// attention.cuh — split-K flash-decode over the fp16 KV ring for one query token, GQA-aware.
//
// Reference semantics (infer.cpp:325-359, 434-444): per q-head h, kv head = h / (n_heads/n_kv_heads);
//   s_t = (sum_i q_i k_{t,i}) / sqrt(head_dim)  for every PHYSICAL slot t in [0, kv_len)   (ring order is irrelevant:
//   softmax is permutation invariant, infer.cpp:340-358 scans slots, not positions)
//   p = softmax(s) (max-subtracted, fp32 expf), out_i = sum_t p_t v_{t,i}.   KV layout (t, kv_head, head_dim), fp16.
//
// Mapping.  The reference walks K and V once per q-head (4-8x re-reads under GQA).  Here a CTA owns one kv head and
// one slice of the sequence and serves all G = n_heads/n_kv_heads query heads from a single pass over its K/V rows:
// HD/8 lanes cover one row with 128-bit loads, so a warp holds 32/(HD/8) timesteps in flight per request and TB
// requests are issued back to back before any arithmetic.  Each lane group keeps an online-softmax state (m, l) per
// head and a partial output for its 8 dims; groups and warps are merged through shared memory, the CTA writes one
// (m, l, acc[G][HD]) partial, and the LAST CTA of the kv head to arrive (atomic ticket) merges the splits in a fixed
// order — no second launch, deterministic result.  The grid is fixed (n_splits x n_kv_heads) so one captured CUDA
// graph serves every kv_len; surplus CTAs retire immediately.
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace xalm {

struct AttnArgs {
	const float* q;        // (n_heads, HD) fp32, already RoPE'd
	const __half* k_cache; // (max_seq_len, n_kv_heads*HD)
	const __half* v_cache;
	float* out;            // (n_heads, HD)
	const StepParams* step; // kv_len read from here when kv_len_fixed < 0
	int kv_len_fixed;
	int n_kv_heads;
	int n_splits;          // gridDim.x
	int min_split;         // smallest slice worth a CTA
	float* part_acc;       // (n_kv_heads, n_splits, G, HD)
	float* part_ml;        // (n_kv_heads, n_splits, G, 2)
	unsigned int* tickets; // (n_kv_heads,) zero-initialised, self-resetting
	const uint8_t* pf_ptr; // first bytes of the next kernel's weights (Wo), pulled into L2 before this kernel waits for q
	unsigned long long pf_bytes;
	// batched decode (BATCH = true, blockIdx.z = sequence): step is the step's StepParams array, k_cache / v_cache are slot 0's
	// caches, and q, out, the split partials and the tickets hold one block per sequence
	int q_stride;          // floats between two sequences' q (and out)
	size_t kv_slot;        // elements between two slots' caches
};

// K/V rows: coherent L2 loads (ld.global.cg).  NOT the read-only path: rows kv_fresh .. kv_pos and the sink rows are written by the QKV
// kernel that may still be running when this kernel's early batch is requested (PDL), and ld.global.nc is only defined for data
// that nobody writes during the kernel's lifetime.
__device__ __forceinline__ uint4 ld_kv16(const __half* p) { return __ldcg(reinterpret_cast<const uint4*>(p)); }

__host__ __device__ inline int attn_split_len(int kv_len, int n_splits, int min_split) {
	int len = (kv_len + n_splits - 1) / n_splits;
	if (len < min_split) len = min_split;
	return len;
}

template <int HD, int G, int NW, bool BATCH = false>
__global__ void __launch_bounds__(NW * 32) attn_decode_kernel(const AttnArgs a) {
	constexpr int LPR = HD / 8;       // lanes per K/V row
	constexpr int RPW = 32 / LPR;     // rows per warp request
	constexpr int TB = 4;             // requests in flight per lane before arithmetic
	constexpr int NGRP = NW * RPW;    // lane groups per CTA
	__shared__ float s_m[NGRP][G], s_l[NGRP][G];
	__shared__ float s_acc[NW][G][HD];
	__shared__ float s_scale[NGRP][G];
	__shared__ bool s_last;

	pdl_launch_dependents();
	int tl = -1;
	if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) tl = tl_begin(300);
	if (threadIdx.x == 0) l2_prefetch_slice(a.pf_ptr, a.pf_bytes, (int) (blockIdx.y * gridDim.x + blockIdx.x), (int) (gridDim.x * gridDim.y));

	// Everything that does not depend on the QKV kernel still running is done BEFORE the dependency wait: the split bounds (the
	// step parameters were written before the graph was launched) and the first batch of K/V rows — only the rows being written
	// this step (kv_fresh .. kv_pos: one row, or the rows of every entry of a span up to this one) and the re-rotated sink rows
	// are fetched again afterwards.
	const int kvh = blockIdx.y, split = blockIdx.x;
	const int z = BATCH ? (int) blockIdx.z : 0;
	const StepParams* step = a.step + z;
	const float* q = a.q + (size_t) z * a.q_stride;
	float* out = a.out + (size_t) z * a.q_stride;
	const size_t kv_off = BATCH ? (size_t) step->slot * a.kv_slot : 0;
	float* part_acc = a.part_acc + (size_t) z * a.n_kv_heads * a.n_splits * G * HD;
	float* part_ml = a.part_ml + (size_t) z * a.n_kv_heads * a.n_splits * G * 2;
	unsigned int* tickets = a.tickets + z * a.n_kv_heads;
	const int kv_len = a.kv_len_fixed >= 0 ? a.kv_len_fixed : step->kv_len;
	const int kv_pos = a.kv_len_fixed >= 0 ? -1 : step->kv_pos;
	const int kv_sink = a.kv_len_fixed >= 0 ? 0 : step->kv_sink;
	const int kv_fresh = a.kv_len_fixed >= 0 ? -1 : step->kv_fresh;
	const int slen = attn_split_len(kv_len, a.n_splits, a.min_split);
	const int n_active = (kv_len + slen - 1) / slen;
	const int t0 = split * slen, t1 = min(kv_len, t0 + slen);

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int sub = lane / LPR, li = lane % LPR; // which row of the request, which 8-dim slice
	const int kv_stride = a.n_kv_heads * HD;
	const float inv_sqrt = 1.0f / sqrtf((float) HD);
	const __half* kbase = a.k_cache + kv_off + (size_t) kvh * HD + li * 8;
	const __half* vbase = a.v_cache + kv_off + (size_t) kvh * HD + li * 8;
	// Batched steps read row t of the sequence where the entry's row map puts it (StepParams::tree).  A tree node i at depth d
	// (xalm_cuda_forward_tree) has kv_fresh = the root's row, kv_pos = kv_fresh + i and kv_len = kv_fresh + d + 1; rows kv_fresh ..
	// kv_len-1 map to its ancestors' rows, root first, then its own.  Since i >= d, kv_pos >= kv_len - 1: every row of this step it
	// reads maps from a t in [kv_fresh, kv_pos], so the re-fetch after the dependency wait below (tested on t) covers all of them.
	// The map is loaded where it is used (read-only path: StepParams rows are written before the step starts) rather than held in a
	// register: that way no BATCH instance spills.
	auto row = [&](int t) -> int {
		if constexpr (!BATCH) {
			return t;
		} else {
			const unsigned int d = (unsigned int) (t - kv_fresh);
			return d < 8u ? kv_fresh + (int) ((__ldg(&step->tree) >> (3u * d)) & 7u) : t;
		}
	};

	uint4 kn[TB], vn[TB]; // next batch, requested one iteration ahead
	auto fetch = [&](int tb) {
#pragma unroll
		for (int j = 0; j < TB; j++) {
			const int t = tb + j * RPW + sub;
			const int tc = row(t < t1 ? t : t0);
			kn[j] = ld_kv16(kbase + (size_t) tc * kv_stride);
			vn[j] = ld_kv16(vbase + (size_t) tc * kv_stride);
		}
	};
	const int tb_first = t0 + warp * RPW * TB;
	const bool early = a.kv_len_fixed < 0 && split < n_active && tb_first < t1;
	if (early) fetch(tb_first);

	pdl_wait();
	tl_mark(tl, 2);
	if (split >= n_active) return;

	// this lane's 8 dims of each of the G query heads
	float qf[G][8];
#pragma unroll
	for (int g = 0; g < G; g++) {
		const float* qp = q + (size_t) (kvh * G + g) * HD + li * 8;
		const float4 u = ld_act4(qp), v = ld_act4(qp + 4);
		qf[g][0] = u.x; qf[g][1] = u.y; qf[g][2] = u.z; qf[g][3] = u.w;
		qf[g][4] = v.x; qf[g][5] = v.y; qf[g][6] = v.z; qf[g][7] = v.w;
	}
	float m[G], l[G], acc[G][8];
#pragma unroll
	for (int g = 0; g < G; g++) {
		m[g] = -CUDART_INF_F; l[g] = 0.f;
#pragma unroll
		for (int i = 0; i < 8; i++) acc[g][i] = 0.f;
	}
	if (early) { // rows the QKV kernel wrote this step: take them again now that it has completed
#pragma unroll
		for (int j = 0; j < TB; j++) {
			const int t = tb_first + j * RPW + sub;
			if (t < t1 && ((t >= kv_fresh && t <= kv_pos) || t < kv_sink)) {
				kn[j] = ld_kv16(kbase + (size_t) row(t) * kv_stride);
				vn[j] = ld_kv16(vbase + (size_t) row(t) * kv_stride);
			}
		}
	} else if (tb_first < t1) fetch(tb_first);
	for (int tb = tb_first; tb < t1; tb += NW * RPW * TB) {
		uint4 kq[TB], vq[TB];
		bool ok[TB];
#pragma unroll
		for (int j = 0; j < TB; j++) {
			ok[j] = tb + j * RPW + sub < t1;
			kq[j] = kn[j];
			vq[j] = vn[j];
		}
		if (tb + NW * RPW * TB < t1) fetch(tb + NW * RPW * TB);
		float s[TB][G];
#pragma unroll
		for (int j = 0; j < TB; j++) {
			const __half2* kh = reinterpret_cast<const __half2*>(&kq[j]);
			float kf[8];
#pragma unroll
			for (int i = 0; i < 4; i++) {
				const float2 f = __half22float2(kh[i]);
				kf[2 * i] = f.x; kf[2 * i + 1] = f.y;
			}
#pragma unroll
			for (int g = 0; g < G; g++) {
				float p = 0.f;
#pragma unroll
				for (int i = 0; i < 8; i++) p += qf[g][i] * kf[i];
#pragma unroll
				for (int o = LPR / 2; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
				s[j][g] = ok[j] ? p * inv_sqrt : -CUDART_INF_F;
			}
		}
#pragma unroll
		for (int g = 0; g < G; g++) {
			float mn = m[g];
#pragma unroll
			for (int j = 0; j < TB; j++) mn = fmaxf(mn, s[j][g]);
			if (mn == -CUDART_INF_F) continue; // nothing valid yet for this lane group
			const float corr = expf(m[g] - mn);   // m = -inf -> 0
			l[g] *= corr;
#pragma unroll
			for (int i = 0; i < 8; i++) acc[g][i] *= corr;
			m[g] = mn;
#pragma unroll
			for (int j = 0; j < TB; j++) {
				const float p = expf(s[j][g] - mn); // masked rows: exp(-inf) = 0
				l[g] += p;
				const __half2* vh = reinterpret_cast<const __half2*>(&vq[j]);
#pragma unroll
				for (int i = 0; i < 4; i++) {
					const float2 f = __half22float2(vh[i]);
					acc[g][2 * i] += p * f.x;
					acc[g][2 * i + 1] += p * f.y;
				}
			}
		}
	}

	// ---- merge lane groups and warps of the CTA ----
	const int grp = warp * RPW + sub;
	if (li == 0) {
#pragma unroll
		for (int g = 0; g < G; g++) { s_m[grp][g] = m[g]; s_l[grp][g] = l[g]; }
	}
	__syncthreads();
	float M[G];
#pragma unroll
	for (int g = 0; g < G; g++) {
		float mm = -CUDART_INF_F;
		for (int i = 0; i < NGRP; i++) mm = fmaxf(mm, s_m[i][g]);
		M[g] = mm;
	}
	// rescale own partial to the CTA max, then reduce the RPW groups of this warp with shuffles
#pragma unroll
	for (int g = 0; g < G; g++) {
		const float sc = m[g] == -CUDART_INF_F ? 0.f : expf(m[g] - M[g]);
		if (li == 0) s_scale[grp][g] = sc;
#pragma unroll
		for (int i = 0; i < 8; i++) {
			float v = acc[g][i] * sc;
#pragma unroll
			for (int o = LPR; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
			acc[g][i] = v;
		}
		if (sub == 0) {
#pragma unroll
			for (int i = 0; i < 8; i++) s_acc[warp][g][li * 8 + i] = acc[g][i];
		}
	}
	__syncthreads();
	float* pacc = part_acc + ((size_t) kvh * a.n_splits + split) * G * HD;
	float* pml = part_ml + ((size_t) kvh * a.n_splits + split) * G * 2;
	if (n_active == 1) {
		// the whole sequence fit in one split: normalise and write the output directly (no partial round trip, no ticket)
		for (int i = threadIdx.x; i < G * HD; i += NW * 32) {
			const int g = i / HD, dpos = i % HD;
			float v = 0.f, L = 0.f;
#pragma unroll
			for (int w = 0; w < NW; w++) v += s_acc[w][g][dpos];
			for (int k = 0; k < NGRP; k++) L += s_l[k][g] * s_scale[k][g];
			out[(size_t) kvh * G * HD + i] = v / L;
		}
		tl_mark(tl, 3);
		return;
	}
	for (int i = threadIdx.x; i < G * HD; i += NW * 32) {
		const int g = i / HD, dpos = i % HD;
		float v = 0.f;
#pragma unroll
		for (int w = 0; w < NW; w++) v += s_acc[w][g][dpos];
		pacc[i] = v;
	}
	if (threadIdx.x < G) {
		const int g = threadIdx.x;
		float L = 0.f;
		for (int i = 0; i < NGRP; i++) L += s_l[i][g] * s_scale[i][g];
		// M recomputed per thread g (registers above are per-thread copies of all G maxima)
		float mm = -CUDART_INF_F;
		for (int i = 0; i < NGRP; i++) mm = fmaxf(mm, s_m[i][g]);
		pml[2 * g] = mm;
		pml[2 * g + 1] = L;
	}

	// ---- last CTA of this kv head merges the splits (fixed order) ----
	__threadfence();
	__syncthreads();
	if (threadIdx.x == 0) {
		const unsigned int ticket = atomicAdd(&tickets[kvh], 1u);
		s_last = ticket == (unsigned int) (n_active - 1);
		if (s_last) tickets[kvh] = 0; // ready for the next launch
	}
	__syncthreads();
	tl_mark(tl, 3);
	if (!s_last) return;
	__threadfence();
	const float* bacc = part_acc + (size_t) kvh * a.n_splits * G * HD;
	const float* bml = part_ml + (size_t) kvh * a.n_splits * G * 2;
	// every partial of this thread's first four outputs is requested BEFORE the scales are computed: one L2 round trip for up
	// to 16 splits, overlapped with the (m, l) pass, instead of a chain of dependent ones after it
	constexpr int MB = 16;
	float4 pv[MB];
	auto preload = [&](int i4, int s0) {
#pragma unroll
		for (int k = 0; k < MB; k++)
			if (s0 + k < n_active) pv[k] = __ldcg(reinterpret_cast<const float4*>(bacc + (size_t) (s0 + k) * G * HD + i4));
	};
	if ((int) threadIdx.x * 4 < G * HD) preload((int) threadIdx.x * 4, 0);
	// (m, l) of every split -> shared memory (reusing s_acc), then per-head max, rescale factors and denominators
	float* s_ml = &s_acc[0][0][0];                 // [n_active][G][2]   (n_active * G * 2 <= NW * G * HD)
	float* s_sc = s_ml + (size_t) n_active * G * 2; // [n_active][G]
	for (int i = threadIdx.x; i < n_active * G * 2; i += NW * 32) s_ml[i] = __ldcg(bml + i);
	__syncthreads();
	__shared__ float s_den[G];
	if (threadIdx.x < G) {
		const int g = threadIdx.x;
		float mm = -CUDART_INF_F;
		for (int sidx = 0; sidx < n_active; sidx++) mm = fmaxf(mm, s_ml[(sidx * G + g) * 2]);
		float den = 0.f;
		for (int sidx = 0; sidx < n_active; sidx++) {
			const float sc = expf(s_ml[(sidx * G + g) * 2] - mm);
			s_sc[sidx * G + g] = sc;
			den += sc * s_ml[(sidx * G + g) * 2 + 1];
		}
		s_den[g] = den;
	}
	__syncthreads();
	for (int i4 = threadIdx.x * 4; i4 < G * HD; i4 += NW * 32 * 4) {
		const int g = i4 / HD;
		float4 num = make_float4(0.f, 0.f, 0.f, 0.f);
		for (int s0 = 0; s0 < n_active; s0 += MB) {
			if (s0 > 0 || i4 != (int) threadIdx.x * 4) preload(i4, s0); // the first batch is already in flight
#pragma unroll
			for (int k = 0; k < MB; k++) {
				if (s0 + k < n_active) {
					const float sc = s_sc[(s0 + k) * G + g];
					num.x += sc * pv[k].x; num.y += sc * pv[k].y; num.z += sc * pv[k].z; num.w += sc * pv[k].w;
				}
			}
		}
		const float den = s_den[g];
		*reinterpret_cast<float4*>(out + (size_t) kvh * G * HD + i4) = make_float4(num.x / den, num.y / den, num.z / den, num.w / den);
	}
}

#ifndef XALM_SECONDARY_TU // non-template kernel: defined once, in xalm_cuda.cu's translation unit
// ---- attention probabilities for the `att` scratch argument of mha (model.h:289-307): test hook only, one CTA per
//      head, the three passes of infer.cpp:340-349 as written. ----
__global__ void attn_probs_kernel(const float* q, const __half* k_cache, float* att, int head_dim, int n_kv_heads,
                                  int n_heads, int kv_len, int max_seq_len) {
	const int h = blockIdx.x;
	const int kvh = h / (n_heads / n_kv_heads);
	const int kv_stride = n_kv_heads * head_dim;
	float* at = att + (size_t) h * max_seq_len;
	__shared__ float s_red[32];
	const float inv_sqrt = 1.0f / sqrtf((float) head_dim);
	float mx = -CUDART_INF_F;
	for (int t = threadIdx.x; t < kv_len; t += blockDim.x) {
		float s = 0.f;
		for (int i = 0; i < head_dim; i++) s += q[(size_t) h * head_dim + i] * __half2float(k_cache[(size_t) t * kv_stride + kvh * head_dim + i]);
		s *= inv_sqrt;
		at[t] = s;
		mx = fmaxf(mx, s);
	}
	mx = warp_max(mx);
	if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = mx;
	__syncthreads();
	mx = -CUDART_INF_F;
	for (int i = 0; i < (blockDim.x + 31) / 32; i++) mx = fmaxf(mx, s_red[i]);
	__syncthreads();
	float sum = 0.f;
	for (int t = threadIdx.x; t < kv_len; t += blockDim.x) {
		const float e = expf(at[t] - mx);
		at[t] = e;
		sum += e;
	}
	sum = warp_sum(sum);
	if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = sum;
	__syncthreads();
	sum = 0.f;
	for (int i = 0; i < (blockDim.x + 31) / 32; i++) sum += s_red[i];
	for (int t = threadIdx.x; t < kv_len; t += blockDim.x) at[t] /= sum;
}

#endif // XALM_SECONDARY_TU

} // namespace xalm
