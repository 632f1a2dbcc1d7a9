// matvec.cuh — the decode hot kernel: xout = W(d,n) · x(n), W in any reference weight format, fp32 activations and
// accumulation (infer.cpp:104-135), with the surrounding element-wise ops of Block::_block_cpu fused in:
//
//   prologue (optional)   x' = rmsnorm(x) * g                                   infer.cpp:224-236, :376, :457, :628
//   epilogue STORE        out[i]  = y_i                                         classifier, infer.cpp:637
//            RESIDUAL     out[i] += y_i                                         infer.cpp:447-452, :490-494
//            GLU          out[i]  = act(y_i^{W1}) * y_i^{W3}                    infer.cpp:468-488
//            QKV          clip -> RoPE(q,k) -> q fp32, k/v fp16 into the KV ring at kv_pos; the block that owns
//                         virtual row 0 also re-rotates the attention sinks     infer.cpp:388-431
//
// Mapping.  HBM-bound: every weight byte is read exactly once, with 128-bit streaming loads that bypass L1
// allocation; x is small (<= 114 KB) and is read through L1, where it stays resident for all warps of the SM.
// One warp owns R consecutive rows so each x chunk it loads is reused R times from registers (otherwise the
// 4-byte activations would cost more L1 bandwidth than the <= 1-byte weights cost HBM bandwidth).  KS warps of a
// CTA split K for the same rows when rows are scarce (Wo/W2: 4096 rows must still cover 148 SMs evenly); partial
// sums are combined in a fixed order through shared memory, so results are deterministic run to run.
//
// PDL.  The kernel is launched with programmatic stream serialisation: it fetches its first weight fragments —
// which no earlier kernel writes — BEFORE griddepcontrol.wait, so the HBM stream does not drain at kernel
// boundaries; activations are only touched after the wait.
#pragma once
#include <math_constants.h>

#include "formats.cuh"

namespace xalm {

enum { EPI_STORE = 0, EPI_RESIDUAL = 1, EPI_GLU = 2, EPI_QKV = 3 };

struct MatvecArgs {
	WMat w;              // weights; for GLU rows [0,d) are W1 and [glu_off, glu_off+d) are W3
	const float* x;      // (n,) input activations
	int n;               // K
	int d;               // number of OUTPUT values (GLU: hidden_dim; else rows)
	int epi;
	int glu_off;         // row offset of W3 inside w (GLU only)
	int act;             // xalm_act (GLU only)
	// rmsnorm prologue
	const uint8_t* norm_w; // nullptr = no norm
	int norm_type;       // XALM_F32 or XALM_BF16
	float norm_eps;
	// outputs
	float* out;          // STORE / RESIDUAL / GLU target, QKV: q (q_dim,)
	// QKV epilogue
	const StepParams* step;
	__half* k_cache;     // (max_seq_len, kv_dim)
	__half* v_cache;
	const float* rope_freq; // (head_dim/2,) 1/powf(theta, j/rotary_dim) computed on the host (0 beyond rotary_dim)
	int q_dim, kv_dim, head_dim;
	float qkv_clip;
	// one-byte LUT formats
	int lut_type;        // 0 = none, else the type id whose 256 values fill the shared-memory table
	// tail prefetch: when this CTA's producer has issued its last weight load it pulls its share of the NEXT kernel's first
	// bytes into L2, so that kernel's ramp-up reads hit L2 instead of paying an HBM round trip after the dependency wait
	const uint8_t* pf_ptr;       // next kernel's weights (or nullptr)
	unsigned long long pf_bytes;
	int pf_kv;                   // 1: also prefetch rows [0, kv_len) of k_cache / v_cache (the attention kernel that follows QKV)
	// rmsnorm weights of the NEXT norm-fused kernel (read once per token, i.e. from DRAM): CTA 0 pulls them into L2 at entry.  That
	// kernel requests them before its dependency wait; coming from DRAM behind its own weight stream they took ~2.5 us, and the
	// activation loads issued after them return in order behind them (profiles/r2_decode_timeline.md)
	const uint8_t* pf_norm_ptr;
	unsigned int pf_norm_bytes;
	// tensor-parallel exchange fused into the matvec kernels, LL style: the row-split matvecs (Wo, W2) PUSH every partial row as
	// an 8-byte {value, sequence tag} word straight into every rank's receive slot over NVLink (posted stores, no fence, no flag,
	// no extra kernel); the next kernel's rmsnorm prologue polls the tags of the words it needs and adds the partials (fixed rank
	// order) to the residual stream (tp_receive).
	uint2* push_dst[8];          // per destination rank: its receive slot for THIS rank's partial, (dim,) {float bits, tag}
	int n_push;                  // 0 = off
	int push_idx;                // exchange index inside the token: tag = step->ar_base + push_idx + 1
	const uint2* recv;           // local receive slot: (n_recv, dim) words
	int n_recv;                  // 0 = off
	int recv_idx;
	float* x_out;                // the first CTAs store x + sum(partials) here: the residual stream after the exchange
	unsigned int* err_flag;      // set to 1 when a wait for a peer's words times out (the host turns it into XALM_ERR_COMM)
	uint2* xl;                   // local (dim,) {value, tag} words: the reducing CTAs publish the summed stream here, every CTA polls it
};

__device__ __forceinline__ float act_gelu(float x) { return 0.5f * x * (1.0f + tanhf(0.797885f * (x + 0.044715f * x * x * x))); }
__device__ __forceinline__ float act_silu(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float clipf(float x, float v) { return x < -v ? -v : (x > v ? v : x); }

// rotate the pair (v0, v1) that sits at even head offset j_head by pos * freq (infer.cpp:305-322)
__device__ __forceinline__ void rope_pair(float& v0, float& v1, int j_head, int pos, const float* freq_tab) {
	const float freq = freq_tab[j_head >> 1];
	const float val = (float) pos * freq;
	float fci, fcr;
	sincosf(val, &fci, &fcr);
	const float a = v0, b = v1;
	v0 = a * fcr - b * fci;
	v1 = a * fci + b * fcr;
}

// Re-rotate the kv_sink attention-sink keys of k_cache by one position, through fp16 (infer.cpp:421-431).  Threads tid = 0 .. nt-1
// of the block share the work: in the warp-specialised kernels nt is the consumer thread count, not blockDim.x, because their
// producer warp has returned by then.
__device__ __forceinline__ void rotate_sinks(const MatvecArgs& a, __half* k_cache, int kv_sink, int tid, int nt) {
	const int pairs = a.kv_dim / 2;
	for (int i = tid; i < kv_sink * pairs; i += nt) {
		const int r = i / pairs, p = i % pairs;
		__half2* kp = reinterpret_cast<__half2*>(k_cache + (size_t) r * a.kv_dim) + p;
		float2 v = __half22float2(*kp);
		rope_pair(v.x, v.y, (2 * p) % a.head_dim, 1, a.rope_freq);
		*kp = __floats2half2_rn(v.x, v.y);
	}
}

// One QKV output pair (row, row + 1) of the sequence sp, row even: clip -> RoPE(q, k) -> q fp32 into out, k / v fp16 into the KV
// ring of slot sp.slot at sp.kv_pos (infer.cpp:388-420).  kv_slot = elements between two slots' caches (0: one cache).
__device__ __forceinline__ void qkv_pair(const MatvecArgs& a, const StepParams& sp, size_t kv_slot, float* out, int row, float y0, float y1) {
	const int pos = sp.pos, kv_pos = sp.kv_pos;
	float v0 = clipf(y0, a.qkv_clip), v1 = clipf(y1, a.qkv_clip);
	if (row < a.q_dim) {
		rope_pair(v0, v1, row % a.head_dim, pos, a.rope_freq);
		out[row] = v0;
		out[row + 1] = v1;
	} else if (row < a.q_dim + a.kv_dim) {
		const int i = row - a.q_dim;
		rope_pair(v0, v1, i % a.head_dim, pos, a.rope_freq);
		__half* kc = a.k_cache + (size_t) sp.slot * kv_slot;
		*reinterpret_cast<__half2*>(kc + (size_t) kv_pos * a.kv_dim + i) = __floats2half2_rn(v0, v1);
	} else {
		const int i = row - a.q_dim - a.kv_dim;
		__half* vc = a.v_cache + (size_t) sp.slot * kv_slot;
		*reinterpret_cast<__half2*>(vc + (size_t) kv_pos * a.kv_dim + i) = __floats2half2_rn(v0, v1);
	}
}

template <int R>
__device__ __forceinline__ void epilogue(const MatvecArgs& a, int row0, const float (&y)[R]) {
	// called by ONE thread per row group with the R finished dot products; row0 = first virtual row
	if (a.epi == EPI_STORE) {
#pragma unroll
		for (int r = 0; r < R; r++)
			if (row0 + r < a.d) a.out[row0 + r] = y[r];
	} else if (a.epi == EPI_RESIDUAL) {
#pragma unroll
		for (int r = 0; r < R; r++)
			if (row0 + r < a.d) a.out[row0 + r] += y[r];
	} else if (a.epi == EPI_GLU) {
		// rows [0,R/2) came from W1, [R/2,R) from W3, output index = row0/2 + r
		const int o0 = row0 / 2;
#pragma unroll
		for (int r = 0; r < R / 2; r++) {
			if (o0 + r < a.d) {
				const float g = a.act == XALM_SILU ? act_silu(y[r]) : act_gelu(y[r]);
				a.out[o0 + r] = g * y[R / 2 + r];
			}
		}
	} else { // EPI_QKV
		const StepParams sp = *a.step;
#pragma unroll
		for (int r = 0; r < R; r += 2) {
			const int row = row0 + r;
			if (row >= a.d) break;
			qkv_pair(a, sp, 0, a.out, row, y[r], y[r + 1]);
		}
	}
}

// ---- shared by the warp-specialised kernels (matvec_tma.cuh, matvec_idp.cuh, matvec_mma.cuh) ---------------------------------------

constexpr unsigned int XALM_SPIN_LIMIT = 1u << 23; // polls of a tagged word (~1 us each) before a tensor-parallel wait gives up

// Four consecutive {value, tag} words: poll until all carry the exchange's tag seq and return the values.  A peer that never
// writes them has died: after XALM_SPIN_LIMIT polls set *err_flag (the host turns it into XALM_ERR_COMM) instead of hanging the GPU.
__device__ __forceinline__ float4 poll_tagged4(const uint2* src, unsigned int seq, unsigned int* err_flag) {
	uint4 w0, w1;
	unsigned int spins = 0;
	do {
		asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w0.x), "=r"(w0.y), "=r"(w0.z), "=r"(w0.w) : "l"(src));
		asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w1.x), "=r"(w1.y), "=r"(w1.z), "=r"(w1.w) : "l"(src + 2));
		if (++spins > XALM_SPIN_LIMIT) { if (err_flag) *err_flag = 1u; break; }
	} while (w0.y != seq || w0.w != seq || w1.y != seq || w1.w != seq);
	return make_float4(__uint_as_float(w0.x), __uint_as_float(w0.z), __uint_as_float(w1.x), __uint_as_float(w1.z));
}

// Tensor-parallel receive (LL style), run by the nt consumer threads of a norm-fused kernel with n_recv set: the first min(grid, 8)
// CTAs each reduce a slice of the stream — x += sum over ranks of the partial rows the previous row-split matvec pushed here (rank
// order: identical bits on every rank; infer.cpp:450-452 / :492-494) — store it to x_out and publish it locally as {value, tag}
// words, so every other CTA reads dim words instead of n_ranks x dim.
__device__ __forceinline__ void tp_receive(const MatvecArgs& a, int tid, int nt) {
	const int n_red = min((int) gridDim.x, 8);
	if ((int) blockIdx.x >= n_red) return;
	const unsigned int seq = a.step->ar_base + (unsigned int) a.recv_idx + 1u;
	const int chunk = ((a.n / 4 + n_red - 1) / n_red) * 4;
	const int i0 = (int) blockIdx.x * chunk, i1 = min(a.n, i0 + chunk);
	for (int i = i0 + tid * 4; i < i1; i += nt * 4) {
		float4 v = ld_act4(a.x + i);
		float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
		for (int p = 0; p < a.n_recv; p++) {
			const float4 w = poll_tagged4(a.recv + (size_t) p * a.n + i, seq, a.err_flag);
			sum.x += w.x; sum.y += w.y; sum.z += w.z; sum.w += w.w;
		}
		v.x += sum.x; v.y += sum.y; v.z += sum.z; v.w += sum.w;
		*reinterpret_cast<float4*>(a.x_out + i) = v;
		*reinterpret_cast<uint4*>(a.xl + i) = make_uint4(__float_as_uint(v.x), seq, __float_as_uint(v.y), seq);
		*reinterpret_cast<uint4*>(a.xl + i + 2) = make_uint4(__float_as_uint(v.z), seq, __float_as_uint(v.w), seq);
	}
}

// The staging input x[8 grp .. 8 grp + 8): with recv, the summed stream the reducing CTAs publish as {value, tag} words (poll this
// exchange's tag), else x itself
__device__ __forceinline__ void load_x8(const MatvecArgs& a, int grp, bool recv, float (&v)[8]) {
	float4 q0, q1;
	if (recv) {
		const unsigned int seq = a.step->ar_base + (unsigned int) a.recv_idx + 1u;
		q0 = poll_tagged4(a.xl + grp * 8, seq, a.err_flag);
		q1 = poll_tagged4(a.xl + grp * 8 + 4, seq, a.err_flag);
	} else {
		q0 = ld_act4(a.x + grp * 8);
		q1 = ld_act4(a.x + grp * 8 + 4);
	}
	v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w;
	v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
}

// rmsnorm weights of the 8-element group grp, raw: two uint4 of F32, or one of BF16
__device__ __forceinline__ void load_norm8(const uint8_t* norm_w, int norm_type, int grp, uint4 (&gw)[2]) {
	if (norm_type == XALM_F32) {
		gw[0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(norm_w) + grp * 8);
		gw[1] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(norm_w) + grp * 8 + 4);
	} else {
		gw[0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(norm_w) + grp * 8);
	}
}
// element e of a group load_norm8 fetched
__device__ __forceinline__ float norm_weight(const uint4 (&gw)[2], int norm_type, int e) {
	if (norm_type == XALM_F32) {
		const uint4 q = gw[e >> 2];
		return __uint_as_float((e & 3) == 0 ? q.x : (e & 3) == 1 ? q.y : (e & 3) == 2 ? q.z : q.w);
	}
	const uint4 q = gw[0];
	const int h = e >> 1;
	const uint32_t u = h == 0 ? q.x : h == 1 ? q.y : h == 2 ? q.z : q.w;
	return __uint_as_float((e & 1) ? (u & 0xFFFF0000u) : (u << 16));
}

// Producer warp, at entry: CTA 0 pulls the next norm-fused kernel's rmsnorm weights into L2 (pf_norm_ptr)
__device__ __forceinline__ void prefetch_next_norm(const MatvecArgs& a) {
	if (blockIdx.x == 0 && a.pf_norm_ptr && a.pf_norm_bytes >= 16)
		asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.pf_norm_ptr), "r"(a.pf_norm_bytes & ~15u) : "memory");
}
// Producer warp, after its last weight load: this CTA's slice of the next kernel's weights and, with kv and pf_kv set, of the K/V
// rows the attention kernel after QKV reads
__device__ __forceinline__ void prefetch_tail(const MatvecArgs& a, bool kv) {
	l2_prefetch_slice(a.pf_ptr, a.pf_bytes, (int) blockIdx.x, (int) gridDim.x);
	if (kv && a.pf_kv) {
		const unsigned long long kvb = (unsigned long long) a.step->kv_len * a.kv_dim * sizeof(__half);
		l2_prefetch_slice(reinterpret_cast<const uint8_t*>(a.k_cache), kvb, (int) blockIdx.x, (int) gridDim.x);
		l2_prefetch_slice(reinterpret_cast<const uint8_t*>(a.v_cache), kvb, (int) blockIdx.x, (int) gridDim.x);
	}
}

// Epilogue of a finished tile of RC rows, run by one whole warp: lane i < RC holds the sum yv of row row0 + i and, for EPI_RESIDUAL,
// the old activation xold of that row.  GLU pairs the W1 row of lane i with the W3 row RC/2 lanes up; otherwise even lanes hand a
// row pair to epilogue<2> (RoPE needs both) or, tensor parallel, push it to every rank.
template <int RC>
__device__ __forceinline__ void row_epilogue(const MatvecArgs& a, int row0, int lane, float yv, float xold) {
	const float ynext = __shfl_down_sync(0xffffffffu, yv, 1);
	if (a.epi == EPI_GLU) {
		const float ypart = __shfl_down_sync(0xffffffffu, yv, RC / 2); // W3 value for the W1 row in this lane
		const int o = row0 / 2 + lane;
		if (lane < RC / 2 && o < a.d) {
			const float g = a.act == XALM_SILU ? act_silu(yv) : act_gelu(yv);
			a.out[o] = g * ypart;
		}
		return;
	}
	const int row = row0 + lane;
	if (lane >= RC || row >= a.d) return;
	if (a.epi == EPI_RESIDUAL) {
		a.out[row] = xold + yv;
	} else if ((lane & 1) == 0) {
		if (a.epi == EPI_STORE && a.n_push) { // tensor parallel: this rank's partial rows go to every rank (NVLink stores)
			const unsigned int seq = a.step->ar_base + (unsigned int) a.push_idx + 1u;
			const uint4 w = make_uint4(__float_as_uint(yv), seq, __float_as_uint(ynext), seq);
			for (int p = 0; p < a.n_push; p++) *reinterpret_cast<uint4*>(a.push_dst[p] + row) = w;
		} else {
			const float y2[2] = {yv, ynext};
			epilogue<2>(a, row, y2);
		}
	}
}

// virtual row (what the epilogue sees) -> physical weight row
__device__ __forceinline__ int phys_row(const MatvecArgs& a, int row0, int r, int R) {
	if (a.epi == EPI_GLU) {
		const int o0 = row0 / 2;
		return r < R / 2 ? o0 + r : a.glu_off + o0 + (r - R / 2);
	}
	return row0 + r;
}
__device__ __forceinline__ bool row_valid(const MatvecArgs& a, int row0, int r, int R) {
	if (a.epi == EPI_GLU) return row0 / 2 + (r % (R / 2)) < a.d;
	return row0 + r < a.d;
}

// TYPE: format tag (an xalm_type, or -1 for the shared-memory LUT path).  R rows per warp, KS warps split K,
// NW warps per CTA.  NORM: fused rmsnorm prologue.
template <int TYPE, int R, int KS, int NW, bool NORM>
__global__ void __launch_bounds__(NW * 32) matvec_kernel(const MatvecArgs a) {
	using F = Fmt<TYPE>;
	constexpr int E = F::E;
	constexpr int GROUPS = NW / KS; // row groups per CTA
	__shared__ float s_part[GROUPS][KS][R];
	__shared__ float s_red[NW];
	__shared__ float s_lut[TYPE == -1 ? 256 : 1];

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int group = warp / KS, ks = warp % KS;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d; // virtual rows
	const int row0 = (blockIdx.x * GROUPS + group) * R;
	const bool active = row0 < vrows;

	pdl_launch_dependents();
	int tl = -1;
	if (blockIdx.x == 0 && threadIdx.x == 0) tl = tl_begin(200 + a.epi);

	RowPtr rp[R];
#pragma unroll
	for (int r = 0; r < R; r++) {
		const int pr = (active && row_valid(a, row0, r, R)) ? phys_row(a, row0, r, R) : (active ? phys_row(a, row0, 0, R) : 0);
		rp[r] = {a.w.p0 + (size_t) pr * a.w.s0, a.w.p1 + (size_t) pr * a.w.s1, a.w.p2 + (size_t) pr * a.w.s2};
	}
	const int nchunks = a.n / E;
	int c = ks * 32 + lane;

	// ---- first weight fragments are requested before we wait on the previous kernel ----
	typename F::Frag frag[R];
	if (active && c < nchunks) {
#pragma unroll
		for (int r = 0; r < R; r++) frag[r] = F::load(rp[r], c);
	}

	if (TYPE == -1) {
		for (int i = threadIdx.x; i < 256; i += NW * 32) s_lut[i] = decode_byte_type(a.lut_type, (uint8_t) i);
	}

	pdl_wait(); // activations (and the KV ring) written by earlier kernels are visible from here on
	tl_mark(tl, 2);

	if (a.epi == EPI_QKV && blockIdx.x == 0 && a.step->kv_sink > 0) rotate_sinks(a, a.k_cache, a.step->kv_sink, threadIdx.x, blockDim.x);

	// ---- rmsnorm prologue: every CTA recomputes the scale (n floats from L1/L2, hidden under the weight fetch) ----
	float scale = 1.0f;
	if (NORM) {
		float ss = 0.f;
		for (int i = threadIdx.x * 4; i < a.n; i += NW * 32 * 4) {
			const float4 v = ld_act4(a.x + i);
			ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
		}
		ss = warp_sum(ss);
		if (lane == 0) s_red[warp] = ss;
		__syncthreads();
		float tot = 0.f;
#pragma unroll
		for (int i = 0; i < NW; i++) tot += s_red[i];
		scale = 1.0f / sqrtf(tot / (float) a.n + a.norm_eps);
	} else if (TYPE == -1) {
		__syncthreads();
	}

	f32x2 acc[R];
#pragma unroll
	for (int r = 0; r < R; r++) acc[r] = pack2(0.f, 0.f);

	if (active) {
		while (c < nchunks) {
			// activations for this chunk
			float xv[E];
#pragma unroll
			for (int i = 0; i < E; i += 4) {
				const float4 v = ld_act4(a.x + (size_t) c * E + i);
				xv[i] = v.x; xv[i + 1] = v.y; xv[i + 2] = v.z; xv[i + 3] = v.w;
			}
			if (NORM) {
				// o[i] = x[i] * scale * weight[i]  (infer.cpp:233-235)
				if (a.norm_type == XALM_F32) {
					const float* g = reinterpret_cast<const float*>(a.norm_w) + (size_t) c * E;
#pragma unroll
					for (int i = 0; i < E; i += 4) {
						const float4 gv = ld_act4(g + i);
						xv[i] = xv[i] * scale * gv.x; xv[i + 1] = xv[i + 1] * scale * gv.y;
						xv[i + 2] = xv[i + 2] * scale * gv.z; xv[i + 3] = xv[i + 3] * scale * gv.w;
					}
				} else {
					const uint16_t* g = reinterpret_cast<const uint16_t*>(a.norm_w) + (size_t) c * E;
#pragma unroll
					for (int i = 0; i < E; i += 4) {
						const uint2 gv = *reinterpret_cast<const uint2*>(g + i);
						xv[i] = xv[i] * scale * __uint_as_float(gv.x << 16); xv[i + 1] = xv[i + 1] * scale * __uint_as_float(gv.x & 0xFFFF0000u);
						xv[i + 2] = xv[i + 2] * scale * __uint_as_float(gv.y << 16); xv[i + 3] = xv[i + 3] * scale * __uint_as_float(gv.y & 0xFFFF0000u);
					}
				}
			}
			// next fragments go out before this chunk's arithmetic
			const int cn = c + KS * 32;
			typename F::Frag nxt[R];
			if (cn < nchunks) {
#pragma unroll
				for (int r = 0; r < R; r++) nxt[r] = F::load(rp[r], cn);
			}
#pragma unroll
			for (int r = 0; r < R; r++) {
				if constexpr (TYPE == -1) F::fma_chunk_lut(frag[r], xv, acc[r], s_lut);
				else F::fma_chunk(frag[r], xv, acc[r]);
			}
			if (cn < nchunks) {
#pragma unroll
				for (int r = 0; r < R; r++) frag[r] = nxt[r];
			}
			c = cn;
		}
	}

	float y[R];
#pragma unroll
	for (int r = 0; r < R; r++) {
		float lo, hi;
		unpack2(acc[r], lo, hi);
		y[r] = warp_sum(lo + hi);
	}
	if (KS == 1) {
		if (active && lane == 0) epilogue<R>(a, row0, y);
	} else {
		if (lane == 0) {
#pragma unroll
			for (int r = 0; r < R; r++) s_part[group][ks][r] = y[r];
		}
		__syncthreads();
		if (active && ks == 0 && lane == 0) {
#pragma unroll
			for (int r = 0; r < R; r++) {
				float t = 0.f;
#pragma unroll
				for (int k = 0; k < KS; k++) t += s_part[group][k][r];
				y[r] = t;
			}
			epilogue<R>(a, row0, y);
		}
	}
	tl_mark(tl, 3);
}

// ---- TQ1_0 (quants.py:664-683): 256 weights in 54 bytes, base-3 packed.  Not a 16-byte-chunk format: one warp
//      walks a row block by block, lane B decodes byte B (5 trits) of qs0, lanes 0-15 byte B of qs1, lanes 0-3 qh. ----
template <int R, int NW, bool NORM>
__global__ void __launch_bounds__(NW * 32) matvec_tq1_kernel(const MatvecArgs a) {
	__shared__ float s_red[NW];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	const int row0 = (blockIdx.x * NW + warp) * R;
	const bool active = row0 < vrows;
	pdl_launch_dependents();
	pdl_wait();
	if (a.epi == EPI_QKV && blockIdx.x == 0 && a.step->kv_sink > 0) rotate_sinks(a, a.k_cache, a.step->kv_sink, threadIdx.x, blockDim.x);
	float scale = 1.0f;
	if (NORM) {
		float ss = 0.f;
		for (int i = threadIdx.x; i < a.n; i += NW * 32) ss += a.x[i] * a.x[i];
		ss = warp_sum(ss);
		if (lane == 0) s_red[warp] = ss;
		__syncthreads();
		float tot = 0.f;
		for (int i = 0; i < NW; i++) tot += s_red[i];
		scale = 1.0f / sqrtf(tot / (float) a.n + a.norm_eps);
	}
	auto xval = [&](int j) -> float {
		float v = a.x[j];
		if (NORM) v = v * scale * (a.norm_type == XALM_F32 ? reinterpret_cast<const float*>(a.norm_w)[j]
		                                                   : bf16_bits_to_f32(reinterpret_cast<const uint16_t*>(a.norm_w)[j]));
		return v;
	};
	float y[R];
#pragma unroll
	for (int r = 0; r < R; r++) y[r] = 0.f;
	if (active) {
		const int nb = a.n / 256;
		for (int b = 0; b < nb; b++) {
			const int base = b * 256;
#pragma unroll
			for (int r = 0; r < R; r++) {
				const int pr = row_valid(a, row0, r, R) ? phys_row(a, row0, r, R) : phys_row(a, row0, 0, R);
				const uint8_t* blk = a.w.p0 + (size_t) pr * a.w.s0 + (size_t) b * 54;
				float s = 0.f;
				uint8_t q = blk[lane];
#pragma unroll
				for (int k = 0; k < 5; k++) {
					const int trit = ((int) q * 3) >> 8;
					s += (float) (trit - 1) * xval(base + k * 32 + lane);
					q = (uint8_t) (q * 3);
				}
				if (lane < 16) {
					q = blk[32 + lane];
#pragma unroll
					for (int k = 0; k < 5; k++) {
						const int trit = ((int) q * 3) >> 8;
						s += (float) (trit - 1) * xval(base + 160 + k * 16 + lane);
						q = (uint8_t) (q * 3);
					}
				}
				if (lane < 4) {
					q = blk[48 + lane];
#pragma unroll
					for (int k = 0; k < 4; k++) {
						const int trit = ((int) q * 3) >> 8;
						s += (float) (trit - 1) * xval(base + 240 + k * 4 + lane);
						q = (uint8_t) (q * 3);
					}
				}
				y[r] += ld_f16_unaligned(blk + 52) * s;
			}
		}
	}
#pragma unroll
	for (int r = 0; r < R; r++) y[r] = warp_sum(y[r]);
	if (active && lane == 0) epilogue<R>(a, row0, y);
}

} // namespace xalm
