// matvec_tma.cuh — the decode hot kernel, TMA edition: persistent CTAs stream weight rows HBM -> shared memory with
// cp.async.bulk (the TMA engine; no LSU / L1TEX involvement), signalled through mbarriers, and consume them with
// conflict-free 128-bit shared loads.  Same math, prologue and epilogues as matvec.cuh (which stays as the path for
// row lengths that are not a multiple of 256 and for the table-decoded formats).
//
// Why (profiles/r1_matvec_ldg_q8_0_w13.md): the LDG version is L1TEX-bound, not HBM-bound — every warp re-reads its
// activation chunk (and the norm weights) through L1 for every 4 rows, 3x the weight traffic, and tops out at ~40 % of
// HBM peak.  Here:
//   * one CTA per SM, grid-strided over row tiles; a dedicated producer warp keeps a ring of NS stages in flight
//     (>= 64 KB per SM, independent of register pressure), each stage = RC rows x U "units";
//   * activations are normalised ONCE per CTA (rmsnorm prologue) into shared memory and reused by every tile;
//   * the producer starts fetching weights BEFORE griddepcontrol.wait (PDL): the HBM stream runs through kernel
//     boundaries; only the consumers wait for the previous kernel's activations.
//
// Device layout ("unit-interleaved", built at upload, same byte count as on disk): a row is n/256 units; a unit holds
// the 256 elements' main bytes followed by their scales / high bits, so ONE bulk copy per row fetches any run of units:
//   F32 1024 | F16,BF16 512 | F8_*,Q8 256 | Q8_0 256+16 | Q4_0 128+16 | Q4_1 128+32 | Q5_0 128+16+32 | Q5_1 128+32+32
// A "piece" is 16 main bytes (E elements); lane-strided pieces make every shared load a full 512-byte wavefront set.
//
// Warp roles: warps 0..7 consume (KW K-slices x RW row groups, R = RC/RW rows per warp), warp 8 produces.
// Cross-warp (K-slice) sums go through shared memory in a fixed order -> bit-reproducible run to run.
#pragma once
#include "matvec.cuh"

namespace xalm {

// on-disk rows -> unit-interleaved rows.  One thread per (row, unit).
__global__ void repack_units_kernel(int t, const uint8_t* __restrict__ raw, size_t raw_stride, int rows, int n, uint8_t* __restrict__ dst,
                                    size_t dst_stride) {
	const int nu = n / 256;
	const int ub = unit_bytes(t);
	TypeInfo ti;
	type_info(t, &ti);
	const size_t total = (size_t) rows * nu;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const size_t r = i / nu;
		const int u = (int) (i % nu);
		uint8_t* o = dst + r * dst_stride + (size_t) u * ub;
		if (ti.block == 1) {
			const uint8_t* src = raw + r * raw_stride + (size_t) u * 256 * ti.bytes;
			for (int j = 0; j < 256 * ti.bytes; j++) o[j] = t == XALM_Q8 ? (uint8_t) (src[j] ^ 0x80) : src[j];
			continue;
		}
		const uint8_t* src = raw + r * raw_stride + (size_t) u * 8 * ti.bytes; // 8 blocks of 32 per unit
		for (int b = 0; b < 8; b++) {
			const uint8_t* s = src + (size_t) b * ti.bytes;
			switch (t) {
				case XALM_Q8_0:
					for (int j = 0; j < 32; j++) o[32 * b + j] = s[2 + j] ^ 0x80;
					o[256 + 2 * b] = s[0]; o[256 + 2 * b + 1] = s[1];
					break;
				case XALM_Q4_0:
					for (int j = 0; j < 16; j++) o[16 * b + j] = s[2 + j];
					o[128 + 2 * b] = s[0]; o[128 + 2 * b + 1] = s[1];
					break;
				case XALM_Q4_1:
					for (int j = 0; j < 16; j++) o[16 * b + j] = s[4 + j];
					for (int j = 0; j < 4; j++) o[128 + 4 * b + j] = s[j];
					break;
				case XALM_Q5_0:
					for (int j = 0; j < 16; j++) o[16 * b + j] = s[6 + j];
					o[128 + 2 * b] = s[0]; o[128 + 2 * b + 1] = s[1];
					for (int j = 0; j < 4; j++) o[144 + 4 * b + j] = s[2 + j];
					break;
				case XALM_Q5_1:
					for (int j = 0; j < 16; j++) o[16 * b + j] = s[8 + j];
					for (int j = 0; j < 4; j++) o[128 + 4 * b + j] = s[j];
					for (int j = 0; j < 4; j++) o[160 + 4 * b + j] = s[4 + j];
					break;
			}
		}
	}
}

__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// ---- per-format access to one piece of a unit held in shared memory --------------------------------------------------
template <int TYPE>
struct UFmt;
#define XALM_UFMT_PLAIN(T, PPU_)                                                                      \
	template <>                                                                                       \
	struct UFmt<T> {                                                                                  \
		static constexpr int PPU = PPU_;                                                              \
		static __device__ __forceinline__ typename Fmt<T>::Frag load(const uint8_t* unit, int p) {    \
			return {*reinterpret_cast<const uint4*>(unit + 16 * p)};                                  \
		}                                                                                             \
	};
XALM_UFMT_PLAIN(XALM_F32, 64)
XALM_UFMT_PLAIN(XALM_F16, 32)
XALM_UFMT_PLAIN(XALM_BF16, 32)
XALM_UFMT_PLAIN(XALM_F8_E4M3, 16)
XALM_UFMT_PLAIN(XALM_F8_E5M2, 16)
XALM_UFMT_PLAIN(XALM_Q8, 16)
#undef XALM_UFMT_PLAIN
template <>
struct UFmt<XALM_Q8_0> {
	static constexpr int PPU = 16;
	static __device__ __forceinline__ Fmt<XALM_Q8_0>::Frag load(const uint8_t* unit, int p) {
		return {*reinterpret_cast<const uint4*>(unit + 16 * p), *reinterpret_cast<const uint16_t*>(unit + 256 + 2 * (p >> 1))};
	}
};
template <>
struct UFmt<XALM_Q4_0> {
	static constexpr int PPU = 8;
	static __device__ __forceinline__ Fmt<XALM_Q4_0>::Frag load(const uint8_t* unit, int p) {
		return {*reinterpret_cast<const uint4*>(unit + 16 * p), *reinterpret_cast<const uint16_t*>(unit + 128 + 2 * p)};
	}
};
template <>
struct UFmt<XALM_Q4_1> {
	static constexpr int PPU = 8;
	static __device__ __forceinline__ Fmt<XALM_Q4_1>::Frag load(const uint8_t* unit, int p) {
		return {*reinterpret_cast<const uint4*>(unit + 16 * p), *reinterpret_cast<const uint32_t*>(unit + 128 + 4 * p)};
	}
};
template <>
struct UFmt<XALM_Q5_0> {
	static constexpr int PPU = 8;
	static __device__ __forceinline__ Fmt<XALM_Q5_0>::Frag load(const uint8_t* unit, int p) {
		return {*reinterpret_cast<const uint4*>(unit + 16 * p), *reinterpret_cast<const uint32_t*>(unit + 144 + 4 * p),
		        *reinterpret_cast<const uint16_t*>(unit + 128 + 2 * p)};
	}
};
template <>
struct UFmt<XALM_Q5_1> {
	static constexpr int PPU = 8;
	static __device__ __forceinline__ Fmt<XALM_Q5_1>::Frag load(const uint8_t* unit, int p) {
		return {*reinterpret_cast<const uint4*>(unit + 16 * p), *reinterpret_cast<const uint32_t*>(unit + 160 + 4 * p),
		        *reinterpret_cast<const uint32_t*>(unit + 128 + 4 * p)};
	}
};

struct TmaArgs {
	MatvecArgs a;   // a.w.p0 = unit-interleaved rows, a.w.s0 = row stride in bytes
	int U;          // units per stage
	int NS;         // ring stages
	int n_tiles;    // ceil(virtual rows / RC)
	int x_global;   // 1: activations are NOT staged in shared memory but read through L1 (long rows without norm: W2), 8-row reuse
};

constexpr int TMA_NW = 8; // consumer warps

__host__ __device__ inline size_t tma_smem_bytes(int type, int n, int RC, int U, int NS) {
	size_t s = 0;
	s += (size_t) n * sizeof(float);            // xb (pass n = 0 when activations are read from global memory)
	s += (size_t) NS * RC * U * unit_bytes(type); // ring
	s += 2 * TMA_NW * 16 * sizeof(float);       // partials, double-buffered  [2][KW<=8][RC<=16]
	s += 2 * (size_t) NS * sizeof(uint64_t);    // full / empty barriers
	s += 64 * sizeof(float);                    // reduction scratch
	return s + 128;
}

// TYPE: weight format; RC: rows per tile; KW: K-slices (RW = 8/KW row groups, R = RC/RW rows per warp); NORM: rmsnorm prologue
template <int TYPE, int RC, int KW, bool NORM>
__global__ void __launch_bounds__((TMA_NW + 1) * 32, 1) matvec_tma_kernel(const TmaArgs ta) {
	using F = Fmt<TYPE>;
	using UF = UFmt<TYPE>;
	constexpr int E = F::E;
	constexpr int PPU = UF::PPU;
	constexpr int RW = TMA_NW / KW;
	constexpr int R = RC / RW;
	static_assert(RC % RW == 0 && R >= 1, "row split");
	const MatvecArgs& a = ta.a;
	const int UB = unit_bytes(TYPE);
	const int U = ta.U, NS = ta.NS;
	const int nu = a.n / 256; // units per row
	const int stages_per_tile = (nu + U - 1) / U;
	const size_t row_stage_bytes = (size_t) U * UB;

	extern __shared__ __align__(128) uint8_t smem[];
	float* xb = reinterpret_cast<float*>(smem);
	const bool xg = !NORM && ta.x_global;
	uint8_t* ring = smem + (xg ? 0 : (((size_t) a.n * sizeof(float) + 127) / 128) * 128);
	float* part = reinterpret_cast<float*>(ring + (size_t) NS * RC * row_stage_bytes);
	uint64_t* full = reinterpret_cast<uint64_t*>(part + 2 * TMA_NW * 16);
	uint64_t* empty = full + NS;
	float* s_red = reinterpret_cast<float*>(empty + NS);

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; s++) {
			mbar_init(&full[s], 1);
			mbar_init(&empty[s], TMA_NW);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	pdl_launch_dependents();
	int tl = -1;
	if (blockIdx.x == 0 && threadIdx.x == 0) tl = tl_begin(100 + a.epi);

	const int my_tiles = ((int) blockIdx.x < ta.n_tiles) ? (ta.n_tiles - 1 - (int) blockIdx.x) / (int) gridDim.x + 1 : 0;

	if (warp == TMA_NW) {
		// ===================== producer: weights only — runs ahead of griddepcontrol.wait =====================
		if (lane == 0) {
			prefetch_next_norm(a);
			int slot = 0, phase = 0;
			for (int tt = 0; tt < my_tiles; tt++) {
				const int row0 = ((int) blockIdx.x + tt * (int) gridDim.x) * RC;
				for (int st = 0; st < stages_per_tile; st++) {
					mbar_wait(&empty[slot], phase ^ 1);
					const int u0 = st * U;
					const int un = min(U, nu - u0);
					const uint32_t bytes = (uint32_t) un * UB;
					mbar_expect_tx(&full[slot], bytes * RC);
					uint8_t* dst = ring + (size_t) slot * RC * row_stage_bytes;
#pragma unroll
					for (int r = 0; r < RC; r++) {
						const int pr = phys_row(a, row0, r, RC);
						bulk_g2s(dst + (size_t) r * row_stage_bytes, a.w.p0 + (size_t) pr * a.w.s0 + (size_t) u0 * UB, bytes, &full[slot]);
					}
					if (++slot == NS) { slot = 0; phase ^= 1; }
				}
			}
			prefetch_tail(a, true);
		}
		return;
	}

	// ===================== consumers =====================
	// the rmsnorm weights do not depend on the previous kernel: request this thread's share (up to 8 chunks = rows of 8192)
	// before the dependency wait, so the scale pass below does not sit on an L2 round trip
	constexpr int GPRE = 8;
	float4 gpre[NORM ? GPRE : 1];
	if (NORM) {
#pragma unroll
		for (int c = 0; c < GPRE; c++) {
			const int i = (int) threadIdx.x * 4 + c * TMA_NW * 32 * 4;
			if (i < a.n) {
				if (a.norm_type == XALM_F32) gpre[c] = ld_act4(reinterpret_cast<const float*>(a.norm_w) + i);
				else {
					const uint2 gv = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(a.norm_w) + i);
					gpre[c] = make_float4(__uint_as_float(gv.x << 16), __uint_as_float(gv.x & 0xFFFF0000u), __uint_as_float(gv.y << 16),
					                      __uint_as_float(gv.y & 0xFFFF0000u));
				}
			}
		}
	}
	pdl_wait(); // activations / KV ring of earlier kernels are visible from here on
	tl_mark(tl, 2);
	if (a.epi == EPI_QKV && blockIdx.x == 0 && a.step->kv_sink > 0) rotate_sinks(a, a.k_cache, a.step->kv_sink, threadIdx.x, TMA_NW * 32);
	if (NORM && a.n_recv) tp_receive(a, threadIdx.x, TMA_NW * 32);
	// ---- stage activations: xb = NORM ? x * scale * g : x ----
	if (!xg) {
		// xb is stored permuted inside each 256-element unit: the E floats a lane needs for one piece are split into
		// E/4 float4s laid out [i][piece], so the 32 lanes of a warp read consecutive float4s (no bank conflicts).
		auto xpos = [](int e) { // e % 4 == 0
			const int u = e >> 8, w = e & 255;
			const int pp = w / E, i4 = (w % E) >> 2;
			return (u << 8) + ((i4 * PPU + pp) << 2);
		};
		float ss = 0.f;
		for (int i = threadIdx.x * 4; i < a.n; i += TMA_NW * 32 * 4) {
			float4 v;
			if (NORM && a.n_recv) { // the summed stream, published by the reducing CTAs above as {value, tag} words: poll this exchange's tag
				v = poll_tagged4(a.xl + i, a.step->ar_base + (unsigned int) a.recv_idx + 1u, a.err_flag);
			} else {
				v = ld_act4(a.x + i);
			}
			*reinterpret_cast<float4*>(xb + xpos(i)) = v;
			ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
		}
		if (NORM) {
			ss = warp_sum(ss);
			if (lane == 0) s_red[warp] = ss;
			consumer_bar_sync();
			float tot = 0.f;
#pragma unroll
			for (int i = 0; i < TMA_NW; i++) tot += s_red[i];
			const float scale = 1.0f / sqrtf(tot / (float) a.n + a.norm_eps);
#pragma unroll
			for (int c = 0; c < GPRE; c++) { // same elements this thread wrote above
				const int i = (int) threadIdx.x * 4 + c * TMA_NW * 32 * 4;
				if (i < a.n) {
					float4 v = *reinterpret_cast<float4*>(xb + xpos(i));
					const float4 g = gpre[c];
					v.x = v.x * scale * g.x; v.y = v.y * scale * g.y; v.z = v.z * scale * g.z; v.w = v.w * scale * g.w; // infer.cpp:233-235
					*reinterpret_cast<float4*>(xb + xpos(i)) = v;
				}
			}
			for (int i = threadIdx.x * 4 + GPRE * TMA_NW * 32 * 4; i < a.n; i += TMA_NW * 32 * 4) { // rows longer than 8192
				float4 v = *reinterpret_cast<float4*>(xb + xpos(i));
				float4 g;
				if (a.norm_type == XALM_F32) g = ld_act4(reinterpret_cast<const float*>(a.norm_w) + i);
				else {
					const uint2 gv = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(a.norm_w) + i);
					g = make_float4(__uint_as_float(gv.x << 16), __uint_as_float(gv.x & 0xFFFF0000u), __uint_as_float(gv.y << 16),
					                __uint_as_float(gv.y & 0xFFFF0000u));
				}
				v.x = v.x * scale * g.x; v.y = v.y * scale * g.y; v.z = v.z * scale * g.z; v.w = v.w * scale * g.w; // infer.cpp:233-235
				*reinterpret_cast<float4*>(xb + xpos(i)) = v;
			}
		}
		consumer_bar_sync();
	}

	const int kw = warp % KW, rw = warp / KW;
	int slot = 0, phase = 0;
	for (int tt = 0; tt < my_tiles; tt++) {
		f32x2 acc[R];
#pragma unroll
		for (int r = 0; r < R; r++) acc[r] = pack2(0.f, 0.f);
		// residual: the reducer warp fetches the old activation now, so its epilogue does not sit on an L2 round trip
		float xold = 0.f;
		if (a.epi == EPI_RESIDUAL && warp == (tt % TMA_NW) && lane < RC) {
			const int row = ((int) blockIdx.x + tt * (int) gridDim.x) * RC + lane;
			if (row < a.d) xold = a.out[row];
		}
		for (int st = 0; st < stages_per_tile; st++) {
			const int u0 = st * U;
			const int un = min(U, nu - u0);
			const int pieces = un * PPU;                 // pieces per row in this stage
			const int per = (pieces + KW - 1) / KW;      // this warp's K-slice [kw*per, ...)
			const int pend = min(pieces, (kw + 1) * per);
			mbar_wait(&full[slot], phase);
			const uint8_t* rows = ring + (size_t) slot * RC * row_stage_bytes + (size_t) (rw * R) * row_stage_bytes;
			for (int p = kw * per + lane; p < pend; p += 32) {
				const int u = p / PPU, pp = p % PPU;
				float xv[E];
				if (xg) { // natural order, straight from global memory through L1 (coherent at a kernel boundary)
					const float* xs = a.x + (size_t) (u0 + u) * 256 + pp * E;
#pragma unroll
					for (int i = 0; i < E; i += 4) {
						const float4 v = ld_act4(xs + i);
						xv[i] = v.x; xv[i + 1] = v.y; xv[i + 2] = v.z; xv[i + 3] = v.w;
					}
				} else {
					const float* xs = xb + (size_t) (u0 + u) * 256 + pp * 4;
#pragma unroll
					for (int i = 0; i < E; i += 4) {
						const float4 v = *reinterpret_cast<const float4*>(xs + i * PPU);
						xv[i] = v.x; xv[i + 1] = v.y; xv[i + 2] = v.z; xv[i + 3] = v.w;
					}
				}
#pragma unroll
				for (int r = 0; r < R; r++) {
					const typename F::Frag f = UF::load(rows + (size_t) r * row_stage_bytes + (size_t) u * UB, pp);
					F::fma_chunk(f, xv, acc[r]);
				}
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&empty[slot]);
			if (++slot == NS) { slot = 0; phase ^= 1; }
		}
		// ---- combine the KW K-slices (fixed order) and run the epilogue; barrier deferred behind the next tile's work ----
		float* pt = part + (tt & 1) * (TMA_NW * 16);
#pragma unroll
		for (int r = 0; r < R; r++) {
			float lo, hi;
			unpack2(acc[r], lo, hi);
			const float y = warp_sum(lo + hi);
			if (lane == 0) pt[kw * 16 + rw * R + r] = y;
		}
		consumer_bar_sync();
		if (warp == (tt % TMA_NW)) { // rotating reducer
			float yv = 0.f;
			if (lane < RC) {
#pragma unroll
				for (int k = 0; k < KW; k++) yv += pt[k * 16 + lane];
			}
			row_epilogue<RC>(a, ((int) blockIdx.x + tt * (int) gridDim.x) * RC, lane, yv, xold);
		}
	}
	tl_mark(tl, 3);
}

} // namespace xalm
