// matvec_mma.cuh — the decode matvec for the integer weight formats on the TENSOR cores' integer path
// (mma.sync.m16n8k32.s32.u8.u8), weights in fragment tiles (frag_layout.cuh).
//
// Why.  The dp4a core (matvec_idp.cuh) spends 24 IDP.4A plus ~30 unpack / convert / scale instructions per 32-weight block and
// lane: 0.112 (q8_0) - 0.124 (q4_0) warp instructions per weight.  ncu (profiles/r2_ncu_q4_0_w13_details.txt): q4_0 W1|W3 runs at
// 30 % of DRAM peak with the issue slots 52 % busy and 0.9 eligible warps per scheduler — the consumers, not HBM, set the pace,
// and q4_0 decodes no faster than q8_0 although it streams half the bytes.  Here ONE mma handles a 16-row x 32-element block
// column (512 weights) against the three activation limbs at once, and the per-block float work is 2 IMAD + 2 I2F + 2 FFMA:
// ~0.04 warp instructions per weight.
//
// Arithmetic (exact in integers, like idp.cuh).  Activations are staged once per CTA as block floating point, x_k ~= dx * X_k
// with |X_k| < 2^23 and one power-of-two dx per 32 elements, but in OFFSET form X'_k = X_k + 2^23 (three unsigned byte limbs
// l0' l1' l2'), because the mma has one signedness per operand.  The B operand (32 k x 8 columns) holds
//     column 0: l2'   column 1: l1'   column 2: l0'   column 3: ones   columns 4-7: zero
// and the stored weight bytes u_k = q_k + BIAS are the A operand.  With the accumulators initialised to
//     c(l2') = -BIAS S2',  c(l1') = -BIAS S1',  c(l0') = -BIAS (S0' - 4096),  c(ones) = 0       (S' = limb sums of the block)
// the lane that holds columns (0, 1) forms v = 256 c1 + c0, the lane that holds (2, 3) forms v = c0 - 128 c1 (this removes the
// 2^23 offset: 2^23 = 128 * 65536), and  sum_k (u_k - BIAS) X_k = 65536 v(2,3) + v(0,1)  exactly.  Each lane accumulates
// float(v) * (d * dx [* 65536]) in fp32; lanes are added at the end of a tile.  With a one-hot x everything is exact and the
// kernel returns the dequantised weight bit for bit (d*q exact, d*q+m rounds once).
//
// Skeleton: as matvec_idp.cuh — persistent CTAs (one per SM), a producer warp streaming records into an mbarrier ring with ONE
// cp.async.bulk per stage (a tile's records are contiguous), 16 consumer warps, rmsnorm prologue (1/rms applied to the row
// sums), QKV / GLU / residual / store epilogues, PDL, the fused tensor-parallel exchange.
#pragma once
#include "frag_layout.cuh"
#include "idp.cuh"
#include "matvec_tma.cuh"

namespace xalm {

constexpr int MMA_RC = 16;  // rows per tile
constexpr int MMA_SB = 64;  // records (32-element block columns) per ring stage
constexpr int MMA_NCW = 16; // consumer warps
constexpr int MMA_NT = MMA_NCW * 32;
constexpr int MMA_MP = 2;   // activation groups a lane keeps in flight (8 elements each): one pass for n <= 8192

// ---- activation image in shared memory: 3 limb planes (stride n + 16 bytes: the three planes a quarter-warp reads fall into
//      different banks) + one 64-byte table entry per block, 16 bytes per lane position: {c-init (l2'), c-init (l1'), dx, sum x} {c-init (l0'), 0, dx * 65536, 0} {0} {0}
struct XmView {
	uint8_t* q;
	int4* tbl;
	int ps; // plane stride
};
__host__ __device__ inline size_t xm_bytes(int n) { return ((size_t) 3 * (n + 16) + (size_t) (n / 32) * 64 + 127) / 128 * 128; }
__device__ __forceinline__ XmView xm_view(uint8_t* base, int n) { return {base, reinterpret_cast<int4*>(base + (size_t) 3 * (n + 16)), n + 16}; }

// one group of eight elements quantised: the three limb words of each half, the block's limb sums (s0 = low limb, u = mid | high
// << 16, summed over the four lanes of the block) and the block exponent dx
struct XmGroup {
	uint32_t w[3][2];
	uint32_t s0, u;
	float dx;
};

// eight consecutive elements per lane, the four lanes 4k .. 4k+3 of a warp share a block (call with all lanes of the warp)
__device__ __forceinline__ void xm_quant_group8(const float (&x)[8], XmGroup& o) {
	uint32_t mb = 0;
#pragma unroll
	for (int e = 0; e < 8; e++) mb = max(mb, __float_as_uint(x[e]) & 0x7fffffffu);
	mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 1));
	mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 2));
	const int eb = (int) (mb >> 23);
	const bool live = eb >= 40 && eb < 255; // as idp.cuh: blocks below 2^-87 contribute nothing, non-finite blocks are dropped
	const float sc = live ? __uint_as_float((uint32_t) (276 - eb) << 23) : 0.f;
	const float dx = live ? __uint_as_float((uint32_t) (eb - 22) << 23) : 0.f;
	uint32_t s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
	for (int q = 0; q < 2; q++) {
		int X[4];
#pragma unroll
		for (int e = 0; e < 4; e++) X[e] = min(__float2int_rn(x[4 * q + e] * sc), 8388607) + 8388608; // offset form: 0 .. 2^24 - 1
#pragma unroll
		for (int k = 0; k < 3; k++) {
			const uint32_t sel = (uint32_t) k | ((uint32_t) (4 + k) << 4);
			const uint32_t lo = prmt((uint32_t) X[0], (uint32_t) X[1], sel), hi = prmt((uint32_t) X[2], (uint32_t) X[3], sel);
			o.w[2 - k][q] = prmt(lo, hi, 0x5410u);
		}
		asm("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(s0) : "r"(o.w[0][q]), "r"(0x01010101u));
		asm("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(s1) : "r"(o.w[1][q]), "r"(0x01010101u));
		asm("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(s2) : "r"(o.w[2][q]), "r"(0x01010101u));
	}
	uint32_t u = s1 | (s2 << 16); // block totals <= 32 * 255 < 2^16
	u += __shfl_xor_sync(0xffffffffu, u, 1);
	u += __shfl_xor_sync(0xffffffffu, u, 2);
	s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
	s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
	o.s0 = s0;
	o.u = u;
	o.dx = dx;
}

// (lanes past the end of the vector pass valid = false and take part in the shuffles only)
template <int BIAS>
__device__ __forceinline__ void xm_store_group8(const XmView& v, int grp, const float (&x)[8], bool valid = true) {
	XmGroup o;
	xm_quant_group8(x, o);
	if (!valid) return;
	const uint32_t(&w)[3][2] = o.w;
	const uint32_t s0 = o.s0, u = o.u;
	const float dx = o.dx;
#pragma unroll
	for (int k = 0; k < 3; k++) *reinterpret_cast<uint2*>(v.q + (size_t) k * v.ps + (size_t) grp * 8) = make_uint2(w[k][0], w[k][1]);
	if ((grp & 3) == 0) {
		const int S0 = (int) s0, S1 = (int) (u & 0xFFFFu), S2 = (int) (u >> 16);
		const int tot = (S0 - 4096) * 65536 + S1 * 256 + S2; // sum of the block's X (the offsets removed)
		const float sx = __int2float_rn(tot) * dx;
		int4* e = v.tbl + 4 * (grp >> 2); // one entry per lane position tig (columns 2 tig, 2 tig + 1); positions 2, 3 hold the zero columns
		e[0] = make_int4(-BIAS * S2, -BIAS * S1, (int) __float_as_uint(dx), (int) __float_as_uint(sx));
		e[1] = make_int4(-BIAS * (S0 - 4096), 0, (int) __float_as_uint(dx * 65536.f), 0);
		e[2] = make_int4(0, 0, 0, 0);
		e[3] = make_int4(0, 0, 0, 0);
	}
}

// d = a * b + c with separate accumulator-in registers: the c-init values are used as they come from the table, no copies
__device__ __forceinline__ void mma_u8(int (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, int c0, int c1) {
	asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%10,%11};"
	             : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
	             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "r"(c0), "r"(c1));
}

// ---- weight side: the A fragment and the scales of one record -------------------------------------------------------------
template <int TYPE>
struct MmaFmt;
template <>
struct MmaFmt<XALM_Q8_0> {
	static constexpr int RB = 544, BIAS = 128;
	static constexpr bool HAS_MIN = false;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int g, uint32_t (&a)[4], float& d0, float& d1, float&, float&) {
		const uint4 q = *reinterpret_cast<const uint4*>(rec + lane * 16);
		a[0] = q.x; a[1] = q.y; a[2] = q.z; a[3] = q.w;
		const float2 d = __half22float2(*reinterpret_cast<const __half2*>(rec + 512 + g * 4));
		d0 = d.x; d1 = d.y;
	}
};
template <>
struct MmaFmt<XALM_Q8> {
	static constexpr int RB = 512, BIAS = 128;
	static constexpr bool HAS_MIN = false;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int, uint32_t (&a)[4], float& d0, float& d1, float&, float&) {
		const uint4 q = *reinterpret_cast<const uint4*>(rec + lane * 16);
		a[0] = q.x; a[1] = q.y; a[2] = q.z; a[3] = q.w;
		d0 = d1 = 1.f / 100.f; // types.h:423-424
	}
};
__device__ __forceinline__ void mma_nibbles(const uint8_t* rec, int lane, uint32_t (&a)[4]) {
	const uint2 q = *reinterpret_cast<const uint2*>(rec + lane * 8);
	a[0] = q.x & 0x0F0F0F0Fu; a[1] = (q.x >> 4) & 0x0F0F0F0Fu;
	a[2] = q.y & 0x0F0F0F0Fu; a[3] = (q.y >> 4) & 0x0F0F0F0Fu;
}
// fifth bits: bit 4j + e of the lane's half-word -> bit 4 of byte e of a[j]  (x * 0x00204081 moves bit i to bits i, i+7, i+14, i+21)
__device__ __forceinline__ void mma_fifth_bits(const uint8_t* rec, int lane, uint32_t (&a)[4]) {
	const uint32_t hb = *reinterpret_cast<const uint16_t*>(rec + 256 + lane * 2);
#pragma unroll
	for (int j = 0; j < 4; j++) a[j] |= ((((hb >> (4 * j)) & 0xFu) * 0x00204081u) & 0x01010101u) << 4;
}
template <>
struct MmaFmt<XALM_Q4_0> { // d * (q - 8)
	static constexpr int RB = 288, BIAS = 8;
	static constexpr bool HAS_MIN = false;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int g, uint32_t (&a)[4], float& d0, float& d1, float&, float&) {
		mma_nibbles(rec, lane, a);
		const float2 d = __half22float2(*reinterpret_cast<const __half2*>(rec + 256 + g * 4));
		d0 = d.x; d1 = d.y;
	}
};
template <>
struct MmaFmt<XALM_Q4_1> { // d * q + m
	static constexpr int RB = 320, BIAS = 0;
	static constexpr bool HAS_MIN = true;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int g, uint32_t (&a)[4], float& d0, float& d1, float& m0, float& m1) {
		mma_nibbles(rec, lane, a);
		const uint2 s = *reinterpret_cast<const uint2*>(rec + 256 + g * 8);
		const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&s.x)), m = __half22float2(*reinterpret_cast<const __half2*>(&s.y));
		d0 = d.x; d1 = d.y; m0 = m.x; m1 = m.y;
	}
};
template <>
struct MmaFmt<XALM_Q5_0> { // d * ((ql | qh << 4) - 16)
	static constexpr int RB = 352, BIAS = 16;
	static constexpr bool HAS_MIN = false;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int g, uint32_t (&a)[4], float& d0, float& d1, float&, float&) {
		mma_nibbles(rec, lane, a);
		mma_fifth_bits(rec, lane, a);
		const float2 d = __half22float2(*reinterpret_cast<const __half2*>(rec + 320 + g * 4));
		d0 = d.x; d1 = d.y;
	}
};
template <>
struct MmaFmt<XALM_Q5_1> { // d * (ql | qh << 4) + m
	static constexpr int RB = 384, BIAS = 0;
	static constexpr bool HAS_MIN = true;
	static __device__ __forceinline__ void load(const uint8_t* rec, int lane, int g, uint32_t (&a)[4], float& d0, float& d1, float& m0, float& m1) {
		mma_nibbles(rec, lane, a);
		mma_fifth_bits(rec, lane, a);
		const uint2 s = *reinterpret_cast<const uint2*>(rec + 320 + g * 8);
		const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&s.x)), m = __half22float2(*reinterpret_cast<const __half2*>(&s.y));
		d0 = d.x; d1 = d.y; m0 = m.x; m1 = m.y;
	}
};

__host__ __device__ inline bool mma_supported(int t) { return frag_record_bytes(t) != 0; }
__host__ __device__ inline int mma_pb(int NS) { return NS + 2 < 8 ? 8 : NS + 2; } // partial-sum buffers (tiles in flight), as idp_pb

__host__ __device__ inline size_t mma_smem_bytes(int type, int n, int NS) {
	size_t s = xm_bytes(n);
	s += (size_t) NS * MMA_SB * frag_record_bytes(type);
	s += (size_t) mma_pb(NS) * MMA_NCW * MMA_RC * sizeof(float);
	s += (2 * (size_t) NS + 2 * mma_pb(NS)) * sizeof(uint64_t);
	s += MMA_NCW * sizeof(float);
	return s + 128;
}

struct MmaArgs {
	MatvecArgs a; // a.w.p0 = fragment tiles, a.w.s0 = bytes of one tile
	int NS;       // ring stages
	int n_tiles;  // virtual rows / 16
};

template <int TYPE, bool NORM>
__global__ void __launch_bounds__((MMA_NCW + 2) * 32, 1) matvec_mma_kernel(const MmaArgs ta) {
	using F = MmaFmt<TYPE>;
	constexpr int RC = MMA_RC, SB = MMA_SB, NCW = MMA_NCW, NT = MMA_NT, RB = F::RB, MP = MMA_MP;
	constexpr int STAGE = SB * RB;
	auto cbar = [] { asm volatile("bar.sync 1, 512;" ::: "memory"); };
	const MatvecArgs& a = ta.a;
	const int NS = ta.NS, PB = mma_pb(ta.NS);
	const int n = a.n, nb = n / 32;
	const int kranges = (nb + SB - 1) / SB; // stages per tile

	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* ring = smem + xm_bytes(n);
	float* part = reinterpret_cast<float*>(ring + (size_t) NS * STAGE);
	float* s_red = part + PB * NCW * RC;
	uint64_t* full = reinterpret_cast<uint64_t*>(s_red + NCW);
	uint64_t* empty = full + NS;
	uint64_t* pbar = empty + NS;
	uint64_t* pfree = pbar + PB; // a partial-sum buffer has been read by the epilogue warp

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; s++) {
			mbar_init(&full[s], 1);
			mbar_init(&empty[s], NCW);
		}
		for (int s = 0; s < PB; s++) {
			mbar_init(&pbar[s], NCW);
			mbar_init(&pfree[s], 1);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	pdl_launch_dependents();
	int tl = -1;
	if (blockIdx.x == 0 && threadIdx.x == 0) tl = tl_begin(100 + a.epi);

	const int my_tiles = ((int) blockIdx.x < ta.n_tiles) ? (ta.n_tiles - 1 - (int) blockIdx.x) / (int) gridDim.x + 1 : 0;

	if (warp == NCW) {
		// ===================== producer: weights only — runs ahead of griddepcontrol.wait =====================
		if (lane == 0) {
			prefetch_next_norm(a);
			int slot = 0, phase = 0;
			for (int tt = 0; tt < my_tiles; tt++) {
				const uint8_t* tile = a.w.p0 + (size_t) ((int) blockIdx.x + tt * (int) gridDim.x) * a.w.s0;
				for (int kr = 0; kr < kranges; kr++) {
					mbar_wait(&empty[slot], phase ^ 1);
					const uint32_t bytes = (uint32_t) min(SB, nb - kr * SB) * RB;
					mbar_expect_tx(&full[slot], bytes);
					bulk_g2s(ring + (size_t) slot * STAGE, tile + (size_t) kr * STAGE, bytes, &full[slot]); // a tile's records are contiguous
					if (++slot == NS) { slot = 0; phase ^= 1; }
				}
			}
			prefetch_tail(a, true);
		}
		return;
	}

	if (warp == NCW + 1) {
		// ===================== epilogue warp: K-slice sums -> rows -> epilogue.  The 16 multiplying warps never wait for each other's
		// partial sums (with a rotating reducer among them, a third of all warp samples sat in that wait: profiles/r2_mma.md) ==========
		pdl_wait();
		float nscale = 1.f;
		int pb = 0, pph = 0;
		for (int tt = 0; tt < my_tiles; tt++) {
			const int row0 = ((int) blockIdx.x + tt * (int) gridDim.x) * RC;
			float xold = 0.f; // residual: fetch the old activation before the wait, so the epilogue does not sit on an L2 round trip
			if (a.epi == EPI_RESIDUAL && lane < RC && row0 + lane < a.d) xold = a.out[row0 + lane];
			mbar_wait(&pbar[pb], pph);
			if (NORM && tt == 0) { // the sums of squares were complete before any warp multiplied a tile
				float tot = 0.f;
#pragma unroll
				for (int i = 0; i < NCW; i++) tot += s_red[i];
				nscale = 1.0f / sqrtf(tot / (float) n + a.norm_eps); // infer.cpp:229-232
			}
			float yv = 0.f;
			if (lane < RC) {
				const float* pt = part + pb * NCW * RC;
#pragma unroll
				for (int w = 0; w < NCW; w++) yv += pt[w * RC + lane];
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&pfree[pb]);
			if (++pb == PB) { pb = 0; pph ^= 1; }
			if (NORM) yv *= nscale;
			const float ynext = __shfl_down_sync(0xffffffffu, yv, 1);
			if (a.epi == EPI_RESIDUAL) {
				if (lane < RC && row0 + lane < a.d) a.out[row0 + lane] = xold + yv;
			} else if (a.epi == EPI_STORE && a.n_push) { // tensor parallel: this rank's partial rows go to every rank (NVLink stores)
				if (lane < RC && (lane & 1) == 0 && row0 + lane < a.d) {
					const unsigned int seq = a.step->ar_base + (unsigned int) a.push_idx + 1u;
					const uint4 w = make_uint4(__float_as_uint(yv), seq, __float_as_uint(ynext), seq);
					for (int p = 0; p < a.n_push; p++) *reinterpret_cast<uint4*>(a.push_dst[p] + row0 + lane) = w;
				}
			} else if (lane < RC && (lane & 1) == 0 && a.epi != EPI_GLU) { // GLU below (partner rows RC/2 apart)
				const float y2[2] = {yv, ynext};
				epilogue<2>(a, row0 + lane, y2);
			}
			if (a.epi == EPI_GLU) {
				const float ypart = __shfl_down_sync(0xffffffffu, yv, RC / 2); // W3 value for the W1 row in this lane
				if (lane < RC / 2) {
					const int o = row0 / 2 + lane;
					if (o < a.d) {
						const float gt = a.act == XALM_SILU ? act_silu(yv) : act_gelu(yv);
						a.out[o] = gt * ypart;
					}
				}
			}
		}
		return;
	}

	// ===================== consumers =====================
	const int tid = threadIdx.x;
	const int ngrp = n / 8;
	// the rmsnorm weights of the first pass do not depend on the previous kernel: request them before the dependency wait
	uint4 gw[NORM ? MP : 1][2];
	auto load_gw = [&](int grp, uint4 (&o)[2]) {
		if (a.norm_type == XALM_F32) {
			o[0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(a.norm_w) + grp * 8);
			o[1] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(a.norm_w) + grp * 8 + 4);
		} else {
			o[0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(a.norm_w) + grp * 8);
		}
	};
	if (NORM) {
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = p * NT + tid;
			if (grp < ngrp) load_gw(grp, gw[p]);
		}
	}
	pdl_wait(); // activations / KV ring of earlier kernels are visible from here on
	tl_mark(tl, 2);
	if (a.epi == EPI_QKV && blockIdx.x == 0 && a.step->kv_sink > 0) { // re-rotate the attention sinks (infer.cpp:393-399)
		const int pairs = a.kv_dim / 2;
		for (int i = threadIdx.x; i < a.step->kv_sink * pairs; i += NT) {
			const int r = i / pairs, p = i % pairs;
			__half2* kp = reinterpret_cast<__half2*>(a.k_cache + (size_t) r * a.kv_dim) + p;
			float2 v = __half22float2(*kp);
			rope_pair(v.x, v.y, (2 * p) % a.head_dim, 1, a.rope_freq);
			*kp = __floats2half2_rn(v.x, v.y);
		}
	}
	// ---- tensor-parallel receive (LL style), as in matvec_tma_kernel: the first CTAs each reduce a slice of the stream and publish
	//      it locally as {value, tag} words ----
	if (NORM && a.n_recv) {
		const int n_red = min((int) gridDim.x, 8);
		if ((int) blockIdx.x < n_red) {
			const unsigned int seq = a.step->ar_base + (unsigned int) a.recv_idx + 1u;
			const int chunk = ((n / 4 + n_red - 1) / n_red) * 4;
			const int i0 = (int) blockIdx.x * chunk, i1 = min(n, i0 + chunk);
			for (int i = i0 + (int) threadIdx.x * 4; i < i1; i += NT * 4) {
				float4 v = ld_act4(a.x + i);
				float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
				for (int p = 0; p < a.n_recv; p++) {
					const uint2* src = a.recv + (size_t) p * n + i; // four {value, tag} words; poll until all carry this exchange's tag
					uint4 w0, w1;
					unsigned int spins = 0;
					do {
						asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w0.x), "=r"(w0.y), "=r"(w0.z), "=r"(w0.w) : "l"(src));
						asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w1.x), "=r"(w1.y), "=r"(w1.z), "=r"(w1.w) : "l"(src + 2));
						if (++spins > XALM_SPIN_LIMIT) { if (a.err_flag) *a.err_flag = 1u; break; } // a peer died: report, do not hang the GPU
					} while (w0.y != seq || w0.w != seq || w1.y != seq || w1.w != seq);
					sum.x += __uint_as_float(w0.x); sum.y += __uint_as_float(w0.z); sum.z += __uint_as_float(w1.x); sum.w += __uint_as_float(w1.z);
				}
				v.x += sum.x; v.y += sum.y; v.z += sum.z; v.w += sum.w;
				*reinterpret_cast<float4*>(a.x_out + i) = v;
				*reinterpret_cast<uint4*>(a.xl + i) = make_uint4(__float_as_uint(v.x), seq, __float_as_uint(v.y), seq);
				*reinterpret_cast<uint4*>(a.xl + i + 2) = make_uint4(__float_as_uint(v.z), seq, __float_as_uint(v.w), seq);
			}
		}
	}
	// ---- stage activations: quantise(NORM ? x * g : x); the scalar 1/rms is applied to the row sums (y = scale * sum w (x g)) ----
	//      xq_batch_kernel repeats this loop (thread -> group map, norm-weight decode, sum-of-squares order) and the epilogue warp's
	//      1/rms expression: batched decode is bit-identical to this kernel only while the two stay the same ----
	const XmView xv = xm_view(smem, n);
	float ss = 0.f;
	{
		auto load_group = [&](int grp, float (&v)[8]) {
			if (NORM && a.n_recv) { // the summed stream, published by the reducing CTAs as {value, tag} words: poll this exchange's tag
				const unsigned int seq = a.step->ar_base + (unsigned int) a.recv_idx + 1u;
#pragma unroll
				for (int c = 0; c < 2; c++) {
					const uint2* src = a.xl + grp * 8 + 4 * c;
					uint4 w0, w1;
					unsigned int spins = 0;
					do {
						asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w0.x), "=r"(w0.y), "=r"(w0.z), "=r"(w0.w) : "l"(src));
						asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w1.x), "=r"(w1.y), "=r"(w1.z), "=r"(w1.w) : "l"(src + 2));
						if (++spins > XALM_SPIN_LIMIT) { if (a.err_flag) *a.err_flag = 1u; break; }
					} while (w0.y != seq || w0.w != seq || w1.y != seq || w1.w != seq);
					v[4 * c] = __uint_as_float(w0.x); v[4 * c + 1] = __uint_as_float(w0.z); v[4 * c + 2] = __uint_as_float(w1.x); v[4 * c + 3] = __uint_as_float(w1.z);
				}
			} else {
				const float4 q0 = ld_act4(a.x + grp * 8), q1 = ld_act4(a.x + grp * 8 + 4);
				v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w;
				v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
			}
		};
		for (int base = 0; base < ngrp; base += MP * NT) {
			float xr[MP][8];
#pragma unroll
			for (int p = 0; p < MP; p++) {
				const int grp = base + p * NT + tid;
				if (grp < ngrp) {
					load_group(grp, xr[p]);
					if (NORM && base > 0) load_gw(grp, gw[p]);
				} else {
#pragma unroll
					for (int e = 0; e < 8; e++) xr[p][e] = 0.f;
				}
			}
#pragma unroll
			for (int p = 0; p < MP; p++) {
				const int grp = base + p * NT + tid;
				if (base + p * NT + warp * 32 < ngrp) { // warp-uniform: the quantiser shuffles within quads of lanes
					const bool valid = grp < ngrp;
					if (NORM && valid) {
#pragma unroll
						for (int e = 0; e < 8; e++) {
							ss += xr[p][e] * xr[p][e];
							float g;
							if (a.norm_type == XALM_F32) {
								const uint4 q = gw[p][e >> 2];
								g = __uint_as_float((e & 3) == 0 ? q.x : (e & 3) == 1 ? q.y : (e & 3) == 2 ? q.z : q.w);
							} else {
								const uint4 q = gw[p][0];
								const int h = e >> 1;
								const uint32_t u = h == 0 ? q.x : h == 1 ? q.y : h == 2 ? q.z : q.w;
								g = __uint_as_float((e & 1) ? (u & 0xFFFF0000u) : (u << 16));
							}
							xr[p][e] = xr[p][e] * g; // infer.cpp:233-235 without the scalar
						}
					}
					xm_store_group8<F::BIAS>(xv, grp, xr[p], valid);
				}
			}
		}
		if (NORM) {
			ss = warp_sum(ss);
			if (lane == 0) s_red[warp] = ss;
		}
		cbar();
	}
	if (tl >= 0) tl_begin(500 + a.epi); // timeline event: activations staged

	// this lane's place in the mma fragments
	const int g = lane >> 2, tig = lane & 3;
	const int vmul = tig == 0 ? 256 : tig == 1 ? -128 : 0; // v = c_odd * vmul + c_even
	const uint8_t* bp = xv.q + (size_t) (g == 0 ? 2 : g == 1 ? 1 : 0) * xv.ps + tig * 4; // B column g: l2', l1', l0' (then ones, zeros)
	const uint32_t bdef = g == 3 ? 0x01010101u : 0u;
	const int4* tp = xv.tbl + tig;

	int slot = 0, phase = 0;
	int pb_next = 0, pph_next = 0;
	for (int tt = 0; tt < my_tiles; tt++) {
		const int pb = pb_next, pph = pph_next;
		if (++pb_next == PB) { pb_next = 0; pph_next ^= 1; }
		float y0 = 0.f, y1 = 0.f; // rows g and g + 8 of the tile, this lane's columns
		for (int kr = 0; kr < kranges; kr++) {
			const int b0 = kr * SB;
			const int nbs = min(SB, nb - b0);
			const uint8_t* st = ring + (size_t) slot * STAGE;
			mbar_wait(&full[slot], phase);
			// one record (16 rows x 32 elements): rec = its bytes, bq = this lane's limb bytes of the block, tq = its table entry
			auto record = [&](const uint8_t* rec, const uint8_t* bq, const int4* tq) {
				uint32_t A[4];
				float d0, d1, m0 = 0.f, m1 = 0.f;
				F::load(rec, lane, g, A, d0, d1, m0, m1);
				uint32_t B0 = bdef, B1 = bdef;
				if (lane < 12) {
					B0 = *reinterpret_cast<const uint32_t*>(bq);
					B1 = *reinterpret_cast<const uint32_t*>(bq + 16);
				}
				const int4 tb = *tq;
				int c[4];
				mma_u8(c, A, B0, B1, tb.x, tb.y);
				const int v0 = c[1] * vmul + c[0], v1 = c[3] * vmul + c[2];
				const float dxl = __int_as_float(tb.z);
				y0 = fmaf(__int2float_rn(v0), d0 * dxl, y0);
				y1 = fmaf(__int2float_rn(v1), d1 * dxl, y1);
				if (F::HAS_MIN) {
					const float sxl = __int_as_float(tb.w);
					y0 = fmaf(m0, sxl, y0);
					y1 = fmaf(m1, sxl, y1);
				}
			};
			if (nbs == SB) { // a full stage: this warp's four records sit at fixed offsets (every address = base + immediate)
				const uint8_t* rec = st + (size_t) warp * RB;
				const uint8_t* bq = bp + (size_t) (b0 + warp) * 32;
				const int4* tq = tp + 4 * (b0 + warp);
#pragma unroll
				for (int i = 0; i < SB / NCW; i++) record(rec + (size_t) i * NCW * RB, bq + (size_t) i * NCW * 32, tq + i * NCW * 4);
			} else {
				for (int j = warp; j < nbs; j += NCW) record(st + (size_t) j * RB, bp + (size_t) (b0 + j) * 32, tp + 4 * (b0 + j));
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&empty[slot]);
			if (++slot == NS) { slot = 0; phase ^= 1; }
		}
		if (tl >= 0 && tt < 4) tl_begin(510 + 10 * tt + a.epi); // timeline event: tile tt multiplied
		// ---- the four lanes of a quad -> one sum per row, warps -> shared memory (fixed order: bit-reproducible run to run) ----
		y0 += __shfl_xor_sync(0xffffffffu, y0, 1);
		y1 += __shfl_xor_sync(0xffffffffu, y1, 1);
		y0 += __shfl_xor_sync(0xffffffffu, y0, 2);
		y1 += __shfl_xor_sync(0xffffffffu, y1, 2);
		if (tt >= PB) mbar_wait(&pfree[pb], pph ^ 1); // the epilogue warp has read what this buffer held PB tiles ago
		if (tig == 0) {
			float* pt = part + (pb * NCW + warp) * RC;
			pt[g] = y0;
			pt[g + 8] = y1;
		}
		__syncwarp();
		if (lane == 0) mbar_arrive(&pbar[pb]); // (release: this warp's partial sums are visible to whoever completes the wait)
	}
	tl_mark(tl, 3);
}

// =============================================================================================================================
// Batched decode: up to 8 independent sequences per pass over the weights.
//
// Column packing.  The B operand has 8 columns and one sequence needs 4 (three limbs and the ones column), so a PAIR of sequences
// shares one mma: sequence 2p in columns 0-3, sequence 2p+1 in columns 4-7.  The lanes with tig 0, 1 then accumulate sequence 2p
// and the lanes with tig 2, 3 sequence 2p+1, each exactly as tig 0, 1 do in matvec_mma_kernel (same records in the same per-lane
// order, same c-init values, same float operations).  The quad reduction adds the two lanes of a sequence (xor 1) and then +0,
// which is what the batch-1 kernel's second shuffle adds from its zero columns; the epilogue warp adds the 16 warps' partial
// sums in the same order.  So each sequence's outputs are bit-identical to the batch-1 kernel's, whatever shares the step.
//
// Activation staging.  One CTA cannot hold eight staged copies of a 14336-element row (5 bytes per element each).  Instead
// xq_batch_kernel quantises every sequence ONCE per matvec into an image in global memory (it stays in L2), laid out by block and
// pair: MMB_PAIR bytes per (32-element block, pair) = the three limb planes of each of the two sequences (32 bytes each) and the
// four 16-byte table entries of the pair's lanes tig 0-3.  The producer bulk-copies a stage's slice of the image into the ring
// next to the stage's weight records, so shared memory no longer grows with n.  The same kernel computes each sequence's 1/rms
// with the batch-1 kernel's reduction order (512 threads, the same thread -> group map, warp shuffles, 16 warp sums in order).
// =============================================================================================================================
constexpr int MMB_PAIR = 256; // image bytes per (block, pair)
constexpr int MMB_SB = 32;    // records per ring stage (any multiple of MMA_NCW keeps each lane's record order)
constexpr int MMB_MAX_SEQS = 8;

struct XqArgs {
	const float* x;         // (nseq, x_stride) activations
	int x_stride, n, nseq, np; // np = pairs in the image
	const uint8_t* norm_w;  // nullptr = no norm
	int norm_type;
	float norm_eps;
	uint8_t* img;           // (n / 32, np, MMB_PAIR)
	float* nscale;          // (nseq,) 1/rms per sequence (norm only)
};

// One CTA of MMA_NT threads per sequence.  The staging loop below (thread -> group map, norm-weight decode, the order of the sum of
// squares) and the 1/rms expression are those of matvec_mma_kernel's staging and epilogue warp: each sequence's image and 1/rms
// are then bit-identical to what the batch-1 kernel stages.  Edit both together.
template <int BIAS, bool NORM>
__global__ void __launch_bounds__(MMA_NT) xq_batch_kernel(const XqArgs q) {
	constexpr int NT = MMA_NT, MP = MMA_MP;
	__shared__ float s_red[MMA_NCW];
	pdl_launch_dependents();
	pdl_wait();
	const int s = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int n = q.n, ngrp = n / 8;
	const float* x = q.x + (size_t) s * q.x_stride;
	uint8_t* mine = q.img + (size_t) (s >> 1) * MMB_PAIR + (s & 1) * 96; // this sequence's limb planes inside a (block, pair) record
	float ss = 0.f;
	for (int base = 0; base < ngrp; base += MP * NT) {
		float xr[MP][8];
		uint4 gw[MP][2];
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = base + p * NT + tid;
			if (grp < ngrp) {
				const float4 q0 = ld_act4(x + grp * 8), q1 = ld_act4(x + grp * 8 + 4);
				xr[p][0] = q0.x; xr[p][1] = q0.y; xr[p][2] = q0.z; xr[p][3] = q0.w;
				xr[p][4] = q1.x; xr[p][5] = q1.y; xr[p][6] = q1.z; xr[p][7] = q1.w;
				if (NORM) {
					if (q.norm_type == XALM_F32) {
						gw[p][0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(q.norm_w) + grp * 8);
						gw[p][1] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(q.norm_w) + grp * 8 + 4);
					} else {
						gw[p][0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(q.norm_w) + grp * 8);
					}
				}
			} else {
#pragma unroll
				for (int e = 0; e < 8; e++) xr[p][e] = 0.f;
			}
		}
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = base + p * NT + tid;
			if (base + p * NT + warp * 32 < ngrp) { // warp-uniform: the quantiser shuffles within quads of lanes
				const bool valid = grp < ngrp;
				if (NORM && valid) {
#pragma unroll
					for (int e = 0; e < 8; e++) {
						ss += xr[p][e] * xr[p][e];
						float g;
						if (q.norm_type == XALM_F32) {
							const uint4 w = gw[p][e >> 2];
							g = __uint_as_float((e & 3) == 0 ? w.x : (e & 3) == 1 ? w.y : (e & 3) == 2 ? w.z : w.w);
						} else {
							const uint4 w = gw[p][0];
							const int h = e >> 1;
							const uint32_t u = h == 0 ? w.x : h == 1 ? w.y : h == 2 ? w.z : w.w;
							g = __uint_as_float((e & 1) ? (u & 0xFFFF0000u) : (u << 16));
						}
						xr[p][e] = xr[p][e] * g;
					}
				}
				XmGroup o;
				xm_quant_group8(xr[p], o);
				if (valid) {
					uint8_t* rec = mine + (size_t) (grp >> 2) * q.np * MMB_PAIR;
#pragma unroll
					for (int k = 0; k < 3; k++) *reinterpret_cast<uint2*>(rec + k * 32 + (grp & 3) * 8) = make_uint2(o.w[k][0], o.w[k][1]);
					if ((grp & 3) == 0) { // this sequence's two table entries (lanes tig 0, 1 of its half of the pair)
						const int S0 = (int) o.s0, S1 = (int) (o.u & 0xFFFFu), S2 = (int) (o.u >> 16);
						const int tot = (S0 - 4096) * 65536 + S1 * 256 + S2;
						const float sx = __int2float_rn(tot) * o.dx;
						int4* e = reinterpret_cast<int4*>(rec - (s & 1) * 96 + 192 + (s & 1) * 32);
						e[0] = make_int4(-BIAS * S2, -BIAS * S1, (int) __float_as_uint(o.dx), (int) __float_as_uint(sx));
						e[1] = make_int4(-BIAS * (S0 - 4096), 0, (int) __float_as_uint(o.dx * 65536.f), 0);
					}
				}
			}
		}
	}
	if (NORM) {
		ss = warp_sum(ss);
		if (lane == 0) s_red[warp] = ss;
		__syncthreads();
		if (tid == 0) {
			float tot = 0.f;
#pragma unroll
			for (int i = 0; i < MMA_NCW; i++) tot += s_red[i];
			q.nscale[s] = 1.0f / sqrtf(tot / (float) n + q.norm_eps); // infer.cpp:229-232
		}
	}
}

__host__ __device__ inline size_t mmb_stage_bytes(int type, int np) { return (size_t) MMB_SB * (frag_record_bytes(type) + (size_t) np * MMB_PAIR); }
__host__ __device__ inline size_t mmb_smem_bytes(int type, int np, int NS) {
	size_t s = (size_t) NS * mmb_stage_bytes(type, np);
	s += (size_t) mma_pb(NS) * MMA_NCW * (2 * np) * MMA_RC * sizeof(float);
	s += (2 * (size_t) NS + 2 * mma_pb(NS)) * sizeof(uint64_t);
	return s + 128;
}

struct MmbArgs {
	MatvecArgs a;          // a.step = the step's StepParams array (one per sequence), a.k_cache / a.v_cache = slot 0's caches
	int NS, n_tiles, nseq;
	const uint8_t* img;    // xq_batch_kernel's image of the input activations
	const float* nscale;   // per-sequence 1/rms, or nullptr
	int out_stride;        // floats between two sequences' outputs
	size_t kv_slot;        // elements between two slots' caches
};

template <int TYPE, int NP>
__global__ void __launch_bounds__((MMA_NCW + 2) * 32, 1) matvec_mma_batch_kernel(const MmbArgs ta) {
	using F = MmaFmt<TYPE>;
	constexpr int RC = MMA_RC, SB = MMB_SB, NCW = MMA_NCW, NT = MMA_NT, RB = F::RB, NS2 = 2 * NP;
	constexpr int WB = SB * RB, XB = SB * NP * MMB_PAIR, STAGE = WB + XB;
	const MatvecArgs& a = ta.a;
	const int NS = ta.NS, PB = mma_pb(ta.NS), nseq = ta.nseq;
	const int n = a.n, nb = n / 32;
	const int kranges = (nb + SB - 1) / SB;

	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* ring = smem;
	float* part = reinterpret_cast<float*>(ring + (size_t) NS * STAGE); // [PB][NCW][NS2][RC]
	uint64_t* full = reinterpret_cast<uint64_t*>(part + PB * NCW * NS2 * RC);
	uint64_t* empty = full + NS;
	uint64_t* pbar = empty + NS;
	uint64_t* pfree = pbar + PB;

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; s++) {
			mbar_init(&full[s], 1);
			mbar_init(&empty[s], NCW);
		}
		for (int s = 0; s < PB; s++) {
			mbar_init(&pbar[s], NCW);
			mbar_init(&pfree[s], 1);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	pdl_launch_dependents();

	const int my_tiles = ((int) blockIdx.x < ta.n_tiles) ? (ta.n_tiles - 1 - (int) blockIdx.x) / (int) gridDim.x + 1 : 0;

	if (warp == NCW) {
		// ===================== producer: the first stages' weights before the dependency wait, the image slices after it =========
		if (lane == 0) {
			const int total = my_tiles * kranges;
			auto wsrc = [&](int i, uint32_t* wbytes, uint32_t* xbytes, uint32_t* xoff) {
				const int tt = i / kranges, kr = i % kranges;
				const int nbs = min(SB, nb - kr * SB);
				*wbytes = (uint32_t) nbs * RB;
				*xbytes = (uint32_t) nbs * NP * MMB_PAIR;
				*xoff = (uint32_t) kr * XB;
				return a.w.p0 + (size_t) ((int) blockIdx.x + tt * (int) gridDim.x) * a.w.s0 + (size_t) kr * WB;
			};
			const int pre = min(NS, total);
			for (int i = 0; i < pre; i++) {
				uint32_t wb, xb, xo;
				const uint8_t* src = wsrc(i, &wb, &xb, &xo);
				mbar_expect_tx(&full[i], wb + xb);
				bulk_g2s(ring + (size_t) i * STAGE, src, wb, &full[i]);
			}
			pdl_wait(); // the image is written by the kernel before this one
			for (int i = 0; i < pre; i++) {
				uint32_t wb, xb, xo;
				wsrc(i, &wb, &xb, &xo);
				bulk_g2s(ring + (size_t) i * STAGE + WB, ta.img + xo, xb, &full[i]);
			}
			for (int i = pre; i < total; i++) {
				const int slot = i % NS, phase = (i / NS) & 1;
				uint32_t wb, xb, xo;
				const uint8_t* src = wsrc(i, &wb, &xb, &xo);
				mbar_wait(&empty[slot], phase ^ 1);
				mbar_expect_tx(&full[slot], wb + xb);
				bulk_g2s(ring + (size_t) slot * STAGE, src, wb, &full[slot]);
				bulk_g2s(ring + (size_t) slot * STAGE + WB, ta.img + xo, xb, &full[slot]);
			}
			prefetch_tail(a, false); // (K/V prefetch is off for batched steps)
		}
		return;
	}

	if (warp == NCW + 1) {
		// ===================== epilogue warp: two sequences per pass, lanes 0-15 and 16-31 each take the 16 rows of one =============
		pdl_wait();
		const int r = lane & (RC - 1);
		int pb = 0, pph = 0;
		for (int tt = 0; tt < my_tiles; tt++) {
			const int row0 = ((int) blockIdx.x + tt * (int) gridDim.x) * RC;
			float xold[NP];
#pragma unroll
			for (int ps = 0; ps < NP; ps++) {
				const int s = 2 * ps + (lane >> 4);
				xold[ps] = 0.f;
				if (a.epi == EPI_RESIDUAL && s < nseq && row0 + r < a.d) xold[ps] = a.out[(size_t) s * ta.out_stride + row0 + r];
			}
			mbar_wait(&pbar[pb], pph);
			const float* pt = part + pb * NCW * NS2 * RC;
#pragma unroll
			for (int ps = 0; ps < NP; ps++) {
				const int s = 2 * ps + (lane >> 4);
				const bool live = s < nseq;
				float yv = 0.f;
				if (live) {
#pragma unroll
					for (int w = 0; w < NCW; w++) yv += pt[(w * NS2 + s) * RC + r];
					if (ta.nscale) yv *= ta.nscale[s];
				}
				const float ynext = __shfl_down_sync(0xffffffffu, yv, 1);
				const float ypart = __shfl_down_sync(0xffffffffu, yv, RC / 2);
				if (!live) continue;
				float* out = a.out + (size_t) s * ta.out_stride;
				const int row = row0 + r;
				if (a.epi == EPI_RESIDUAL) {
					if (row < a.d) out[row] = xold[ps] + yv;
				} else if (a.epi == EPI_STORE) {
					if (row < a.d) out[row] = yv;
				} else if (a.epi == EPI_GLU) {
					const int o = row0 / 2 + r;
					if (r < RC / 2 && o < a.d) {
						const float gt = a.act == XALM_SILU ? act_silu(yv) : act_gelu(yv);
						out[o] = gt * ypart;
					}
				} else if ((r & 1) == 0 && row < a.d) { // EPI_QKV into this slot's ring
					qkv_pair(a, a.step[s], ta.kv_slot, out, row, yv, ynext);
				}
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&pfree[pb]);
			if (++pb == PB) { pb = 0; pph ^= 1; }
		}
		return;
	}

	// ===================== consumers =====================
	pdl_wait();
	if (a.epi == EPI_QKV && blockIdx.x == 0) { // re-rotate the attention sinks of every sequence past its window
		for (int s = 0; s < nseq; s++) rotate_sinks(a, a.k_cache + (size_t) a.step[s].slot * ta.kv_slot, a.step[s].kv_sink, threadIdx.x, NT);
	}

	// this lane's place in the mma fragments: column g of the B operand is limb plane (2 - g) of sequence 2p (g < 3), the ones column
	// (g = 3, 7) or limb plane (6 - g) of sequence 2p + 1 (4 <= g < 7); accumulator columns 2 tig, 2 tig + 1
	const int g = lane >> 2, tig = lane & 3;
	const int vmul = (tig & 1) ? -128 : 256;
	const bool ones = (g & 3) == 3;
	const int boff = (g < 4 ? (2 - g) * 32 : 96 + (6 - g) * 32) + tig * 4;
	const int toff = 192 + tig * 16;

	int slot = 0, phase = 0;
	int pb_next = 0, pph_next = 0;
	for (int tt = 0; tt < my_tiles; tt++) {
		const int pb = pb_next, pph = pph_next;
		if (++pb_next == PB) { pb_next = 0; pph_next ^= 1; }
		float y0[NP], y1[NP]; // rows g and g + 8 of the tile, this lane's sequence of each pair
#pragma unroll
		for (int p = 0; p < NP; p++) y0[p] = y1[p] = 0.f;
		for (int kr = 0; kr < kranges; kr++) {
			const int nbs = min(SB, nb - kr * SB);
			const uint8_t* st = ring + (size_t) slot * STAGE;
			mbar_wait(&full[slot], phase);
			auto record = [&](int j) {
				const uint8_t* rec = st + (size_t) j * RB;
				const uint8_t* xr = st + WB + (size_t) j * NP * MMB_PAIR;
				uint32_t A[4];
				float d0, d1, m0 = 0.f, m1 = 0.f;
				F::load(rec, lane, g, A, d0, d1, m0, m1);
#pragma unroll
				for (int p = 0; p < NP; p++) {
					const uint8_t* xp = xr + p * MMB_PAIR;
					uint32_t B0 = 0x01010101u, B1 = 0x01010101u;
					if (!ones) {
						B0 = *reinterpret_cast<const uint32_t*>(xp + boff);
						B1 = *reinterpret_cast<const uint32_t*>(xp + boff + 16);
					}
					const int4 tb = *reinterpret_cast<const int4*>(xp + toff);
					int c[4];
					mma_u8(c, A, B0, B1, tb.x, tb.y);
					const int v0 = c[1] * vmul + c[0], v1 = c[3] * vmul + c[2];
					const float dxl = __int_as_float(tb.z);
					y0[p] = fmaf(__int2float_rn(v0), d0 * dxl, y0[p]);
					y1[p] = fmaf(__int2float_rn(v1), d1 * dxl, y1[p]);
					if (F::HAS_MIN) {
						const float sxl = __int_as_float(tb.w);
						y0[p] = fmaf(m0, sxl, y0[p]);
						y1[p] = fmaf(m1, sxl, y1[p]);
					}
				}
			};
			if (nbs == SB) {
#pragma unroll
				for (int i = 0; i < SB / NCW; i++) record(warp + i * NCW);
			} else {
				for (int j = warp; j < nbs; j += NCW) record(j);
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&empty[slot]);
			if (++slot == NS) { slot = 0; phase ^= 1; }
		}
		// ---- the two lanes of a sequence -> one sum per row (+0: the batch-1 kernel's zero-column lanes), warps -> shared memory ----
#pragma unroll
		for (int p = 0; p < NP; p++) {
			y0[p] += __shfl_xor_sync(0xffffffffu, y0[p], 1);
			y1[p] += __shfl_xor_sync(0xffffffffu, y1[p], 1);
			y0[p] = __fadd_rn(y0[p], 0.f);
			y1[p] = __fadd_rn(y1[p], 0.f);
		}
		if (tt >= PB) mbar_wait(&pfree[pb], pph ^ 1);
		if ((tig & 1) == 0) {
#pragma unroll
			for (int p = 0; p < NP; p++) {
				float* pt = part + ((pb * NCW + warp) * NS2 + 2 * p + (tig >> 1)) * RC;
				pt[g] = y0[p];
				pt[g + 8] = y1[p];
			}
		}
		__syncwarp();
		if (lane == 0) mbar_arrive(&pbar[pb]);
	}
}

} // namespace xalm
