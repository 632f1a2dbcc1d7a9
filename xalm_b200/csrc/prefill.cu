// prefill.cu — batched prefill / perplexity (BASELINE config 3): the whole prompt goes through every layer at once,
// the seven per-layer contractions become GEMMs on the 5th-generation tensor cores (tcgen05.mma, accumulators in
// TMEM), everything else stays the reference's arithmetic (infer.cpp:365-496) applied to T rows instead of one.
//
// What the reference does instead: main.cpp:244-254 (perplexity) and :94-100 (prompt hydrate) call Model::forward once
// per position — T matvec passes over all weights.  Here the weights are read once per prompt.
//
// Data flow per layer (T = tokens in this call, all buffers in HBM, sized for Tp = ceil(T/128)*128 rows):
//   x fp32 (T,dim) --rmsnorm_rows--> xb  [A tiles fp16]
//   xb . Wqkv^T    --gemm, QKV epilogue (clip, RoPE at pos0+row, fp16)--> q (T,q_dim) fp16; K/V cache rows pos0..pos0+T-1
//   causal attention over the fp16 cache: tcgen05 QK^T / PV with S and O in TMEM for head_dim 128 (attn_tc_kernel), mma.sync
//   tiles for head_dim 64 (attn_prefill_kernel); fp32 online softmax either way --> xb2 [A tiles]
//   xb2 . Wo^T     --gemm, residual epilogue--> x += .
//   x --rmsnorm_rows--> xb;  xb . (W1|W3)^T --gemm, GLU epilogue act(g)*u--> hb [A tiles]
//   hb . W2^T      --gemm, residual epilogue--> x += .
// then final rmsnorm, classifier GEMM -> logits fp32 (rows, vocab), and softmax-at-target for perplexity.
// Past the context window (window mode) the same loop runs over the KV ring with its two attention sinks: see
// gather_ring_kernel / sink_versions_kernel and the window-mode notes of the attention kernels.
//
// Operand layout ("A tiles"/"B tiles"): 128 (A) or 256 (B) rows x 64 K-elements of fp16, stored as the exact
// shared-memory image tcgen05.mma wants for a K-major SWIZZLE_128B operand (8-row x 128-byte atoms, 16-byte chunks
// XOR-swizzled by row%8), tile after tile.  One cp.async.bulk (TMA engine) brings a whole 16/32 KB tile into shared
// memory — no tensor map, no per-thread staging.  Weights are dequantised from their decode layout into B tiles once
// per GEMM (dequant_tiles_kernel: every format the decode path takes), which costs 2 bytes written + read per weight
// against 2*T flops per weight: ~10 % of the GEMM at T = 4096.
//
// Numerics: tensor-core operands are fp16 with fp32 accumulation.  split=1 rounds every operand to fp16 (fastest; ten rounding
// stages per layer add up to ~4e-2 on the logits of a 32-layer model).  split=2 keeps the activations to ~fp32 by feeding
// hi = fp16(a) and lo = fp16(a - hi) as two MMAs against the same weight tile.  split=3 (default) does the same for the weights
// (hi.hi + lo.hi + hi.lo) and for q and the softmax probabilities in attention: logits within ~1e-3 of the token-at-a-time
// fp32 path at 32 layers x 4096 tokens.  Tolerance in tests: 1e-2 (north star: "within max-abs 1e-2 (fp16)").
#define XALM_SECONDARY_TU
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <float.h>
#include <limits.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "matvec.cuh"
#include "frag_layout.cuh"
#include "nccl_api.h"
#include "prefill.h"

namespace xalm {

// ------------------------------------------------------------------------------------------------------------------
// tile geometry
// ------------------------------------------------------------------------------------------------------------------
constexpr int GB_M = 128;  // rows of an A tile = UMMA M
constexpr int GB_N = 256;  // rows of a B tile = UMMA N
constexpr int GB_K = 64;   // K elements per tile = one 128-byte swizzle row of fp16
constexpr int A_TILE_BYTES = GB_M * GB_K * 2;
constexpr int B_TILE_BYTES = GB_N * GB_K * 2;
constexpr int UMMA_K = 16;

// byte offset of element (r, c) inside a tile (r < 128 or 256, c < 64): 8-row atoms of 1024 bytes, chunk ^= row % 8
__host__ __device__ __forceinline__ size_t tile_inner_off(int r, int c) {
	return (size_t) (r >> 3) * 1024 + (size_t) (r & 7) * 128 + (size_t) ((((c >> 3) ^ r) & 7) << 4) + (size_t) (c & 7) * 2;
}
__host__ __device__ __forceinline__ size_t a_off(int m, int k, int KT) {
	return ((size_t) (m / GB_M) * KT + (size_t) (k / GB_K)) * A_TILE_BYTES + tile_inner_off(m % GB_M, k % GB_K);
}

struct ATiles {      // activations as tensor-core operands
	uint8_t* hi = nullptr;
	uint8_t* lo = nullptr; // residual plane (split = 2), else nullptr
	int KT = 0;      // K tiles per row block
};

// pack 8 floats into 8 fp16 (hi) and, optionally, the fp16 of the rounding residuals (lo)
__device__ __forceinline__ void store_a8(const ATiles& a, int m, int k0, const float (&v)[8]) {
	const size_t off = a_off(m, k0, a.KT);
	__half2 h[4];
#pragma unroll
	for (int i = 0; i < 4; i++) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
	*reinterpret_cast<uint4*>(a.hi + off) = *reinterpret_cast<const uint4*>(h);
	if (a.lo) {
		__half2 l[4];
#pragma unroll
		for (int i = 0; i < 4; i++) {
			const float2 f = __half22float2(h[i]);
			l[i] = __floats2half2_rn(v[2 * i] - f.x, v[2 * i + 1] - f.y);
		}
		*reinterpret_cast<uint4*>(a.lo + off) = *reinterpret_cast<const uint4*>(l);
	}
}

// ------------------------------------------------------------------------------------------------------------------
// weights -> B tiles: element (row, k) of a WMat in ANY of the decode layouts -> fp16
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ld_h(const uint8_t* p) { return __half2float(*reinterpret_cast<const __half*>(p)); }

// 8 consecutive elements k0..k0+7 (k0 % 8 == 0) of physical row `r`
// TT: compile-time type (the switch folds away) or -1 for "whatever w.type says"; LU: 2 = fragment tiles, 1 = unit-interleaved, 0 = planar, -1 = runtime
template <int TT, int LU>
__device__ __forceinline__ void wmat_decode8(const WMat& w, int r, int k0, float (&v)[8]) {
	const int t = TT >= 0 ? TT : w.type;
	if (LU == 2 || (LU < 0 && w.layout_frag)) { // fragment tiles of the tensor-core decode matvec (frag_layout.cuh)
		frag_decode8(w, t, r, k0, v);
		return;
	}
	const uint8_t* row = w.p0 + (size_t) r * w.s0;
	switch (t) {
		case XALM_F32: {
			const float4 a = *reinterpret_cast<const float4*>(row + (size_t) k0 * 4);
			const float4 b = *reinterpret_cast<const float4*>(row + (size_t) k0 * 4 + 16);
			v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
			return;
		}
		case XALM_F16: case XALM_BF16: {
			const uint4 q = *reinterpret_cast<const uint4*>(row + (size_t) k0 * 2);
			const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
			for (int i = 0; i < 4; i++) {
				if (t == XALM_F16) {
					const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
					v[2 * i] = f.x; v[2 * i + 1] = f.y;
				} else {
					v[2 * i] = __uint_as_float(u[i] << 16); v[2 * i + 1] = __uint_as_float(u[i] & 0xFFFF0000u);
				}
			}
			return;
		}
		case XALM_F8_E2M5: case XALM_F8_E3M4: case XALM_F8_E4M3: case XALM_F8_E5M2: case XALM_U8: case XALM_Q8: case XALM_QI8: {
			const uint2 q = *reinterpret_cast<const uint2*>(row + k0);
			const uint32_t u[2] = {q.x, q.y};
#pragma unroll
			for (int i = 0; i < 8; i++) {
				uint8_t b = (uint8_t) (u[i >> 2] >> (8 * (i & 3)));
				if (t == XALM_Q8) b ^= 0x80; // stored biased on the device (formats.cuh)
				v[i] = decode_byte_type(t, b);
			}
			return;
		}
		case XALM_TQ1_0: {
			const uint8_t* blk = row + (size_t) (k0 / 256) * 54;
#pragma unroll
			for (int i = 0; i < 8; i++) v[i] = decode_block_elem(t, blk, (k0 % 256) + i);
			return;
		}
	}
	// ---- 32-element block formats: locate main bytes / scales / high bits in the unit-interleaved or planar layout ----
	const int blk = k0 / 32, j0 = k0 % 32;
	const uint8_t *mainp, *scp, *qhp = nullptr;
	const int sc_bytes = (t == XALM_Q4_1 || t == XALM_Q5_1) ? 4 : 2;
	const int main_per_blk = t == XALM_Q8_0 ? 32 : 16;
	if (LU >= 0 ? LU != 0 : w.layout_units != 0) {
		const int ub = t == XALM_Q8_0 ? 272 : t == XALM_Q4_0 ? 144 : t == XALM_Q4_1 ? 160 : t == XALM_Q5_0 ? 176 : 192;
		const uint8_t* unit = row + (size_t) (k0 / 256) * ub;
		const int b = blk & 7;
		const int main_bytes = main_per_blk * 8;
		mainp = unit + b * main_per_blk;
		scp = unit + main_bytes + b * sc_bytes;
		if (t == XALM_Q5_0) qhp = unit + 144 + 4 * b;
		if (t == XALM_Q5_1) qhp = unit + 160 + 4 * b;
	} else {
		mainp = row + (size_t) blk * main_per_blk;
		scp = w.p1 + (size_t) r * w.s1 + (size_t) blk * sc_bytes;
		if (w.p2) qhp = w.p2 + (size_t) r * w.s2 + (size_t) blk * 4;
	}
	const float d = ld_h(scp);
	if (t == XALM_Q8_0) {
		const uint2 q = *reinterpret_cast<const uint2*>(mainp + j0);
		const uint32_t u[2] = {q.x, q.y};
#pragma unroll
		for (int i = 0; i < 8; i++) v[i] = __fmul_rn(d, (float) ((int) ((u[i >> 2] >> (8 * (i & 3))) & 0xFF) - 128));
		return;
	}
	const float mn = sc_bytes == 4 ? ld_h(scp + 2) : 0.f;
	const uint2 q = *reinterpret_cast<const uint2*>(mainp + (j0 & 15)); // nibble bytes of elements j0..j0+7 (low half: j < 16)
	const uint32_t u[2] = {q.x, q.y};
	const uint32_t qh = qhp ? *reinterpret_cast<const uint32_t*>(qhp) : 0u;
#pragma unroll
	for (int i = 0; i < 8; i++) {
		const uint32_t byte = (u[i >> 2] >> (8 * (i & 3))) & 0xFF;
		int qv = (j0 < 16) ? (int) (byte & 0x0F) : (int) (byte >> 4);
		if (qhp) qv |= (int) ((qh >> (j0 + i)) & 1u) << 4;
		switch (t) {
			case XALM_Q4_0: v[i] = __fmul_rn(d, (float) (qv - 8)); break;
			case XALM_Q5_0: v[i] = __fmul_rn(d, (float) (qv - 16)); break;
			default: v[i] = __fadd_rn(__fmul_rn(d, (float) qv), mn); break; // Q4_1, Q5_1
		}
	}
}

// One thread per 16-byte chunk of the destination, in destination order (coalesced stores).  Destination row n of
// B tile `nt`: plain matrices -> physical row nt*256 + n;  GLU (glu_off > 0 or glu) -> n < 128: W1 row nt*128 + n,
// else W3 row glu_off + nt*128 + (n-128), so gate and up of the same hidden unit land in one accumulator row block.
template <int TT, int LU>
__global__ void dequant_tiles_kernel(const WMat w, int glu, int glu_off, int n_valid, int K, int NT, int KT, uint8_t* __restrict__ dst,
                                     uint8_t* __restrict__ dst_lo) {
	const size_t chunks_per_tile = B_TILE_BYTES / 16;
	const size_t total = (size_t) NT * KT * chunks_per_tile;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const size_t tile = i / chunks_per_tile;
		const int ci = (int) (i % chunks_per_tile);
		const int nt = (int) (tile / KT), kt = (int) (tile % KT);
		const int r = (ci >> 6) * 8 + ((ci & 63) >> 3);
		const int lc = (ci & 7) ^ (r & 7);
		const int k0 = kt * GB_K + lc * 8;
		int prow;
		bool valid;
		if (glu) {
			const int o = nt * (GB_N / 2) + (r % (GB_N / 2));
			valid = o < n_valid;
			prow = r < GB_N / 2 ? o : glu_off + o;
		} else {
			prow = nt * GB_N + r;
			valid = prow < n_valid;
		}
		uint4 out = make_uint4(0, 0, 0, 0), out_lo = make_uint4(0, 0, 0, 0);
		if (valid && k0 < K) {
			float v[8];
			wmat_decode8<TT, LU>(w, prow, k0, v);
			__half2 h[4], l[4];
#pragma unroll
			for (int j = 0; j < 4; j++) {
				h[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
				const float2 f = __half22float2(h[j]);
				l[j] = __floats2half2_rn(v[2 * j] - f.x, v[2 * j + 1] - f.y); // what fp16 dropped (exact difference, then rounded)
			}
			out = *reinterpret_cast<const uint4*>(h);
			out_lo = *reinterpret_cast<const uint4*>(l);
		}
		*reinterpret_cast<uint4*>(dst + i * 16) = out;
		if (dst_lo) *reinterpret_cast<uint4*>(dst_lo + i * 16) = out_lo;
	}
}

// ------------------------------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier, bulk copy, tcgen05
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_u32(bar)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "WAIT_%=:\n"
	    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	    "@p bra DONE_%=;\n"
	    "bra WAIT_%=;\n"
	    "DONE_%=:\n"
	    "}\n" ::"r"(s_u32(bar)),
	    "r"(parity)
	    : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s_u32(dst)), "l"(src),
	             "r"(bytes), "r"(s_u32(bar))
	             : "memory");
}
// one lane of a converged warp (elect.sync): lets the compiler keep the tcgen05 issue in a warp-uniform branch
__device__ __forceinline__ bool elect_one() {
	uint32_t pred;
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "elect.sync _|p, 0xffffffff;\n"
	    "selp.u32 %0, 1, 0, p;\n"
	    "}\n"
	    : "=r"(pred));
	return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// whole warp: allocate `cols` TMEM columns (power of two >= 32), base address -> *slot (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
	asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_u32(slot)), "r"(cols) : "memory");
	asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
	asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, fp16 operands, fp32 accumulate; issued by ONE thread for the CTA
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "setp.ne.b32 p, %4, 0;\n"
	    "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
	    "}\n" ::"r"(tmem_d),
	    "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
	    : "memory");
}
// all MMAs issued so far by this thread -> one arrival on `bar` when they have completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
	asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_u32(bar)) : "memory");
}
// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row atoms 1024 bytes apart (SBO), sm_100 descriptor version 1
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
	return (uint64_t) ((saddr & 0x3FFFFu) >> 4) | ((uint64_t) (1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor, kind::f16: D fp32 (bits 4-5 = 1), A/B fp16 (0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t instr_desc_f16(int M, int N) {
	return (1u << 4) | ((uint32_t) (N >> 3) << 17) | ((uint32_t) (M >> 4) << 24);
}
// 32 lanes x 16 consecutive fp32 columns of this warp's TMEM quadrant
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
	uint32_t r[16];
	__syncwarp(); // .sync.aligned: the whole warp, converged
	asm volatile(
	    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
	    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
	      "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
	    : "r"(taddr));
	asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
	for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
	uint32_t r[32];
	__syncwarp();
	asm volatile(
	    "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
	    "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
	    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
	      "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
	      "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
	      "=r"(r[30]), "=r"(r[31])
	    : "r"(taddr));
	asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
	for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
// issue only (no wait): lets several loads fly before one tmem_wait_ld()
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, float* v) {
	uint32_t r[32];
	asm volatile(
	    "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
	    "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
	    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
	      "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
	      "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
	      "=r"(r[30]), "=r"(r[31])
	    : "r"(taddr));
#pragma unroll
	for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
	asm volatile(
	    "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
	    "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
	    "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
	    "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])),
	    "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
	    "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])), "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])),
	    "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])), "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])),
	    "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])), "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])),
	    "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])), "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])),
	    "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
	    : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
	uint32_t r[8];
	__syncwarp();
	asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
	             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
	             : "r"(taddr));
	asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
	for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}

// ------------------------------------------------------------------------------------------------------------------
// the GEMM: out(M, N) = A(M, K) . B(N, K)^T, persistent warp-specialised CTAs, one per SM
//   warp 0    producer: one lane issues cp.async.bulk for the A tile(s) + B tile of each K step into a ring of NS stages
//   warp 1    allocates TMEM; one lane issues tcgen05.mma (4 x K=16 per stage, x NA activation planes) and commits
//   warps 2-5 epilogue: tcgen05.ld the 128 x 256 fp32 accumulator (one TMEM lane quadrant per warp) and apply the
//             fused epilogue, while the MMA warp already fills the OTHER accumulator buffer (2 x 256 of the 512 columns)
// ------------------------------------------------------------------------------------------------------------------
enum { GEPI_STORE = 0, GEPI_RESID = 1, GEPI_GLU = 2, GEPI_QKV = 3 };

struct GemmArgs {
	const uint8_t* a_hi;
	const uint8_t* a_lo;
	const uint8_t* b;
	const uint8_t* b_lo; // residual plane of the weights (NB = 2)
	int MT, NT, KT;     // tile counts; M tiles are [mt0, mt0 + MT)
	int mt0;
	int M;              // valid rows
	int N;              // valid outputs (GLU: hidden units; else columns)
	int epi;
	float* out;         // STORE / RESID: row-major, leading dimension ldo, row index (m - out_row0)
	int ldo;
	int out_row0;
	// QKV
	__half* q_out;      // (T, q_dim) row-major fp16, RoPE applied
	__half* q_lo;       // fp16 of what q_out's rounding dropped (precise mode), or nullptr
	uint8_t* qt_hi;     // when set: q goes into 128-row x 64-column operand tiles ((head, row block, hd half) order) for attn_tc_kernel
	uint8_t* qt_lo;     // instead of row-major q_out / q_lo
	int n_qb;           // row blocks of 128
	uint8_t* kt;        // when set (pos0 == 0, head_dim 128): K and V^T operand tiles of attn_tc_kernel are written here as well,
	uint8_t* vt;        // so no re-tiling pass over the cache is needed
	int n_kb_total;     // 128-key blocks per kv head in kt / vt
	__half* k_cache;
	__half* v_cache;
	int ring;           // window mode: the KV cache is a ring of this many data slots after 2 sinks (cache row 2 + (pos - 2) % ring); 0 = linear
	__half* k_stage;    // window mode: K / V rows also go to these linear staging buffers, row stage_row0 + m (attention reads them)
	__half* v_stage;
	int stage_row0;
	const float2* rope_cs; // (T, head_dim/2): {cos, sin}(pos * freq) per row, from rope_table_kernel
	int q_dim, kv_dim, head_dim, pos0; // pos0: position of row 0 (the cache row in linear mode)
	float qkv_clip;
	// GLU
	ATiles o;
	int act;
};

constexpr int GEMM_THREADS = 192;
// NA activation planes x NB weight planes: (1,1) fp16 x fp16; (2,1) hi+lo activations; (2,2) hi+lo on both sides, three MMAs per
// K step (hi.hi + lo.hi + hi.lo; lo.lo is below fp32 resolution) = fp32-grade products on the fp16 tensor pipe
template <int NA, int NB>
struct GemmCfg {
	static constexpr int STAGE = NA * A_TILE_BYTES + NB * B_TILE_BYTES;
	static constexpr int NS = (200 * 1024) / STAGE;
	static constexpr size_t SMEM = (size_t) NS * STAGE + 1024 /* alignment slack */ + 256 /* barriers */;
};

template <int NA, int NB>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_tc_kernel(const GemmArgs g) {
	using Cfg = GemmCfg<NA, NB>;
	constexpr int NS = Cfg::NS;
	extern __shared__ uint8_t smem_raw[];
	// 1024-byte alignment in the SHARED address space (the swizzle pattern is a function of the address bits)
	const uint32_t raw_s = s_u32(smem_raw);
	uint8_t* smem = smem_raw + (((raw_s + 1023u) & ~1023u) - raw_s);
	uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t) NS * Cfg::STAGE);
	uint64_t* empty = full + NS;
	uint64_t* tfull = empty + NS;   // [2] accumulator ready
	uint64_t* tempty = tfull + 2;   // [2] accumulator drained
	uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; s++) {
			mb_init(&full[s], 1);
			mb_init(&empty[s], 1);
		}
		for (int i = 0; i < 2; i++) {
			mb_init(&tfull[i], 1);
			mb_init(&tempty[i], 4);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	if (warp == 1) tmem_alloc(tmem_slot, 512);
	tc_fence_before();
	__syncthreads();
	tc_fence_after();
	const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

	const int n_tiles = g.MT * g.NT;
	const int KT = g.KT;

	if (warp == 0) {
		if (lane == 0) {
			int slot = 0, phase = 0;
			for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
				const int mt = g.mt0 + tile % g.MT, nt = tile / g.MT;
				const uint8_t* ah = g.a_hi + (size_t) mt * KT * A_TILE_BYTES;
				const uint8_t* al = NA == 2 ? g.a_lo + (size_t) mt * KT * A_TILE_BYTES : nullptr;
				const uint8_t* bt = g.b + (size_t) nt * KT * B_TILE_BYTES;
				const uint8_t* bl = NB == 2 ? g.b_lo + (size_t) nt * KT * B_TILE_BYTES : nullptr;
				for (int kt = 0; kt < KT; kt++) {
					mb_wait(&empty[slot], phase ^ 1);
					uint8_t* st = smem + (size_t) slot * Cfg::STAGE;
					mb_expect_tx(&full[slot], Cfg::STAGE);
					bulk_load(st, ah + (size_t) kt * A_TILE_BYTES, A_TILE_BYTES, &full[slot]);
					if (NA == 2) bulk_load(st + A_TILE_BYTES, al + (size_t) kt * A_TILE_BYTES, A_TILE_BYTES, &full[slot]);
					bulk_load(st + NA * A_TILE_BYTES, bt + (size_t) kt * B_TILE_BYTES, B_TILE_BYTES, &full[slot]);
					if (NB == 2) bulk_load(st + NA * A_TILE_BYTES + B_TILE_BYTES, bl + (size_t) kt * B_TILE_BYTES, B_TILE_BYTES, &full[slot]);
					if (++slot == NS) { slot = 0; phase ^= 1; }
				}
			}
		}
		__syncwarp();
	} else if (warp == 1) {
		if (lane == 0) {
			constexpr uint32_t idesc = instr_desc_f16(GB_M, GB_N);
			int slot = 0, phase = 0, acc = 0, acc_phase = 0;
			for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
				mb_wait(&tempty[acc], acc_phase ^ 1);
				tc_fence_after();
				const uint32_t d_tmem = tmem_base + (uint32_t) acc * GB_N;
				for (int kt = 0; kt < KT; kt++) {
					mb_wait(&full[slot], phase);
					tc_fence_after();
					const uint32_t sa = s_u32(smem + (size_t) slot * Cfg::STAGE);
#pragma unroll
					for (int p = 0; p < NA + NB - 1; p++) { // (a_hi, b_hi), (a_lo, b_hi), (a_hi, b_lo)
						const uint64_t adesc = smem_desc(sa + (p == 1 ? A_TILE_BYTES : 0));
						const uint64_t bdesc = smem_desc(sa + NA * A_TILE_BYTES + (p == 2 ? B_TILE_BYTES : 0));
#pragma unroll
						for (int k = 0; k < GB_K / UMMA_K; k++) {
							// advancing K by 16 fp16 = 32 bytes inside the 128-byte swizzle row: +2 in the (>>4) address field
							umma_f16(d_tmem, adesc + (uint64_t) (2 * k), bdesc + (uint64_t) (2 * k), idesc, (uint32_t) ((kt | k | p) != 0));
						}
					}
					umma_commit(&empty[slot]); // frees the stage once these MMAs have read it
					if (++slot == NS) { slot = 0; phase ^= 1; }
				}
				umma_commit(&tfull[acc]);
				acc ^= 1;
				if (acc == 0) acc_phase ^= 1;
			}
		}
		__syncwarp();
	} else {
		const int quad = warp & 3; // TMEM lanes [32*quad, 32*quad+32) are the ones this warp may read
		int acc = 0, acc_phase = 0;
		for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
			const int mt = g.mt0 + tile % g.MT, nt = tile / g.MT;
			mb_wait(&tfull[acc], acc_phase);
			tc_fence_after();
			const int m = mt * GB_M + quad * 32 + lane;
			const bool mrow = m < g.M;
			const uint32_t taddr = tmem_base + ((uint32_t) (quad * 32) << 16) + (uint32_t) acc * GB_N;
			if (g.epi == GEPI_GLU) {
				for (int c = 0; c < GB_N / 2; c += 8) {
					float gt[8], up[8];
					tmem_ld8(taddr + c, gt);
					tmem_ld8(taddr + GB_N / 2 + c, up);
					const int o0 = nt * (GB_N / 2) + c;
					if (mrow && o0 < g.N) {
						float h[8];
#pragma unroll
						for (int i = 0; i < 8; i++) h[i] = (g.act == XALM_SILU ? act_silu(gt[i]) : act_gelu(gt[i])) * up[i]; // infer.cpp:470-488
						store_a8(g.o, m, o0, h);
					}
				}
			} else if (g.epi == GEPI_QKV) {
				// 16 columns = 8 rotation pairs at a time; q_dim, kv_dim and head_dim are multiples of 16, so a chunk never straddles
				// the q | k | v regions or a head, and leaves as two 16-byte stores
				const int pos = g.pos0 + m;
				const int crow = g.ring ? 2 + (pos - 2) % g.ring : pos; // KV cache row of this position
				const float2* cs_row = g.rope_cs + (size_t) (mrow ? m : 0) * (g.head_dim / 2);
				for (int c = 0; c < GB_N; c += 16) {
					float v[16];
					tmem_ld16(taddr + c, v);
					const int n0 = nt * GB_N + c;
					if (!mrow || n0 >= g.N) continue;
					const int region = n0 < g.q_dim ? 0 : (n0 < g.q_dim + g.kv_dim ? 1 : 2);
					const int j0 = n0 - (region == 0 ? 0 : region == 1 ? g.q_dim : g.q_dim + g.kv_dim); // column inside the region
#pragma unroll
					for (int i = 0; i < 16; i++) v[i] = clipf(v[i], g.qkv_clip); // infer.cpp:389-399
					if (region < 2) { // rope (infer.cpp:305-322) on q and k: the same sincosf(pos * freq) values as the decode kernels
						const float4* cs4 = reinterpret_cast<const float4*>(cs_row + ((j0 % g.head_dim) >> 1));
#pragma unroll
						for (int i = 0; i < 4; i++) {
							const float4 t = cs4[i]; // {cos, sin} of two consecutive pairs
							const float a0 = v[4 * i], b0 = v[4 * i + 1], a1 = v[4 * i + 2], b1 = v[4 * i + 3];
							v[4 * i] = a0 * t.x - b0 * t.y; v[4 * i + 1] = a0 * t.y + b0 * t.x;
							v[4 * i + 2] = a1 * t.z - b1 * t.w; v[4 * i + 3] = a1 * t.w + b1 * t.z;
						}
					}
					__half2 h[8];
#pragma unroll
					for (int i = 0; i < 8; i++) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
					if (region == 0 && g.qt_hi) { // head_dim 128: tile ((head * n_qb + m / 128) * 2 + hd half), row m % 128
						const int head = j0 >> 7, hc = j0 & 127;
						const size_t toff = ((size_t) (head * g.n_qb + (m >> 7)) * 2 + (hc >> 6)) * A_TILE_BYTES;
						const size_t o0 = toff + tile_inner_off(m & 127, hc & 63), o1 = toff + tile_inner_off(m & 127, (hc & 63) + 8);
						*reinterpret_cast<uint4*>(g.qt_hi + o0) = reinterpret_cast<const uint4*>(h)[0];
						*reinterpret_cast<uint4*>(g.qt_hi + o1) = reinterpret_cast<const uint4*>(h)[1];
						if (g.qt_lo) {
							__half2 l[8];
#pragma unroll
							for (int i = 0; i < 8; i++) {
								const float2 f = __half22float2(h[i]);
								l[i] = __floats2half2_rn(v[2 * i] - f.x, v[2 * i + 1] - f.y);
							}
							*reinterpret_cast<uint4*>(g.qt_lo + o0) = reinterpret_cast<const uint4*>(l)[0];
							*reinterpret_cast<uint4*>(g.qt_lo + o1) = reinterpret_cast<const uint4*>(l)[1];
						}
						continue;
					}
					__half* dst = region == 0 ? g.q_out + (size_t) m * g.q_dim + j0
					            : region == 1 ? g.k_cache + (size_t) crow * g.kv_dim + j0 : g.v_cache + (size_t) crow * g.kv_dim + j0;
					reinterpret_cast<uint4*>(dst)[0] = reinterpret_cast<const uint4*>(h)[0];
					reinterpret_cast<uint4*>(dst)[1] = reinterpret_cast<const uint4*>(h)[1];
					if (region > 0 && g.k_stage) {
						__half* sd = (region == 1 ? g.k_stage : g.v_stage) + (size_t) (g.stage_row0 + m) * g.kv_dim + j0;
						reinterpret_cast<uint4*>(sd)[0] = reinterpret_cast<const uint4*>(h)[0];
						reinterpret_cast<uint4*>(sd)[1] = reinterpret_cast<const uint4*>(h)[1];
					}
					if (region > 0 && g.kt) { // the same values as operand tiles (key = pos: this path is only taken with pos0 == 0)
						const int kvh = j0 >> 7, hc = j0 & 127;
						const size_t blk = (size_t) (kvh * g.n_kb_total + (pos >> 7)) * 2;
						if (region == 1) { // K tile (kv head, 128-key block, hd half): row = key, 64 hd columns
							uint8_t* t = g.kt + (blk + (hc >> 6)) * A_TILE_BYTES;
							*reinterpret_cast<uint4*>(t + tile_inner_off(pos & 127, hc & 63)) = reinterpret_cast<const uint4*>(h)[0];
							*reinterpret_cast<uint4*>(t + tile_inner_off(pos & 127, (hc & 63) + 8)) = reinterpret_cast<const uint4*>(h)[1];
						} else {           // V^T tile (kv head, 128-key block, key half): row = hd, 64 key columns; a warp covers 32 consecutive keys
							uint8_t* t = g.vt + (blk + ((pos & 127) >> 6)) * A_TILE_BYTES;
							const __half* hv = reinterpret_cast<const __half*>(h);
#pragma unroll
							for (int i = 0; i < 16; i++) *reinterpret_cast<__half*>(t + tile_inner_off(hc + i, pos & 63)) = hv[i];
						}
					}
					if (region == 0 && g.q_lo) {
						__half2 l[8];
#pragma unroll
						for (int i = 0; i < 8; i++) {
							const float2 f = __half22float2(h[i]);
							l[i] = __floats2half2_rn(v[2 * i] - f.x, v[2 * i + 1] - f.y);
						}
						uint4* dl = reinterpret_cast<uint4*>(g.q_lo + (size_t) m * g.q_dim + j0);
						dl[0] = reinterpret_cast<const uint4*>(l)[0];
						dl[1] = reinterpret_cast<const uint4*>(l)[1];
					}
				}
			} else {
				for (int c = 0; c < GB_N; c += 32) { // 32 columns = one full 128-byte line per thread
					float v[32];
					tmem_ld32(taddr + c, v);
					const int n0 = nt * GB_N + c;
					if (!mrow || n0 >= g.N) continue;
					float* o = g.out + (size_t) (m - g.out_row0) * g.ldo + n0;
#pragma unroll
					for (int i = 0; i < 32; i += 4) {
						if (n0 + i >= g.N) break;
						float4 r = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
						if (g.epi == GEPI_RESID) {
							const float4 x = *reinterpret_cast<const float4*>(o + i);
							r.x += x.x; r.y += x.y; r.z += x.z; r.w += x.w; // infer.cpp:450-452, :492-494
						}
						*reinterpret_cast<float4*>(o + i) = r;
					}
				}
			}
			tc_fence_before();
			__syncwarp();
			if (lane == 0) mb_arrive(&tempty[acc]);
			acc ^= 1;
			if (acc == 0) acc_phase ^= 1;
		}
	}
	tc_fence_before();
	__syncthreads();
	if (warp == 1) {
		tc_fence_after();
		tmem_dealloc(tmem_base, 512);
	}
}

// ------------------------------------------------------------------------------------------------------------------
// row-wise kernels
// ------------------------------------------------------------------------------------------------------------------
// _copy_embedding (infer.cpp:553-602) for T tokens
__global__ void embed_rows_kernel(int type, const uint8_t* __restrict__ table, size_t row_bytes, int dim, const int* __restrict__ tokens, int T,
                                  float* __restrict__ x) {
	const size_t total = (size_t) T * dim;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int m = (int) (i / dim), j = (int) (i % dim);
		x[i] = decode_disk_elem(type, table + (size_t) tokens[m] * row_bytes, (size_t) j);
	}
}

// {cos, sin}(pos * freq_j) for every row and rotation pair: the very expression rope_pair (matvec.cuh) evaluates per token
__global__ void rope_table_kernel(const float* __restrict__ freq, int half_dim, int T, int pos0, float2* __restrict__ cs) {
	const int total = T * half_dim;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
		const int m = i / half_dim, j = i % half_dim;
		const float val = (float) (pos0 + m) * freq[j];
		float sn, cn;
		sincosf(val, &sn, &cn);
		cs[i] = make_float2(cn, sn);
	}
}

// rmsnorm (infer.cpp:224-236) of each row, result as an A-tile operand.  One 128-thread CTA per row: the row stays in registers
// (up to 8 chunks of 8 floats per thread = 8192 elements; longer rows re-read), the norm weights are requested before the
// block reduction so both loads overlap.
__global__ void __launch_bounds__(128) rmsnorm_rows_kernel(const float* __restrict__ x, int T, int dim, const uint8_t* __restrict__ w, int wtype, float eps,
                                                           ATiles o) {
	__shared__ float red[4];
	constexpr int MAXC = 8;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (int m = blockIdx.x; m < T; m += gridDim.x) {
		const float* xr = x + (size_t) m * dim;
		float4 buf[MAXC][2];
		float ss = 0.f;
#pragma unroll
		for (int c = 0; c < MAXC; c++) {
			const int j = threadIdx.x * 8 + c * 1024;
			if (j < dim) {
				buf[c][0] = *reinterpret_cast<const float4*>(xr + j);
				buf[c][1] = *reinterpret_cast<const float4*>(xr + j + 4);
			}
		}
#pragma unroll
		for (int c = 0; c < MAXC; c++) {
			const int j = threadIdx.x * 8 + c * 1024;
			if (j < dim) {
				const float4 a = buf[c][0], b = buf[c][1];
				ss += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w + b.x * b.x + b.y * b.y + b.z * b.z + b.w * b.w;
			}
		}
		for (int j = threadIdx.x * 8 + MAXC * 1024; j < dim; j += 1024) {
			const float4 a = *reinterpret_cast<const float4*>(xr + j), b = *reinterpret_cast<const float4*>(xr + j + 4);
			ss += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w + b.x * b.x + b.y * b.y + b.z * b.z + b.w * b.w;
		}
		ss = warp_sum(ss);
		__syncthreads(); // red[] of the previous row has been read by everyone
		if (lane == 0) red[warp] = ss;
		__syncthreads();
		const float tot = red[0] + red[1] + red[2] + red[3];
		const float scale = 1.0f / sqrtf(tot / (float) dim + eps);
		auto emit = [&](int j, const float4& a, const float4& b) {
			const float xv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
			float gw[8];
			if (wtype == XALM_F32) {
				const float4 g0 = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(w) + j);
				const float4 g1 = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(w) + j + 4);
				gw[0] = g0.x; gw[1] = g0.y; gw[2] = g0.z; gw[3] = g0.w; gw[4] = g1.x; gw[5] = g1.y; gw[6] = g1.z; gw[7] = g1.w;
			} else {
				const uint4 gq = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(w) + j);
				const uint32_t u[4] = {gq.x, gq.y, gq.z, gq.w};
#pragma unroll
				for (int i = 0; i < 4; i++) { gw[2 * i] = __uint_as_float(u[i] << 16); gw[2 * i + 1] = __uint_as_float(u[i] & 0xFFFF0000u); }
			}
			float v[8];
#pragma unroll
			for (int i = 0; i < 8; i++) v[i] = xv[i] * scale * gw[i]; // infer.cpp:233-235
			store_a8(o, m, j, v);
		};
#pragma unroll
		for (int c = 0; c < MAXC; c++) {
			const int j = threadIdx.x * 8 + c * 1024;
			if (j < dim) emit(j, buf[c][0], buf[c][1]);
		}
		for (int j = threadIdx.x * 8 + MAXC * 1024; j < dim; j += 1024)
			emit(j, *reinterpret_cast<const float4*>(xr + j), *reinterpret_cast<const float4*>(xr + j + 4));
	}
}

// Sampler::sample_prob (sampler.cpp:18-33) per row: softmax(logits)[target], the FLT_MIN-seeded max included
__global__ void target_prob_kernel(const float* __restrict__ logits, int vocab, const int* __restrict__ targets, float* __restrict__ probs) {
	__shared__ float red[32];
	const float* l = logits + (size_t) blockIdx.x * vocab;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
	float mx = FLT_MIN;
	for (int i = threadIdx.x; i < vocab; i += blockDim.x) mx = fmaxf(mx, l[i]);
	mx = warp_max(mx);
	if (lane == 0) red[warp] = mx;
	__syncthreads();
	mx = red[0];
	for (int i = 1; i < nw; i++) mx = fmaxf(mx, red[i]);
	__syncthreads();
	float sum = 0.f;
	for (int i = threadIdx.x; i < vocab; i += blockDim.x) sum += expf(l[i] - mx);
	sum = warp_sum(sum);
	if (lane == 0) red[warp] = sum;
	__syncthreads();
	if (threadIdx.x == 0) {
		float tot = 0.f;
		for (int i = 0; i < nw; i++) tot += red[i];
		probs[blockIdx.x] = expf(l[targets[blockIdx.x]] - mx) / tot;
	}
}

// ------------------------------------------------------------------------------------------------------------------
// causal attention over the fp16 KV cache for a block of 64 query rows of one head (attn + softmax, infer.cpp:325-359,
// 280-297, for T rows at once).  Flash-style: S = Q K^T and O += P V on mma.sync m16n8k16 tiles (fp16 in, fp32 out),
// online softmax in fp32 with expf.  Query row i (position pos0+i) sees cache rows [0, pos0+i].
// Window mode (win > 0, past the context window): k/v point at a linear staging copy of the ring, query row i sees only the
// band of rows (pos0+i-win, pos0+i], plus two attention-sink keys of its own (sink_k row i) scored in fp32; the sink scores
// seed the running maximum and enter the sum and the output at the end.
// Not a tcgen05 kernel: attention is ~7 % of the prefill flops at 4k; the GEMMs above are where the tensor time goes.
// ------------------------------------------------------------------------------------------------------------------
struct AttnPArgs {
	const __half* q;       // (T, q_dim)
	const __half* q_lo;    // rounding residual of q (PRECISE), or nullptr
	const __half* k_cache; // (max_seq_len, kv_dim)
	const __half* v_cache;
	ATiles o;              // xb2
	int T, pos0, q_dim, kv_dim, n_heads, n_kv_heads, n_qt;
	int win;               // window mode: keys per query in the band; 0 = linear (causal over [0, pos0+i])
	const __half* sink_k;  // window mode: (T, 2, kv_dim) the sink keys as query row i sees them
	const __half* sink_v;  // window mode: (2, kv_dim) the sink values
};

// window mode: the two sink scores of query row `row`, q.k in fp32 over head_dim from the (hi + lo) q held in global memory,
// split over the 4 lanes of a quad (each lane: HD/4 elements), reduced over the quad
template <int HD>
__device__ __forceinline__ void sink_scores_quad(const AttnPArgs& a, int row, int h, int kvh, int lane, float (&sc)[2]) {
	const int r = min(row, a.T - 1);
	const __half* qh = a.q + (size_t) r * a.q_dim + h * HD;
	const __half* ql = a.q_lo ? a.q_lo + (size_t) r * a.q_dim + h * HD : nullptr;
#pragma unroll
	for (int s = 0; s < 2; s++) {
		const __half* kp = a.sink_k + ((size_t) r * 2 + s) * a.kv_dim + kvh * HD;
		float acc = 0.f;
		for (int d = (lane & 3) * (HD / 4); d < (lane & 3) * (HD / 4) + HD / 4; d++) {
			const float qv = __half2float(qh[d]) + (ql ? __half2float(ql[d]) : 0.f);
			acc = fmaf(qv, __half2float(kp[d]), acc);
		}
		acc += __shfl_xor_sync(0xffffffffu, acc, 1);
		acc += __shfl_xor_sync(0xffffffffu, acc, 2);
		sc[s] = acc;
	}
}

__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t saddr) {
	asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldsm4_t(uint32_t (&r)[4], uint32_t saddr) {
	asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
	asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
	             : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
	             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g, bool valid) {
	const int sz = valid ? 16 : 0; // src-size 0 -> zero fill
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(sz) : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
	const __half2 h = __floats2half2_rn(a, b);
	return *reinterpret_cast<const uint32_t*>(&h);
}

// PRECISE: q and the softmax probabilities enter the tensor cores as hi+lo fp16 pairs (two MMAs each) — with the split GEMMs
// this keeps the whole prefill at fp32-grade operand precision (K and V are fp16 in the reference too).
template <int HD, bool PRECISE>
__global__ void __launch_bounds__(128) attn_prefill_kernel(const AttnPArgs a) {
	constexpr int BQ = 64, BKV = 64;
	constexpr int CPR = HD / 8;         // 16-byte chunks per row
	constexpr int ROWB = HD * 2;        // bytes per row
	extern __shared__ __align__(128) uint8_t sm[];
	uint8_t* sQ = sm;                   // [1 or 2][BQ][HD]
	uint8_t* sK = sQ + (PRECISE ? 2 : 1) * BQ * ROWB; // [2][BKV][HD]
	uint8_t* sV = sK + 2 * BKV * ROWB;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int qt = a.n_qt - 1 - (int) blockIdx.x; // longest (latest) query tiles first
	const int h = blockIdx.y;
	const int kvh = h / (a.n_heads / a.n_kv_heads);
	const int q0 = qt * BQ;
	const int q_last = min(q0 + BQ, a.T) - 1;
	const int kv_total = a.pos0 + q_last + 1;  // cache rows any row of this tile may see
	const int n_kb = (kv_total + BKV - 1) / BKV;
	const int kb0 = a.win ? max(0, a.pos0 + q0 - a.win + 1) / BKV : 0; // window mode: blocks wholly below the band are skipped
	// chunk (r, c) lives at r*ROWB + ((c ^ (r & 7)) * 16): conflict-free for ldmatrix (8 rows x 16 bytes per phase)
	auto soff = [](int r, int c) { return (uint32_t) (r * ROWB + ((c ^ (r & 7)) << 4)); };

	// ---- async loads: Q once, K/V blocks double-buffered ----
	for (int i = threadIdx.x; i < BQ * CPR; i += 128) {
		const int r = i / CPR, c = i % CPR;
		const bool ok = q0 + r < a.T;
		cp_async16(s_u32(sQ) + soff(r, c), a.q + (size_t) (ok ? q0 + r : 0) * a.q_dim + h * HD + c * 8, ok);
		if (PRECISE) cp_async16(s_u32(sQ) + BQ * ROWB + soff(r, c), a.q_lo + (size_t) (ok ? q0 + r : 0) * a.q_dim + h * HD + c * 8, ok);
	}
	auto load_kv = [&](int kb, int buf) {
		for (int i = threadIdx.x; i < BKV * CPR; i += 128) {
			const int r = i / CPR, c = i % CPR;
			const int key = kb * BKV + r;
			const bool ok = key < kv_total;
			const size_t g = (size_t) (ok ? key : 0) * a.kv_dim + kvh * HD + c * 8;
			cp_async16(s_u32(sK) + buf * BKV * ROWB + soff(r, c), a.k_cache + g, ok);
			cp_async16(s_u32(sV) + buf * BKV * ROWB + soff(r, c), a.v_cache + g, ok);
		}
	};
	load_kv(kb0, 0);
	asm volatile("cp.async.commit_group;" ::: "memory");

	float o_acc[HD / 8][4];
#pragma unroll
	for (int i = 0; i < HD / 8; i++)
#pragma unroll
		for (int j = 0; j < 4; j++) o_acc[i][j] = 0.f;
	float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
	uint32_t qf[HD / 16][4];
	uint32_t qlf[PRECISE ? HD / 16 : 1][4];
	const float scale = 1.0f / sqrtf((float) HD);
	const int row_a = q0 + warp * 16 + (lane >> 2); // this thread's two query rows: row_a and row_a + 8
	bool q_loaded = false;
	float sink_s[2][2]; // [row_a, row_a + 8][sink], scaled
	if (a.win) {
#pragma unroll
		for (int r = 0; r < 2; r++) {
			sink_scores_quad<HD>(a, row_a + 8 * r, h, kvh, lane, sink_s[r]);
			sink_s[r][0] *= scale; sink_s[r][1] *= scale;
			m_run[r] = fmaxf(sink_s[r][0], sink_s[r][1]); // every row has a finite maximum even where a block masks all its keys
		}
	}

	for (int kb = kb0; kb < n_kb; kb++) {
		const int buf = (kb - kb0) & 1;
		if (kb + 1 < n_kb) load_kv(kb + 1, buf ^ 1);
		asm volatile("cp.async.commit_group;" ::: "memory");
		asm volatile("cp.async.wait_group 1;" ::: "memory");
		__syncthreads();
		if (!q_loaded) {
#pragma unroll
			for (int ks = 0; ks < HD / 16; ks++) {
				ldsm4(qf[ks], s_u32(sQ) + soff(warp * 16 + (lane & 15), ks * 2 + (lane >> 4)));
				if (PRECISE) ldsm4(qlf[ks], s_u32(sQ) + BQ * ROWB + soff(warp * 16 + (lane & 15), ks * 2 + (lane >> 4)));
			}
			q_loaded = true;
		}
		// ---- S = Q K^T (16 query rows x 64 keys per warp) ----
		float s[BKV / 8][4];
#pragma unroll
		for (int i = 0; i < BKV / 8; i++)
#pragma unroll
			for (int j = 0; j < 4; j++) s[i][j] = 0.f;
		const uint32_t kbase = s_u32(sK) + buf * BKV * ROWB;
#pragma unroll
		for (int ks = 0; ks < HD / 16; ks++) {
#pragma unroll
			for (int nb = 0; nb < BKV / 16; nb++) {
				uint32_t kf[4];
				ldsm4(kf, kbase + soff(nb * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 2 + ((lane >> 3) & 1)));
				mma16816(s[2 * nb], qf[ks], kf[0], kf[1]);
				mma16816(s[2 * nb + 1], qf[ks], kf[2], kf[3]);
				if (PRECISE) {
					mma16816(s[2 * nb], qlf[ks], kf[0], kf[1]);
					mma16816(s[2 * nb + 1], qlf[ks], kf[2], kf[3]);
				}
			}
		}
		// ---- scale, causal mask, online softmax ----
		const bool need_mask = kb * BKV + BKV - 1 > a.pos0 + q0 + warp * 16  // some key of this block is beyond the warp's first row
		                    || (a.win && kb * BKV < a.pos0 + q0 + warp * 16 + 15 - a.win + 1); // or below the band of its last row
		float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
		for (int i = 0; i < BKV / 8; i++) {
#pragma unroll
			for (int j = 0; j < 4; j++) {
				float v = s[i][j] * scale;
				if (need_mask) {
					const int key = kb * BKV + i * 8 + 2 * (lane & 3) + (j & 1);
					const int row = row_a + (j >> 1) * 8;
					if (key > a.pos0 + row || (a.win && key <= a.pos0 + row - a.win)) v = -INFINITY;
				}
				s[i][j] = v;
				mx[j >> 1] = fmaxf(mx[j >> 1], v);
			}
		}
		float corr[2];
#pragma unroll
		for (int r = 0; r < 2; r++) {
			mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
			mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
			const float m_new = fmaxf(m_run[r], mx[r]);
			corr[r] = expf(m_run[r] - m_new); // first block: exp(-inf) = 0
			m_run[r] = m_new;
		}
		float rs[2] = {0.f, 0.f};
#pragma unroll
		for (int i = 0; i < BKV / 8; i++) {
#pragma unroll
			for (int j = 0; j < 4; j++) {
				const float p = expf(s[i][j] - m_run[j >> 1]);
				s[i][j] = p;
				rs[j >> 1] += p;
			}
		}
#pragma unroll
		for (int r = 0; r < 2; r++) l_run[r] = l_run[r] * corr[r] + rs[r]; // per-thread partial row sums, reduced over the quad at the end
#pragma unroll
		for (int i = 0; i < HD / 8; i++) {
			o_acc[i][0] *= corr[0]; o_acc[i][1] *= corr[0];
			o_acc[i][2] *= corr[1]; o_acc[i][3] *= corr[1];
		}
		// ---- O += P V ----
		const uint32_t vbase = s_u32(sV) + buf * BKV * ROWB;
#pragma unroll
		for (int kk = 0; kk < BKV / 16; kk++) {
			uint32_t pf[4], pl[4];
#pragma unroll
			for (int f = 0; f < 4; f++) {
				const float p0 = s[2 * kk + (f >> 1)][2 * (f & 1)], p1 = s[2 * kk + (f >> 1)][2 * (f & 1) + 1];
				const __half2 hh = __floats2half2_rn(p0, p1);
				pf[f] = *reinterpret_cast<const uint32_t*>(&hh);
				if (PRECISE) {
					const float2 back = __half22float2(hh);
					pl[f] = pack_h2(p0 - back.x, p1 - back.y);
				}
			}
#pragma unroll
			for (int nb = 0; nb < HD / 16; nb++) {
				uint32_t vf[4];
				ldsm4_t(vf, vbase + soff(kk * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), nb * 2 + (lane >> 4)));
				mma16816(o_acc[2 * nb], pf, vf[0], vf[1]);
				mma16816(o_acc[2 * nb + 1], pf, vf[2], vf[3]);
				if (PRECISE) {
					mma16816(o_acc[2 * nb], pl, vf[0], vf[1]);
					mma16816(o_acc[2 * nb + 1], pl, vf[2], vf[3]);
				}
			}
		}
		__syncthreads(); // everyone is done with `buf` before the next iteration's prefetch overwrites it
	}
	// ---- normalise and store as an A-tile operand (xb2) ----
#pragma unroll
	for (int r = 0; r < 2; r++) {
		l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
		l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
	}
	float sink_p[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
	if (a.win) {
#pragma unroll
		for (int r = 0; r < 2; r++) {
			sink_p[r][0] = expf(sink_s[r][0] - m_run[r]);
			sink_p[r][1] = expf(sink_s[r][1] - m_run[r]);
			l_run[r] += sink_p[r][0] + sink_p[r][1];
		}
	}
#pragma unroll
	for (int r = 0; r < 2; r++) {
		const int row = row_a + r * 8;
		if (row >= a.T) continue;
		const float inv = 1.0f / l_run[r];
#pragma unroll
		for (int i = 0; i < HD / 8; i++) {
			float o0 = o_acc[i][2 * r], o1 = o_acc[i][2 * r + 1];
			if (a.win) {
				const int d = kvh * HD + i * 8 + 2 * (lane & 3);
				const float2 v0s = __half22float2(*reinterpret_cast<const __half2*>(a.sink_v + d));
				const float2 v1s = __half22float2(*reinterpret_cast<const __half2*>(a.sink_v + a.kv_dim + d));
				o0 += sink_p[r][0] * v0s.x + sink_p[r][1] * v1s.x;
				o1 += sink_p[r][0] * v0s.y + sink_p[r][1] * v1s.y;
			}
			const float v0 = o0 * inv, v1 = o1 * inv;
			const int col = h * HD + i * 8 + 2 * (lane & 3);
			const size_t off = a_off(row, col, a.o.KT);
			const __half2 hh = __floats2half2_rn(v0, v1);
			*reinterpret_cast<__half2*>(a.o.hi + off) = hh;
			if (a.o.lo) {
				const float2 f = __half22float2(hh);
				*reinterpret_cast<__half2*>(a.o.lo + off) = __floats2half2_rn(v0 - f.x, v1 - f.y);
			}
		}
	}
}

// ------------------------------------------------------------------------------------------------------------------
// causal attention on tcgen05 (head_dim 128): S = Q K^T and O_blk = P V as UMMA 128x128x16 tiles with accumulators in TMEM.
//   Q operand   tiles written by the QKV epilogue: (head, 128-row block, hd half) -> 128 rows x 64
//   K operand   tiles (kv head, 128-key block, hd half) -> 128 keys x 64            } retile_kv_kernel, once per layer, from the
//   V^T operand tiles (kv head, 128-key block, key half) -> 128 hd rows x 64 keys   } fp16 cache rows [0, pos0 + T)
// One CTA = 128 query rows of one head.  warp 0: bulk-copy producer (Q once; one K slot and one V slot — K and V are needed
// at different times, so single slots already overlap load and use).  warp 1: MMA issuer; QK of block j+1 is issued before
// it waits for P of block j (S is double-buffered in TMEM).  warps 2-5: softmax, thread = query row: two passes over S in
// TMEM (row max, then exp), P as fp16 (hi, lo) into a shared-memory operand tile, running (max, sum) and the fp32 output
// row in registers; O_blk comes back from TMEM one block later and is folded in with the rescale.
// Window mode (win > 0): the tiles hold a linear staging copy of the ring, query row i sees the band (pos0+i-win, pos0+i] —
// key blocks wholly below a tile's band are not loaded — plus two sink keys of its own whose fp32 scores seed the running
// maximum and are added to the sum and the output row at the end.
// ------------------------------------------------------------------------------------------------------------------
struct AttnTcArgs {
	const uint8_t* qt_hi;
	const uint8_t* qt_lo;
	const uint8_t* kt;   // K tiles
	const uint8_t* vt;   // V^T tiles
	ATiles o;            // xb2
	int T, pos0, n_heads, n_kv_heads, n_qb, n_kb_total;
	int win;              // window mode: keys per query in the band; 0 = linear
	const __half* sink_k; // window mode: (T, 2, kv_dim) the sink keys as query row i sees them
	const __half* sink_v; // window mode: (2, kv_dim)
	int kv_dim;
	int dbg; // timing knock-outs (XALM_ATTN_DBG, results are then meaningless): 1 = no QK MMAs, 2 = no PV MMAs, 4 = no softmax math / P stores
};

// cache rows -> K tiles and V^T tiles.  grid (64-key blocks, kv heads), 256 threads.
__global__ void __launch_bounds__(256) retile_kv_kernel(const __half* __restrict__ k_cache, const __half* __restrict__ v_cache, int kv_dim,
                                                        int kv_total, int n_kb_total, uint8_t* __restrict__ kt, uint8_t* __restrict__ vt) {
	__shared__ __align__(16) __half sv[64][136];
	const int kb64 = blockIdx.x, kvh = blockIdx.y;
	const int key0 = kb64 * 64;
	const int kb = kb64 >> 1, half = kb64 & 1; // 128-key block and which half of it
	// K: 64 keys x 128 hd -> rows [64*half, 64*half+64) of tiles (kvh, kb, 0) and (kvh, kb, 1)
	uint8_t* ktile = kt + ((size_t) (kvh * n_kb_total + kb) * 2) * A_TILE_BYTES;
	for (int i = threadIdx.x; i < 64 * 16; i += 256) {
		const int r = i >> 4, c = i & 15; // key row, 16-byte chunk of the 128 hd values
		const int key = key0 + r;
		uint4 kvv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
		if (key < kv_total) {
			kvv = *reinterpret_cast<const uint4*>(k_cache + (size_t) key * kv_dim + kvh * 128 + c * 8);
			vv = *reinterpret_cast<const uint4*>(v_cache + (size_t) key * kv_dim + kvh * 128 + c * 8);
		}
		*reinterpret_cast<uint4*>(ktile + (size_t) (c >> 3) * A_TILE_BYTES + tile_inner_off(half * 64 + r, (c & 7) * 8)) = kvv;
		*reinterpret_cast<uint4*>(&sv[r][c * 8]) = vv;
	}
	__syncthreads();
	// V^T: tile (kvh, kb, half): row = hd d, columns = these 64 keys
	uint8_t* vtile = vt + ((size_t) (kvh * n_kb_total + kb) * 2 + half) * A_TILE_BYTES;
	for (int i = threadIdx.x; i < 128 * 8; i += 256) {
		const int d = i & 127, c = i >> 7; // chunk c = keys 8c .. 8c+7
		__half h[8];
#pragma unroll
		for (int j = 0; j < 8; j++) h[j] = sv[c * 8 + j][d];
		*reinterpret_cast<uint4*>(vtile + tile_inner_off(d, c * 8)) = *reinterpret_cast<const uint4*>(h);
	}
}

constexpr int ATT_THREADS = 192;
constexpr int ATT_BKV = 64; // keys per block
template <bool PRECISE>
struct AttnTcCfg {
	static constexpr int NP = PRECISE ? 2 : 1;                 // operand planes for Q and P
	static constexpr int NKV = PRECISE ? 3 : 4;                // K / V ring depth: a block's tiles take ~1.5 us to arrive from L2 and are consumed in
	                                                           // ~0.3 us, so the loads must run several blocks ahead (ncu: with one slot the softmax
	                                                           // warps sat on s_full — the MMA thread was waiting for K — 22 % of all samples)
	static constexpr int Q_BYTES = NP * 2 * A_TILE_BYTES;      // 128 rows x 128 hd
	static constexpr int P_TILE = A_TILE_BYTES;                // 128 rows x 64 keys, one plane
	static constexpr int P_BYTES = 2 * NP * P_TILE;            // double-buffered
	static constexpr int KV_SLOT = A_TILE_BYTES;               // 64 keys x 128 hd (K, two 8 KB halves) or 128 hd x 64 keys (V^T)
	static constexpr size_t SMEM = Q_BYTES + P_BYTES + 2 * NKV * KV_SLOT + 1024 + 256;
};

template <bool PRECISE>
__global__ void __launch_bounds__(ATT_THREADS, 1) attn_tc_kernel(const AttnTcArgs a) {
	using Cfg = AttnTcCfg<PRECISE>;
	constexpr int NP = Cfg::NP, NKV = Cfg::NKV;
	extern __shared__ uint8_t smem_raw[];
	const uint32_t raw_s = s_u32(smem_raw);
	uint8_t* smem = smem_raw + (((raw_s + 1023u) & ~1023u) - raw_s);
	uint8_t* sQ = smem;
	uint8_t* sP = sQ + Cfg::Q_BYTES;            // [2][NP][128 x 64]
	uint8_t* sK = sP + Cfg::P_BYTES;            // [NKV][2 hd halves][64 keys x 64]
	uint8_t* sV = sK + NKV * Cfg::KV_SLOT;      // [NKV][128 hd x 64 keys]
	uint64_t* bars = reinterpret_cast<uint64_t*>(sV + NKV * Cfg::KV_SLOT);
	uint64_t* q_full = bars;          // tx
	uint64_t* k_full = bars + 1;      // [4] tx
	uint64_t* k_empty = bars + 5;     // [4] commit
	uint64_t* v_full = bars + 9;      // [4] tx
	uint64_t* v_empty = bars + 13;    // [4] commit
	uint64_t* s_full = bars + 17;     // [4] commit
	uint64_t* s_empty = bars + 21;    // [4] 4 softmax warps
	uint64_t* p_full = bars + 25;     // [2] 4 softmax warps
	uint64_t* o_full = bars + 27;     // [2] commit (alternating by block parity, so a waiter is never two phases behind)
	uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 29);
	constexpr int LA = NKV - 1;       // the scores of LA blocks ahead are already in flight on the tensor pipe (S ring of 4 in TMEM)

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	// CTAs are dispatched in linear order (x fastest): make that order longest-first over the WHOLE launch — all heads' last
	// query block, then all heads' second-to-last, ... — so the causal tail is made of the shortest tiles, not of one head's longest
	const int lin = (int) (blockIdx.y * gridDim.x + blockIdx.x);
	const int qb = a.n_qb - 1 - lin / a.n_heads;
	const int h = lin % a.n_heads;
	const int kvh = h / (a.n_heads / a.n_kv_heads);
	const int q0 = qb * 128;
	const int q_last = min(q0 + 128, a.T) - 1;
	const int n_kb = (a.pos0 + q_last) / ATT_BKV + 1; // 64-key blocks any row of this tile sees
	const int kb0 = a.win ? max(0, a.pos0 + q0 - a.win + 1) / ATT_BKV : 0; // window mode: first block inside the tile's band
	const int n_it = n_kb - kb0;                       // blocks this tile visits; the rings below count visits, not block indices

	if (threadIdx.x == 0) {
		mb_init(q_full, 1);
		for (int i = 0; i < 4; i++) {
			mb_init(&k_full[i], 1); mb_init(&k_empty[i], 1); mb_init(&v_full[i], 1); mb_init(&v_empty[i], 1);
			mb_init(&s_full[i], 1); mb_init(&s_empty[i], 4);
		}
		for (int i = 0; i < 2; i++) { mb_init(&p_full[i], 4); mb_init(&o_full[i], 1); }
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	if (warp == 1) tmem_alloc(tmem_slot, 512);
	tc_fence_before();
	__syncthreads();
	tc_fence_after();
	const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
	const uint32_t TM_S0 = tmem_base, TM_O = tmem_base + 256; // S[j & 3] at columns 64 * (j & 3), O at 256

	if (warp == 0) {
		if (lane == 0) {
			const size_t qoff = ((size_t) (h * a.n_qb + qb) * 2) * A_TILE_BYTES;
			mb_expect_tx(q_full, Cfg::Q_BYTES);
			bulk_load(sQ, a.qt_hi + qoff, 2 * A_TILE_BYTES, q_full);
			if (PRECISE) bulk_load(sQ + 2 * A_TILE_BYTES, a.qt_lo + qoff, 2 * A_TILE_BYTES, q_full);
			for (int it = 0; it < n_it; it++) {
				const int j = kb0 + it;
				const int slot = it % NKV, use = it / NKV; // use-th fill of this slot
				// the retiled cache holds 128-key tiles; block j is rows [64 (j & 1), +64) of K tile (kvh, j / 2, hd half) — a contiguous
				// 8 KB run of whole 8-row atoms — and V^T tile (kvh, j / 2, j & 1)
				const uint8_t* ksrc = a.kt + ((size_t) (kvh * a.n_kb_total + (j >> 1)) * 2) * A_TILE_BYTES + (size_t) (j & 1) * (A_TILE_BYTES / 2);
				const uint8_t* vsrc = a.vt + ((size_t) (kvh * a.n_kb_total + (j >> 1)) * 2 + (j & 1)) * A_TILE_BYTES;
				mb_wait(&k_empty[slot], (use & 1) ^ 1);
				mb_expect_tx(&k_full[slot], Cfg::KV_SLOT);
				bulk_load(sK + slot * Cfg::KV_SLOT, ksrc, A_TILE_BYTES / 2, &k_full[slot]);
				bulk_load(sK + slot * Cfg::KV_SLOT + A_TILE_BYTES / 2, ksrc + A_TILE_BYTES, A_TILE_BYTES / 2, &k_full[slot]);
				mb_wait(&v_empty[slot], (use & 1) ^ 1);
				mb_expect_tx(&v_full[slot], Cfg::KV_SLOT);
				bulk_load(sV + slot * Cfg::KV_SLOT, vsrc, A_TILE_BYTES, &v_full[slot]);
			}
		}
		__syncwarp();
	} else if (warp == 1) {
		// The whole warp runs the control flow (barrier waits included) and ONE elected lane issues the MMAs and commits inside a
		// warp-uniform branch.  With the loop under `if (lane == 0)` instead, ncu showed ~210 instructions per 64-key block on this
		// single thread (ELECT / PLOP3 / R2UR around every UTCHMMA) — the MMA issuer, not the tensor pipe (28 % active) or the
		// softmax warps, was setting the pace.
		constexpr uint32_t idesc_s = instr_desc_f16(128, ATT_BKV); // S = Q K^T: 128 rows x 64 keys
		constexpr uint32_t idesc_o = instr_desc_f16(128, 128);     // O += P V: 128 rows x 128 hd
		const uint32_t q_s = s_u32(sQ), p_s = s_u32(sP), k_s = s_u32(sK), v_s = s_u32(sV);
		uint64_t qd[NP * 2], kd[NKV * 2], pd[2 * NP], vd[NKV]; // operand descriptors of every slot, built once
#pragma unroll
		for (int i = 0; i < NP * 2; i++) qd[i] = smem_desc(q_s + i * A_TILE_BYTES);
#pragma unroll
		for (int i = 0; i < NKV * 2; i++) kd[i] = smem_desc(k_s + (i >> 1) * Cfg::KV_SLOT + (i & 1) * (A_TILE_BYTES / 2));
#pragma unroll
		for (int i = 0; i < 2 * NP; i++) pd[i] = smem_desc(p_s + i * Cfg::P_TILE);
#pragma unroll
		for (int i = 0; i < NKV; i++) vd[i] = smem_desc(v_s + i * Cfg::KV_SLOT);
		auto issue_qk = [&](int j) {
			const int b = j & 3, slot = j % NKV, use = j / NKV;
			mb_wait(&k_full[slot], use & 1);
			mb_wait(&s_empty[b], ((j >> 2) & 1) ^ 1);
			tc_fence_after();
			if (elect_one()) {
				uint64_t kd0 = kd[0], kd1 = kd[1];
#pragma unroll
				for (int i = 1; i < NKV; i++)
					if (slot == i) { kd0 = kd[2 * i]; kd1 = kd[2 * i + 1]; }
				const uint32_t d = TM_S0 + ATT_BKV * b;
#pragma unroll
				for (int p = 0; p < NP; p++)
#pragma unroll
					for (int t = 0; t < 2; t++) // hd halves
#pragma unroll
						for (int k = 0; k < 4; k++)
							if (!(a.dbg & 1)) umma_f16(d, qd[p * 2 + t] + 2 * k, (t ? kd1 : kd0) + 2 * k, idesc_s, (uint32_t) ((p | t | k) != 0));
				umma_commit(&k_empty[slot]);
				umma_commit(&s_full[b]);
			}
			__syncwarp();
		};
		mb_wait(q_full, 0);
		for (int j = 0; j < LA && j < n_it; j++) issue_qk(j);
		for (int j = 0; j < n_it; j++) {
			if (j + LA < n_it) issue_qk(j + LA); // the tensor pipe works on later scores while the softmax warps turn these into P
			const int b = j & 1, slot = j % NKV, use = j / NKV;
			mb_wait(&p_full[b], (j >> 1) & 1);
			mb_wait(&v_full[slot], use & 1);
			tc_fence_after();
			if (elect_one()) {
				uint64_t vdd = vd[0];
#pragma unroll
				for (int i = 1; i < NKV; i++)
					if (slot == i) vdd = vd[i];
#pragma unroll
				for (int p = 0; p < NP; p++) {
					const uint64_t pdd = b ? pd[NP + p] : pd[p];
#pragma unroll
					for (int k = 0; k < 4; k++)
						if (!(a.dbg & 2)) umma_f16(TM_O, pdd + 2 * k, vdd + 2 * k, idesc_o, (uint32_t) ((j | p | k) != 0)); // O accumulates over all blocks
				}
				umma_commit(&v_empty[slot]);
				umma_commit(&o_full[b]);
			}
			__syncwarp();
		}
	} else {
		const int quad = warp & 3;
		const int r = quad * 32 + lane; // query row inside the tile = TMEM lane
		const int row = q0 + r;
		const uint32_t lane_addr = (uint32_t) (quad * 32) << 16;
		// softmax in the log2 domain on the RAW scores: p = 2^(s*c1 - m*c1), c1 = log2(e)/sqrt(head_dim) -> one FFMA + one MUFU per
		// element (ex2.approx: 2^-22 relative, far below the fp16 rounding of P even as a hi+lo pair)
		const float c1 = 1.4426950408889634f / sqrtf(128.0f);
		auto ex2 = [](float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; };
		// The output accumulates in TMEM (PV with accumulate); it is rescaled only when a row's maximum grows by more than TAU
		// (in natural-log units: exp(8) = 2981 still fits fp16 comfortably) over the maximum its probabilities are expressed against.
		const float TAU_RAW = 8.0f * sqrtf(128.0f);
		float m_run = -INFINITY, l_run = 0.f; // m_run: maximum of the raw scores
		float sink_s[2] = {-INFINITY, -INFINITY};
		if (a.win) { // q row r from the Q tiles in shared memory (hi + lo in the precise mode) . this row's sink keys, fp32
			mb_wait(q_full, 0);
			const int rr = min(row, a.T - 1);
#pragma unroll
			for (int s = 0; s < 2; s++) {
				const __half* kp = a.sink_k + ((size_t) rr * 2 + s) * a.kv_dim + kvh * 128;
				float acc = 0.f;
				for (int c8 = 0; c8 < 16; c8++) { // 8 hd values = one 16-byte chunk of a Q tile row
					const size_t off = (size_t) (c8 >> 3) * A_TILE_BYTES + tile_inner_off(r, (c8 & 7) * 8);
					const uint4 qh4 = *reinterpret_cast<const uint4*>(sQ + off);
					const uint4 k4 = *reinterpret_cast<const uint4*>(kp + c8 * 8);
					const __half* qh = reinterpret_cast<const __half*>(&qh4);
					const __half* kh = reinterpret_cast<const __half*>(&k4);
					uint4 ql4 = make_uint4(0, 0, 0, 0);
					if (PRECISE) ql4 = *reinterpret_cast<const uint4*>(sQ + 2 * A_TILE_BYTES + off);
					const __half* ql = reinterpret_cast<const __half*>(&ql4);
#pragma unroll
					for (int i = 0; i < 8; i++) acc = fmaf(__half2float(qh[i]) + (PRECISE ? __half2float(ql[i]) : 0.f), __half2float(kh[i]), acc);
				}
				sink_s[s] = acc;
			}
			m_run = fmaxf(sink_s[0], sink_s[1]); // finite for every row, even where a block masks all of its keys
		}
		for (int it = 0; it < n_it; it++) {
			const int j = kb0 + it;            // key block
			const int b = it & 1, sb = it & 3; // ring positions
			mb_wait(&s_full[sb], (it >> 2) & 1);
			tc_fence_after();
			const bool need_mask = j * ATT_BKV + ATT_BKV - 1 > a.pos0 + q0   // some key of this block is beyond the tile's first row
			                    || (a.win && j * ATT_BKV < a.pos0 + q_last - a.win + 1); // or below the band of its last row
			const int lim = a.pos0 + row - j * ATT_BKV;                      // keys with index (inside the block) > lim are masked
			const int lo = a.win ? lim - a.win + 1 : INT_MIN;                // window mode: and those < lo
			float sv[ATT_BKV];
			__syncwarp();
#pragma unroll
			for (int c = 0; c < ATT_BKV / 32; c++) tmem_ld32_issue(TM_S0 + lane_addr + ATT_BKV * sb + 32 * c, sv + 32 * c);
			tmem_wait_ld();
			float mx = -INFINITY;
			if (need_mask) {
#pragma unroll
				for (int i = 0; i < ATT_BKV; i++) {
					if (i > lim || i < lo) sv[i] = -INFINITY;
					mx = fmaxf(mx, sv[i]);
				}
			} else {
#pragma unroll
				for (int i = 0; i < ATT_BKV; i++) mx = fmaxf(mx, sv[i]);
			}
			// this P buffer was last read by the P V of block j-2: it must have completed (it has, long ago, in steady state)
			if (it >= 2) mb_wait(&o_full[b], ((it >> 1) - 1) & 1);
			const bool grow = mx > m_run + TAU_RAW;   // block 0: m_run = -inf -> true, but there is nothing to rescale yet
			if (it == 0) m_run = fmaxf(m_run, mx);    // (window mode: m_run holds the sink maximum)
			else if (__any_sync(0xffffffffu, grow)) {
				// rare: O must be quiescent, i.e. the P V of block j-1 (the last one issued) has completed
				mb_wait(&o_full[(it - 1) & 1], ((it - 1) >> 1) & 1);
				const float m_new = grow ? mx : m_run;
				const float corr = ex2((m_run - m_new) * c1); // 1 for the rows that keep their maximum
				tc_fence_after();
#pragma unroll
				for (int c = 0; c < 4; c++) {
					float v[32];
					tmem_ld32(TM_O + lane_addr + 32 * c, v);
#pragma unroll
					for (int i = 0; i < 32; i++) v[i] *= corr;
					tmem_st32(TM_O + lane_addr + 32 * c, v);
				}
				tmem_wait_st();
				l_run *= corr;
				m_run = m_new;
			}
			const float nm = -m_run * c1;
			// ---- probabilities -> fp16 operand tile (hi, lo), row sum ----
			uint8_t* pt = sP + (size_t) (b * NP) * Cfg::P_TILE;
			float rs = 0.f;
#pragma unroll
			for (int g8 = 0; g8 < ((a.dbg & 4) ? 0 : ATT_BKV / 8); g8++) { // 8 keys = one 16-byte chunk
				__half2 hh[4], ll[4];
#pragma unroll
				for (int i = 0; i < 4; i++) {
					const float p0 = ex2(fmaf(sv[8 * g8 + 2 * i], c1, nm)), p1 = ex2(fmaf(sv[8 * g8 + 2 * i + 1], c1, nm));
					rs += p0 + p1;
					hh[i] = __floats2half2_rn(p0, p1);
					if (PRECISE) {
						const float2 f = __half22float2(hh[i]);
						ll[i] = __floats2half2_rn(p0 - f.x, p1 - f.y);
					}
				}
				const size_t off = tile_inner_off(r, 8 * g8);
				*reinterpret_cast<uint4*>(pt + off) = *reinterpret_cast<const uint4*>(hh);
				if (PRECISE) *reinterpret_cast<uint4*>(pt + Cfg::P_TILE + off) = *reinterpret_cast<const uint4*>(ll);
			}
			l_run += rs;
			tc_fence_before();
			asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // generic-proxy writes of P -> visible to the MMA (async proxy)
			__syncwarp();
			if (lane == 0) {
				mb_arrive(&s_empty[sb]);
				mb_arrive(&p_full[b]);
			}
		}
		{ // the last P V (and with it every earlier one: MMAs complete in order)
			const int jl = n_it - 1;
			mb_wait(&o_full[jl & 1], (jl >> 1) & 1);
		}
		tc_fence_after();
		float sp0 = 0.f, sp1 = 0.f;
		if (a.win) {
			sp0 = ex2((sink_s[0] - m_run) * c1);
			sp1 = ex2((sink_s[1] - m_run) * c1);
			l_run += sp0 + sp1;
		}
		const float inv = 1.0f / l_run;
#pragma unroll
		for (int c = 0; c < 4; c++) {
			float v[32];
			tmem_ld32(TM_O + lane_addr + 32 * c, v);
			if (a.win) { // + the sinks' share of the output row
				const __half* v0 = a.sink_v + kvh * 128 + 32 * c;
				const __half* v1 = v0 + a.kv_dim;
#pragma unroll
				for (int i = 0; i < 32; i++) v[i] += sp0 * __half2float(v0[i]) + sp1 * __half2float(v1[i]);
			}
			if (row < a.T) {
#pragma unroll
				for (int g8 = 0; g8 < 4; g8++) {
					float out[8];
#pragma unroll
					for (int i = 0; i < 8; i++) out[i] = v[8 * g8 + i] * inv;
					store_a8(a.o, row, h * 128 + 32 * c + 8 * g8, out);
				}
			}
		}
	}
	tc_fence_before();
	__syncthreads();
	if (warp == 1) {
		tc_fence_after();
		tmem_dealloc(tmem_base, 512);
	}
}

// ------------------------------------------------------------------------------------------------------------------
// window mode (positions pos0 .. pos0+T-1, all >= max_seq_len): the KV cache is a ring, slot 2 + (p - 2) % S of S = max_seq_len - 2
// data slots after two attention sinks (infer.cpp:608-613).  The batch's own K/V rows overwrite ring rows that its earlier
// queries still need, so attention reads a linear staging copy instead: rows [0, S-1) = positions pos0-S+1 .. pos0-1
// (gathered from the ring before the QKV GEMM), rows [S-1, S-1+T) = the new rows (QKV epilogue).
// ------------------------------------------------------------------------------------------------------------------
__global__ void gather_ring_kernel(const __half* __restrict__ k_cache, const __half* __restrict__ v_cache, int kv_dim, int S, int pos0,
                                   __half* __restrict__ k_stage, __half* __restrict__ v_stage) {
	const int cpr = kv_dim / 8; // 16-byte chunks per row
	const size_t total = (size_t) (S - 1) * cpr;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int r = (int) (i / cpr), c = (int) (i % cpr);
		const int p = pos0 - S + 1 + r;  // >= 3: below the window its slot is p itself, which the same formula gives
		const size_t src = (size_t) (2 + (p - 2) % S) * kv_dim + c * 8, dst = (size_t) r * kv_dim + c * 8;
		*reinterpret_cast<uint4*>(k_stage + dst) = *reinterpret_cast<const uint4*>(k_cache + src);
		*reinterpret_cast<uint4*>(v_stage + dst) = *reinterpret_cast<const uint4*>(v_cache + src);
	}
}

// The sink keys (cache rows 0 and 1) as each query of the batch sees them: the token-at-a-time path re-rotates them by one
// position per token before that token's attention (rotate_sinks, matvec.cuh), so query i sees them i+1 rotations on from the
// state before the call.  One thread per rotation pair walks the T steps with the same expression, rounding through fp16 each
// step (bit-identical to T forwards); version i -> sink_k row i, the last one goes back to the cache.
__global__ void sink_versions_kernel(__half* __restrict__ k_cache, int kv_dim, int head_dim, const float* __restrict__ rope_freq, int T,
                                     __half* __restrict__ sink_k) {
	const int pairs = kv_dim / 2;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= 2 * pairs) return;
	const int r = i / pairs, p = i % pairs;
	__half2* kp = reinterpret_cast<__half2*>(k_cache + (size_t) r * kv_dim) + p;
	__half2 h = *kp;
	for (int t = 0; t < T; t++) {
		float2 v = __half22float2(h);
		rope_pair(v.x, v.y, (2 * p) % head_dim, 1, rope_freq);
		h = __floats2half2_rn(v.x, v.y);
		reinterpret_cast<__half2*>(sink_k + ((size_t) t * 2 + r) * kv_dim)[p] = h;
	}
	*kp = h;
}

// fp32 row-major (T, K) -> A tiles (op-level hook and tests)
__global__ void pack_a_kernel(const float* __restrict__ a, int T, int K, ATiles o) {
	const size_t total = (size_t) T * (K / 8);
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int m = (int) (i / (K / 8)), k0 = (int) (i % (K / 8)) * 8;
		float v[8];
#pragma unroll
		for (int j = 0; j < 8; j++) v[j] = a[(size_t) m * K + k0 + j];
		store_a8(o, m, k0, v);
	}
}

// tensor parallel: the all-gathered classifier shards (P, rows, vocab_l) -> (rows, P * vocab_l), the one-GPU layout
__global__ void unshard_logits_kernel(const float* __restrict__ shards, int P, int rows, int vocab_l, float* __restrict__ out) {
	const int q = vocab_l / 4; // float4 per shard row (vocab_l % 32 == 0)
	const size_t total = (size_t) P * rows * q;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int j = (int) (i % q);
		const size_t pr = i / q;
		const int r = (int) (pr % rows), p = (int) (pr / rows);
		reinterpret_cast<float4*>(out + (size_t) r * P * vocab_l + (size_t) p * vocab_l)[j] = reinterpret_cast<const float4*>(shards)[i];
	}
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
static int g_sms = 0;
static int sm_count() {
	if (!g_sms) {
		int dev = 0;
		cudaGetDevice(&dev);
		cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
		if (g_sms <= 0) g_sms = 148;
	}
	return g_sms;
}
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

struct DevBuf {
	uint8_t* p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes, bool zero, cudaStream_t s) {
		if (bytes <= cap) return XALM_OK;
		if (p) {
			XALM_CUDA_CHECK(cudaStreamSynchronize(s));
			XALM_CUDA_CHECK(cudaFree(p));
			p = nullptr; cap = 0;
		}
		XALM_CUDA_CHECK(cudaMalloc((void**) &p, bytes));
		cap = bytes;
		if (zero) XALM_CUDA_CHECK(cudaMemsetAsync(p, 0, bytes, s));
		return XALM_OK;
	}
	void release() {
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
	}
};

struct PrefillScratch {
	DevBuf x, xb_hi, xb_lo, xb2_hi, xb2_lo, hb_hi, hb_lo, q, q_lo, wt[2], wt_lo[2], logits, tokens, targets, probs, rope, qt_hi, qt_lo, kt, vt,
	    k_stage, v_stage, sink_k, // window mode
	    part, logits_tp;          // tensor parallel: this rank's partial sums of Wo / W2; the all-gathered classifier shards
	int logits_rows = 0;
	cudaStream_t side = nullptr;          // dequantises the NEXT GEMM's weights while the current GEMM runs
	cudaEvent_t ev_start = nullptr, ev_deq[2] = {nullptr, nullptr}, ev_gemm[2] = {nullptr, nullptr};
};

void prefill_free(PrefillScratch* s) {
	if (!s) return;
	DevBuf* all[] = {&s->x, &s->xb_hi, &s->xb_lo, &s->xb2_hi, &s->xb2_lo, &s->hb_hi, &s->hb_lo, &s->q, &s->q_lo, &s->wt[0], &s->wt[1],
	                 &s->wt_lo[0], &s->wt_lo[1], &s->logits, &s->tokens, &s->targets, &s->probs, &s->rope, &s->qt_hi, &s->qt_lo, &s->kt, &s->vt,
	                 &s->k_stage, &s->v_stage, &s->sink_k, &s->part, &s->logits_tp};
	for (DevBuf* b : all) b->release();
	if (s->side) cudaStreamDestroy(s->side);
	if (s->ev_start) cudaEventDestroy(s->ev_start);
	for (int i = 0; i < 2; i++) {
		if (s->ev_deq[i]) cudaEventDestroy(s->ev_deq[i]);
		if (s->ev_gemm[i]) cudaEventDestroy(s->ev_gemm[i]);
	}
	delete s;
}
const float* prefill_logits_dev(const PrefillScratch* s, int* rows) {
	if (rows) *rows = s ? s->logits_rows : 0;
	return s ? reinterpret_cast<const float*>(s->logits.p) : nullptr;
}

template <int NA, int NB>
static int launch_gemm_inst(const GemmArgs& g, int grid, cudaStream_t s) {
	static bool attr = false;
	if (!attr) {
		XALM_CUDA_CHECK(cudaFuncSetAttribute(gemm_tc_kernel<NA, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) GemmCfg<NA, NB>::SMEM));
		attr = true;
	}
	gemm_tc_kernel<NA, NB><<<grid, GEMM_THREADS, GemmCfg<NA, NB>::SMEM, s>>>(g);
	return XALM_OK;
}
static int launch_gemm(const GemmArgs& g, int na, int nb, cudaStream_t s) {
	const int tiles = g.MT * g.NT;
	if (tiles <= 0) return XALM_OK;
	const int grid = std::min(tiles, sm_count());
	if (na == 2 && nb == 2) XALM_TRY((launch_gemm_inst<2, 2>(g, grid, s)));
	else if (na == 2) XALM_TRY((launch_gemm_inst<2, 1>(g, grid, s)));
	else XALM_TRY((launch_gemm_inst<1, 1>(g, grid, s)));
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "gemm_tc launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// weights of `w` (rows [0, n_valid) or the GLU pairing) -> B tiles in `dst` (+ rounding residuals in dst_lo when not NULL)
static int launch_dequant_tiles(const WMat& w, bool glu, int glu_off, int n_valid, int K, int NT, int KT, uint8_t* dst, uint8_t* dst_lo,
                                cudaStream_t s) {
	const size_t chunks = (size_t) NT * KT * (B_TILE_BYTES / 16);
	const int grid = (int) std::min<size_t>((chunks + 255) / 256, (size_t) sm_count() * 16);
	// the common formats get a kernel with the type and layout folded in at compile time (2x the generic one's throughput)
#define XALM_DQ(TT, LU) dequant_tiles_kernel<TT, LU><<<grid, 256, 0, s>>>(w, glu ? 1 : 0, glu_off, n_valid, K, NT, KT, dst, dst_lo)
	if (w.type == XALM_Q8_0 && w.layout_frag) XALM_DQ(XALM_Q8_0, 2);
	else if (w.type == XALM_Q4_0 && w.layout_frag) XALM_DQ(XALM_Q4_0, 2);
	else if (w.type == XALM_Q8_0 && w.layout_units) XALM_DQ(XALM_Q8_0, 1);
	else if (w.type == XALM_Q4_0 && w.layout_units) XALM_DQ(XALM_Q4_0, 1);
	else if (w.type == XALM_F16) XALM_DQ(XALM_F16, 0);
	else if (w.type == XALM_BF16) XALM_DQ(XALM_BF16, 0);
	else if (w.type == XALM_F8_E4M3) XALM_DQ(XALM_F8_E4M3, 0);
	else XALM_DQ(-1, -1);
#undef XALM_DQ
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "dequant_tiles launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

static bool prefill_type_ok(int t) {
	TypeInfo ti;
	return type_info(t, &ti);
}

template <bool PRECISE>
static int launch_attn_tc(const AttnTcArgs& a, cudaStream_t s) {
	static bool attr = false;
	if (!attr) {
		XALM_CUDA_CHECK(cudaFuncSetAttribute(attn_tc_kernel<PRECISE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) AttnTcCfg<PRECISE>::SMEM));
		attr = true;
	}
	attn_tc_kernel<PRECISE><<<dim3(a.n_qb, a.n_heads), ATT_THREADS, AttnTcCfg<PRECISE>::SMEM, s>>>(a);
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "attn_tc launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

template <int HD, bool PRECISE>
static int launch_attn_p(const AttnPArgs& a, cudaStream_t s) {
	const size_t smem = (size_t) 64 * HD * 2 * (PRECISE ? 6 : 5);
	static bool attr = false;
	if (!attr) {
		XALM_CUDA_CHECK(cudaFuncSetAttribute(attn_prefill_kernel<HD, PRECISE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
		attr = true;
	}
	attn_prefill_kernel<HD, PRECISE><<<dim3(a.n_qt, a.n_heads), 128, smem, s>>>(a);
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "attn_prefill launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// Tensor parallel: every rank learns the worst status of the group (XALM_OK = 0, errors > 0) before anything touches a cache.  A
// scratch allocation can fail on one rank only; then every rank returns an error and none is left waiting in a collective.
static int agree_status(const PrefillModel& pm, int rc) {
	int v = rc;
	XALM_CUDA_CHECK(cudaMemcpyAsync(pm.status_dev, &v, sizeof v, cudaMemcpyHostToDevice, pm.stream));
	XALM_NCCL_CHECK(g_nccl.AllReduce(pm.status_dev, pm.status_dev, 1, ncclInt32, ncclMax, pm.comm, pm.stream));
	XALM_CUDA_CHECK(cudaMemcpyAsync(&v, pm.status_dev, sizeof v, cudaMemcpyDeviceToHost, pm.stream));
	XALM_CUDA_CHECK(cudaStreamSynchronize(pm.stream));
	if (v == XALM_OK || rc != XALM_OK) return rc; // a rank that failed keeps its own message
	return set_error(v, "prefill: another rank of the tensor-parallel group failed (status %d)", v);
}

int prefill_run(const PrefillModel& pm, PrefillScratch** scratch, const int* tokens, int n, int pos0, int want_logits, float* logits_host,
                const int* targets, float* probs_host, int split, int* n_launches, bool window) {
	const xalm_config& c = pm.c;
	if (n <= 0) return set_error(XALM_ERR_INVALID, "prefill: n = %d", n);
	if (!window && (pos0 < 0 || (long long) pos0 + n > c.max_seq_len))
		return set_error(XALM_ERR_INVALID,
		                 "prefill: positions [%d, %d) do not fit the %d-slot KV cache without wrapping (use xalm_cuda_prefill_window past it)", pos0,
		                 pos0 + n, c.max_seq_len);
	if (window && pos0 < c.max_seq_len)
		return set_error(XALM_ERR_INVALID, "prefill_window: pos0 %d is inside the %d-position window (use xalm_cuda_prefill below it)", pos0,
		                 c.max_seq_len);
	if (window && n > c.max_seq_len - 2)
		return set_error(XALM_ERR_INVALID, "prefill_window: n = %d exceeds the %d ring slots (split it into chunks of at most that many)", n,
		                 c.max_seq_len - 2);
	if (window && (long long) pos0 + n > INT_MAX) return set_error(XALM_ERR_INVALID, "prefill_window: positions overflow");
	if (c.head_dim != 64 && c.head_dim != 128) return set_error(XALM_ERR_UNSUPPORTED, "prefill: head_dim %d (64 or 128)", c.head_dim);
	if (c.dim % 16 || pm.hidden % 16 || pm.q_dim % 16 || pm.kv_dim % 16) return set_error(XALM_ERR_UNSUPPORTED, "prefill: dims must be multiples of 16");
	if (pm.tp_size > 1 && (!pm.comm || !pm.status_dev)) return set_error(XALM_ERR_STATE, "prefill: tensor-parallel model without a communicator");
	if (targets && want_logits != 2) return set_error(XALM_ERR_INVALID, "prefill: target probabilities need the logits of every position");
	if (want_logits < 0 || want_logits > 2) return set_error(XALM_ERR_INVALID, "prefill: want_logits = %d", want_logits);
	for (int i = 0; i < n; i++)
		if (tokens[i] < 0 || tokens[i] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "prefill: token %d out of range", tokens[i]);
	// everything that can be refused is refused HERE, before anything is enqueued: an error return must not leave half a pass in
	// flight on two streams and a partly overwritten KV cache
	if (targets)
		for (int i = 0; i < n; i++)
			if (targets[i] < 0 || targets[i] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "prefill: target %d out of range", targets[i]);
	for (const PrefillLayer& P : pm.layers)
		if (!prefill_type_ok(P.wqkv.type) || !prefill_type_ok(P.wo.type) || !prefill_type_ok(P.w13.type) || !prefill_type_ok(P.w2.type))
			return set_error(XALM_ERR_UNSUPPORTED, "prefill: weight type %d", P.wqkv.type);
	if (want_logits && !prefill_type_ok(pm.wcls.type)) return set_error(XALM_ERR_UNSUPPORTED, "prefill: weight type %d", pm.wcls.type);
	// split: 1 = fp16 x fp16; 2 = hi+lo activations; 3 = hi+lo activations AND weights AND attention operands (fp32-grade)
	const int na = split >= 2 ? 2 : 1;
	const bool precise = split >= 3;
	const bool tp = pm.tp_size > 1;
	cudaStream_t s = pm.stream;
	const int T = n, MT = cdiv(T, GB_M), Tp = MT * GB_M;
	const int KT_dim = cdiv(c.dim, GB_K), KT_q = cdiv(pm.q_dim, GB_K), KT_h = cdiv(pm.hidden, GB_K);
	const int n_qkv = pm.q_dim + 2 * pm.kv_dim;
	const int NT_qkv = cdiv(n_qkv, GB_N), NT_dim = cdiv(c.dim, GB_N), NT_glu = cdiv(pm.hidden, GB_N / 2), NT_cls = cdiv(pm.vocab, GB_N);
	// tensor parallel: the Wo / W2 partial sums are reduce-scattered in blocks of Tr / P rows of x (Tr = T rounded up to a multiple of
	// P); rows [T, Tr) carry values nothing reads
	const int Tr = cdiv(T, pm.tp_size) * pm.tp_size;
	// head_dim 128: attention on tcgen05 (attn_tc_kernel); otherwise the mma.sync kernel on row-major q
	const bool attn_tc = c.head_dim == 128 && getenv("XALM_ATTN_MMA_SYNC") == nullptr;
	// window mode: attention reads the staging copy, rows [0, S-1+T), as if it were a cache prefix of S-1 rows (pos0 of the kernels)
	const int S = c.max_seq_len - 2;
	const int attn_pos0 = window ? S - 1 : pos0;
	const int n_qb = MT, n_kb_total = cdiv(attn_pos0 + T, 128);
	size_t wt_tiles = std::max({(size_t) NT_qkv * KT_dim, (size_t) NT_dim * KT_q, (size_t) NT_glu * KT_dim, (size_t) NT_dim * KT_h});
	if (want_logits) wt_tiles = std::max(wt_tiles, (size_t) NT_cls * KT_dim);
	// want 1: only the last M tile goes through the classifier; its valid rows are stored, the last one is the answer
	const int logit_row0 = want_logits == 1 ? (MT - 1) * GB_M : 0;
	const int logit_rows = want_logits ? T - logit_row0 : 0;
	if (!*scratch) *scratch = new PrefillScratch();
	PrefillScratch& sc = **scratch;
	// ---- scratch (grown on demand; (re)allocation synchronises, steady state does not) ----
	auto grow = [&]() -> int {
		if (!sc.side) {
			XALM_CUDA_CHECK(cudaStreamCreateWithFlags(&sc.side, cudaStreamNonBlocking));
			XALM_CUDA_CHECK(cudaEventCreateWithFlags(&sc.ev_start, cudaEventDisableTiming));
			for (int i = 0; i < 2; i++) {
				XALM_CUDA_CHECK(cudaEventCreateWithFlags(&sc.ev_deq[i], cudaEventDisableTiming));
				XALM_CUDA_CHECK(cudaEventCreateWithFlags(&sc.ev_gemm[i], cudaEventDisableTiming));
			}
		}
		XALM_TRY(sc.x.ensure((size_t) std::max(Tp, Tr) * c.dim * 4, true, s));
		XALM_TRY(sc.xb_hi.ensure((size_t) MT * KT_dim * A_TILE_BYTES, true, s));
		XALM_TRY(sc.xb2_hi.ensure((size_t) MT * KT_q * A_TILE_BYTES, true, s));
		XALM_TRY(sc.hb_hi.ensure((size_t) MT * KT_h * A_TILE_BYTES, true, s));
		if (na == 2) {
			XALM_TRY(sc.xb_lo.ensure((size_t) MT * KT_dim * A_TILE_BYTES, true, s));
			XALM_TRY(sc.xb2_lo.ensure((size_t) MT * KT_q * A_TILE_BYTES, true, s));
			XALM_TRY(sc.hb_lo.ensure((size_t) MT * KT_h * A_TILE_BYTES, true, s));
		}
		if (window) {
			XALM_TRY(sc.k_stage.ensure((size_t) (S - 1 + T) * pm.kv_dim * 2, false, s));
			XALM_TRY(sc.v_stage.ensure((size_t) (S - 1 + T) * pm.kv_dim * 2, false, s));
			XALM_TRY(sc.sink_k.ensure((size_t) T * 2 * pm.kv_dim * 2, false, s));
		}
		if (attn_tc) {
			XALM_TRY(sc.qt_hi.ensure((size_t) pm.n_heads * n_qb * 2 * A_TILE_BYTES, true, s));
			if (precise) XALM_TRY(sc.qt_lo.ensure((size_t) pm.n_heads * n_qb * 2 * A_TILE_BYTES, true, s));
			XALM_TRY(sc.kt.ensure((size_t) pm.n_kv_heads * n_kb_total * 2 * A_TILE_BYTES, true, s)); // zeroed: tail keys of the last tile must stay finite
			XALM_TRY(sc.vt.ensure((size_t) pm.n_kv_heads * n_kb_total * 2 * A_TILE_BYTES, true, s));
		} else {
			XALM_TRY(sc.q.ensure((size_t) Tp * pm.q_dim * 2, true, s));
			if (precise) XALM_TRY(sc.q_lo.ensure((size_t) Tp * pm.q_dim * 2, true, s));
		}
		XALM_TRY(sc.rope.ensure((size_t) T * (c.head_dim / 2) * sizeof(float2), false, s));
		for (int i = 0; i < 2; i++) {
			XALM_TRY(sc.wt[i].ensure(wt_tiles * B_TILE_BYTES, false, s));
			if (precise) XALM_TRY(sc.wt_lo[i].ensure(wt_tiles * B_TILE_BYTES, false, s));
		}
		XALM_TRY(sc.tokens.ensure((size_t) T * 4, false, s));
		if (logit_rows) XALM_TRY(sc.logits.ensure((size_t) logit_rows * c.vocab_size * 4, false, s));
		if (want_logits && targets && probs_host) {
			XALM_TRY(sc.targets.ensure((size_t) T * 4, false, s));
			XALM_TRY(sc.probs.ensure((size_t) T * 4, false, s));
		}
		if (tp) {
			XALM_TRY(sc.part.ensure((size_t) Tr * c.dim * 4, true, s));
			if (logit_rows) XALM_TRY(sc.logits_tp.ensure((size_t) logit_rows * c.vocab_size * 4, false, s));
		}
		return XALM_OK;
	};
	int rc = grow();
	if (tp) rc = agree_status(pm, rc);
	if (rc != XALM_OK) return rc;
	sc.logits_rows = logit_rows;
	const bool timing = getenv("XALM_PREFILL_TIMING") != nullptr; // per-category CUDA-event timing, everything on one stream
	cudaStream_t ds = timing ? s : sc.side;
	int launches = tp ? 1 : 0; // the status vote
	struct Span { const char* what; cudaEvent_t a, b; };
	std::vector<Span> spans;
	auto t_begin = [&](const char* what) {
		if (!timing) return;
		Span sp{what, nullptr, nullptr};
		cudaEventCreate(&sp.a); cudaEventCreate(&sp.b);
		cudaEventRecord(sp.a, s);
		spans.push_back(sp);
	};
	auto t_end = [&]() { if (timing) cudaEventRecord(spans.back().b, s); };

	ATiles xb{sc.xb_hi.p, na == 2 ? sc.xb_lo.p : nullptr, KT_dim};
	ATiles xb2{sc.xb2_hi.p, na == 2 ? sc.xb2_lo.p : nullptr, KT_q};
	ATiles hb{sc.hb_hi.p, na == 2 ? sc.hb_lo.p : nullptr, KT_h};
	float* x = reinterpret_cast<float*>(sc.x.p);
	__half* q = reinterpret_cast<__half*>(sc.q.p);
	__half* q_lo = precise ? reinterpret_cast<__half*>(sc.q_lo.p) : nullptr;
	const float2* rope_cs = reinterpret_cast<const float2*>(sc.rope.p);

	// ---- weight dequantisation runs one GEMM ahead on the side stream, ping-ponging two tile buffers ----
	XALM_CUDA_CHECK(cudaEventRecord(sc.ev_start, s));
	XALM_CUDA_CHECK(cudaStreamWaitEvent(ds, sc.ev_start, 0));
	int job = 0;      // GEMMs issued so far
	int prepared = 0; // weight sets dequantised (issued) so far
	auto nb_of = [&](const WMat& w) { return precise && w.type != XALM_F16 ? 2 : 1; }; // f16 weights are exact in one plane
	auto prep = [&](const WMat& w, bool glu, int glu_off, int n_valid, int K, int NT, int KT) -> int {
		const int b = prepared & 1;
		if (prepared >= 2) XALM_CUDA_CHECK(cudaStreamWaitEvent(ds, sc.ev_gemm[b], 0)); // the GEMM that last read this buffer
		t_begin("dequant");
		XALM_TRY(launch_dequant_tiles(w, glu, glu_off, n_valid, K, NT, KT, sc.wt[b].p, nb_of(w) == 2 ? sc.wt_lo[b].p : nullptr, ds));
		t_end();
		XALM_CUDA_CHECK(cudaEventRecord(sc.ev_deq[b], ds));
		prepared++;
		launches++;
		return XALM_OK;
	};
	auto run = [&](GemmArgs& g, const WMat& w, const char* what) -> int {
		const int b = job & 1;
		g.b = sc.wt[b].p;
		g.b_lo = sc.wt_lo[b].p;
		XALM_CUDA_CHECK(cudaStreamWaitEvent(s, sc.ev_deq[b], 0));
		t_begin(what);
		XALM_TRY(launch_gemm(g, na, nb_of(w), s));
		t_end();
		XALM_CUDA_CHECK(cudaEventRecord(sc.ev_gemm[b], s));
		job++;
		launches++;
		return XALM_OK;
	};
	// Wo / W2 under tensor parallelism: each rank holds a slice of the input axis, so its GEMM gives a partial (T, dim) sum.  Rank 0
	// adds it to x (residual epilogue), the others store it to `part`; a reduce-scatter sums the P contributions of each row block
	// into the owning rank's rows of x, and an in-place all-gather copies every block to every rank.  Each element is summed once,
	// by one rank, so x stays bit-identical on every rank.  One GPU: the residual epilogue alone.
	float* part = reinterpret_cast<float*>(sc.part.p);
	auto row_split = [&](GemmArgs& g, const WMat& w, const char* what) -> int {
		const bool partial = tp && pm.tp_rank != 0;
		g.epi = partial ? GEPI_STORE : GEPI_RESID; g.out = partial ? part : x; g.ldo = c.dim;
		XALM_TRY(run(g, w, what));
		if (!tp) return XALM_OK;
		t_begin("exchange");
		const size_t cnt = (size_t) (Tr / pm.tp_size) * c.dim;
		float* mine = x + (size_t) pm.tp_rank * cnt;
		XALM_NCCL_CHECK(g_nccl.ReduceScatter(partial ? part : x, mine, cnt, ncclFloat32, ncclSum, pm.comm, s));
		XALM_NCCL_CHECK(g_nccl.AllGather(mine, x, cnt, ncclFloat32, pm.comm, s));
		t_end();
		launches += 2;
		return XALM_OK;
	};
	const size_t L = pm.layers.size();
	auto prep_qkv = [&](size_t l) { return prep(pm.layers[l].wqkv, false, 0, n_qkv, c.dim, NT_qkv, KT_dim); };

	XALM_CUDA_CHECK(cudaMemcpyAsync(sc.tokens.p, tokens, (size_t) T * 4, cudaMemcpyHostToDevice, s));
	embed_rows_kernel<<<std::min(cdiv(T * c.dim, 256), sm_count() * 8), 256, 0, s>>>(pm.embed_type, pm.embed_raw, pm.embed_row_bytes, c.dim,
	                                                                                  reinterpret_cast<const int*>(sc.tokens.p), T, x);
	rope_table_kernel<<<std::min(cdiv(T * (c.head_dim / 2), 256), sm_count() * 8), 256, 0, s>>>(pm.rope_freq, c.head_dim / 2, T, pos0,
	                                                                                             reinterpret_cast<float2*>(sc.rope.p));
	launches += 2;
	const int norm_grid = std::min(T, sm_count() * 16);
	if (L) XALM_TRY(prep_qkv(0));
	for (size_t l = 0; l < L; l++) {
		const PrefillLayer& P = pm.layers[l];
		if (!prefill_type_ok(P.wqkv.type)) return set_error(XALM_ERR_UNSUPPORTED, "prefill: weight type %d", P.wqkv.type);
		// ---- attention half ----
		t_begin("rmsnorm");
		rmsnorm_rows_kernel<<<norm_grid, 128, 0, s>>>(x, T, c.dim, P.rms_att, P.rms_att_type, c.norm_eps, xb);
		t_end();
		__half* k_stage = reinterpret_cast<__half*>(sc.k_stage.p);
		__half* v_stage = reinterpret_cast<__half*>(sc.v_stage.p);
		__half* sink_k = reinterpret_cast<__half*>(sc.sink_k.p);
		if (window) { // before the QKV epilogue overwrites the ring slots of positions pos0-S .. pos0+T-1-S
			t_begin("ring");
			gather_ring_kernel<<<std::min(cdiv((S - 1) * (pm.kv_dim / 8), 256), sm_count() * 8), 256, 0, s>>>(P.k_cache, P.v_cache, pm.kv_dim, S, pos0,
			                                                                                                   k_stage, v_stage);
			sink_versions_kernel<<<cdiv(pm.kv_dim, 128), 128, 0, s>>>(P.k_cache, pm.kv_dim, c.head_dim, pm.rope_freq, T, sink_k);
			t_end();
			launches += 2;
		}
		XALM_TRY(prep(P.wo, false, 0, c.dim, pm.q_dim, NT_dim, KT_q));
		GemmArgs g = {};
		g.a_hi = xb.hi; g.a_lo = xb.lo;
		g.MT = MT; g.NT = NT_qkv; g.KT = KT_dim; g.mt0 = 0; g.M = T; g.N = n_qkv; g.epi = GEPI_QKV;
		g.q_out = q; g.q_lo = q_lo; g.k_cache = P.k_cache; g.v_cache = P.v_cache; g.rope_cs = rope_cs;
		g.q_dim = pm.q_dim; g.kv_dim = pm.kv_dim; g.head_dim = c.head_dim; g.pos0 = pos0; g.qkv_clip = c.qkv_clip;
		if (attn_tc) { g.qt_hi = sc.qt_hi.p; g.qt_lo = precise ? sc.qt_lo.p : nullptr; g.n_qb = n_qb; }
		if (window) { g.ring = S; g.k_stage = k_stage; g.v_stage = v_stage; g.stage_row0 = S - 1; }
		// later chunks (and the window mode) re-tile the whole cache prefix / staging copy
		const bool tiles_from_epilogue = attn_tc && !window && pos0 == 0 && getenv("XALM_ATTN_RETILE") == nullptr;
		if (tiles_from_epilogue) { g.kt = sc.kt.p; g.vt = sc.vt.p; g.n_kb_total = n_kb_total; }
		XALM_TRY(run(g, P.wqkv, "gemm_qkv"));
		t_begin("attention");
		if (attn_tc) {
			if (!tiles_from_epilogue)
				retile_kv_kernel<<<dim3(2 * n_kb_total, pm.n_kv_heads), 256, 0, s>>>(window ? k_stage : P.k_cache, window ? v_stage : P.v_cache, pm.kv_dim,
				                                                                    attn_pos0 + T, n_kb_total, sc.kt.p, sc.vt.p);
			AttnTcArgs at = {sc.qt_hi.p, precise ? sc.qt_lo.p : nullptr, sc.kt.p, sc.vt.p, xb2, T, attn_pos0, pm.n_heads, pm.n_kv_heads, n_qb, n_kb_total,
			                 window ? S : 0, window ? sink_k : nullptr, window ? P.v_cache : nullptr, pm.kv_dim,
			                 getenv("XALM_ATTN_DBG") ? atoi(getenv("XALM_ATTN_DBG")) : 0};
			XALM_TRY(precise ? launch_attn_tc<true>(at, s) : launch_attn_tc<false>(at, s));
			launches++;
		} else {
			AttnPArgs at = {q, q_lo, window ? k_stage : P.k_cache, window ? v_stage : P.v_cache, xb2, T, attn_pos0, pm.q_dim, pm.kv_dim, pm.n_heads,
			                pm.n_kv_heads, cdiv(T, 64), window ? S : 0, window ? sink_k : nullptr, window ? P.v_cache : nullptr};
			if (c.head_dim == 128) XALM_TRY(precise ? (launch_attn_p<128, true>(at, s)) : (launch_attn_p<128, false>(at, s)));
			else XALM_TRY(precise ? (launch_attn_p<64, true>(at, s)) : (launch_attn_p<64, false>(at, s)));
		}
		t_end();
		XALM_TRY(prep(P.w13, true, P.glu_off, pm.hidden, c.dim, NT_glu, KT_dim));
		g = {};
		g.a_hi = xb2.hi; g.a_lo = xb2.lo;
		g.MT = MT; g.NT = NT_dim; g.KT = KT_q; g.M = T; g.N = c.dim;
		XALM_TRY(row_split(g, P.wo, "gemm_wo"));
		// ---- feed-forward half ----
		t_begin("rmsnorm");
		rmsnorm_rows_kernel<<<norm_grid, 128, 0, s>>>(x, T, c.dim, P.rms_ffn, P.rms_ffn_type, c.norm_eps, xb);
		t_end();
		XALM_TRY(prep(P.w2, false, 0, c.dim, pm.hidden, NT_dim, KT_h));
		g = {};
		g.a_hi = xb.hi; g.a_lo = xb.lo;
		g.MT = MT; g.NT = NT_glu; g.KT = KT_dim; g.M = T; g.N = pm.hidden; g.epi = GEPI_GLU; g.o = hb; g.act = c.act;
		XALM_TRY(run(g, P.w13, "gemm_w13"));
		if (l + 1 < L) XALM_TRY(prep_qkv(l + 1));
		else if (want_logits) XALM_TRY(prep(pm.wcls, false, 0, pm.vocab, c.dim, NT_cls, KT_dim));
		g = {};
		g.a_hi = hb.hi; g.a_lo = hb.lo;
		g.MT = MT; g.NT = NT_dim; g.KT = KT_h; g.M = T; g.N = c.dim;
		XALM_TRY(row_split(g, P.w2, "gemm_w2"));
		launches += 3;
	}
	if (want_logits) {
		if (!L) XALM_TRY(prep(pm.wcls, false, 0, pm.vocab, c.dim, NT_cls, KT_dim));
		rmsnorm_rows_kernel<<<norm_grid, 128, 0, s>>>(x, T, c.dim, pm.rms_final, pm.rms_final_type, c.norm_eps, xb);
		GemmArgs g = {};
		g.a_hi = xb.hi; g.a_lo = xb.lo;
		g.NT = NT_cls; g.KT = KT_dim; g.M = T; g.N = pm.vocab; g.epi = GEPI_STORE;
		// tensor parallel: this rank's (rows, vocab_l) block of the all-gathered shards, then back to the one-GPU layout
		float* logits_tp = reinterpret_cast<float*>(sc.logits_tp.p);
		const size_t shard = (size_t) logit_rows * pm.vocab;
		g.out = tp ? logits_tp + pm.tp_rank * shard : reinterpret_cast<float*>(sc.logits.p); g.ldo = pm.vocab;
		g.mt0 = want_logits == 1 ? MT - 1 : 0;
		g.MT = want_logits == 1 ? 1 : MT;
		g.out_row0 = logit_row0;
		XALM_TRY(run(g, pm.wcls, "gemm_cls"));
		launches++;
		if (tp) {
			t_begin("exchange");
			XALM_NCCL_CHECK(g_nccl.AllGather(logits_tp + pm.tp_rank * shard, logits_tp, shard, ncclFloat32, pm.comm, s));
			t_end();
			unshard_logits_kernel<<<(int) std::min<size_t>((logit_rows * (size_t) c.vocab_size / 4 + 255) / 256, (size_t) sm_count() * 8), 256, 0, s>>>(
			    logits_tp, pm.tp_size, logit_rows, pm.vocab, reinterpret_cast<float*>(sc.logits.p));
			launches += 2;
		}
		if (targets && probs_host) {
			for (int i = 0; i < T; i++)
				if (targets[i] < 0 || targets[i] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "prefill: target %d out of range", targets[i]);
			XALM_CUDA_CHECK(cudaMemcpyAsync(sc.targets.p, targets, (size_t) T * 4, cudaMemcpyHostToDevice, s));
			target_prob_kernel<<<T, 256, 0, s>>>(reinterpret_cast<const float*>(sc.logits.p), c.vocab_size, reinterpret_cast<const int*>(sc.targets.p),
			                                     reinterpret_cast<float*>(sc.probs.p));
			launches++;
			XALM_CUDA_CHECK(cudaMemcpyAsync(probs_host, sc.probs.p, (size_t) T * 4, cudaMemcpyDeviceToHost, s));
		}
		if (logits_host) {
			if (want_logits == 2)
				XALM_CUDA_CHECK(cudaMemcpyAsync(logits_host, sc.logits.p, (size_t) T * c.vocab_size * 4, cudaMemcpyDeviceToHost, s));
			else
				XALM_CUDA_CHECK(cudaMemcpyAsync(logits_host, sc.logits.p + (size_t) (sc.logits_rows - 1) * c.vocab_size * 4, (size_t) c.vocab_size * 4,
				                                cudaMemcpyDeviceToHost, s));
		}
	}
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "prefill launch failed: %s", cudaGetErrorString(e));
	if (n_launches) *n_launches = launches;
	if (timing) {
		cudaStreamSynchronize(s);
		std::vector<std::pair<std::string, float>> tot;
		for (auto& sp : spans) {
			float ms = 0.f;
			cudaEventElapsedTime(&ms, sp.a, sp.b);
			bool found = false;
			for (auto& t : tot)
				if (t.first == sp.what) { t.second += ms; found = true; }
			if (!found) tot.push_back({sp.what, ms});
			cudaEventDestroy(sp.a); cudaEventDestroy(sp.b);
		}
		fprintf(stderr, "[prefill timing, T=%d split=%d]", T, split);
		for (auto& t : tot) fprintf(stderr, " %s %.2f ms;", t.first.c_str(), t.second);
		fprintf(stderr, "\n");
	}
	return XALM_OK;
}

// ---- op-level hook -----------------------------------------------------------------------------------------------------
int prefill_gemm_dev(const WMat& w, const float* a_dev, int T, float* out_dev, int split, cudaStream_t s) {
	const int K = w.n, N = w.rows;
	if (K % 8) return set_error(XALM_ERR_INVALID, "gemm: K %% 8 != 0");
	const int na = split >= 2 ? 2 : 1, nb = split >= 3 ? 2 : 1;
	const int MT = cdiv(T, GB_M), KT = cdiv(K, GB_K), NT = cdiv(N, GB_N);
	DevBuf ah, al, bt, bl;
	XALM_TRY(ah.ensure((size_t) MT * KT * A_TILE_BYTES, true, s));
	if (na == 2) XALM_TRY(al.ensure((size_t) MT * KT * A_TILE_BYTES, true, s));
	XALM_TRY(bt.ensure((size_t) NT * KT * B_TILE_BYTES, false, s));
	if (nb == 2) XALM_TRY(bl.ensure((size_t) NT * KT * B_TILE_BYTES, false, s));
	ATiles at{ah.p, na == 2 ? al.p : nullptr, KT};
	pack_a_kernel<<<std::min(cdiv(T * (K / 8), 256), sm_count() * 8), 256, 0, s>>>(a_dev, T, K, at);
	int rc = launch_dequant_tiles(w, false, 0, N, K, NT, KT, bt.p, nb == 2 ? bl.p : nullptr, s);
	if (rc == XALM_OK) {
		GemmArgs g = {};
		g.a_hi = at.hi; g.a_lo = at.lo; g.b = bt.p; g.b_lo = bl.p;
		g.MT = MT; g.NT = NT; g.KT = KT; g.M = T; g.N = N; g.epi = GEPI_STORE; g.out = out_dev; g.ldo = N;
		rc = launch_gemm(g, na, nb, s);
	}
	cudaError_t e = cudaStreamSynchronize(s);
	ah.release(); al.release(); bt.release(); bl.release();
	if (rc != XALM_OK) return rc;
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "gemm failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

int prefill_bench_gemm(int T, int N, int K, int split, int iters, float* ms_per_launch) {
	const int na = split >= 2 ? 2 : 1, nb = split >= 3 ? 2 : 1;
	const int MT = cdiv(T, GB_M), KT = cdiv(K, GB_K), NT = cdiv(N, GB_N);
	cudaStream_t s;
	XALM_CUDA_CHECK(cudaStreamCreate(&s));
	DevBuf ah, al, bt, bl, out;
	XALM_TRY(ah.ensure((size_t) MT * KT * A_TILE_BYTES, true, s));
	if (na == 2) XALM_TRY(al.ensure((size_t) MT * KT * A_TILE_BYTES, true, s));
	XALM_TRY(bt.ensure((size_t) NT * KT * B_TILE_BYTES, true, s));
	if (nb == 2) XALM_TRY(bl.ensure((size_t) NT * KT * B_TILE_BYTES, true, s));
	XALM_TRY(out.ensure((size_t) MT * GB_M * N * 4, true, s));
	// fill the operands with a pattern of small finite fp16 values (0x2C00 = 0.0625)
	XALM_CUDA_CHECK(cudaMemsetAsync(ah.p, 0x2C, (size_t) MT * KT * A_TILE_BYTES, s));
	XALM_CUDA_CHECK(cudaMemsetAsync(bt.p, 0x2C, (size_t) NT * KT * B_TILE_BYTES, s));
	GemmArgs g = {};
	g.a_hi = ah.p; g.a_lo = al.p; g.b = bt.p; g.b_lo = bl.p;
	g.MT = MT; g.NT = NT; g.KT = KT; g.M = T; g.N = N; g.epi = GEPI_STORE; g.out = reinterpret_cast<float*>(out.p); g.ldo = N;
	cudaEvent_t e0, e1;
	XALM_CUDA_CHECK(cudaEventCreate(&e0));
	XALM_CUDA_CHECK(cudaEventCreate(&e1));
	for (int i = 0; i < 3; i++) XALM_TRY(launch_gemm(g, na, nb, s));
	XALM_CUDA_CHECK(cudaEventRecord(e0, s));
	for (int i = 0; i < iters; i++) XALM_TRY(launch_gemm(g, na, nb, s));
	XALM_CUDA_CHECK(cudaEventRecord(e1, s));
	XALM_CUDA_CHECK(cudaStreamSynchronize(s));
	float ms = 0.f;
	XALM_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
	*ms_per_launch = ms / (float) iters;
	cudaEventDestroy(e0); cudaEventDestroy(e1);
	ah.release(); al.release(); bt.release(); bl.release(); out.release();
	cudaStreamDestroy(s);
	return XALM_OK;
}

} // namespace xalm
