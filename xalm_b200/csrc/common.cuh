// common.cuh — small device/host helpers shared by every kernel of the sm_100a backend.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/xalm_cuda.h"

namespace xalm {

// ---- error plumbing (no exceptions cross the C ABI: status code + thread-local message) ----------------
extern thread_local std::string g_last_error;
int set_error(int status, const char* fmt, ...);

#define XALM_CUDA_CHECK(expr)                                                                                   \
	do {                                                                                                        \
		cudaError_t _e = (expr);                                                                                \
		if (_e != cudaSuccess)                                                                                  \
			return ::xalm::set_error(XALM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
			                         __LINE__);                                                                 \
	} while (0)

#define XALM_TRY(expr)                  \
	do {                                \
		int _s = (expr);                \
		if (_s != XALM_OK) return _s;   \
	} while (0)

// ---- per-token scalars every kernel reads from device memory, so one captured graph serves every position ----
struct StepParams {
	int token;
	int pos;
	int kv_sink; // infer.cpp:611
	int kv_pos;  // infer.cpp:612
	int kv_len;  // infer.cpp:613
	int mode;
	unsigned int ar_base; // peer allreduce sequence base of this token (same on every rank)
	int slot;    // batched decode: the sequence slot (KV cache) this entry drives
	int kv_fresh; // first ring row of this entry's slot written in this step: kv_pos, or the span's first row when the slot has
	              // several entries (consecutive positions, xalm_cuda_forward_spans); rows kv_fresh .. kv_pos are written by the QKV kernel
	uint32_t tree; // batched attention's row map (xalm_cuda_forward_tree): for 0 <= t - kv_fresh <= 7, row t of the entry's sequence is
	               // read from row kv_fresh + ((tree >> 3 * (t - kv_fresh)) & 7); every other row is read where it is.  TREE_IDENTITY
	               // everywhere but in a tree step.
};
constexpr uint32_t TREE_IDENTITY = 0xFAC688u; // 3-bit fields 0, 1, .., 7: row t is read from row t

// ---- loads ---------------------------------------------------------------------------------------------
// Weights are streamed exactly once per token: read-only path, do not allocate in L1 (activations live there).
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
	uint4 r;
	asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4];"
	             : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
	             : "l"(p));
	return r;
}
__device__ __forceinline__ uint32_t ld_stream4(const void* p) {
	uint32_t r;
	asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
	return r;
}
__device__ __forceinline__ uint16_t ld_stream2(const void* p) {
	uint16_t r;
	asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(r) : "l"(p));
	return r;
}
// Activations: plain cached loads (x is re-read by every warp of the SM and sits in L1).
__device__ __forceinline__ float4 ld_act4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// ---- programmatic dependent launch (sm_90+): let the next kernel's prologue overlap this kernel's tail ----
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

// ---- L2 prefetch of a slice of the NEXT kernel's first bytes (cp.async.bulk.prefetch.L2): CTA `cta` of `n_ctas` takes its share ----
__device__ __forceinline__ void l2_prefetch_slice(const uint8_t* ptr, unsigned long long bytes, int cta, int n_ctas) {
	if (!ptr || !bytes) return;
	unsigned long long per = ((bytes + n_ctas - 1) / n_ctas + 127ull) & ~127ull;
	const unsigned long long off = per * (unsigned long long) cta;
	if (off >= bytes) return;
	if (off + per > bytes) per = (bytes - off) & ~15ull;
	if (per) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr + off), "r"((unsigned int) per) : "memory");
}

// ---- mbarrier / bulk-copy primitives ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "WAIT_%=:\n"
	    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	    "@p bra DONE_%=;\n"
	    "bra WAIT_%=;\n"
	    "DONE_%=:\n"
	    "}\n" ::"r"(smem_u32(bar)),
	    "r"(parity)
	    : "memory");
}
// global -> shared bulk copy (TMA, 1-D); completion is credited to `bar` in bytes.  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
	             "r"(bytes), "r"(smem_u32(bar))
	             : "memory");
}
// ---- packed fp32x2 arithmetic (new on sm_100: two FMAs per issued instruction) ---------------------------
struct f32x2 {
	unsigned long long v;
};
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
	f32x2 r;
	asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
	return r;
}
__device__ __forceinline__ void unpack2(f32x2 a, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
	f32x2 r;
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
	return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
	f32x2 r;
	asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
	return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
	f32x2 r;
	asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
	return r;
}

// ---- optional in-kernel timeline (debug/profiling: no nsys in this environment).  When enabled, block 0 of every kernel
//      records %globaltimer at entry, after the dependency wait and at exit. ----
struct Timeline {
	unsigned long long* buf; // 4 x u64 per record: kernel id, t_entry, t_after_wait, t_exit
	unsigned int cap;
	unsigned int count;
};
__device__ __forceinline__ unsigned long long gtime() {
	unsigned long long t;
	asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
	return t;
}
#ifndef XALM_SECONDARY_TU // the timeline lives in xalm_cuda.cu's translation unit only
__device__ Timeline d_timeline = {nullptr, 0, 0};
__device__ __forceinline__ int tl_begin(int kid) {
	if (d_timeline.buf == nullptr) return -1;
	const unsigned int slot = atomicAdd(&d_timeline.count, 1u);
	if (slot >= d_timeline.cap) return -1;
	d_timeline.buf[4 * slot] = (unsigned long long) kid;
	d_timeline.buf[4 * slot + 1] = gtime();
	return (int) slot;
}
__device__ __forceinline__ void tl_mark(int slot, int which) {
	if (slot >= 0) d_timeline.buf[4 * slot + which] = gtime();
}
#else
__device__ __forceinline__ int tl_begin(int) { return -1; }
__device__ __forceinline__ void tl_mark(int, int) {}
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
	return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
	return v;
}

__device__ __forceinline__ float bf16_bits_to_f32(uint16_t h) { return __uint_as_float((uint32_t) h << 16); }
__device__ __forceinline__ float f16_bits_to_f32(uint16_t h) { return __half2float(__ushort_as_half(h)); }

} // namespace xalm
