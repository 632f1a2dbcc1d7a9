// formats.cuh — every weight format the reference defines, on the device.
//
//   * type table (block elements / bytes)                       quants.py:45-77, types.h:505-514
//   * scalar decode of one element from the ON-DISK layout       types.h:302-325,406-427; quants.py dequantize_blocks
//     (used by the dequant entry point, the embedding gather and the repack/scan kernels)
//   * the PLANAR device layout weights are repacked into at upload (quants ‖ scales ‖ high bits as separate
//     16-byte-aligned planes, same byte count as on disk) and, per format, the 16-byte "chunk" a lane loads
//     with one 128-bit request plus the fused dequant·x arithmetic the matvec kernel runs on it.
//
// Bit-exactness notes (SURVEY.md §7): an f16 scale (11 significant bits) times a <=8-bit integer is exact in
// fp32, so d*q never rounds and d*q+m rounds once whether or not it is fused; Q8 multiplies by fp32(1/100);
// fp8 codes that IEEE-style decoders call NaN/Inf are ordinary finite numbers in the reference.
#pragma once
#include "common.cuh"

namespace xalm {

struct TypeInfo {
	int block; // elements per block
	int bytes; // bytes per block
};

__host__ __device__ inline bool type_info(int t, TypeInfo* ti) {
	switch (t) {
		case XALM_F32: *ti = {1, 4}; return true;
		case XALM_F16: case XALM_BF16: *ti = {1, 2}; return true;
		case XALM_F8_E2M5: case XALM_F8_E3M4: case XALM_F8_E4M3: case XALM_F8_E5M2: case XALM_U8: case XALM_Q8:
		case XALM_QI8: *ti = {1, 1}; return true;
		case XALM_Q4_0: *ti = {32, 18}; return true;
		case XALM_Q4_1: *ti = {32, 20}; return true;
		case XALM_Q5_0: *ti = {32, 22}; return true;
		case XALM_Q5_1: *ti = {32, 24}; return true;
		case XALM_Q8_0: *ti = {32, 34}; return true;
		case XALM_TQ1_0: *ti = {256, 54}; return true;
	}
	return false;
}

// bytes of one 256-element "unit" of the unit-interleaved device layout (matvec_tma.cuh, matvec_idp.cuh); 0 = not a unit format
__host__ __device__ inline int unit_bytes(int t) {
	switch (t) {
		case XALM_F32: return 1024;
		case XALM_F16: case XALM_BF16: return 512;
		case XALM_F8_E4M3: case XALM_F8_E5M2: case XALM_Q8: return 256;
		case XALM_Q8_0: return 272;
		case XALM_Q4_0: return 144;
		case XALM_Q4_1: return 160;
		case XALM_Q5_0: return 176;
		case XALM_Q5_1: return 192;
	}
	return 0; // not a TMA-path format
}

// ---------------------------------------------------------------------------------------------------------
// Scalar decode from the on-disk layout.
// ---------------------------------------------------------------------------------------------------------

// f8_t<E,M>::to_float (types.h:302-314): sign -> bit 31, low 7 bits -> top of exponent|mantissa, times 2^(127-bias).
template <int E, int M>
__device__ __forceinline__ float f8_decode(uint8_t b) {
	constexpr int bias = (1 << (E - 1)) - 1;
	const uint32_t bits = ((uint32_t) (b & 0x80) << 24) | ((uint32_t) (b & 0x7F) << (23 - M));
	return __fmul_rn(__uint_as_float(bits), __uint_as_float((uint32_t) (127 + 127 - bias) << 23)); // * 2^(127-bias)
}

__device__ __forceinline__ float decode_byte_type(int t, uint8_t b) {
	switch (t) {
		case XALM_F8_E2M5: return f8_decode<2, 5>(b);
		case XALM_F8_E3M4: return f8_decode<3, 4>(b);
		case XALM_F8_E4M3: return f8_decode<4, 3>(b);
		case XALM_F8_E5M2: return f8_decode<5, 2>(b);
		case XALM_Q8: return __fmul_rn(1.f / 100.f, (float) (int8_t) b);                  // types.h:423-424
		case XALM_QI8: return __fsub_rn(__fdiv_rn((float) b, 127.5f), 1.0f);               // convert.py:550-551
		case XALM_U8: return (float) b;
	}
	return 666.66f; // types.h:426
}

// one element of a scalar (non-block) type
__device__ __forceinline__ float decode_scalar(int t, const uint8_t* p, size_t i) {
	switch (t) {
		case XALM_F32: return reinterpret_cast<const float*>(p)[i];
		case XALM_F16: return f16_bits_to_f32(reinterpret_cast<const uint16_t*>(p)[i]);
		case XALM_BF16: return bf16_bits_to_f32(reinterpret_cast<const uint16_t*>(p)[i]);
		default: return decode_byte_type(t, p[i]);
	}
}

__device__ __forceinline__ float ld_f16_unaligned(const uint8_t* p) { return f16_bits_to_f32((uint16_t) (p[0] | (p[1] << 8))); }

// element j of an on-disk block (quants.py:302-313, 337-350, 376-393, 419-438, 458-464, 664-683; SURVEY App. B)
__device__ inline float decode_block_elem(int t, const uint8_t* b, int j) {
	switch (t) {
		case XALM_Q8_0: return __fmul_rn((float) (int8_t) b[2 + j], ld_f16_unaligned(b));
		case XALM_Q4_0: {
			const int q = j < 16 ? (b[2 + j] & 0x0F) : (b[2 + j - 16] >> 4);
			return __fmul_rn(ld_f16_unaligned(b), (float) (q - 8));
		}
		case XALM_Q4_1: {
			const int q = j < 16 ? (b[4 + j] & 0x0F) : (b[4 + j - 16] >> 4);
			return __fadd_rn(__fmul_rn(ld_f16_unaligned(b), (float) q), ld_f16_unaligned(b + 2));
		}
		case XALM_Q5_0: {
			const uint32_t qh = b[2] | (b[3] << 8) | (b[4] << 16) | ((uint32_t) b[5] << 24);
			const int ql = j < 16 ? (b[6 + j] & 0x0F) : (b[6 + j - 16] >> 4);
			const int q = ql | (((qh >> j) & 1) << 4);
			return __fmul_rn(ld_f16_unaligned(b), (float) (q - 16));
		}
		case XALM_Q5_1: {
			const uint32_t qh = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t) b[7] << 24);
			const int ql = j < 16 ? (b[8 + j] & 0x0F) : (b[8 + j - 16] >> 4);
			const int q = ql | (((qh >> j) & 1) << 4);
			return __fadd_rn(__fmul_rn(ld_f16_unaligned(b), (float) q), ld_f16_unaligned(b + 2));
		}
		case XALM_TQ1_0: {
			int k, B;
			if (j < 160) { k = j / 32; B = j % 32; }
			else if (j < 240) { k = (j - 160) / 16; B = 32 + (j - 160) % 16; }
			else { k = (j - 240) / 4; B = 48 + (j - 240) % 4; }
			const int pow3[5] = {1, 3, 9, 27, 81};
			const uint8_t q = (uint8_t) (b[B] * pow3[k]);
			const int trit = ((int) q * 3) >> 8;
			return __fmul_rn(ld_f16_unaligned(b + 52), (float) (trit - 1));
		}
	}
	return 666.66f;
}

// generic "element i of a tensor in its on-disk layout"
__device__ __forceinline__ float decode_disk_elem(int t, const uint8_t* base, size_t i) {
	TypeInfo ti;
	type_info(t, &ti);
	if (ti.block == 1) return decode_scalar(t, base, i);
	return decode_block_elem(t, base + (i / ti.block) * (size_t) ti.bytes, (int) (i % ti.block));
}

// ---------------------------------------------------------------------------------------------------------
// Planar device layout.
// ---------------------------------------------------------------------------------------------------------
// One weight matrix W(rows, n) on the device.  p0 = main plane (element bytes / quants, 16-byte aligned rows),
// p1 = scales (f16 d, or half2 {d,m}), p2 = high bits (u32 qh per block).  Strides in bytes.
//   F32/F16/BF16/F8_*    p0 = the on-disk row                                   (no repack)
//   Q8 (int8 x 1/100)    p0 = q + 128 as uint8                                  (bias removes a sign fix-up per element)
//   QI8                  p0 = the on-disk row
//   Q8_0                 p0 = (q + 128) uint8 [n]        p1 = f16 d [n/32]
//   Q4_0                 p0 = nibbles [n/2]              p1 = f16 d [n/32]
//   Q4_1                 p0 = nibbles [n/2]              p1 = half2 {d,m} [n/32]
//   Q5_0                 p0 = nibbles [n/2]              p1 = f16 d [n/32]        p2 = u32 qh [n/32]
//   Q5_1                 p0 = nibbles [n/2]              p1 = half2 {d,m} [n/32]  p2 = u32 qh [n/32]
//   TQ1_0                p0 = the on-disk row (54-byte blocks)
struct WMat {
	int type = 0;
	int rows = 0;
	int n = 0;
	int flags = 0; // bit0: fp8 tensor contains codes an IEEE decoder maps to NaN/Inf -> take the exact LUT path
	int layout_units = 0; // block format stored unit-interleaved for the TMA kernel (matvec_tma.cuh) instead of planar
	int layout_frag = 0;  // integer format stored as fragment tiles (frag_layout.cuh): p0 = records, s0 = bytes of one 16-row tile
	int glu_half = 0;     // fragment tiles of a gate|up matrix: rows [0, glu_half) are W1, the rest W3, interleaved 8 + 8 per tile
	const uint8_t* p0 = nullptr;
	const uint8_t* p1 = nullptr;
	const uint8_t* p2 = nullptr;
	size_t s0 = 0, s1 = 0, s2 = 0;
};
enum { WMAT_FP8_NONFINITE = 1 };

struct PlaneSizes {
	size_t s0, s1, s2;
};
__host__ inline PlaneSizes plane_row_bytes(int t, int n) {
	switch (t) {
		case XALM_F32: return {(size_t) n * 4, 0, 0};
		case XALM_F16: case XALM_BF16: return {(size_t) n * 2, 0, 0};
		case XALM_Q8_0: return {(size_t) n, (size_t) n / 32 * 2, 0};
		case XALM_Q4_0: return {(size_t) n / 2, (size_t) n / 32 * 2, 0};
		case XALM_Q4_1: return {(size_t) n / 2, (size_t) n / 32 * 4, 0};
		case XALM_Q5_0: return {(size_t) n / 2, (size_t) n / 32 * 2, (size_t) n / 32 * 4};
		case XALM_Q5_1: return {(size_t) n / 2, (size_t) n / 32 * 4, (size_t) n / 32 * 4};
		case XALM_TQ1_0: return {(size_t) n / 256 * 54, 0, 0};
		default: return {(size_t) n, 0, 0}; // one byte per element
	}
}

#ifndef XALM_SECONDARY_TU // non-template kernels: defined once, in xalm_cuda.cu's translation unit
// raw (on-disk rows, `raw_stride` bytes apart) -> planes.  One thread per block (or per 16 bytes for scalar types).
__global__ void repack_kernel(int t, const uint8_t* __restrict__ raw, size_t raw_stride, int rows, int n, uint8_t* p0,
                              size_t s0, uint8_t* p1, size_t s1, uint8_t* p2, size_t s2) {
	TypeInfo ti;
	type_info(t, &ti);
	if (ti.block == 1 || t == XALM_TQ1_0) {
		// byte copy (Q8: re-bias int8 -> uint8)
		const size_t row_bytes = (size_t) n / ti.block * ti.bytes;
		const size_t total = (size_t) rows * row_bytes;
		for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
			const size_t r = i / row_bytes, c = i % row_bytes;
			uint8_t v = raw[r * raw_stride + c];
			if (t == XALM_Q8) v ^= 0x80;
			p0[r * s0 + c] = v;
		}
		return;
	}
	const int nb = n / 32;
	const size_t total = (size_t) rows * nb;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const size_t r = i / nb;
		const int b = (int) (i % nb);
		const uint8_t* src = raw + r * raw_stride + (size_t) b * ti.bytes;
		uint8_t* q = p0 + r * s0;
		uint8_t* sc = p1 + r * s1;
		switch (t) {
			case XALM_Q8_0:
				sc[2 * b] = src[0]; sc[2 * b + 1] = src[1];
				for (int j = 0; j < 32; j++) q[32 * b + j] = src[2 + j] ^ 0x80;
				break;
			case XALM_Q4_0:
				sc[2 * b] = src[0]; sc[2 * b + 1] = src[1];
				for (int j = 0; j < 16; j++) q[16 * b + j] = src[2 + j];
				break;
			case XALM_Q4_1:
				for (int j = 0; j < 4; j++) sc[4 * b + j] = src[j];
				for (int j = 0; j < 16; j++) q[16 * b + j] = src[4 + j];
				break;
			case XALM_Q5_0:
				sc[2 * b] = src[0]; sc[2 * b + 1] = src[1];
				for (int j = 0; j < 4; j++) (p2 + r * s2)[4 * b + j] = src[2 + j];
				for (int j = 0; j < 16; j++) q[16 * b + j] = src[6 + j];
				break;
			case XALM_Q5_1:
				for (int j = 0; j < 4; j++) sc[4 * b + j] = src[j];
				for (int j = 0; j < 4; j++) (p2 + r * s2)[4 * b + j] = src[4 + j];
				for (int j = 0; j < 16; j++) q[16 * b + j] = src[8 + j];
				break;
		}
	}
}

// does an fp8 tensor contain a code the hardware converter would turn into NaN/Inf?
__global__ void fp8_scan_nonfinite_kernel(int t, const uint8_t* __restrict__ p, size_t nbytes, int* flag) {
	bool bad = false;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < nbytes; i += (size_t) gridDim.x * blockDim.x) {
		const uint8_t b = p[i] & 0x7F;
		if (t == XALM_F8_E4M3) bad |= (b == 0x7F);
		else bad |= (b >= 0x7C);
	}
	if (bad) *flag = 1;
}
#endif // XALM_SECONDARY_TU

// ---------------------------------------------------------------------------------------------------------
// Chunk arithmetic for the matvec kernel.  A "chunk" is what one lane fetches with ONE 16-byte load from the
// main plane: E consecutive elements of a row.  fma_chunk accumulates  sum_j w_j * x_j  into a packed pair of
// fp32 partial sums (even/odd lanes of fma.rn.f32x2).
// ---------------------------------------------------------------------------------------------------------
struct RowPtr {
	const uint8_t* p0;
	const uint8_t* p1;
	const uint8_t* p2;
};

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
	uint32_t r;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
	return r;
}
// byte k of w as the float 2^23 + byte  (exact integer -> float without the I2F pipe)
template <int K>
__device__ __forceinline__ float magic_byte(uint32_t w) {
	return __uint_as_float(prmt(w, 0x4B000000u, 0x7540u | K));
}

// sum over the 4 bytes of w:  (byte - BIAS) * x[0..3]   accumulated into acc
template <int BIAS>
__device__ __forceinline__ void fma_bytes4(uint32_t w, const float* x, f32x2& acc) {
	const float C = -(8388608.0f + (float) BIAS);
	const f32x2 c2 = pack2(C, C);
	const f32x2 a = add2(pack2(magic_byte<0>(w), magic_byte<1>(w)), c2);
	const f32x2 b = add2(pack2(magic_byte<2>(w), magic_byte<3>(w)), c2);
	acc = fma2(a, pack2(x[0], x[1]), acc);
	acc = fma2(b, pack2(x[2], x[3]), acc);
}
// same, but each weight is d*q + m (rounded once, like numpy's (d*q)+m with exact d*q)
__device__ __forceinline__ void fma_bytes4_dm(uint32_t w, f32x2 d2, f32x2 m2, const float* x, f32x2& acc) {
	const f32x2 c2 = pack2(-8388608.0f, -8388608.0f);
	const f32x2 a = fma2(add2(pack2(magic_byte<0>(w), magic_byte<1>(w)), c2), d2, m2);
	const f32x2 b = fma2(add2(pack2(magic_byte<2>(w), magic_byte<3>(w)), c2), d2, m2);
	acc = fma2(a, pack2(x[0], x[1]), acc);
	acc = fma2(b, pack2(x[2], x[3]), acc);
}

template <int TYPE>
struct Fmt;

// ---- F32 ----
template <>
struct Fmt<XALM_F32> {
	static constexpr int E = 4;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		acc = fma2(pack2(__uint_as_float(f.w.x), __uint_as_float(f.w.y)), pack2(x[0], x[1]), acc);
		acc = fma2(pack2(__uint_as_float(f.w.z), __uint_as_float(f.w.w)), pack2(x[2], x[3]), acc);
	}
};
// ---- F16 ----
template <>
struct Fmt<XALM_F16> {
	static constexpr int E = 8;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
#pragma unroll
		for (int i = 0; i < 4; i++) {
			const float2 v = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
			acc = fma2(pack2(v.x, v.y), pack2(x[2 * i], x[2 * i + 1]), acc);
		}
	}
};
// ---- BF16 (types.h:322-325: bits << 16) ----
template <>
struct Fmt<XALM_BF16> {
	static constexpr int E = 8;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
#pragma unroll
		for (int i = 0; i < 4; i++)
			acc = fma2(pack2(__uint_as_float(w[i] << 16), __uint_as_float(w[i] & 0xFFFF0000u)), pack2(x[2 * i], x[2 * i + 1]), acc);
	}
};
// ---- F8_E4M3 / F8_E5M2 fast path: hardware fp8->f16 conversion, valid when the tensor holds no NaN/Inf code
//      (fp8_scan_nonfinite_kernel); every finite code converts to exactly the reference's value. ----
template <>
struct Fmt<XALM_F8_E4M3> {
	static constexpr int E = 16;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
#pragma unroll
		for (int i = 0; i < 4; i++) {
			uint32_t h0, h1;
			asm("{ .reg .b16 lo, hi; mov.b32 {lo, hi}, %2; cvt.rn.f16x2.e4m3x2 %0, lo; cvt.rn.f16x2.e4m3x2 %1, hi; }"
			    : "=r"(h0), "=r"(h1)
			    : "r"(w[i]));
			const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&h0));
			const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&h1));
			acc = fma2(pack2(a.x, a.y), pack2(x[4 * i], x[4 * i + 1]), acc);
			acc = fma2(pack2(b.x, b.y), pack2(x[4 * i + 2], x[4 * i + 3]), acc);
		}
	}
};
template <>
struct Fmt<XALM_F8_E5M2> {
	static constexpr int E = 16;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
#pragma unroll
		for (int i = 0; i < 4; i++) {
			// an e5m2 code is the high byte of the f16 with the same value
			const uint32_t h0 = prmt(w[i], 0u, 0x1404u); // {0,b0,0,b1}
			const uint32_t h1 = prmt(w[i], 0u, 0x3424u); // {0,b2,0,b3}
			const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&h0));
			const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&h1));
			acc = fma2(pack2(a.x, a.y), pack2(x[4 * i], x[4 * i + 1]), acc);
			acc = fma2(pack2(b.x, b.y), pack2(x[4 * i + 2], x[4 * i + 3]), acc);
		}
	}
};
// ---- any one-byte type through a 256-entry table in shared memory (exact for every code): F8_E2M5, F8_E3M4,
//      QI8, and E4M3/E5M2 tensors that do contain NaN/Inf codes.  TYPE tag -1. ----
template <>
struct Fmt<-1> {
	static constexpr int E = 16;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk_lut(const Frag& f, const float* x, f32x2& acc, const float* lut) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
#pragma unroll
		for (int i = 0; i < 4; i++) {
			acc = fma2(pack2(lut[w[i] & 0xFF], lut[(w[i] >> 8) & 0xFF]), pack2(x[4 * i], x[4 * i + 1]), acc);
			acc = fma2(pack2(lut[(w[i] >> 16) & 0xFF], lut[w[i] >> 24]), pack2(x[4 * i + 2], x[4 * i + 3]), acc);
		}
	}
};
// ---- Q8: int8 * fp32(1/100) (types.h:423-424); plane holds q+128 ----
template <>
struct Fmt<XALM_Q8> {
	static constexpr int E = 16;
	struct Frag { uint4 w; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) { return {ld_stream16(r.p0 + (size_t) c * 16)}; }
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		f32x2 s = pack2(0.f, 0.f);
		fma_bytes4<128>(f.w.x, x, s);
		fma_bytes4<128>(f.w.y, x + 4, s);
		fma_bytes4<128>(f.w.z, x + 8, s);
		fma_bytes4<128>(f.w.w, x + 12, s);
		const float k = 1.f / 100.f;
		acc = fma2(pack2(k, k), s, acc);
	}
};
// ---- Q8_0: d * q (quants.py:458-464); plane0 = q+128, plane1 = f16 d per 32 ----
template <>
struct Fmt<XALM_Q8_0> {
	static constexpr int E = 16;
	struct Frag { uint4 w; uint16_t d; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) {
		return {ld_stream16(r.p0 + (size_t) c * 16), ld_stream2(r.p1 + (size_t) (c >> 1) * 2)};
	}
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		f32x2 s = pack2(0.f, 0.f);
		fma_bytes4<128>(f.w.x, x, s);
		fma_bytes4<128>(f.w.y, x + 4, s);
		fma_bytes4<128>(f.w.z, x + 8, s);
		fma_bytes4<128>(f.w.w, x + 12, s);
		const float d = f16_bits_to_f32(f.d);
		acc = fma2(pack2(d, d), s, acc);
	}
};
// ---- Q4_0: d * (q - 8) (quants.py:302-313): byte j = {lo: elem j, hi: elem j+16}; one chunk = one block ----
template <>
struct Fmt<XALM_Q4_0> {
	static constexpr int E = 32;
	struct Frag { uint4 w; uint16_t d; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) {
		return {ld_stream16(r.p0 + (size_t) c * 16), ld_stream2(r.p1 + (size_t) c * 2)};
	}
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
		f32x2 s = pack2(0.f, 0.f);
#pragma unroll
		for (int i = 0; i < 4; i++) {
			fma_bytes4<8>(w[i] & 0x0F0F0F0Fu, x + 4 * i, s);
			fma_bytes4<8>((w[i] >> 4) & 0x0F0F0F0Fu, x + 16 + 4 * i, s);
		}
		const float d = f16_bits_to_f32(f.d);
		acc = fma2(pack2(d, d), s, acc);
	}
};
// ---- Q4_1: d * q + m (quants.py:337-350) ----
template <>
struct Fmt<XALM_Q4_1> {
	static constexpr int E = 32;
	struct Frag { uint4 w; uint32_t dm; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) {
		return {ld_stream16(r.p0 + (size_t) c * 16), ld_stream4(r.p1 + (size_t) c * 4)};
	}
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
		const float d = f16_bits_to_f32((uint16_t) (f.dm & 0xFFFF)), m = f16_bits_to_f32((uint16_t) (f.dm >> 16));
		const f32x2 d2 = pack2(d, d), m2 = pack2(m, m);
#pragma unroll
		for (int i = 0; i < 4; i++) {
			fma_bytes4_dm(w[i] & 0x0F0F0F0Fu, d2, m2, x + 4 * i, acc);
			fma_bytes4_dm((w[i] >> 4) & 0x0F0F0F0Fu, d2, m2, x + 16 + 4 * i, acc);
		}
	}
};
// bits [4i, 4i+4) of qh spread to bit 4 of four bytes
__device__ __forceinline__ uint32_t spread_hi4(uint32_t qh, int shift) {
	return (((qh >> shift) & 0xFu) * 0x02040810u) & 0x10101010u;
}
// ---- Q5_0: d * ((ql | qh<<4) - 16) (quants.py:376-393) ----
template <>
struct Fmt<XALM_Q5_0> {
	static constexpr int E = 32;
	struct Frag { uint4 w; uint32_t qh; uint16_t d; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) {
		return {ld_stream16(r.p0 + (size_t) c * 16), ld_stream4(r.p2 + (size_t) c * 4), ld_stream2(r.p1 + (size_t) c * 2)};
	}
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
		f32x2 s = pack2(0.f, 0.f);
#pragma unroll
		for (int i = 0; i < 4; i++) {
			fma_bytes4<16>((w[i] & 0x0F0F0F0Fu) | spread_hi4(f.qh, 4 * i), x + 4 * i, s);
			fma_bytes4<16>(((w[i] >> 4) & 0x0F0F0F0Fu) | spread_hi4(f.qh, 16 + 4 * i), x + 16 + 4 * i, s);
		}
		const float d = f16_bits_to_f32(f.d);
		acc = fma2(pack2(d, d), s, acc);
	}
};
// ---- Q5_1: d * (ql | qh<<4) + m (quants.py:419-438) ----
template <>
struct Fmt<XALM_Q5_1> {
	static constexpr int E = 32;
	struct Frag { uint4 w; uint32_t qh; uint32_t dm; };
	static __device__ __forceinline__ Frag load(const RowPtr& r, int c) {
		return {ld_stream16(r.p0 + (size_t) c * 16), ld_stream4(r.p2 + (size_t) c * 4), ld_stream4(r.p1 + (size_t) c * 4)};
	}
	static __device__ __forceinline__ void fma_chunk(const Frag& f, const float* x, f32x2& acc) {
		const uint32_t w[4] = {f.w.x, f.w.y, f.w.z, f.w.w};
		const float d = f16_bits_to_f32((uint16_t) (f.dm & 0xFFFF)), m = f16_bits_to_f32((uint16_t) (f.dm >> 16));
		const f32x2 d2 = pack2(d, d), m2 = pack2(m, m);
#pragma unroll
		for (int i = 0; i < 4; i++) {
			fma_bytes4_dm((w[i] & 0x0F0F0F0Fu) | spread_hi4(f.qh, 4 * i), d2, m2, x + 4 * i, acc);
			fma_bytes4_dm(((w[i] >> 4) & 0x0F0F0F0Fu) | spread_hi4(f.qh, 16 + 4 * i), d2, m2, x + 16 + 4 * i, acc);
		}
	}
};

} // namespace xalm
