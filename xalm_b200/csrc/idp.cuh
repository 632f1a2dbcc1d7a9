// idp.cuh — the integer-dot-product core of the decode matvec for the integer weight formats
// (Q8_0, Q4_0, Q4_1, Q5_0, Q5_1 of quants.py:281-464, and Q8 = int8 x 1/100 of types.h:423-424).
//
// The reference multiplies dequantised weights d*q (+m) by fp32 activations (infer.cpp:104-135).  On the CUDA cores
// that costs ~2.2 issue slots per 8-bit weight and ~4.3 per 4-bit weight (byte -> fp32 via PRMT, FADD2, FFMA2):
// profiles/r1_matvec_tma_q8_0_w13.md shows the q8_0 kernel latency/issue-bound at 75 % of HBM peak and the 4/5-bit
// formats ALU-bound at 26-29 %.  Here the sum over a 32-element block is taken in INTEGERS with dp4a:
//
//     sum_j (d*q_j) * x_j  =  d * dx * sum_j q_j * X_j          x_j ~= dx * X_j,  X_j a 24-bit integer,
//
// where the activation block is held as block floating point — one power-of-two scale dx per 32 elements and three
// int8 limbs per element (X = 65536*l0 + 256*l1 + l2; l0 signed, l1, l2 unsigned), so one IDP.4A handles four weights
// against one limb: 24 dp4a per 32-weight block instead of 64-136 PRMT/FADD2/FFMA2.  The integer sums are exact; the
// only rounding beyond the reference's is x -> 23 bits + sign relative to its block maximum (<= 2^-23 of the largest
// |x| of the block — measured against fp64 the result is CLOSER than sequential fp32 accumulation, tests/test_idp_cpu.py).
// With a one-hot x the arithmetic is exact and returns the dequantised weight bit for bit (d*q is exact in fp32,
// d*q+m rounds once, as in quants.py).
//
// Biased storage (q+128 for Q8_0/Q8 in the unit layout, q-8 / q-16 semantics of Q4_0 / Q5_0) is folded into the
// accumulator's initial value: -BIAS * (sum of the block's limbs), kept per block next to dx.
#pragma once
#include "matvec.cuh"

namespace xalm {

// ---- activation side ----------------------------------------------------------------------------------------------
// Shared-memory image of a quantised activation vector of n elements (n % 32 == 0):
//   limb plane k at q + k * n (n bytes each, natural element order), then n/32 meta entries {S0, S1, S2, dx bits}.
struct XqView {
	uint8_t* q;   // 3 planes of n bytes
	int4* meta;   // n / 32 entries
	int n;
};
__host__ __device__ inline size_t xq_bytes(int n) { return (size_t) 3 * n + (size_t) (n / 32) * 16; }
__device__ __forceinline__ XqView xq_view(uint8_t* base, int n) { return {base, reinterpret_cast<int4*>(base + (size_t) 3 * n), n}; }

// The staging: EIGHT consecutive elements per lane, the four lanes 4k..4k+3 of a warp share a block (call with all lanes of the
// warp).  Loads are coalesced (32 bytes per lane, 1 KB per warp instruction) and every thread of the CTA works; a thread-per-block
// staging left half the CTA idle behind 32 line-strided loads per lane and took 7 us of a 25 us kernel
// (profiles/r2_decode_timeline.md).
__device__ __forceinline__ void xq_store_group8(const XqView& v, int grp, const float (&x)[8]) {
	uint32_t mb = 0; // block maximum of |x| (non-negative floats order like their bit patterns)
#pragma unroll
	for (int e = 0; e < 8; e++) mb = max(mb, __float_as_uint(x[e]) & 0x7fffffffu);
	mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 1));
	mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 2));
	const int eb = (int) (mb >> 23);                 // biased exponent of the maximum: max < 2^(eb-126)
	const bool live = eb >= 40 && eb < 255;          // blocks below 2^-87 contribute nothing; non-finite blocks are dropped
	const float sc = live ? __uint_as_float((uint32_t) (276 - eb) << 23) : 0.f;  // 2^(149-eb): |x*sc| < 2^23
	const float dx = live ? __uint_as_float((uint32_t) (eb - 22) << 23) : 0.f;   // 2^(eb-149)
	uint32_t w[3][2];
	int s0 = 0;
	uint32_t s1 = 0, s2 = 0;
#pragma unroll
	for (int q = 0; q < 2; q++) {
		int X[4];
#pragma unroll
		for (int e = 0; e < 4; e++) X[e] = min(__float2int_rn(x[4 * q + e] * sc), 8388607);
		// byte k of X[0..3] -> word k (limb 2 = low byte, limb 0 = signed high byte)
#pragma unroll
		for (int k = 0; k < 3; k++) {
			const uint32_t sel = (uint32_t) k | ((uint32_t) (4 + k) << 4);
			const uint32_t lo = prmt((uint32_t) X[0], (uint32_t) X[1], sel), hi = prmt((uint32_t) X[2], (uint32_t) X[3], sel);
			w[2 - k][q] = prmt(lo, hi, 0x5410u);
		}
		asm("dp4a.s32.u32 %0, %1, %2, %0;" : "+r"(s0) : "r"(w[0][q]), "r"(0x01010101u));
		asm("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(s1) : "r"(w[1][q]), "r"(0x01010101u));
		asm("dp4a.u32.u32 %0, %1, %2, %0;" : "+r"(s2) : "r"(w[2][q]), "r"(0x01010101u));
	}
	uint32_t u = s1 | (s2 << 16); // block totals <= 32 * 255 < 2^16 each: one shuffle pair reduces both
	u += __shfl_xor_sync(0xffffffffu, u, 1);
	u += __shfl_xor_sync(0xffffffffu, u, 2);
	s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
	s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
#pragma unroll
	for (int k = 0; k < 3; k++) *reinterpret_cast<uint2*>(v.q + (size_t) k * v.n + (size_t) grp * 8) = make_uint2(w[k][0], w[k][1]);
	if ((grp & 3) == 0) v.meta[grp >> 2] = make_int4(s0, (int) (u & 0xFFFFu), (int) (u >> 16), (int) __float_as_uint(dx));
}

// what one lane holds of an activation block while it walks the R rows of a tile
struct XqBlock {
	uint4 a[3];   // limb k, the 16 elements of half hA of the block
	uint4 b[3];   // limb k, the other half
	int s[3];     // limb sums of the block
	float dx;     // block scale
	float sx;     // sum of the block's activations (formats with a per-block minimum)
};
// hA = (lane >> 2) & 1: lanes 0-3 of every group of eight read the first half of their block first, lanes 4-7 the second, so
// the eight 16-byte requests of a quarter-warp fall into eight different bank groups (blocks are 32 bytes apart).
__device__ __forceinline__ void xq_load(const XqView& v, int gb, int hA, XqBlock& o) {
#pragma unroll
	for (int k = 0; k < 3; k++) {
		const uint8_t* p = v.q + (size_t) k * v.n + (size_t) gb * 32;
		o.a[k] = *reinterpret_cast<const uint4*>(p + 16 * hA);
		o.b[k] = *reinterpret_cast<const uint4*>(p + 16 * (1 - hA));
	}
	const int4 m = v.meta[gb];
	o.s[0] = m.x; o.s[1] = m.y; o.s[2] = m.z;
	o.dx = __uint_as_float((uint32_t) m.w);
	o.sx = (__int2float_rn(m.x) * 65536.f + __int2float_rn((m.y << 8) + m.z)) * o.dx;
}

__device__ __forceinline__ int dp4a_us(uint32_t w, uint32_t x, int c) { // unsigned weights x signed limb
	int r;
	asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(x), "r"(c));
	return r;
}
__device__ __forceinline__ int dp4a_uu(uint32_t w, uint32_t x, int c) { // unsigned weights x unsigned limb
	int r;
	asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(x), "r"(c));
	return r;
}
// four weight words against the matching four words of each limb
__device__ __forceinline__ void idp16(const uint32_t (&w)[4], const uint4 (&x)[3], int (&acc)[3]) {
	const uint32_t x0[4] = {x[0].x, x[0].y, x[0].z, x[0].w}, x1[4] = {x[1].x, x[1].y, x[1].z, x[1].w}, x2[4] = {x[2].x, x[2].y, x[2].z, x[2].w};
#pragma unroll
	for (int i = 0; i < 4; i++) {
		acc[0] = dp4a_us(w[i], x0[i], acc[0]);
		acc[1] = dp4a_uu(w[i], x1[i], acc[1]);
		acc[2] = dp4a_uu(w[i], x2[i], acc[2]);
	}
}
// integer block sums -> fp32:  65536*a0 + 256*a1 + a2 (|a_k| < 2^21: the first conversion is exact, the second rounds 29 -> 24 bits
// of a term 2^-8 of the first)
__device__ __forceinline__ float idp_combine(const int (&acc)[3]) {
	return fmaf(__int2float_rn(acc[0]), 65536.f, __int2float_rn((acc[1] << 8) + acc[2]));
}

// ---- weight side: one 32-element block of one row, from a unit held in shared memory ------------------------------------
// block(unit, j, hA, xb, y): y += sum over block j of the unit of w * x.
template <int TYPE>
struct IdpFmt;

template <int BIAS>
__device__ __forceinline__ void idp_init(const XqBlock& xb, int (&acc)[3]) {
	acc[0] = -BIAS * xb.s[0]; acc[1] = -BIAS * xb.s[1]; acc[2] = -BIAS * xb.s[2];
}

// 8-bit quants stored biased (+128): Q8_0 (f16 scale per block) and Q8 (fixed scale 1/100)
template <>
struct IdpFmt<XALM_Q8_0> {
	static constexpr int UB = 272;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		const uint4 wa = *reinterpret_cast<const uint4*>(unit + 32 * j + 16 * hA);
		const uint4 wb = *reinterpret_cast<const uint4*>(unit + 32 * j + 16 * (1 - hA));
		const float d = f16_bits_to_f32(*reinterpret_cast<const uint16_t*>(unit + 256 + 2 * j));
		int acc[3];
		idp_init<128>(xb, acc);
		const uint32_t a[4] = {wa.x, wa.y, wa.z, wa.w}, b[4] = {wb.x, wb.y, wb.z, wb.w};
		idp16(a, xb.a, acc);
		idp16(b, xb.b, acc);
		y = fmaf(idp_combine(acc), d * xb.dx, y);
	}
};
template <>
struct IdpFmt<XALM_Q8> {
	static constexpr int UB = 256;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		const uint4 wa = *reinterpret_cast<const uint4*>(unit + 32 * j + 16 * hA);
		const uint4 wb = *reinterpret_cast<const uint4*>(unit + 32 * j + 16 * (1 - hA));
		int acc[3];
		idp_init<128>(xb, acc);
		const uint32_t a[4] = {wa.x, wa.y, wa.z, wa.w}, b[4] = {wb.x, wb.y, wb.z, wb.w};
		idp16(a, xb.a, acc);
		idp16(b, xb.b, acc);
		y = fmaf(idp_combine(acc), (1.f / 100.f) * xb.dx, y); // types.h:423-424
	}
};
// 4-bit: byte i of the block's 16 = {low nibble: element i, high nibble: element 16+i} (quants.py:302-313).  The half a lane
// pairs with its first activation load is picked with a per-lane shift, so no select is needed.
template <int BIAS, bool HAS_MIN, int SC_OFF, int SC_STRIDE>
__device__ __forceinline__ void idp_block4(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
	const uint4 wq = *reinterpret_cast<const uint4*>(unit + 16 * j);
	const uint32_t w[4] = {wq.x, wq.y, wq.z, wq.w};
	const int shA = 4 * hA, shB = 4 - shA;
	uint32_t a[4], b[4];
#pragma unroll
	for (int i = 0; i < 4; i++) {
		a[i] = (w[i] >> shA) & 0x0F0F0F0Fu;
		b[i] = (w[i] >> shB) & 0x0F0F0F0Fu;
	}
	int acc[3];
	idp_init<BIAS>(xb, acc);
	idp16(a, xb.a, acc);
	idp16(b, xb.b, acc);
	if (HAS_MIN) {
		const uint32_t dm = *reinterpret_cast<const uint32_t*>(unit + SC_OFF + SC_STRIDE * j);
		const float d = f16_bits_to_f32((uint16_t) (dm & 0xFFFF)), m = f16_bits_to_f32((uint16_t) (dm >> 16));
		y = fmaf(idp_combine(acc), d * xb.dx, y);
		y = fmaf(m, xb.sx, y);
	} else {
		const float d = f16_bits_to_f32(*reinterpret_cast<const uint16_t*>(unit + SC_OFF + SC_STRIDE * j));
		y = fmaf(idp_combine(acc), d * xb.dx, y);
	}
}
template <>
struct IdpFmt<XALM_Q4_0> { // d * (q - 8)
	static constexpr int UB = 144;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		idp_block4<8, false, 128, 2>(unit, j, hA, xb, y);
	}
};
template <>
struct IdpFmt<XALM_Q4_1> { // d * q + m (quants.py:337-350)
	static constexpr int UB = 160;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		idp_block4<0, true, 128, 4>(unit, j, hA, xb, y);
	}
};
// 5-bit: fifth bits in a u32 per block, bit e -> element e (quants.py:376-393, 419-438)
template <int BIAS, bool HAS_MIN, int SC_OFF, int SC_STRIDE, int QH_OFF>
__device__ __forceinline__ void idp_block5(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
	const uint4 wq = *reinterpret_cast<const uint4*>(unit + 16 * j);
	const uint32_t qh = *reinterpret_cast<const uint32_t*>(unit + QH_OFF + 4 * j);
	const uint32_t w[4] = {wq.x, wq.y, wq.z, wq.w};
	const int shA = 4 * hA, shB = 4 - shA;
	const uint32_t hbA = qh >> (16 * hA), hbB = qh >> (16 - 16 * hA); // the 16 fifth bits of each half in the low half-word
	uint32_t a[4], b[4];
#pragma unroll
	for (int i = 0; i < 4; i++) {
		a[i] = ((w[i] >> shA) & 0x0F0F0F0Fu) | ((((hbA >> (4 * i)) & 0xFu) * 0x02040810u) & 0x10101010u);
		b[i] = ((w[i] >> shB) & 0x0F0F0F0Fu) | ((((hbB >> (4 * i)) & 0xFu) * 0x02040810u) & 0x10101010u);
	}
	int acc[3];
	idp_init<BIAS>(xb, acc);
	idp16(a, xb.a, acc);
	idp16(b, xb.b, acc);
	if (HAS_MIN) {
		const uint32_t dm = *reinterpret_cast<const uint32_t*>(unit + SC_OFF + SC_STRIDE * j);
		const float d = f16_bits_to_f32((uint16_t) (dm & 0xFFFF)), m = f16_bits_to_f32((uint16_t) (dm >> 16));
		y = fmaf(idp_combine(acc), d * xb.dx, y);
		y = fmaf(m, xb.sx, y);
	} else {
		const float d = f16_bits_to_f32(*reinterpret_cast<const uint16_t*>(unit + SC_OFF + SC_STRIDE * j));
		y = fmaf(idp_combine(acc), d * xb.dx, y);
	}
}
template <>
struct IdpFmt<XALM_Q5_0> { // d * ((ql | qh << 4) - 16): unit = 128 quants, 16 scales, 32 high bits
	static constexpr int UB = 176;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		idp_block5<16, false, 128, 2, 144>(unit, j, hA, xb, y);
	}
};
template <>
struct IdpFmt<XALM_Q5_1> { // d * (ql | qh << 4) + m: unit = 128 quants, 32 {d,m}, 32 high bits
	static constexpr int UB = 192;
	static __device__ __forceinline__ void block(const uint8_t* unit, int j, int hA, const XqBlock& xb, float& y) {
		idp_block5<0, true, 128, 4, 160>(unit, j, hA, xb, y);
	}
};

__host__ __device__ inline bool idp_supported(int t) {
	return t == XALM_Q8_0 || t == XALM_Q8 || t == XALM_Q4_0 || t == XALM_Q4_1 || t == XALM_Q5_0 || t == XALM_Q5_1;
}

} // namespace xalm
