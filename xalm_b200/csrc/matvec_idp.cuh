// matvec_idp.cuh — the TMA decode matvec (matvec_tma.cuh) for the integer weight formats, on the integer-dot core (idp.cuh).
//
// Same skeleton as matvec_tma_kernel — persistent CTAs, a producer warp streaming rows into an mbarrier ring with
// cp.async.bulk, 8 consumer warps, rmsnorm prologue, QKV / GLU / residual / store epilogues, PDL, the fused tensor-parallel
// exchange — but the consumers work in integers: the activations are staged ONCE per CTA as block floating point (three int8
// limbs per element + one power-of-two scale per 32), and a 32-weight block costs 24 dp4a plus ~8 finishing instructions
// instead of 64-136 PRMT / FADD2 / FFMA2.  Measured on the float core (profiles/r1_matvec_tma_q8_0_w13.md): q8_0 issue /
// latency-bound at 75 % of HBM peak (3.9 issue slots per weight with its per-tile reductions), q4_0..q5_1 ALU-bound at 26-29 %.
//
// Mapping: a tile is 8 rows, a ring stage 8 rows x 16 units (4096 elements).  Warp (kw, rw) = K-slice kw of 4 (32 blocks of 32
// elements: one block per lane) x row group rw of 2 (4 rows).  Per stage a lane loads its activation block once (7 shared
// loads) and walks its 4 rows.  Lane sums are reduced with a 6-shuffle transposed butterfly; K-slices are combined through
// shared memory in a fixed order (bit-reproducible run to run); a rotating warp runs the epilogue.
#pragma once
#include "idp.cuh"
#include "matvec_tma.cuh"

namespace xalm {

constexpr int IDP_KW = 4, IDP_RW = 2, IDP_R = 4, IDP_RC = IDP_RW * IDP_R, IDP_U = 16;
// Partial sums of the K-slice warps are handed to the tile's reducer warp through PB buffers, each with an mbarrier the 8 consumer
// warps arrive on: nobody but the reducer ever waits (a CTA-wide bar.sync per tile was 26 % of all stall cycles, profiles/r2_idp_ncu.md).
// A buffer is reused PB tiles later; a warp cannot run more than NS stages (<= NS tiles) ahead of the slowest warp of its group (ring).
__host__ __device__ inline int idp_pb(int NS) { return NS + 2 < 8 ? 8 : NS + 2; }
constexpr int IDP_MP = 4; // staging passes of a norm-fused kernel: 8 elements x 256 lanes x 4 = n <= 8192

__host__ __device__ inline size_t idp_smem_bytes(int type, int n, int NS, int NG = 1) {
	size_t s = (xq_bytes(n) + 127) / 128 * 128;
	s += (size_t) NS * IDP_RC * IDP_U * unit_bytes(type);
	s += (size_t) idp_pb(NS) * NG * IDP_KW * IDP_RC * sizeof(float); // partials, idp_pb(NS) tiles deep
	s += (2 * (size_t) NS + idp_pb(NS)) * sizeof(uint64_t); // full / empty / partial barriers
	s += 16 * sizeof(float);                    // reduction scratch
	return s + 128;
}

struct IdpArgs {
	MatvecArgs a;   // a.w.p0 = unit-interleaved rows, a.w.s0 = row stride in bytes
	int NS;         // ring stages
	int n_tiles;    // virtual rows / 8
};

// NG = consumer groups of 8 warps.  NG = 1: two CTAs per SM, each with its own staged activations and a 2-stage ring.  NG = 2: ONE CTA
// per SM — the activations are fetched and quantised once per SM instead of twice (the broadcast read of x by every CTA is an L2
// hot spot: 1-1.6 us) and the shared memory that bought goes to the ring (6 stages instead of 2 x 2), so the producer keeps HBM busy
// through the dependency wait + staging of the consumers.  The two groups take alternate ring stages.
template <int TYPE, bool NORM, int NG>
// <= 96 registers: the register file is per scheduler (16 K each); 17 warps (or two CTAs of 9) put 5 warps on one of them: 16384 / 5 / 32 = 102
__global__ void __maxnreg__(96) matvec_idp_kernel(const IdpArgs ta) {
	using F = IdpFmt<TYPE>;
	constexpr int KW = IDP_KW, R = IDP_R, RC = IDP_RC, U = IDP_U, UB = F::UB;
	constexpr int NCW = NG * TMA_NW, NT = NCW * 32; // consumer warps / threads
	auto cbar = [] { if (NG == 1) asm volatile("bar.sync 1, 256;" ::: "memory"); else asm volatile("bar.sync 1, 512;" ::: "memory"); };
	constexpr int ROW_STAGE = U * UB;
	constexpr int SLOT = RC * ROW_STAGE;
	const MatvecArgs& a = ta.a;
	const int NS = ta.NS, PB = idp_pb(ta.NS);
	const int n = a.n, nu = n / 256;
	const int kranges = (nu + U - 1) / U;

	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* xq_base = smem;
	uint8_t* ring = smem + (xq_bytes(n) + 127) / 128 * 128;
	float* part = reinterpret_cast<float*>(ring + (size_t) NS * SLOT);
	float* s_red = part + PB * NG * KW * RC;
	uint64_t* full = reinterpret_cast<uint64_t*>(s_red + 16);
	uint64_t* empty = full + NS;
	uint64_t* pbar = empty + NS;

	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; s++) {
			mbar_init(&full[s], 1);
			mbar_init(&empty[s], TMA_NW);
		}
		for (int s = 0; s < PB; s++) mbar_init(&pbar[s], (kranges >= NG ? NG : 1) * TMA_NW); // the warps that hold a piece of a tile
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
				const int row0 = ((int) blockIdx.x + tt * (int) gridDim.x) * RC;
				for (int kr = 0; kr < kranges; kr++) {
					mbar_wait(&empty[slot], phase ^ 1);
					const int u0 = kr * U;
					const int un = min(U, nu - u0);
					const uint32_t bytes = (uint32_t) un * UB;
					mbar_expect_tx(&full[slot], bytes * RC);
					uint8_t* dst = ring + (size_t) slot * SLOT;
					if (un == nu && nu == U && a.w.s0 == (size_t) ROW_STAGE) {
						// the stage spans whole rows and a tile's rows are neighbours in memory: ONE copy per run of rows instead of
						// one per row (the copy engine is bound by the NUMBER of bulk copies when they are a few KB each: q4_0 rows of
						// 2304 bytes streamed no faster than q8_0 rows of 4352, profiles/r2_decode_timeline.md)
						if (a.epi == EPI_GLU) { // rows [0, RC/2) are W1[o0..], rows [RC/2, RC) are W3[o0..]
							const int o0 = row0 / 2;
							bulk_g2s(dst, a.w.p0 + (size_t) o0 * a.w.s0, bytes * (RC / 2), &full[slot]);
							bulk_g2s(dst + (size_t) (RC / 2) * ROW_STAGE, a.w.p0 + (size_t) (a.glu_off + o0) * a.w.s0, bytes * (RC / 2), &full[slot]);
						} else {
							bulk_g2s(dst, a.w.p0 + (size_t) row0 * a.w.s0, bytes * RC, &full[slot]);
						}
					} else {
#pragma unroll
						for (int r = 0; r < RC; r++) {
							const int pr = phys_row(a, row0, r, RC);
							bulk_g2s(dst + (size_t) r * ROW_STAGE, a.w.p0 + (size_t) pr * a.w.s0 + (size_t) u0 * UB, bytes, &full[slot]);
						}
					}
					if (++slot == NS) { slot = 0; phase ^= 1; }
				}
			}
			prefetch_tail(a, true);
		}
		return;
	}

	// ===================== consumers =====================
	// Staging: lane t of the CTA owns the 8-element groups t, t + 256, ... (four lanes per 32-element block).  The rmsnorm weights do
	// not depend on the previous kernel: request them before the dependency wait (host: NORM only with n <= 8192 = IDP_MP passes).
	const int tid = threadIdx.x;
	const int ngrp = n / 8;
	constexpr int MP = IDP_MP / NG; // staging passes of a norm-fused kernel (n <= 8192)
	uint4 gw[NORM ? MP : 1][2];
	if (NORM) {
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = p * NT + tid;
			if (grp < ngrp) load_norm8(a.norm_w, a.norm_type, grp, gw[p]);
		}
	}
	pdl_wait(); // activations / KV ring of earlier kernels are visible from here on
	tl_mark(tl, 2);
	if (a.epi == EPI_QKV && blockIdx.x == 0 && a.step->kv_sink > 0) rotate_sinks(a, a.k_cache, a.step->kv_sink, tid, NT);
	if (NORM && a.n_recv) tp_receive(a, tid, NT);
	// ---- stage activations: xq = quantise(NORM ? x * scale * g : x) ----
	const XqView xv = xq_view(xq_base, n);
	if (NORM) {
		float xr[MP][8];
		float ss = 0.f;
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = p * NT + tid;
			if (grp < ngrp) load_x8(a, grp, NORM && a.n_recv, xr[p]);
		}
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = p * NT + tid;
			if (grp < ngrp) {
#pragma unroll
				for (int e = 0; e < 8; e++) ss += xr[p][e] * xr[p][e];
			}
		}
		ss = warp_sum(ss);
		if (tl >= 0) tl_begin(600 + a.epi); // event: x arrived
		if (lane == 0) s_red[warp] = ss;
		// The staged vector is x * g; the scalar 1/rms is applied to the row sums in the epilogue (y = scale * sum w * (x * g)), so
		// the staging does not wait for the CTA-wide sum of squares: one barrier instead of two between x arriving and the first tile
#pragma unroll
		for (int p = 0; p < MP; p++) {
			const int grp = p * NT + tid;
			if (grp < ngrp) { // (warp-uniform: n % 256 == 0)
#pragma unroll
				for (int e = 0; e < 8; e++) xr[p][e] = xr[p][e] * norm_weight(gw[p], a.norm_type, e); // infer.cpp:233-235 without the scalar
				xq_store_group8(xv, grp, xr[p]);
			}
		}
	} else {
		constexpr int UNR = 4; // groups in flight per lane (n = 14336 on 512 threads: one round of loads)
		for (int base = 0; base < ngrp; base += UNR * NT) {
			float xr[UNR][8];
#pragma unroll
			for (int p = 0; p < UNR; p++) {
				const int grp = base + p * NT + tid;
				if (grp < ngrp) load_x8(a, grp, NORM && a.n_recv, xr[p]);
			}
#pragma unroll
			for (int p = 0; p < UNR; p++) {
				const int grp = base + p * NT + tid;
				if (grp < ngrp) xq_store_group8(xv, grp, xr[p]);
			}
		}
	}
	cbar();
	float nscale = 1.f; // 1/rms of the input (infer.cpp:229-232), applied to the row sums
	if (NORM) {
		float tot = 0.f;
#pragma unroll
		for (int i = 0; i < NCW; i++) tot += s_red[i];
		nscale = 1.0f / sqrtf(tot / (float) n + a.norm_eps);
	}
	if (tl >= 0) tl_begin(500 + a.epi); // timeline event: activations staged

	const int cg = warp / TMA_NW, wl = warp % TMA_NW; // consumer group, warp within it
	const int kw = wl % KW, rw = wl / KW;
	const int hA = (lane >> 2) & 1;
	const bool both = kranges >= NG; // every group holds a piece of every tile (else tiles alternate between the groups)
	int slot = 0, phase = 0, gi = 0; // gi: stage counter of the CTA; group gi % NG takes it
	int pb_next = 0, pph_next = 0;   // partial buffer of the tile and the phase of its barrier (tt % PB, (tt / PB) & 1 without the divisions)
	for (int tt = 0; tt < my_tiles; tt++) {
		const int pb = pb_next, pph = pph_next;
		if (++pb_next == PB) { pb_next = 0; pph_next ^= 1; }
		const int row0 = ((int) blockIdx.x + tt * (int) gridDim.x) * RC;
		const int g_last = (gi + kranges - 1) % NG; // the group that takes the tile's last stage supplies the reducer
		const bool mine = both || (gi % NG) == cg;
		const bool reducer = cg == g_last && wl == ((tt / (both ? 1 : NG)) % TMA_NW);
		float xold = 0.f; // residual: the reducer warp fetches the old activation now, so its epilogue does not sit on an L2 round trip
		if (a.epi == EPI_RESIDUAL && reducer && lane < RC && row0 + lane < a.d) xold = a.out[row0 + lane];
		float y[R];
#pragma unroll
		for (int r = 0; r < R; r++) y[r] = 0.f;
		for (int kr = 0; kr < kranges; kr++, gi++) {
			if (NG == 1 || (gi % NG) == cg) {
				const int u0 = kr * U;
				const int nb = 8 * min(U, nu - u0); // blocks per row in this stage
				const int b = kw * 32 + lane;
				mbar_wait(&full[slot], phase);
				if (b < nb) {
					XqBlock xb;
					xq_load(xv, u0 * 8 + b, hA, xb);
					const uint8_t* unit = ring + (size_t) slot * SLOT + (size_t) (rw * R) * ROW_STAGE + (size_t) (b >> 3) * UB;
#pragma unroll
					for (int r = 0; r < R; r++) F::block(unit + (size_t) r * ROW_STAGE, b & 7, hA, xb, y[r]);
				}
				__syncwarp();
				if (lane == 0) mbar_arrive(&empty[slot]);
			}
			if (++slot == NS) { slot = 0; phase ^= 1; }
		}
		if (!mine) continue;
		if (tl >= 0 && tt < 4) tl_begin(510 + 10 * tt + a.epi); // timeline event: tile tt multiplied
		// ---- lanes -> one sum per row (transposed butterfly: 6 shuffles for 4 rows), K-slices -> shared memory (fixed order) ----
		{
			const bool b4 = lane & 16, b3 = lane & 8;
			float k0 = b4 ? y[2] : y[0], k1 = b4 ? y[3] : y[1];
			const float s0 = b4 ? y[0] : y[2], s1 = b4 ? y[1] : y[3];
			k0 += __shfl_xor_sync(0xffffffffu, s0, 16);
			k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
			float k = b3 ? k1 : k0;
			const float s = b3 ? k0 : k1;
			k += __shfl_xor_sync(0xffffffffu, s, 8);
			k += __shfl_xor_sync(0xffffffffu, k, 4);
			k += __shfl_xor_sync(0xffffffffu, k, 2);
			k += __shfl_xor_sync(0xffffffffu, k, 1);
			if ((lane & 7) == 0) part[(pb * NG + cg) * (KW * RC) + kw * RC + rw * R + (b4 ? 2 : 0) + (b3 ? 1 : 0)] = k;
		}
		__syncwarp();
		if (lane == 0) mbar_arrive(&pbar[pb]); // (release: this warp's partial sums are visible to whoever completes the wait)
		if (reducer) { // rotating reducer: lane i owns row i of the tile
			mbar_wait(&pbar[pb], pph);
			float yv = 0.f;
			if (lane < RC) {
#pragma unroll
				for (int g = 0; g < NG; g++) {
					if (!both && g != cg) continue;
					const float* pt = part + (pb * NG + g) * (KW * RC);
#pragma unroll
					for (int k = 0; k < KW; k++) yv += pt[k * RC + lane];
				}
			}
			if (NORM) yv *= nscale;
			row_epilogue<RC>(a, row0, lane, yv, xold);
		}
	}
	tl_mark(tl, 3);
}

} // namespace xalm
