// xalm_cuda.cu — implementation of the C ABI in include/xalm_cuda.h: model handle, sharded upload + repack, the
// per-token kernel sequence (captured once as a CUDA graph with programmatic dependent launches), NCCL plumbing
// for tensor parallelism, and the op-level entry points the parity tests call.
//
// Per token (Model::_forward_cpu, infer.cpp:604-638 / Block::_block_cpu, infer.cpp:365-496):
//   embed                                   x = dequant(embed[token])
//   per layer  matvec[norm -> QKV -> rope]  q fp32, k/v fp16 -> KV ring   (+ sink re-rotation)
//              attn_decode                  xb2 = softmax(q k^T / sqrt(hd)) v      (split-K, GQA)
//              matvec[Wo, residual]         x += Wo xb2                    (TP: partial -> allreduce -> add)
//              matvec[norm -> W1|W3 -> GLU] hb = act(W1 xb) * (W3 xb)
//              matvec[W2, residual]         x += W2 hb                     (TP: partial -> allreduce -> add)
//   matvec[norm -> classifier]              logits                         (skipped in HYDRATE_KV_CACHE mode)
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "attention.cuh"
#include "matvec.cuh"
#include "matvec_tma.cuh"
#include "matvec_idp.cuh"
#include "matvec_mma.cuh"
#include "nccl_api.h"
#include "prefill.h"

namespace xalm {

thread_local std::string g_last_error;

int set_error(int status, const char* fmt, ...) {
	char buf[1024];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof buf, fmt, ap);
	va_end(ap);
	g_last_error = buf;
	return status;
}

// ---------------------------------------------------------------------------------------------------------
// tuning knobs (xalm_cuda_tune): integers looked up by name, so GPU sweeps need no recompilation
// ---------------------------------------------------------------------------------------------------------
static std::map<std::string, int>& tuning() {
	static std::map<std::string, int> t = {
	    {"pdl", 1},          // programmatic dependent launch between the kernels of a token
	    {"graph", 1},        // replay a captured CUDA graph per token
	    {"attn_splits", 0},  // 0 = auto (~1 CTA per SM, at most 32 splits per kv head)
	    {"attn_min_split", 128},
	    {"tma", 1},          // stream weights with cp.async.bulk into a shared-memory ring (matvec_tma.cuh)
	    {"idp", 1},          // integer weight formats: integer-dot consumers (matvec_idp.cuh) instead of the float ones
	    {"tma_smem_kb", 100}, // shared-memory budget per CTA for the TMA kernel (two kernels co-reside under PDL)
	    {"tma_xstage_max_kb", 32}, // rows longer than this (in fp32 bytes) are not staged in smem when there is no norm
	    {"tma_ns_max", 4},   // most ring stages
	    {"tma_ctas_per_sm", 2},
	    {"tma_short_rows", 1}, // rows of <= 64 pieces without a norm prologue: 16-row tiles with 1-2 K-slices (all lanes busy)
	    {"tp_fused", 1},     // tensor parallel: fuse the two per-layer exchanges into the matvec kernels (push over NVLink + receive in the next prologue)
	    {"idp_per_sm", 2},
	    {"mma", 2},         // integer formats on the tensor-core matvec (fragment tiles + mma.sync int8, matvec_mma.cuh): 0 = never (unit layout + dp4a), 1 = all six, 2 = the 4/5-bit formats, and the 8-bit ones under tensor parallelism (measured on one GPU: q4_0 1.68 vs 1.86 ms/token; q8_0 1.90 vs 1.86)
    {"idp_ng", 0},      // consumer groups per CTA of the integer-dot matvec: 0 = by format, 2 = one 17-warp CTA per SM, 1 = two 9-warp CTAs
	    {"tail_prefetch_mb", 8}, // each decode kernel pulls this many MB of the NEXT kernel's first weights into L2 once its own loads are issued
	    {"prefill_split", 3}, // batched prefill operand precision: 1 = fp16 x fp16 (fastest; logits drift ~4e-2 over 32 layers), 2 = hi+lo fp16
	                          // activations, 3 = hi+lo on activations, weights and attention operands (default: logits within ~1e-3 of the decode path)
	};
	return t;
}
static int tune(const char* k) {
	const char* e = nullptr;
	std::string env = std::string("XALM_") + k;
	for (auto& ch : env) ch = (char) toupper(ch);
	if ((e = getenv(env.c_str()))) return atoi(e);
	return tuning()[k];
}

// ---------------------------------------------------------------------------------------------------------
// launch helper (optionally with the programmatic-stream-serialisation attribute = PDL)
// ---------------------------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
static cudaError_t launch_smem(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args&&... args) {
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid;
	cfg.blockDim = block;
	cfg.dynamicSmemBytes = smem;
	cfg.stream = stream;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
	cfg.attrs = attr;
	cfg.numAttrs = 1;
	return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

template <typename... KArgs, typename... Args>
static cudaError_t launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, bool pdl, Args&&... args) {
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid;
	cfg.blockDim = block;
	cfg.dynamicSmemBytes = 0;
	cfg.stream = stream;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
	cfg.attrs = attr;
	cfg.numAttrs = 1;
	return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---------------------------------------------------------------------------------------------------------
// matvec dispatch
// ---------------------------------------------------------------------------------------------------------
struct MvCfg {
	int R, KS, NW;
};
static const MvCfg CFG_A = {4, 1, 4}; // many rows: 16 virtual rows per 128-thread CTA
static const MvCfg CFG_B = {2, 4, 8}; // few rows (Wo, W2): 4 rows per CTA, K split over 4 warps

template <int TYPE>
static cudaError_t launch_matvec_typed(const MatvecArgs& a, const MvCfg& c, bool norm, cudaStream_t s, bool pdl) {
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	if (c.KS == 1) {
		const int rows_per_cta = (CFG_A.NW / CFG_A.KS) * CFG_A.R;
		dim3 grid((vrows + rows_per_cta - 1) / rows_per_cta), block(CFG_A.NW * 32);
		if (norm) return launch(matvec_kernel<TYPE, 4, 1, 4, true>, grid, block, s, pdl, a);
		return launch(matvec_kernel<TYPE, 4, 1, 4, false>, grid, block, s, pdl, a);
	}
	const int rows_per_cta = (CFG_B.NW / CFG_B.KS) * CFG_B.R;
	dim3 grid((vrows + rows_per_cta - 1) / rows_per_cta), block(CFG_B.NW * 32);
	if (norm) return launch(matvec_kernel<TYPE, 2, 4, 8, true>, grid, block, s, pdl, a);
	return launch(matvec_kernel<TYPE, 2, 4, 8, false>, grid, block, s, pdl, a);
}

// ---------------------------------------------------------------------------------------------------------
// TMA matvec dispatch (matvec_tma.cuh)
// ---------------------------------------------------------------------------------------------------------
static int current_device() {
	int dev = 0;
	cudaGetDevice(&dev);
	return dev;
}
// SM count of the CURRENT device (function attributes, occupancy and SM counts are per device: a handle may live on any GPU)
static int num_sms() {
	static std::map<int, int> cache;
	const int dev = current_device();
	auto it = cache.find(dev);
	if (it == cache.end()) {
		int n = 148;
		cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
		it = cache.emplace(dev, n).first;
	}
	return it->second;
}
// opt a kernel into > 48 KB of dynamic shared memory, once per (kernel, device)
template <typename K>
static cudaError_t ensure_smem_attr(K kern, int bytes) {
	static std::map<std::pair<const void*, int>, bool> done; // (kernel, device): one instantiation serves every kernel of a signature
	const std::pair<const void*, int> key(reinterpret_cast<const void*>(kern), current_device());
	if (done.count(key)) return cudaSuccess;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
	if (e == cudaSuccess) done[key] = true;
	return e;
}

template <int TYPE, int RC, int KW, bool NORM>
static cudaError_t launch_tma_inst(const TmaArgs& ta, int max_ctas_per_sm, size_t smem, cudaStream_t s, bool pdl) {
	static std::map<std::pair<int, size_t>, int> occ_cache; // (device, smem) -> resident CTAs per SM
	auto kern = matvec_tma_kernel<TYPE, RC, KW, NORM>;
	{
		cudaError_t e = ensure_smem_attr(kern, 200 * 1024);
		if (e != cudaSuccess) return e;
	}
	// persistent grid: exactly as many CTAs as can be resident at once (a second wave would serialise behind the first)
	const std::pair<int, size_t> key(current_device(), smem);
	auto it = occ_cache.find(key);
	if (it == occ_cache.end()) {
		int occ = 1;
		cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, (TMA_NW + 1) * 32, smem);
		if (e != cudaSuccess) return e;
		it = occ_cache.emplace(key, occ < 1 ? 1 : occ).first;
	}
	int per_sm = it->second < max_ctas_per_sm ? it->second : max_ctas_per_sm;
	int grid = num_sms() * per_sm;
	if (grid > ta.n_tiles) grid = ta.n_tiles;
	return launch_smem(kern, dim3(grid), dim3((TMA_NW + 1) * 32), smem, s, pdl, ta);
}

template <int TYPE>
static cudaError_t launch_tma_typed(const TmaArgs& ta, int RC, int KW, bool norm, int grid, size_t smem, cudaStream_t s, bool pdl) {
#define XALM_TMA_CASE(rc, kw)                                                                     \
	if (RC == rc && KW == kw)                                                                     \
		return norm ? launch_tma_inst<TYPE, rc, kw, true>(ta, grid, smem, s, pdl)                 \
		            : launch_tma_inst<TYPE, rc, kw, false>(ta, grid, smem, s, pdl);
	XALM_TMA_CASE(8, 8)
	XALM_TMA_CASE(8, 4)
#undef XALM_TMA_CASE
	// short rows (the row-split Wo / W2 under tensor parallelism: n = q_dim / P): 16-row tiles, one or two K-slices, so every lane
	// of a warp has a piece to work on
	if (!norm && RC == 16 && KW == 2) return launch_tma_inst<TYPE, 16, 2, false>(ta, grid, smem, s, pdl);
	if (!norm && RC == 16 && KW == 1) return launch_tma_inst<TYPE, 16, 1, false>(ta, grid, smem, s, pdl);
	return cudaErrorInvalidValue;
}

static int pieces_per_unit(int t) {
	switch (t) {
		case XALM_F32: return 64;
		case XALM_F16: case XALM_BF16: return 32;
		case XALM_Q4_0: case XALM_Q4_1: case XALM_Q5_0: case XALM_Q5_1: return 8;
		default: return 16;
	}
}

// can this matrix go down the TMA path?
static bool tma_eligible(const WMat& w, int n) {
	if (!tune("tma")) return false;
	if (!unit_bytes(w.type) || n % 256) return false;
	if ((w.type == XALM_F8_E4M3 || w.type == XALM_F8_E5M2) && (w.flags & WMAT_FP8_NONFINITE)) return false;
	return true;
}

static int launch_matvec_tma(const MatvecArgs& a, cudaStream_t s, bool pdl) {
	const int t = a.w.type;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	const int ppu = pieces_per_unit(t);
	const int nu = a.n / 256;
	int RC = 8, KW = 8;
	if (ppu == 8) KW = 4;                 // 4/5-bit: 8 pieces per unit -> fewer K-slices
	if (nu * ppu / 8 < 32) KW = 4;        // short rows: keep 32 lanes busy
	if (a.norm_w == nullptr && vrows % 16 == 0 && tune("tma_short_rows")) {
		if (nu * ppu <= 32) { RC = 16; KW = 1; }
		else if (nu * ppu <= 64) { RC = 16; KW = 2; }
	}
	if (vrows % RC) return -1;
	const int ub = unit_bytes(t);
	const size_t budget = (size_t) tune("tma_smem_kb") * 1024;
	// long rows without a norm prologue (W2): do not spend shared memory on x, read it through L1 with 8-row reuse
	const bool x_global = a.norm_w == nullptr && RC == 8 && (size_t) a.n * sizeof(float) > (size_t) tune("tma_xstage_max_kb") * 1024;
	const int n_stage = x_global ? 0 : a.n;
	const size_t fixed = tma_smem_bytes(t, n_stage, RC, 0, 0) + 2 * 4 * sizeof(uint64_t);
	if (fixed + 2 * (size_t) RC * ub > 200 * 1024) return -1; // activations do not fit: LDG path
	// stage: U units per row, chosen to keep >= 32 pieces per K-slice, as large as the budget allows with >= 2 stages
	int umin = (32 * KW + ppu - 1) / ppu;
	if (umin > nu) umin = nu;
	int U = umin, NS = 2;
	size_t best = 0;
	for (int u = umin; u <= nu && u <= 64; u++) {
		if (u != nu && (u % umin)) continue;
		const size_t stage = (size_t) RC * u * ub;
		size_t avail = budget > fixed ? budget - fixed : 0;
		int ns = (int) (avail / stage);
		if (ns > tune("tma_ns_max")) ns = tune("tma_ns_max");
		if (ns < 2) continue;
		if ((size_t) ns * stage > best) { best = (size_t) ns * stage; U = u; NS = ns; }
	}
	if (best == 0) { U = umin; NS = 2; }
	const size_t smem = tma_smem_bytes(t, n_stage, RC, U, NS);
	if (smem > 200 * 1024) return -1;
	TmaArgs ta;
	ta.a = a;
	ta.U = U; ta.NS = NS;
	ta.x_global = x_global ? 1 : 0;
	ta.n_tiles = (vrows + RC - 1) / RC;
	const int grid = tune("tma_ctas_per_sm"); // upper bound on resident CTAs per SM; the launcher asks the occupancy API
	const bool norm = a.norm_w != nullptr;
	cudaError_t e;
	switch (t) {
		case XALM_F32: e = launch_tma_typed<XALM_F32>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_F16: e = launch_tma_typed<XALM_F16>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_BF16: e = launch_tma_typed<XALM_BF16>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_F8_E4M3: e = launch_tma_typed<XALM_F8_E4M3>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_F8_E5M2: e = launch_tma_typed<XALM_F8_E5M2>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q8: e = launch_tma_typed<XALM_Q8>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q8_0: e = launch_tma_typed<XALM_Q8_0>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q4_0: e = launch_tma_typed<XALM_Q4_0>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q4_1: e = launch_tma_typed<XALM_Q4_1>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q5_0: e = launch_tma_typed<XALM_Q5_0>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		case XALM_Q5_1: e = launch_tma_typed<XALM_Q5_1>(ta, RC, KW, norm, grid, smem, s, pdl); break;
		default: return -1;
	}
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "matvec (tma) launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// integer-dot matvec dispatch (matvec_idp.cuh): the integer weight formats in unit layout
// ---------------------------------------------------------------------------------------------------------
template <int TYPE, bool NORM, int NG>
static cudaError_t launch_idp_inst(const IdpArgs& ta, size_t smem, int max_ctas_per_sm, cudaStream_t s, bool pdl) {
	static std::map<std::pair<int, size_t>, int> occ_cache;
	auto kern = matvec_idp_kernel<TYPE, NORM, NG>;
	constexpr int threads = (NG * TMA_NW + 1) * 32;
	cudaError_t e = ensure_smem_attr(kern, 227 * 1024);
	if (e != cudaSuccess) return e;
	const std::pair<int, size_t> key(current_device(), smem);
	auto it = occ_cache.find(key);
	if (it == occ_cache.end()) {
		int occ = 1;
		e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem);
		if (e != cudaSuccess) return e;
		it = occ_cache.emplace(key, occ < 1 ? 1 : occ).first;
	}
	const int per_sm = it->second < max_ctas_per_sm ? it->second : max_ctas_per_sm;
	int grid = num_sms() * per_sm; // persistent: exactly the CTAs that can be resident at once
	if (grid > ta.n_tiles) grid = ta.n_tiles;
	return launch_smem(kern, dim3(grid), dim3(threads), smem, s, pdl, ta);
}
template <int TYPE>
static cudaError_t launch_idp_typed(const IdpArgs& ta, bool norm, int ng, size_t smem, int per_sm, cudaStream_t s, bool pdl) {
	if (ng == 2) return norm ? launch_idp_inst<TYPE, true, 2>(ta, smem, 1, s, pdl) : launch_idp_inst<TYPE, false, 2>(ta, smem, 1, s, pdl);
	return norm ? launch_idp_inst<TYPE, true, 1>(ta, smem, per_sm, s, pdl) : launch_idp_inst<TYPE, false, 1>(ta, smem, per_sm, s, pdl);
}
// returns -1 when the matrix cannot go down this path (the caller falls back to the float kernels)
static int launch_matvec_idp(const MatvecArgs& a, cudaStream_t s, bool pdl) {
	const int t = a.w.type;
	if (!tune("idp") || !tune("tma") || !idp_supported(t)) return -1;
	TypeInfo ti;
	type_info(t, &ti);
	if (ti.block > 1 ? !a.w.layout_units : a.w.s0 != (size_t) a.n) return -1;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	if (a.n % 256 || vrows % IDP_RC) return -1;
	const bool norm = a.norm_w != nullptr;
	if (norm && a.n > 8192) return -1; // the norm-fused staging keeps its 8-element groups in registers (IDP_MP passes)
	int NS = 0, per_sm = 1, ng = tune("idp_ng");
	if (ng == 0) ng = unit_bytes(t) >= 256 ? 2 : 1; // the 4/5-bit formats are bound by the consumers, not by the ring depth: measured faster as two CTAs
	if (ng == 2) { // one CTA per SM, two consumer groups, the whole shared memory behind one copy of the activations
		// NS even: a slot then always serves the same group (a group that skipped a completion of a slot's barrier could not tell
		// the phase it waits for from the one before it: mbarrier waits carry one parity bit)
		for (int ns = 12; ns >= 4; ns -= 2)
			if (idp_smem_bytes(t, a.n, ns, 2) <= 226 * 1024) { NS = ns; break; }
		if (!NS) ng = 1;
	}
	if (ng != 2) {
		ng = 1;
		// two CTAs per SM when the staged activations leave room for >= 2 ring stages each (kernels overlap under PDL), else one deep ring
		const size_t budget2 = (size_t) tune("tma_smem_kb") * 1024;
		per_sm = tune("idp_per_sm");
		for (int ns = tune("tma_ns_max"); ns >= 2; ns--)
			if (idp_smem_bytes(t, a.n, ns) <= budget2) { NS = ns; break; }
		if (!NS) {
			per_sm = 1;
			for (int ns = 5; ns >= 2; ns--)
				if (idp_smem_bytes(t, a.n, ns) <= 216 * 1024) { NS = ns; break; }
		}
	}
	if (!NS) return -1;
	IdpArgs ta;
	ta.a = a;
	ta.NS = NS;
	ta.n_tiles = vrows / IDP_RC;
	const size_t smem = idp_smem_bytes(t, a.n, NS, ng);
	cudaError_t e;
	switch (t) {
		case XALM_Q8_0: e = launch_idp_typed<XALM_Q8_0>(ta, norm, ng, smem, per_sm, s, pdl); break;
		case XALM_Q8: e = launch_idp_typed<XALM_Q8>(ta, norm, ng, smem, per_sm, s, pdl); break;
		case XALM_Q4_0: e = launch_idp_typed<XALM_Q4_0>(ta, norm, ng, smem, per_sm, s, pdl); break;
		case XALM_Q4_1: e = launch_idp_typed<XALM_Q4_1>(ta, norm, ng, smem, per_sm, s, pdl); break;
		case XALM_Q5_0: e = launch_idp_typed<XALM_Q5_0>(ta, norm, ng, smem, per_sm, s, pdl); break;
		case XALM_Q5_1: e = launch_idp_typed<XALM_Q5_1>(ta, norm, ng, smem, per_sm, s, pdl); break;
		default: return -1;
	}
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "matvec (idp) launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// tensor-core matvec dispatch (matvec_mma.cuh): the integer weight formats in fragment tiles
// ---------------------------------------------------------------------------------------------------------
template <int TYPE, bool NORM>
static cudaError_t launch_mma_inst(const MmaArgs& ta, size_t smem, cudaStream_t s, bool pdl) {
	auto kern = matvec_mma_kernel<TYPE, NORM>;
	cudaError_t e = ensure_smem_attr(kern, 227 * 1024);
	if (e != cudaSuccess) return e;
	int grid = num_sms(); // persistent: one CTA per SM
	if (grid > ta.n_tiles) grid = ta.n_tiles;
	return launch_smem(kern, dim3(grid), dim3((MMA_NCW + 2) * 32), smem, s, pdl, ta);
}
static int launch_matvec_mma(const MatvecArgs& a, cudaStream_t s, bool pdl) {
	const int t = a.w.type;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	if (!mma_supported(t) || a.n % 32 || vrows % MMA_RC || vrows != a.w.rows)
		return set_error(XALM_ERR_STATE, "matrix is in fragment layout but the tensor-core matvec cannot take it (type=%d n=%d rows=%d)", t, a.n, vrows);
	if ((a.epi == EPI_GLU) != (a.w.glu_half != 0))
		return set_error(XALM_ERR_STATE, "fragment layout: gate|up interleave (%d) does not match the epilogue (%d)", a.w.glu_half, a.epi);
	const bool norm = a.norm_w != nullptr;
	int NS = 0;
	for (int ns = 8; ns >= 2; ns--)
		if (mma_smem_bytes(t, a.n, ns) <= 226 * 1024) { NS = ns; break; }
	if (!NS) return set_error(XALM_ERR_UNSUPPORTED, "matmul: rows of %d elements do not fit the tensor-core matvec's shared memory", a.n);
	MmaArgs ta;
	ta.a = a;
	ta.NS = NS;
	ta.n_tiles = vrows / MMA_RC;
	const size_t smem = mma_smem_bytes(t, a.n, NS);
	cudaError_t e;
#define XALM_MMA_CASE(T) case T: e = norm ? launch_mma_inst<T, true>(ta, smem, s, pdl) : launch_mma_inst<T, false>(ta, smem, s, pdl); break;
	switch (t) {
		XALM_MMA_CASE(XALM_Q8_0)
		XALM_MMA_CASE(XALM_Q8)
		XALM_MMA_CASE(XALM_Q4_0)
		XALM_MMA_CASE(XALM_Q4_1)
		XALM_MMA_CASE(XALM_Q5_0)
		XALM_MMA_CASE(XALM_Q5_1)
		default: return set_error(XALM_ERR_STATE, "fragment layout with type %d", t);
	}
#undef XALM_MMA_CASE
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "matvec (mma) launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// batched tensor-core matvec (matvec_mma.cuh): xq_batch_kernel quantises the nseq input rows once, then one pass over the weights
// serves them all.  a.x / a.out hold one row per sequence (x_stride / out_stride floats apart), a.step the step's StepParams array.
// ---------------------------------------------------------------------------------------------------------
struct BatchIo {
	int nseq, x_stride, out_stride;
	uint8_t* img;       // activation image, (n / 32) x ceil(nseq / 2) x MMB_PAIR bytes
	float* nscale;      // (nseq,) 1/rms
	size_t kv_slot;
};
template <int BIAS>
static cudaError_t launch_xq(const XqArgs& q, bool norm, cudaStream_t s, bool pdl) {
	return norm ? launch(xq_batch_kernel<BIAS, true>, dim3(q.nseq), dim3(MMA_NT), s, pdl, q)
	            : launch(xq_batch_kernel<BIAS, false>, dim3(q.nseq), dim3(MMA_NT), s, pdl, q);
}
template <int TYPE, int NP>
static cudaError_t launch_mmb_inst(const MmbArgs& ta, size_t smem, cudaStream_t s, bool pdl) {
	auto kern = matvec_mma_batch_kernel<TYPE, NP>;
	cudaError_t e = ensure_smem_attr(kern, 227 * 1024);
	if (e != cudaSuccess) return e;
	int grid = num_sms();
	if (grid > ta.n_tiles) grid = ta.n_tiles;
	return launch_smem(kern, dim3(grid), dim3((MMA_NCW + 2) * 32), smem, s, pdl, ta);
}
template <int TYPE>
static cudaError_t launch_mmb_typed(const MatvecArgs& a, const BatchIo& io, cudaStream_t s, bool pdl) {
	const int np = (io.nseq + 1) / 2;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	XqArgs q = {};
	q.x = a.x; q.x_stride = io.x_stride; q.n = a.n; q.nseq = io.nseq; q.np = np;
	q.norm_w = a.norm_w; q.norm_type = a.norm_type; q.norm_eps = a.norm_eps; q.img = io.img; q.nscale = io.nscale;
	cudaError_t e = launch_xq<MmaFmt<TYPE>::BIAS>(q, a.norm_w != nullptr, s, pdl);
	if (e != cudaSuccess) return e;
	int NS = 0;
	for (int ns = 8; ns >= 2; ns--)
		if (mmb_smem_bytes(TYPE, np, ns) <= 226 * 1024) { NS = ns; break; }
	MmbArgs ta;
	ta.a = a; ta.NS = NS; ta.n_tiles = vrows / MMA_RC; ta.nseq = io.nseq;
	ta.img = io.img; ta.nscale = a.norm_w ? io.nscale : nullptr; ta.out_stride = io.out_stride; ta.kv_slot = io.kv_slot;
	const size_t smem = mmb_smem_bytes(TYPE, np, NS);
	switch (np) {
		case 1: return launch_mmb_inst<TYPE, 1>(ta, smem, s, pdl);
		case 2: return launch_mmb_inst<TYPE, 2>(ta, smem, s, pdl);
		case 3: return launch_mmb_inst<TYPE, 3>(ta, smem, s, pdl);
		case 4: return launch_mmb_inst<TYPE, 4>(ta, smem, s, pdl);
	}
	return cudaErrorInvalidValue;
}
// two launches: the quantiser and the matvec
static int launch_matvec_batch(const MatvecArgs& a, const BatchIo& io, cudaStream_t s, bool pdl) {
	const int t = a.w.type;
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	if (!a.w.layout_frag || a.n % 32 || vrows % MMA_RC || vrows != a.w.rows || io.nseq < 1 || io.nseq > MMB_MAX_SEQS)
		return set_error(XALM_ERR_STATE, "batched matvec: matrix not in fragment layout or bad shape (type=%d n=%d rows=%d nseq=%d)", t, a.n, vrows, io.nseq);
	if (a.norm_w && a.norm_type != XALM_F32 && a.norm_type != XALM_BF16)
		return set_error(XALM_ERR_UNSUPPORTED, "rmsnorm: unsupported data type %d", a.norm_type);
	cudaError_t e;
	switch (t) {
		case XALM_Q8_0: e = launch_mmb_typed<XALM_Q8_0>(a, io, s, pdl); break;
		case XALM_Q8: e = launch_mmb_typed<XALM_Q8>(a, io, s, pdl); break;
		case XALM_Q4_0: e = launch_mmb_typed<XALM_Q4_0>(a, io, s, pdl); break;
		case XALM_Q4_1: e = launch_mmb_typed<XALM_Q4_1>(a, io, s, pdl); break;
		case XALM_Q5_0: e = launch_mmb_typed<XALM_Q5_0>(a, io, s, pdl); break;
		case XALM_Q5_1: e = launch_mmb_typed<XALM_Q5_1>(a, io, s, pdl); break;
		default: return set_error(XALM_ERR_STATE, "batched matvec: fragment layout with type %d", t);
	}
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "batched matvec launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

static int launch_matvec(MatvecArgs a, cudaStream_t s, bool pdl) {
	const bool norm = a.norm_w != nullptr;
	if (norm && a.norm_type != XALM_F32 && a.norm_type != XALM_BF16)
		return set_error(XALM_ERR_UNSUPPORTED, "rmsnorm: unsupported data type %d", a.norm_type); // infer.cpp:248-249
	if (a.n % 32 || (a.epi != EPI_GLU && a.d % 2))
		return set_error(XALM_ERR_INVALID, "matmul: n=%d d=%d must be multiples of 32", a.n, a.d); // infer.cpp:110-111
	const int vrows = a.epi == EPI_GLU ? 2 * a.d : a.d;
	int t = a.w.type;
	cudaError_t e;
	if (a.w.layout_frag) return launch_matvec_mma(a, s, pdl);
	{
		const int rc = launch_matvec_idp(a, s, pdl);
		if (rc >= 0) return rc;
	}
	if (a.w.layout_units) {
		const int rc = launch_matvec_tma(a, s, pdl);
		if (rc >= 0) return rc;
		return set_error(XALM_ERR_STATE, "matrix is in unit layout but the TMA kernel cannot take it (n=%d d=%d)", a.n, a.d);
	}
	if (tma_eligible(a.w, a.n)) {
		const int rc = launch_matvec_tma(a, s, pdl);
		if (rc >= 0) return rc;
	}
	if (a.n_push || a.n_recv) return set_error(XALM_ERR_STATE, "fused tensor-parallel exchange needs the TMA matvec kernel (n=%d d=%d type=%d)", a.n, a.d, t);
	if (t == XALM_TQ1_0) {
		if (a.n % 256) return set_error(XALM_ERR_INVALID, "TQ1_0 rows must be a multiple of 256 elements (n=%d)", a.n);
		dim3 grid((vrows + 4 * 4 - 1) / (4 * 4)), block(4 * 32);
		e = norm ? launch(matvec_tq1_kernel<4, 4, true>, grid, block, s, pdl, a)
		         : launch(matvec_tq1_kernel<4, 4, false>, grid, block, s, pdl, a);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "matvec launch failed: %s", cudaGetErrorString(e));
		return XALM_OK;
	}
	// config: enough CTAs to cover 148 SMs several times over with balanced shares
	const MvCfg c = vrows >= 6144 ? CFG_A : CFG_B;
	a.lut_type = 0;
	if (t == XALM_F8_E2M5 || t == XALM_F8_E3M4 || t == XALM_QI8 ||
	    ((t == XALM_F8_E4M3 || t == XALM_F8_E5M2) && (a.w.flags & WMAT_FP8_NONFINITE))) {
		a.lut_type = t;
		t = -1;
	}
	switch (t) {
		case -1: e = launch_matvec_typed<-1>(a, c, norm, s, pdl); break;
		case XALM_F32: e = launch_matvec_typed<XALM_F32>(a, c, norm, s, pdl); break;
		case XALM_F16: e = launch_matvec_typed<XALM_F16>(a, c, norm, s, pdl); break;
		case XALM_BF16: e = launch_matvec_typed<XALM_BF16>(a, c, norm, s, pdl); break;
		case XALM_F8_E4M3: e = launch_matvec_typed<XALM_F8_E4M3>(a, c, norm, s, pdl); break;
		case XALM_F8_E5M2: e = launch_matvec_typed<XALM_F8_E5M2>(a, c, norm, s, pdl); break;
		case XALM_Q8: e = launch_matvec_typed<XALM_Q8>(a, c, norm, s, pdl); break;
		case XALM_Q8_0: e = launch_matvec_typed<XALM_Q8_0>(a, c, norm, s, pdl); break;
		case XALM_Q4_0: e = launch_matvec_typed<XALM_Q4_0>(a, c, norm, s, pdl); break;
		case XALM_Q4_1: e = launch_matvec_typed<XALM_Q4_1>(a, c, norm, s, pdl); break;
		case XALM_Q5_0: e = launch_matvec_typed<XALM_Q5_0>(a, c, norm, s, pdl); break;
		case XALM_Q5_1: e = launch_matvec_typed<XALM_Q5_1>(a, c, norm, s, pdl); break;
		default:
			return set_error(XALM_ERR_UNSUPPORTED, "matmul: unsupported data type: %d", a.w.type); // infer.cpp:211-214
	}
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "matvec launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------------------
// _copy_embedding (infer.cpp:553-602) from the ON-DISK layout of the table (block formats: extension); one row per step entry
// (blockIdx.y), x is (entries, dim)
__global__ void embed_rows_kernel(int type, const uint8_t* __restrict__ table, size_t row_bytes, int dim, const StepParams* steps,
                                  float* __restrict__ x) {
	pdl_launch_dependents();
	pdl_wait();
	const uint8_t* row = table + (size_t) steps[blockIdx.y].token * row_bytes;
	float* xs = x + (size_t) blockIdx.y * dim;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < dim; i += gridDim.x * blockDim.x) xs[i] = decode_disk_elem(type, row, i);
}

__global__ void dequant_kernel(int type, const uint8_t* __restrict__ src, size_t n, float* __restrict__ dst) {
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x)
		dst[i] = decode_disk_elem(type, src, i);
}

// Sampler::sample_argmax (sampler.cpp:3-16) on the device: running maximum seeded with FLT_MIN (the reference's quirk: with no
// logit above 1.18e-38 the answer is 0), strict '>' so the FIRST maximum wins.  One CTA per row.
__device__ __forceinline__ void argmax_row(const float* __restrict__ logits, int n, int* __restrict__ out) {
	__shared__ float s_v[32];
	__shared__ int s_i[32];
	float best = 1.17549435e-38f; // numeric_limits<float>::min()
	int bi = 0;
	for (int i = threadIdx.x; i < n; i += blockDim.x) {
		const float v = logits[i];
		if (v > best) { best = v; bi = i; }
	}
	auto better = [](float v, int i, float bv, int b) { return v > bv || (v == bv && i < b); };
	// a thread that saw nothing above the seed keeps index 0, which the tie rule turns into "lowest index": patch it to n so real hits win
	if (best == 1.17549435e-38f && bi == 0 && !(logits[0] > 1.17549435e-38f)) bi = n;
	for (int o = 16; o > 0; o >>= 1) {
		const float ov = __shfl_xor_sync(0xffffffffu, best, o);
		const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
		if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
	}
	if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = bi; }
	__syncthreads();
	if (threadIdx.x < 32) {
		const int nw = (blockDim.x + 31) / 32;
		best = threadIdx.x < nw ? s_v[threadIdx.x] : 1.17549435e-38f;
		bi = threadIdx.x < nw ? s_i[threadIdx.x] : n;
		for (int o = 16; o > 0; o >>= 1) {
			const float ov = __shfl_xor_sync(0xffffffffu, best, o);
			const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
			if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
		}
		if (threadIdx.x == 0) *out = bi >= n ? 0 : bi;
	}
}
// row b of (rows, n) logits -> out[b]
__global__ void argmax_rows_kernel(const float* __restrict__ logits, int n, int* __restrict__ out) {
	argmax_row(logits + (size_t) blockIdx.x * n, n, out + blockIdx.x);
}

// an entry's token, position and mode, and its ring / sink indices: infer.cpp:611-613, KV_SINKS = 2 (model.h:10).  On the host for
// every step the host sets up, on the device for the steps of a greedy chain (argmax_next_step_kernel).
static __host__ __device__ void fill_step_entry(const xalm_config& c, StepParams& p, int token, int pos, int mode) {
	p.token = token; p.pos = pos;
	p.kv_sink = pos >= c.max_seq_len ? 2 : 0;
	p.kv_pos = p.kv_sink + (pos - p.kv_sink) % (c.max_seq_len - p.kv_sink);
	p.kv_len = pos >= c.max_seq_len ? c.max_seq_len : pos + 1;
	p.mode = mode;
	p.tree = TREE_IDENTITY;
}

// One link of a greedy chain (xalm_cuda_forward_greedy): Sampler::sample_argmax of the single-sequence logits into *out and, unless
// `next` is NULL (the chain's last step), the single-sequence StepParams row of the next step, which decodes that token at next_pos.
// Freshness: every kernel of a step reads StepParams from d_step, some of them before their PDL dependency wait.  This kernel is
// therefore launched WITHOUT the PDL attribute: it starts only once the step that read the row has completed, and the next step's
// first kernel (the embedding, also launched without PDL) starts only once this one has completed.
__global__ void argmax_next_step_kernel(const float* __restrict__ logits, int n, int* __restrict__ out, StepParams* __restrict__ next,
                                        xalm_config c, int next_pos, unsigned int ar_base) {
	argmax_row(logits, n, out);
	if (next && threadIdx.x == 0) { // the thread that wrote *out
		StepParams p;
		fill_step_entry(c, p, *out, next_pos, XALM_OUTPUT_LOGITS);
		p.kv_fresh = p.kv_pos;
		p.ar_base = ar_base;
		p.slot = 0;
		*next = p;
	}
}

// xalm_cuda_tree_accept: move j copies row src[j] to row dst[j] of one K or V cache, for j = 0 .. n-1 in that order, each once
// the one before has landed.  The order matters: a move may write the row an earlier move read (never one a later move reads,
// because sources lie above every earlier destination; xalm_cuda.h).  One CTA per cache: caches[2 l] / caches[2 l + 1] are layer l's
// K / V caches, offset is the slot's first element, a row is kv_dim halves.  Launched without PDL, like argmax_next_step_kernel: it
// starts once the verifying step has completed, and the next step's embedding (also launched without PDL) once it has.
struct TreeMoves {
	int n;
	int src[MMB_MAX_SEQS], dst[MMB_MAX_SEQS]; // rows within the slot
};
__global__ void tree_accept_kernel(__half* const* __restrict__ caches, size_t offset, int kv_dim, const TreeMoves mv) {
	__half* base = caches[blockIdx.x] + offset;
	const int n16 = kv_dim / 8; // uint4 per row
	for (int j = 0; j < mv.n; j++) {
		const uint4* src = reinterpret_cast<const uint4*>(base + (size_t) mv.src[j] * kv_dim);
		uint4* dst = reinterpret_cast<uint4*>(base + (size_t) mv.dst[j] * kv_dim);
		for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = src[i];
		__syncthreads();
	}
}

__global__ void residual_add_kernel(float* __restrict__ x, const float* __restrict__ y, int n) {
	pdl_launch_dependents();
	pdl_wait();
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) x[i] += y[i];
}

// ---- one-shot allreduce + residual over NVLink peer memory (tensor parallel) -------------------------------------------
// Every rank's matvec wrote its partial vector into ITS OWN exchange buffer (slot = call index & 1).  This kernel
//   1. publishes "my partial #seq is ready" into every peer's flag array (system-scope release after the kernel boundary),
//   2. waits until all peers have published #seq in MY flag array (local polling),
//   3. reads the P partials straight from peer memory (volatile loads: peer lines must not be served from a stale L1),
//      sums them in rank order — identical bits on every rank — and adds the result to the residual stream x.
// Two slots suffice: a rank can only reach call k+2 after every peer has signalled k+1, i.e. finished reading k.
struct PeerArgs {
	float* data[8];          // exchange buffers of all ranks (peer-mapped), [2][stride] floats each
	unsigned int* flags[8];  // flag arrays of all ranks, [2][8] u32 each
	int rank, size, stride;
	uint2* recv[8];          // per rank: its receive area [2 slots][8 source ranks][dim] of {value, tag} words (fused exchange, matvec_tma.cuh)
};
__global__ void peer_allreduce_residual_kernel(const PeerArgs pa, float* __restrict__ x, int n, int idx, const StepParams* step) {
	pdl_launch_dependents();
	pdl_wait();
	const int slot = idx & 1;
	const unsigned int seq = step->ar_base + (unsigned int) idx + 1u;
	if (blockIdx.x == 0 && threadIdx.x < pa.size) {
		__threadfence_system();
		unsigned int* f = pa.flags[threadIdx.x] + slot * 8 + pa.rank;
		asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(seq) : "memory");
	}
	if (threadIdx.x < pa.size) {
		const unsigned int* f = pa.flags[pa.rank] + slot * 8 + threadIdx.x;
		unsigned int v;
		do {
			asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
		} while ((int) (v - seq) < 0);
	}
	__syncthreads();
	for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += gridDim.x * blockDim.x * 4) {
		float4 acc = *reinterpret_cast<const float4*>(x + i);
		float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
		for (int p = 0; p < pa.size; p++) {
			const float* src = pa.data[p] + (size_t) slot * pa.stride + i;
			float4 v;
			asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(src));
			sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
		}
		acc.x += sum.x; acc.y += sum.y; acc.z += sum.z; acc.w += sum.w;
		*reinterpret_cast<float4*>(x + i) = acc;
	}
}

// Fused exchange, HYDRATE tokens: the classifier that would receive the last exchange of the token is not run, but the exchange
// must still be CONSUMED before this rank moves on — the two-slot scheme is only safe while every rank executes
// push(i), recv(i), push(i+1), ... (tests/test_tp_exchange_protocol.py shows the overwrite / deadlock without this).  One CTA polls
// the tags of all P partials of that exchange and discards the values.
__global__ void tp_drain_kernel(const uint2* __restrict__ recv, int n_ranks, int dim, int idx, const StepParams* step, unsigned int* err_flag) {
	pdl_launch_dependents();
	pdl_wait();
	const unsigned int seq = step->ar_base + (unsigned int) idx + 1u;
	for (int i = threadIdx.x; i < n_ranks * dim; i += blockDim.x) {
		unsigned int tag, spins = 0;
		do {
			asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(tag) : "l"(&recv[i].y));
			if (++spins > xalm::XALM_SPIN_LIMIT) { if (err_flag) *err_flag = 1u; break; }
		} while (tag != seq);
	}
}

// standalone rmsnorm / rope for the op-level entry points (the hot path fuses both into the matvec kernel)
__global__ void rmsnorm_kernel(float* o, const float* x, const uint8_t* w, int wtype, int size, float eps) {
	__shared__ float s_red[32];
	float ss = 0.f;
	for (int i = threadIdx.x; i < size; i += blockDim.x) ss += x[i] * x[i];
	ss = warp_sum(ss);
	if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = ss;
	__syncthreads();
	float tot = 0.f;
	for (int i = 0; i < (int) (blockDim.x + 31) / 32; i++) tot += s_red[i];
	const float scale = 1.0f / sqrtf(tot / (float) size + eps);
	for (int i = threadIdx.x; i < size; i += blockDim.x) {
		const float g = wtype == XALM_F32 ? reinterpret_cast<const float*>(w)[i] : bf16_bits_to_f32(reinterpret_cast<const uint16_t*>(w)[i]);
		o[i] = x[i] * scale * g;
	}
}
__global__ void rope_kernel(float* vec, int d, int head_dim, int pos, const float* freq) {
	for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d / 2; p += gridDim.x * blockDim.x) {
		float v0 = vec[2 * p], v1 = vec[2 * p + 1];
		rope_pair(v0, v1, (2 * p) % head_dim, pos, freq);
		vec[2 * p] = v0;
		vec[2 * p + 1] = v1;
	}
}

// 1/powf(theta, j/rotary_dim) on the HOST, exactly the expression of infer.cpp:310-312 (0 beyond rotary_dim)
static std::vector<float> rope_freq_table(int head_dim, int rotary_dim, float theta) {
	std::vector<float> f(head_dim / 2);
	for (int j = 0; j < head_dim; j += 2)
		f[j / 2] = j >= rotary_dim ? 0.f : 1.0f / powf(theta, (float) j / (float) rotary_dim);
	return f;
}

// ---------------------------------------------------------------------------------------------------------
// attention dispatch
// ---------------------------------------------------------------------------------------------------------
template <int HD, bool BATCH>
static cudaError_t launch_attn_hd(const AttnArgs& a, int G, int nseq, cudaStream_t s, bool pdl) {
	dim3 grid(a.n_splits, a.n_kv_heads, nseq), block(256);
	constexpr int NW8 = HD >= 256 ? 4 : 8; // 8 query heads x 256 dims: keep the per-warp partials within 48 KB of static smem
	switch (G) {
		case 1: return launch(attn_decode_kernel<HD, 1, 8, BATCH>, grid, block, s, pdl, a);
		case 2: return launch(attn_decode_kernel<HD, 2, 8, BATCH>, grid, block, s, pdl, a);
		case 4: return launch(attn_decode_kernel<HD, 4, 8, BATCH>, grid, block, s, pdl, a);
		case 8: return launch(attn_decode_kernel<HD, 8, NW8, BATCH>, grid, dim3(NW8 * 32), s, pdl, a);
	}
	return cudaErrorInvalidValue;
}
// nseq > 0: the batched kernel, one grid layer per sequence (AttnArgs' batched fields); 0: one sequence
static int launch_attn(const AttnArgs& a, int head_dim, int G, cudaStream_t s, bool pdl, int nseq = 0) {
	cudaError_t e;
	const bool b = nseq > 0;
	const int z = b ? nseq : 1;
	switch (head_dim) {
		case 32: e = b ? launch_attn_hd<32, true>(a, G, z, s, pdl) : launch_attn_hd<32, false>(a, G, z, s, pdl); break;
		case 64: e = b ? launch_attn_hd<64, true>(a, G, z, s, pdl) : launch_attn_hd<64, false>(a, G, z, s, pdl); break;
		case 128: e = b ? launch_attn_hd<128, true>(a, G, z, s, pdl) : launch_attn_hd<128, false>(a, G, z, s, pdl); break;
		case 256: e = b ? launch_attn_hd<256, true>(a, G, z, s, pdl) : launch_attn_hd<256, false>(a, G, z, s, pdl); break;
		default: return set_error(XALM_ERR_UNSUPPORTED, "attention: head_dim %d not in {32,64,128,256}", head_dim);
	}
	if (e == cudaErrorInvalidValue && (G != 1 && G != 2 && G != 4 && G != 8))
		return set_error(XALM_ERR_UNSUPPORTED, "attention: %d query heads per kv head not in {1,2,4,8}", G);
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "attention launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}
static int attn_auto_splits(int n_kv_heads) {
	int forced = tune("attn_splits");
	if (forced > 0) return forced;
	int sms = 148;
	int dev = 0;
	if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	// about one CTA per SM, and never so many splits that the last-CTA merge dominates (measured: profiles/r1_attention_splits.md)
	int s = sms / n_kv_heads;
	if (s > 32) s = 32;
	return s < 1 ? 1 : s;
}

// ---------------------------------------------------------------------------------------------------------
// device weight storage
// ---------------------------------------------------------------------------------------------------------
struct DevAlloc {
	std::vector<void*> ptrs;
	size_t total = 0;
	int alloc(void** p, size_t bytes) {
		if (bytes == 0) bytes = 16;
		cudaError_t e = cudaMalloc(p, bytes);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
		ptrs.push_back(*p);
		total += bytes;
		return XALM_OK;
	}
	void free_all() {
		for (void* p : ptrs) cudaFree(p);
		ptrs.clear();
	}
};

// A weight matrix being assembled from one or more uploaded pieces stacked along rows (q|k|v, gate|up).
struct WSlot {
	WMat m;            // planes for ALL rows of the fused matrix
	int total_rows = 0;
	bool allocated = false;
};

// can the tensor-core matvec take this matrix (batch 1: its activations staged whole in shared memory)?
static bool mma_takes(int type, int rows, int n, int glu_half) {
	return mma_supported(type) && n % 32 == 0 && rows % MMA_RC == 0 && glu_half % 8 == 0 && mma_smem_bytes(type, n, 2) <= 226 * 1024;
}

// batched: the matrix goes to fragment tiles whatever the knobs say (the caller has checked mma_takes)
static int alloc_wmat(DevAlloc& da, WMat& m, int type, int rows, int n, int glu_half = 0, bool sharded = false, bool batched = false) {
	m.type = type; m.rows = rows; m.n = n; m.flags = 0; m.layout_units = 0; m.layout_frag = 0; m.glu_half = 0;
	TypeInfo tinfo;
	type_info(type, &tinfo);
	// 2 (default): the 4/5-bit formats always; the 8-bit ones under tensor parallelism, where the per-rank rows are short (the dp4a kernel
	// maps one 32-element block to a lane: rows of 512 elements keep 16 of its 256 lanes busy) — TP2 611 -> 637 tok/s
	const bool mma_on = tune("mma") == 1 || (tune("mma") == 2 && (sharded || (type != XALM_Q8_0 && type != XALM_Q8)));
	if (mma_takes(type, rows, n, glu_half) && (batched || (mma_on && tune("tma")))) {
		// integer formats on the tensor-core path: fragment tiles (frag_layout.cuh); same byte count as on disk
		m.layout_frag = 1;
		m.glu_half = glu_half;
		m.s0 = (size_t) n / 32 * frag_record_bytes(type); m.s1 = m.s2 = 0;
		uint8_t* p = nullptr;
		XALM_TRY(da.alloc((void**) &p, m.s0 * (rows / MMA_RC)));
		m.p0 = p; m.p1 = m.p2 = nullptr;
		return XALM_OK;
	}
	if (tinfo.block > 1 && unit_bytes(type) && n % 256 == 0 && rows % 8 == 0 && tune("tma")) {
		// block formats on the TMA path: unit-interleaved rows (matvec_tma.cuh); same byte count as planar
		m.layout_units = 1;
		m.s0 = (size_t) n / 256 * unit_bytes(type); m.s1 = m.s2 = 0;
		uint8_t* p = nullptr;
		XALM_TRY(da.alloc((void**) &p, m.s0 * rows));
		m.p0 = p; m.p1 = m.p2 = nullptr;
		return XALM_OK;
	}
	const PlaneSizes ps = plane_row_bytes(type, n);
	m.s0 = ps.s0; m.s1 = ps.s1; m.s2 = ps.s2;
	uint8_t *p0 = nullptr, *p1 = nullptr, *p2 = nullptr;
	XALM_TRY(da.alloc((void**) &p0, ps.s0 * rows));
	if (ps.s1) XALM_TRY(da.alloc((void**) &p1, ps.s1 * rows));
	if (ps.s2) XALM_TRY(da.alloc((void**) &p2, ps.s2 * rows));
	m.p0 = p0; m.p1 = p1; m.p2 = p2;
	return XALM_OK;
}

// Copy rows [r0,r1) x element columns [c0,c1) of a host tensor (on-disk layout, `n_full` elements per row) to the
// device and repack them into rows [dst_row, ...) of `m`.  `staging` is a reusable device scratch buffer.
struct Staging {
	uint8_t* p = nullptr;
	size_t cap = 0;
	int* flag = nullptr;
};
static int upload_piece(WMat& m, int dst_row, int type, const uint8_t* host, int n_full, int r0, int r1, int c0, int c1,
                        Staging& st, cudaStream_t s) {
	TypeInfo ti;
	type_info(type, &ti);
	if (n_full % ti.block || c0 % ti.block || c1 % ti.block)
		return set_error(XALM_ERR_INVALID, "column range [%d,%d) of %d splits a %d-element block", c0, c1, n_full, ti.block);
	const size_t full_row = (size_t) n_full / ti.block * ti.bytes;
	const size_t width = (size_t) (c1 - c0) / ti.block * ti.bytes;
	const size_t off = (size_t) c0 / ti.block * ti.bytes;
	const int rows = r1 - r0;
	const size_t need = width * rows;
	if (need > st.cap) {
		if (st.p) cudaFree(st.p);
		st.p = nullptr; st.cap = 0;
		XALM_CUDA_CHECK(cudaMalloc((void**) &st.p, need));
		st.cap = need;
	}
	if (!st.flag) XALM_CUDA_CHECK(cudaMalloc((void**) &st.flag, sizeof(int)));
	XALM_CUDA_CHECK(cudaMemcpy2DAsync(st.p, width, host + (size_t) r0 * full_row + off, full_row, width, rows, cudaMemcpyHostToDevice, s));
	const int n = c1 - c0;
	uint8_t* p0 = const_cast<uint8_t*>(m.p0) + (size_t) dst_row * m.s0;
	uint8_t* p1 = m.p1 ? const_cast<uint8_t*>(m.p1) + (size_t) dst_row * m.s1 : nullptr;
	uint8_t* p2 = m.p2 ? const_cast<uint8_t*>(m.p2) + (size_t) dst_row * m.s2 : nullptr;
	if (m.layout_frag) repack_frag_kernel<<<1024, 256, 0, s>>>(type, st.p, width, dst_row, rows, m.rows, n, m.glu_half, const_cast<uint8_t*>(m.p0));
	else if (m.layout_units) repack_units_kernel<<<1024, 256, 0, s>>>(type, st.p, width, rows, n, p0, m.s0);
	else repack_kernel<<<1024, 256, 0, s>>>(type, st.p, width, rows, n, p0, m.s0, p1, m.s1, p2, m.s2);
	XALM_CUDA_CHECK(cudaGetLastError());
	if (type == XALM_F8_E4M3 || type == XALM_F8_E5M2) {
		XALM_CUDA_CHECK(cudaMemsetAsync(st.flag, 0, sizeof(int), s));
		fp8_scan_nonfinite_kernel<<<256, 256, 0, s>>>(type, st.p, need, st.flag);
		int h = 0;
		XALM_CUDA_CHECK(cudaMemcpyAsync(&h, st.flag, sizeof(int), cudaMemcpyDeviceToHost, s));
		XALM_CUDA_CHECK(cudaStreamSynchronize(s));
		if (h) m.flags |= WMAT_FP8_NONFINITE;
	}
	XALM_CUDA_CHECK(cudaStreamSynchronize(s));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// NCCL, loaded lazily (nccl_api.h)
// ---------------------------------------------------------------------------------------------------------
NcclApi g_nccl;
int nccl_load() {
	if (g_nccl.h) return XALM_OK;
	const char* names[] = {"libnccl.so.2", "libnccl.so"};
	for (const char* n : names)
		if ((g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
	if (!g_nccl.h) return set_error(XALM_ERR_COMM, "cannot load libnccl: %s", dlerror());
#define XALM_NCCL_SYM(field, sym)                                                                      \
	if (!(*(void**) (&g_nccl.field) = dlsym(g_nccl.h, sym))) {                                         \
		g_nccl.h = nullptr;                                                                            \
		return set_error(XALM_ERR_COMM, "libnccl lacks %s", sym);                                      \
	}
	XALM_NCCL_SYM(GetUniqueId, "ncclGetUniqueId");
	XALM_NCCL_SYM(CommInitRank, "ncclCommInitRank");
	XALM_NCCL_SYM(AllReduce, "ncclAllReduce");
	XALM_NCCL_SYM(AllGather, "ncclAllGather");
	XALM_NCCL_SYM(ReduceScatter, "ncclReduceScatter");
	XALM_NCCL_SYM(CommDestroy, "ncclCommDestroy");
	XALM_NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef XALM_NCCL_SYM
	return XALM_OK;
}

} // namespace xalm

using namespace xalm;

// ---------------------------------------------------------------------------------------------------------
// the model handle
// ---------------------------------------------------------------------------------------------------------
struct LayerDev {
	WSlot wqkv, wo, w13, w2;
	const uint8_t* rms_att = nullptr;
	const uint8_t* rms_ffn = nullptr;
	int rms_att_type = 0, rms_ffn_type = 0;
	__half* k_cache = nullptr;
	__half* v_cache = nullptr;
	bool got[9] = {false, false, false, false, false, false, false, false, false};
	int piece_type[9] = {0};
};
enum { P_ATT_NORM = 0, P_FFN_NORM, P_Q, P_K, P_V, P_O, P_GATE, P_DOWN, P_UP };

struct StepGraph {
	cudaGraphExec_t exec;
	int launches;
};

struct xalm_cuda_model {
	xalm_config c;
	int device = 0, tp_rank = 0, tp_size = 1;
	// batched decode (xalm_cuda_set_batch): max_seqs sequence slots, each with its own KV cache, slot_stride elements apart
	int max_seqs = 1;
	bool batched = false;
	bool uploaded = false;
	int cur_seq = 0;                  // the slot the single-sequence calls use (xalm_cuda_select_seq)
	size_t kv_slot = 0;
	uint8_t* ximg = nullptr;          // activation image of the batched matvec
	float* nscale = nullptr;          // (max_seqs,) 1/rms of the batched matvec's norm prologue
	// (mode, n) -> captured step; n = 0: the single-sequence kernel sequence, else a batched step of n entries (run_step)
	std::map<std::pair<int, int>, StepGraph> graphs;
	// local (per-rank) sizes
	int q_dim = 0, kv_dim = 0, q_dim_l = 0, kv_dim_l = 0, n_heads_l = 0, n_kv_heads_l = 0, hidden_l = 0, vocab_l = 0;
	DevAlloc da;
	Staging staging;
	// weights
	uint8_t* embed_raw = nullptr; // on-disk layout, all rows (replicated)
	int embed_type = 0;
	size_t embed_row_bytes = 0;
	bool got_embed = false, got_final_norm = false, got_cls = false;
	WSlot wcls;
	const uint8_t* rms_final = nullptr;
	int rms_final_type = 0;
	std::vector<LayerDev> layers;
	// state (InferenceState, model.h:96-156 — only what the fused kernels still materialise)
	float *x = nullptr, *xb2 = nullptr, *hb = nullptr, *q = nullptr, *logits = nullptr, *logits_full = nullptr, *part = nullptr;
	float* rope_freq = nullptr;
	float *attn_acc = nullptr, *attn_ml = nullptr;
	unsigned int* tickets = nullptr;
	int attn_splits = 0;
	StepParams* d_step = nullptr;
	StepParams* h_step = nullptr; // pinned ring
	cudaEvent_t h_step_ev[64];
	bool h_step_ev_used[64];
	int step_slot = 0;
	float* h_logits = nullptr; // pinned
	cudaStream_t own_stream = nullptr, stream = nullptr;
	bool finalized = false;
	int last_launches = 0;
	ncclComm_t comm = nullptr;
	// peer-memory allreduce
	float* xchg = nullptr;            // [2][dim] floats + [2][8] u32 flags, cudaMalloc'd (IPC-exportable)
	bool peer_ready = false;
	bool tp_fused = false;            // exchanges fused into the matvec kernels (push + receive in the next prologue)
	float* x_alt = nullptr;           // second residual-stream buffer (the fused exchange ping-pongs x)
	unsigned int* h_err = nullptr;    // pinned: a tensor-parallel wait that gave up sets it
	uint2* xl = nullptr;              // [2][dim] {value, tag} words: the summed stream published inside a receiving kernel
	xalm::PeerArgs peer = {};
	std::vector<void*> peer_opened;
	unsigned int token_serial = 0;
	__half** kv_table = nullptr;      // device: every layer's K and V cache (tree_accept_kernel)
	int* d_argmax = nullptr;          // device-side sampler result
	int* h_argmax = nullptr;          // pinned
	// batched prefill (prefill.cu)
	PrefillScratch* prefill = nullptr;
	int last_prefill_launches = 0;
	int* prefill_status = nullptr;    // tensor parallel: the one int the ranks' status vote reduces (allocated by finalize)
};

static int parse_tensor_name(const char* name, int n_layers, int* layer, int* piece) {
	// model.cpp:83-114
	*layer = -1;
	*piece = -1;
	if (!strcmp(name, "embed.weight")) { *piece = 100; return XALM_OK; }
	if (!strcmp(name, "output.norm.weight")) { *piece = 101; return XALM_OK; }
	if (!strcmp(name, "output.weight")) { *piece = 102; return XALM_OK; }
	int l = -1;
	char rest[64] = {0};
	if (sscanf(name, "l.%d.%63s", &l, rest) == 2 && l >= 0 && l < n_layers) {
		static const char* names[9] = {"attn.norm.weight", "mlp.norm.weight", "attn.q.weight", "attn.k.weight", "attn.v.weight",
		                               "attn.down.weight", "mlp.gate.weight", "mlp.down.weight", "mlp.up.weight"};
		for (int i = 0; i < 9; i++)
			if (!strcmp(rest, names[i])) { *layer = l; *piece = i; return XALM_OK; }
	}
	return set_error(XALM_ERR_INVALID, "unknown tensor name '%s'", name);
}

extern "C" {

int xalm_cuda_abi_version(void) { return XALM_CUDA_ABI_VERSION; }
const char* xalm_cuda_last_error(void) { return g_last_error.c_str(); }

int xalm_cuda_device_count(int* count) {
	if (!count) return set_error(XALM_ERR_INVALID, "count is NULL");
	XALM_CUDA_CHECK(cudaGetDeviceCount(count));
	return XALM_OK;
}

int xalm_cuda_type_info(int type_id, int* block_elems, int* block_bytes) {
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	if (block_elems) *block_elems = ti.block;
	if (block_bytes) *block_bytes = ti.bytes;
	return XALM_OK;
}

int xalm_cuda_tune(const char* key, int value) {
	if (!key || !tuning().count(key)) return set_error(XALM_ERR_INVALID, "unknown tuning key '%s'", key ? key : "(null)");
	tuning()[key] = value;
	return XALM_OK;
}

int xalm_cuda_create(const xalm_config* cfg, int device, int tp_rank, int tp_size, xalm_cuda_model** out) {
	if (!cfg || !out) return set_error(XALM_ERR_INVALID, "cfg/out is NULL");
	*out = nullptr;
	const xalm_config& c = *cfg;
	if (c.dim <= 0 || c.hidden_dim <= 0 || c.head_dim <= 0 || c.n_layers <= 0 || c.n_heads <= 0 || c.n_kv_heads <= 0 ||
	    c.vocab_size <= 0 || c.max_seq_len <= 0)
		return set_error(XALM_ERR_INVALID, "config has a non-positive dimension");
	if (c.n_heads % c.n_kv_heads) return set_error(XALM_ERR_INVALID, "n_heads %d not a multiple of n_kv_heads %d", c.n_heads, c.n_kv_heads);
	if (c.dim % 32 || c.hidden_dim % 32 || c.vocab_size % 32 || (c.n_heads * c.head_dim) % 32 || (c.n_kv_heads * c.head_dim) % 32)
		return set_error(XALM_ERR_INVALID, "matmul dimensions must be multiples of 32 (infer.cpp:110-111)");
	if (c.head_dim % 2 || c.rotary_dim > c.head_dim || c.rotary_dim < 0) return set_error(XALM_ERR_INVALID, "bad head_dim/rotary_dim");
	if (c.max_seq_len <= 2) return set_error(XALM_ERR_INVALID, "max_seq_len must exceed KV_SINKS (2)");
	if (c.norm_type != 0) return set_error(XALM_ERR_UNSUPPORTED, "unsupported norm type");
	if (c.act != XALM_GELU && c.act != XALM_SILU) return set_error(XALM_ERR_UNSUPPORTED, "unsupported activation type");
	if (tp_size < 1 || tp_rank < 0 || tp_rank >= tp_size) return set_error(XALM_ERR_INVALID, "bad tp_rank/tp_size %d/%d", tp_rank, tp_size);
	if (c.n_kv_heads % tp_size || c.n_heads % tp_size || c.hidden_dim % (32 * tp_size) || c.vocab_size % (32 * tp_size) ||
	    ((c.n_heads / tp_size) * c.head_dim) % 32)
		return set_error(XALM_ERR_INVALID, "tp_size %d does not divide heads/hidden/vocab into 32-aligned shards", tp_size);
	int ndev = 0;
	XALM_CUDA_CHECK(cudaGetDeviceCount(&ndev));
	if (device < 0 || device >= ndev) return set_error(XALM_ERR_CUDA, "device %d not available (%d devices)", device, ndev);
	XALM_CUDA_CHECK(cudaSetDevice(device));
	xalm_cuda_model* m = new xalm_cuda_model();
	m->c = c;
	m->device = device; m->tp_rank = tp_rank; m->tp_size = tp_size;
	m->q_dim = c.n_heads * c.head_dim;
	m->kv_dim = c.n_kv_heads * c.head_dim;
	m->n_heads_l = c.n_heads / tp_size;
	m->n_kv_heads_l = c.n_kv_heads / tp_size;
	m->q_dim_l = m->n_heads_l * c.head_dim;
	m->kv_dim_l = m->n_kv_heads_l * c.head_dim;
	m->hidden_l = c.hidden_dim / tp_size;
	m->vocab_l = c.vocab_size / tp_size;
	m->layers.resize(c.n_layers);
	memset(m->h_step_ev_used, 0, sizeof m->h_step_ev_used);
	cudaError_t e = cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking);
	if (e != cudaSuccess) { delete m; return set_error(XALM_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e)); }
	m->stream = m->own_stream;
	*out = m;
	return XALM_OK;
}

void xalm_cuda_destroy(xalm_cuda_model* m) {
	if (!m) return;
	cudaSetDevice(m->device);
	prefill_free(m->prefill);
	m->prefill = nullptr;
	cudaSetDevice(m->device);
	cudaStreamSynchronize(m->stream);
	for (auto& kv : m->graphs) cudaGraphExecDestroy(kv.second.exec);
	if (m->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(m->comm);
	for (int i = 0; i < 64; i++)
		if (m->h_step_ev_used[i]) cudaEventDestroy(m->h_step_ev[i]);
	if (m->h_argmax) cudaFreeHost(m->h_argmax);
	for (void* p : m->peer_opened) cudaIpcCloseMemHandle(p);
	if (m->xchg) cudaFree(m->xchg);
	m->da.free_all();
	if (m->staging.p) cudaFree(m->staging.p);
	if (m->staging.flag) cudaFree(m->staging.flag);
	if (m->h_step) cudaFreeHost(m->h_step);
	if (m->h_logits) cudaFreeHost(m->h_logits);
	if (m->h_err) cudaFreeHost(m->h_err);
	if (m->own_stream) cudaStreamDestroy(m->own_stream);
	delete m;
}

int xalm_cuda_set_stream(xalm_cuda_model* m, void* cuda_stream) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	m->stream = cuda_stream ? (cudaStream_t) cuda_stream : m->own_stream;
	return XALM_OK;
}

int xalm_cuda_ipc_export(xalm_cuda_model* m, void* handle64) {
	if (!m || !handle64) return set_error(XALM_ERR_INVALID, "model/handle is NULL");
	if (m->finalized) return set_error(XALM_ERR_STATE, "ipc_export must precede finalize");
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	static_assert(sizeof(cudaIpcMemHandle_t) == XALM_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
	if (!m->xchg) {
		// [2][dim] pull slots | [2][8] flags | [2][8][dim] receive slots of 8-byte {value, tag} words
		const size_t bytes = (size_t) (2 + 32) * m->c.dim * sizeof(float) + 2 * 8 * sizeof(unsigned int);
		XALM_CUDA_CHECK(cudaMalloc((void**) &m->xchg, bytes)); // its own allocation: the IPC handle covers exactly this buffer
		XALM_CUDA_CHECK(cudaMemset(m->xchg, 0, bytes));
		XALM_CUDA_CHECK(cudaDeviceSynchronize());
	}
	cudaIpcMemHandle_t h;
	XALM_CUDA_CHECK(cudaIpcGetMemHandle(&h, m->xchg));
	memcpy(handle64, &h, sizeof h);
	return XALM_OK;
}

int xalm_cuda_ipc_import(xalm_cuda_model* m, const void* handles) {
	if (!m || !handles) return set_error(XALM_ERR_INVALID, "model/handles is NULL");
	if (m->finalized) return set_error(XALM_ERR_STATE, "ipc_import must precede finalize");
	if (!m->xchg) return set_error(XALM_ERR_STATE, "ipc_import before ipc_export");
	if (m->tp_size > 8) return set_error(XALM_ERR_UNSUPPORTED, "peer allreduce supports up to 8 ranks");
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	const size_t data_floats = (size_t) 2 * m->c.dim;
	for (int p = 0; p < m->tp_size; p++) {
		float* base = nullptr;
		if (p == m->tp_rank) base = m->xchg;
		else {
			cudaIpcMemHandle_t h;
			memcpy(&h, (const char*) handles + (size_t) p * XALM_IPC_HANDLE_BYTES, sizeof h);
			void* ptr = nullptr;
			XALM_CUDA_CHECK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
			m->peer_opened.push_back(ptr);
			base = (float*) ptr;
		}
		m->peer.data[p] = base;
		m->peer.flags[p] = reinterpret_cast<unsigned int*>(base + data_floats);
		m->peer.recv[p] = reinterpret_cast<uint2*>(base + data_floats + 16);
	}
	m->peer.rank = m->tp_rank; m->peer.size = m->tp_size; m->peer.stride = m->c.dim;
	m->peer_ready = true;
	return XALM_OK;
}

int xalm_cuda_comm_unique_id(void* id128) {
	if (!id128) return set_error(XALM_ERR_INVALID, "id is NULL");
	XALM_TRY(nccl_load());
	static_assert(sizeof(ncclUniqueId) == XALM_COMM_ID_BYTES, "ncclUniqueId size");
	ncclUniqueId id;
	XALM_NCCL_CHECK(g_nccl.GetUniqueId(&id));
	memcpy(id128, &id, sizeof id);
	return XALM_OK;
}

int xalm_cuda_comm_init(xalm_cuda_model* m, const void* id128) {
	if (!m || !id128) return set_error(XALM_ERR_INVALID, "model/id is NULL");
	if (m->tp_size == 1) return XALM_OK;
	if (m->finalized) return set_error(XALM_ERR_STATE, "comm_init must precede finalize");
	XALM_TRY(nccl_load());
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	ncclUniqueId id;
	memcpy(&id, id128, sizeof id);
	XALM_NCCL_CHECK(g_nccl.CommInitRank(&m->comm, m->tp_size, id, m->tp_rank));
	return XALM_OK;
}

// the rows / columns of tensor `piece` (full element shape er x ec) that rank R of P keeps (SURVEY.md 8e)
static void shard_range_of(const xalm_cuda_model* m, int piece, int er, int ec, int* r0, int* r1, int* c0, int* c1) {
	const int R = m->tp_rank;
	*r0 = 0; *r1 = er; *c0 = 0; *c1 = ec;
	switch (piece) {
		case 102: *r0 = R * m->vocab_l; *r1 = (R + 1) * m->vocab_l; break;                       // classifier: vocab rows
		case 100: break;                                                                          // embedding: replicated (gathered by row)
		case P_Q: *r0 = R * m->q_dim_l; *r1 = (R + 1) * m->q_dim_l; break;                        // heads
		case P_K: case P_V: *r0 = R * m->kv_dim_l; *r1 = (R + 1) * m->kv_dim_l; break;            // kv heads
		case P_O: *c0 = R * m->q_dim_l; *c1 = (R + 1) * m->q_dim_l; break;                        // input (quantised) axis
		case P_GATE: case P_UP: *r0 = R * m->hidden_l; *r1 = (R + 1) * m->hidden_l; break;
		case P_DOWN: *c0 = R * m->hidden_l; *c1 = (R + 1) * m->hidden_l; break;
	}
}

static int expected_shape(const xalm_cuda_model* m, int piece, int* er, int* ec, bool* is_norm) {
	const xalm_config& c = m->c;
	*er = 0; *ec = 0; *is_norm = false;
	switch (piece) { // model.cpp:83-114
		case 100: case 102: *er = c.vocab_size; *ec = c.dim; break;
		case 101: case P_ATT_NORM: case P_FFN_NORM: *er = c.dim; *is_norm = true; break;
		case P_Q: *er = m->q_dim; *ec = c.dim; break;
		case P_K: case P_V: *er = m->kv_dim; *ec = c.dim; break;
		case P_O: *er = c.dim; *ec = m->q_dim; break;
		case P_GATE: case P_UP: *er = c.hidden_dim; *ec = c.dim; break;
		case P_DOWN: *er = c.dim; *ec = c.hidden_dim; break;
		default: return set_error(XALM_ERR_INVALID, "unknown tensor");
	}
	return XALM_OK;
}

void* xalm_cuda_host_alloc(size_t nbytes) {
	void* p = nullptr;
	cudaError_t e = cudaMallocHost(&p, nbytes ? nbytes : 16);
	if (e != cudaSuccess) { set_error(XALM_ERR_CUDA, "cudaMallocHost(%zu) failed: %s", nbytes, cudaGetErrorString(e)); return nullptr; }
	return p;
}
void xalm_cuda_host_free(void* p) {
	if (p) cudaFreeHost(p);
}

int xalm_cuda_shard_range(xalm_cuda_model* m, const char* name, int* range4) {
	if (!m || !name || !range4) return set_error(XALM_ERR_INVALID, "NULL argument");
	int layer, piece, er, ec;
	bool is_norm;
	XALM_TRY(parse_tensor_name(name, m->c.n_layers, &layer, &piece));
	XALM_TRY(expected_shape(m, piece, &er, &ec, &is_norm));
	if (is_norm) { range4[0] = 0; range4[1] = er; range4[2] = 0; range4[3] = 1; return XALM_OK; }
	shard_range_of(m, piece, er, ec, &range4[0], &range4[1], &range4[2], &range4[3]);
	if (piece == 100 && m->c.tie_word_embeddings) { range4[0] = 0; range4[1] = er; } // also feeds the classifier shard: keep it whole
	return XALM_OK;
}

static int upload_impl(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank, const void* data, size_t nbytes,
                       const int* sub /* NULL = data is the full tensor; else {r0, r1, c0, c1} = the block data holds */);

int xalm_cuda_upload_tensor(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank, const void* data,
                            size_t nbytes) {
	return upload_impl(m, name, type_id, shape, rank, data, nbytes, nullptr);
}

int xalm_cuda_upload_tensor_shard(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank, const int* range4,
                                  const void* data, size_t nbytes) {
	if (!range4) return set_error(XALM_ERR_INVALID, "NULL argument");
	return upload_impl(m, name, type_id, shape, rank, data, nbytes, range4);
}

static int upload_impl(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank, const void* data, size_t nbytes,
                       const int* sub) {
	if (!m || !name || !shape || !data) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (m->finalized) return set_error(XALM_ERR_STATE, "upload after finalize");
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	const xalm_config& c = m->c;
	int layer, piece;
	XALM_TRY(parse_tensor_name(name, c.n_layers, &layer, &piece));
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	int er = 0, ec = 0;
	bool is_norm = false;
	XALM_TRY(expected_shape(m, piece, &er, &ec, &is_norm));
	if ((is_norm && (rank != 1 || shape[0] != er)) || (!is_norm && (rank != 2 || shape[0] != er || shape[1] != ec))) {
		if (rank == 2) return set_error(XALM_ERR_INVALID, "shape mismatch for %s: [%d, %d] vs [%d, %d] expected!", name, shape[0], shape[1], er, ec);
		return set_error(XALM_ERR_INVALID, "shape mismatch for %s: rank %d, [%d] vs [%d] expected!", name, rank, shape[0], er);
	}
	size_t elems = is_norm ? (size_t) er : (size_t) er * ec;
	if (elems % ti.block || (!is_norm && ec % ti.block)) return set_error(XALM_ERR_INVALID, "%s: row length %d is not a multiple of the block size %d", name, ec, ti.block);
	// shard upload: `data` holds only rows [sr0, sr1) x columns [sc0, sc1) of the tensor, which must be exactly what this rank keeps
	int sr0 = 0, sr1 = er, sc0 = 0, sc1 = ec;
	if (sub && !is_norm) {
		int need[4];
		XALM_TRY(xalm_cuda_shard_range(m, name, need));
		if (sub[0] != need[0] || sub[1] != need[1] || sub[2] != need[2] || sub[3] != need[3])
			return set_error(XALM_ERR_INVALID, "%s: rank %d keeps rows [%d, %d) x columns [%d, %d), the upload holds [%d, %d) x [%d, %d)", name, m->tp_rank,
			                 need[0], need[1], need[2], need[3], sub[0], sub[1], sub[2], sub[3]);
		sr0 = sub[0]; sr1 = sub[1]; sc0 = sub[2]; sc1 = sub[3];
		if ((sc1 - sc0) % ti.block) return set_error(XALM_ERR_INVALID, "%s: column range splits a block", name);
		elems = (size_t) (sr1 - sr0) * (sc1 - sc0);
	}
	if (nbytes != elems / ti.block * ti.bytes) return set_error(XALM_ERR_INVALID, "buffer size mismatch for %s: %zu vs %zu", name, nbytes, elems / ti.block * ti.bytes);
	m->uploaded = true;
	const uint8_t* host = (const uint8_t*) data;
	// geometry of `host`: its rows are (sc1 - sc0) elements long and its first row / column is (sr0, sc0) of the tensor
	auto put = [&](WMat& w, int dst_row, int r0, int r1, int c0, int c1) -> int {
		return upload_piece(w, dst_row, type_id, host, sc1 - sc0, r0 - sr0, r1 - sr0, c0 - sc0, c1 - sc0, m->staging, m->stream);
	};
	const int P = m->tp_size, R = m->tp_rank;

	if (is_norm) {
		if (type_id != XALM_F32 && type_id != XALM_BF16) return set_error(XALM_ERR_UNSUPPORTED, "rmsnorm: unsupported data type %d for %s", type_id, name);
		uint8_t* d = nullptr;
		XALM_TRY(m->da.alloc((void**) &d, nbytes));
		XALM_CUDA_CHECK(cudaMemcpy(d, host, nbytes, cudaMemcpyHostToDevice));
		if (piece == 101) { m->rms_final = d; m->rms_final_type = type_id; m->got_final_norm = true; }
		else if (piece == P_ATT_NORM) { m->layers[layer].rms_att = d; m->layers[layer].rms_att_type = type_id; m->layers[layer].got[piece] = true; }
		else { m->layers[layer].rms_ffn = d; m->layers[layer].rms_ffn_type = type_id; m->layers[layer].got[piece] = true; }
		return XALM_OK;
	}
	if (type_id == XALM_U8) return set_error(XALM_ERR_UNSUPPORTED, "matmul: unsupported data type: U8 (%s)", name);

	auto ensure = [&](WSlot& slot, int rows, int n, int glu_half = 0) -> int {
		if (slot.allocated) {
			if (slot.m.type != type_id) return set_error(XALM_ERR_UNSUPPORTED, "%s: tensors fused into one matrix must share a type (%d vs %d)", name, type_id, slot.m.type);
			return XALM_OK;
		}
		if (m->batched && !mma_takes(type_id, rows, n, glu_half))
			return set_error(XALM_ERR_UNSUPPORTED, "%s%s: a batched handle takes only matrices the tensor-core matvec can (the six integer block "
			                 "formats, rows a multiple of 16, input rows that fit the batch-1 kernel's shared memory); type %d, %d x %d", name,
			                 piece == 100 ? " (tied classifier)" : "", type_id, rows, n);
		XALM_TRY(alloc_wmat(m->da, slot.m, type_id, rows, n, glu_half, m->tp_size > 1, m->batched));
		slot.total_rows = rows;
		slot.allocated = true;
		return XALM_OK;
	};

	if (piece == 100 || piece == 102) {
		if (piece == 100) {
			// embedding table: replicated, kept in on-disk layout for the row gather
			if (sr0 != 0 || sr1 != er) return set_error(XALM_ERR_INVALID, "embed.weight is replicated: upload all of its rows");
			XALM_TRY(m->da.alloc((void**) &m->embed_raw, nbytes));
			XALM_CUDA_CHECK(cudaMemcpy(m->embed_raw, host, nbytes, cudaMemcpyHostToDevice));
			m->embed_type = type_id;
			m->embed_row_bytes = (size_t) c.dim / ti.block * ti.bytes;
			m->got_embed = true;
			if (!c.tie_word_embeddings) return XALM_OK;
			// tied: the classifier reads the same values (model.cpp:112-114) — built from this upload, no second host pass
		} else if (c.tie_word_embeddings) {
			return XALM_OK; // ignored, like the reference (model.cpp:112-114 loads embed.weight instead)
		}
		XALM_TRY(ensure(m->wcls, m->vocab_l, c.dim));
		XALM_TRY(put(m->wcls.m, 0, R * m->vocab_l, (R + 1) * m->vocab_l, 0, c.dim));
		m->got_cls = true;
		return XALM_OK;
	}

	LayerDev& L = m->layers[layer];
	L.piece_type[piece] = type_id;
	switch (piece) {
		case P_Q:
			XALM_TRY(ensure(L.wqkv, m->q_dim_l + 2 * m->kv_dim_l, c.dim));
			XALM_TRY(put(L.wqkv.m, 0, R * m->q_dim_l, (R + 1) * m->q_dim_l, 0, c.dim));
			break;
		case P_K:
			XALM_TRY(ensure(L.wqkv, m->q_dim_l + 2 * m->kv_dim_l, c.dim));
			XALM_TRY(put(L.wqkv.m, m->q_dim_l, R * m->kv_dim_l, (R + 1) * m->kv_dim_l, 0, c.dim));
			break;
		case P_V:
			XALM_TRY(ensure(L.wqkv, m->q_dim_l + 2 * m->kv_dim_l, c.dim));
			XALM_TRY(put(L.wqkv.m, m->q_dim_l + m->kv_dim_l, R * m->kv_dim_l, (R + 1) * m->kv_dim_l, 0, c.dim));
			break;
		case P_O: // row-split under TP = slice of the INPUT (quantised) axis
			XALM_TRY(ensure(L.wo, c.dim, m->q_dim_l));
			XALM_TRY(put(L.wo.m, 0, 0, c.dim, R * m->q_dim_l, (R + 1) * m->q_dim_l));
			break;
		case P_GATE:
			XALM_TRY(ensure(L.w13, 2 * m->hidden_l, c.dim, m->hidden_l));
			XALM_TRY(put(L.w13.m, 0, R * m->hidden_l, (R + 1) * m->hidden_l, 0, c.dim));
			break;
		case P_UP:
			XALM_TRY(ensure(L.w13, 2 * m->hidden_l, c.dim, m->hidden_l));
			XALM_TRY(put(L.w13.m, m->hidden_l, R * m->hidden_l, (R + 1) * m->hidden_l, 0, c.dim));
			break;
		case P_DOWN:
			XALM_TRY(ensure(L.w2, c.dim, m->hidden_l));
			XALM_TRY(put(L.w2.m, 0, 0, c.dim, R * m->hidden_l, (R + 1) * m->hidden_l));
			break;
	}
	L.got[piece] = true;
	(void) P;
	return XALM_OK;
}

} // extern "C" (templates below)

// kv_seq: the slot whose K/V cache the arguments point at (the batched kernels add step[i].slot * kv_slot to slot 0's)
static void fill_layer_args(xalm_cuda_model* m, int l, int kv_seq, MatvecArgs* qkv, AttnArgs* at, MatvecArgs* wo, MatvecArgs* w13,
                            MatvecArgs* w2) {
	const xalm_config& c = m->c;
	LayerDev& L = m->layers[l];
	const bool tp = m->tp_size > 1;
	__half* k_cache = L.k_cache + (size_t) kv_seq * m->kv_slot;
	__half* v_cache = L.v_cache + (size_t) kv_seq * m->kv_slot;
	{ // attention pre-norm + q,k,v + clip + rope + KV write (+ sinks)
		MatvecArgs a = {};
		a.w = L.wqkv.m; a.x = m->x; a.n = c.dim; a.d = m->q_dim_l + 2 * m->kv_dim_l; a.epi = EPI_QKV;
		a.norm_w = L.rms_att; a.norm_type = L.rms_att_type; a.norm_eps = c.norm_eps;
		a.out = m->q; a.step = m->d_step; a.k_cache = k_cache; a.v_cache = v_cache; a.rope_freq = m->rope_freq;
		a.q_dim = m->q_dim_l; a.kv_dim = m->kv_dim_l; a.head_dim = c.head_dim; a.qkv_clip = c.qkv_clip;
		*qkv = a;
	}
	{
		AttnArgs a = {};
		a.q = m->q; a.k_cache = k_cache; a.v_cache = v_cache; a.out = m->xb2; a.step = m->d_step; a.kv_len_fixed = -1;
		a.n_kv_heads = m->n_kv_heads_l; a.n_splits = m->attn_splits; a.min_split = tune("attn_min_split");
		a.part_acc = m->attn_acc; a.part_ml = m->attn_ml; a.tickets = m->tickets;
		*at = a;
	}
	{ // Wo + residual
		MatvecArgs a = {};
		a.w = L.wo.m; a.x = m->xb2; a.n = m->q_dim_l; a.d = c.dim;
		a.epi = tp ? EPI_STORE : EPI_RESIDUAL; a.out = tp ? m->part : m->x;
		*wo = a;
	}
	{ // ffn pre-norm + W1,W3 + act*gate
		MatvecArgs a = {};
		a.w = L.w13.m; a.x = m->x; a.n = c.dim; a.d = m->hidden_l; a.epi = EPI_GLU; a.glu_off = m->hidden_l; a.act = c.act;
		a.norm_w = L.rms_ffn; a.norm_type = L.rms_ffn_type; a.norm_eps = c.norm_eps; a.out = m->hb;
		*w13 = a;
	}
	{ // W2 + residual
		MatvecArgs a = {};
		a.w = L.w2.m; a.x = m->hb; a.n = m->hidden_l; a.d = c.dim;
		a.epi = tp ? EPI_STORE : EPI_RESIDUAL; a.out = tp ? m->part : m->x;
		*w2 = a;
	}
}

// bytes of a matrix's first plane: in fragment layout s0 bytes hold a tile row of 16 matrix rows (alloc_wmat), else one row
static size_t plane0_bytes(const WMat& w) { return w.s0 * (size_t) (w.layout_frag ? w.rows / MMA_RC : w.rows); }

// the tail-prefetch chain of layer l: every kernel warms L2 with the first pf_mb MB of the next kernel's weights
static void chain_tail_prefetch(xalm_cuda_model* m, int l, int mode, int pf_mb, AttnArgs* at, MatvecArgs* wo, MatvecArgs* w13, MatvecArgs* w2) {
	auto head = [&](const WMat& w, const uint8_t** ptr, unsigned long long* bytes) {
		*ptr = w.p0;
		*bytes = std::min<unsigned long long>(plane0_bytes(w), (unsigned long long) pf_mb << 20);
	};
	head(wo->w, &at->pf_ptr, &at->pf_bytes);
	head(w13->w, &wo->pf_ptr, &wo->pf_bytes);
	head(w2->w, &w13->pf_ptr, &w13->pf_bytes);
	if (l + 1 < m->c.n_layers) head(m->layers[l + 1].wqkv.m, &w2->pf_ptr, &w2->pf_bytes);
	else if (mode == XALM_OUTPUT_LOGITS) head(m->wcls.m, &w2->pf_ptr, &w2->pf_bytes);
}

// a step's first kernel: one embedding row per entry, launched without PDL, so it starts only after the previous step has completed
static int launch_embed(xalm_cuda_model* m, int n, cudaStream_t s) {
	cudaError_t e = launch(embed_rows_kernel, dim3(4, n), dim3(256), s, false, m->embed_type, (const uint8_t*) m->embed_raw, m->embed_row_bytes,
	                       m->c.dim, (const StepParams*) m->d_step, m->x);
	if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "embed launch failed: %s", cudaGetErrorString(e));
	return XALM_OK;
}

extern "C" {

// ---- the per-token kernel sequence ---------------------------------------------------------------------------
static int enqueue_token(xalm_cuda_model* m, int mode, cudaStream_t s, int* n_launches) {
	const xalm_config& c = m->c;
	const bool pdl = tune("pdl") != 0;
	const bool tp = m->tp_size > 1;
	int nl = 0;
	cudaError_t e;
	XALM_TRY(launch_embed(m, 1, s));
	nl++;
	const int G = c.n_heads / c.n_kv_heads;
	// fused tensor-parallel exchange: Wo / W2 push their partial rows to every rank, the next norm-prologue kernel receives
	const bool fused = tp && m->peer_ready && m->tp_fused;
	float* X[2] = {m->x, m->x_alt};
	int cur = 0; // which buffer holds the residual stream
	auto set_push = [&](MatvecArgs& a, int idx) {
		const int slot = idx & 1;
		a.epi = EPI_STORE; a.out = nullptr; a.step = m->d_step;
		a.n_push = m->tp_size; a.push_idx = idx;
		for (int p = 0; p < m->tp_size; p++) a.push_dst[p] = m->peer.recv[p] + (size_t) (slot * 8 + m->tp_rank) * c.dim;
	};
	auto set_recv = [&](MatvecArgs& a, int idx) {
		const int slot = idx & 1;
		a.step = m->d_step; a.n_recv = m->tp_size; a.recv_idx = idx;
		a.recv = m->peer.recv[m->tp_rank] + (size_t) slot * 8 * c.dim;
		a.xl = m->xl + (size_t) slot * c.dim;
		a.err_flag = m->h_err; // pinned host word, written over PCIe only when a wait gives up
		a.x = X[cur]; a.x_out = X[cur ^ 1];
		cur ^= 1;
	};
	// Wo / W2 + residual; idx: the exchange (2l, 2l + 1) under tensor parallelism
	auto residual = [&](MatvecArgs a, int idx) -> int {
		if (tp && m->peer_ready && !fused) a.out = m->xchg + (size_t) (idx & 1) * c.dim;
		XALM_TRY(launch_matvec(a, s, pdl));
		nl++;
		if (fused) {
		} else if (tp && m->peer_ready) {
			e = launch(peer_allreduce_residual_kernel, dim3(4), dim3(256), s, pdl, m->peer, m->x, c.dim, idx, (const StepParams*) m->d_step);
			if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "peer allreduce launch failed: %s", cudaGetErrorString(e));
			nl++;
		} else if (tp) {
			XALM_NCCL_CHECK(g_nccl.AllReduce(m->part, m->part, c.dim, ncclFloat32, ncclSum, m->comm, s));
			e = launch(residual_add_kernel, dim3(8), dim3(256), s, false, m->x, (const float*) m->part, c.dim);
			if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "residual launch failed: %s", cudaGetErrorString(e));
			nl += 2;
		}
		return XALM_OK;
	};
	for (int l = 0; l < c.n_layers; l++) {
		LayerDev& L = m->layers[l];
		MatvecArgs a_qkv, a_wo, a_w13, a_w2;
		AttnArgs a_at;
		fill_layer_args(m, l, m->cur_seq, &a_qkv, &a_at, &a_wo, &a_w13, &a_w2);
		if (fused) {
			if (l > 0) set_recv(a_qkv, 2 * l - 1);
			set_push(a_wo, 2 * l);
			set_recv(a_w13, 2 * l);
			set_push(a_w2, 2 * l + 1);
		}
		if (const int pf_mb = tune("tail_prefetch_mb")) {
			a_qkv.pf_kv = 1;
			chain_tail_prefetch(m, l, mode, pf_mb, &a_at, &a_wo, &a_w13, &a_w2);
			// ... and with the rmsnorm weights the next norm-fused kernel asks for before its dependency wait
			auto norm_bytes = [&](int type) { return (unsigned int) ((size_t) c.dim * (type == XALM_F32 ? 4 : 2)); };
			a_wo.pf_norm_ptr = (const uint8_t*) L.rms_ffn; a_wo.pf_norm_bytes = norm_bytes(L.rms_ffn_type);
			if (l + 1 < c.n_layers) {
				a_w2.pf_norm_ptr = (const uint8_t*) m->layers[l + 1].rms_att; a_w2.pf_norm_bytes = norm_bytes(m->layers[l + 1].rms_att_type);
			} else if (mode == XALM_OUTPUT_LOGITS) {
				a_w2.pf_norm_ptr = (const uint8_t*) m->rms_final; a_w2.pf_norm_bytes = norm_bytes(m->rms_final_type);
			}
		}
		XALM_TRY(launch_matvec(a_qkv, s, pdl)); // attention pre-norm + q,k,v + clip + rope + KV write (+ sinks)
		XALM_TRY(launch_attn(a_at, c.head_dim, G, s, pdl));
		nl += 2;
		XALM_TRY(residual(a_wo, 2 * l));
		XALM_TRY(launch_matvec(a_w13, s, pdl && (!tp || m->peer_ready))); // ffn pre-norm + W1,W3 + act*gate
		nl++;
		XALM_TRY(residual(a_w2, 2 * l + 1));
	}
	if (fused && mode != XALM_OUTPUT_LOGITS && c.n_layers > 0) { // nobody else receives the token's last exchange: drain it
		const int idx = 2 * c.n_layers - 1;
		e = launch(tp_drain_kernel, dim3(1), dim3(1024), s, pdl, (const uint2*) (m->peer.recv[m->tp_rank] + (size_t) (idx & 1) * 8 * c.dim),
		           m->tp_size, c.dim, idx, (const StepParams*) m->d_step, m->h_err);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "tp drain launch failed: %s", cudaGetErrorString(e));
		nl++;
	}
	if (mode == XALM_OUTPUT_LOGITS) { // final norm + classifier (infer.cpp:625-637)
		MatvecArgs a = {};
		a.w = m->wcls.m; a.x = m->x; a.n = c.dim; a.d = m->vocab_l; a.epi = EPI_STORE;
		a.norm_w = m->rms_final; a.norm_type = m->rms_final_type; a.norm_eps = c.norm_eps; a.out = m->logits;
		if (fused && c.n_layers > 0) set_recv(a, 2 * c.n_layers - 1);
		XALM_TRY(launch_matvec(a, s, pdl && (!tp || fused)));
		nl++;
		if (tp) {
			XALM_NCCL_CHECK(g_nccl.AllGather(m->logits, m->logits_full, m->vocab_l, ncclFloat32, m->comm, s));
			nl++;
		}
	}
	if (n_launches) *n_launches = nl;
	return XALM_OK;
}

int xalm_cuda_finalize(xalm_cuda_model* m) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (m->finalized) return XALM_OK;
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	const xalm_config& c = m->c;
	if (!m->got_embed) return set_error(XALM_ERR_STATE, "missing tensor embed.weight");
	if (!m->got_final_norm) return set_error(XALM_ERR_STATE, "missing tensor output.norm.weight");
	if (!m->got_cls) return set_error(XALM_ERR_STATE, "missing tensor output.weight");
	static const char* names[9] = {"attn.norm", "mlp.norm", "attn.q", "attn.k", "attn.v", "attn.down", "mlp.gate", "mlp.down", "mlp.up"};
	for (int l = 0; l < c.n_layers; l++)
		for (int p = 0; p < 9; p++)
			if (!m->layers[l].got[p]) return set_error(XALM_ERR_STATE, "missing tensor l.%d.%s.weight", l, names[p]);
	if (m->tp_size > 1 && !m->comm) return set_error(XALM_ERR_STATE, "tp_size %d but xalm_cuda_comm_init was not called", m->tp_size);
	if (m->tp_size > 1 && 2 * c.n_layers > 1024)
		return set_error(XALM_ERR_UNSUPPORTED, "tensor parallel: %d layers need %d exchange tags per token, the tag space has 1024", c.n_layers, 2 * c.n_layers);
	if (m->staging.p) { cudaFree(m->staging.p); m->staging.p = nullptr; m->staging.cap = 0; }

	auto fzero = [&](float** p, size_t n) -> int {
		XALM_TRY(m->da.alloc((void**) p, n * sizeof(float)));
		XALM_CUDA_CHECK(cudaMemset(*p, 0, n * sizeof(float)));
		return XALM_OK;
	};
	// one row per sequence slot (the single-sequence calls use row 0)
	const int S = m->max_seqs;
	XALM_TRY(fzero(&m->x, (size_t) S * c.dim));
	XALM_TRY(fzero(&m->xb2, (size_t) S * m->q_dim_l));
	XALM_TRY(fzero(&m->hb, (size_t) S * m->hidden_l));
	XALM_TRY(fzero(&m->q, (size_t) S * m->q_dim_l));
	XALM_TRY(fzero(&m->logits, (size_t) S * m->vocab_l));
	if (m->batched) {
		const int nmax = std::max(c.dim, std::max(m->q_dim_l, m->hidden_l));
		XALM_TRY(m->da.alloc((void**) &m->ximg, (size_t) nmax / 32 * ((S + 1) / 2) * MMB_PAIR));
		XALM_CUDA_CHECK(cudaMemset(m->ximg, 0, (size_t) nmax / 32 * ((S + 1) / 2) * MMB_PAIR));
		XALM_TRY(fzero(&m->nscale, S));
	}
	XALM_TRY(fzero(&m->part, c.dim));
	XALM_TRY(fzero(&m->x_alt, c.dim));
	XALM_TRY(m->da.alloc((void**) &m->xl, (size_t) 2 * c.dim * sizeof(uint2)));
	XALM_CUDA_CHECK(cudaMemset(m->xl, 0, (size_t) 2 * c.dim * sizeof(uint2)));
	if (m->tp_size > 1 && m->peer_ready && tune("tp_fused")) {
		auto takes = [&](const WMat& w, int n) { return w.layout_frag || ((w.layout_units || tma_eligible(w, n)) && w.rows % 8 == 0 && n % 256 == 0); };
		bool ok = takes(m->wcls.m, c.dim) && (size_t) c.dim * sizeof(float) <= 64 * 1024;
		for (auto& L : m->layers)
			ok = ok && takes(L.wqkv.m, c.dim) && takes(L.wo.m, m->q_dim_l) && takes(L.w13.m, c.dim) && takes(L.w2.m, m->hidden_l);
		m->tp_fused = ok;
	}
	if (m->tp_size > 1) {
		XALM_TRY(fzero(&m->logits_full, c.vocab_size));
		XALM_TRY(m->da.alloc((void**) &m->prefill_status, sizeof(int)));
	} else {
		m->logits_full = m->logits;
	}
	m->kv_slot = (size_t) c.max_seq_len * m->kv_dim_l;
	const size_t kv_elems = m->kv_slot * S;
	for (auto& L : m->layers) {
		XALM_TRY(m->da.alloc((void**) &L.k_cache, kv_elems * sizeof(__half)));
		XALM_TRY(m->da.alloc((void**) &L.v_cache, kv_elems * sizeof(__half)));
		XALM_CUDA_CHECK(cudaMemset(L.k_cache, 0, kv_elems * sizeof(__half)));
		XALM_CUDA_CHECK(cudaMemset(L.v_cache, 0, kv_elems * sizeof(__half)));
	}
	if (m->batched) {
		std::vector<__half*> table;
		for (auto& L : m->layers) { table.push_back(L.k_cache); table.push_back(L.v_cache); }
		XALM_TRY(m->da.alloc((void**) &m->kv_table, table.size() * sizeof(__half*)));
		XALM_CUDA_CHECK(cudaMemcpy(m->kv_table, table.data(), table.size() * sizeof(__half*), cudaMemcpyHostToDevice));
	}
	const std::vector<float> freq = rope_freq_table(c.head_dim, c.rotary_dim, c.rope_theta);
	XALM_TRY(m->da.alloc((void**) &m->rope_freq, freq.size() * sizeof(float)));
	XALM_CUDA_CHECK(cudaMemcpy(m->rope_freq, freq.data(), freq.size() * sizeof(float), cudaMemcpyHostToDevice));
	const int G = c.n_heads / c.n_kv_heads;
	m->attn_splits = attn_auto_splits(m->n_kv_heads_l);
	// the last-CTA merge parks 3 floats per (split, head) in the 8 x G x head_dim floats of the per-warp partial area (attention.cuh)
	if (m->attn_splits > 8 * c.head_dim / 3) m->attn_splits = 8 * c.head_dim / 3;
	XALM_TRY(fzero(&m->attn_acc, (size_t) S * m->n_kv_heads_l * m->attn_splits * G * c.head_dim));
	XALM_TRY(fzero(&m->attn_ml, (size_t) S * m->n_kv_heads_l * m->attn_splits * G * 2));
	XALM_TRY(m->da.alloc((void**) &m->tickets, S * m->n_kv_heads_l * sizeof(unsigned int)));
	XALM_CUDA_CHECK(cudaMemset(m->tickets, 0, S * m->n_kv_heads_l * sizeof(unsigned int)));
	XALM_TRY(m->da.alloc((void**) &m->d_step, S * sizeof(StepParams)));
	XALM_CUDA_CHECK(cudaMallocHost((void**) &m->h_step, 64 * S * sizeof(StepParams)));
	XALM_CUDA_CHECK(cudaMemset(m->d_step, 0, S * sizeof(StepParams)));
	XALM_CUDA_CHECK(cudaMallocHost((void**) &m->h_logits, (size_t) S * c.vocab_size * sizeof(float)));
	XALM_CUDA_CHECK(cudaMallocHost((void**) &m->h_err, 64));
	memset(m->h_err, 0, 64);
	XALM_TRY(m->da.alloc((void**) &m->d_argmax, 64));
	XALM_CUDA_CHECK(cudaMemset(m->d_argmax, 0, 64));
	XALM_CUDA_CHECK(cudaMallocHost((void**) &m->h_argmax, 64));
	XALM_CUDA_CHECK(cudaDeviceSynchronize());
	m->finalized = true;
	return XALM_OK;
}

// the batched kernel sequence: n entries (several sequence slots, or consecutive positions of one), one pass over the weights
static int enqueue_batch(xalm_cuda_model* m, int mode, int n, cudaStream_t s, int* n_launches) {
	const xalm_config& c = m->c;
	const bool pdl = tune("pdl") != 0;
	const int G = c.n_heads / c.n_kv_heads;
	int nl = 0;
	XALM_TRY(launch_embed(m, n, s));
	nl++;
	auto io = [&](int x_stride, int out_stride) { return BatchIo{n, x_stride, out_stride, m->ximg, m->nscale, m->kv_slot}; };
	for (int l = 0; l < c.n_layers; l++) {
		MatvecArgs a_qkv, a_wo, a_w13, a_w2;
		AttnArgs a_at;
		fill_layer_args(m, l, 0, &a_qkv, &a_at, &a_wo, &a_w13, &a_w2);
		a_at.q_stride = m->q_dim_l; a_at.kv_slot = m->kv_slot;
		if (const int pf_mb = tune("tail_prefetch_mb")) chain_tail_prefetch(m, l, mode, pf_mb, &a_at, &a_wo, &a_w13, &a_w2);
		XALM_TRY(launch_matvec_batch(a_qkv, io(c.dim, m->q_dim_l), s, pdl));
		XALM_TRY(launch_attn(a_at, c.head_dim, G, s, pdl, n));
		XALM_TRY(launch_matvec_batch(a_wo, io(m->q_dim_l, c.dim), s, pdl));
		XALM_TRY(launch_matvec_batch(a_w13, io(c.dim, m->hidden_l), s, pdl));
		XALM_TRY(launch_matvec_batch(a_w2, io(m->hidden_l, c.dim), s, pdl));
		nl += 9;
	}
	if (mode == XALM_OUTPUT_LOGITS) {
		MatvecArgs a = {};
		a.w = m->wcls.m; a.x = m->x; a.n = c.dim; a.d = m->vocab_l; a.epi = EPI_STORE;
		a.norm_w = m->rms_final; a.norm_type = m->rms_final_type; a.norm_eps = c.norm_eps; a.out = m->logits;
		XALM_TRY(launch_matvec_batch(a, io(c.dim, m->vocab_l), s, pdl));
		nl += 2;
	}
	if (n_launches) *n_launches = nl;
	return XALM_OK;
}

// Enqueue the kernels of one step: n = 0 the single-sequence sequence, else a batched step of n entries.  With the graph knob on
// the step is captured into a CUDA graph on first use and replayed after that.
static int run_step(xalm_cuda_model* m, int mode, int n) {
	cudaStream_t s = m->stream;
	auto enqueue = [&](int* nl) { return n ? enqueue_batch(m, mode, n, s, nl) : enqueue_token(m, mode, s, nl); };
	if (!tune("graph")) return enqueue(&m->last_launches);
	const std::pair<int, int> key(mode, n);
	auto it = m->graphs.find(key);
	if (it == m->graphs.end()) {
		cudaGraph_t g = nullptr;
		XALM_CUDA_CHECK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
		int nl = 0;
		int rc = enqueue(&nl);
		cudaError_t e = cudaStreamEndCapture(s, &g);
		if (rc != XALM_OK) { if (g) cudaGraphDestroy(g); return rc; }
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
		cudaGraphExec_t ge = nullptr;
		e = cudaGraphInstantiate(&ge, g, 0);
		cudaGraphDestroy(g);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
		it = m->graphs.emplace(key, StepGraph{ge, nl}).first;
	}
	XALM_CUDA_CHECK(cudaGraphLaunch(it->second.exec, s));
	m->last_launches = it->second.launches;
	return XALM_OK;
}

// the next row group of the pinned StepParams ring, once the copy that last read it has run
static int claim_step_rows(xalm_cuda_model* m, StepParams** rows) {
	const int slot = m->step_slot;
	m->step_slot = (slot + 1) % 64;
	if (m->h_step_ev_used[slot]) XALM_CUDA_CHECK(cudaEventSynchronize(m->h_step_ev[slot]));
	else { XALM_CUDA_CHECK(cudaEventCreateWithFlags(&m->h_step_ev[slot], cudaEventDisableTiming)); m->h_step_ev_used[slot] = true; }
	*rows = m->h_step + (size_t) slot * m->max_seqs;
	return XALM_OK;
}

// copy the first n rows of a claimed row group to the device, and mark the group free again once the copy has run
static int upload_step_rows(xalm_cuda_model* m, const StepParams* rows, int n) {
	const int slot = (int) ((rows - m->h_step) / m->max_seqs);
	XALM_CUDA_CHECK(cudaMemcpyAsync(m->d_step, rows, (size_t) n * sizeof(StepParams), cudaMemcpyHostToDevice, m->stream));
	XALM_CUDA_CHECK(cudaEventRecord(m->h_step_ev[slot], m->stream));
	return XALM_OK;
}

int xalm_cuda_forward_async(xalm_cuda_model* m, int token, int pos, int mode) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "forward before finalize");
	if (mode != XALM_HYDRATE_KV_CACHE && mode != XALM_OUTPUT_LOGITS) return set_error(XALM_ERR_INVALID, "bad mode %d", mode);
	const xalm_config& c = m->c;
	if (token < 0 || token >= c.vocab_size) return set_error(XALM_ERR_INVALID, "token %d out of range [0,%d)", token, c.vocab_size);
	if (pos < 0) return set_error(XALM_ERR_INVALID, "negative position");
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	StepParams* sp = nullptr;
	XALM_TRY(claim_step_rows(m, &sp));
	fill_step_entry(c, *sp, token, pos, mode);
	sp->kv_fresh = sp->kv_pos;
	sp->ar_base = m->token_serial++ * 1024u; // 2 x n_layers <= 1024 exchanges per token; wraps consistently on every rank
	sp->slot = 0;                            // the single-sequence kernels address the cache of cur_seq directly
	XALM_TRY(upload_step_rows(m, sp, 1));
	return run_step(m, mode, 0);
}

// a tensor-parallel wait that timed out inside a kernel (a peer died): report it instead of hanging
static int check_tp_error(xalm_cuda_model* m) {
	if (m->h_err && *reinterpret_cast<volatile unsigned int*>(m->h_err))
		return set_error(XALM_ERR_COMM, "tensor-parallel exchange timed out waiting for a peer rank");
	return XALM_OK;
}

int xalm_cuda_sync(xalm_cuda_model* m) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	return check_tp_error(m);
}

// after a step of n entries (1 for the single-sequence calls): copy their logits back (logits_host may be NULL) and wait
static int finish_step(xalm_cuda_model* m, int n, int mode, float* logits_host) {
	const size_t bytes = (size_t) n * m->c.vocab_size * sizeof(float);
	if (mode == XALM_OUTPUT_LOGITS && logits_host) {
		XALM_CUDA_CHECK(cudaMemcpyAsync(m->h_logits, m->logits_full, bytes, cudaMemcpyDeviceToHost, m->stream));
		XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
		if (logits_host != m->h_logits) memcpy(logits_host, m->h_logits, bytes);
	} else {
		XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	}
	return check_tp_error(m);
}

// after a step of n entries with logits: Sampler::sample_argmax of every row on the device, next_tokens[i] for entry i
static int finish_step_argmax(xalm_cuda_model* m, int n, int* next_tokens) {
	argmax_rows_kernel<<<n, 1024, 0, m->stream>>>(m->logits_full, m->c.vocab_size, m->d_argmax);
	XALM_CUDA_CHECK(cudaGetLastError());
	// a pinned buffer of its own: the host logits buffer (InferenceState::_logits alias) stays untouched
	XALM_CUDA_CHECK(cudaMemcpyAsync(m->h_argmax, m->d_argmax, (size_t) n * sizeof(int), cudaMemcpyDeviceToHost, m->stream));
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	XALM_TRY(check_tp_error(m));
	memcpy(next_tokens, m->h_argmax, (size_t) n * sizeof(int));
	return XALM_OK;
}

int xalm_cuda_forward(xalm_cuda_model* m, int token, int pos, int mode, float* logits_host) {
	XALM_TRY(xalm_cuda_forward_async(m, token, pos, mode));
	return finish_step(m, 1, mode, logits_host);
}

// Model::forward + Sampler::sample_argmax with the sampler on the device: 4 bytes come back instead of vocab * 4
int xalm_cuda_forward_argmax(xalm_cuda_model* m, int token, int pos, int* next_token) {
	if (!next_token) return set_error(XALM_ERR_INVALID, "next_token is NULL");
	XALM_TRY(xalm_cuda_forward_async(m, token, pos, XALM_OUTPUT_LOGITS));
	return finish_step_argmax(m, 1, next_token);
}

// The loop forward(HYDRATE) x (n_in - 1), forward_argmax, then forward_argmax of each result, with one host synchronisation.  The
// steps fed from `tokens` are set up by the host as xalm_cuda_forward_async sets them up; after every logits step
// argmax_next_step_kernel writes the greedy token to d_argmax[i] and, but for the last, the next step's row of d_step, and that
// step's graph (the single-sequence logits graph) is replayed without an upload.  The n_out tokens come back in one copy.
int xalm_cuda_forward_greedy(xalm_cuda_model* m, int n_in, const int* tokens, int pos, int n_out, int* out_tokens) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (m->tp_size > 1)
		return set_error(XALM_ERR_UNSUPPORTED, "forward_greedy: tensor-parallel exchange tags are assigned per token on the host (tp_size %d)", m->tp_size);
	if (!m->finalized) return set_error(XALM_ERR_STATE, "forward_greedy before finalize");
	if (n_in < 1 || n_in > 8) return set_error(XALM_ERR_INVALID, "forward_greedy: n_in = %d not in [1, 8]", n_in);
	if (n_out < 1 || n_out > 16) return set_error(XALM_ERR_INVALID, "forward_greedy: n_out = %d not in [1, 16]", n_out); // d_argmax holds 16
	if (!tokens || !out_tokens) return set_error(XALM_ERR_INVALID, "NULL argument");
	const xalm_config& c = m->c;
	for (int j = 0; j < n_in; j++)
		if (tokens[j] < 0 || tokens[j] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "token %d out of range [0,%d)", tokens[j], c.vocab_size);
	if (pos < 0) return set_error(XALM_ERR_INVALID, "negative position");
	if (pos > INT_MAX - n_in - n_out) return set_error(XALM_ERR_INVALID, "forward_greedy: position %d overflows", pos);
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	for (int j = 0; j < n_in; j++) XALM_TRY(xalm_cuda_forward_async(m, tokens[j], pos + j, j + 1 < n_in ? XALM_HYDRATE_KV_CACHE : XALM_OUTPUT_LOGITS));
	for (int i = 0; i < n_out; i++) {
		const bool last = i + 1 == n_out;
		StepParams* next = last ? nullptr : m->d_step;
		cudaError_t e = launch(argmax_next_step_kernel, dim3(1), dim3(1024), m->stream, false, (const float*) m->logits_full, c.vocab_size,
		                       m->d_argmax + i, next, c, pos + n_in + i, m->token_serial * 1024u);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "argmax launch failed: %s", cudaGetErrorString(e));
		if (last) break;
		m->token_serial++; // the step's ar_base, as xalm_cuda_forward_async counts them
		XALM_TRY(run_step(m, XALM_OUTPUT_LOGITS, 0));
	}
	XALM_CUDA_CHECK(cudaMemcpyAsync(m->h_argmax, m->d_argmax, (size_t) n_out * sizeof(int), cudaMemcpyDeviceToHost, m->stream));
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	XALM_TRY(check_tp_error(m));
	memcpy(out_tokens, m->h_argmax, (size_t) n_out * sizeof(int));
	return XALM_OK;
}

// ---- batched decode: several sequence slots, one pass over the weights per step ------------------------------------------
int xalm_cuda_set_batch(xalm_cuda_model* m, int max_seqs) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (m->tp_size > 1) return set_error(XALM_ERR_UNSUPPORTED, "set_batch: batched decode runs on one GPU (tp_size %d)", m->tp_size);
	if (m->uploaded || m->finalized) return set_error(XALM_ERR_STATE, "set_batch must precede the first upload");
	if (max_seqs < 1 || max_seqs > MMB_MAX_SEQS) return set_error(XALM_ERR_INVALID, "set_batch: max_seqs %d not in [1, %d]", max_seqs, MMB_MAX_SEQS);
	m->max_seqs = max_seqs;
	m->batched = true;
	return XALM_OK;
}

int xalm_cuda_select_seq(xalm_cuda_model* m, int seq) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (seq < 0 || seq >= m->max_seqs) return set_error(XALM_ERR_INVALID, "select_seq: slot %d not in [0, %d)", seq, m->max_seqs);
	if (seq == m->cur_seq) return XALM_OK;
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	for (auto it = m->graphs.begin(); it != m->graphs.end();) // the single-sequence graphs hold the previous slot's cache pointers
		if (it->first.second == 0) { cudaGraphExecDestroy(it->second.exec); it = m->graphs.erase(it); }
		else ++it;
	m->cur_seq = seq;
	return XALM_OK;
}

// The checks every call on a batched handle's slots starts with: a finalized batched handle, 1 <= n <= max_seqs.
static int check_batched(xalm_cuda_model* m, const char* fn, int n) {
	if (!m) return set_error(XALM_ERR_INVALID, "model is NULL");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "%s before finalize", fn);
	if (!m->batched) return set_error(XALM_ERR_STATE, "%s on a handle without xalm_cuda_set_batch", fn);
	if (n < 1 || n > m->max_seqs) return set_error(XALM_ERR_INVALID, "%s: n = %d not in [1, %d]", fn, n, m->max_seqs);
	return XALM_OK;
}

// Claim a row group of the StepParams ring, let fill(rows) write its n entries, upload them and run the batched step of n entries.
extern "C++" {
template <class Fill>
static int run_batched_rows(xalm_cuda_model* m, int n, int mode, Fill fill) {
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	StepParams* sp = nullptr;
	XALM_TRY(claim_step_rows(m, &sp));
	fill(sp);
	XALM_TRY(upload_step_rows(m, sp, n));
	return run_step(m, mode, n);
}
}

// One step of n entries: entry i drives slot seqs[i] with tokens[i] at pos[i].  spans = false (forward_batch): every slot at most
// once.  spans = true (forward_spans): a slot may take several consecutive positions, all inside the window; the attention of
// each such entry re-reads, after its dependency wait, every row the step writes for its slot up to its own (kv_fresh .. kv_pos).
// Everything is validated before anything is enqueued, so a refusal leaves every cache untouched.
static int forward_step_async(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, int mode, bool spans) {
	const char* fn = spans ? "forward_spans" : "forward_batch";
	XALM_TRY(check_batched(m, fn, n));
	if (mode != XALM_HYDRATE_KV_CACHE && mode != XALM_OUTPUT_LOGITS) return set_error(XALM_ERR_INVALID, "bad mode %d", mode);
	if (!seqs || !tokens || !pos) return set_error(XALM_ERR_INVALID, "NULL argument");
	const xalm_config& c = m->c;
	int first[MMB_MAX_SEQS], last[MMB_MAX_SEQS]; // per slot: its first and latest entry so far (-1: none)
	for (int s = 0; s < MMB_MAX_SEQS; s++) first[s] = last[s] = -1;
	for (int i = 0; i < n; i++) {
		const int s = seqs[i];
		if (s < 0 || s >= m->max_seqs) return set_error(XALM_ERR_INVALID, "%s: slot %d not in [0, %d)", fn, s, m->max_seqs);
		if (last[s] >= 0 && !spans) return set_error(XALM_ERR_INVALID, "forward_batch: slot %d named twice", s);
		if (last[s] >= 0 && (long long) pos[i] != (long long) pos[last[s]] + 1)
			return set_error(XALM_ERR_INVALID, "forward_spans: slot %d takes position %d after %d (a span's positions are consecutive)", s, pos[i], pos[last[s]]);
		if (first[s] < 0) first[s] = i;
		last[s] = i;
		if (tokens[i] < 0 || tokens[i] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "token %d out of range [0,%d)", tokens[i], c.vocab_size);
		if (pos[i] < 0) return set_error(XALM_ERR_INVALID, "negative position");
	}
	for (int s = 0; s < m->max_seqs; s++) // positions of a span increase, so its last one is its largest
		if (first[s] != last[s] && pos[last[s]] >= c.max_seq_len)
			return set_error(XALM_ERR_INVALID, "forward_spans: the span of slot %d reaches position %d, spans stay below max_seq_len %d", s,
			                 pos[last[s]], c.max_seq_len);
	return run_batched_rows(m, n, mode, [&](StepParams* sp) {
		for (int i = 0; i < n; i++) {
			fill_step_entry(c, sp[i], tokens[i], pos[i], mode);
			sp[i].kv_fresh = sp[first[seqs[i]]].kv_pos; // == kv_pos unless an earlier entry of this step drives the same slot
			sp[i].ar_base = 0;
			sp[i].slot = seqs[i];
		}
	});
}

// One step of a tree of n drafted nodes of one slot (xalm_cuda_forward_tree): node i decodes tokens[i] at position pos + depth(i),
// writes its K/V to row pos + i, and its attention reads rows pos .. pos + depth(i) through the row map (StepParams::tree), which
// sends depth e to the row of its ancestor at depth e.  Everything is validated before anything is enqueued.
static int forward_tree_async(xalm_cuda_model* m, int slot, int n, const int* tokens, const int* parents, int pos) {
	XALM_TRY(check_batched(m, "forward_tree", n));
	if (!tokens || !parents) return set_error(XALM_ERR_INVALID, "NULL argument");
	const xalm_config& c = m->c;
	if (slot < 0 || slot >= m->max_seqs) return set_error(XALM_ERR_INVALID, "forward_tree: slot %d not in [0, %d)", slot, m->max_seqs);
	if (pos < 0) return set_error(XALM_ERR_INVALID, "negative position");
	if (pos > c.max_seq_len - n)
		return set_error(XALM_ERR_INVALID, "forward_tree: rows %d .. %d reach max_seq_len %d, trees stay below the window", pos, pos + n - 1,
		                 c.max_seq_len);
	int depth[MMB_MAX_SEQS];
	for (int i = 0; i < n; i++) {
		if (tokens[i] < 0 || tokens[i] >= c.vocab_size) return set_error(XALM_ERR_INVALID, "token %d out of range [0,%d)", tokens[i], c.vocab_size);
		if (i == 0 ? parents[0] != -1 : parents[i] < 0 || parents[i] >= i)
			return set_error(XALM_ERR_INVALID, "forward_tree: parents[%d] = %d (the root's is -1, node i's lies in [0, i))", i, parents[i]);
		depth[i] = i == 0 ? 0 : depth[parents[i]] + 1;
	}
	return run_batched_rows(m, n, XALM_OUTPUT_LOGITS, [&](StepParams* sp) {
		for (int i = 0; i < n; i++) {
			fill_step_entry(c, sp[i], tokens[i], pos + depth[i], XALM_OUTPUT_LOGITS); // kv_len = pos + depth + 1: the branch's length
			sp[i].kv_pos = pos + i;
			sp[i].kv_fresh = pos;
			sp[i].ar_base = 0;
			sp[i].slot = slot;
			for (int v = i; v >= 0; v = parents[v])
				sp[i].tree = (sp[i].tree & ~(7u << 3 * depth[v])) | (uint32_t) v << 3 * depth[v];
		}
	});
}

int xalm_cuda_forward_tree(xalm_cuda_model* m, int slot, int n, const int* tokens, const int* parents, int pos, float* logits_host) {
	XALM_TRY(forward_tree_async(m, slot, n, tokens, parents, pos));
	return finish_step(m, n, XALM_OUTPUT_LOGITS, logits_host);
}

int xalm_cuda_forward_tree_argmax(xalm_cuda_model* m, int slot, int n, const int* tokens, const int* parents, int pos, int* next_tokens) {
	if (!next_tokens) return set_error(XALM_ERR_INVALID, "next_tokens is NULL");
	XALM_TRY(forward_tree_async(m, slot, n, tokens, parents, pos));
	return finish_step_argmax(m, n, next_tokens);
}

int xalm_cuda_tree_accept(xalm_cuda_model* m, int slot, int pos, int n, const int* nodes) {
	XALM_TRY(check_batched(m, "tree_accept", n));
	if (!nodes) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (slot < 0 || slot >= m->max_seqs) return set_error(XALM_ERR_INVALID, "tree_accept: slot %d not in [0, %d)", slot, m->max_seqs);
	if (pos < 0) return set_error(XALM_ERR_INVALID, "negative position");
	if (nodes[0] != 0) return set_error(XALM_ERR_INVALID, "tree_accept: nodes[0] = %d, a path starts at the root (0)", nodes[0]);
	for (int j = 1; j < n; j++)
		if (nodes[j] <= nodes[j - 1] || nodes[j] >= m->max_seqs)
			return set_error(XALM_ERR_INVALID, "tree_accept: nodes[%d] = %d after %d (a path's nodes increase and stay below %d)", j, nodes[j],
			                 nodes[j - 1], m->max_seqs);
	if (pos > m->c.max_seq_len - 1 - nodes[n - 1])
		return set_error(XALM_ERR_INVALID, "tree_accept: row %d reaches max_seq_len %d, trees stay below the window", pos + nodes[n - 1],
		                 m->c.max_seq_len);
	TreeMoves mv = {};
	for (int j = 0; j < n; j++)
		if (nodes[j] != j) { mv.src[mv.n] = pos + nodes[j]; mv.dst[mv.n] = pos + j; mv.n++; }
	if (!mv.n) return XALM_OK;
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	XALM_CUDA_CHECK(launch(tree_accept_kernel, dim3(2 * m->c.n_layers), dim3(128), m->stream, false, (__half* const*) m->kv_table,
	                       (size_t) slot * m->kv_slot, m->kv_dim_l, mv));
	return XALM_OK;
}

int xalm_cuda_forward_batch_async(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, int mode) {
	return forward_step_async(m, n, seqs, tokens, pos, mode, false);
}

int xalm_cuda_forward_batch(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, int mode, float* logits_host) {
	XALM_TRY(forward_step_async(m, n, seqs, tokens, pos, mode, false));
	return finish_step(m, n, mode, logits_host);
}

int xalm_cuda_forward_batch_argmax(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, int* next_tokens) {
	if (!next_tokens) return set_error(XALM_ERR_INVALID, "next_tokens is NULL");
	XALM_TRY(forward_step_async(m, n, seqs, tokens, pos, XALM_OUTPUT_LOGITS, false));
	return finish_step_argmax(m, n, next_tokens);
}

int xalm_cuda_forward_spans(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, float* logits_host) {
	XALM_TRY(forward_step_async(m, n, seqs, tokens, pos, XALM_OUTPUT_LOGITS, true));
	return finish_step(m, n, XALM_OUTPUT_LOGITS, logits_host);
}

int xalm_cuda_forward_spans_argmax(xalm_cuda_model* m, int n, const int* seqs, const int* tokens, const int* pos, int* next_tokens) {
	if (!next_tokens) return set_error(XALM_ERR_INVALID, "next_tokens is NULL");
	XALM_TRY(forward_step_async(m, n, seqs, tokens, pos, XALM_OUTPUT_LOGITS, true));
	return finish_step_argmax(m, n, next_tokens);
}

float* xalm_cuda_logits_host(xalm_cuda_model* m) { return m ? m->h_logits : nullptr; }

int xalm_cuda_last_launch_count(xalm_cuda_model* m, int* n) {
	if (!m || !n) return set_error(XALM_ERR_INVALID, "NULL argument");
	*n = m->last_launches;
	return XALM_OK;
}

int xalm_cuda_active_bytes(xalm_cuda_model* m, long long pos, long long* bytes) {
	if (!m || !bytes) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "active_bytes before finalize");
	const xalm_config& c = m->c;
	auto wb = [](int type, long long elems) -> long long {
		TypeInfo ti;
		type_info(type, &ti);
		return elems / ti.block * ti.bytes;
	};
	long long b = 0;
	b += wb(m->embed_type, c.dim);
	b += wb(m->rms_final_type, c.dim);
	b += wb(m->wcls.m.type, (long long) m->vocab_l * c.dim);
	for (auto& L : m->layers) {
		b += wb(L.rms_att_type, c.dim) + wb(L.rms_ffn_type, c.dim);
		b += wb(L.wqkv.m.type, (long long) (m->q_dim_l + 2 * m->kv_dim_l) * c.dim);
		b += wb(L.wo.m.type, (long long) c.dim * m->q_dim_l);
		b += wb(L.w13.m.type, 2LL * m->hidden_l * c.dim);
		b += wb(L.w2.m.type, (long long) c.dim * m->hidden_l);
		const long long kv_len = pos + 1 < c.max_seq_len ? pos + 1 : c.max_seq_len;
		b += 2 * kv_len * m->kv_dim_l * 2;
	}
	*bytes = b;
	return XALM_OK;
}

int xalm_cuda_read_state(xalm_cuda_model* m, int which, float* dst, size_t n) {
	if (!m || !dst) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "read_state before finalize");
	const float* src = nullptr;
	size_t cap = 0;
	switch (which) {
		case XALM_S_X: src = m->x; cap = m->c.dim; break;
		case XALM_S_XB2: src = m->xb2; cap = m->q_dim_l; break;
		case XALM_S_HB: src = m->hb; cap = m->hidden_l; break;
		case XALM_S_Q: src = m->q; cap = m->q_dim_l; break;
		case XALM_S_LOGITS: src = m->logits_full; cap = m->c.vocab_size; break;
		default: return set_error(XALM_ERR_INVALID, "state buffer %d is not materialised by the fused kernels", which);
	}
	if (n > cap) return set_error(XALM_ERR_INVALID, "read_state: %zu > %zu", n, cap);
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	XALM_CUDA_CHECK(cudaMemcpy(dst, src, n * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_read_kv(xalm_cuda_model* m, int layer, int which, uint16_t* dst, size_t n_elems) {
	if (!m || !dst) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "read_kv before finalize");
	if (layer < 0 || layer >= m->c.n_layers || (which != 0 && which != 1)) return set_error(XALM_ERR_INVALID, "bad layer/which");
	const size_t cap = (size_t) m->c.max_seq_len * m->kv_dim_l;
	if (n_elems > cap) return set_error(XALM_ERR_INVALID, "read_kv: %zu > %zu", n_elems, cap);
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	XALM_CUDA_CHECK(cudaStreamSynchronize(m->stream));
	const __half* src = (which == 0 ? m->layers[layer].k_cache : m->layers[layer].v_cache) + (size_t) m->cur_seq * m->kv_slot;
	XALM_CUDA_CHECK(cudaMemcpy(dst, src, n_elems * sizeof(uint16_t), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// op-level entry points (host in / host out) — the same kernels the model path launches
// ---------------------------------------------------------------------------------------------------------
struct TmpDev {
	std::vector<void*> v;
	~TmpDev() { for (void* p : v) cudaFree(p); }
	int alloc(void** p, size_t n) {
		cudaError_t e = cudaMalloc(p, n ? n : 16);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "cudaMalloc(%zu) failed: %s", n, cudaGetErrorString(e));
		v.push_back(*p);
		return XALM_OK;
	}
	int put(void** p, const void* h, size_t n) {
		XALM_TRY(alloc(p, n));
		XALM_CUDA_CHECK(cudaMemcpy(*p, h, n, cudaMemcpyHostToDevice));
		return XALM_OK;
	}
};

static int need_device() {
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0) return set_error(XALM_ERR_CUDA, "no CUDA device: %s", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
	return XALM_OK;
}

int xalm_cuda_dequant(int type_id, const void* src, size_t n_elems, float* dst) {
	if (!src || !dst) return set_error(XALM_ERR_INVALID, "NULL argument");
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	if (n_elems % ti.block) return set_error(XALM_ERR_INVALID, "%zu elements is not a multiple of the block size %d", n_elems, ti.block);
	XALM_TRY(need_device());
	if (n_elems == 0) return XALM_OK;
	TmpDev t;
	void *d_src, *d_dst;
	XALM_TRY(t.put(&d_src, src, n_elems / ti.block * ti.bytes));
	XALM_TRY(t.alloc(&d_dst, n_elems * sizeof(float)));
	dequant_kernel<<<1024, 256>>>(type_id, (const uint8_t*) d_src, n_elems, (float*) d_dst);
	XALM_CUDA_CHECK(cudaGetLastError());
	XALM_CUDA_CHECK(cudaMemcpy(dst, d_dst, n_elems * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

// device-resident weight from host bytes via the same repack path the model upload uses
static int tmp_weight(TmpDev& t, WMat& w, int type_id, const void* host, int rows, int n) {
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	if (type_id == XALM_U8) return set_error(XALM_ERR_UNSUPPORTED, "matmul: unsupported data type: U8");
	if (n % ti.block) return set_error(XALM_ERR_INVALID, "row length %d is not a multiple of the block size %d", n, ti.block);
	DevAlloc da;
	int rc = alloc_wmat(da, w, type_id, rows, n);
	for (void* p : da.ptrs) t.v.push_back(p);
	XALM_TRY(rc);
	Staging st;
	rc = upload_piece(w, 0, type_id, (const uint8_t*) host, n, 0, rows, 0, n, st, 0);
	if (st.p) t.v.push_back(st.p);
	if (st.flag) t.v.push_back(st.flag);
	return rc;
}

int xalm_cuda_matmul(float* xout, const float* x, const void* w, int type_id, int n, int d) {
	if (!xout || !x || !w) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (n <= 0 || d <= 0 || n % 32 || d % 32) return set_error(XALM_ERR_INVALID, "matmul: n=%d d=%d must be positive multiples of 32", n, d);
	XALM_TRY(need_device());
	TmpDev t;
	WMat wm;
	XALM_TRY(tmp_weight(t, wm, type_id, w, d, n));
	void *dx, *dy;
	XALM_TRY(t.put(&dx, x, (size_t) n * sizeof(float)));
	XALM_TRY(t.alloc(&dy, (size_t) d * sizeof(float)));
	MatvecArgs a = {};
	a.w = wm; a.x = (const float*) dx; a.n = n; a.d = d; a.epi = EPI_STORE; a.out = (float*) dy;
	XALM_TRY(launch_matvec(a, 0, false));
	XALM_CUDA_CHECK(cudaMemcpy(xout, dy, (size_t) d * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_mha(float* xout, float* att, const uint16_t* kb, const uint16_t* vb, const float* q, int head_dim, int kv_len,
                  int max_seq_len, int n_heads, int n_kv_heads) {
	if (!xout || !kb || !vb || !q) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (head_dim <= 0 || n_heads <= 0 || n_kv_heads <= 0 || n_heads % n_kv_heads || kv_len <= 0 || kv_len > max_seq_len)
		return set_error(XALM_ERR_INVALID, "mha: bad dimensions");
	XALM_TRY(need_device());
	TmpDev t;
	const size_t kv_bytes = (size_t) max_seq_len * n_kv_heads * head_dim * sizeof(uint16_t);
	void *dk, *dv, *dq, *dout, *dacc, *dml, *dtick, *datt = nullptr;
	XALM_TRY(t.put(&dk, kb, kv_bytes));
	XALM_TRY(t.put(&dv, vb, kv_bytes));
	XALM_TRY(t.put(&dq, q, (size_t) n_heads * head_dim * sizeof(float)));
	XALM_TRY(t.alloc(&dout, (size_t) n_heads * head_dim * sizeof(float)));
	const int G = n_heads / n_kv_heads;
	const int splits = attn_auto_splits(n_kv_heads);
	XALM_TRY(t.alloc(&dacc, (size_t) n_kv_heads * splits * G * head_dim * sizeof(float)));
	XALM_TRY(t.alloc(&dml, (size_t) n_kv_heads * splits * G * 2 * sizeof(float)));
	XALM_TRY(t.alloc(&dtick, n_kv_heads * sizeof(unsigned int)));
	XALM_CUDA_CHECK(cudaMemset(dtick, 0, n_kv_heads * sizeof(unsigned int)));
	AttnArgs a = {};
	a.q = (const float*) dq; a.k_cache = (const __half*) dk; a.v_cache = (const __half*) dv; a.out = (float*) dout;
	a.kv_len_fixed = kv_len; a.n_kv_heads = n_kv_heads; a.n_splits = splits; a.min_split = tune("attn_min_split");
	a.part_acc = (float*) dacc; a.part_ml = (float*) dml; a.tickets = (unsigned int*) dtick;
	XALM_TRY(launch_attn(a, head_dim, G, 0, false));
	if (att) {
		XALM_TRY(t.alloc(&datt, (size_t) n_heads * max_seq_len * sizeof(float)));
		XALM_CUDA_CHECK(cudaMemset(datt, 0, (size_t) n_heads * max_seq_len * sizeof(float)));
		attn_probs_kernel<<<n_heads, 256>>>((const float*) dq, (const __half*) dk, (float*) datt, head_dim, n_kv_heads, n_heads, kv_len, max_seq_len);
		XALM_CUDA_CHECK(cudaGetLastError());
		XALM_CUDA_CHECK(cudaMemcpy(att, datt, (size_t) n_heads * max_seq_len * sizeof(float), cudaMemcpyDeviceToHost));
	}
	XALM_CUDA_CHECK(cudaMemcpy(xout, dout, (size_t) n_heads * head_dim * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_rmsnorm(float* o, const float* x, const void* weight, int weight_type, int size, float eps) {
	if (!o || !x || !weight || size <= 0) return set_error(XALM_ERR_INVALID, "bad argument");
	if (weight_type != XALM_F32 && weight_type != XALM_BF16) return set_error(XALM_ERR_UNSUPPORTED, "rmsnorm: unsupported data type %d", weight_type);
	XALM_TRY(need_device());
	TmpDev t;
	void *dx, *dw, *dout;
	XALM_TRY(t.put(&dx, x, (size_t) size * sizeof(float)));
	XALM_TRY(t.put(&dw, weight, (size_t) size * (weight_type == XALM_F32 ? 4 : 2)));
	XALM_TRY(t.alloc(&dout, (size_t) size * sizeof(float)));
	rmsnorm_kernel<<<1, 256>>>((float*) dout, (const float*) dx, (const uint8_t*) dw, weight_type, size, eps);
	XALM_CUDA_CHECK(cudaGetLastError());
	XALM_CUDA_CHECK(cudaMemcpy(o, dout, (size_t) size * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_rope(float* vec, int d, int head_dim, int pos, float theta, int rotary_dim) {
	if (!vec || d <= 0 || d % 2 || head_dim <= 0 || head_dim % 2 || d % head_dim || rotary_dim < 0)
		return set_error(XALM_ERR_INVALID, "rope: bad argument");
	XALM_TRY(need_device());
	TmpDev t;
	const std::vector<float> freq = rope_freq_table(head_dim, rotary_dim, theta);
	void *dv, *df;
	XALM_TRY(t.put(&dv, vec, (size_t) d * sizeof(float)));
	XALM_TRY(t.put(&df, freq.data(), freq.size() * sizeof(float)));
	rope_kernel<<<(d / 2 + 255) / 256, 256>>>((float*) dv, d, head_dim, pos, (const float*) df);
	XALM_CUDA_CHECK(cudaGetLastError());
	XALM_CUDA_CHECK(cudaMemcpy(vec, dv, (size_t) d * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_ffn(float* xout, const float* x, const void* w1, const void* w2, const void* w3, int type_id, int hidden_dim, int dim,
                  int act) {
	if (!xout || !x || !w1 || !w2 || !w3) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (dim <= 0 || hidden_dim <= 0 || dim % 32 || hidden_dim % 32) return set_error(XALM_ERR_INVALID, "ffn: dims must be positive multiples of 32");
	if (act != XALM_GELU && act != XALM_SILU) return set_error(XALM_ERR_UNSUPPORTED, "unsupported activation type");
	XALM_TRY(need_device());
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	TmpDev t;
	// W1|W3 stacked along rows, exactly as the model path fuses gate|up
	DevAlloc da;
	WMat w13;
	int rc = alloc_wmat(da, w13, type_id, 2 * hidden_dim, dim, hidden_dim);
	for (void* p : da.ptrs) t.v.push_back(p);
	XALM_TRY(rc);
	Staging st;
	rc = upload_piece(w13, 0, type_id, (const uint8_t*) w1, dim, 0, hidden_dim, 0, dim, st, 0);
	if (rc == XALM_OK) rc = upload_piece(w13, hidden_dim, type_id, (const uint8_t*) w3, dim, 0, hidden_dim, 0, dim, st, 0);
	if (st.p) t.v.push_back(st.p);
	if (st.flag) t.v.push_back(st.flag);
	XALM_TRY(rc);
	WMat wd;
	XALM_TRY(tmp_weight(t, wd, type_id, w2, dim, hidden_dim));
	void *dx, *dhb, *dout;
	XALM_TRY(t.put(&dx, x, (size_t) dim * sizeof(float)));
	XALM_TRY(t.alloc(&dhb, (size_t) hidden_dim * sizeof(float)));
	XALM_TRY(t.alloc(&dout, (size_t) dim * sizeof(float)));
	MatvecArgs a = {};
	a.w = w13; a.x = (const float*) dx; a.n = dim; a.d = hidden_dim; a.epi = EPI_GLU; a.glu_off = hidden_dim; a.act = act; a.out = (float*) dhb;
	XALM_TRY(launch_matvec(a, 0, false));
	MatvecArgs b = {};
	b.w = wd; b.x = (const float*) dhb; b.n = hidden_dim; b.d = dim; b.epi = EPI_STORE; b.out = (float*) dout;
	XALM_TRY(launch_matvec(b, 0, false));
	XALM_CUDA_CHECK(cudaMemcpy(xout, dout, (size_t) dim * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

static void fill_prefill_model(xalm_cuda_model* m, PrefillModel& pm) {
	pm.c = m->c;
	pm.q_dim = m->q_dim_l; pm.kv_dim = m->kv_dim_l; pm.n_heads = m->n_heads_l; pm.n_kv_heads = m->n_kv_heads_l;
	pm.hidden = m->hidden_l; pm.vocab = m->vocab_l;
	pm.tp_rank = m->tp_rank; pm.tp_size = m->tp_size; pm.comm = m->comm; pm.status_dev = m->prefill_status;
	pm.embed_raw = m->embed_raw; pm.embed_type = m->embed_type; pm.embed_row_bytes = m->embed_row_bytes;
	pm.wcls = m->wcls.m; pm.rms_final = m->rms_final; pm.rms_final_type = m->rms_final_type;
	pm.rope_freq = m->rope_freq;
	pm.stream = m->stream;
	pm.layers.resize(m->layers.size());
	for (size_t l = 0; l < m->layers.size(); l++) {
		LayerDev& L = m->layers[l];
		PrefillLayer& P = pm.layers[l];
		P.wqkv = L.wqkv.m; P.wo = L.wo.m; P.w13 = L.w13.m; P.w2 = L.w2.m; P.glu_off = m->hidden_l;
		P.rms_att = L.rms_att; P.rms_ffn = L.rms_ffn; P.rms_att_type = L.rms_att_type; P.rms_ffn_type = L.rms_ffn_type;
		P.k_cache = L.k_cache + (size_t) m->cur_seq * m->kv_slot; P.v_cache = L.v_cache + (size_t) m->cur_seq * m->kv_slot;
	}
}

// ---- batched prefill / perplexity on the tensor-core path (prefill.cu); a collective under tensor parallelism --------------
// fn names the entry point in error messages; window: past the context window (prefill_run's ring regime); sync: wait for the
// stream (the synchronous calls also check want_logits up front, the async one leaves that to prefill_run)
static int prefill_call(const char* fn, xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits, float* logits_host,
                        const int* targets, float* probs_host, bool window, bool sync) {
	if (!m || !tokens) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (!m->finalized) return set_error(XALM_ERR_STATE, "prefill before finalize");
	if (sync && (want_logits < 0 || want_logits > 2)) return set_error(XALM_ERR_INVALID, "%s: want_logits = %d", fn, want_logits);
	XALM_CUDA_CHECK(cudaSetDevice(m->device));
	PrefillModel pm;
	fill_prefill_model(m, pm);
	XALM_TRY(prefill_run(pm, &m->prefill, tokens, n, pos0, want_logits, logits_host, targets, probs_host, tune("prefill_split"),
	                     &m->last_prefill_launches, window));
	if (sync) {
		cudaError_t e = cudaStreamSynchronize(m->stream);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "%s failed: %s", fn, cudaGetErrorString(e));
	}
	m->last_launches = m->last_prefill_launches;
	return XALM_OK;
}

int xalm_cuda_prefill(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits, float* logits_host, const int* targets,
                      float* probs_host) {
	return prefill_call("prefill", m, tokens, n, pos0, want_logits, logits_host, targets, probs_host, false, true);
}

int xalm_cuda_prefill_window(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits, float* logits_host, const int* targets,
                             float* probs_host) {
	return prefill_call("prefill_window", m, tokens, n, pos0, want_logits, logits_host, targets, probs_host, true, true);
}

// same as xalm_cuda_prefill without the host synchronisation and read-back (bench.py's device-timed leg)
int xalm_cuda_prefill_async(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits) {
	return prefill_call("prefill", m, tokens, n, pos0, want_logits, nullptr, nullptr, nullptr, false, false);
}

// out(T,N) = a(T,K) . W(N,K)^T — the batched form of matmul (model.h:315) on the tcgen05 path, host pointers in and out
int xalm_cuda_gemm(float* out, const float* a, const void* w, int type_id, int T, int K, int N, int split) {
	if (!out || !a || !w) return set_error(XALM_ERR_INVALID, "NULL argument");
	if (T <= 0 || K <= 0 || N <= 0 || K % 32 || N % 32) return set_error(XALM_ERR_INVALID, "gemm: T=%d K=%d N=%d (K, N positive multiples of 32)", T, K, N);
	XALM_TRY(need_device());
	TmpDev t;
	WMat wm;
	XALM_TRY(tmp_weight(t, wm, type_id, w, N, K));
	void *da, *dout;
	XALM_TRY(t.put(&da, a, (size_t) T * K * sizeof(float)));
	XALM_TRY(t.alloc(&dout, (size_t) T * N * sizeof(float)));
	XALM_TRY(prefill_gemm_dev(wm, (const float*) da, T, (float*) dout, split, 0));
	XALM_CUDA_CHECK(cudaMemcpy(out, dout, (size_t) T * N * sizeof(float), cudaMemcpyDeviceToHost));
	return XALM_OK;
}

int xalm_cuda_bench_gemm(int T, int N, int K, int split, int iters, float* ms_per_launch) {
	if (!ms_per_launch || T <= 0 || N <= 0 || K <= 0 || iters <= 0) return set_error(XALM_ERR_INVALID, "bench_gemm: bad argument");
	XALM_TRY(need_device());
	return prefill_bench_gemm(T, N, K, split, iters, ms_per_launch);
}

int xalm_cuda_timeline(int n_records, unsigned long long* out, int* n_out) {
	// n_records > 0 and out == NULL: start recording (up to n_records kernels); out != NULL: stop, copy records (4 x u64 each)
	XALM_TRY(need_device());
	static unsigned long long* dbuf = nullptr;
	static int cap = 0;
	XALM_CUDA_CHECK(cudaDeviceSynchronize());
	if (!out) {
		if (dbuf) cudaFree(dbuf);
		dbuf = nullptr;
		cap = n_records;
		Timeline t = {nullptr, 0, 0};
		if (n_records > 0) {
			XALM_CUDA_CHECK(cudaMalloc((void**) &dbuf, (size_t) n_records * 4 * sizeof(unsigned long long)));
			XALM_CUDA_CHECK(cudaMemset(dbuf, 0, (size_t) n_records * 4 * sizeof(unsigned long long)));
			t.buf = dbuf; t.cap = (unsigned) n_records;
		}
		XALM_CUDA_CHECK(cudaMemcpyToSymbol(d_timeline, &t, sizeof t));
		return XALM_OK;
	}
	Timeline t;
	XALM_CUDA_CHECK(cudaMemcpyFromSymbol(&t, d_timeline, sizeof t));
	int n = (int) (t.count < (unsigned) cap ? t.count : (unsigned) cap);
	if (n > n_records) n = n_records;
	if (n > 0) XALM_CUDA_CHECK(cudaMemcpy(out, dbuf, (size_t) n * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
	if (n_out) *n_out = n;
	Timeline z = {nullptr, 0, 0};
	XALM_CUDA_CHECK(cudaMemcpyToSymbol(d_timeline, &z, sizeof z));
	if (dbuf) { cudaFree(dbuf); dbuf = nullptr; }
	return XALM_OK;
}

// Times one matvec over n_buffers rotating copies of a random weight matrix.  n_seqs = 0: the kernel the single-sequence path
// picks for the matrix; 1..8: the batched tensor-core matvec (activation quantiser + matvec) at that many sequences.
static int bench_matvec_run(int type_id, int n, int d, int epi, int with_norm, int n_seqs, int n_buffers, int iters, float* ms_per_launch) {
	if (!ms_per_launch || n <= 0 || d <= 0 || n % 32 || d % 32 || n_buffers <= 0 || iters <= 0) return set_error(XALM_ERR_INVALID, "bad argument");
	if (epi != EPI_STORE && epi != EPI_GLU && epi != EPI_RESIDUAL) return set_error(XALM_ERR_INVALID, "bench epi must be 0 (store), 1 (residual) or 2 (glu)");
	TypeInfo ti;
	if (!type_info(type_id, &ti)) return set_error(XALM_ERR_INVALID, "invalid type: %d", type_id);
	if (n % ti.block) return set_error(XALM_ERR_INVALID, "n %% block");
	const int rows = epi == EPI_GLU ? 2 * d : d;
	if (n_seqs && !mma_takes(type_id, rows, n, epi == EPI_GLU ? d : 0))
		return set_error(XALM_ERR_UNSUPPORTED, "the batched matvec cannot take type %d, %d x %d", type_id, rows, n);
	XALM_TRY(need_device());
	const int nx = n_seqs ? n_seqs : 1; // activation rows
	DevAlloc da;
	Staging sg;
	cudaEvent_t e0 = nullptr, e1 = nullptr;
	cudaStream_t s = nullptr;
	auto run = [&]() -> int {
		std::vector<WMat> ws(n_buffers);
		const size_t raw_bytes = (size_t) rows * n / ti.block * ti.bytes;
		// random but decodable bytes: scales must be finite f16 -> build on host once
		std::vector<uint8_t> host(raw_bytes);
		uint32_t st = 12345;
		for (size_t i = 0; i < raw_bytes; i++) { st = st * 1664525u + 1013904223u; host[i] = (uint8_t) ((st >> 24) & 0x3F); }
		for (WMat& w : ws) {
			XALM_TRY(alloc_wmat(da, w, type_id, rows, n, epi == EPI_GLU ? d : 0, false, n_seqs > 0));
			XALM_TRY(upload_piece(w, 0, type_id, host.data(), n, 0, rows, 0, n, sg, 0));
		}
		float *dx = nullptr, *dy = nullptr, *dg = nullptr, *dsc = nullptr;
		uint8_t* img = nullptr;
		if (with_norm) {
			const std::vector<float> hg(n, 1.0f);
			XALM_TRY(da.alloc((void**) &dg, (size_t) n * sizeof(float)));
			XALM_CUDA_CHECK(cudaMemcpy(dg, hg.data(), (size_t) n * sizeof(float), cudaMemcpyHostToDevice));
		}
		const std::vector<float> hx((size_t) nx * n, 0.01f);
		XALM_TRY(da.alloc((void**) &dx, hx.size() * sizeof(float)));
		XALM_CUDA_CHECK(cudaMemcpy(dx, hx.data(), hx.size() * sizeof(float), cudaMemcpyHostToDevice));
		XALM_TRY(da.alloc((void**) &dy, (size_t) nx * d * sizeof(float)));
		XALM_CUDA_CHECK(cudaMemset(dy, 0, (size_t) nx * d * sizeof(float)));
		if (n_seqs) {
			XALM_TRY(da.alloc((void**) &dsc, (size_t) n_seqs * sizeof(float)));
			XALM_TRY(da.alloc((void**) &img, (size_t) n / 32 * ((n_seqs + 1) / 2) * MMB_PAIR));
		}
		XALM_CUDA_CHECK(cudaEventCreate(&e0));
		XALM_CUDA_CHECK(cudaEventCreate(&e1));
		XALM_CUDA_CHECK(cudaStreamCreate(&s));
		const bool pdl = tune("pdl") != 0;
		const BatchIo io = {n_seqs, n, d, img, dsc, 0};
		for (int it = -3 * n_buffers; it < iters; it++) {
			if (it == 0) XALM_CUDA_CHECK(cudaEventRecord(e0, s));
			MatvecArgs a = {};
			a.w = ws[((it % n_buffers) + n_buffers) % n_buffers]; a.x = dx; a.n = n; a.d = d; a.epi = epi; a.out = dy;
			a.glu_off = d; a.act = XALM_SILU;
			if (with_norm) { a.norm_w = (const uint8_t*) dg; a.norm_type = XALM_F32; a.norm_eps = 1e-5f; }
			XALM_TRY(n_seqs ? launch_matvec_batch(a, io, s, pdl) : launch_matvec(a, s, pdl));
		}
		XALM_CUDA_CHECK(cudaEventRecord(e1, s));
		cudaError_t e = cudaStreamSynchronize(s);
		if (e != cudaSuccess) return set_error(XALM_ERR_CUDA, "bench failed: %s", cudaGetErrorString(e));
		float ms = 0.f;
		XALM_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
		*ms_per_launch = ms / iters;
		return XALM_OK;
	};
	const int rc = run();
	if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } // a failed launch may leave earlier ones in flight on the buffers freed below
	if (e0) cudaEventDestroy(e0);
	if (e1) cudaEventDestroy(e1);
	if (sg.p) cudaFree(sg.p);
	if (sg.flag) cudaFree(sg.flag);
	da.free_all();
	return rc;
}

int xalm_cuda_bench_matvec(int type_id, int n, int d, int epi, int with_norm, int n_buffers, int iters, float* ms_per_launch) {
	return bench_matvec_run(type_id, n, d, epi, with_norm, 0, n_buffers, iters, ms_per_launch);
}

int xalm_cuda_bench_matvec_batch(int type_id, int n, int d, int epi, int with_norm, int n_seqs, int n_buffers, int iters, float* ms_per_launch) {
	if (n_seqs < 1 || n_seqs > MMB_MAX_SEQS) return set_error(XALM_ERR_INVALID, "bad argument");
	return bench_matvec_run(type_id, n, d, epi, with_norm, n_seqs, n_buffers, iters, ms_per_launch);
}

} // extern "C"
