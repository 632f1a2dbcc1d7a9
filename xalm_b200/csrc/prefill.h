// prefill.h — seam between xalm_cuda.cu (model handle, uploads, decode path) and prefill.cu (the batched
// prefill / perplexity path on tcgen05 tensor cores).  Plain structs, no templates: the two translation units
// compile independently.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <nccl.h>

#include <vector>

#include "formats.cuh"

namespace xalm {

struct PrefillLayer {
	WMat wqkv, wo, w13, w2;       // device layouts of the decode path (matvec.cuh / matvec_tma.cuh); w13 = W1 rows then W3 rows
	int glu_off = 0;              // first W3 row inside w13
	const uint8_t* rms_att = nullptr;
	const uint8_t* rms_ffn = nullptr;
	int rms_att_type = 0, rms_ffn_type = 0;
	__half* k_cache = nullptr;    // (max_seq_len, kv_dim)
	__half* v_cache = nullptr;
};

struct PrefillModel {
	xalm_config c;
	// this rank's shard of the sharded dimensions (one GPU: the full sizes; tensor parallel: SURVEY.md 8e)
	int q_dim = 0, kv_dim = 0, n_heads = 0, n_kv_heads = 0, hidden = 0, vocab = 0;
	// tensor parallel (tp_size > 1): the pass is a collective over `comm`; status_dev: one device int for the status vote
	int tp_rank = 0, tp_size = 1;
	ncclComm_t comm = nullptr;
	int* status_dev = nullptr;
	const uint8_t* embed_raw = nullptr; // on-disk rows
	int embed_type = 0;
	size_t embed_row_bytes = 0;
	WMat wcls;
	const uint8_t* rms_final = nullptr;
	int rms_final_type = 0;
	const float* rope_freq = nullptr;   // (head_dim/2,) device
	std::vector<PrefillLayer> layers;
	cudaStream_t stream = nullptr;
};

struct PrefillScratch; // device scratch + pinned staging, grown on demand; owned by the model handle

// Positions pos0 .. pos0+n-1 in one pass.  want_logits: 0 = hydrate the KV cache only (final norm + classifier skipped,
// like InferenceMode::HYDRATE_KV_CACHE), 1 = logits of the last position only, 2 = logits of every position.
// logits_host: NULL, or vocab floats (want 1) / n*vocab floats (want 2).  targets/probs_host: NULL, or n entries —
// probs_host[i] = softmax(logits_i)[targets[i]] as Sampler::sample_prob computes it (needs want 2).
// split: 1 = activations as one fp16 operand, 2 = hi+lo fp16 pair (two MMAs per weight tile, ~fp32 activations).
// Tensor parallel (pm.tp_size > 1): every rank calls it with the same arguments; each fills its KV-cache shard and receives the
// full logits / probabilities.  A refusal is the same on every rank and leaves every cache untouched.
// window = false: the linear regime, pos0 + n <= max_seq_len.  window = true: the ring regime past the context window,
// pos0 >= max_seq_len and n <= max_seq_len - 2 (each ring slot written at most once); new rows go to their ring slots and the
// two sink keys are re-rotated n times, as n token-at-a-time forwards would leave the cache.
int prefill_run(const PrefillModel& pm, PrefillScratch** scratch, const int* tokens, int n, int pos0, int want_logits,
                float* logits_host, const int* targets, float* probs_host, int split, int* n_launches, bool window = false);
void prefill_free(PrefillScratch* s);
// device pointer of the logits of the last prefill (rows x vocab) — bench / tests
const float* prefill_logits_dev(const PrefillScratch* s, int* rows);

// Op-level hook: out(T,N) = a(T,K) . W(N,K)^T on the tensor-core path, all pointers on the device; W in its decode layout.
int prefill_gemm_dev(const WMat& w, const float* a_dev, int T, float* out_dev, int split, cudaStream_t s);
// Times `iters` launches of the GEMM kernel alone (operands resident, dequantised tiles prepared once).
int prefill_bench_gemm(int T, int N, int K, int split, int iters, float* ms_per_launch);

} // namespace xalm
