/* =============================================================================================
 * xalm_cuda.h — C ABI of the B200 (sm_100a) `-d cuda` backend for Xalm's transformer forward pass.
 *
 * The reference has no plugin/FFI interface; its only device seam is three C++ call sites
 * (SURVEY.md §8b).  Each entry point below names the reference interface it stands in for.
 * Paths are relative to the reference tree (jubruckne/Xalm).
 *
 *   - nothing but POD, raw pointers and sizes crosses this boundary; no exceptions: every call
 *     returns 0 on success or a non-zero xalm_status, and xalm_cuda_last_error() describes it;
 *   - the backend owns all device memory (weights, KV cache, scratch) behind the opaque handle;
 *   - there is NO CPU fallback: without a usable CUDA device every compute call fails.
 * ============================================================================================= */
#ifndef XALM_CUDA_H
#define XALM_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XALM_CUDA_ABI_VERSION 1

/* Tensor element types.  0..9: `Type` ids, src/types.h:505-514.  1007..1012: the gguf-style block
 * formats convert.py writes (XType values, convert.py:56-61; layouts quants.py:281-464,638-683) which
 * the reference runtime never learned to load (SURVEY.md §0.4).  2007: convert.py's qi8 (:538-551). */
enum xalm_type {
	XALM_UNKNOWN = 0,
	XALM_F32 = 1, XALM_F16 = 2, XALM_BF16 = 3,
	XALM_F8_E2M5 = 4, XALM_F8_E3M4 = 5, XALM_F8_E4M3 = 6, XALM_F8_E5M2 = 7,
	XALM_U8 = 8, XALM_Q8 = 9,
	XALM_Q4_0 = 1007, XALM_Q4_1 = 1008, XALM_Q5_0 = 1009, XALM_Q5_1 = 1010, XALM_Q8_0 = 1011, XALM_TQ1_0 = 1012,
	XALM_QI8 = 2007
};

/* InferenceMode, src/model.h:249-252 */
enum xalm_mode { XALM_HYDRATE_KV_CACHE = 0, XALM_OUTPUT_LOGITS = 1 };
/* ActivationType, src/model.h:12-15 */
enum xalm_act { XALM_GELU = 0, XALM_SILU = 1 };

enum xalm_status {
	XALM_OK = 0,
	XALM_ERR_INVALID = 1,      /* bad argument / shape / unknown tensor name (load-time std::invalid_argument in the reference) */
	XALM_ERR_UNSUPPORTED = 2,  /* dtype the op does not take (infer.cpp:211-214, :248-249) */
	XALM_ERR_CUDA = 3,         /* CUDA runtime / driver error, or no device */
	XALM_ERR_STATE = 4,        /* call out of order (forward before finalize, missing tensors, ...) */
	XALM_ERR_COMM = 5          /* NCCL error */
};

/* Config, src/model.h:25-42 (same fields, same order; enums as int). */
typedef struct xalm_config {
	int dim;
	int hidden_dim;
	int head_dim;
	int n_layers;
	int n_heads;
	int n_kv_heads;
	int vocab_size;
	int max_seq_len;      /* after the 4096 clamp / -T override of Config::from_xalm (model.h:54-59) */
	float rope_theta;
	int rotary_dim;
	float norm_eps;
	int act;              /* xalm_act */
	int norm_type;        /* 0 = RMSNorm (the only LayerNormType, model.h:17-19) */
	float qkv_clip;       /* FLT_MAX when the checkpoint has none (model.h:84-85) */
	int tie_word_embeddings;
} xalm_config;

typedef struct xalm_cuda_model xalm_cuda_model; /* opaque: Model + InferenceState + KV caches on one GPU */

/* ---- diagnostics ------------------------------------------------------------------------- */
int xalm_cuda_abi_version(void);
/* Message for the last failing call on this thread ("" if none). Stands in for the reference's exceptions. */
const char* xalm_cuda_last_error(void);
int xalm_cuda_device_count(int* count);
/* (block elements, block bytes) of a type — Type::bit_size (types.h:350) generalised to quants.py:45-77. */
int xalm_cuda_type_info(int type_id, int* block_elems, int* block_bytes);

/* ---- model lifecycle: Model::from_xalm (model.cpp:48-118) + the commented-out
 *      `model.cuda(); state.cuda();` (main.cpp:211-212, :283-284) ------------------------------ */
/* tp_rank/tp_size: tensor-parallel shard this handle holds (1 GPU: 0/1).  Sharding per SURVEY.md §8e. */
int xalm_cuda_create(const xalm_config* cfg, int device, int tp_rank, int tp_size, xalm_cuda_model** out);
/* One call per tensor of model.cpp:83-114 ("embed.weight", "l.{i}.attn.{norm,q,k,v,down}.weight",
 * "l.{i}.mlp.{norm,gate,down,up}.weight", "output.norm.weight", "output.weight").  `shape` is the ELEMENT
 * shape (rows, cols), `data` the full (unsharded) host tensor in its on-disk byte layout; the backend keeps
 * only this rank's shard.  The host buffer may be freed on return. */
int xalm_cuda_upload_tensor(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank,
                            const void* data, size_t nbytes);
/* Shard-aware upload for tensor-parallel handles, so that a rank reads / generates only what it keeps (the reference loader it
 * stands in for reads every tensor whole, model.cpp:48-118).  xalm_cuda_shard_range: range4 = {row0, row1, col0, col1} of the
 * ELEMENT shape this rank keeps of tensor `name` (norms and the embedding table: everything).  xalm_cuda_upload_tensor_shard:
 * `data` holds exactly that block, dense, in on-disk bytes (rows of (col1 - col0) elements); `shape` is still the full shape. */
int xalm_cuda_shard_range(xalm_cuda_model* m, const char* name, int* range4);
int xalm_cuda_upload_tensor_shard(xalm_cuda_model* m, const char* name, int type_id, const int* shape, int rank, const int* range4,
                                  const void* data, size_t nbytes);
/* Page-locked host memory for upload staging (H2D copies from it run at full PCIe rate and may be asynchronous). */
void* xalm_cuda_host_alloc(size_t nbytes);
void xalm_cuda_host_free(void* p);
/* Checks every tensor arrived, builds fused/concatenated device layouts, captures the per-token CUDA graphs. */
int xalm_cuda_finalize(xalm_cuda_model* m);
void xalm_cuda_destroy(xalm_cuda_model* m);

/* Tensor parallel plumbing (no reference analogue; north star).  Rank 0 makes an id, the host side ships it to
 * the other ranks (torch.distributed / MPI / a file), every rank calls comm_init before finalize. */
#define XALM_COMM_ID_BYTES 128
int xalm_cuda_comm_unique_id(void* id128);
int xalm_cuda_comm_init(xalm_cuda_model* m, const void* id128);

/* Optional: one-shot allreduce over NVLink peer memory instead of NCCL for the two per-layer exchanges.  Every rank exports
 * a CUDA IPC handle of its exchange buffer, the host gathers all of them (rank order) and hands the table to every rank.
 * Call after create and before finalize; without it the backend uses ncclAllReduce. */
#define XALM_IPC_HANDLE_BYTES 64
int xalm_cuda_ipc_export(xalm_cuda_model* m, void* handle64);
int xalm_cuda_ipc_import(xalm_cuda_model* m, const void* handles /* tp_size x 64 bytes */);

/* Run on a caller-provided cudaStream_t (e.g. the framework's current stream) instead of the model's own. */
int xalm_cuda_set_stream(xalm_cuda_model* m, void* cuda_stream);

/* ---- forward: Model::forward(state, token, pos, mode)  (model.h:272, infer.cpp:604-638) ---------------- */
/* Synchronous: on return with mode == XALM_OUTPUT_LOGITS, `logits_host` (vocab_size floats, caller-owned,
 * may be pageable) holds what InferenceState::logits() would.  logits_host may be NULL (leave them on device). */
int xalm_cuda_forward(xalm_cuda_model* m, int token, int pos, int mode, float* logits_host);
/* forward(OUTPUT_LOGITS) followed by Sampler::sample_argmax (sampler.cpp:3-16, FLT_MIN-seeded running maximum, first
 * maximum wins) on the device: only the 4-byte token id crosses PCIe.  Leaves the host logits buffer untouched. */
int xalm_cuda_forward_argmax(xalm_cuda_model* m, int token, int pos, int* next_token);
/* Enqueue only (no host sync, logits stay on the device): the device-timed leg of bench.py. */
int xalm_cuda_forward_async(xalm_cuda_model* m, int token, int pos, int mode);
int xalm_cuda_sync(xalm_cuda_model* m);
/* ---- batched prefill: the loops of main.cpp:94-100 (prompt hydrate) and :244-254 (perplexity), which call
 *      Model::forward once per position, as ONE pass over the weights on the tcgen05 tensor-core path ---------- */
/* Positions pos0 .. pos0+n-1 (pos0 + n <= max_seq_len: no ring wrap; past that use xalm_cuda_prefill_window).  Fills the KV
 * cache exactly as n forward calls would (fp16-operand rounding aside).  want_logits: 0 = none (HYDRATE_KV_CACHE for
 * every position), 1 = logits of the last position -> logits_host[vocab], 2 = every position -> logits_host[n*vocab].
 * targets/probs_host (n entries each, or NULL; needs want_logits 2): probs_host[i] = Sampler::sample_prob(targets[i])
 * on the logits of position pos0+i (sampler.cpp:18-33) — what perplexity mode takes the log of (main.cpp:251).
 * logits_host may be NULL.  Synchronous.  Tensor-core operands are fp16 with fp32 accumulation; the "prefill_split"
 * knob (xalm_cuda_tune) picks how fp32 values enter them: 3 (default) = hi+lo fp16 pairs for activations, weights and the
 * attention operands (3 MMAs per product; 32-layer 4k-token logits within ~1e-3 of the token-at-a-time path), 2 = pairs
 * for activations only, 1 = plain fp16 (fastest; ~4e-2 at that depth).  North star tolerance: 1e-2.
 * Tensor-parallel handles: a collective.  Every rank of the group calls it with the same arguments, in the same order; each
 * fills its own KV-cache shard (its kv heads) and receives the FULL logits and probabilities, as xalm_cuda_forward returns
 * full logits on every rank.  A refusal (bad argument, or a scratch allocation that failed on any one rank) is the same
 * error on every rank and leaves every rank's cache untouched. */
int xalm_cuda_prefill(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits, float* logits_host,
                      const int* targets, float* probs_host);
/* The same batched pass past the context window, where the KV cache is a ring: positions pos0 .. pos0+n-1 with
 * pos0 >= max_seq_len and 1 <= n <= max_seq_len - 2 (each ring slot is written at most once per call; longer runs go in
 * chunks).  Leaves the KV cache as n xalm_cuda_forward calls would: each new row in its ring slot 2 + (pos - 2) % (max_seq_len - 2),
 * and the two attention-sink keys in slots 0 and 1 re-rotated n more times (bit-identical to the token loop).  Each
 * position attends to the two sinks and the max_seq_len - 2 latest positions, itself included.  want_logits, logits_host,
 * targets, probs_host and the "prefill_split" knob mean what they mean for xalm_cuda_prefill.  Anything else — positions
 * below the window, n too large, a token out of range — is XALM_ERR_INVALID before anything runs (the cache is untouched).
 * Synchronous.  A collective on tensor-parallel handles, with the same per-rank results and refusals as xalm_cuda_prefill. */
int xalm_cuda_prefill_window(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits, float* logits_host,
                             const int* targets, float* probs_host);
/* Enqueue only (no read-back, no host sync) — bench.py's device-timed leg.  A collective on tensor-parallel handles; a
 * refusal there is agreed between the ranks, which takes one host synchronisation before the pass is enqueued. */
int xalm_cuda_prefill_async(xalm_cuda_model* m, const int* tokens, int n, int pos0, int want_logits);
/* Pinned host buffer the logits are copied into by xalm_cuda_forward (alias it as InferenceState::_logits). */
float* xalm_cuda_logits_host(xalm_cuda_model* m);
/* Model::active_bytes(pos) (model.cpp:12-35), 64-bit, per-format bytes; this rank's shard only. */
int xalm_cuda_active_bytes(xalm_cuda_model* m, long long pos, long long* bytes);
/* Kernels launched by the last forward (bench.py's gpu_launches). */
int xalm_cuda_last_launch_count(xalm_cuda_model* m, int* n);

/* ---- state read-back for parity tests (InferenceState accessors model.h:124-139, Block KV model.h:222-223) -- */
enum xalm_state_buf { XALM_S_X = 0, XALM_S_XB = 1, XALM_S_XB2 = 2, XALM_S_HB = 3, XALM_S_Q = 5, XALM_S_LOGITS = 9 };
int xalm_cuda_read_state(xalm_cuda_model* m, int which, float* dst, size_t n);
/* which: 0 = key_cache, 1 = value_cache; fp16 bits, (max_seq_len, local kv_dim) */
int xalm_cuda_read_kv(xalm_cuda_model* m, int layer, int which, uint16_t* dst, size_t n_elems);

/* ---- op-level entry points: the functions model.h:286-316 exposes "for tests", host pointers in and out ---- */
/* Type::get_float over a buffer (types.h:406-427) / quants.py dequantize: n_elems elements -> fp32. */
int xalm_cuda_dequant(int type_id, const void* src, size_t n_elems, float* dst);
/* matmul(xout, x, w, n, d) (model.h:315, infer.cpp:185-216): W(d,n) row-major in on-disk bytes of `type_id`. */
int xalm_cuda_matmul(float* xout, const float* x, const void* w, int type_id, int n, int d);
/* mha_cuda — the prototype the reference declares and never defines (model.h:308-313). att may be NULL. */
int xalm_cuda_mha(float* xout, float* att, const uint16_t* kb, const uint16_t* vb, const float* q, int head_dim,
                  int kv_len, int max_seq_len, int n_heads, int n_kv_heads);
/* The batched form of matmul: out(T,N) = a(T,K) . W(N,K)^T on the tcgen05 path (dequantise to fp16 tiles, UMMA, fp32
 * accumulate).  split: 1 = fp16 activations, 2 = hi+lo fp16 pair. */
int xalm_cuda_gemm(float* out, const float* a, const void* w, int type_id, int T, int K, int N, int split);
/* rmsnorm(o, x, weight, size, eps) (infer.cpp:224-251); weight F32 or BF16 only. */
int xalm_cuda_rmsnorm(float* o, const float* x, const void* weight, int weight_type, int size, float eps);
/* rope(vec, d, head_dim, pos, theta, rotary_dim) (infer.cpp:305-322), in place. */
int xalm_cuda_rope(float* vec, int d, int head_dim, int pos, float theta, int rotary_dim);
/* ffn: hb = act(W1 x) * (W3 x); xout = W2 hb   (ffn_cpu, infer.cpp:519-551) with weights of `type_id`. */
int xalm_cuda_ffn(float* xout, const float* x, const void* w1, const void* w2, const void* w3, int type_id,
                  int hidden_dim, int dim, int act);

/* Integer tuning knobs by name ("pdl", "graph", "attn_splits", "attn_min_split", "prefill_split", "idp", "mma",
 * "tail_prefetch_mb", ...); an XALM_<KEY> environment variable overrides the stored value.  Takes effect for graphs captured
 * afterwards; "mma" (which matvec kernel and device layout the integer formats take: 0 = dp4a + unit layout, 1 = tensor-core mma +
 * fragment tiles, 2 = default: mma for the 4/5-bit formats and, under tensor parallelism, the 8-bit ones) is read when a
 * matrix is uploaded. */
int xalm_cuda_tune(const char* key, int value);

/* In-kernel timeline (there is no nsys here): with out == NULL start recording up to n_records kernels; with out != NULL
 * stop and fetch the records — 4 x u64 each: kernel id (100+epi = TMA matvec, 200+epi = LDG matvec, 300 = attention),
 * %globaltimer (ns) of block 0 at entry, after the dependency wait, at exit. */
int xalm_cuda_timeline(int n_records, unsigned long long* out, int* n_out);

/* ---- kernel micro-benchmark hook (bench.py roofline leg; README.md:62-84 `-k matmul`) ------------------- */
/* Times `iters` back-to-back launches of the matvec kernel on resident weights of `type_id` (random bytes), rotating
 * over `n_buffers` distinct copies so the working set exceeds L2.  epi: 0 = plain store of d outputs from a (d,n) matrix,
 * 2 = the fused gate|up kernel (2d rows -> d outputs through act*gate); with_norm: fuse the rmsnorm prologue.  Returns
 * mean milliseconds per launch (CUDA events on the launch stream). */
int xalm_cuda_bench_matvec(int type_id, int n, int d, int epi, int with_norm, int n_buffers, int iters, float* ms_per_launch);

/* Times `iters` launches of the tcgen05 GEMM kernel alone on resident fp16 tiles (T x K activations, N x K weights);
 * mean milliseconds per launch.  2*T*N*K flops per launch. */
int xalm_cuda_bench_gemm(int T, int N, int K, int split, int iters, float* ms_per_launch);

#ifdef __cplusplus
}
#endif
#endif /* XALM_CUDA_H */
