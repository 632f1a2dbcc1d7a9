// model.h — C++ host side of the `-d cuda` backend: the reference's operator surface for the forward path
// (Type, Tensor, Xalm::load, Config, InferenceState, Model, Sampler, Tokenizer — same names, argument meaning and
// error behaviour as /root/reference/src/{types,tensor,xalm,model,sampler,tokenizer}.h) with the compute behind the
// C ABI of include/xalm_cuda.h.  Portable C++20 (g++ 13, x86-64): no NEON, no <print>.
//
// What changes relative to the reference, by design (SURVEY.md §8b):
//   * Device gains CUDA (model.h:21-23); Model::cuda() / InferenceState::cuda() exist (main.cpp:211-212 has them
//     commented out); Model::forward on a model that is not on the device throws — there is no CPU path here.
//   * Type::parse also accepts the block formats convert.py writes (q4_0 q4_1 q5_0 q5_1 q8_0 tq1_0, qi8) and the
//     loader maps their byte-shaped headers back to element shapes (SURVEY.md §0.4).
#pragma once
#include <cfloat>
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <string_view>
#include <vector>

#include "xalm_cuda.h"

constexpr int KV_SINKS = 2; // model.h:10

// ---- Type (types.h:337-514) ------------------------------------------------------------------------------
struct Type {
	int id = XALM_UNKNOWN;
	int block = 1;  // elements per block
	int bytes = 0;  // bytes per block

	static Type from_id(int id);
	static Type parse(std::string_view name); // case-insensitive; throws std::invalid_argument on an unknown name
	std::string_view name() const;
	size_t nbytes(size_t elems) const { return elems / (size_t) block * (size_t) bytes; }
	bool operator==(const Type& o) const { return id == o.id; }
	bool operator!=(const Type& o) const { return id != o.id; }
};

// ---- Tensor (tensor.h:241-298): name / type / element shape / 16-byte aligned host buffer ----------------------
class Tensor {
public:
	Tensor() = default;
	Tensor(Tensor&&) noexcept = default;
	Tensor& operator=(Tensor&&) noexcept = default;
	Tensor(const Tensor&) = delete;
	Tensor& operator=(const Tensor&) = delete;

	std::string name;
	Type type;
	std::vector<int> shape;   // ELEMENT shape
	size_t size = 0;          // bytes
	size_t linear_length = 0; // elements

	static Tensor zeroes(Type type, const std::vector<int>& shape, const std::string& name = "");
	// Tensor::convert_to (tensor.cpp:226-296), extended to the block formats the reference only defines in Python: an F32 / F16 /
	// BF16 tensor re-encoded as F32, F16, BF16, Q8 or Q8_0 / Q4_0 / Q4_1 / Q5_0 / Q5_1 / TQ1_0 with quants.py's quantiser rules
	// (byte-identical to quants.py, tests/test_quantize.py).  Throws std::invalid_argument for a pair it does not take.
	[[nodiscard]] Tensor convert_to(Type target_type) const;
	template <typename T>
	const T* get_data() const { return reinterpret_cast<const T*>(data_.get()); }
	uint8_t* bytes() { return data_.get(); }
	const uint8_t* bytes() const { return data_.get(); }

private:
	struct Free { void operator()(uint8_t* p) const { std::free(p); } };
	std::unique_ptr<uint8_t, Free> data_;
};

// ---- Xalm (xalm.h:11-193) ---------------------------------------------------------------------------------------
struct Xalm {
	struct tensor_info {
		std::string name;
		Type type;
		std::vector<int> shape;      // element shape
		std::vector<int> disk_shape; // as stored (byte shape for block formats)
		std::string file_name;
		size_t offset = 0; // absolute
		size_t size = 0;
		uint64_t hash = 0;
		bool has_hash = false;
	};
	struct file_info {
		std::string file_name;
		std::string arch;
		std::map<std::string, std::string> metadata; // the "config" object: every value is a string
		std::map<std::string, tensor_info> tensors;
		Tensor load_tensor(const std::string& name) const;
		// reads the payload (one descriptor per file, pread) and verifies its xxh3_64 against the header's "hash" when present
		void load_tensor_data(const tensor_info& ti, uint8_t* dst, size_t n) const;
		file_info() = default;
		file_info(file_info&& o) noexcept : file_name(std::move(o.file_name)), arch(std::move(o.arch)), metadata(std::move(o.metadata)),
		                                    tensors(std::move(o.tensors)), fd_(o.fd_) { o.fd_ = -1; }
		file_info(const file_info&) = delete;
		~file_info();
	private:
		mutable int fd_ = -1;
	};
	static file_info load(const std::string& file_name);
	static bool hash_check_available(); // libxxhash found on this box
	static unsigned long long xxh3(const void* p, size_t n); // XXH3_64bits (0 when the library is missing)
};

// ---- Config (model.h:25-91) -------------------------------------------------------------------------------------
enum class ActivationType { GELU, SILU };
enum class LayerNormType { RMSNorm };
enum class Device { CPU, CUDA };

struct Config {
	int dim, hidden_dim, head_dim, n_layers, n_heads, n_kv_heads, vocab_size, max_seq_len;
	float rope_theta;
	int rotary_dim;
	float norm_eps;
	ActivationType act;
	LayerNormType norm_type;
	float qkv_clip;
	bool tie_word_embeddings;
	static Config from_xalm(const Xalm::file_info& xalm, int context = 0);
	xalm_config to_c() const;
};

// ---- InferenceState (model.h:96-156) ----------------------------------------------------------------------------
// On the device the scratch activations belong to the backend handle; what remains on the host is the logits
// vector the Sampler reads.  After cuda() it aliases the backend's pinned buffer (no extra copy per token).
struct InferenceState {
	explicit InferenceState(const Config& config);
	void cuda() { device = Device::CUDA; }
	float* logits() const { return logits_ptr_ ? logits_ptr_ : const_cast<float*>(own_logits_.data()); }
	Device device = Device::CPU;

private:
	friend struct Model;
	std::vector<float> own_logits_;
	mutable float* logits_ptr_ = nullptr;
};

enum class InferenceMode { HYDRATE_KV_CACHE, OUTPUT_LOGITS };

// Tensor parallel over peer memory: gets this rank's XALM_IPC_HANDLE_BYTES handle, returns every rank's, in rank order.
using IpcExchange = std::function<std::vector<uint8_t>(const std::vector<uint8_t>& mine)>;

// ---- Model (model.h:254-284) ------------------------------------------------------------------------------------
struct Model {
	// defer_load: do not read the weights into host memory now — model.cuda() then streams each tensor disk -> pinned staging
	// buffer -> device, and a tensor-parallel rank reads only the rows it keeps (the reference reads everything whole first,
	// model.cpp:48-118).  The file_info must outlive the cuda() call.
	static Model from_xalm(Xalm::file_info& xalm, int context, bool defer_load = false);
	Model(Model&&) noexcept;
	Model(const Model&) = delete;
	Model& operator=(const Model&) = delete;
	~Model();

	Config config;
	Device device = Device::CPU;

	// model.cuda(): upload every tensor (sharded for tp_size > 1), release the host copies, finalize.  With tp_size > 1 and an
	// ipc_exchange, the ranks also swap CUDA IPC handles (after the communicator, before the uploads), which enables the fused
	// peer-memory exchange; without one the decode exchange is ncclAllReduce.
	// max_seqs > 1: a batched handle with that many sequence slots (xalm_cuda_set_batch; one GPU, integer block formats only).
	void cuda(int device_index = 0, int tp_rank = 0, int tp_size = 1, const void* comm_id = nullptr, const IpcExchange& ipc_exchange = {},
	          int max_seqs = 1);
	[[nodiscard]] size_t active_bytes(size_t pos) const;
	// Kernels launched by the last forward / prefill call (xalm_cuda_last_launch_count).
	[[nodiscard]] int last_launch_count() const;
	void forward(const InferenceState& s, int token, int pos, InferenceMode mode = InferenceMode::OUTPUT_LOGITS) const;
	// The per-position loops of main.cpp:94-100 / :244-254 as one batched pass on the tensor cores (xalm_cuda_prefill).
	// Positions pos0 .. pos0+n-1; mode OUTPUT_LOGITS leaves the LAST position's logits in s.logits().  With `targets` and
	// `probs` (n entries) also returns Sampler::sample_prob(targets[i]) at every position.  Returns false — and does nothing —
	// when the batch cannot take this path (ring-buffer wrap past max_seq_len): callers fall back to forward().  Under tensor
	// parallelism it is a collective: every rank calls it with the same arguments and gets the full logits.
	bool prefill(const InferenceState& s, const int* tokens, int n, int pos0, InferenceMode mode = InferenceMode::OUTPUT_LOGITS,
	             const int* targets = nullptr, float* probs = nullptr) const;
	// The same past the context window, where the KV cache is a ring with two attention sinks (xalm_cuda_prefill_window):
	// pos0 >= max_seq_len and n <= max_seq_len - 2 (longer runs go in chunks).  Leaves the cache as n forward() calls would.
	// Returns false — and does nothing — when the batch cannot take this path (positions outside that range).  Collective under
	// tensor parallelism, as prefill().
	bool prefill_window(const InferenceState& s, const int* tokens, int n, int pos0, InferenceMode mode = InferenceMode::OUTPUT_LOGITS,
	                    const int* targets = nullptr, float* probs = nullptr) const;

	// Batched decode on a max_seqs > 1 handle: one step of n sequences, slot seqs[i] takes tokens[i] at pos[i]
	// (xalm_cuda_forward_batch).  OUTPUT_LOGITS fills logits with n x vocab_size floats (may be null).  A refused call throws.
	void forward_batch(int n, const int* seqs, const int* tokens, const int* pos, InferenceMode mode, float* logits) const;
	// forward_batch + Sampler::sample_argmax of every row on the device: next[i] for seqs[i].
	void forward_batch_argmax(int n, const int* seqs, const int* tokens, const int* pos, int* next) const;
	// forward_batch_argmax where a slot may take several consecutive positions in one step (xalm_cuda_forward_spans_argmax):
	// how drafted tokens are verified in one pass over the weights.  next[i] is the greedy token after entry i.  A refused call throws.
	void forward_spans_argmax(int n, const int* seqs, const int* tokens, const int* pos, int* next) const;
	// Tree verification on one slot (xalm_cuda_forward_tree_argmax): node i decodes tokens[i] after its ancestors (parents[0] == -1,
	// 0 <= parents[i] < i) at position pos + depth(i); next[i] is the greedy token after node i.  A refused call throws.
	void forward_tree_argmax(int slot, int n, const int* tokens, const int* parents, int pos, int* next) const;
	// Move the accepted root-to-node path nodes[0 .. n-1] of the tree last verified at pos into rows pos .. pos+n-1 of the slot
	// (xalm_cuda_tree_accept; enqueue only, nothing for a chain).  A refused call throws.
	void tree_accept(int slot, int pos, int n, const int* nodes) const;
	// Greedy chain (xalm_cuda_forward_greedy): tokens[0 .. n_in-2] hydrate positions pos .. pos+n_in-2, tokens[n_in-1] decodes at
	// pos+n_in-1, and each of the n_out - 1 further steps decodes the previous step's greedy token; out[i] is step i's token.  One
	// host synchronisation per call, as a draft model drafts.  1 <= n_in <= 8, 1 <= n_out <= 16.  A refused call throws.
	void forward_greedy(const int* tokens, int n_in, int pos, int n_out, int* out) const;
	// The slot forward / prefill / prefill_window work on (default 0): how a prompt is hydrated into a slot.
	void select_seq(int seq) const;

private:
	explicit Model(const Config& c) : config(c) {}
	bool prefill_call(bool window, const InferenceState& s, const int* tokens, int n, int pos0, InferenceMode mode, const int* targets,
	                  float* probs) const;
	std::map<std::string, Tensor> host_; // until cuda()
	std::map<std::string, Type> types_;  // kept for active_bytes after the host copies are gone
	const Xalm::file_info* deferred_ = nullptr; // defer_load: where cuda() reads the tensors from
	xalm_cuda_model* handle_ = nullptr;
};

// ---- Sampler (sampler.h / sampler.cpp): host-side, unchanged semantics incl. the FLT_MIN seed (SURVEY.md §0.8) ---
struct Sampler {
	int vocab_size;
	explicit Sampler(const Config& config) noexcept : vocab_size(config.vocab_size) {}
	[[nodiscard]] float sample_prob(int index, const InferenceState& s) const;
	[[nodiscard]] int sample_argmax(const InferenceState& s) const;
};

// ---- Tokenizer (tokenizer.h / tokenizer.cpp) --------------------------------------------------------------------
struct Tokenizer {
	std::vector<std::string> vocab;
	int bos_id = -1, eos_id = -1, eot_id = -1;
	int byte_fallback_start = -1;
	explicit Tokenizer(const Xalm::file_info& data);
	std::vector<int> encode(const std::string& text, bool encode_bos) const;
	std::string decode_one(int prev_token, int token) const;
	std::string encoding_to_debug_string(const std::vector<int>& encoding) const;

private:
	// flat trie: node -> (byte -> child), children in one map keyed by (node << 8 | byte)
	std::map<uint64_t, int> edges_;
	std::vector<int> node_token_;
};

// helpers shared with main.cpp
[[noreturn]] void xalm_throw_last(const char* what);
extern "C" {
int xalm_host_quantize(int type_id, const float* src, long long n_rows, long long n_cols, uint8_t* dst);
void xalm_host_normal(uint64_t seed, uint64_t stream, long long n, float mean, float std, float* out);
}
