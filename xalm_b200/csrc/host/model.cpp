// model.cpp — host-side implementation of the reference surface declared in model.h, over the C ABI.
#include "model.h"

#include <dlfcn.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <fstream>
#include <limits>

#include "json.h"

[[noreturn]] void xalm_throw_last(const char* what) {
	throw std::runtime_error(std::string(what) + ": " + xalm_cuda_last_error());
}

// ---- Type ------------------------------------------------------------------------------------------------------
namespace {
struct TypeRow { int id; const char* name; int block; int bytes; };
// ids/sizes: types.h:505-514, convert.py:56-61, quants.py:45-77
const TypeRow kTypes[] = {
    {XALM_F32, "F32", 1, 4}, {XALM_F16, "F16", 1, 2}, {XALM_BF16, "BF16", 1, 2}, {XALM_F8_E2M5, "F8_E2M5", 1, 1},
    {XALM_F8_E3M4, "F8_E3M4", 1, 1}, {XALM_F8_E4M3, "F8_E4M3", 1, 1}, {XALM_F8_E5M2, "F8_E5M2", 1, 1}, {XALM_U8, "U8", 1, 1},
    {XALM_Q8, "Q8", 1, 1}, {XALM_Q4_0, "Q4_0", 32, 18}, {XALM_Q4_1, "Q4_1", 32, 20}, {XALM_Q5_0, "Q5_0", 32, 22},
    {XALM_Q5_1, "Q5_1", 32, 24}, {XALM_Q8_0, "Q8_0", 32, 34}, {XALM_TQ1_0, "TQ1_0", 256, 54}, {XALM_QI8, "QI8", 1, 1},
};
} // namespace

Type Type::from_id(int id) {
	for (const auto& r : kTypes)
		if (r.id == id) return Type{r.id, r.block, r.bytes};
	return Type{};
}
Type Type::parse(std::string_view s) {
	std::string up(s);
	std::transform(up.begin(), up.end(), up.begin(), [](unsigned char c) { return (char) std::toupper(c); });
	for (const auto& r : kTypes)
		if (up == r.name) return Type{r.id, r.block, r.bytes};
	throw std::invalid_argument("invalid type: " + up); // the reference prints and asserts (types.h:496-498)
}
std::string_view Type::name() const {
	for (const auto& r : kTypes)
		if (r.id == id) return r.name;
	return "UNKNOWN";
}

// ---- Tensor ----------------------------------------------------------------------------------------------------
Tensor Tensor::zeroes(Type type, const std::vector<int>& shape, const std::string& name) {
	if (shape.size() > 4) throw std::invalid_argument("Shape cannot have more than 4 dimensions");
	Tensor t;
	t.name = name;
	t.type = type;
	t.shape = shape;
	size_t n = 1;
	for (int d : shape) {
		if (d < 0) throw std::invalid_argument("Shape dimensions must be positive");
		if (d != 0) n *= (size_t) d;
	}
	if (n % (size_t) type.block) throw std::invalid_argument("tensor length is not a multiple of the block size");
	t.linear_length = n;
	t.size = type.nbytes(n);
	const size_t alloc = (t.size + 63) / 64 * 64;
	void* p = std::aligned_alloc(64, alloc ? alloc : 64);
	if (!p) throw std::bad_alloc();
	std::memset(p, 0, alloc ? alloc : 64);
	t.data_.reset(static_cast<uint8_t*>(p));
	return t;
}

Tensor Tensor::convert_to(const Type target_type) const {
	if (!data_) throw std::invalid_argument("Tensor data cannot be null");
	if (type == target_type) throw std::invalid_argument("Tensor is already of target dtype."); // the reference prints this and exits
	if (type.id != XALM_F32 && type.id != XALM_F16 && type.id != XALM_BF16)
		throw std::invalid_argument(std::string("Unsupported conversion from dtype: ") + std::string(type.name()));
	const size_t cols = shape.empty() ? 1 : (size_t) shape.back();
	if (cols % (size_t) target_type.block) throw std::invalid_argument("row length is not a multiple of the target block size");
	std::vector<float> f(linear_length);
	if (type.id == XALM_F32) std::memcpy(f.data(), data_.get(), linear_length * 4);
	else if (type.id == XALM_F16) {
		const _Float16* h = reinterpret_cast<const _Float16*>(data_.get());
		for (size_t i = 0; i < linear_length; i++) f[i] = (float) h[i];
	} else {
		const uint16_t* b = reinterpret_cast<const uint16_t*>(data_.get());
		for (size_t i = 0; i < linear_length; i++) {
			const uint32_t u = (uint32_t) b[i] << 16; // types.h:322-325
			std::memcpy(&f[i], &u, 4);
		}
	}
	Tensor out = Tensor::zeroes(target_type, shape, name);
	if (xalm_host_quantize(target_type.id, f.data(), (long long) (linear_length / cols), (long long) cols, out.bytes()) != 0)
		throw std::invalid_argument(std::string("Unsupported conversion to dtype: ") + std::string(target_type.name()));
	return out;
}

// ---- Xalm::load (xalm.h:90-192) --------------------------------------------------------------------------------
static std::string expand_tilde(const std::string& path) {
	if (path.empty() || path[0] != '~') return path;
	const char* home = std::getenv("HOME");
	if (!home) throw std::runtime_error("HOME environment variable not set");
	return std::string(home) + path.substr(1);
}

Xalm::file_info Xalm::load(const std::string& file_name_in) {
	const std::string file_name = expand_tilde(file_name_in);
	std::ifstream stream(file_name, std::ios::binary);
	if (!stream) throw std::invalid_argument("cannot open " + file_name);
	const uint64_t file_size = std::filesystem::file_size(file_name);
	uint64_t header_end = 0;
	stream.read(reinterpret_cast<char*>(&header_end), sizeof header_end);
	if (header_end == 0 || header_end > file_size - sizeof(uint64_t))
		throw std::invalid_argument("bad json size: " + std::to_string(header_end) + " for file size: " + std::to_string(file_size));
	std::vector<char> buf(header_end - sizeof(uint64_t) + 1, 0);
	stream.read(buf.data(), (std::streamsize) (header_end - sizeof(uint64_t)));
	const size_t json_len = std::strlen(buf.data()); // the header is NUL-padded up to the data blob
	const xjson::Value header = xjson::Parser::parse(buf.data(), json_len);
	if (!header.contains("xalm")) throw std::invalid_argument("invalid file format!");
	const xjson::Value* ver = header.at("xalm").find("version");
	if (!ver || ver->inum != 1) throw std::invalid_argument("xalm version mismatch: " + std::to_string(ver ? ver->inum : 0));

	file_info fi;
	fi.file_name = file_name;
	for (const auto& [arch, val] : header.obj) {
		if (arch == "xalm") continue;
		if (arch != "LlamaForCausalLM" && arch != "MistralForCausalLM")
			throw std::invalid_argument("unsupported model architecture: " + arch); // console::error + exit(1) in the reference
		fi.arch = arch;
		for (const auto& [k, v] : val.at("config").obj) fi.metadata[k] = v.kind == xjson::Value::String ? v.str : std::to_string(v.num);
		for (const auto& [name, tv] : val.at("tensors").obj) {
			tensor_info ti;
			ti.name = name;
			const xjson::Value* ty = tv.find("type");
			ti.type = Type::parse(ty ? ty->str : "<missing>");
			const auto& shp = tv.at("shape").arr;
			if (shp.size() > 4) throw std::invalid_argument("shape exceeds 4 dimensions");
			for (const auto& d : shp) {
				if (d.kind != xjson::Value::Number || !d.is_int) throw std::invalid_argument("bad shape");
				ti.disk_shape.push_back((int) d.inum);
			}
			ti.shape = ti.disk_shape;
			if (ti.type.block > 1 && !ti.shape.empty()) {
				// block formats store uint8 rows: [rows, cols/block*bytes] (quants.py:79-83) -> element shape
				if (ti.shape.back() % ti.type.bytes)
					throw std::invalid_argument("bytes per row of " + name + " is not a multiple of the " + std::string(ti.type.name()) + " type size");
				ti.shape.back() = ti.shape.back() / ti.type.bytes * ti.type.block;
			}
			const xjson::Value* off = tv.find("offset");
			const xjson::Value* sz = tv.find("size");
			if (!off || off->inum < 0) throw std::invalid_argument("bad offset");
			if (!sz || sz->inum < 0) throw std::invalid_argument("bad size");
			if (sz->inum == 0 || header_end + (uint64_t) off->inum + (uint64_t) sz->inum > file_size)
				throw std::invalid_argument("offset out of range");
			ti.offset = header_end + (size_t) off->inum;
			ti.size = (size_t) sz->inum;
			if (const xjson::Value* hv = tv.find("hash"); hv && hv->kind == xjson::Value::Number && hv->is_int) {
				ti.hash = hv->unum; // xxh3_64 of the payload (convert.py:265-266)
				ti.has_hash = true;
			}
			size_t n = 1;
			for (int d : ti.shape) n *= (size_t) d;
			if (n % (size_t) ti.type.block || ti.type.nbytes(n) != ti.size)
				throw std::invalid_argument("size mismatch for " + name);
			ti.file_name = file_name;
			fi.tensors.emplace(name, std::move(ti));
		}
	}
	if (fi.arch.empty()) throw std::invalid_argument("no model architecture in header");
	return fi;
}

// XXH3_64bits from the system's libxxhash (0.8.x, the library convert.py's `xxhash` module wraps), resolved at run time so the
// host library has no link-time dependency on it; nullptr when the box has none (the check is then skipped, as the reference
// always does: xalm.h:90-192 parses "hash" and never looks at it).
using xxh3_fn = unsigned long long (*)(const void*, size_t);
static xxh3_fn xxh3_64bits() {
	static xxh3_fn fn = []() -> xxh3_fn {
		if (std::getenv("XALM_NO_HASH_CHECK")) return nullptr;
		for (const char* lib : {"libxxhash.so.0", "libxxhash.so"})
			if (void* h = dlopen(lib, RTLD_NOW | RTLD_LOCAL))
				if (void* f = dlsym(h, "XXH3_64bits")) return reinterpret_cast<xxh3_fn>(f);
		return nullptr;
	}();
	return fn;
}
bool Xalm::hash_check_available() { return xxh3_64bits() != nullptr; }
unsigned long long Xalm::xxh3(const void* p, size_t n) { const xxh3_fn h = xxh3_64bits(); return h ? h(p, n) : 0ull; }

Xalm::file_info::~file_info() {
	if (fd_ >= 0) ::close(fd_);
}

// One descriptor per checkpoint, positional reads: no reopen + seek per tensor (model.cpp:57 constructs an ifstream per tensor).
void Xalm::file_info::load_tensor_data(const tensor_info& ti, uint8_t* dst, size_t n) const {
	if (n != ti.size) throw std::runtime_error("buffer size mismatch"); // xalm.h:27-29
	if (fd_ < 0) {
		fd_ = ::open(ti.file_name.c_str(), O_RDONLY);
		if (fd_ < 0) throw std::runtime_error("cannot open " + ti.file_name);
	}
	size_t done = 0;
	while (done < n) {
		const ssize_t r = ::pread(fd_, dst + done, n - done, (off_t) (ti.offset + done));
		if (r <= 0) throw std::runtime_error("short read for tensor " + ti.name);
		done += (size_t) r;
	}
	if (ti.has_hash) {
		if (const xxh3_fn h = xxh3_64bits()) {
			const unsigned long long got = h(dst, n);
			if (got != ti.hash)
				throw std::runtime_error("hash mismatch for tensor " + ti.name + ": header " + std::to_string(ti.hash) + ", payload " + std::to_string(got));
		}
	}
}

Tensor Xalm::file_info::load_tensor(const std::string& name) const {
	const tensor_info& ti = tensors.at(name);
	Tensor t = Tensor::zeroes(ti.type, ti.shape, ti.name);
	load_tensor_data(ti, t.bytes(), t.size);
	return t;
}

// ---- Config::from_xalm (model.h:44-90) -------------------------------------------------------------------------
Config Config::from_xalm(const Xalm::file_info& xalm, const int context) {
	const auto& md = xalm.metadata;
	auto geti = [&](const char* k) { return std::stoi(md.at(k)); };
	auto value = [&](const char* k, const char* dflt) -> std::string {
		auto it = md.find(k);
		return it == md.end() ? dflt : it->second;
	};
	Config c{};
	c.dim = geti("dim");
	c.hidden_dim = geti("hidden_dim");
	c.head_dim = geti("head_dim");
	c.n_layers = geti("n_layers");
	c.n_heads = geti("n_heads");
	c.n_kv_heads = geti("n_kv_heads");
	c.vocab_size = geti("vocab_size");
	c.max_seq_len = std::min(geti("max_seq_len"), 4096); // model.h:54-56
	if (context) c.max_seq_len = context;              // -T (model.h:57-59)
	c.rope_theta = std::stof(md.at("rope_theta"));
	c.rotary_dim = geti("rotary_dim");
	c.norm_eps = std::stof(value("norm_eps", "1e-5"));
	const std::string act = value("act_type", "gelu");
	if (act == "silu") c.act = ActivationType::SILU;
	else {
		if (act != "gelu") std::fprintf(stderr, "unsupported act_type, defaulting to gelu\n");
		c.act = ActivationType::GELU;
	}
	if (value("norm_type", "rmsnorm") != "rmsnorm") std::fprintf(stderr, "unsupported norm_type, defaulting to rmsnorm\n");
	c.norm_type = LayerNormType::RMSNorm;
	c.qkv_clip = md.count("qkv_clip") ? std::stof(md.at("qkv_clip")) : FLT_MAX;
	c.tie_word_embeddings = md.at("tie_word_embeddings") == "True";
	return c;
}

xalm_config Config::to_c() const {
	xalm_config c{};
	c.dim = dim; c.hidden_dim = hidden_dim; c.head_dim = head_dim; c.n_layers = n_layers; c.n_heads = n_heads;
	c.n_kv_heads = n_kv_heads; c.vocab_size = vocab_size; c.max_seq_len = max_seq_len; c.rope_theta = rope_theta;
	c.rotary_dim = rotary_dim; c.norm_eps = norm_eps; c.act = act == ActivationType::SILU ? XALM_SILU : XALM_GELU;
	c.norm_type = 0; c.qkv_clip = qkv_clip; c.tie_word_embeddings = tie_word_embeddings ? 1 : 0;
	return c;
}

InferenceState::InferenceState(const Config& config) : own_logits_((size_t) config.vocab_size, 0.f) {}

// ---- Model -------------------------------------------------------------------------------------------------------
Model::Model(Model&& o) noexcept : config(o.config), device(o.device), host_(std::move(o.host_)), types_(std::move(o.types_)),
                                   deferred_(o.deferred_), handle_(o.handle_) {
	o.deferred_ = nullptr;
	o.handle_ = nullptr;
}
Model::~Model() {
	if (handle_) xalm_cuda_destroy(handle_);
}

// Model::from_xalm (model.cpp:48-118): same tensor names, same expected shapes, same failure modes
Model Model::from_xalm(Xalm::file_info& xalm, const int context, const bool defer_load) {
	const Config config = Config::from_xalm(xalm, context);
	Model m(config);
	auto load = [&](const std::string& name, const std::vector<int>& expected) {
		const auto it = xalm.tensors.find(name);
		if (it == xalm.tensors.end()) throw std::out_of_range("tensor not found: " + name); // std::map::at
		const auto& ti = it->second;
		if (expected != ti.shape) {
			auto fmt = [](const std::vector<int>& v) {
				std::string s = "[";
				for (size_t i = 0; i < v.size(); i++) s += (i ? ", " : "") + std::to_string(v[i]);
				return s + "]";
			};
			throw std::invalid_argument("shape mismatch for " + name + ": " + fmt(ti.shape) + " vs " + fmt(expected) + " expected!");
		}
		m.types_[name] = ti.type;
		if (!defer_load) m.host_.emplace(name, xalm.load_tensor(name));
	};
	if (defer_load) m.deferred_ = &xalm;
	const int q_dim = config.n_heads * config.head_dim, kv_dim = config.n_kv_heads * config.head_dim;
	load("embed.weight", {config.vocab_size, config.dim});
	for (int i = 0; i < config.n_layers; ++i) {
		const std::string p = "l." + std::to_string(i) + ".";
		load(p + "attn.norm.weight", {config.dim});
		load(p + "mlp.norm.weight", {config.dim});
		load(p + "attn.q.weight", {q_dim, config.dim});
		load(p + "attn.k.weight", {kv_dim, config.dim});
		load(p + "attn.v.weight", {kv_dim, config.dim});
		load(p + "attn.down.weight", {config.dim, q_dim});
		load(p + "mlp.gate.weight", {config.hidden_dim, config.dim});
		load(p + "mlp.down.weight", {config.dim, config.hidden_dim});
		load(p + "mlp.up.weight", {config.hidden_dim, config.dim});
	}
	load("output.norm.weight", {config.dim});
	if (!config.tie_word_embeddings) load("output.weight", {config.vocab_size, config.dim}); // tied: embed is reused (model.cpp:112-114)
	return m;
}

void Model::cuda(int device_index, int tp_rank, int tp_size, const void* comm_id, const IpcExchange& ipc_exchange, int max_seqs) {
	if (handle_) return;
	const xalm_config c = config.to_c();
	if (xalm_cuda_create(&c, device_index, tp_rank, tp_size, &handle_) != XALM_OK) xalm_throw_last("model.cuda()");
	if (max_seqs != 1 && xalm_cuda_set_batch(handle_, max_seqs) != XALM_OK) xalm_throw_last("model.cuda()");
	if (tp_size > 1) {
		if (!comm_id) throw std::invalid_argument("model.cuda(): tensor parallel needs a communicator id");
		if (xalm_cuda_comm_init(handle_, comm_id) != XALM_OK) xalm_throw_last("model.cuda()");
		if (ipc_exchange) {
			std::vector<uint8_t> mine(XALM_IPC_HANDLE_BYTES);
			if (xalm_cuda_ipc_export(handle_, mine.data()) != XALM_OK) xalm_throw_last("model.cuda()");
			const std::vector<uint8_t> table = ipc_exchange(mine);
			if (table.size() != (size_t) tp_size * XALM_IPC_HANDLE_BYTES)
				throw std::invalid_argument("model.cuda(): the IPC exchange must return tp_size x 64 bytes");
			if (xalm_cuda_ipc_import(handle_, table.data()) != XALM_OK) xalm_throw_last("model.cuda()");
		}
	}
	if (deferred_) {
		// disk -> pinned staging -> device, one tensor at a time; row-sharded tensors read only this rank's rows
		size_t cap = 0;
		for (const auto& [name, ty] : types_) cap = std::max(cap, deferred_->tensors.at(name).size);
		uint8_t* stage = static_cast<uint8_t*>(xalm_cuda_host_alloc(cap));
		if (!stage) xalm_throw_last("model.cuda()");
		struct Guard { uint8_t* p; ~Guard() { xalm_cuda_host_free(p); } } guard{stage};
		for (const auto& [name, ty] : types_) {
			const Xalm::tensor_info& ti = deferred_->tensors.at(name);
			int rng[4];
			if (xalm_cuda_shard_range(handle_, name.c_str(), rng) != XALM_OK) xalm_throw_last("model.cuda()");
			const int rows = ti.shape.empty() ? 1 : ti.shape[0];
			const int cols = ti.shape.size() > 1 ? ti.shape[1] : 1;
			const bool row_shard = ti.shape.size() == 2 && rng[2] == 0 && rng[3] == cols && (rng[0] != 0 || rng[1] != rows);
			int rc;
			if (row_shard) { // a contiguous byte range of the payload (the header's hash covers the whole tensor: not checked here)
				const size_t row_bytes = ti.type.nbytes((size_t) cols);
				Xalm::tensor_info part = ti;
				part.offset = ti.offset + (size_t) rng[0] * row_bytes;
				part.size = (size_t) (rng[1] - rng[0]) * row_bytes;
				part.has_hash = false;
				deferred_->load_tensor_data(part, stage, part.size);
				rc = xalm_cuda_upload_tensor_shard(handle_, name.c_str(), ti.type.id, ti.shape.data(), (int) ti.shape.size(), rng, stage, part.size);
			} else { // replicated or column-split: the whole tensor (hash verified), the backend keeps its columns
				deferred_->load_tensor_data(ti, stage, ti.size);
				rc = xalm_cuda_upload_tensor(handle_, name.c_str(), ti.type.id, ti.shape.data(), (int) ti.shape.size(), stage, ti.size);
			}
			if (rc != XALM_OK) xalm_throw_last("model.cuda()");
		}
		deferred_ = nullptr;
	}
	for (auto it = host_.begin(); it != host_.end();) {
		const Tensor& t = it->second;
		if (xalm_cuda_upload_tensor(handle_, it->first.c_str(), t.type.id, t.shape.data(), (int) t.shape.size(), t.bytes(), t.size) != XALM_OK)
			xalm_throw_last("model.cuda()");
		it = host_.erase(it); // the device owns the weights from here on
	}
	if (xalm_cuda_finalize(handle_) != XALM_OK) xalm_throw_last("model.cuda()");
	device = Device::CUDA;
}

size_t Model::active_bytes(const size_t pos) const {
	// model.cpp:12-35 in 64-bit with per-format bytes (the reference's int arithmetic overflows at 128256 x 4096 x 16)
	auto wb = [&](const std::string& name, size_t elems) { return types_.at(name).nbytes(elems); };
	const size_t dim = config.dim, hidden = config.hidden_dim, q_dim = (size_t) config.n_heads * config.head_dim,
	             kv_dim = (size_t) config.n_kv_heads * config.head_dim;
	size_t bytes = wb("embed.weight", dim) + wb("output.norm.weight", dim) +
	               wb(config.tie_word_embeddings ? "embed.weight" : "output.weight", (size_t) config.vocab_size * dim);
	for (int l = 0; l < config.n_layers; ++l) {
		const std::string p = "l." + std::to_string(l) + ".";
		bytes += wb(p + "attn.norm.weight", dim) + wb(p + "mlp.norm.weight", dim);
		bytes += wb(p + "attn.q.weight", q_dim * dim) + wb(p + "attn.k.weight", kv_dim * dim) + wb(p + "attn.v.weight", kv_dim * dim) +
		         wb(p + "attn.down.weight", q_dim * dim);
		bytes += wb(p + "mlp.gate.weight", dim * hidden) + wb(p + "mlp.down.weight", dim * hidden) + wb(p + "mlp.up.weight", dim * hidden);
		const size_t kv_len = std::min((size_t) config.max_seq_len, pos + 1);
		bytes += 2 * kv_len * kv_dim * sizeof(uint16_t);
	}
	return bytes;
}

int Model::last_launch_count() const {
	int n = 0;
	if (!handle_ || xalm_cuda_last_launch_count(handle_, &n) != XALM_OK) return 0;
	return n;
}

void Model::forward(const InferenceState& s, const int token, const int pos, const InferenceMode mode) const {
	if (device != Device::CUDA || !handle_)
		throw std::runtime_error("Model::forward: model is not on a CUDA device (call model.cuda()); this backend has no CPU path");
	if (!s.logits_ptr_ && s.device == Device::CUDA) s.logits_ptr_ = xalm_cuda_logits_host(handle_); // alias the pinned buffer
	const int m = mode == InferenceMode::OUTPUT_LOGITS ? XALM_OUTPUT_LOGITS : XALM_HYDRATE_KV_CACHE;
	if (xalm_cuda_forward(handle_, token, pos, m, m == XALM_OUTPUT_LOGITS ? s.logits() : nullptr) != XALM_OK) {
		// forward-time failures abort in the reference (noexcept matmul + assert, infer.cpp:211-214)
		std::fprintf(stderr, "Model::forward: %s\n", xalm_cuda_last_error());
		std::abort();
	}
}

bool Model::prefill(const InferenceState& s, const int* tokens, const int n, const int pos0, const InferenceMode mode, const int* targets,
                    float* probs) const {
	if (n <= 0 || pos0 < 0 || (long long) pos0 + n > config.max_seq_len) return false;
	return prefill_call(false, s, tokens, n, pos0, mode, targets, probs);
}

bool Model::prefill_window(const InferenceState& s, const int* tokens, const int n, const int pos0, const InferenceMode mode, const int* targets,
                           float* probs) const {
	if (n <= 0 || pos0 < config.max_seq_len || n > config.max_seq_len - 2) return false;
	return prefill_call(true, s, tokens, n, pos0, mode, targets, probs);
}

bool Model::prefill_call(const bool window, const InferenceState& s, const int* tokens, const int n, const int pos0, const InferenceMode mode,
                         const int* targets, float* probs) const {
	if (device != Device::CUDA || !handle_)
		throw std::runtime_error("Model::prefill: model is not on a CUDA device (call model.cuda()); this backend has no CPU path");
	if (!s.logits_ptr_ && s.device == Device::CUDA) s.logits_ptr_ = xalm_cuda_logits_host(handle_);
	auto call = window ? xalm_cuda_prefill_window : xalm_cuda_prefill;
	int rc;
	if (targets && probs) rc = call(handle_, tokens, n, pos0, 2, nullptr, targets, probs);
	else if (mode == InferenceMode::OUTPUT_LOGITS) rc = call(handle_, tokens, n, pos0, 1, s.logits(), nullptr, nullptr);
	else rc = call(handle_, tokens, n, pos0, 0, nullptr, nullptr, nullptr);
	if (rc == XALM_ERR_UNSUPPORTED) return false; // e.g. a head_dim the batched attention kernel does not take
	if (rc != XALM_OK) {
		std::fprintf(stderr, "Model::%s: %s\n", window ? "prefill_window" : "prefill", xalm_cuda_last_error());
		std::abort();
	}
	return true;
}

void Model::forward_batch(const int n, const int* seqs, const int* tokens, const int* pos, const InferenceMode mode, float* logits) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::forward_batch: model is not on a CUDA device (call model.cuda())");
	const int m = mode == InferenceMode::OUTPUT_LOGITS ? XALM_OUTPUT_LOGITS : XALM_HYDRATE_KV_CACHE;
	if (xalm_cuda_forward_batch(handle_, n, seqs, tokens, pos, m, logits) != XALM_OK) xalm_throw_last("Model::forward_batch");
}

void Model::forward_batch_argmax(const int n, const int* seqs, const int* tokens, const int* pos, int* next) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::forward_batch_argmax: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_forward_batch_argmax(handle_, n, seqs, tokens, pos, next) != XALM_OK) xalm_throw_last("Model::forward_batch_argmax");
}

void Model::forward_spans_argmax(const int n, const int* seqs, const int* tokens, const int* pos, int* next) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::forward_spans_argmax: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_forward_spans_argmax(handle_, n, seqs, tokens, pos, next) != XALM_OK) xalm_throw_last("Model::forward_spans_argmax");
}

void Model::forward_tree_argmax(const int slot, const int n, const int* tokens, const int* parents, const int pos, int* next) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::forward_tree_argmax: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_forward_tree_argmax(handle_, slot, n, tokens, parents, pos, next) != XALM_OK) xalm_throw_last("Model::forward_tree_argmax");
}

void Model::tree_accept(const int slot, const int pos, const int n, const int* nodes) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::tree_accept: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_tree_accept(handle_, slot, pos, n, nodes) != XALM_OK) xalm_throw_last("Model::tree_accept");
}

void Model::forward_greedy(const int* tokens, const int n_in, const int pos, const int n_out, int* out) const {
	if (device != Device::CUDA || !handle_) throw std::runtime_error("Model::forward_greedy: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_forward_greedy(handle_, n_in, tokens, pos, n_out, out) != XALM_OK) xalm_throw_last("Model::forward_greedy");
}

void Model::select_seq(const int seq) const {
	if (!handle_) throw std::runtime_error("Model::select_seq: model is not on a CUDA device (call model.cuda())");
	if (xalm_cuda_select_seq(handle_, seq) != XALM_OK) xalm_throw_last("Model::select_seq");
}

// ---- Sampler (sampler.cpp:3-30) ----------------------------------------------------------------------------------
// The running maximum starts at numeric_limits<float>::min() — the smallest POSITIVE normal — exactly like the
// reference; with all logits <= 1.18e-38 argmax answers 0.  Token-exact parity depends on keeping this.
float Sampler::sample_prob(const int index, const InferenceState& s) const {
	const float* lg = s.logits();
	float top = std::numeric_limits<float>::min();
	for (int i = 0; i < vocab_size; ++i) top = lg[i] > top ? lg[i] : top;
	float denom = 0;
	for (int i = 0; i < vocab_size; ++i) denom += expf(lg[i] - top);
	return expf(lg[index] - top) / denom;
}
int Sampler::sample_argmax(const InferenceState& s) const {
	const float* lg = s.logits();
	int best = 0;
	float top = std::numeric_limits<float>::min();
	for (int i = 0; i < vocab_size; ++i)
		if (lg[i] > top) { top = lg[i]; best = i; }
	return best;
}

// ---- Tokenizer (tokenizer.cpp) -----------------------------------------------------------------------------------
static int first_int(const std::string& s) { // "[1, 2]" or "1" -> 1 (tokenizer.cpp:4-21)
	size_t i = 0;
	while (i < s.size() && (s[i] == '[' || s[i] == ' ')) i++;
	return std::stoi(s.substr(i));
}

Tokenizer::Tokenizer(const Xalm::file_info& data) {
	bos_id = first_int(data.metadata.at("bos_token_id"));
	eos_id = first_int(data.metadata.at("eos_token_id"));
	const Tensor toks = data.load_tensor("tokenizer.tokens");
	if (toks.type.id != XALM_U8) throw std::invalid_argument("tokenizer.tokens must be U8");
	const char* p = toks.get_data<char>();
	const char* end = p + toks.linear_length;
	while (p < end) { // NUL-separated strings
		const char* s = p;
		while (p < end && *p != '\0') p++;
		vocab.emplace_back(s, (size_t) (p - s));
		p++;
	}
	node_token_.push_back(-1); // root
	for (size_t i = 0; i < vocab.size(); i++) {
		const std::string& w = vocab[i];
		if (w == "<0x00>") byte_fallback_start = (int) i;
		else if (w == "<|eot_id|>" || w == "<|end|>" || w == "<|im_end|>") eot_id = (int) i;
		int node = 0;
		for (unsigned char ch : w) {
			const uint64_t key = ((uint64_t) node << 8) | ch;
			auto it = edges_.find(key);
			if (it == edges_.end()) {
				node_token_.push_back(-1);
				it = edges_.emplace(key, (int) node_token_.size() - 1).first;
			}
			node = it->second;
		}
		node_token_[node] = (int) i; // a later duplicate wins, as in the reference's trie build
	}
}

std::vector<int> Tokenizer::encode(const std::string& text, const bool encode_bos) const {
	std::vector<int> out;
	if (encode_bos) out.push_back(bos_id);
	for (size_t i = 0; i < text.size();) {
		int node = 0, best = -1;
		size_t best_len = 0;
		for (size_t l = 0; i + l < text.size(); l++) { // greedy longest match
			const auto it = edges_.find(((uint64_t) node << 8) | (unsigned char) text[i + l]);
			if (it == edges_.end()) break;
			node = it->second;
			if (node_token_[node] >= 0) { best = node_token_[node]; best_len = l + 1; }
		}
		if (best < 0) {
			if (byte_fallback_start >= 0) out.push_back((unsigned char) text[i] + byte_fallback_start);
			i += 1;
		} else {
			out.push_back(best);
			i += best_len;
		}
	}
	return out;
}

std::string Tokenizer::decode_one(const int prev_token, const int token) const {
	const std::string& piece = vocab.at((size_t) token);
	if (prev_token == bos_id && !piece.empty() && piece[0] == ' ') return piece.substr(1); // sentencepiece strips it after BOS
	if (byte_fallback_start >= 0 && token >= byte_fallback_start && token - byte_fallback_start < 256)
		return std::string(1, (char) (token - byte_fallback_start));
	return piece;
}

std::string Tokenizer::encoding_to_debug_string(const std::vector<int>& encoding) const {
	std::string s;
	for (const int id : encoding) {
		if (id == bos_id) s += "[<s>:" + std::to_string(id) + "]";
		else if (id == eos_id) s += "[</s>:" + std::to_string(id) + "]";
		else s += "[" + vocab.at((size_t) id) + ":" + std::to_string(id) + "]";
	}
	return s;
}
