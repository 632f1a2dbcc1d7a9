// main.cpp — the reference's CLI surface (src/main.cpp:417-547) on top of the CUDA backend.
//
//   xalm_main <checkpoint.xalm> [-d cuda] [-m completion|passkey|perplexity] [-T ctx] [-i prompt | -f file] [-n steps] [-l pos] [-g gpus]
//
// Same flags, same prefix matching for -m/-d, same defaults (mode completion, -n 128, the default prompt), same stats
// block, plus the roofline fraction.  Differences, on purpose:
//   * `-d` defaults to cuda here and `-d cpu` is refused: this build IS the cuda backend, it carries no CPU forward
//     (the reference's usage text already says "default - cuda", main.cpp:24);
//   * run_completion honours -d (the reference drops it, main.cpp:44,537);
//   * elapsed time is wall clock (the reference divides by user+system CPU time, main.cpp:101,117);
//   * `-g P` runs the model tensor-parallel on CUDA devices 0 .. P-1 (launch.h): P worker processes run the same mode function,
//     rank 0 prints.  The reference has no multi-GPU path.  Without -g, or with -g 1, nothing forks.
//
// Under -g P every decision the mode functions take must come out the same on every rank, or the ranks' collectives (each
// forward / prefill call) stop matching up.  They depend only on the arguments, the inherited environment, the checkpoint and
// the logits — which every rank receives whole and bit-identical — so they do; the comments below name the less obvious ones.
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>

#include "launch.h"
#include "model.h"

namespace {

[[noreturn]] void error_usage() {
	fprintf(stderr, "Usage:   xalm_main <checkpoint> [options]\n");
	fprintf(stderr, "Example: xalm_main model.xalm -i \"Q: What is the meaning of life?\"\n");
	fprintf(stderr, "Options:\n");
	fprintf(stderr, "  -h Display this help message\n");
	fprintf(stderr, "  -d [cuda] which device to use (default - cuda; this build has no cpu path)\n");
	fprintf(stderr, "  -m [completion,passkey,perplexity] which mode to run in (default - completion)\n");
	fprintf(stderr, "  -T <int> sliding window context length (0 - max)\n");
	fprintf(stderr, "  -g <int> number of GPUs to run tensor-parallel on (default - 1; not with -m verify)\n");
	fprintf(stderr, "\nPerplexity mode options:\n  Choose one:\n    -i <string> input prompt\n    -f <filepath> input file with prompt\n");
	fprintf(stderr, "Completion mode options:\n  -n <int>    number of steps to run for in completion mode, default 128. 0 = max_seq_len, -1 = infinite\n");
	fprintf(stderr, "  Choose one:\n    -i <string> input prompt\n    -f <filepath> input file with prompt\n");
	fprintf(stderr, "Passkey mode options:\n  -n <int>    number of junk lines to insert (default - 250)\n  -l <int>    passkey position (-1 - random)\n");
	exit(1);
}

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

double hbm_peak_gbs() {
	// measured on this pool (MEASURED_PEAKS.json); XALM_HBM_PEAK_GBS overrides
	if (const char* e = getenv("XALM_HBM_PEAK_GBS")) return atof(e);
	return 6538.3;
}

// model.cuda() for this rank; the one-GPU TpRank makes it the plain model.cuda().
void to_device(Model& model, const TpRank& tp) { model.cuda(tp.device, tp.rank, tp.size, tp.comm_id, tp.ipc_exchange); }

// Under tensor parallelism: which GPUs, and how many kernels one decode token takes (this shows which exchange path runs).
void print_tp_stats(const TpRank& tp, int launches) {
	if (tp.size > 1) printf("  tensor parallel: %d GPUs, %d launches/token\n", tp.size, launches);
}

void run_completion(const TpRank& tp, const std::string& checkpoint_path, const std::string& prompt, int context, int num_steps) {
	auto model_data = Xalm::load(checkpoint_path);
	std::cout << "loading model " << checkpoint_path << std::endl;
	Model model = Model::from_xalm(model_data, context, /*defer_load=*/true); // weights go disk -> pinned -> device in model.cuda()
	printf("Model active bytes(m): %zu\n", model.active_bytes(model.config.max_seq_len) / (1024 * 1024));
	std::cout << "Using CUDA" << std::endl;
	to_device(model, tp);
	InferenceState state(model.config);
	state.cuda();
	Sampler sampler(model.config);
	Tokenizer tokenizer(model_data);
	if (num_steps == 0) num_steps = model.config.max_seq_len; // `-n 0` = full context (main.cpp:67-70)
	model.forward(state, 0, 0);                               // warm-up (main.cpp:72): captures the CUDA graph
	const int launches = model.last_launch_count();

	double t0 = now_s();
	std::vector<int> encoding = tokenizer.encode(prompt, true);
	std::cout << tokenizer.encoding_to_debug_string(encoding) << std::endl;
	const double enc_s = now_s() - t0;
	printf("Encoding stats: (%zu tokens, throughput: %.5gtok/s, latency: %.5gs/tok, total: %.5gs)\n\n", encoding.size(),
	       encoding.size() / enc_s, enc_s / encoding.size(), enc_s);

	t0 = now_s();
	size_t read_bytes = 0;
	// hydrate the KV cache (main.cpp:94-100).  The reference walks the prompt token by token; here the part of the prompt
	// that fits the cache without wrapping goes through ONE batched pass (tcgen05 GEMMs), the part past the context window
	// through batched passes over the KV ring, and whatever those refuse (e.g. a head_dim the batched attention does not take)
	// through the same loop.  The chunk sizes depend on the prompt and the config only, and a refusal is agreed between the
	// ranks (xalm_cuda.h), so under -g every rank makes the same calls and falls back at the same position.
	size_t pos = 0;
	if (getenv("XALM_NO_PREFILL") == nullptr && encoding.size() > 1) {
		const size_t W = (size_t) model.config.max_seq_len;
		const size_t n = std::min(encoding.size(), W);
		const InferenceMode mode = n == encoding.size() ? InferenceMode::OUTPUT_LOGITS : InferenceMode::HYDRATE_KV_CACHE;
		if (model.prefill(state, encoding.data(), (int) n, 0, mode)) {
			read_bytes += model.active_bytes(n - 1); // the weights are streamed once for the whole batch
			pos = n;
		}
		while (pos >= W && pos < encoding.size()) {
			const size_t c = std::min({encoding.size() - pos, W - 2, (size_t) 4096});
			const InferenceMode cmode = pos + c == encoding.size() ? InferenceMode::OUTPUT_LOGITS : InferenceMode::HYDRATE_KV_CACHE;
			if (!model.prefill_window(state, encoding.data() + pos, (int) c, (int) pos, cmode)) break;
			read_bytes += model.active_bytes(pos + c - 1);
			pos += c;
		}
	}
	for (; pos < encoding.size(); pos++) {
		const InferenceMode mode = pos + 1 == encoding.size() ? InferenceMode::OUTPUT_LOGITS : InferenceMode::HYDRATE_KV_CACHE;
		model.forward(state, encoding[pos], (int) pos, mode);
		read_bytes += model.active_bytes(pos);
	}
	const double hydrate_s = now_s() - t0;
	for (int i = 0; i < num_steps || num_steps == -1; i++) { // main.cpp:105-115
		// the logits are all-gathered under -g, so every rank picks the same token and stops at the same step
		const int token_id = sampler.sample_argmax(state);
		std::cout << tokenizer.decode_one(encoding.back(), token_id) << std::flush;
		encoding.push_back(token_id);
		if (token_id == tokenizer.eos_id || token_id == tokenizer.eot_id) break;
		model.forward(state, token_id, (int) encoding.size() - 1);
		read_bytes += model.active_bytes(encoding.size() - 1);
	}
	std::cout << "\n" << std::endl;
	const double elapsed_s = now_s() - t0;
	// bandwidth: the whole model's bytes (every rank streams its shard of them), against the P GPUs' aggregate peak
	const double gbs = (double) read_bytes / 1e9 / elapsed_s, peak = tp.size * hbm_peak_gbs();
	printf("Generation stats:\n  %zu tokens\n  throughput: %.5gtok/s\n  latency: %.5gs/tok\n  hydrate: %.5gs\n  bandwidth: %.5gGB/s\n"
	       "  roofline: %.1f%% of %.0f GB/s HBM\n  total: %.5gs\n",
	       encoding.size(), encoding.size() / elapsed_s, elapsed_s / encoding.size(), hydrate_s, gbs, 100.0 * gbs / peak, peak, elapsed_s);
	print_tp_stats(tp, launches);
}

void run_perplexity(const TpRank& tp, const std::string& checkpoint_path, const std::string& prompt, int context) {
	auto model_data = Xalm::load(checkpoint_path);
	Model model = Model::from_xalm(model_data, context, /*defer_load=*/true); // weights go disk -> pinned -> device in model.cuda()
	std::cout << "Model active bytes with full context window: " << model.active_bytes(model.config.max_seq_len) << std::endl;
	std::cout << "Using CUDA" << std::endl;
	to_device(model, tp);
	InferenceState state(model.config);
	state.cuda();
	Sampler sampler(model.config);
	Tokenizer tokenizer(model_data);
	model.forward(state, 0, 0);
	const int launches = model.last_launch_count();
	std::vector<int> encoding = tokenizer.encode(prompt, true);
	std::cout << tokenizer.encoding_to_debug_string(encoding) << std::endl;
	if (encoding.size() < 2) { fprintf(stderr, "Error: perplexity needs at least two tokens\n"); exit(1); }
	double sum_logprob = 0.0, ss_logprob = 0.0;
	const double t0 = now_s();
	size_t read_bytes = 0;
	const size_t N = encoding.size() - 1;
	size_t pos = 0;
	// main.cpp:244-254 evaluates one position per forward; here positions are evaluated in batched passes of up to 4096 (every
	// position's logits on the device, softmax-at-target there too): those that fit the cache without wrapping through prefill,
	// those past the context window through prefill_window (at most max_seq_len - 2 per pass), whatever they refuse as before
	// (a refusal is the same on every rank, so under -g the ranks leave this loop together).
	if (getenv("XALM_NO_PREFILL") == nullptr) {
		std::vector<float> probs;
		const size_t W = (size_t) model.config.max_seq_len;
		while (pos < N) {
			const bool window = pos >= W;
			const size_t n = std::min({N - pos, window ? W - 2 : W - pos, (size_t) 4096});
			probs.resize(n);
			const int* tg = encoding.data() + pos + 1;
			if (!(window ? model.prefill_window(state, encoding.data() + pos, (int) n, (int) pos, InferenceMode::OUTPUT_LOGITS, tg, probs.data())
			             : model.prefill(state, encoding.data() + pos, (int) n, (int) pos, InferenceMode::OUTPUT_LOGITS, tg, probs.data())))
				break;
			std::cout << "\r Computing perplexity..." << pos + n << "/" << N << std::flush;
			read_bytes += model.active_bytes(pos + n - 1);
			for (size_t i = 0; i < n; i++) {
				const double logprob = std::log(probs[i]);
				sum_logprob += logprob;
				ss_logprob += logprob * logprob;
			}
			pos += n;
		}
	}
	for (; pos + 1 < encoding.size(); pos++) {
		std::cout << "\r Computing perplexity..." << pos + 1 << "/" << N << std::flush;
		model.forward(state, encoding[pos], (int) pos);
		read_bytes += model.active_bytes(pos);
		const double logprob = std::log(sampler.sample_prob(encoding[pos + 1], state));
		sum_logprob += logprob;
		ss_logprob += logprob * logprob;
	}
	std::cout << std::endl;
	const double elapsed_s = now_s() - t0;
	const double perplexity = std::exp(-sum_logprob / N);
	const double perplexity_error = perplexity * std::sqrt((ss_logprob - sum_logprob * sum_logprob / N) / N / N);
	printf("Stats:\n  %zu tokens\n  perplexity: %.5g ± %.5g\n  throughput: %.5gtok/s\n  latency: %.5gs/tok\n  bandwidth: %.5gGB/s\n  total: %.5gs\n", N,
	       perplexity, perplexity_error, N / elapsed_s, elapsed_s / N, (double) read_bytes / 1e9 / elapsed_s, elapsed_s);
	print_tp_stats(tp, launches);
}

void run_passkey(const TpRank& tp, const std::string& checkpoint_path, int context, int n_junk, int passkey_pos) {
	auto model_data = Xalm::load(checkpoint_path);
	Model model = Model::from_xalm(model_data, context, /*defer_load=*/true); // weights go disk -> pinned -> device in model.cuda()
	std::cout << "Model active bytes with full context window: " << model.active_bytes(model.config.max_seq_len) << std::endl;
	std::cout << "Using CUDA" << std::endl;
	to_device(model, tp);
	InferenceState state(model.config);
	state.cuda();
	Sampler sampler(model.config);
	Tokenizer tokenizer(model_data);
	model.forward(state, 0, 0);
	const std::string PROMPT_PREFIX = "There is an important info hidden inside a lot of irrelevant text. "
	                                  "Find it and memorize them. I will quiz you about the important information there.";
	const std::string PROMPT_SUFFIX = " What is the pass key? The pass key is";
	// unseeded, like the reference (main.cpp:298).  Under -g every rank must draw the same values, so nothing may call rand()
	// before this on some ranks only; the one call rank 0 alone makes, for the NCCL id, does not (libnccl takes no rand()).
	const int passkey = std::rand() % 50000 + 1;
	const int pos = passkey_pos == -1 ? std::rand() % n_junk : passkey_pos;
	std::string prompt = PROMPT_PREFIX;
	for (int i = 0; i < n_junk; i++) {
		if (i % n_junk == pos)
			prompt += " The pass key is " + std::to_string(passkey) + ". Remember it. " + std::to_string(passkey) + " is the pass key.";
		prompt += " The grass is green. The sky is blue. The sun is yellow. Here we go. There and back again.";
	}
	prompt += PROMPT_SUFFIX;
	std::vector<int> encoding = tokenizer.encode(prompt, true);
	printf("Passkey test:\n  prompt: %zu tokens\n  passkey: %d\n  passkey token index: ~%d\n", encoding.size(), passkey,
	       (int) ((float) pos / n_junk * encoding.size()));
	const size_t N = encoding.size();
	for (size_t p = 0; p < N; p++) {
		std::cout << "\r Running passkey test..." << p + 1 << "/" << N << std::flush;
		model.forward(state, encoding[p], (int) p, p + 1 == N ? InferenceMode::OUTPUT_LOGITS : InferenceMode::HYDRATE_KV_CACHE);
	}
	std::cout << std::endl << PROMPT_SUFFIX << std::flush;
	for (size_t p = N; p < N + 16; p++) { // at most 16 steps (main.cpp:323)
		const int token_id = sampler.sample_argmax(state);
		std::cout << tokenizer.decode_one(encoding.back(), token_id) << std::flush;
		encoding.push_back(token_id);
		if (token_id == tokenizer.eos_id || token_id == tokenizer.eot_id) break;
		model.forward(state, token_id, (int) p);
	}
	std::cout << std::endl;
}

// -m verify: read every tensor of the checkpoint once and check its xxh3_64 against the header (host only, no device needed).
// With -t <type>: additionally re-encode every F32/F16/BF16 matrix with Tensor::convert_to and print "<name> <type> <bytes> <xxh3>"
// (the call sites the reference has commented out at main.cpp:54-63).
int run_verify(const std::string& checkpoint_path, const std::string& convert_type) {
	auto data = Xalm::load(checkpoint_path);
	if (!Xalm::hash_check_available()) std::cout << "warning: libxxhash not found, hashes are NOT checked" << std::endl;
	size_t n = 0, bytes = 0, hashed = 0;
	for (const auto& [name, ti] : data.tensors) {
		Tensor t = data.load_tensor(name); // throws std::runtime_error on a hash mismatch
		n++; bytes += t.size; hashed += ti.has_hash ? 1 : 0;
		if (!convert_type.empty() && t.shape.size() == 2 && (t.type.id == XALM_F32 || t.type.id == XALM_F16 || t.type.id == XALM_BF16)) {
			const Type target = Type::parse(convert_type);
			if (target == t.type) continue;
			const Tensor c = t.convert_to(target);
			std::cout << name << " " << c.type.name() << " " << c.size << " " << Xalm::xxh3(c.bytes(), c.size) << std::endl;
		}
	}
	std::cout << "verified " << n << " tensors (" << hashed << " with a hash), " << bytes << " bytes" << std::endl;
	return 0;
}

bool is_prefix_of(const std::string& full, const std::string& s) { return !s.empty() && full.compare(0, s.size(), s) == 0; }

// -g: a whole positive number, anything else is a usage error
int parse_gpus(const std::string& v) {
	char* end = nullptr;
	errno = 0;
	const long n = strtol(v.c_str(), &end, 10);
	if (v.empty() || *end != '\0' || errno || n < 1 || n > 1024) error_usage();
	return (int) n;
}

} // namespace

int main(int argc, char* argv[]) {
	std::string checkpoint_path, device = "cuda", mode = "completion";
	std::string prompt = "Q: What is the meaning of life? A:"; // main.cpp:421
	std::string prompt_path;
	std::string convert_type;
	int context = 0, num_steps = 128, n_junk = 250, passkey_pos = -1, gpus = 1;
	if (argc >= 2) checkpoint_path = argv[1];
	else error_usage();
	for (int i = 2; i < argc;) { // main.cpp:435-512
		if (i + 1 >= argc || argv[i][0] != '-' || strlen(argv[i]) != 2) error_usage();
		const char f = argv[i][1];
		const std::string v = argv[i + 1];
		if (f == 'm') {
			if (is_prefix_of("completion", v)) mode = "completion";
			else if (is_prefix_of("passkey", v)) mode = "passkey";
			else if (is_prefix_of("perplexity", v)) mode = "perplexity";
			else if (is_prefix_of("verify", v)) mode = "verify";
			else error_usage();
		} else if (f == 'd') {
			if (is_prefix_of("cpu", v)) device = "cpu";
			else if (is_prefix_of("cuda", v)) device = "cuda";
			else error_usage();
		} else if (f == 'i') prompt = v;
		else if (f == 'f') prompt_path = v;
		else if (f == 'T') context = std::stoi(v);
		else if (f == 't') convert_type = v;
		else if (f == 'l') passkey_pos = std::stoi(v);
		else if (f == 'g') gpus = parse_gpus(v);
		else if (f == 'n') { num_steps = std::stoi(v); n_junk = num_steps; }
		else error_usage();
		i += 2;
	}
	if (mode == "verify") {
		if (gpus != 1) {
			fprintf(stderr, "Error: -m verify runs on the host only and takes no -g\n");
			error_usage();
		}
		try {
			return run_verify(checkpoint_path, convert_type);
		} catch (const std::exception& e) {
			fprintf(stderr, "error: %s\n", e.what());
			return 1;
		}
	}
	if (device != "cuda") {
		fprintf(stderr, "Error: this binary is the CUDA backend; it carries no CPU forward pass (use the reference for -d cpu)\n");
		return 1;
	}
	if (mode == "completion" || mode == "perplexity") {
		if (!prompt_path.empty()) { // the reference's default prompt makes `-f` alone an error (main.cpp:513-517); -f simply wins here
			std::ifstream file(prompt_path);
			if (!file.is_open()) { std::cerr << "Error: could not open file " << prompt_path << std::endl; return 1; }
			std::stringstream buffer;
			buffer << file.rdbuf();
			prompt = buffer.str();
		} else if (prompt.empty()) error_usage();
	} else if (passkey_pos != -1 && (passkey_pos >= n_junk || passkey_pos < 0)) {
		std::cerr << "Error: passkey position must be between 0 and " << n_junk - 1 << std::endl;
		return 1;
	}
	auto run = [&](const TpRank& tp) {
		try {
			if (mode == "completion") run_completion(tp, checkpoint_path, prompt, context, num_steps);
			else if (mode == "passkey") run_passkey(tp, checkpoint_path, context, n_junk, passkey_pos);
			else run_perplexity(tp, checkpoint_path, prompt, context);
		} catch (const std::exception& e) {
			fprintf(stderr, "error: %s\n", e.what());
			return 1;
		}
		return 0;
	};
	return gpus == 1 ? run(TpRank{}) : run_tp_ranks(gpus, run);
}
