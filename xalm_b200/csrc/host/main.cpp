// main.cpp — the reference's CLI surface (src/main.cpp:417-547) on top of the CUDA backend.
//
//   xalm_main <checkpoint.xalm> [-d cuda] [-m completion|passkey|perplexity|batch] [-T ctx] [-i prompt | -f file] [-n steps] [-l pos] [-g gpus] [-b seqs]
//             [-s draft] [-w branches] [-D draft.xalm]
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
#include <optional>
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
	fprintf(stderr, "  -m [completion,passkey,perplexity,batch] which mode to run in (default - completion)\n");
	fprintf(stderr, "  -T <int> sliding window context length (0 - max)\n");
	fprintf(stderr, "  -g <int> number of GPUs to run tensor-parallel on (default - 1; not with -m verify)\n");
	fprintf(stderr, "\nPerplexity mode options:\n  Choose one:\n    -i <string> input prompt\n    -f <filepath> input file with prompt\n");
	fprintf(stderr, "Completion mode options:\n  -n <int>    number of steps to run for in completion mode, default 128. 0 = max_seq_len, -1 = infinite\n");
	fprintf(stderr, "  -s <int>    speculative decoding: verify up to this many prompt-lookup draft tokens per pass (1..7; one GPU,\n"
	                "              integer block formats; same output as without -s)\n");
	fprintf(stderr, "  -w <int>    with -s k: verify up to this many prompt-lookup continuations per pass as one tree (1..k,\n"
	                "              default 1; not with -D)\n");
	fprintf(stderr, "  -D <filepath> with -s: draft the tokens with this model (same tokenizer, any weight format, same GPU) instead of\n"
	                "              prompt lookup\n");
	fprintf(stderr, "  Choose one:\n    -i <string> input prompt\n    -f <filepath> input file with prompt\n");
	fprintf(stderr, "Batch mode options (one GPU; integer block formats):\n  -f <filepath> prompts, one per non-empty line\n"
	                "  -b <int>    sequences decoded together (1..8, default 8)\n  -n <int>    tokens per prompt, default 128. 0 = max_seq_len\n");
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

// Hydrate the KV cache with a prompt (main.cpp:94-100) and leave the last position's logits in `state`.  The reference walks the
// prompt token by token; here the part of the prompt that fits the cache without wrapping goes through ONE batched pass (tcgen05
// GEMMs), the part past the context window through batched passes over the KV ring, and whatever those refuse (e.g. a head_dim
// the batched attention does not take) through the same loop.  The chunk sizes depend on the prompt and the config only, and a
// refusal is agreed between the ranks (xalm_cuda.h), so under -g every rank makes the same calls and falls back at the same
// position.  Returns the bytes the calls streamed (Model::active_bytes per pass).
size_t hydrate(const Model& model, const InferenceState& state, const std::vector<int>& encoding) {
	size_t read_bytes = 0;
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
	return read_bytes;
}

// Drafted tokens to verify in one pass, as a tree under the sequence's last token (node 0, not stored here): drafted node i + 1
// decodes tokens[i] after node parents[i] (0: the last token itself).  Nodes are numbered in insertion order, so parents[i] <= i.
struct DraftTree {
	std::vector<int> tokens, parents;
};

// Prompt lookup: the continuations after earlier occurrences of the sequence's last 3 tokens, most recent first, then after those
// of its last 2 (a single token is too weak a match to be worth a wider pass), up to k tokens each.  The first b that each add a
// token the ones before do not already propose are merged into a trie under the last token, which grows level by level (every
// candidate's first token, then every candidate's second, ...) in candidate order until it holds k drafted nodes.  With b = 1 this
// is the chain after the most recent occurrence.  Empty when neither suffix occurred before.
DraftTree draft_lookup(const std::vector<int>& seq, int k, int b) {
	const size_t N = seq.size();
	std::vector<std::vector<int>> cand;
	auto adds_nothing = [&](const std::vector<int>& c) {
		for (const auto& o : cand)
			if (o.size() >= c.size() && std::equal(c.begin(), c.end(), o.begin())) return true;
		return false;
	};
	for (size_t n = 3; n >= 2 && (int) cand.size() < b; n--) {
		if (N <= n) continue;
		for (size_t s = N - n; s-- > 0 && (int) cand.size() < b;) // occurrences starting before the suffix itself, latest first
			if (std::equal(seq.begin() + s, seq.begin() + s + n, seq.end() - n)) {
				const size_t from = s + n, len = std::min((size_t) k, N - from);
				std::vector<int> c(seq.begin() + from, seq.begin() + from + len);
				if (!adds_nothing(c)) cand.push_back(std::move(c));
			}
	}
	DraftTree t;
	std::vector<int> at(cand.size(), 0); // the node each candidate has reached
	for (size_t d = 0; (int) t.tokens.size() < k; d++) {
		bool any = false;
		for (size_t c = 0; c < cand.size() && (int) t.tokens.size() < k; c++) {
			if (d >= cand[c].size()) continue;
			any = true;
			int child = -1;
			for (size_t i = 0; i < t.tokens.size() && child < 0; i++)
				if (t.parents[i] == at[c] && t.tokens[i] == cand[c][d]) child = (int) i + 1;
			if (child < 0) {
				t.tokens.push_back(cand[c][d]);
				t.parents.push_back(at[c]);
				child = (int) t.tokens.size();
			}
			at[c] = child;
		}
		if (!any) break;
	}
	return t;
}

struct SpecStats {
	size_t passes = 0, drafted = 0, accepted = 0, decoded = 0; // decoded: tokens the passes produced (accepted + one per pass)
	size_t branched = 0;                                       // passes whose tree had more than one branch
};

// Where the drafts of -m completion -s k come from: prompt lookup, or a draft model (-D) decoding greedily on its own handle.
struct Drafter {
	const Model* model = nullptr; // the draft model; nullptr: prompt lookup
	size_t valid = 0;             // draft model: its KV rows 0 .. valid-1 hold the accepted sequence
	size_t steps = 0, calls = 0;  // draft model: forward steps run, and forward_greedy calls that ran them
	double seconds = 0.0;

	// up to k tokens to follow seq; P = seq.size() - 1 is the target's next position and P + k stays inside the window.  The draft
	// model catches up on the accepted tokens it has not decoded (seq[valid .. P]) and drafts k tokens in one greedy chain.
	// b: prompt lookup's candidates per pass (-w); the draft model gives one, a chain.
	DraftTree draft(const std::vector<int>& seq, int k, int b) {
		if (!model) return draft_lookup(seq, k, b);
		const size_t P = seq.size() - 1;
		DraftTree t;
		t.tokens.resize(k);
		const double t0 = now_s();
		model->forward_greedy(seq.data() + valid, (int) (P + 1 - valid), (int) valid, k, t.tokens.data());
		seconds += now_s() - t0;
		steps += P + 1 - valid + k - 1;
		calls++;
		for (int i = 0; i < k; i++) t.parents.push_back(i);
		return t;
	}
	// a of the drafts of a round at P were accepted.  The chain wrote draft rows P+1 .. P+n-1 for its first n-1 drafts, and those
	// of the accepted ones hold accepted tokens; rows of rejected drafts are rewritten before they are read, as a span's are
	// (xalm_cuda.h).  So the next round feeds one token, or two when every draft was accepted.
	void accepted(size_t P, int a, int n) {
		if (model) valid = P + std::min(a, n - 1) + 1;
	}
};

// The generation loop of -m completion -s k [-w b]: the same greedy tokens, fewer passes over the weights.  Each step drafts a tree
// of up to k tokens (Drafter; a chain unless prompt lookup has several candidates) and verifies it with the last token as its
// root in ONE pass (Model::forward_tree_argmax): node i's greedy token is what a plain step would produce after the branch from
// the root to i.  So starting at the root, the walk moves to the child whose token is the current node's greedy token while there
// is one; the drafts it passes are accepted, plus the model's own token after the last.  Model::tree_accept moves that branch's
// rows into place (nothing for a chain, or the lowest-numbered branch); rows of rejected drafts need no cleanup (xalm_cuda.h).
// Without a draft, or past the context window where trees are refused, the step is a plain forward on slot 0.  Prints the tokens
// as run_completion does; returns the bytes read.
size_t generate_speculative(const Model& model, const InferenceState& state, const Sampler& sampler, const Tokenizer& tokenizer,
                            std::vector<int>& encoding, int num_steps, int k, int b, Drafter& drafter, SpecStats& st) {
	const size_t W = (size_t) model.config.max_seq_len;
	const size_t kv_row = W > 1 ? model.active_bytes(1) - model.active_bytes(0) : 0, weights = model.active_bytes(0) - kv_row;
	size_t read_bytes = 0;
	std::vector<int> pending = {sampler.sample_argmax(state)}; // greedy tokens known but not printed yet
	std::vector<int> toks, parents, depth, out, path;
	for (int i = 0;;) {
		bool stop = false;
		for (const int token_id : pending) {
			if (!(i < num_steps || num_steps == -1)) { stop = true; break; }
			std::cout << tokenizer.decode_one(encoding.back(), token_id) << std::flush;
			encoding.push_back(token_id);
			i++;
			if (token_id == tokenizer.eos_id || token_id == tokenizer.eot_id) { stop = true; break; }
		}
		if (stop || !(i < num_steps || num_steps == -1)) break;
		const size_t P = encoding.size() - 1;            // position of the last token, not yet decoded
		const size_t room = P + 1 < W ? W - 1 - P : 0;    // draft positions P+1 .. P+len stay inside the window
		const DraftTree draft = room ? drafter.draft(encoding, (int) std::min(room, (size_t) k), b) : DraftTree{};
		st.passes++;
		if (draft.tokens.empty()) {
			model.forward(state, encoding.back(), (int) P);
			read_bytes += model.active_bytes(P);
			pending = {sampler.sample_argmax(state)};
			st.decoded++;
			continue;
		}
		const int n = (int) draft.tokens.size() + 1;
		toks.assign(1, encoding.back());
		toks.insert(toks.end(), draft.tokens.begin(), draft.tokens.end());
		parents.assign(1, -1);
		parents.insert(parents.end(), draft.parents.begin(), draft.parents.end());
		depth.assign(1, 0);
		for (int i = 1; i < n; i++) depth.push_back(depth[parents[i]] + 1);
		out.resize(n);
		model.forward_tree_argmax(0, n, toks.data(), parents.data(), (int) P, out.data());
		read_bytes += weights;
		for (int i = 0; i < n; i++) read_bytes += (P + depth[i] + 1) * kv_row;
		path.assign(1, 0);
		for (int i = 1; i < n; i++) // children come after their parent: one scan finds the accepted branch
			if (parents[i] == path.back() && toks[i] == out[path.back()]) path.push_back(i);
		model.tree_accept(0, (int) P, (int) path.size(), path.data());
		const int a = (int) path.size() - 1;
		drafter.accepted(P, a, n - 1);
		pending.clear();
		for (int j = 1; j <= a; j++) pending.push_back(toks[path[j]]);
		pending.push_back(out[path.back()]);
		st.drafted += n - 1;
		st.accepted += a;
		st.decoded += a + 1;
		if (*std::max_element(depth.begin(), depth.end()) < n - 1) st.branched++;
	}
	return read_bytes;
}

void run_completion(const TpRank& tp, const std::string& checkpoint_path, const std::string& prompt, int context, int num_steps, int spec,
                    int width, const std::string& draft_path) {
	auto model_data = Xalm::load(checkpoint_path);
	std::cout << "loading model " << checkpoint_path << std::endl;
	Model model = Model::from_xalm(model_data, context, /*defer_load=*/true); // weights go disk -> pinned -> device in model.cuda()
	// -D: the draft model must speak the target's tokens: the same vocabulary size and tokenizer, checked before any device work
	std::optional<Xalm::file_info> draft_data;
	std::optional<Model> draft;
	if (!draft_path.empty()) {
		draft_data.emplace(Xalm::load(draft_path));
		draft.emplace(Model::from_xalm(*draft_data, context, /*defer_load=*/true));
		if (draft->config.vocab_size != model.config.vocab_size)
			throw std::invalid_argument("draft model " + draft_path + ": vocab_size " + std::to_string(draft->config.vocab_size) + " differs from the target's " +
			                            std::to_string(model.config.vocab_size));
		const Tensor a = model_data.load_tensor("tokenizer.tokens"), b = draft_data->load_tensor("tokenizer.tokens");
		if (a.size != b.size || std::memcmp(a.bytes(), b.bytes(), a.size) != 0)
			throw std::invalid_argument("draft model " + draft_path + ": tokenizer.tokens differ from the target's");
	}
	printf("Model active bytes(m): %zu\n", model.active_bytes(model.config.max_seq_len) / (1024 * 1024));
	std::cout << "Using CUDA" << std::endl;
	if (spec) model.cuda(0, 0, 1, nullptr, {}, spec + 1); // -s k: a batched handle wide enough for a span of k drafts + the last token
	else to_device(model, tp);
	InferenceState state(model.config);
	state.cuda();
	Sampler sampler(model.config);
	Tokenizer tokenizer(model_data);
	if (num_steps == 0) num_steps = model.config.max_seq_len; // `-n 0` = full context (main.cpp:67-70)
	model.forward(state, 0, 0);                               // warm-up (main.cpp:72): captures the CUDA graph
	const int launches = model.last_launch_count();
	std::optional<InferenceState> draft_state;
	Drafter drafter;
	if (draft) { // the same GPU, a plain batch-1 handle: any weight format
		draft->cuda();
		draft_state.emplace(draft->config);
		draft_state->cuda();
		draft->forward(*draft_state, 0, 0);
		drafter.model = &*draft;
	}

	double t0 = now_s();
	std::vector<int> encoding = tokenizer.encode(prompt, true);
	std::cout << tokenizer.encoding_to_debug_string(encoding) << std::endl;
	const double enc_s = now_s() - t0;
	printf("Encoding stats: (%zu tokens, throughput: %.5gtok/s, latency: %.5gs/tok, total: %.5gs)\n\n", encoding.size(),
	       encoding.size() / enc_s, enc_s / encoding.size(), enc_s);

	t0 = now_s();
	size_t read_bytes = hydrate(model, state, encoding);
	if (draft) {
		hydrate(*draft, *draft_state, encoding);
		drafter.valid = encoding.size();
	}
	const double hydrate_s = now_s() - t0;
	SpecStats spec_stats;
	if (spec) read_bytes += generate_speculative(model, state, sampler, tokenizer, encoding, num_steps, spec, width, drafter, spec_stats);
	else for (int i = 0; i < num_steps || num_steps == -1; i++) { // main.cpp:105-115
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
	if (spec)
		printf("  speculative: %zu passes, %zu drafted, %zu accepted, %.3g tokens/pass\n", spec_stats.passes, spec_stats.drafted, spec_stats.accepted,
		       spec_stats.passes ? (double) spec_stats.decoded / spec_stats.passes : 0.0);
	if (width > 1) printf("  tree: up to %d branches, %zu passes verified more than one\n", width, spec_stats.branched);
	if (draft) printf("  draft: %s, %zu steps in %zu calls, %.5gs\n", draft_path.c_str(), drafter.steps, drafter.calls, drafter.seconds);
}

// -m batch: every non-empty line of the prompt file is one prompt; up to `max_batch` of them decode together on one batched handle,
// greedy, with continuous batching: when a sequence ends (eos / eot or num_steps tokens) the next prompt is hydrated into its slot
// (select_seq + the completion mode's hydrate) and joins the following step.  Each sequence's tokens are what -m completion
// produces for that prompt (the batched matvec is bit-identical to the single-sequence tensor-core kernel).
void run_batch(const std::string& checkpoint_path, const std::vector<std::string>& prompts, int context, int num_steps, int max_batch) {
	auto model_data = Xalm::load(checkpoint_path);
	std::cout << "loading model " << checkpoint_path << std::endl;
	Model model = Model::from_xalm(model_data, context, /*defer_load=*/true);
	const int B = std::max(1, std::min(max_batch, (int) prompts.size()));
	std::cout << "Using CUDA, " << B << " sequence slots" << std::endl;
	model.cuda(0, 0, 1, nullptr, {}, std::max(B, 2)); // a batched handle even when one slot is enough
	InferenceState state(model.config);
	state.cuda();
	Sampler sampler(model.config);
	Tokenizer tokenizer(model_data);
	if (num_steps == 0) num_steps = model.config.max_seq_len;
	// bytes of one cached position (K and V of every layer) and of the weights alone, for the bandwidth figure
	const size_t kv_row = model.config.max_seq_len > 1 ? model.active_bytes(1) - model.active_bytes(0) : 0;
	const size_t weights = model.active_bytes(0) - kv_row;

	struct Seq {
		int prompt = -1;  // -1: slot idle
		std::vector<int> enc;
		int generated = 0;
	};
	std::vector<Seq> slot(B);
	std::vector<std::string> text(prompts.size());
	size_t next_prompt = 0, generated = 0, read_bytes = 0, steps = 0, seq_steps = 0;
	double hydrate_s = 0.0;
	const double t0 = now_s();
	// emit the sequence's next token (as run_completion prints it); true when the sequence has ended
	auto emit = [&](Seq& q, int token) {
		text[q.prompt] += tokenizer.decode_one(q.enc.back(), token);
		q.enc.push_back(token);
		q.generated++;
		generated++;
		return token == tokenizer.eos_id || token == tokenizer.eot_id || q.generated == num_steps;
	};
	// hydrate the next prompt into slot s and emit its first token; prompts that end at once free the slot for the next one
	auto start = [&](int s) {
		slot[s].prompt = -1;
		while (next_prompt < prompts.size()) {
			Seq& q = slot[s];
			q = Seq{(int) next_prompt, tokenizer.encode(prompts[next_prompt], true), 0};
			next_prompt++;
			const double h0 = now_s();
			model.select_seq(s);
			read_bytes += hydrate(model, state, q.enc);
			hydrate_s += now_s() - h0;
			if (!emit(q, sampler.sample_argmax(state))) return;
			q.prompt = -1;
		}
	};
	for (int s = 0; s < B; s++) start(s);
	std::vector<int> seqs, toks, pos, nxt(B);
	for (;;) {
		seqs.clear(); toks.clear(); pos.clear();
		for (int s = 0; s < B; s++)
			if (slot[s].prompt >= 0) {
				seqs.push_back(s);
				toks.push_back(slot[s].enc.back());
				pos.push_back((int) slot[s].enc.size() - 1);
			}
		if (seqs.empty()) break;
		const int n = (int) seqs.size();
		model.forward_batch_argmax(n, seqs.data(), toks.data(), pos.data(), nxt.data());
		steps++;
		seq_steps += n;
		read_bytes += weights;
		for (int i = 0; i < n; i++) read_bytes += std::min((size_t) pos[i] + 1, (size_t) model.config.max_seq_len) * kv_row;
		for (int i = 0; i < n; i++)
			if (emit(slot[seqs[i]], nxt[i])) start(seqs[i]);
	}
	const double elapsed_s = now_s() - t0;
	for (size_t i = 0; i < prompts.size(); i++) printf("[prompt %zu]\n%s\n", i, text[i].c_str());
	const double gbs = (double) read_bytes / 1e9 / elapsed_s;
	printf("\nBatch stats:\n  %zu prompts\n  %zu generated tokens\n  throughput: %.5gtok/s\n  hydrate: %.5gs\n  mean sequences per step: %.3g\n"
	       "  bandwidth: %.5gGB/s\n  roofline: %.1f%% of %.0f GB/s HBM\n  total: %.5gs\n",
	       prompts.size(), generated, generated / elapsed_s, hydrate_s, steps ? (double) seq_steps / steps : 0.0, gbs, 100.0 * gbs / hbm_peak_gbs(),
	       hbm_peak_gbs(), elapsed_s);
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
	std::string convert_type, draft_path;
	int context = 0, num_steps = 128, n_junk = 250, passkey_pos = -1, gpus = 1, max_batch = 8, spec = 0, width = 0;
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
			else if (is_prefix_of("batch", v)) mode = "batch";
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
		else if (f == 'b') {
			max_batch = parse_gpus(v);
			if (max_batch > 8) error_usage();
		}
		else if (f == 's') {
			spec = parse_gpus(v);
			if (spec > 7) error_usage();
		}
		else if (f == 'w') width = parse_gpus(v);
		else if (f == 'D') draft_path = v;
		else if (f == 'n') { num_steps = std::stoi(v); n_junk = num_steps; }
		else error_usage();
		i += 2;
	}
	if (spec && (mode != "completion" || gpus != 1)) {
		fprintf(stderr, "Error: -s runs -m completion on one GPU (no -g)\n");
		error_usage();
	}
	if (!draft_path.empty() && !spec) {
		fprintf(stderr, "Error: -D drafts for -s (speculative -m completion on one GPU)\n");
		error_usage();
	}
	if (width && (!spec || width > spec || !draft_path.empty())) {
		fprintf(stderr, "Error: -w b widens -s k's prompt-lookup drafts to a tree of up to b branches, 1 <= b <= k (not with -D)\n");
		error_usage();
	}
	if (!width) width = 1;
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
	if (mode == "batch") {
		if (gpus != 1 || num_steps < 0 || prompt_path.empty()) {
			fprintf(stderr, "Error: -m batch runs on one GPU (no -g), needs -f <prompts> and -n >= 0\n");
			error_usage();
		}
		std::ifstream file(prompt_path);
		if (!file.is_open()) { std::cerr << "Error: could not open file " << prompt_path << std::endl; return 1; }
		std::vector<std::string> prompts;
		for (std::string line; std::getline(file, line);)
			if (!line.empty()) prompts.push_back(line);
		if (prompts.empty()) { std::cerr << "Error: no prompts in " << prompt_path << std::endl; return 1; }
		try {
			run_batch(checkpoint_path, prompts, context, num_steps, max_batch);
		} catch (const std::exception& e) {
			fprintf(stderr, "error: %s\n", e.what());
			return 1;
		}
		return 0;
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
			if (mode == "completion") run_completion(tp, checkpoint_path, prompt, context, num_steps, spec, width, draft_path);
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
