"""Perplexity past the context window on one GPU: the batched path (prefill over [0, W), then prefill_window in chunks of
at most W - 2) against the token-at-a-time decode path, on a synthetic model.  Prints one JSON line.

    python scripts/bench_prefill_window.py --model m7 --wtype q8_0 --window 4096 --tokens 16384

Times: host clock around calls that end in a device synchronise (prefill and prefill_window are synchronous; the token
loop syncs on every forward).  The batched pass is the perplexity workload (every position's softmax at its target, the
logits stay on the device).  The token loop is timed over a sample of the same positions: the first --loop positions of the
last window chunk, replayed from the same cache state; the logits of --sample positions spread over that range are compared
between the two paths.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from xalm_b200 import capi, synth, types as T, xalm_file as X


def gpu_name_and_power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers below are still printed, marked as lacking their hardware context
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="m7")
    ap.add_argument("--wtype", default="q8_0")
    ap.add_argument("--layers", type=int, default=0, help="override n_layers (0 = the shape's own)")
    ap.add_argument("--window", type=int, default=4096, help="context window W (the -T override)")
    ap.add_argument("--tokens", type=int, default=16384, help="positions evaluated")
    ap.add_argument("--chunk", type=int, default=4096, help="largest window chunk (capped at W - 2)")
    ap.add_argument("--split", type=int, default=0, help="prefill_split knob (0 = library default)")
    ap.add_argument("--loop", type=int, default=1024, help="positions replayed by the token loop")
    ap.add_argument("--sample", type=int, default=32, help="positions whose logits are compared")
    args = ap.parse_args()
    import bench as B
    from xalm_b200.model import InferenceState

    if args.split:
        capi.tune("prefill_split", args.split)
    W, N = args.window, args.tokens
    if N <= W:
        ap.error("--tokens must exceed --window")
    over = {"n_layers": args.layers} if args.layers else {}
    cfg_full = synth.model_config(args.model, **over)
    cfg = X.parse_config(synth.metadata_strings(cfg_full), W)
    model, _ = B.build_model_streaming(cfg_full, cfg, T.parse(args.wtype), 0, False, device=0)
    toks = np.random.default_rng(5).integers(3, cfg["vocab_size"], size=N + 1).astype(np.int32)
    C = min(args.chunk, W - 2)
    starts = list(range(W, N, C))

    def linear():
        return model.prefill(toks[:W], 0, want_logits=2, targets=toks[1:W + 1], fetch_logits=False)[1]

    def window(p0):
        n = min(C, N - p0)
        return model.prefill_window(toks[p0:p0 + n], p0, want_logits=2, targets=toks[p0 + 1:p0 + n + 1], fetch_logits=False)[1]

    # warm-up of both prefill shapes and the decode path (the linear pass rewrites every cache slot, so the timed pass starts
    # from the same state)
    st = InferenceState(cfg).cuda()
    linear(); window(W)
    model.forward(st, int(toks[0]), 0, 1)  # the decode path's first call captures its CUDA graph
    t0 = time.perf_counter()
    probs = [linear()]
    t_lin = time.perf_counter() - t0
    t1 = time.perf_counter()
    for p0 in starts:
        probs.append(window(p0))
    t_win = time.perf_counter() - t1
    probs = np.concatenate(probs)
    ppl = float(np.exp(-np.mean(np.log(probs.astype(np.float64)))))

    # the token loop over the first `loop` positions of the last chunk that has that many, from the cache state the batched
    # path reached there
    k = max([i for i, p0 in enumerate(starts) if N - p0 >= args.loop] or [len(starts) - 1])
    last = starts[k]
    n_loop = min(args.loop, N - last)
    linear()
    for p0 in starts[:k]:
        window(p0)
    ref = model.prefill_window(toks[last:last + n_loop], last, want_logits=2)
    linear()
    for p0 in starts[:k]:
        window(p0)
    sample = set(np.linspace(0, n_loop - 1, min(args.sample, n_loop)).astype(int).tolist())
    worst = 0.0
    t2 = time.perf_counter()
    for i in range(n_loop):
        model.forward(st, int(toks[last + i]), last + i, 1)
        if i in sample:
            worst = max(worst, float(np.max(np.abs(st.logits() - ref[i]))))
    t_loop = time.perf_counter() - t2
    name, limit = gpu_name_and_power_limit()
    n_win = N - W
    batched = N / (t_lin + t_win)
    loop = n_loop / t_loop
    print(json.dumps({
        "bench": "prefill_window", "model": args.model, "wtype": args.wtype, "n_layers": cfg["n_layers"], "window": W, "tokens": N,
        "chunk": C, "prefill_split": args.split or "default (3)",
        "batched_tok_s": round(batched, 1), "linear_tok_s": round(W / t_lin, 1), "window_tok_s": round(n_win / t_win, 1),
        "token_loop_tok_s": round(loop, 1), "token_loop_positions": n_loop, "speedup_vs_token_loop": round(batched / loop, 2),
        "window_speedup_vs_token_loop": round(n_win / t_win / loop, 2), "max_abs_logit_diff": worst, "sampled_positions": len(sample),
        "perplexity": ppl, "gpu": name, "power_limit": limit,
        "timing": "host clock around synchronous calls; warm-up pass of both shapes first",
    }), flush=True)
    model.close()


if __name__ == "__main__":
    main()
