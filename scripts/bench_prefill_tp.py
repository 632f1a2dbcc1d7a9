"""Batched prefill on a tensor-parallel model (one GPU per rank) against the token loop on the same handles.  Prints one JSON
line from rank 0 (and appends it to --out when given).  Run it under torch.distributed.run; one process is the single-GPU case:

    python -m torch.distributed.run --nproc-per-node 2 scripts/bench_prefill_tp.py --model m7 --wtype q8_0 --tokens 4096
    python -m torch.distributed.run --nproc-per-node 8 scripts/bench_prefill_tp.py --model l70 --context 32768 --tokens 4096 \\
        --window-chunks 2

Timing: CUDA events bracketing prefill_async + a synchronise of the model stream (device synchronises on both sides), after a warm-up pass of the same shape,
averaged over --steps passes (every pass rewrites the same cache rows).  Window chunks (--window-chunks K, past a context of
--context positions hydrated by linear prefills) go through the synchronous prefill_window with the same events around it.  The
exchange share comes from a separate pass with XALM_PREFILL_TIMING=1 (one stream, per-category events).  The token loop is timed
with the host clock over --loop positions at the end of the prompt, replayed from the cache the prefill left (each forward
synchronises); its logits at --sample of them are compared with the prefill's.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def gpu_name_and_power_limit(device):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # the numbers are still printed, marked as lacking their hardware context
        return f"unknown ({e})", "unknown"


def timing_spans(fn):
    """Run fn() with XALM_PREFILL_TIMING set and return the per-category milliseconds the library prints to stderr."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        os.environ["XALM_PREFILL_TIMING"] = "1"
        try:
            fn()
        finally:
            del os.environ["XALM_PREFILL_TIMING"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read()
    spans = {}
    for line in text.splitlines():
        for what, ms in re.findall(r" (\w+) ([0-9.]+) ms;", line):
            spans[what] = spans.get(what, 0.0) + float(ms)
    return spans


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="m7")
    ap.add_argument("--wtype", default="q8_0")
    ap.add_argument("--layers", type=int, default=0, help="override n_layers (0 = the shape's own)")
    ap.add_argument("--tokens", type=int, default=4096, help="positions of the timed linear pass")
    ap.add_argument("--context", type=int, default=0, help="max_seq_len (the -T override; 0 = --tokens)")
    ap.add_argument("--window-chunks", type=int, default=0, help="window chunks timed past a hydrated context (0 = none)")
    ap.add_argument("--chunk", type=int, default=4096, help="window chunk size and linear hydrate chunk (capped at context - 2)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--loop", type=int, default=64, help="positions replayed by the token loop")
    ap.add_argument("--sample", type=int, default=16, help="positions whose logits are compared with the token loop")
    ap.add_argument("--out", default="", help="append the JSON line to this file")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    W = args.context or args.tokens
    T_ = args.tokens
    if T_ > W:
        ap.error("--tokens must not exceed --context")
    import torch
    import torch.distributed as dist
    import bench as B
    from xalm_b200 import synth, tp, types as T, xalm_file as X
    from xalm_b200.model import InferenceState

    over = {"n_layers": args.layers} if args.layers else {}
    cfg_full = synth.model_config(args.model, **over)
    cfg = X.parse_config(synth.metadata_strings(cfg_full), W)
    torch.cuda.set_device(local)
    kw = dict(device=local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
        kw.update(tp_rank=rank, tp_size=world, comm_id=tp.broadcast_comm_id(dist, rank, device="cuda"),
                  ipc_exchange=tp.make_ipc_exchange(dist, world))
    model, _ = B.build_model_streaming(cfg_full, cfg, T.parse(args.wtype), 0, False, **kw)
    toks = np.random.default_rng(5).integers(3, cfg["vocab_size"], size=max(T_, W) + args.chunk * (args.window_chunks + 2) + 1).astype(np.int32)

    def timed(fn):  # the model runs on its own stream: the events bracket it through device synchronises
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        model.sync()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 1e3

    lin = lambda: model.prefill_async(toks[:T_], 0, want_logits=2)
    lin(); model.sync()                                   # warm-up (scratch growth, first launches)
    t_lin = np.mean([timed(lin) for _ in range(args.steps)])
    spans_lin = timing_spans(lambda: model.prefill(toks[:T_], 0, want_logits=2, fetch_logits=False))
    res = {"bench": "prefill_tp", "model": args.model, "wtype": args.wtype, "n_layers": cfg["n_layers"], "tp": world, "context": W,
           "tokens": T_, "steps": args.steps, "linear_tok_s": round(T_ / t_lin, 1), "linear_ms": round(t_lin * 1e3, 2),
           "linear_spans_ms": {k: round(v, 2) for k, v in spans_lin.items()},
           "linear_exchange_share": round(spans_lin.get("exchange", 0.0) / max(sum(spans_lin.values()), 1e-9), 4)}

    # the token loop on the same handles: the last `loop` positions of the prompt, from the cache the prefill left
    ref = model.prefill(toks[:T_], 0, want_logits=2)
    st = InferenceState(cfg).cuda()
    p_first = T_ - args.loop
    model.forward(st, int(toks[p_first]), p_first, 1)     # warm-up (graph capture)
    sample = set(np.linspace(0, args.loop - 1, min(args.sample, args.loop)).astype(int).tolist())
    worst = 0.0
    t0 = time.perf_counter()
    for i in range(args.loop):
        model.forward(st, int(toks[p_first + i]), p_first + i, 1)
        if i in sample:
            worst = max(worst, float(np.max(np.abs(st.logits() - ref[p_first + i]))))
    t_loop = time.perf_counter() - t0
    del ref
    res.update({"token_loop_tok_s": round(args.loop / t_loop, 1), "token_loop_positions": args.loop,
                "speedup_vs_token_loop": round(T_ / t_lin / (args.loop / t_loop), 1), "max_abs_logit_diff_vs_token_loop": worst,
                "sampled_positions": len(sample)})

    if args.window_chunks:
        C = min(args.chunk, W - 2)
        for p0 in range(0, W, C):                        # hydrate [0, W)
            model.prefill(toks[p0:min(W, p0 + C)], p0, want_logits=0)
        pos = W
        win = lambda p0: model.prefill_window(toks[p0:p0 + C], p0, want_logits=2, targets=toks[p0 + 1:p0 + C + 1], fetch_logits=False)
        win(pos); pos += C                                # warm-up of the window shape
        ts = []
        for _ in range(args.window_chunks):
            p0 = pos
            ts.append(timed(lambda: win(p0)))
            pos += C
        spans_win = timing_spans(lambda: win(pos))
        res.update({"window_chunk": C, "window_chunks": args.window_chunks, "window_tok_s": round(C / np.mean(ts), 1),
                    "window_spans_ms": {k: round(v, 2) for k, v in spans_win.items()},
                    "window_exchange_share": round(spans_win.get("exchange", 0.0) / max(sum(spans_win.values()), 1e-9), 4)})
    name, limit = gpu_name_and_power_limit(local)
    res.update({"gpu": name, "power_limit": limit,
                "timing": "CUDA events around prefill_async + synchronise after a warm-up pass; token loop: host clock, synchronous forwards"})
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
