"""Batched decode on one GPU: Mistral-7B shape (synthetic weights), 1 / 2 / 4 / 8 sequences per step on a batched handle.

One JSON line per (format, sequence count): device step time (CUDA events around `steps` enqueued steps on the model's stream),
aggregate and per-sequence tok/s, bytes per step from the shapes (weights once + each sequence's K/V rows), that over the
measured 6.54 TB/s, and a parity key (4 greedy steps of every sequence in the batch against the same sequence decoded alone by
the batch-1 kernel).  Then the batched W1|W3 matvec alone (`xalm_cuda_bench_matvec_batch`) next to the batch-1 kernel.  Each
step's positions are spread over [0, 4096) as in bench.py, at every sequence count; the card name and power limit are read in
the same run.

    python scripts/bench_batch.py [--formats q8_0,q4_0] [--steps 64] [--out profiles/r6_batch_decode.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from xalm_b200 import capi, synth  # noqa: E402
from xalm_b200 import types as T  # noqa: E402
from xalm_b200 import xalm_file as X  # noqa: E402
from xalm_b200.model import Model  # noqa: E402
from bench import positions_for  # noqa: E402

PEAK_GBS = 6540.0   # measured HBM rate of the B200 (DESIGN.md §5)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--formats", default="q8_0,q4_0")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join("profiles", "r6_batch_decode.jsonl"))
    args = ap.parse_args()
    gpu = card()
    cfg_full = synth.model_config("m7")
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    kv_dim = cfg["n_kv_heads"] * cfg["head_dim"]
    kv_row = 2 * kv_dim * 2 * cfg["n_layers"]            # K and V, fp16, every layer
    lines = []
    for wname in args.formats.split(","):
        wtype = T.parse(wname)
        stream = torch.cuda.Stream()
        m = Model.from_tensors(cfg, synth.iter_tensors(cfg_full, wtype, 0, std=0.02)).cuda(max_seqs=8, release_host=True,
                                                                                             stream=stream.cuda_stream)
        weights = m.active_bytes(0) - kv_row
        rng = np.random.default_rng(1)
        for n in (1, 2, 4, 8):
            seqs = list(range(n))
            # as bench.py: every step's positions spread over [0, ctx); sequence i of step k takes position k * n + i of the spread
            pl = positions_for(args.steps * n, args.ctx)
            step_pos = [[int(pl[k * n + i]) for i in range(n)] for k in range(args.steps)]
            toks = [int(t) for t in rng.integers(0, cfg["vocab_size"], n)]
            for k in range(4):                            # warm-up: the graph of this n is captured
                m.forward_batch_async(seqs, toks, step_pos[k])
            m.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.steps):
                m.forward_batch_async(seqs, toks, step_pos[k])
            e1.record(stream)
            e1.synchronize()
            dt = e0.elapsed_time(e1) / 1e3 / args.steps
            kv_bytes = sum(min(p + 1, args.ctx) for row in step_pos for p in row) / args.steps * kv_row
            step_bytes = weights + kv_bytes
            # parity: 4 greedy steps of the batch against each sequence decoded alone by the batch-1 kernel (select_seq + forward)
            start = [min(p + 1, args.ctx - 5) for p in step_pos[-1]]   # inside the window: re-running a step rewrites the same rows
            got, cur = [], list(toks)
            for k in range(4):
                cur = m.forward_batch_argmax(seqs, cur, [p + k for p in start])
                got.append(cur)
            alone = []
            for i in range(n):
                m.select_seq(i)
                t, row = toks[i], []
                for k in range(4):
                    t = m.forward_argmax(t, start[i] + k)
                    row.append(t)
                alone.append(row)
            m.select_seq(0)
            parity = all([got[k][i] for k in range(4)] == alone[i] for i in range(n))
            rec = {"gpu": gpu, "shape": "m7", "wtype": wname, "n_seqs": n, "step_ms": dt * 1e3, "tok_s": n / dt, "tok_s_per_seq": 1 / dt,
                   "bytes_per_step": int(step_bytes), "weight_bytes": int(weights), "kv_bytes_per_step": int(kv_bytes),
                   "frac_of_6540_gbs": step_bytes / dt / 1e9 / PEAK_GBS, "parity_vs_alone": parity,
                   "positions": f"spread uniformly over [0, {args.ctx}) as in bench.py, {args.steps} timed steps",
                   "timing": "CUDA events on the model's stream", "parity": "4 greedy steps vs each sequence alone on the batch-1 kernel"}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        m.close()
        tid = wtype.id
        for n in (1, 2, 4, 8):
            ms = capi.bench_matvec_batch(tid, 4096, 14336, n, 4, 100, epi=2, with_norm=True)
            rec = {"gpu": gpu, "kernel": "batched W1|W3 (quantiser + matvec)", "wtype": wname, "n_seqs": n, "us": ms * 1e3,
                   "weight_bytes": 2 * 14336 * 4096 * wtype.bytes // wtype.block}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        ms = capi.bench_matvec(tid, 4096, 14336, 4, 100, epi=2, with_norm=True)
        rec = {"gpu": gpu, "kernel": "batch-1 W1|W3 (the kernel bench.py's handle runs)", "wtype": wname, "n_seqs": 1, "us": ms * 1e3}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
