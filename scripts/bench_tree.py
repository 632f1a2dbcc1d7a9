"""Tree verification on one GPU: Mistral-7B shape (synthetic weights), one batched handle (max_seqs = 8).

For each format, one JSON line per measurement:
  * the plain greedy step on the batched handle (`forward_argmax`, slot 0: what -s runs without a draft);
  * for n = 2 .. 8 nodes: `forward_tree_argmax` of a chain, of a bushy tree (2 branches for n <= 5, else 3, numbered level by
    level as xalm_main numbers them), and `forward_spans_argmax` of n entries;
  * `tree_accept` of a 7-row path that moves 6 rows (each call followed by a synchronise), against the synchronise alone;
  * parity: an 8-node tree of two branches at position 3988, every node bit-identical to plain steps along its branch.
Every call is synchronous, so each time is a host clock around `steps` calls that each end in a device synchronise.  Start
positions are spread over [0, 4096 - 8] with bench.positions_for.  The card name and power limit are read in the same run.

--compare-lib PATH: a libxalm_cuda.so built from another commit (e.g. the parent).  Then the same process also loads that
library, builds the same q8_0 model on it, and times `forward_spans_argmax` and `forward_batch_argmax` at n = 2, 4, 8 on both
libraries, alternating them over --rounds rounds; the JSON lines give every round's time and the spread.

    python scripts/bench_tree.py [--formats q8_0,q4_0] [--steps 64] [--compare-lib /path/libxalm_cuda.so] [--out profiles/r9_tree_verify.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402

from bench import positions_for  # noqa: E402
from bench_batch import card  # noqa: E402
from xalm_b200 import capi, synth  # noqa: E402
from xalm_b200 import types as T  # noqa: E402
from xalm_b200 import xalm_file as X  # noqa: E402
from xalm_b200.model import InferenceState, Model  # noqa: E402

N_MAX = 8


def timed(fn, steps):
    """seconds per call of fn(k), k = 0 .. steps-1, after 4 warm-up calls (graph capture); every call ends in a synchronise"""
    for k in range(4):
        fn(k)
    t0 = time.perf_counter()
    for k in range(steps):
        fn(k)
    return (time.perf_counter() - t0) / steps


def chain(n):
    return [-1] + list(range(n - 1))


def bushy(n):
    """n nodes, 2 branches (n <= 5) or 3, level by level: node i >= 1 continues node i - nb (or the root)"""
    nb = 2 if n <= 5 else 3
    return [-1] + [0 if i <= nb else i - nb for i in range(1, n)]


def path_to(parents, i):
    p = []
    while i >= 0:
        p.append(i)
        i = parents[i]
    return p[::-1]


def load_lib(path):
    L = C.CDLL(path)
    for name, (res, args) in capi.SYMBOLS.items():
        if hasattr(L, name):
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
    return L


def parity(m, cfg, toks, P):
    """an 8-node two-branch tree on slot 1 at P against plain steps (batch-1 tensor-core kernel) along each branch on slot 1"""
    parents = [-1, 0, 0, 1, 2, 3, 4, 5]              # branches 1-3-5-7 and 2-4-6
    tt = list(toks)
    st = InferenceState(cfg)
    m.select_seq(1)
    ref = [None] * N_MAX
    for leaf in (6, 7):
        for e, node in enumerate(path_to(parents, leaf)):
            m.forward(st, tt[node], P + e, 1)
            ref[node] = st.logits().copy()
    m.select_seq(0)
    lg = m.forward_tree(1, tt, parents, P)
    return all(np.array_equal(lg[i].view(np.uint32), ref[i].view(np.uint32)) for i in range(N_MAX))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--formats", default="q8_0,q4_0")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--compare-lib", default="")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--out", default=os.path.join("profiles", "r9_tree_verify.jsonl"))
    args = ap.parse_args()
    gpu = card()
    cfg_full = synth.model_config("m7")
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    starts = positions_for(args.steps, args.ctx - N_MAX + 1)
    rng = np.random.default_rng(1)
    toks = [int(t) for t in rng.integers(3, cfg["vocab_size"], N_MAX)]
    lines = []

    def emit(rec):
        rec = {"gpu": gpu, "shape": "m7", **rec}
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    for wname in args.formats.split(","):
        tensors = list(synth.iter_tensors(cfg_full, T.parse(wname), 0, std=0.02))
        m = Model.from_tensors(cfg, tensors).cuda(max_seqs=N_MAX)
        t_plain = timed(lambda k: m.forward_argmax(toks[0], starts[k]), args.steps)
        emit({"wtype": wname, "what": "plain greedy step (batched handle, slot 0)", "step_ms": t_plain * 1e3})
        for n in range(2, N_MAX + 1):
            t_chain = timed(lambda k: m.forward_tree_argmax(0, toks[:n], chain(n), starts[k]), args.steps)
            t_bushy = timed(lambda k: m.forward_tree_argmax(0, toks[:n], bushy(n), starts[k]), args.steps)
            t_span = timed(lambda k: m.forward_spans_argmax([0] * n, toks[:n], list(range(starts[k], starts[k] + n))), args.steps)
            emit({"wtype": wname, "what": "tree", "nodes": n, "chain_ms": t_chain * 1e3, "bushy_ms": t_bushy * 1e3,
                  "bushy_branches": 2 if n <= 5 else 3, "span_ms": t_span * 1e3,
                  "bushy_minus_span_us": (t_bushy - t_span) * 1e6, "chain_minus_span_us": (t_chain - t_span) * 1e6})
        nodes = [0, 2, 3, 4, 5, 6, 7]                   # 7 rows, 6 of them moved
        t_acc = timed(lambda k: (m.tree_accept(0, starts[k % args.steps], nodes), m.sync()), args.steps * 4)
        t_sync = timed(lambda k: m.sync(), args.steps * 4)
        emit({"wtype": wname, "what": "tree_accept", "rows": len(nodes), "moved": 6, "accept_and_sync_us": t_acc * 1e6,
              "sync_alone_us": t_sync * 1e6, "accept_us": (t_acc - t_sync) * 1e6})
        emit({"wtype": wname, "what": "parity", "position": args.ctx - N_MAX - 100, "nodes": N_MAX, "branches": 2,
              "tree_bit_identical_to_plain_steps": parity(m, cfg, toks, args.ctx - N_MAX - 100)})
        m.close()
        if args.compare_lib and wname == "q8_0":
            compare(args, cfg, tensors, toks, starts, emit)
        del tensors
    for r in lines:
        r["timing"] = f"host clock around {args.steps} synchronous calls after 4 warm-up calls"
        r["positions"] = f"start positions spread over [0, {args.ctx - N_MAX}] with bench.positions_for"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


def compare(args, cfg, tensors, toks, starts, emit):
    """spans and batched steps at n = 2, 4, 8 on this tree's library and on --compare-lib, in one process, alternating"""
    libs = {"this": capi.lib(), "other": load_lib(args.compare_lib)}
    models = {}
    for name, L in libs.items():
        capi._LIB = L
        models[name] = Model.from_tensors(cfg, tensors).cuda(max_seqs=N_MAX)
    res = {(name, what, n): [] for name in libs for what in ("spans", "batch") for n in (2, 4, 8)}
    for r in range(args.rounds):
        for name in (("this", "other") if r % 2 == 0 else ("other", "this")):
            capi._LIB = libs[name]
            m = models[name]
            for n in (2, 4, 8):
                res[(name, "spans", n)].append(timed(lambda k: m.forward_spans_argmax([0] * n, toks[:n], list(range(starts[k], starts[k] + n))), args.steps) * 1e3)
                res[(name, "batch", n)].append(timed(lambda k: m.forward_batch_argmax(list(range(n)), toks[:n], [starts[k]] * n), args.steps) * 1e3)
    for name in libs:
        capi._LIB = libs[name]
        models[name].close()
    capi._LIB = libs["this"]
    for what in ("spans", "batch"):
        for n in (2, 4, 8):
            a, b = res[("this", what, n)], res[("other", what, n)]
            emit({"wtype": "q8_0", "what": f"compare {what}", "n": n, "this_ms": a, "other_ms": b, "other_lib": args.compare_lib,
                  "this_mean_ms": float(np.mean(a)), "other_mean_ms": float(np.mean(b)),
                  "this_spread_ms": float(max(a) - min(a)), "other_spread_ms": float(max(b) - min(b)),
                  "diff_pct": float(100 * (np.mean(a) / np.mean(b) - 1)), "rounds": args.rounds, "order": "alternating, this first in even rounds"})


if __name__ == "__main__":
    main()
