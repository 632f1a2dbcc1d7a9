"""Spans on one GPU (speculative decoding's verify pass): Mistral-7B shape (synthetic weights), one batched handle (max_seqs = 8).

For L = 1 .. 8 entries on one slot, one JSON line per (format, L): the time of one greedy span step
(`xalm_cuda_forward_spans_argmax`, which is what `xalm_main -m completion -s k` calls), tok/s when every draft is accepted
(L / step) and when none is (1 / step), and the break-even tokens per pass against the batch-1 handle's greedy step
(`xalm_cuda_forward_argmax` on a handle made as bench.py makes it), timed in the same run.  At L = 2 / 4 / 8 the same step with L
independent sequences (`forward_batch_argmax`, one entry per slot, the same positions) is timed too: the span's entries read the
same K/V rows, the independent sequences each read their own.  Every call is synchronous, so each step time is a host clock
around `steps` calls that each end in a device synchronise, the same for every variant.  Span start positions are spread over
[0, 4096 - 8] with bench.positions_for.  Parity: an 8-entry span fed 8 plain steps' own greedy tokens (batch-1 tensor-core
kernel, same slot, same positions) gives bit-identical logits.  The card name and power limit are read in the same run.

    python scripts/bench_spec.py [--formats q8_0,q4_0] [--steps 64] [--out profiles/r7_spec_decode.jsonl]
"""
import argparse
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
from xalm_b200 import synth  # noqa: E402
from xalm_b200 import types as T  # noqa: E402
from xalm_b200 import xalm_file as X  # noqa: E402
from xalm_b200.model import InferenceState, Model  # noqa: E402

MAX_SPAN = 8


def timed(fn, steps):
    """seconds per call of fn(k), k = 0 .. steps-1, after 4 warm-up calls (graph capture); every call ends in a synchronise"""
    for k in range(4):
        fn(k)
    t0 = time.perf_counter()
    for k in range(steps):
        fn(k)
    return (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--formats", default="q8_0,q4_0")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join("profiles", "r7_spec_decode.jsonl"))
    args = ap.parse_args()
    gpu = card()
    cfg_full = synth.model_config("m7")
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    starts = positions_for(args.steps, args.ctx - MAX_SPAN + 1)          # span starts over [0, ctx - 8]
    rng = np.random.default_rng(1)
    toks = [int(t) for t in rng.integers(3, cfg["vocab_size"], MAX_SPAN)]
    lines = []
    for wname in args.formats.split(","):
        wtype = T.parse(wname)
        # the batch-1 handle bench.py measures (default kernels: dp4a for q8_0, tensor cores for q4_0)
        solo = Model.from_tensors(cfg, synth.iter_tensors(cfg_full, wtype, 0, std=0.02)).cuda(release_host=True)
        t_solo = timed(lambda k: solo.forward_argmax(toks[0], starts[k]), args.steps)
        solo.close()
        m = Model.from_tensors(cfg, synth.iter_tensors(cfg_full, wtype, 0, std=0.02)).cuda(max_seqs=MAX_SPAN, release_host=True)
        t_plain = timed(lambda k: m.forward_argmax(toks[0], starts[k]), args.steps)   # -s's no-draft step: batched handle, slot 0
        rec = {"gpu": gpu, "shape": "m7", "wtype": wname, "what": "batch-1 greedy step", "batch1_handle_ms": t_solo * 1e3,
               "batch1_handle_tok_s": 1 / t_solo, "batched_handle_plain_ms": t_plain * 1e3, "batched_handle_plain_tok_s": 1 / t_plain}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        for L in range(1, MAX_SPAN + 1):
            t_span = timed(lambda k: m.forward_spans_argmax([0] * L, toks[:L], list(range(starts[k], starts[k] + L))), args.steps)
            rec = {"gpu": gpu, "shape": "m7", "wtype": wname, "what": "span", "entries": L, "step_ms": t_span * 1e3,
                   "tok_s_all_accepted": L / t_span, "tok_s_none_accepted": 1 / t_span,
                   "break_even_tokens_per_pass": t_span / t_solo, "vs_batch1_handle_ms": t_solo * 1e3}
            if L in (2, 4, 8):
                t_ind = timed(lambda k: m.forward_batch_argmax(list(range(L)), toks[:L], [starts[k] + i for i in range(L)]), args.steps)
                rec["independent_seqs_ms"] = t_ind * 1e3
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        # parity: 8 plain greedy steps on slot 1 (batch-1 tensor-core kernel) against one 8-entry span of the same tokens
        st = InferenceState(cfg)
        P = args.ctx - MAX_SPAN - 100
        m.select_seq(1)
        fed, ref, t = [], [], toks[0]
        for q in range(MAX_SPAN):
            fed.append(t)
            m.forward(st, t, P + q, 1)
            ref.append(st.logits().copy())
            t = int(np.argmax(ref[-1]))
        m.select_seq(0)
        lg = m.forward_spans([1] * MAX_SPAN, fed, list(range(P, P + MAX_SPAN)))
        parity = all(np.array_equal(lg[j].view(np.uint32), ref[j].view(np.uint32)) for j in range(MAX_SPAN))
        rec = {"gpu": gpu, "shape": "m7", "wtype": wname, "what": "parity", "position": P, "entries": MAX_SPAN,
               "span_bit_identical_to_plain_steps": parity}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        m.close()
    for r in lines:
        r["timing"] = f"host clock around {args.steps} synchronous greedy calls after 4 warm-up calls"
        r["positions"] = f"span starts spread over [0, {args.ctx - MAX_SPAN}] with bench.positions_for"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
