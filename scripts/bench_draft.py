"""Drafting by a model on one GPU: the greedy chain (`xalm_cuda_forward_greedy`) of a TinyLlama-1.1B-shaped draft, and one
speculative round of `xalm_main -m completion -s k -D draft` with a Mistral-7B-shaped target.  Synthetic weights throughout.

(a) Chain against host loop.  d1 in each draft format on a plain batch-1 handle, its cache hydrated by prefill over the whole
    4096-token context.  For k = 1, 2, 4, 8: one `forward_greedy(n_in = 1, n_out = k)` call (one synchronise) against k
    `forward_argmax` calls (k synchronises), both starting at positions spread over [0, 4096 - k] with bench.positions_for.
    Reported as ms per drafted token.
(b) Round cost.  The target (m7, --target format) on the batched handle `-s 7` makes (max_seqs = 8); the draft (d1, --round-draft
    format).  A round at position P is the chain of k drafts (n_in = 1) and the span of k + 1 entries that verifies them, alternated
    as the CLI runs them; the components are also timed alone.  Against the batch-1 handle's plain greedy step (the handle bench.py
    makes), a round that accepts a drafts yields a + 1 tokens, so it breaks even at a = round / step - 1 accepted drafts.

Every timed call ends in a device synchronise, so each time is a host clock around `steps` calls after 4 warm-up calls.  Parity:
each chain's tokens equal the host loop's at the same positions (the loop runs second and rewrites the same rows).  The card
name and power limit are read in the same run.

    python scripts/bench_draft.py [--draft-formats q8_0,q4_0] [--target q8_0] [--round-draft q4_0] [--steps 64] [--out ...]
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
from xalm_b200.model import Model  # noqa: E402

CHAIN_K = [1, 2, 4, 8]
ROUND_K = [1, 2, 4, 7]       # -s k verifies k drafts plus the last token: at most 8 entries


def timed(fn, steps):
    """seconds per call of fn(i), i = 0 .. steps-1, after 4 warm-up calls (graph capture); every call ends in a synchronise"""
    for i in range(4):
        fn(i)
    t0 = time.perf_counter()
    for i in range(steps):
        fn(i)
    return (time.perf_counter() - t0) / steps


def shape_cfg(shape, ctx):
    full = synth.model_config(shape)
    return full, X.parse_config(synth.metadata_strings(full), ctx)


def load(shape, wname, ctx, **cuda_kw):
    full, cfg = shape_cfg(shape, ctx)
    return cfg, Model.from_tensors(cfg, synth.iter_tensors(full, T.parse(wname), 0, std=0.02)).cuda(release_host=True, **cuda_kw)


def hydrate(m, cfg, ctx):
    m.prefill(np.random.default_rng(2).integers(3, cfg["vocab_size"], ctx).astype(np.int32), 0, 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draft-formats", default="q8_0,q4_0")
    ap.add_argument("--target", default="q8_0")
    ap.add_argument("--round-draft", default="q4_0")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join("profiles", "r8_draft_model.jsonl"))
    args = ap.parse_args()
    gpu = card()
    lines = []

    def emit(rec):
        rec = {"gpu": gpu, **rec}
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    tok = 1000
    # (a) chain against host loop
    for wname in args.draft_formats.split(","):
        cfg, d = load("d1", wname, args.ctx)
        hydrate(d, cfg, args.ctx)
        for k in CHAIN_K:
            starts = positions_for(args.steps, args.ctx - k + 1)
            chains, loops = {}, {}

            def chain(i):
                chains[i] = d.forward_greedy([tok], starts[i], k)

            def loop(i):
                t, out = tok, []
                for j in range(k):
                    t = d.forward_argmax(t, starts[i] + j)
                    out.append(t)
                loops[i] = out

            t_chain = timed(chain, args.steps)
            t_loop = timed(loop, args.steps)
            emit({"shape": "d1", "wtype": wname, "what": "chain vs loop", "k": k, "chain_call_ms": t_chain * 1e3,
                  "loop_ms": t_loop * 1e3, "chain_ms_per_token": t_chain * 1e3 / k, "loop_ms_per_token": t_loop * 1e3 / k,
                  "chain_saves_pct": 100.0 * (1 - t_chain / t_loop), "tokens_identical": chains == loops})
        d.close()

    # (b) round cost: chain of k (draft) + span of k + 1 (target)
    tcfg, solo = load("m7", args.target, args.ctx)
    plain = positions_for(args.steps, args.ctx)
    t_step = timed(lambda i: solo.forward_argmax(tok, plain[i]), args.steps)
    solo.close()
    emit({"shape": "m7", "wtype": args.target, "what": "target batch-1 step", "step_ms": t_step * 1e3, "tok_s": 1 / t_step})
    _, tgt = load("m7", args.target, args.ctx, max_seqs=8)
    dcfg, d = load("d1", args.round_draft, args.ctx)
    hydrate(d, dcfg, args.ctx)
    for k in ROUND_K:
        starts = positions_for(args.steps, args.ctx - k)                  # positions P .. P + k stay inside the window
        span = lambda i: tgt.forward_spans_argmax([0] * (k + 1), [tok] * (k + 1), list(range(starts[i], starts[i] + k + 1)))
        chain = lambda i: d.forward_greedy([tok], starts[i], k)
        t_chain = timed(chain, args.steps)
        t_span = timed(span, args.steps)
        t_round = timed(lambda i: (chain(i), span(i)), args.steps)
        emit({"shape": "m7+d1", "wtype": f"{args.target}+{args.round_draft}", "what": "round", "k": k, "chain_ms": t_chain * 1e3,
              "span_ms": t_span * 1e3, "round_ms": t_round * 1e3, "target_step_ms": t_step * 1e3,
              "break_even_accepted_per_round": t_round / t_step - 1, "tok_s_all_accepted": (k + 1) / t_round,
              "tok_s_none_accepted": 1 / t_round})
    d.close()
    tgt.close()
    for r in lines:
        r["timing"] = f"host clock around {args.steps} synchronous calls after 4 warm-up calls"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
