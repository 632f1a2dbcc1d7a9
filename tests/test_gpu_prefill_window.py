"""Batched prefill past the context window (xalm_cuda_prefill_window): the KV cache is a ring of max_seq_len - 2 slots after
two attention sinks, and every position attends to the sinks plus the max_seq_len - 2 latest positions.

Checked against the CPU oracle run token by token (logits, KV cache, perplexity, the CLI) and against the token-at-a-time
decode kernels (the sink keys, which both re-rotate through fp16 once per position, must agree bit for bit).
"""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import oracle
from xalm_b200 import build, capi
from xalm_b200.model import InferenceState, Sampler

from gpu_util import LOGIT_TOL, synth_pair

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _chunks(S, total):
    """Window chunk sizes covering `total` positions: mixed sizes, including 1 and the largest allowed (S = W - 2)."""
    pattern = [1, S, 17, S - 3, 5, S, 2]
    out, left, i = [], total, 0
    while left > 0:
        c = min(pattern[i % len(pattern)], left)
        out.append(c)
        left -= c
        i += 1
    return out


def _kv(gm, config):
    return [[gm.read_kv(l, w).copy() for w in (0, 1)] for l in range(config["n_layers"])]


def _run(gm, tokens, W, chunks, targets=None):
    """Linear prefill of [0, W), then window chunks; every position's logits (and target probabilities)."""
    tg = None if targets is None else targets[:W]
    r = gm.prefill(tokens[:W], 0, want_logits=2, targets=tg)
    lgs, prs = ([r[0]], [r[1]]) if targets is not None else ([r], [])
    pos = W
    for c in chunks:
        tg = None if targets is None else targets[pos:pos + c]
        r = gm.prefill_window(tokens[pos:pos + c], pos, want_logits=2, targets=tg)
        if targets is not None:
            lgs.append(r[0]); prs.append(r[1])
        else:
            lgs.append(r)
        pos += c
    return np.concatenate(lgs), (np.concatenate(prs) if prs else None)


CASES = [("f16", "tiny", 48), ("q8_0", "tiny", 48), ("q4_0", "tiny", 48),   # head_dim 64: the mma.sync attention
         ("q8_0", "small", 256), ("f16", "small", 256)]                      # head_dim 128, GQA 8:2: the tcgen05 attention


@pytest.mark.parametrize("wtype,shape,W", CASES)
@pytest.mark.parametrize("split", [1, 2, 3])
def test_window_logits_and_cache_match_oracle(wtype, shape, W, split):
    capi.tune("prefill_split", split)
    try:
        over = dict(n_layers=2) if shape == "small" else {}
        config, om, gm = synth_pair(shape, wtype, seed=7, context=W, std=0.06 if shape == "tiny" else 0.03, **over)
        assert config["max_seq_len"] == W
        S = W - 2
        chunks = _chunks(S, 3 * W + 5)
        n = W + sum(chunks)
        tokens = np.random.default_rng(1).integers(3, config["vocab_size"], size=n).astype(np.int32)
        ref = np.stack([om.forward(int(t), pos, 1).copy() for pos, t in enumerate(tokens)])
        got, _ = _run(gm, tokens, W, chunks)
        diff = float(np.max(np.abs(got - ref)))
        # split 3 (the precise default): 1e-3 as in test_prefill_logits_match_oracle, except f16 on the head_dim-128 shape, measured
        # at 1.6e-3 from the oracle (1.3e-3 from the decode kernels) over these ~1000 positions on a B200; the linear prefill is held
        # to 1e-2 at such lengths (test_prefill_4096_tokens_vs_oracle)
        tol = LOGIT_TOL if split < 3 else (2e-3 if (wtype, shape) == ("f16", "small") else 1e-3)
        assert diff <= tol, f"{wtype}/{shape}/split {split}: window prefill logits differ from the oracle by {diff}"
        kvd = config["n_kv_heads"] * config["head_dim"]
        for layer in range(config["n_layers"]):
            for which in (0, 1):
                a = gm.read_kv(layer, which).view(np.float16).astype(np.float32)[: W * kvd].reshape(W, kvd)
                b = om.kv(layer, which).view(np.float16).astype(np.float32)[: W * kvd].reshape(W, kvd)
                # the data slots; the sinks are checked bit for bit against the token loop in test_sink_keys_bit_identical_to_token_loop
                # (against the oracle they carry hundreds of fp16 re-roundings of slightly different starting values)
                assert np.max(np.abs(a[2:] - b[2:])) <= 1e-2 * max(1.0, float(np.abs(b[2:]).max()))
        gm.close(); om.close()
    finally:
        capi.tune("prefill_split", 3)


@pytest.mark.parametrize("shape,W", [("tiny", 48), ("small", 256)])
def test_sink_keys_bit_identical_to_token_loop(shape, W):
    over = dict(n_layers=2) if shape == "small" else {}
    std = 0.06 if shape == "tiny" else 0.03
    config, om, gm = synth_pair(shape, "q8_0", seed=5, context=W, std=std, **over)
    _, om2, ref = synth_pair(shape, "q8_0", seed=5, context=W, std=std, **over)
    S = W - 2
    chunks = [1, S, 9, S - 1]
    n = W + sum(chunks)
    tokens = np.random.default_rng(2).integers(3, config["vocab_size"], size=n).astype(np.int32)
    _run(gm, tokens, W, chunks)
    ref.prefill(tokens[:W], 0, want_logits=0)
    st = InferenceState(config)
    for pos in range(W, n):
        ref.forward(st, int(tokens[pos]), pos, 0)
    kvd = config["n_kv_heads"] * config["head_dim"]
    for layer in range(config["n_layers"]):
        for which in (0, 1):
            a = gm.read_kv(layer, which)[: 2 * kvd]
            b = ref.read_kv(layer, which)[: 2 * kvd]
            assert np.array_equal(a, b), f"layer {layer} {'kv'[which]}: sink rows differ from the token loop"
    gm.close(); om.close(); ref.close(); om2.close()


def test_window_perplexity_probabilities():
    config, om, gm = synth_pair("tiny", "q8_0", seed=12, context=48, std=0.06)
    W = 48
    N = 4 * W + 3
    toks = np.random.default_rng(4).integers(3, config["vocab_size"], size=N + 1).astype(np.int32)
    ref_lp = np.array([np.log(oracle.sample_prob(om.forward(int(toks[p]), p, 1), int(toks[p + 1]))) for p in range(N)])
    _, probs = _run(gm, toks[:N], W, _chunks(W - 2, N - W), targets=toks[1:])
    lp = np.log(probs)
    assert np.max(np.abs(lp - ref_lp)) <= 2e-2
    ppl_ref, ppl = np.exp(-np.mean(ref_lp)), np.exp(-np.mean(lp))
    assert abs(ppl - ppl_ref) <= 2e-3 * ppl_ref
    gm.close(); om.close()


def test_decode_continues_after_window_prefill():
    config, om, gm = synth_pair("tiny", "q8_0", seed=9, context=48, std=0.06)
    W = 48
    prompt = np.random.default_rng(3).integers(3, config["vocab_size"], size=W + 70).astype(np.int32)
    for pos, tok in enumerate(prompt):
        lg_o = om.forward(int(tok), pos, 1 if pos + 1 == len(prompt) else 0)
    gm.prefill(prompt[:W], 0, want_logits=0)
    gm.prefill_window(prompt[W:W + 46], W, want_logits=0)
    lg = gm.prefill_window(prompt[W + 46:], W + 46, want_logits=1)
    assert np.max(np.abs(lg - lg_o)) <= LOGIT_TOL
    state, sampler = InferenceState(config), Sampler(config)
    state.logits()[:] = lg
    otoks, gtoks = [], []
    for i in range(16):
        to, tg = oracle.sample_argmax(lg_o), sampler.sample_argmax(state)
        otoks.append(to); gtoks.append(tg)
        pos = len(prompt) + i
        lg_o = om.forward(to, pos, 1)
        gm.forward(state, tg, pos, 1)
        assert np.max(np.abs(state.logits() - lg_o)) <= LOGIT_TOL
    assert otoks == gtoks
    gm.close(); om.close()


@pytest.mark.parametrize("shape,W", [("tiny", 48), ("small", 256)])
def test_chunking_and_determinism(shape, W):
    over = dict(n_layers=2) if shape == "small" else {}
    std = 0.06 if shape == "tiny" else 0.03
    handles = [synth_pair(shape, "f16", seed=6, context=W, std=std, **over) for _ in range(3)]
    config = handles[0][0]
    S = W - 2
    tokens = np.random.default_rng(8).integers(3, config["vocab_size"], size=W + S).astype(np.int32)
    outs = []
    for i, (_, _, gm) in enumerate(handles):
        gm.prefill(tokens[:W], 0, want_logits=0)
        if i < 2:   # one call of the largest size, twice on identical handles
            outs.append(gm.prefill_window(tokens[W:], W, want_logits=2))
        else:       # the same positions in three calls
            cuts = [W, W + 7, W + S - 5, W + S]
            outs.append(np.concatenate([gm.prefill_window(tokens[a:b], a, want_logits=2) for a, b in zip(cuts, cuts[1:])]))
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32)), "two runs of the same call differ"
    assert np.max(np.abs(outs[0] - outs[2])) <= 1e-3
    kvd = config["n_kv_heads"] * config["head_dim"]
    for layer in range(config["n_layers"]):
        assert np.array_equal(handles[0][2].read_kv(layer, 0)[: 2 * kvd], handles[2][2].read_kv(layer, 0)[: 2 * kvd])
    for _, om, gm in handles:
        gm.close(); om.close()


def test_refusals_leave_the_cache_untouched():
    config, om, gm = synth_pair("tiny", "q8_0", seed=13, context=48, std=0.06)
    W, V = 48, config["vocab_size"]
    tokens = np.random.default_rng(6).integers(3, V, size=2 * W).astype(np.int32)
    gm.prefill(tokens[:W], 0, want_logits=0)
    before = _kv(gm, config)
    bad = [(tokens[:1], W - 1),                                      # inside the window: xalm_cuda_prefill's range
           (tokens[W:2 * W - 1], W),                                 # n = W - 1: would write a ring slot twice
           (np.array([5, V, 7], dtype=np.int32), W)]                 # token out of range
    for toks, pos0 in bad:
        with pytest.raises(capi.XalmError):
            gm.prefill_window(toks, pos0, want_logits=2)
        after = _kv(gm, config)
        for l in range(config["n_layers"]):
            for w in (0, 1):
                assert np.array_equal(before[l][w], after[l][w])
    with pytest.raises(capi.XalmError):                              # the linear entry point still refuses to wrap
        gm.prefill(tokens[W:W + 4], W, want_logits=0)
    gm.close(); om.close()


def _cli_oracle(path, context, enc):
    from xalm_b200 import xalm_file as X
    f = X.XalmFile(path)
    cfg = X.parse_config(f.metadata, context)
    return oracle.OracleModel(cfg, {k: (ti.type.id, f.raw(k)) for k, ti in f.tensors.items()})


def test_cli_perplexity_past_the_window():
    from xalm_b200 import xalm_file as X
    from xalm_b200.model import Tokenizer
    path = os.path.join(GOLD, "tiny_bf16.xalm")
    prompt = " ".join(["the meaning of life is in the the of a"] * 8)
    tok = Tokenizer(X.XalmFile(path))
    enc = tok.encode(prompt, True)
    assert len(enc) >= 60
    om = _cli_oracle(path, 16, enc)
    om.forward(0, 0, 1)
    s = sum(np.log(oracle.sample_prob(om.forward(enc[p], p, 1), enc[p + 1])) for p in range(len(enc) - 1))
    ppl = float(np.exp(-s / (len(enc) - 1)))
    build.build_cuda(); build.build_host()
    with tempfile.NamedTemporaryFile("w", suffix=".txt", delete=False) as fh:
        fh.write(prompt)
    try:
        r = subprocess.run([build.MAIN, path, "-m", "perplexity", "-T", "16", "-f", fh.name], capture_output=True, text=True)
    finally:
        os.unlink(fh.name)
    assert r.returncode == 0, r.stderr
    got = float([l for l in r.stdout.splitlines() if "perplexity:" in l][0].split("perplexity:")[1].split()[0])
    assert abs(got - ppl) / ppl < 2e-3, (got, ppl)


def test_cli_completion_prompt_longer_than_the_window():
    from xalm_b200 import xalm_file as X
    from xalm_b200.model import Tokenizer
    path = os.path.join(GOLD, "tiny_q8_0.xalm")
    prompt = "Q: What is the meaning of life, the universe and everything else there is? A:"
    tok = Tokenizer(X.XalmFile(path))
    enc = tok.encode(prompt, True)
    assert len(enc) > 16
    om = _cli_oracle(path, 16, enc)
    om.forward(0, 0, 1)
    for pos, t in enumerate(enc):
        lg = om.forward(t, pos, 1 if pos + 1 == len(enc) else 0)
    text = b""
    for _ in range(12):
        t = oracle.sample_argmax(lg)
        text += tok.decode_one(enc[-1], t)
        enc.append(t)
        if t in (tok.eos_id, tok.eot_id):
            break
        lg = om.forward(t, len(enc) - 1, 1)
    build.build_cuda(); build.build_host()
    r = subprocess.run([build.MAIN, path, "-d", "cuda", "-m", "completion", "-n", "12", "-T", "16", "-i", prompt], capture_output=True)
    assert r.returncode == 0, r.stderr.decode(errors="replace")
    assert text in r.stdout, (text, r.stdout[-600:])


def test_window_perplexity_large_shape():
    """A perplexity pass over 3 windows at W = 1024 on the tcgen05 attention: many key blocks below the band, multi-tile
    queries; logits at ~60 positions spread over the run plus the last 8, and the perplexity of the whole run."""
    W, n = 1024, 3072
    config, om, gm = synth_pair("small", "q8_0", seed=3, context=W, std=0.03, n_layers=2)
    toks = np.random.default_rng(17).integers(3, config["vocab_size"], size=n + 1).astype(np.int32)
    check = sorted(set(list(range(0, n, 52)) + list(range(n - 8, n)) + [W, W + 1, W + 127, W + 128, 2 * W - 2, 2 * W - 1]))
    want, probs_o = {}, np.zeros(n, np.float32)
    for pos in range(n):
        lg = om.forward(int(toks[pos]), pos, 1)
        probs_o[pos] = oracle.sample_prob(lg, int(toks[pos + 1]))
        if pos in check:
            want[pos] = lg.copy()
    S = W - 2
    lg_all, probs = _run(gm, toks[:n], W, [min(S, n - p) for p in range(W, n, S)], targets=toks[1:])
    worst = max(float(np.max(np.abs(lg_all[pos] - want[pos]))) for pos in check)
    assert worst <= LOGIT_TOL, f"window prefill logits differ from the oracle by {worst}"
    ppl_g, ppl_o = float(np.exp(-np.mean(np.log(probs)))), float(np.exp(-np.mean(np.log(probs_o))))
    assert abs(ppl_g - ppl_o) <= 1e-3 * ppl_o, (ppl_g, ppl_o)
    gm.close(); om.close()
