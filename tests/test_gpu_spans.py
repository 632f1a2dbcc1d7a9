"""Spans (xalm_cuda_forward_spans): several consecutive positions of one sequence in one step, as speculative decoding verifies
drafted tokens.  Each entry's logits and the KV rows it writes must be bit-identical to decoding the same tokens one step at a
time on a batch-1 handle with the tensor-core matvec; rows written for rejected drafts must never be read."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_batch import FORMATS, PROMPT, PROMPTS, argmax, bits, check_kv, hydrate, kv_state, oracle_tokens, solo_handle, solo_run, tensors_of
from xalm_b200 import capi
from xalm_b200.model import InferenceState, Model

pytestmark = pytest.mark.gpu

LENGTHS = [2, 3, 4, 5, 6, 7, 8]


def fed_tokens(prompt, toks):
    """the token decoded at each step of a solo run: the prompt's last token, then every greedy token but the last"""
    return [prompt[-1]] + toks[:-1]


def verify_spans(b, slot, seq, lgs, p0, lengths):
    """feed seq (the solo run's own tokens, from position p0) as spans of the given lengths; every entry must equal the solo
    logits at its position.  Returns the greedy tokens of every entry."""
    k, out = 0, []
    for L in lengths:
        L = min(L, len(seq) - k)
        if L <= 0:
            break
        lg = b.forward_spans([slot] * L, seq[k:k + L], list(range(p0 + k, p0 + k + L)))
        for j in range(L):
            assert np.array_equal(bits(lg[j]), bits(lgs[k + j])), f"span of {L} at position {p0 + k}: entry {j}"
        out += [argmax(r) for r in lg]
        k += L
    assert k == len(seq)
    return out


@pytest.mark.parametrize("shape", ["tiny", "small"])
@pytest.mark.parametrize("wtype", FORMATS)
def test_accepted_spans_are_bit_identical_to_solo(shape, wtype):
    steps = sum(LENGTHS)
    cfg, tensors = tensors_of(shape, wtype, 2, 0.06, 0)
    solo = solo_handle(cfg, tensors)
    lgs, toks, kv = solo_run(solo, cfg, PROMPT, steps)
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    hydrate(b, 3, PROMPT)
    got = verify_spans(b, 3, fed_tokens(PROMPT, toks), lgs, len(PROMPT) - 1, LENGTHS)
    assert got == toks
    check_kv(b, cfg, 3, kv, len(PROMPT) - 1 + steps)
    b.close()
    if shape == "tiny":
        assert got == oracle_tokens(cfg, tensors, PROMPT, steps), f"{wtype}: span tokens differ from the oracle"


@pytest.mark.parametrize("graph,pdl", [(1, 1), (0, 0), (0, 1)])
def test_rejected_drafts_are_rewritten_cleanly(graph, pdl):
    """Each step verifies a span whose draft is wrong from index j on: entries 0..j still match solo; decoding goes on from the
    accepted prefix, so the next span re-verifies, with the right tokens, positions that already hold rows of wrong drafts."""
    steps = 40
    cfg, tensors = tensors_of("tiny", "q4_0", 3, 0.06, 0)
    solo = solo_handle(cfg, tensors)
    lgs, toks, kv = solo_run(solo, cfg, PROMPT, steps + 8)
    solo.close()
    seq, p0, V = fed_tokens(PROMPT, toks), len(PROMPT) - 1, cfg["vocab_size"]
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    hydrate(b, 0, PROMPT)
    rng = np.random.default_rng(11)
    capi.tune("graph", graph); capi.tune("pdl", pdl)
    try:
        k, wrote = 0, 0
        while k < steps:
            L = int(rng.integers(2, 9))
            j = int(rng.integers(0, L - 1))                      # draft index of the first wrong token: entry j + 1
            span = list(seq[k:k + L])
            for e in range(j + 1, L):
                span[e] = int((span[e] + 1 + rng.integers(0, V - 1)) % V)
                assert span[e] != seq[k + e]
            lg = b.forward_spans([0] * L, span, list(range(p0 + k, p0 + k + L)))
            for e in range(j + 1):
                assert np.array_equal(bits(lg[e]), bits(lgs[k + e])), f"span at {p0 + k}, wrong from entry {j + 1}: entry {e}"
            assert [argmax(r) for r in lg[:j + 1]] == toks[k:k + j + 1]
            wrote = max(wrote, k + L)
            k += j + 1                                          # accepted: entries 0..j-1's drafts, plus entry j's own token
        assert wrote > k                                        # rows of rejected drafts lie beyond the accepted prefix
        # re-verify everything past the accepted prefix with the right tokens, then plain steps through the end of the run
        verify_spans(b, 0, seq[k:wrote], lgs[k:wrote], p0 + k, LENGTHS * 4)
        for q in range(wrote, steps + 8):
            lg = b.forward_batch([0], [seq[q]], [p0 + q])
            assert np.array_equal(bits(lg[0]), bits(lgs[q])), f"plain step at {p0 + q}"
    finally:
        capi.tune("graph", 1); capi.tune("pdl", 1)
    check_kv(b, cfg, 0, kv, p0 + steps + 8)
    b.close()


def test_mixed_step_spans_and_a_slot_past_its_window():
    """One call holds two slots with spans (3 and 2 entries, interleaved) and one single-entry slot past its window with the
    attention sinks active; each matches its own solo run."""
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 32)
    assert cfg["max_seq_len"] == 32
    pa, pb, pc = [1, 200, 31], PROMPTS[4], [1] + list(range(100, 133))     # pc: 34 tokens, already past the window
    steps = 8
    solo = solo_handle(cfg, tensors)
    ra = solo_run(solo, cfg, pa, 3 * steps)
    rb = solo_run(solo, cfg, pb, 2 * steps)
    rc = solo_run(solo, cfg, pc, steps)
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    for s, p in ((6, pa), (1, pb), (4, pc)):
        hydrate(b, s, p)
    sa, sb, sc = fed_tokens(pa, ra[1]), fed_tokens(pb, rb[1]), fed_tokens(pc, rc[1])
    for k in range(steps):
        a0, b0 = len(pa) - 1 + 3 * k, len(pb) - 1 + 2 * k
        seqs = [6, 1, 6, 4, 1, 6]
        toks = [sa[3 * k], sb[2 * k], sa[3 * k + 1], sc[k], sb[2 * k + 1], sa[3 * k + 2]]
        pos = [a0, b0, a0 + 1, len(pc) - 1 + k, b0 + 1, a0 + 2]
        lg = b.forward_spans(seqs, toks, pos)
        want = [ra[0][3 * k], rb[0][2 * k], ra[0][3 * k + 1], rc[0][k], rb[0][2 * k + 1], ra[0][3 * k + 2]]
        for i in range(6):
            assert np.array_equal(bits(lg[i]), bits(want[i])), f"step {k}: entry {i} (slot {seqs[i]}, pos {pos[i]})"
    check_kv(b, cfg, 6, ra[2], len(pa) - 1 + 3 * steps)
    check_kv(b, cfg, 1, rb[2], len(pb) - 1 + 2 * steps)
    check_kv(b, cfg, 4, rc[2], len(pc) - 1 + steps)
    b.close()


def test_run_to_run_bit_identical():
    cfg, tensors = tensors_of("small", "q5_1", 4, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    runs = []
    for _ in range(2):
        hydrate(b, 2, PROMPT)
        hydrate(b, 5, PROMPTS[2])
        ta, tb, pa, pb, lgs = PROMPT[-1], PROMPTS[2][-1], len(PROMPT) - 1, len(PROMPTS[2]) - 1, []
        for L in LENGTHS[:-1]:                                 # with slot 5's entry: n <= max_seqs
            # draft = the previous greedy token repeated: some entries are accepted, the rest are rewritten by the next span
            lg = b.forward_spans([2] * L + [5], [ta] * L + [tb], list(range(pa, pa + L)) + [pb])
            lgs.append(bits(lg).copy())
            nxt = [argmax(r) for r in lg]
            a = 0
            while a < L - 1 and nxt[a] == ta:
                a += 1
            ta, pa, tb, pb = nxt[a], pa + a + 1, nxt[L], pb + 1
        kv = []
        for s in (2, 5):
            b.select_seq(s)
            kv.append([x.copy() for x in kv_state(b, cfg, pa + 8 if s == 2 else pb)])
        b.select_seq(0)
        runs.append((lgs, kv))
    assert all(np.array_equal(x, y) for x, y in zip(runs[0][0], runs[1][0]))
    assert all(np.array_equal(x, y) for s in range(2) for x, y in zip(runs[0][1][s], runs[1][1][s]))
    b.close()


def test_refusals_leave_every_cache_untouched():
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 0)
    W, V = cfg["max_seq_len"], cfg["vocab_size"]
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    for s in range(4):
        hydrate(b, s, PROMPTS[s])
    snap = []
    for s in range(4):
        b.select_seq(s)
        snap.append([b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)])
    b.select_seq(0)
    cases = [([0, 0], [1, 2], [3, 5]),                    # not consecutive
             ([0, 0], [1, 2], [3, 3]),                    # repeated
             ([0, 0], [1, 2], [4, 3]),                    # decreasing
             ([1, 0, 1, 1], [1] * 4, [3, 3, 4, 6]),       # a gap after an interleaved entry
             ([0, 0], [1, 2], [W - 1, W]),                # a span reaching max_seq_len
             ([2, 2, 2], [1] * 3, [W + 4, W + 5, W + 6]), # a span past the window
             ([0, 1, 2, 3, 0], [1] * 5, [3, 3, 3, 3, 4]), # n > max_seqs
             ([4], [1], [3]),                             # slot out of range
             ([0, 0], [1, V], [3, 4]),                    # token out of range
             ([0, 0], [1, 2], [-1, 0])]                   # negative position
    for seqs, toks, pos in cases:
        for call in (b.forward_spans, b.forward_spans_argmax):
            with pytest.raises(capi.XalmError) as e:
                call(seqs, toks, pos)
            assert e.value.status == 1, (seqs, toks, pos)
    L = capi.lib()
    z, o = (C.c_int * 1)(0), (C.c_int * 1)(0)
    assert L.xalm_cuda_forward_spans(b._h, 0, z, z, z, None) == 1
    for args in ((None, z, z), (z, None, z), (z, z, None)):
        assert L.xalm_cuda_forward_spans(b._h, 1, *args, None) == 1
        assert L.xalm_cuda_forward_spans_argmax(b._h, 1, *args, o) == 1
    assert L.xalm_cuda_forward_spans_argmax(b._h, 1, z, z, z, None) == 1
    with pytest.raises(capi.XalmError) as e:                 # forward_batch keeps refusing a slot named twice
        b.forward_batch([0, 0], [1, 2], [3, 4])
    assert e.value.status == 1
    for s in range(4):
        b.select_seq(s)
        now = [b.read_kv(l, w) for l in range(cfg["n_layers"]) for w in (0, 1)]
        assert all(np.array_equal(x, y) for x, y in zip(now, snap[s])), f"slot {s} changed by a refused call"
    b.close()
    solo = solo_handle(cfg, tensors)                         # a handle without set_batch
    for call in (solo.forward_spans, solo.forward_spans_argmax):
        with pytest.raises(capi.XalmError) as e:
            call([0, 0], [1, 2], [0, 1])
        assert e.value.status == 4
    solo.close()


def test_spans_argmax_matches_host_sampler():
    cfg, tensors = tensors_of("tiny", "q5_0", 21, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    hydrate(b, 1, PROMPT)
    tok, pos = PROMPT[-1], len(PROMPT) - 1
    for _ in range(6):
        span = [tok, 7, 9, 11]
        lg = b.forward_spans([1] * 4, span, list(range(pos, pos + 4)))
        dev = b.forward_spans_argmax([1] * 4, span, list(range(pos, pos + 4)))  # same inputs: the rows are rewritten unchanged
        assert dev == [argmax(r) for r in lg]
        tok, pos = dev[0], pos + 1
    b.close()


def test_full_size_mistral_7b_q8_0_spans_of_eight():
    """Mistral-7B shape, q8_0: an 8-entry span at position 100 and at position 4000 (where the attention's early fetch covers
    only part of the rows the span reads), bit-identical to 8 solo steps."""
    cfg, tensors = tensors_of("m7", "q8_0", 0, 0.02, 0)
    rng = np.random.default_rng(5)
    ctx = [1] + [int(v) for v in rng.integers(3, cfg["vocab_size"], 4000)]
    solo = solo_handle(cfg, tensors)
    refs = {}
    st = InferenceState(cfg)
    for P in (100, 4000):
        solo.prefill(ctx[:P], 0, 0)
        tok, lgs, fed = ctx[P], [], []
        for q in range(8):
            fed.append(tok)
            solo.forward(st, tok, P + q, 1)
            lgs.append(st.logits().copy())
            tok = argmax(lgs[-1])
        refs[P] = (fed, lgs)
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    del tensors
    for P in (100, 4000):
        b.select_seq(0)
        b.prefill(ctx[:P], 0, 0)
        fed, lgs = refs[P]
        lg = b.forward_spans([0] * 8, fed, list(range(P, P + 8)))
        for j in range(8):
            assert np.array_equal(bits(lg[j]), bits(lgs[j])), f"span at {P}: entry {j}"
    b.close()
