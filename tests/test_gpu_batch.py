"""Batched decode (xalm_cuda_set_batch / forward_batch): several sequences per pass over the weights.  Every sequence's logits
and KV cache must be bit-identical to decoding it alone on a batch-1 handle with the tensor-core matvec, whatever shares the
step, and its greedy tokens must match the oracle."""
import os

import numpy as np
import pytest

from oracle import oracle
from xalm_b200 import capi, synth
from xalm_b200 import types as T
from xalm_b200 import xalm_file as X
from xalm_b200.model import InferenceState, Model

pytestmark = pytest.mark.gpu

FORMATS = ["q8_0", "q8", "q4_0", "q4_1", "q5_0", "q5_1"]
PROMPT = [1, 84, 61, 35, 90, 107, 100, 119]
PROMPTS = [PROMPT, [1, 200, 31], [1, 7, 9, 11, 13, 17, 19, 23, 29, 31, 37, 41], [1, 400], [1, 55, 66, 77, 88],
           [1, 300, 301, 302, 303, 304, 305], [1, 9], [1, 120, 121, 122, 123, 124, 125, 126, 127, 128]]
FLT_MIN = np.float32(np.finfo(np.float32).tiny)


def argmax(lg):
    i = int(np.argmax(lg))
    return i if lg[i] > FLT_MIN else 0


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def tensors_of(shape, wtype, seed, std, context):
    c = synth.model_config(shape)
    cfg = X.parse_config(synth.metadata_strings(c), context)
    return cfg, list(synth.iter_tensors(c, T.parse(wtype), seed, std=std))


def solo_handle(cfg, tensors):
    """batch-1 handle on the tensor-core matvec for every integer format (the reference the batched path must match bit for bit)"""
    capi.tune("mma", 1)
    try:
        return Model.from_tensors(cfg, tensors).cuda()
    finally:
        capi.tune("mma", 2)


def solo_run(m, cfg, prompt, steps):
    """prompt token by token, then `steps` greedy steps: (logits per step, tokens, KV rows written) on a batch-1 handle"""
    st = InferenceState(cfg)
    for pos, tok in enumerate(prompt[:-1]):
        m.forward(st, tok, pos, 0)
    tok, pos, lgs, toks = prompt[-1], len(prompt) - 1, [], []
    for _ in range(steps):
        m.forward(st, tok, pos, 1)
        lgs.append(st.logits().copy())
        tok, pos = argmax(lgs[-1]), pos + 1
        toks.append(tok)
    return lgs, toks, kv_state(m, cfg, pos)


def kv_state(m, cfg, next_pos):
    rows = min(next_pos, cfg["max_seq_len"])
    kv = cfg["n_kv_heads"] * cfg["head_dim"]
    return [m.read_kv(l, w)[: rows * kv].copy() for l in range(cfg["n_layers"]) for w in (0, 1)]


def hydrate(b, slot, prompt):
    for pos, tok in enumerate(prompt[:-1]):
        b.forward_batch([slot], [tok], [pos], 0)


def oracle_tokens(cfg, tensors, prompt, steps):
    om = oracle.OracleModel(cfg, {n: (t.id, np.ascontiguousarray(a).view(np.uint8).reshape(-1)) for n, t, a in tensors
                                  if n in X.expected_tensors(cfg)}, 1)
    for pos, tok in enumerate(prompt[:-1]):
        om.forward(tok, pos, 0)
    tok, out = prompt[-1], []
    for i in range(steps):
        tok = oracle.sample_argmax(om.forward(tok, len(prompt) - 1 + i, 1))
        out.append(tok)
    om.close()
    return out


def check_kv(b, cfg, slot, ref, next_pos):
    b.select_seq(slot)
    got = kv_state(b, cfg, next_pos)
    b.select_seq(0)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r), f"slot {slot}: KV cache differs from the solo run"


@pytest.mark.parametrize("shape", ["tiny", "small"])
@pytest.mark.parametrize("wtype", FORMATS)
def test_lock_step_batch_is_bit_identical_to_solo(shape, wtype):
    steps, prompts = 24, PROMPTS[:4]
    cfg, tensors = tensors_of(shape, wtype, 2, 0.06, 0)
    solo = solo_handle(cfg, tensors)
    refs = [solo_run(solo, cfg, p, steps) for p in prompts]
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    slots = [5, 0, 3, 6]                                           # not 0..3: slots are independent of their order
    for s, p in zip(slots, prompts):
        hydrate(b, s, p)
    toks = [p[-1] for p in prompts]
    pos = [len(p) - 1 for p in prompts]
    for k in range(steps):
        lg = b.forward_batch(slots, toks, pos)
        for i in range(4):
            assert np.array_equal(bits(lg[i]), bits(refs[i][0][k])), f"{wtype} {shape}: sequence {i} step {k}"
        toks = [argmax(r) for r in lg]
        pos = [q + 1 for q in pos]
        assert toks == [refs[i][1][k] for i in range(4)]
    for i, s in enumerate(slots):
        check_kv(b, cfg, s, refs[i][2], pos[i])
    b.close()
    if shape == "tiny":
        for i, p in enumerate(prompts):
            assert refs[i][1] == oracle_tokens(cfg, tensors, p, steps), f"{wtype}: sequence {i} differs from the oracle"


def test_run_to_run_bit_identical():
    """The same batched schedule twice (slots re-hydrated from position 0): the same logits and caches, bit for bit."""
    cfg, tensors = tensors_of("small", "q5_1", 4, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    runs = []
    for _ in range(2):
        for s, p in enumerate(PROMPTS):
            hydrate(b, s, p)
        toks, pos, lgs = [p[-1] for p in PROMPTS], [len(p) - 1 for p in PROMPTS], []
        for _ in range(12):
            lg = b.forward_batch(list(range(8)), toks, pos)
            lgs.append(bits(lg).copy())
            toks, pos = [argmax(r) for r in lg], [q + 1 for q in pos]
        kv = []
        for s in range(8):
            b.select_seq(s)
            kv.append(kv_state(b, cfg, pos[s]))
        b.select_seq(0)
        runs.append((lgs, kv))
    assert all(np.array_equal(x, y) for x, y in zip(runs[0][0], runs[1][0]))
    assert all(np.array_equal(x, y) for s in range(8) for x, y in zip(runs[0][1][s], runs[1][1][s]))
    b.close()


@pytest.mark.parametrize("graph,pdl", [(1, 1), (0, 0), (0, 1)])
def test_changing_compositions_join_and_leave(graph, pdl):
    """n = 1 .. 8 per step, permuted slots, sequences that join late and leave early: each sequence still matches its solo run."""
    steps = 16
    cfg, tensors = tensors_of("tiny", "q4_0", 3, 0.06, 0)
    solo = solo_handle(cfg, tensors)
    refs = [solo_run(solo, cfg, p, steps) for p in PROMPTS]
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    rng = np.random.default_rng(7)
    for s, p in enumerate(PROMPTS):
        hydrate(b, s, p)
    done = [0] * 8
    toks = [p[-1] for p in PROMPTS]
    pos = [len(p) - 1 for p in PROMPTS]
    seen_n = set()
    capi.tune("graph", graph); capi.tune("pdl", pdl)
    try:
        while min(done) < steps:
            live = [s for s in range(8) if done[s] < steps]
            n = int(rng.integers(1, len(live) + 1))
            pick = [int(v) for v in rng.permutation(live)[:n]]
            seen_n.add(n)
            lg = b.forward_batch(pick, [toks[s] for s in pick], [pos[s] for s in pick])
            for j, s in enumerate(pick):
                assert np.array_equal(bits(lg[j]), bits(refs[s][0][done[s]])), f"slot {s} step {done[s]} in a batch of {pick}"
                toks[s] = argmax(lg[j])
                pos[s] += 1
                done[s] += 1
    finally:
        capi.tune("graph", 1); capi.tune("pdl", 1)
    assert len(seen_n) >= 4
    for s in range(8):
        check_kv(b, cfg, s, refs[s][2], pos[s])
    b.close()


def test_ring_and_sinks_per_slot():
    """-T 24: some slots wrap their ring (and re-rotate their sinks) while others have not yet."""
    steps = 28
    prompts = [PROMPT, [1, 5], PROMPTS[2], [1, 300, 301, 302, 303, 304, 305, 306, 307, 308, 309, 310, 311, 312, 313, 314, 315, 316, 317, 318]]
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 24)
    assert cfg["max_seq_len"] == 24
    solo = solo_handle(cfg, tensors)
    refs = [solo_run(solo, cfg, p, steps) for p in prompts]
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    for s, p in enumerate(prompts):
        hydrate(b, s, p)
    toks = [p[-1] for p in prompts]
    pos = [len(p) - 1 for p in prompts]
    mixed = False
    for k in range(steps):
        mixed |= len({q >= 24 for q in pos}) == 2
        lg = b.forward_batch([0, 1, 2, 3], toks, pos)
        for i in range(4):
            assert np.array_equal(bits(lg[i]), bits(refs[i][0][k])), f"sequence {i} step {k} (pos {pos[i]})"
        toks = [argmax(r) for r in lg]
        pos = [q + 1 for q in pos]
    assert mixed
    for s in range(4):
        check_kv(b, cfg, s, refs[s][2], pos[s])
    b.close()
    for i, p in enumerate(prompts):
        assert refs[i][1] == oracle_tokens(cfg, tensors, p, steps)


def test_prefill_into_a_slot():
    """select_seq + prefill (+ prefill_window past the window), then batched decoding: the same logits, bit for bit, as prefill and
    decoding on a batch-1 handle; the other slots' caches are untouched."""
    cfg, tensors = tensors_of("tiny", "q4_1", 5, 0.06, 24)
    long_prompt = [1] + list(range(40, 70))                        # 31 tokens: 24 by prefill, 6 by prefill_window, the last decoded
    short = PROMPTS[2]
    solo = solo_handle(cfg, tensors)
    st = InferenceState(cfg)
    ref_lg = []
    solo.prefill(long_prompt[:24], 0, 0)
    solo.prefill_window(long_prompt[24:30], 24, 0)
    tok, pos = long_prompt[30], 30
    for _ in range(8):
        solo.forward(st, tok, pos, 1)
        ref_lg.append(st.logits().copy())
        tok, pos = argmax(ref_lg[-1]), pos + 1
    short_ref = solo_run(solo, cfg, short, 8)
    solo.close()

    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    hydrate(b, 1, short)
    b.select_seq(1)
    before = [b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)]
    b.select_seq(2)
    b.prefill(long_prompt[:24], 0, 0)
    b.prefill_window(long_prompt[24:30], 24, 0)
    b.select_seq(1)
    after = [b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)]
    assert all(np.array_equal(x, y) for x, y in zip(before, after)), "prefill into slot 2 touched slot 1"
    b.select_seq(0)
    toks, pos = [long_prompt[30], short[-1]], [30, len(short) - 1]
    for k in range(8):
        lg = b.forward_batch([2, 1], toks, pos)
        assert np.array_equal(bits(lg[0]), bits(ref_lg[k])), f"prefilled slot, step {k}"
        assert np.array_equal(bits(lg[1]), bits(short_ref[0][k])), f"other slot, step {k}"
        toks = [argmax(r) for r in lg]
        pos = [q + 1 for q in pos]
    b.close()


def test_device_argmax_matches_host_sampler():
    cfg, tensors = tensors_of("tiny", "q5_0", 21, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=3)
    toks, pos = [5, 6, 7], [0, 3, 9]
    for _ in range(16):
        lg = b.forward_batch([2, 0, 1], toks, pos)
        dev = b.forward_batch_argmax([2, 0, 1], toks, pos)   # same inputs inside the window: the KV rows are rewritten unchanged
        assert dev == [argmax(r) for r in lg]
        toks, pos = dev, [q + 1 for q in pos]
    b.close()


def test_refusals_leave_every_cache_untouched():
    import ctypes as C
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    for s in range(4):
        hydrate(b, s, PROMPTS[s])
    snap = []
    for s in range(4):
        b.select_seq(s)
        snap.append([b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)])
    b.select_seq(0)
    V = cfg["vocab_size"]
    cases = [([0, 0], [1, 2], [3, 3], 1),        # slot twice
             ([4], [1], [3], 1),                 # slot out of range
             ([-1], [1], [3], 1),
             ([0, 1, 2, 3, 0], [1] * 5, [3] * 5, 1),  # n > max_seqs
             ([0, 1], [1, V], [3, 3], 1),        # token out of range
             ([0, 1], [1, -1], [3, 3], 1),
             ([0, 1], [1, 2], [3, -1], 1),       # negative position
             ([0, 1], [1, 2], [3, 3], 7)]        # bad mode
    for seqs, toks, pos, mode in cases:
        with pytest.raises(capi.XalmError) as e:
            b.forward_batch(seqs, toks, pos, mode)
        assert e.value.status == 1, (seqs, toks, pos, mode)
    L = capi.lib()
    z = (C.c_int * 1)(0)
    assert L.xalm_cuda_forward_batch(b._h, 0, z, z, z, 1, None) == 1
    with pytest.raises(capi.XalmError):
        b.forward_batch_argmax([1, 1], [2, 2], [3, 3])
    with pytest.raises(capi.XalmError) as e:
        b.select_seq(4)
    assert e.value.status == 1
    for s in range(4):
        b.select_seq(s)
        now = [b.read_kv(l, w) for l in range(cfg["n_layers"]) for w in (0, 1)]
        assert all(np.array_equal(x, y) for x, y in zip(now, snap[s])), f"slot {s} changed by a refused call"
    b.close()

    # set_batch: after an upload, or on a tensor-parallel handle; F16 matrices on a batched handle
    h = C.c_void_p()
    xc = capi.XalmConfig.from_dict(cfg)
    capi.check(L.xalm_cuda_create(C.byref(xc), 0, 0, 1, C.byref(h)))
    m = Model.from_tensors(cfg, tensors)
    m._h = h
    name = "output.norm.weight"
    t, shape, raw = m.tensors[name]
    m.upload(name, t, shape, raw)
    assert L.xalm_cuda_set_batch(h, 4) == 4
    m.close()
    capi.check(L.xalm_cuda_create(C.byref(xc), 0, 0, 2, C.byref(h)))
    assert L.xalm_cuda_set_batch(h, 4) == 2
    L.xalm_cuda_destroy(h)
    cfg16, t16 = tensors_of("tiny", "f16", 2, 0.06, 0)
    with pytest.raises(capi.XalmError) as e:
        Model.from_tensors(cfg16, t16).cuda(max_seqs=2)
    assert e.value.status == 2 and "batched handle" in str(e.value)


@pytest.mark.parametrize("t", ["q8_0", "q4_0"])
def test_convert_py_checkpoints_decode_in_a_batch(golden_dir, t):
    path = os.path.join(golden_dir, f"tiny_{t}.xalm")
    f = X.XalmFile(path)
    model = Model.from_xalm(f)
    cfg = model.config
    prompts = [[1, 266, 267, 268, 269], [1, 270, 200], [1, 280, 281, 282, 283, 284, 285], [1, 250]]   # vocab 288
    otensors = {n: (tt.id, raw) for n, (tt, shape, raw) in model.tensors.items()}
    want = []
    for p in prompts:
        om = oracle.OracleModel(cfg, otensors, 1)
        for pos, tok in enumerate(p[:-1]):
            om.forward(tok, pos, 0)
        tok, out = p[-1], []
        for i in range(20):
            tok = oracle.sample_argmax(om.forward(tok, len(p) - 1 + i, 1))
            out.append(tok)
        want.append(out)
        om.close()
    model.cuda(max_seqs=4)
    for s, p in enumerate(prompts):
        hydrate(model, s, p)
    toks, pos, got = [p[-1] for p in prompts], [len(p) - 1 for p in prompts], [[] for _ in prompts]
    for _ in range(20):
        toks = model.forward_batch_argmax([0, 1, 2, 3], toks, pos)
        pos = [q + 1 for q in pos]
        for i, v in enumerate(toks):
            got[i].append(v)
    assert got == want
    model.close()


def test_full_size_mistral_7b_q8_0_eight_sequences():
    """Mistral-7B shape, q8_0, 32 layers (synthetic): 8 sequences, 8 greedy steps each, bit-identical to the solo mma runs."""
    cfg, tensors = tensors_of("m7", "q8_0", 0, 0.02, 0)
    prompts = [[1, 415 + i, 28747, 1824 + 3 * i][: 2 + i % 3] for i in range(8)]
    solo = solo_handle(cfg, tensors)
    refs = [solo_run(solo, cfg, p, 8) for p in prompts]
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    del tensors
    for s, p in enumerate(prompts):
        hydrate(b, s, p)
    toks, pos = [p[-1] for p in prompts], [len(p) - 1 for p in prompts]
    for k in range(8):
        lg = b.forward_batch(list(range(8)), toks, pos)
        for i in range(8):
            assert np.array_equal(bits(lg[i]), bits(refs[i][0][k])), f"sequence {i} step {k}"
        toks = [argmax(r) for r in lg]
        pos = [q + 1 for q in pos]
    b.close()
