"""The greedy chain (xalm_cuda_forward_greedy), which is how a draft model drafts: tokens, every layer's K/V and the logits left on
the device must be bit-identical to the loop it stands for (forward HYDRATE for all tokens but the last, then forward_argmax
of each result) run on a second handle of the same kind, past the context window too."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_batch import PROMPT, argmax, bits, tensors_of
from xalm_b200 import capi, synth
from xalm_b200 import xalm_file as X
from xalm_b200.model import InferenceState, Model, Sampler

pytestmark = pytest.mark.gpu


def loop(m, tokens, pos, n_out, host_sampler=False):
    """the loop forward_greedy is equivalent to; host_sampler: forward + Sampler.sample_argmax instead of forward_argmax"""
    for j, t in enumerate(tokens[:-1]):
        m.forward_async(t, pos + j, 0)
    t, p, out = tokens[-1], pos + len(tokens) - 1, []
    st, sampler = InferenceState(m.config), Sampler(m.config)
    for _ in range(n_out):
        if host_sampler:
            m.forward(st, t, p, 1)
            t = sampler.sample_argmax(st)
        else:
            t = m.forward_argmax(t, p)
        out.append(t)
        p += 1
    return out


def state_of(m):
    cfg = m.config
    kv = [m.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)]
    return kv, bits(m.read_state(capi.S_LOGITS, cfg["vocab_size"])).copy()


def same_state(a, b, what):
    (kva, lga), (kvb, lgb) = state_of(a), state_of(b)
    for i, (x, y) in enumerate(zip(kva, kvb)):
        assert np.array_equal(x, y), f"{what}: layer {i // 2} {'KV'[i % 2]} cache differs"
    assert np.array_equal(lga, lgb), f"{what}: logits on the device differ"


def pair(shape, wtype, seed=2, context=0, **cuda_kw):
    cfg, tensors = tensors_of(shape, wtype, seed, 0.06, context)
    return cfg, Model.from_tensors(cfg, tensors).cuda(**cuda_kw), Model.from_tensors(cfg, tensors).cuda(**cuda_kw)


# (n_in, n_out) calls made one after the other, each continuing where the previous one stopped
CALLS = [(n_in, n_out) for n_in in (1, 2, 8) for n_out in (1, 5, 16)]


def run_calls(chain, ref, cfg, calls, pos=0, host_sampler=False, what=""):
    V = cfg["vocab_size"]
    rng = np.random.default_rng(3)
    for n_in, n_out in calls:
        toks = [int(v) for v in rng.integers(3, V, n_in)]
        got = chain.forward_greedy(toks, pos, n_out)
        want = loop(ref, toks, pos, n_out, host_sampler)
        assert got == want, f"{what}: n_in {n_in}, n_out {n_out} at position {pos}"
        same_state(chain, ref, f"{what}: n_in {n_in}, n_out {n_out} at position {pos}")
        pos += n_in + n_out - 1
    return pos


@pytest.mark.parametrize("shape", ["tiny", "small"])
@pytest.mark.parametrize("wtype", ["q8_0", "q4_0", "f16", "f8_e4m3"])
def test_chain_is_bit_identical_to_the_loop(shape, wtype):
    """q8_0 on the dp4a matvec, q4_0 on the tensor-core matvec, f16 and f8_e4m3 on the float matvec"""
    cfg, chain, ref = pair(shape, wtype)
    for j, t in enumerate(PROMPT):
        chain.forward_async(t, j, 0)
        ref.forward_async(t, j, 0)
    run_calls(chain, ref, cfg, CALLS, len(PROMPT), what=f"{shape} {wtype}")
    chain.close()
    ref.close()


@pytest.mark.parametrize("graph,pdl", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_graph_and_pdl_on_and_off(graph, pdl):
    capi.tune("graph", graph); capi.tune("pdl", pdl)
    try:
        cfg, chain, ref = pair("tiny", "q4_0", seed=3)
        run_calls(chain, ref, cfg, CALLS, 0, host_sampler=True, what=f"graph {graph} pdl {pdl}")
    finally:
        capi.tune("graph", 1); capi.tune("pdl", 1)
    chain.close()
    ref.close()


@pytest.mark.parametrize("wtype", ["q8_0", "f16"])
def test_chain_across_the_window(wtype):
    """max_seq_len 32: a chain from position 25 runs 16 steps into the KV ring; the sinks are re-rotated as the loop does it"""
    cfg, chain, ref = pair("tiny", wtype, seed=4, context=32)
    assert cfg["max_seq_len"] == 32
    for p in range(25):
        chain.forward_async(PROMPT[p % len(PROMPT)], p, 0)
        ref.forward_async(PROMPT[p % len(PROMPT)], p, 0)
    pos = run_calls(chain, ref, cfg, [(1, 16)], 25, what=f"{wtype} across the window")
    assert pos == 41
    run_calls(chain, ref, cfg, [(2, 16), (8, 16)], pos, what=f"{wtype} past the window")
    chain.close()
    ref.close()


def test_slot_of_a_batched_handle():
    cfg, chain, ref = pair("tiny", "q4_0", seed=5, max_seqs=4)
    for m in (chain, ref):
        m.select_seq(1)
        for j, t in enumerate(PROMPT):
            m.forward_async(t, j, 0)
        m.select_seq(2)
    run_calls(chain, ref, cfg, CALLS[:5], 0, what="slot 2")
    for m in (chain, ref):
        m.select_seq(1)
    same_state(chain, ref, "slot 1, not driven by the chain")
    chain.close()
    ref.close()


def test_run_to_run_bit_identical():
    cfg, tensors = tensors_of("small", "q4_0", 6, 0.06, 0)
    m = Model.from_tensors(cfg, tensors).cuda()
    runs = []
    for _ in range(2):
        for j, t in enumerate(PROMPT):
            m.forward_async(t, j, 0)
        toks = [m.forward_greedy([7, 9], len(PROMPT), 16), m.forward_greedy([11], len(PROMPT) + 17, 16)]
        runs.append((toks, state_of(m)))
    assert runs[0][0] == runs[1][0]
    assert all(np.array_equal(x, y) for x, y in zip(runs[0][1][0], runs[1][1][0]))
    assert np.array_equal(runs[0][1][1], runs[1][1][1])
    m.close()


def test_refusals_leave_the_cache_untouched():
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 0)
    V = cfg["vocab_size"]
    m = Model.from_tensors(cfg, tensors).cuda()
    for j, t in enumerate(PROMPT):
        m.forward_async(t, j, 0)
    before = state_of(m)
    L = capi.lib()
    out = (C.c_int * 16)()
    toks = (C.c_int * 9)(*[5] * 9)
    bad = (C.c_int * 2)(5, V)
    neg = (C.c_int * 1)(-1)
    for n_in, tk, pos, n_out in ((0, toks, 8, 1), (9, toks, 8, 1), (1, toks, 8, 0), (1, toks, 8, 17), (2, bad, 8, 1), (1, neg, 8, 1),
                                 (1, toks, -1, 1)):
        assert L.xalm_cuda_forward_greedy(m._h, n_in, tk, pos, n_out, out) == 1, (n_in, pos, n_out)
    assert L.xalm_cuda_forward_greedy(m._h, 1, None, 8, 1, out) == 1
    assert L.xalm_cuda_forward_greedy(m._h, 1, toks, 8, 1, None) == 1
    after = state_of(m)
    assert all(np.array_equal(x, y) for x, y in zip(before[0], after[0])), "a refused call changed the cache"
    assert np.array_equal(before[1], after[1])
    assert m.forward_greedy([5], 8, 3) == loop_tokens_after(cfg, tensors, 3)
    m.close()


def loop_tokens_after(cfg, tensors, n_out):
    """the loop's tokens for the refusal test's valid call, on a fresh handle"""
    r = Model.from_tensors(cfg, tensors).cuda()
    for j, t in enumerate(PROMPT):
        r.forward_async(t, j, 0)
    out = loop(r, [5], 8, n_out)
    r.close()
    return out


def test_tensor_parallel_handle_is_unsupported():
    cfg = X.parse_config(synth.metadata_strings(synth.model_config("tp")))
    L = capi.lib()
    h = C.c_void_p()
    xc = capi.XalmConfig.from_dict(cfg)
    capi.check(L.xalm_cuda_create(C.byref(xc), 0, 0, 2, C.byref(h)))
    try:
        out = (C.c_int * 4)()
        assert L.xalm_cuda_forward_greedy(h, 1, (C.c_int * 1)(5), 0, 4, out) == 2
        assert b"tensor-parallel" in L.xalm_cuda_last_error()
    finally:
        L.xalm_cuda_destroy(h)


def test_device_tokens_match_the_host_sampler():
    cfg, chain, ref = pair("tiny", "q5_0", seed=21)
    st, sampler = InferenceState(cfg), Sampler(cfg)
    got = chain.forward_greedy([PROMPT[0]], 0, 16)
    t, want = PROMPT[0], []
    for p in range(16):
        ref.forward(st, t, p, 1)
        assert argmax(st.logits()) == sampler.sample_argmax(st)
        t = sampler.sample_argmax(st)
        want.append(t)
    assert got == want
    chain.close()
    ref.close()
