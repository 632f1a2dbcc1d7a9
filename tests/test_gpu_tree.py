"""Trees (xalm_cuda_forward_tree, xalm_cuda_tree_accept): several drafted continuations of one sequence verified in one step.
Each node's logits must be bit-identical to decoding its root-to-node branch one step at a time on a batch-1 handle with the
tensor-core matvec, and after tree_accept of any branch the slot's cache must be the one that branch's solo run leaves."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle
from test_gpu_batch import FORMATS, PROMPT, PROMPTS, argmax, bits, hydrate, kv_state, solo_handle, solo_run, tensors_of
from xalm_b200 import capi
from xalm_b200 import xalm_file as X
from xalm_b200.model import InferenceState, Model

pytestmark = pytest.mark.gpu

SHAPES = {
    "chain8": [-1, 0, 1, 2, 3, 4, 5, 6],
    "star8": [-1, 0, 0, 0, 0, 0, 0, 0],
    "two_branches_of_3": [-1, 0, 0, 1, 2, 3, 4],     # level by level, as xalm_main numbers them: 1-3-5 and 2-4-6
    "binary_depth2": [-1, 0, 0, 1, 1, 2, 2],
    "random": None,                                  # seeded below
}


def shape_parents(name, seed=3):
    if SHAPES[name] is not None:
        return list(SHAPES[name])
    rng = np.random.default_rng(seed)
    return [-1] + [int(rng.integers(0, i)) for i in range(1, 8)]


def path_to(parents, i):
    p = []
    while i >= 0:
        p.append(i)
        i = parents[i]
    return p[::-1]


def depths(parents):
    d = [0]
    for i in range(1, len(parents)):
        d.append(d[parents[i]] + 1)
    return d


def tree_tokens(parents, true_leaf, seq, V, rng):
    """nodes on the path to true_leaf carry seq (the solo run's fed tokens: the root's, then its greedy tokens); every other node
    a token that differs from seq at its depth"""
    on = set(path_to(parents, true_leaf))
    d = depths(parents)
    toks = []
    for i in range(len(parents)):
        if i in on:
            toks.append(seq[d[i]])
        else:
            t = int(rng.integers(3, V))
            toks.append(t if t != seq[d[i]] else (t + 1) % V)
    return toks


def branch_refs(solo, cfg, prompt, parents, toks, hydrated=False):
    """per node: the logits a batch-1 handle gives when it decodes the node's branch one token at a time from the prompt's last
    position; the prefix is decoded once (hydrated: already in the cache).  Also per leaf: the KV rows that branch leaves."""
    st = InferenceState(cfg)
    for pos, tok in enumerate([] if hydrated else prompt[:-1]):
        solo.forward(st, tok, pos, 0)
    P = len(prompt) - 1
    ref, kv = [None] * len(parents), {}
    leaves = [i for i in range(len(parents)) if i not in parents]
    for leaf in leaves:
        path = path_to(parents, leaf)
        for e, node in enumerate(path):
            solo.forward(st, toks[node], P + e, 1)
            lg = st.logits().copy()
            if ref[node] is None:
                ref[node] = lg
            else:                                      # a shared ancestor: the same logits from every branch through it
                assert np.array_equal(bits(lg), bits(ref[node]))
        kv[leaf] = kv_state(solo, cfg, P + len(path))
    return ref, kv


def check_rows(b, cfg, slot, ref, rows):
    b.select_seq(slot)
    got = kv_state(b, cfg, rows)
    b.select_seq(0)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r[: g.size]), f"slot {slot}: KV rows 0 .. {rows - 1} differ from the solo run"


@pytest.mark.parametrize("shape", ["tiny", "small"])
@pytest.mark.parametrize("wtype", FORMATS)
def test_every_node_is_bit_identical_to_its_branch_decoded_solo(shape, wtype):
    cfg, tensors = tensors_of(shape, wtype, 2, 0.06, 0)
    V, P = cfg["vocab_size"], len(PROMPT) - 1
    solo = solo_handle(cfg, tensors)
    _, toks, _ = solo_run(solo, cfg, PROMPT, 8)
    seq = [PROMPT[-1]] + toks
    rng = np.random.default_rng(17)
    cases = []
    for name in SHAPES:
        parents = shape_parents(name)
        true_leaf = len(parents) - 1
        tt = tree_tokens(parents, true_leaf, seq, V, rng)
        cases.append((name, parents, tt, true_leaf) + branch_refs(solo, cfg, PROMPT, parents, tt))
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    hydrate(b, 5, PROMPT)
    for name, parents, tt, true_leaf, ref, kv in cases:
        lg = b.forward_tree(5, tt, parents, P)
        for i in range(len(parents)):
            assert np.array_equal(bits(lg[i]), bits(ref[i])), f"{shape} {wtype} {name}: node {i}"
        assert b.forward_tree_argmax(5, tt, parents, P) == [argmax(r) for r in lg]
        path = path_to(parents, true_leaf)
        assert [argmax(lg[i]) for i in path[:-1]] == [tt[i] for i in path[1:]]   # the true branch is accepted whole
        b.tree_accept(5, P, path)
        check_rows(b, cfg, 5, kv[true_leaf], P + len(path))
    b.close()


def greedy_tree_walk(parents, toks, nxt):
    path = [0]
    for i in range(1, len(parents)):
        if parents[i] == path[-1] and toks[i] == nxt[path[-1]]:
            path.append(i)
    return path


@pytest.mark.parametrize("graph,pdl", [(1, 1), (0, 0), (0, 1)])
def test_accept_a_later_branch_and_continue(graph, pdl):
    """Each round verifies a tree whose LAST-numbered branch holds the solo run's tokens and whose lower-numbered branches are
    wrong, accepts the walk's branch (so tree_accept moves rows), and goes on.  Forty more steps then mix forward_batch, spans and
    further trees; everything stays bit-identical to the solo run, cache included."""
    cfg, tensors = tensors_of("tiny", "q4_0", 3, 0.06, 0)
    V = cfg["vocab_size"]
    total = 120
    solo = solo_handle(cfg, tensors)
    lgs, toks, kv = solo_run(solo, cfg, PROMPT, total)
    solo.close()
    seq, p0 = [PROMPT[-1]] + toks, len(PROMPT) - 1
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    hydrate(b, 2, PROMPT)
    hydrate(b, 6, PROMPTS[2])
    b.select_seq(6)
    other = [b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)]
    b.select_seq(0)
    rng = np.random.default_rng(23)
    capi.tune("graph", graph); capi.tune("pdl", pdl)
    try:
        k, moved = 0, 0
        def tree_round(k):
            # two or three branches; the last one follows seq for its whole depth, the others go wrong at their first token
            nb = int(rng.integers(2, 4))
            depth = max(1, (8 - 1) // nb)
            parents, tt = [-1], [seq[k]]
            for br in range(nb):
                par = 0
                for e in range(depth):
                    if br == nb - 1:
                        t = seq[k + 1 + e]
                    else:
                        t = int(rng.integers(3, V))
                        if e == 0 and t == seq[k + 1]:
                            t = (t + 1) % V
                    parents.append(par); tt.append(t)
                    par = len(parents) - 1
            lg = b.forward_tree(2, tt, parents, p0 + k)
            d = depths(parents)
            for i in range(len(parents)):
                if d[i] == 0 or i > len(parents) - 1 - depth:   # the root and the true branch: the solo run's own logits
                    assert np.array_equal(bits(lg[i]), bits(lgs[k + d[i]])), f"tree at {p0 + k}: node {i}"
            nxt = [argmax(r) for r in lg]
            path = greedy_tree_walk(parents, tt, nxt)
            assert path == [0] + list(range(len(parents) - depth, len(parents)))
            b.tree_accept(2, p0 + k, path)
            return len(path) - 1, path != list(range(len(path)))
        while k < 60:
            a, mv = tree_round(k)
            moved += mv
            k += a + 1
        assert moved > 0
        check_rows(b, cfg, 2, kv, p0 + k)
        # forty more steps: plain batched steps, spans and trees in turn
        end = k + 40
        while k < end:
            kind = k % 3
            if kind == 0:
                lg = b.forward_batch([2], [seq[k]], [p0 + k])
                assert np.array_equal(bits(lg[0]), bits(lgs[k])), f"plain step at {p0 + k}"
                k += 1
            elif kind == 1:
                L = 4
                lg = b.forward_spans([2] * L, seq[k:k + L], list(range(p0 + k, p0 + k + L)))
                for j in range(L):
                    assert np.array_equal(bits(lg[j]), bits(lgs[k + j])), f"span at {p0 + k}: entry {j}"
                k += L
            else:
                a, mv = tree_round(k)
                moved += mv
                k += a + 1
        check_rows(b, cfg, 2, kv, p0 + k)
    finally:
        capi.tune("graph", 1); capi.tune("pdl", 1)
    b.select_seq(6)
    now = [b.read_kv(l, w) for l in range(cfg["n_layers"]) for w in (0, 1)]
    b.select_seq(0)
    assert all(np.array_equal(x, y) for x, y in zip(now, other)), "slot 6 changed by tree calls on slot 2"
    b.close()


def test_chain_tree_equals_span():
    cfg, tensors = tensors_of("small", "q8_0", 4, 0.06, 0)
    rng = np.random.default_rng(2)
    toks = [PROMPT[-1]] + [int(v) for v in rng.integers(3, cfg["vocab_size"], 7)]
    P = len(PROMPT) - 1
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    hydrate(b, 1, PROMPT)
    hydrate(b, 4, PROMPT)
    for n in (1, 2, 5, 8):
        ls = b.forward_spans([1] * n, toks[:n], list(range(P, P + n)))
        lt = b.forward_tree(4, toks[:n], [-1] + list(range(n - 1)), P)
        assert np.array_equal(bits(ls), bits(lt)), f"chain of {n}"
        b.tree_accept(4, P, list(range(n)))                    # a chain: nothing to move
        b.select_seq(1)
        ks = kv_state(b, cfg, P + n)
        b.select_seq(4)
        kt = kv_state(b, cfg, P + n)
        b.select_seq(0)
        assert all(np.array_equal(x, y) for x, y in zip(ks, kt)), f"chain of {n}: caches differ"
    b.close()


def test_refusals_leave_every_cache_untouched():
    cfg, tensors = tensors_of("tiny", "q8_0", 2, 0.06, 0)
    W, V = cfg["max_seq_len"], cfg["vocab_size"]
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=4)
    for s in range(4):
        hydrate(b, s, PROMPTS[s])

    def snapshot():
        out = []
        for s in range(4):
            b.select_seq(s)
            out.append([b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)])
        b.select_seq(0)
        return out
    snap = snapshot()
    tree_cases = [(0, [1, 2], [0, 0], 3),            # root's parent not -1
                  (0, [1, 2], [-1, 1], 3),           # a node its own parent
                  (0, [1, 2, 3], [-1, 2, 0], 3),     # a parent after its child
                  (0, [1, 2], [-1, -1], 3),          # two roots
                  (0, [1, V], [-1, 0], 3),           # token out of range
                  (0, [1, -1], [-1, 0], 3),          # negative token
                  (0, [1, 2], [-1, 0], -1),          # negative position
                  (4, [1, 2], [-1, 0], 3),           # slot out of range
                  (-1, [1, 2], [-1, 0], 3),
                  (0, [1, 2], [-1, 0], W - 1),       # a tree reaching max_seq_len
                  (0, [1, 2], [-1, 0], W + 5),       # a tree past the window
                  (0, [1] * 5, [-1, 0, 0, 0, 0], 3)] # n > max_seqs
    for slot, toks, parents, pos in tree_cases:
        for call in (b.forward_tree, b.forward_tree_argmax):
            with pytest.raises(capi.XalmError) as e:
                call(slot, toks, parents, pos)
            assert e.value.status == 1, (slot, toks, parents, pos)
    # a real tree, so that accept has something it could move; then refused accepts
    b.forward_tree(1, [PROMPTS[1][-1], 5, 6, 7], [-1, 0, 0, 1], len(PROMPTS[1]) - 1)
    snap = snapshot()
    p1 = len(PROMPTS[1]) - 1
    accept_cases = [(1, p1, [1, 2]),                 # not starting at the root
                    (1, p1, [0, 2, 2]),              # not increasing
                    (1, p1, [0, 3, 2]),
                    (1, p1, [0, 4]),                 # a node past max_seqs
                    (1, W - 2, [0, 2]),              # a row reaching max_seq_len
                    (1, -1, [0, 2]),                 # negative position
                    (4, p1, [0, 2]),                 # slot out of range
                    (1, p1, [0, 1, 2, 3, 3])]        # n > max_seqs
    for slot, pos, nodes in accept_cases:
        with pytest.raises(capi.XalmError) as e:
            b.tree_accept(slot, pos, nodes)
        assert e.value.status == 1, (slot, pos, nodes)
    L = capi.lib()
    z, o = (C.c_int * 2)(0, 0), (C.c_int * 2)(0, 0)
    par = (C.c_int * 2)(-1, 0)
    assert L.xalm_cuda_forward_tree(b._h, 0, 0, z, par, 3, None) == 1
    for t, p in ((None, par), (z, None)):
        assert L.xalm_cuda_forward_tree(b._h, 0, 2, t, p, 3, None) == 1
        assert L.xalm_cuda_forward_tree_argmax(b._h, 0, 2, t, p, 3, o) == 1
    assert L.xalm_cuda_forward_tree_argmax(b._h, 0, 2, z, par, 3, None) == 1
    assert L.xalm_cuda_tree_accept(b._h, 0, 3, 1, None) == 1
    assert L.xalm_cuda_tree_accept(b._h, 0, 3, 0, z) == 1
    b.sync()
    now = snapshot()
    for s in range(4):
        assert all(np.array_equal(x, y) for x, y in zip(now[s], snap[s])), f"slot {s} changed by a refused call"
    b.close()
    solo = solo_handle(cfg, tensors)                         # a handle without set_batch
    for call in (solo.forward_tree, solo.forward_tree_argmax):
        with pytest.raises(capi.XalmError) as e:
            call(0, [1, 2], [-1, 0], 0)
        assert e.value.status == 4
    with pytest.raises(capi.XalmError) as e:
        solo.tree_accept(0, 0, [0, 1])
    assert e.value.status == 4
    solo.close()


def test_tree_and_accept_leave_other_slots_untouched():
    cfg, tensors = tensors_of("tiny", "q5_0", 6, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    for s in range(8):
        hydrate(b, s, PROMPTS[s])

    def slot_kv(s):
        b.select_seq(s)
        out = [b.read_kv(l, w).copy() for l in range(cfg["n_layers"]) for w in (0, 1)]
        b.select_seq(0)
        return out
    before = {s: slot_kv(s) for s in range(8) if s != 3}
    P = len(PROMPTS[3]) - 1
    parents = [-1, 0, 0, 1, 2, 2, 5, 3]
    b.forward_tree(3, [PROMPTS[3][-1], 10, 11, 12, 13, 14, 15, 16], parents, P)
    b.tree_accept(3, P, [0, 2, 5, 6])
    for s, kv in before.items():
        assert all(np.array_equal(x, y) for x, y in zip(slot_kv(s), kv)), f"slot {s} changed"
    b.close()


def test_run_to_run_bit_identical():
    cfg, tensors = tensors_of("small", "q5_1", 4, 0.06, 0)
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    runs = []
    for _ in range(2):
        hydrate(b, 2, PROMPT)
        tok, pos, lgs = PROMPT[-1], len(PROMPT) - 1, []
        for r in range(6):
            parents = shape_parents("random", seed=r)
            tt = [tok] + [(tok + 3 * i) % cfg["vocab_size"] for i in range(1, 8)]
            lg = b.forward_tree(2, tt, parents, pos)
            lgs.append(bits(lg).copy())
            nxt = [argmax(v) for v in lg]
            path = greedy_tree_walk(parents, tt, nxt)
            b.tree_accept(2, pos, path)
            tok, pos = nxt[path[-1]], pos + len(path)
        b.select_seq(2)
        kv = [x.copy() for x in kv_state(b, cfg, pos)]
        b.select_seq(0)
        runs.append((lgs, kv))
    assert all(np.array_equal(x, y) for x, y in zip(runs[0][0], runs[1][0]))
    assert all(np.array_equal(x, y) for x, y in zip(runs[0][1], runs[1][1]))
    b.close()


def test_full_size_mistral_7b_q8_0_tree_of_eight():
    """Mistral-7B shape, q8_0: an 8-node tree of two branches at position 100 and at position 4000, every node bit-identical to
    its branch decoded solo."""
    cfg, tensors = tensors_of("m7", "q8_0", 0, 0.02, 0)
    rng = np.random.default_rng(5)
    V = cfg["vocab_size"]
    ctx = [1] + [int(v) for v in rng.integers(3, V, 4000)]
    parents = [-1, 0, 0, 1, 2, 3, 4, 5]                          # branches 1-3-5-7 and 2-4-6
    tt = [0] + [int(v) for v in rng.integers(3, V, 7)]
    solo = solo_handle(cfg, tensors)
    refs = {}
    for P in (100, 4000):
        tt[0] = ctx[P]
        solo.prefill(ctx[:P], 0, 0)
        refs[P] = branch_refs(solo, cfg, ctx[:P + 1], parents, tt, hydrated=True)[0]
    solo.close()
    b = Model.from_tensors(cfg, tensors).cuda(max_seqs=8)
    del tensors
    for P in (100, 4000):
        tt[0] = ctx[P]
        b.select_seq(0)
        b.prefill(ctx[:P], 0, 0)
        lg = b.forward_tree(0, tt, parents, P)
        for i in range(8):
            assert np.array_equal(bits(lg[i]), bits(refs[P][i])), f"tree at {P}: node {i}"
    b.close()


def test_tree_verified_greedy_tokens_equal_the_oracle(golden_dir):
    """tiny_q4_0 (a convert.py checkpoint): greedy decoding where every pass verifies a tree of two branches (one made of
    repeats of the last token, one of the previous pass's rejected greedy tokens) gives the oracle's tokens."""
    path = os.path.join(golden_dir, "tiny_q4_0.xalm")
    model = Model.from_xalm(X.XalmFile(path))
    cfg = model.config
    prompt, steps = [1, 266, 267, 268, 266, 267], 32
    otensors = {n: (tt.id, raw) for n, (tt, shape, raw) in model.tensors.items()}
    om = oracle.OracleModel(cfg, otensors, 1)
    for pos, tok in enumerate(prompt[:-1]):
        om.forward(tok, pos, 0)
    tok, want = prompt[-1], []
    for i in range(steps):
        tok = oracle.sample_argmax(om.forward(tok, len(prompt) - 1 + i, 1))
        want.append(tok)
    om.close()
    model.cuda(max_seqs=8)
    hydrate(model, 0, prompt)
    got, tok, pos, guess = [], prompt[-1], len(prompt) - 1, [7, 8, 9]
    while len(got) < steps and pos + 7 < cfg["max_seq_len"]:
        parents = [-1, 0, 0, 1, 2, 3, 4]
        tt = [tok, tok, guess[0], tok, guess[1], tok, guess[2]]
        if tt[2] == tt[1]:
            tt[2] = (tt[2] + 1) % cfg["vocab_size"]
        nxt = model.forward_tree_argmax(0, tt, parents, pos)
        wp = greedy_tree_walk(parents, tt, nxt)
        model.tree_accept(0, pos, wp)
        got += [tt[i] for i in wp[1:]] + [nxt[wp[-1]]]
        guess = [nxt[i] for i in (0, 2, 4)]
        tok, pos = nxt[wp[-1]], pos + len(wp)
    n = min(len(got), steps)
    assert n >= 16
    assert got[:n] == want[:n]
    model.close()
