"""The forward pass pinned to the REFERENCE ITSELF.

tests/golden/ref_fwd_*.npz hold logits, greedy tokens, sampler probabilities and KV-cache bits produced by the unmodified
reference C++ (src/infer.cpp, model.cpp, sampler.cpp compiled by oracle/Makefile.ref; generator: tests/golden/make_ref_forward.py).

  * CPU: the oracle restatement (oracle/xalm_oracle.cpp) must reproduce them — same greedy tokens, logits within fp32
    reassociation noise, identical KV bits up to libm/accumulation-order rounding of single entries.
  * GPU: the CUDA path must reproduce them — token-exact, logits within the north star's 1e-2.
  * when oracle/_ref/libxalm_ref.so is present (dev container), the oracle is also compared with the live reference on a
    checkpoint no fixture covers.
"""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest

from oracle import oracle
from xalm_b200 import synth
from xalm_b200 import types as T
from xalm_b200 import xalm_file as X
from xalm_b200.model import InferenceState, Model, Sampler

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CASES = sorted(os.path.basename(p)[len("ref_fwd_"):-4] for p in glob.glob(os.path.join(GOLDEN, "ref_fwd_*.npz")))


def load_case(name, tmp_path):
    g = np.load(os.path.join(GOLDEN, f"ref_fwd_{name}.npz"))
    case = json.loads(bytes(g["case"]).decode())
    if "file" in case:
        path = os.path.join(GOLDEN, case["file"])
    else:
        path = str(tmp_path / f"{name}.xalm")
        kw = dict(case["synth"])
        synth.write_checkpoint(path, kw.pop("shape"), kw.pop("wtype"), kw.pop("seed"), std=kw.pop("std"), **kw)
    f = X.XalmFile(path)
    model = Model.from_xalm(f, case["context"])
    return g, case, model


def test_fixtures_exist():
    assert len(CASES) >= 8


def kv_close(a_bits, b_bits):
    a = a_bits.view(np.float16).astype(np.float32)
    b = b_bits.view(np.float16).astype(np.float32)
    mism = float(np.mean(a_bits != b_bits))
    worst = float(np.max(np.abs(a - b))) if a.size else 0.0
    return mism, worst, float(np.abs(b).max()) if b.size else 1.0


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_the_reference(name, tmp_path):
    g, case, model = load_case(name, tmp_path)
    config = model.config
    otensors = {n: (t.id, raw) for n, (t, shape, raw) in model.tensors.items()}
    om = oracle.OracleModel(config, otensors, 1)
    assert list(g["config"][:8]) == [config[k] for k in ("dim", "hidden_dim", "head_dim", "n_layers", "n_heads", "n_kv_heads", "vocab_size", "max_seq_len")]
    toks = [int(t) for t in g["tokens"]]
    n_prompt = len(case["prompt"])
    lg = None
    for pos in range(n_prompt):
        lg = om.forward(toks[pos], pos, 1 if pos + 1 == n_prompt else 0)
    worst = 0.0
    for step in range(case["steps"] + 1):
        ref = g["logits"][step]
        worst = max(worst, float(np.max(np.abs(lg - ref))))
        if step == case["steps"]:
            break
        nxt = oracle.sample_argmax(lg)
        assert nxt == toks[n_prompt + step], f"{name}: greedy token {step} differs from the reference"       # sampler.cpp:3-16
        assert abs(oracle.sample_prob(lg, nxt) - float(g["probs"][step])) <= 1e-4                             # sampler.cpp:18-33
        lg = om.forward(nxt, n_prompt + step, 1)
    # Not bit-identical by construction: infer.cpp:121 accumulates under `#pragma omp simd` (lane order and FMA contraction are the
    # compiler's: g++ here, clang/NEON on the reference's own platform), and every difference of one fp32 ulp that crosses an
    # fp16 rounding boundary in the KV cache feeds back.  Measured: <= 3e-4 in all three oracle accumulation modes (strict
    # sequential 1.1e-4, vectorised 2.7e-4, fp64 3.1e-4 on the 4-layer model) — 30x inside the 1e-2 contract; tokens identical.
    assert worst <= 5e-4, f"{name}: oracle logits differ from the reference by {worst}"
    for l in range(config["n_layers"]):
        for which, nm in ((0, "k"), (1, "v")):
            ref_bits = g[f"{nm}_{l}"]
            mism, wdiff, scale = kv_close(om.kv(l, which)[: ref_bits.size], ref_bits)
            # one fp16 ulp where the fp32 noise above crosses a rounding boundary (grows with depth: up to ~10 % of entries by layer 3)
            assert wdiff <= 2e-3 * max(1.0, scale) and mism < 0.2, f"{name}: {nm} cache of layer {l}: {mism:.4f} of entries differ, worst {wdiff}"
    assert np.max(np.abs(om.state(0, config["dim"]) - g["x"])) <= 5e-4 * max(1.0, float(np.abs(g["x"]).max()))
    om.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_cuda_reproduces_the_reference(name, tmp_path):
    g, case, model = load_case(name, tmp_path)
    config = model.config
    model.cuda()
    state = InferenceState(config)
    sampler = Sampler(config)
    toks = [int(t) for t in g["tokens"]]
    n_prompt = len(case["prompt"])
    for pos in range(n_prompt):
        model.forward(state, toks[pos], pos, 1 if pos + 1 == n_prompt else 0)
    worst = 0.0
    for step in range(case["steps"] + 1):
        worst = max(worst, float(np.max(np.abs(state.logits() - g["logits"][step]))))
        if step == case["steps"]:
            break
        nxt = sampler.sample_argmax(state)
        assert nxt == toks[n_prompt + step], f"{name}: greedy token {step} differs from the reference CPU path"
        model.forward(state, nxt, n_prompt + step, 1)
    assert worst <= 1e-2, f"{name}: logits differ from the reference by {worst}"                              # north star tolerance
    for l in range(config["n_layers"]):
        for which, nm in ((0, "k"), (1, "v")):
            ref_bits = g[f"{nm}_{l}"]
            mism, wdiff, scale = kv_close(model.read_kv(l, which)[: ref_bits.size], ref_bits)
            # never more than one fp16 ulp; how many entries sit on the other side of a rounding boundary grows with depth
            # (fp32 sums in a different order than the CPU's: ~1e-4 relative by layer 3, a fifth of an ulp at |k| ~ 3)
            assert wdiff <= 2e-3 * max(1.0, scale) and mism < 0.4, f"{name}: {nm} cache of layer {l}: {mism:.4f} differ, worst {wdiff}"
    model.close()


REF_SO = os.path.join(ROOT, "oracle", "_ref", "libxalm_ref.so")


@pytest.mark.skipif(not os.path.exists(REF_SO), reason="oracle/_ref/libxalm_ref.so not built (build() builds it when XALM_REFERENCE names the reference's sources)")
def test_oracle_against_the_live_reference(tmp_path):
    """A checkpoint no fixture covers (bf16 weights, 3 kv heads' worth of GQA, window 20 with the prompt running past it)."""
    path = str(tmp_path / "live.xalm")
    synth.write_checkpoint(path, "tiny", "bf16", 11, std=0.06)
    L = C.CDLL(REF_SO)
    L.xref_load.restype = C.c_void_p
    L.xref_load.argtypes = [C.c_char_p, C.c_int]
    L.xref_forward.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    L.xref_free.argtypes = [C.c_void_p]
    h = L.xref_load(path.encode(), 20)
    assert h
    model = Model.from_xalm(X.XalmFile(path), 20)
    om = oracle.OracleModel(model.config, {n: (t.id, raw) for n, (t, shape, raw) in model.tensors.items()}, 1)
    lg_r = np.zeros(model.config["vocab_size"], np.float32)
    rng = np.random.default_rng(5)
    for pos in range(45):
        tok = int(rng.integers(3, model.config["vocab_size"]))
        assert L.xref_forward(h, tok, pos, 1, lg_r.ctypes.data_as(C.c_void_p)) == 0
        lg_o = om.forward(tok, pos, 1)
        assert np.max(np.abs(lg_o - lg_r)) <= 5e-4, f"position {pos}"
        assert int(np.argmax(lg_o)) == int(np.argmax(lg_r))
    L.xref_free(h)
    om.close()
