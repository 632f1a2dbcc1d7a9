"""Full forward parity: the CUDA backend behind Model/InferenceState vs the CPU oracle on identical checkpoints —
token-exact greedy decoding, logits within max-abs 1e-2, fp16 KV cache, ring buffer + attention sinks, modes."""
import os

import numpy as np
import pytest

from oracle import oracle
from xalm_b200 import capi, synth
from xalm_b200 import types as T
from xalm_b200.model import InferenceState, Model, Sampler

from gpu_util import LOGIT_TOL, greedy_compare, load_pair, synth_pair

pytestmark = pytest.mark.gpu

PROMPT = [1, 84, 61, 35, 90, 107, 100, 119]


@pytest.mark.parametrize("t", ["f16", "bf16", "q8_0", "q4_0", "f8_e4m3"])
def test_convert_py_checkpoints_greedy_parity(golden_dir, t):
    """Checkpoints written by the reference's own convert.py; 40 greedy tokens."""
    config, om, gm = load_pair(os.path.join(golden_dir, f"tiny_{t}.xalm"))
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, [1, 266, 267, 268, 269], 40)
    assert maxdiff <= LOGIT_TOL, f"logits differ by {maxdiff}"
    assert otoks == gtoks, f"greedy tokens diverge (min top-2 margin {margin})"
    gm.close(); om.close()


@pytest.mark.parametrize("wtype", ["f32", "f16", "bf16", "f8_e4m3", "f8_e5m2", "q8", "q8_0", "q4_0", "q4_1", "q5_0", "q5_1", "tq1_0", "qi8"])
def test_every_weight_format_full_model(wtype):
    config, om, gm = synth_pair("tiny", wtype, seed=2, std=0.06)
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, PROMPT, 24)
    assert maxdiff <= LOGIT_TOL, f"{wtype}: logits differ by {maxdiff}"
    assert otoks == gtoks, f"{wtype}: greedy tokens diverge (min margin {margin})"
    gm.close(); om.close()


def test_ring_buffer_and_attention_sinks(golden_dir):
    """-T 6: from pos 6 on the KV cache is a ring with 2 sinks that are re-rotated every step through fp16
    (infer.cpp:416-431, 608-613)."""
    config, om, gm = load_pair(os.path.join(golden_dir, "tiny_f16.xalm"), context=6)
    assert config["max_seq_len"] == 6
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, [1, 266, 267], 30)
    assert maxdiff <= LOGIT_TOL
    assert otoks == gtoks
    # the caches themselves: same fp16 bits except where a 1-ulp fp32 libm difference crosses a rounding boundary
    for layer in range(config["n_layers"]):
        for which in (0, 1):
            a = gm.read_kv(layer, which).view(np.float16).astype(np.float32)
            b = om.kv(layer, which).view(np.float16).astype(np.float32)
            assert np.max(np.abs(a - b)) <= 2e-3 * max(1.0, np.abs(b).max())
            assert np.mean(a != b) < 0.02
    gm.close(); om.close()


def test_hydrate_mode_and_state_buffers():
    config, om, gm = synth_pair("tiny", "q8_0", seed=4, std=0.06)
    state = InferenceState(config)
    state.logits()[:] = -7.0
    for pos, tok in enumerate(PROMPT):
        om.forward(tok, pos, 0)
        gm.forward(state, tok, pos, 0)          # HYDRATE_KV_CACHE: no classifier, logits untouched (infer.cpp:620-623)
    assert np.all(state.logits() == -7.0)
    x_g = gm.read_state(capi.S_X, config["dim"])
    x_o = om.state(0, config["dim"])
    assert np.max(np.abs(x_g - x_o)) <= 1e-3 * max(1.0, np.abs(x_o).max())
    lg_o = om.forward(5, len(PROMPT), 1)
    gm.forward(state, 5, len(PROMPT), 1)
    assert np.max(np.abs(state.logits() - lg_o)) <= LOGIT_TOL
    assert np.array_equal(gm.read_state(capi.S_LOGITS, config["vocab_size"]), state.logits())
    # launches per token: embed + 5 fused kernels per layer + classifier
    assert gm.last_launch_count() == 1 + 5 * config["n_layers"] + 1
    gm.close(); om.close()


def test_graph_and_pdl_do_not_change_results():
    outs = {}
    for graph, pdl in ((1, 1), (0, 1), (1, 0), (0, 0)):
        capi.tune("graph", graph); capi.tune("pdl", pdl)
        config, om, gm = synth_pair("tiny", "q4_0", seed=6, std=0.06)
        state = InferenceState(config)
        seq = []
        for pos, tok in enumerate(PROMPT + [7, 9, 300, 2]):
            gm.forward(state, tok, pos, 1)
            seq.append(state.logits().copy())
        outs[(graph, pdl)] = np.stack(seq)
        gm.close(); om.close()
    capi.tune("graph", 1); capi.tune("pdl", 1)
    base = outs[(1, 1)]
    for k, v in outs.items():
        assert np.array_equal(base, v), f"graph/pdl={k} changed the logits"


def test_gelu_tied_embeddings_partial_rotary_and_clip():
    config, om, gm = synth_pair("tiny", "f16", seed=8, std=0.06, act_type="gelu", tie_word_embeddings=True, rotary_dim=32)
    assert config["act"] == 0 and config["tie_word_embeddings"] and config["rotary_dim"] == 32
    otoks, gtoks, maxdiff, _ = greedy_compare(config, om, gm, PROMPT, 16)
    assert maxdiff <= LOGIT_TOL and otoks == gtoks
    gm.close(); om.close()


def test_finite_qkv_clip():
    """qkv_clip = 0.5 with q/k/v entries of ~1: the clamp of infer.cpp:388-399 is active on most rows."""
    config, om, gm = synth_pair("tiny", "q8_0", seed=9, std=0.06, qkv_clip=0.5)
    assert config["qkv_clip"] == 0.5
    otoks, gtoks, maxdiff, _ = greedy_compare(config, om, gm, PROMPT, 16)
    assert maxdiff <= LOGIT_TOL and otoks == gtoks
    q = gm.read_state(capi.S_Q, config["n_heads"] * config["head_dim"])
    assert np.max(np.abs(q)) <= 0.5 * np.sqrt(2) + 1e-6 and np.max(np.abs(q)) > 0.45      # clipped, then rotated pairwise
    gm.close(); om.close()
    # and the unclipped model gives different tokens / logits, i.e. the clip was not a no-op
    config2, om2, gm2 = synth_pair("tiny", "q8_0", seed=9, std=0.06)
    st = InferenceState(config2)
    gm2.forward(st, PROMPT[0], 0, 1)
    assert np.max(np.abs(gm2.read_state(capi.S_Q, config2["n_heads"] * config2["head_dim"]))) > 0.75
    gm2.close(); om2.close()


def test_small_model_longer_context():
    """GQA 8:2, head_dim 128, 4 layers, 200 positions: exercises multi-split attention inside the model path."""
    config, om, gm = synth_pair("small", "q8_0", seed=1, std=0.03)
    prompt = list(np.random.default_rng(0).integers(3, config["vocab_size"], size=180))
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, [int(t) for t in prompt], 24)
    assert maxdiff <= LOGIT_TOL
    assert otoks == gtoks, f"min margin {margin}"
    gm.close(); om.close()


def test_load_time_errors_mirror_the_reference():
    c = synth.model_config("tiny")
    from xalm_b200 import xalm_file as X
    cfg = X.parse_config(synth.metadata_strings(c))
    tensors = list(synth.iter_tensors(c, T.F16, 0))
    # missing tensor -> finalize fails (std::map::at throws in model.cpp:63)
    m = Model.from_tensors(cfg, [t for t in tensors if t[0] != "l.1.mlp.up.weight"])
    with pytest.raises(capi.XalmError) as e:
        m.cuda()
    assert "l.1.mlp.up" in str(e.value)
    # shape mismatch (model.cpp:66-75)
    m = Model.from_tensors(cfg, tensors)
    t, shape, raw = m.tensors["l.0.attn.k.weight"]
    m.tensors["l.0.attn.k.weight"] = (t, (shape[0] * 2, shape[1] // 2), raw)
    with pytest.raises(capi.XalmError) as e:
        m.cuda()
    assert "shape mismatch for l.0.attn.k.weight" in str(e.value)
    # rmsnorm weight must be F32/BF16 (infer.cpp:248-249)
    m = Model.from_tensors(cfg, tensors)
    t, shape, raw = m.tensors["output.norm.weight"]
    m.tensors["output.norm.weight"] = (T.F16, shape, raw[: shape[0] * 2])
    with pytest.raises(capi.XalmError):
        m.cuda()
    # token out of range
    m = Model.from_tensors(cfg, tensors).cuda()
    with pytest.raises(capi.XalmError):
        m.forward(InferenceState(cfg), cfg["vocab_size"], 0)
    m.close()


def test_sampler_quirk_on_device_logits():
    """sampler.cpp seeds its max with FLT_MIN: all-non-positive logits -> token 0."""
    cfg = {"vocab_size": 8}
    st = InferenceState(cfg)
    st.logits()[:] = [-1, -2, -0.5, -3, -4, -5, -6, -7]
    assert Sampler(cfg).sample_argmax(st) == 0 == oracle.sample_argmax(st.logits())
    st.logits()[3] = 0.25
    assert Sampler(cfg).sample_argmax(st) == 3
    assert abs(Sampler(cfg).sample_prob(3, st) - oracle.sample_prob(st.logits(), 3)) < 1e-6


@pytest.mark.parametrize("shape,wtype,layers", [("l70", "q8_0", 1), ("l8", "q4_0", 2)])
def test_baseline_shapes_depth_reduced(shape, wtype, layers):
    """BASELINE configs 4/5 at reduced depth (SURVEY.md §7 '70B parity'): Llama-70B dims (8192/28672, 64 q heads on 8 kv heads,
    128k vocab) and Llama-8B dims, full width — exercises GQA 8:1, 28672-long rows (activations read through L1), big vocab."""
    config, om, gm = synth_pair(shape, wtype, seed=3, std=0.02, n_layers=layers)
    prompt = [int(t) for t in np.random.default_rng(1).integers(3, config["vocab_size"], size=6)]
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, prompt, 4)
    assert maxdiff <= LOGIT_TOL, f"{shape}: logits differ by {maxdiff}"
    assert otoks == gtoks, f"{shape}: greedy tokens diverge (min margin {margin})"
    gm.close(); om.close()


def test_full_size_mistral_7b_q8_0_parity():
    """BASELINE config 2 at FULL size (32 layers, 7.2 B weights, q8_0): the CPU oracle manages ~8 tok/s on the GPU box's
    cores, so direct parity is affordable: 4 prompt tokens + 12 greedy steps, token-exact, logits within 1e-2, and the
    ring/sink path exercised right after (-T is not needed: positions stay < 4096)."""
    config, om, gm = synth_pair("m7", "q8_0", seed=0, std=0.02)
    assert config["max_seq_len"] == 4096 and config["n_layers"] == 32
    otoks, gtoks, maxdiff, margin = greedy_compare(config, om, gm, [1, 415, 28747, 1824], 12)
    assert maxdiff <= LOGIT_TOL, f"logits differ by {maxdiff}"
    assert otoks == gtoks, f"greedy tokens diverge (min margin {margin})"
    # algorithmic bytes: Model::active_bytes == SURVEY.md §8d formula (7.555 GB + 0.131 MB per cached position)
    from xalm_b200.model import active_bytes_formula
    assert gm.active_bytes(0) == active_bytes_formula(config, 34 / 32, 0) == om.active_bytes(0)
    assert abs(gm.active_bytes(0) / 1e9 - 7.555) < 0.01
    gm.close(); om.close()


def test_device_sampler_matches_host_sampler():
    """xalm_cuda_forward_argmax == Model.forward + Sampler.sample_argmax (incl. first-maximum-wins), greedy loop of 24 tokens."""
    config, om, gm = synth_pair("tiny", "q8_0", seed=21, std=0.06)
    state, sampler = InferenceState(config), Sampler(config)
    tok_h = tok_d = 5
    for pos in range(24):
        gm.forward(state, tok_h, pos, 1)
        nxt_h = sampler.sample_argmax(state)
        nxt_d = gm.forward_argmax(tok_h, pos)      # same input token: the KV row is simply rewritten with the same values
        assert nxt_d == nxt_h == oracle.sample_argmax(om.forward(tok_h, pos, 1))
        tok_h = nxt_h
    gm.close(); om.close()
