#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ from the REFERENCE's own executable Python.

Run in the dev container only (it needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

What it pins (SURVEY.md §8c — the reference has no tests of its own, so these are the only
executable pins there are):

  blocks_<fmt>.npz   /root/reference/quants.py quantize() and dequantize() for the six block formats
                     convert.py exposes (convert.py:55-61), on seeded gaussian rows AND on raw random
                     blocks (every nibble/byte code, random f16 scales incl. subnormals and negatives).
  fp8_codes.npz      all 256 codes of float8_e4m3fn / float8_e5m2 decoded by torch (what convert.py
                     writes, convert.py:162-167) + the values types.h:302-314 assigns to the NaN/Inf
                     codes it does not special-case.
  tiny_<type>.xalm   complete checkpoints written by /root/reference/convert.py from a synthetic HF
                     directory (config.json + tokenizer.json + model.safetensors), for
                     f16 / bf16 / q8_0 / q4_0 / f8_e4m3.
                     Their fp32 source weights are not stored: torch.Generator seed 1234 regenerates them
                     bit for bit (make_tiny_checkpoints).
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)

import quants  # noqa: E402  (the reference's module)
from quants import GGMLQuantizationType as Q  # noqa: E402

FORMATS = {"q4_0": Q.Q4_0, "q4_1": Q.Q4_1, "q5_0": Q.Q5_0, "q5_1": Q.Q5_1, "q8_0": Q.Q8_0, "tq1_0": Q.TQ1_0}


def random_scales_f16(rng, n):
    """random finite f16 bit patterns (no Inf/NaN): all exponents 0..30, both signs, subnormals included"""
    bits = rng.integers(0, 1 << 16, size=n, dtype=np.uint16)
    exp = (bits >> 10) & 0x1F
    bits = np.where(exp == 31, bits & np.uint16(0xBFFF), bits).astype(np.uint16)
    return bits


def make_blocks():
    rng = np.random.default_rng(20241018)
    for name, qt in FORMATS.items():
        bs, ts = quants.GGML_QUANT_SIZES[qt]
        # (1) quantize path: gaussian rows like real weights + a few adversarial rows
        cols = 512
        x = (rng.standard_normal((12, cols)) * 0.02).astype(np.float32)
        x[1] *= 50.0
        x[2] = 0.0                      # all-zero blocks (d == 0 branch)
        x[3, ::2] = 0.0
        x[4] = np.round(x[4] * 400) / 400  # many ties
        x[5, :32] = np.linspace(-1, 1, 32, dtype=np.float32)
        x[6] = np.abs(x[6])             # one-sided blocks (min > 0 for the *_1 formats)
        x[7] = -np.abs(x[7])
        qbytes = quants.quantize(x, qt)
        deq = quants.dequantize(qbytes, qt)
        # (2) raw random blocks: exercise every code point of the decoder
        n_raw = 256
        raw = rng.integers(0, 256, size=(n_raw, ts), dtype=np.uint8)
        scales = random_scales_f16(rng, n_raw * 2).view(np.uint8).reshape(n_raw, 4)
        if name == "tq1_0":
            raw[:, 52:54] = scales[:, :2]
        else:
            raw[:, 0:2] = scales[:, :2]
            if name in ("q4_1", "q5_1"):
                raw[:, 2:4] = scales[:, 2:4]
        raw_rows = raw.reshape(4, -1)   # 4 rows of 64 blocks
        raw_deq = quants.dequantize(raw_rows, qt)
        np.savez_compressed(os.path.join(HERE, f"blocks_{name}.npz"), x=x, qbytes=qbytes, deq=deq, raw=raw_rows,
                            raw_deq=raw_deq, block=np.int32(bs), type_size=np.int32(ts))
        print(f"blocks_{name}.npz: q {qbytes.shape} raw {raw_rows.shape}")


def make_fp8():
    import torch
    codes = torch.arange(256, dtype=torch.uint8)
    e4m3 = codes.view(torch.float8_e4m3fn).to(torch.float32).numpy()
    e5m2 = codes.view(torch.float8_e5m2).to(torch.float32).numpy()
    # what types.h:302-314 computes for the codes torch decodes to NaN/Inf: (1+m/2^M) * 2^(e-bias)
    def ref_rule(code, E, M):
        s = -1.0 if code & 0x80 else 1.0
        e = (code & 0x7F) >> M
        m = code & ((1 << M) - 1)
        bias = (1 << (E - 1)) - 1
        return np.float32(s * (1.0 + m / (1 << M)) * 2.0 ** (e - bias)) if e else np.float32(s * (m / (1 << M)) * 2.0 ** (1 - bias))
    e4m3_ref = e4m3.copy()
    e5m2_ref = e5m2.copy()
    for c in range(256):
        if not np.isfinite(e4m3[c]):
            e4m3_ref[c] = ref_rule(c, 4, 3)
        if not np.isfinite(e5m2[c]):
            e5m2_ref[c] = ref_rule(c, 5, 2)
    np.savez_compressed(os.path.join(HERE, "fp8_codes.npz"), e4m3_torch=e4m3, e5m2_torch=e5m2, e4m3_ref=e4m3_ref,
                        e5m2_ref=e5m2_ref)
    print("fp8_codes.npz: non-finite torch codes:", int((~np.isfinite(e4m3)).sum()), int((~np.isfinite(e5m2)).sum()))


TINY = dict(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
            vocab_size=288, max_position_embeddings=64, bos_token_id=1, eos_token_id=2, rope_theta=10000.0,
            rms_norm_eps=1e-5, tie_word_embeddings=False, hidden_act="silu", architectures=["MistralForCausalLM"])


def make_tiny_checkpoints():
    import torch
    from safetensors.torch import save_file
    tmp = tempfile.mkdtemp(prefix="xalm_golden_")
    try:
        with open(os.path.join(tmp, "config.json"), "w") as f:
            json.dump(TINY, f)
        vocab = {"<unk>": 0, "<s>": 1, "</s>": 2}
        for b in range(256):
            vocab[f"<0x{b:02X}>"] = 3 + b
        words = ["▁", "▁the", "▁a", "e", "t", "▁Q", ":", "▁What", "▁is", "▁meaning", "▁of",
                 "▁life", "?", "▁A", "in", "er", "th", "▁▁", "an", "on", "re", "at", "en", "or", "es", "is",
                 "it", "ing", "▁of▁the"]
        for i, w in enumerate(words):
            vocab[w] = 259 + i
        with open(os.path.join(tmp, "tokenizer.json"), "w") as f:
            json.dump({"model": {"vocab": vocab, "byte_fallback": True}, "added_tokens": []}, f)
        g = torch.Generator().manual_seed(1234)
        d, h, L = TINY["hidden_size"], TINY["intermediate_size"], TINY["num_hidden_layers"]
        nh, nkv = TINY["num_attention_heads"], TINY["num_key_value_heads"]
        hd = d // nh
        w = {}
        def rnd(*shape, std=0.05):
            return torch.randn(*shape, generator=g) * std
        w["model.embed_tokens.weight"] = rnd(TINY["vocab_size"], d, std=0.5)
        w["lm_head.weight"] = rnd(TINY["vocab_size"], d, std=0.1)
        w["model.norm.weight"] = 1.0 + rnd(d, std=0.1)
        for l in range(L):
            p = f"model.layers.{l}."
            w[p + "input_layernorm.weight"] = 1.0 + rnd(d, std=0.1)
            w[p + "post_attention_layernorm.weight"] = 1.0 + rnd(d, std=0.1)
            w[p + "self_attn.q_proj.weight"] = rnd(nh * hd, d, std=0.1)
            w[p + "self_attn.k_proj.weight"] = rnd(nkv * hd, d, std=0.1)
            w[p + "self_attn.v_proj.weight"] = rnd(nkv * hd, d, std=0.1)
            w[p + "self_attn.o_proj.weight"] = rnd(d, nh * hd, std=0.1)
            w[p + "mlp.gate_proj.weight"] = rnd(h, d, std=0.1)
            w[p + "mlp.up_proj.weight"] = rnd(h, d, std=0.1)
            w[p + "mlp.down_proj.weight"] = rnd(d, h, std=0.1)
        w = {k: v.contiguous() for k, v in w.items()}
        save_file(w, os.path.join(tmp, "model.safetensors"))
        for t in ["f16", "bf16", "q8_0", "q4_0", "f8_e4m3"]:
            out = os.path.join(HERE, f"tiny_{t}.xalm")
            r = subprocess.run([sys.executable, os.path.join(REF, "convert.py"), "--input", tmp, "--type", t, "--output", out],
                               cwd=REF, capture_output=True, text=True)
            if r.returncode != 0:
                print(r.stdout[-2000:], r.stderr[-2000:])
                raise SystemExit(f"convert.py failed for {t}")
            print(f"tiny_{t}.xalm: {os.path.getsize(out)} bytes")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    make_blocks()
    make_fp8()
    make_tiny_checkpoints()
