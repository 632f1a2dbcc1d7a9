"""Synthetic random-init checkpoints for the BASELINE configs (SURVEY.md §8d).

Weights ~ N(0, 0.02^2) from a counter-based generator (seeded, thread-count independent), norm weights 1.0,
a byte-fallback tokenizer, cast/quantised to the requested format by the host library's writers
(csrc/host/quantize.cpp — byte-identical to the reference's quants.py, see tests/test_quantize.py).
Must run on the GPU box, which has neither the reference tree nor room to ship 7B-70B files.
"""
from __future__ import annotations

import ctypes as C
import os
import zlib
from collections import OrderedDict

import numpy as np

from . import build as _build
from . import types as T
from . import xalm_file as X

_HOST = None

SHAPES = {
    # Mistral-7B-v0.2 (BASELINE configs 1-3)
    "m7": dict(dim=4096, hidden_dim=14336, head_dim=128, n_layers=32, n_heads=32, n_kv_heads=8, vocab_size=32000,
               max_seq_len=32768, rope_theta=1000000.0, arch="MistralForCausalLM"),
    # Llama-3-8B style (config 4)
    "l8": dict(dim=4096, hidden_dim=14336, head_dim=128, n_layers=32, n_heads=32, n_kv_heads=8, vocab_size=128256,
               max_seq_len=8192, rope_theta=500000.0, arch="LlamaForCausalLM"),
    # Llama-3-70B style (config 5)
    "l70": dict(dim=8192, hidden_dim=28672, head_dim=128, n_layers=80, n_heads=64, n_kv_heads=8, vocab_size=128256,
                max_seq_len=8192, rope_theta=500000.0, arch="LlamaForCausalLM"),
    # TinyLlama-1.1B, a draft model for m7 (same vocabulary size); context 4096 rather than 2048 so that it drafts across m7's
    # default window
    "d1": dict(dim=2048, hidden_dim=5632, head_dim=64, n_layers=22, n_heads=32, n_kv_heads=4, vocab_size=32000,
               max_seq_len=4096, rope_theta=10000.0, arch="LlamaForCausalLM"),
    # small shapes for tests / smoke
    "tiny": dict(dim=256, hidden_dim=512, head_dim=64, n_layers=2, n_heads=4, n_kv_heads=2, vocab_size=512,
                 max_seq_len=128, rope_theta=10000.0, arch="MistralForCausalLM"),
    # every per-rank dimension stays a multiple of 256 up to TP=4 (the fused exchange rides on the TMA matvec kernels)
    "tp": dict(dim=1024, hidden_dim=3072, head_dim=128, n_layers=4, n_heads=8, n_kv_heads=4, vocab_size=4096,
               max_seq_len=1024, rope_theta=10000.0, arch="LlamaForCausalLM"),
    # TP=8: one kv head and 256 q / 768 hidden / 512 vocab columns per rank
    "tp8": dict(dim=2048, hidden_dim=6144, head_dim=128, n_layers=2, n_heads=16, n_kv_heads=8, vocab_size=4096,
                max_seq_len=512, rope_theta=10000.0, arch="LlamaForCausalLM"),
    "small": dict(dim=1024, hidden_dim=2816, head_dim=128, n_layers=4, n_heads=8, n_kv_heads=2, vocab_size=4096,
                  max_seq_len=1024, rope_theta=10000.0, arch="LlamaForCausalLM"),
}


def host():
    global _HOST
    if _HOST is None:
        if not os.path.exists(_build.HOSTLIB):
            _build.build_host()
        L = C.CDLL(_build.HOSTLIB)
        L.xalm_host_quantize.argtypes = [C.c_int, C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p]
        L.xalm_host_normal.argtypes = [C.c_uint64, C.c_uint64, C.c_longlong, C.c_float, C.c_float, C.c_void_p]
        L.xalm_host_normal.restype = None
        L.xalm_host_normal_block.argtypes = [C.c_uint64, C.c_uint64, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong,
                                             C.c_float, C.c_float, C.c_void_p]
        L.xalm_host_set_threads.argtypes = [C.c_int]
        L.xalm_host_set_threads.restype = None
        _HOST = L
    return _HOST


def set_threads(n: int):
    host().xalm_host_set_threads(int(n))


def normal(seed: int, stream: int, n: int, std: float, mean: float = 0.0) -> np.ndarray:
    out = np.empty(n, dtype=np.float32)
    host().xalm_host_normal(seed, stream, n, mean, std, out.ctypes.data_as(C.c_void_p))
    return out


def normal_block(seed: int, stream: int, n_cols: int, r0: int, r1: int, c0: int, c1: int, std: float, mean: float = 0.0) -> np.ndarray:
    """Rows [r0, r1) x columns [c0, c1) of the (rows, n_cols) matrix normal(seed, stream, rows * n_cols, std) would give."""
    out = np.empty((r1 - r0, c1 - c0), dtype=np.float32)
    if host().xalm_host_normal_block(seed, stream, n_cols, r0, r1, c0, c1, mean, std, out.ctypes.data_as(C.c_void_p)):
        raise ValueError("normal_block: column bounds must be even")
    return out


def quantize(t: T.XType, x: np.ndarray) -> np.ndarray:
    """fp32 (rows, cols) -> on-disk bytes of type t as a uint8 array shaped like the .xalm header shape."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    rows, cols = (1, x.shape[0]) if x.ndim == 1 else x.shape
    if t in (T.F8_E4M3, T.F8_E5M2):
        import torch  # what convert.py does for fp8 (convert.py:162-167)
        dt = torch.float8_e4m3fn if t is T.F8_E4M3 else torch.float8_e5m2
        return torch.from_numpy(x).to(dt).view(torch.uint8).numpy().reshape(x.shape)
    if t is T.QI8:      # convert.py:538-543
        q = np.clip(np.round((np.clip(x, -1, 1) + np.float32(1.0)) * np.float32(127.5)), 0, 255).astype(np.uint8)
        return q
    out = np.empty(t.nbytes(rows * cols), dtype=np.uint8)
    rc = host().xalm_host_quantize(t.id, x.ctypes.data_as(C.c_void_p), rows, cols, out.ctypes.data_as(C.c_void_p))
    if rc:
        raise ValueError(f"cannot quantize shape {x.shape} to {t.name}")
    if t.block > 1:
        return out.reshape(t.byte_shape(x.shape))
    return out.view({4: np.float32, 2: np.uint16, 1: np.uint8}[t.bytes]).reshape(x.shape)


def byte_fallback_tokens(vocab_size: int) -> list:
    """<unk>, <s>, </s>, <0x00>..<0xFF>, then printable ASCII singles and a few words; the rest empty strings
    (tokenizer.h:21-45 describes the layout)."""
    toks = [b"<unk>", b"<s>", b"</s>"] + [f"<0x{b:02X}>".encode() for b in range(256)]
    extra = [bytes([c]) for c in range(32, 127)]
    extra += [b" the", b" of", b" is", b" What", b" meaning", b" life", b" Q", b" A", b"ing", b"er", b"in", b"an"]
    for e in extra:
        if len(toks) < vocab_size:
            toks.append(e)
    toks += [b""] * (vocab_size - len(toks))
    return toks[:vocab_size]


def model_config(shape: str, **over) -> dict:
    c = dict(SHAPES[shape])
    c.update(over)
    c.setdefault("rotary_dim", c["head_dim"])
    c.setdefault("norm_eps", 1e-5)
    c.setdefault("act_type", "silu")
    c.setdefault("tie_word_embeddings", False)
    c.setdefault("bos_token_id", 1)
    c.setdefault("eos_token_id", 2)
    return c


def metadata_strings(c: dict) -> OrderedDict:
    """The header "config" object exactly as Metadata.to_dict writes it (convert.py:223-245): all strings."""
    keys = ["dim", "hidden_dim", "head_dim", "n_layers", "n_heads", "n_kv_heads", "vocab_size", "max_seq_len",
            "bos_token_id", "eos_token_id", "rope_theta", "rotary_dim", "norm_eps"]
    md = OrderedDict((k, str(c[k])) for k in keys)
    md["norm_type"] = "rmsnorm"
    md["act_type"] = c["act_type"]
    md["tie_word_embeddings"] = str(bool(c["tie_word_embeddings"]))
    if "qkv_clip" in c:
        md["qkv_clip"] = str(c["qkv_clip"])   # optional key (model.h:84-85)
    return md


def iter_tensors(c: dict, wtype: T.XType, seed: int = 0, std: float = 0.02, norm_type: T.XType = T.F32,
                 embed_type: T.XType | None = None, shard_range=None):
    """Yield (name, XType, array-with-header-shape) in the order convert.py's load_weights emits them
    (convert.py:825-848).  Each tensor has its own RNG stream, so any subset can be generated on its own.
    shard_range(name) -> (r0, r1, c0, c1): generate and quantise only that block of every matrix (what a tensor-parallel
    rank keeps, xalm_cuda_shard_range) and yield (name, XType, block, (r0, r1, c0, c1)) — the same values the full tensor has
    there: rows are quantised independently and column bounds are multiples of 256, so no quant block is split."""
    q_dim, kv_dim = c["n_heads"] * c["head_dim"], c["n_kv_heads"] * c["head_dim"]
    embed_type = embed_type or wtype

    def w(name, rows, cols, t):
        if shard_range is not None:
            r0, r1, c0, c1 = shard_range(name)
            x = normal_block(seed, zlib.crc32(name.encode()), cols, r0, r1, c0, c1, std)
            return name, t, quantize(t, x), (r0, r1, c0, c1)
        x = normal(seed, zlib.crc32(name.encode()), rows * cols, std).reshape(rows, cols)
        return name, t, quantize(t, x)

    def ones(name):
        r = name, norm_type, quantize(norm_type, np.ones(c["dim"], dtype=np.float32))
        return r + ((0, c["dim"], 0, 1),) if shard_range is not None else r

    yield w("embed.weight", c["vocab_size"], c["dim"], embed_type)
    for l in range(c["n_layers"]):
        yield ones(f"l.{l}.attn.norm.weight")
        yield w(f"l.{l}.attn.q.weight", q_dim, c["dim"], wtype)
        yield w(f"l.{l}.attn.k.weight", kv_dim, c["dim"], wtype)
        yield w(f"l.{l}.attn.v.weight", kv_dim, c["dim"], wtype)
        yield w(f"l.{l}.attn.down.weight", c["dim"], q_dim, wtype)
        yield ones(f"l.{l}.mlp.norm.weight")
        yield w(f"l.{l}.mlp.gate.weight", c["hidden_dim"], c["dim"], wtype)
        yield w(f"l.{l}.mlp.down.weight", c["dim"], c["hidden_dim"], wtype)
        yield w(f"l.{l}.mlp.up.weight", c["hidden_dim"], c["dim"], wtype)
    if not c["tie_word_embeddings"]:
        yield w("output.weight", c["vocab_size"], c["dim"], embed_type)
    yield ones("output.norm.weight")


def write_checkpoint(path: str, shape: str, wtype: str, seed: int = 0, std: float = 0.02, **over) -> dict:
    """Write a complete .xalm (weights + tokenizer.tokens) for `shape` in format `wtype`; returns the config."""
    c = model_config(shape, **over)
    t = T.parse(wtype)
    tensors = OrderedDict()
    for name, xt, arr in iter_tensors(c, t, seed, std=std):
        tensors[name] = (xt.name.lower(), arr)
    toks = b"".join(tok + b"\x00" for tok in byte_fallback_tokens(c["vocab_size"]))
    tensors["tokenizer.tokens"] = ("u8", np.frombuffer(toks, dtype=np.uint8))
    X.write_xalm(path, c["arch"], metadata_strings(c), tensors)
    return c
