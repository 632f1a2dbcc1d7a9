"""ctypes binding of the C ABI in include/xalm_cuda.h (libxalm_cuda.so).

Fails loudly: if the shared library is missing it is (re)built with nvcc; if that is impossible, or no CUDA
device is present, the calls raise — there is no CPU or PyTorch fallback behind this module.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

HYDRATE_KV_CACHE, OUTPUT_LOGITS = 0, 1          # InferenceMode, model.h:249-252
GELU, SILU = 0, 1                               # ActivationType, model.h:12-15
S_X, S_XB2, S_HB, S_Q, S_LOGITS = 0, 2, 3, 5, 9


class XalmError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"xalm_cuda status {status}: {msg}")
        self.status = status


class XalmConfig(C.Structure):
    # xalm_config (include/xalm_cuda.h) == Config (model.h:25-42)
    _fields_ = [("dim", C.c_int), ("hidden_dim", C.c_int), ("head_dim", C.c_int), ("n_layers", C.c_int),
                ("n_heads", C.c_int), ("n_kv_heads", C.c_int), ("vocab_size", C.c_int), ("max_seq_len", C.c_int),
                ("rope_theta", C.c_float), ("rotary_dim", C.c_int), ("norm_eps", C.c_float), ("act", C.c_int),
                ("norm_type", C.c_int), ("qkv_clip", C.c_float), ("tie_word_embeddings", C.c_int)]

    @classmethod
    def from_dict(cls, c: dict) -> "XalmConfig":
        return cls(c["dim"], c["hidden_dim"], c["head_dim"], c["n_layers"], c["n_heads"], c["n_kv_heads"], c["vocab_size"],
                   c["max_seq_len"], c["rope_theta"], c["rotary_dim"], c["norm_eps"], c["act"], c.get("norm_type", 0),
                   c.get("qkv_clip", float(np.finfo(np.float32).max)), int(c["tie_word_embeddings"]))


# every symbol include/xalm_cuda.h declares: (restype, argtypes)
_vp, _i, _sz, _fp = C.c_void_p, C.c_int, C.c_size_t, C.POINTER(C.c_float)
SYMBOLS = {
    "xalm_cuda_abi_version": (_i, []),
    "xalm_cuda_last_error": (C.c_char_p, []),
    "xalm_cuda_device_count": (_i, [C.POINTER(_i)]),
    "xalm_cuda_type_info": (_i, [_i, C.POINTER(_i), C.POINTER(_i)]),
    "xalm_cuda_create": (_i, [C.POINTER(XalmConfig), _i, _i, _i, C.POINTER(_vp)]),
    "xalm_cuda_upload_tensor": (_i, [_vp, C.c_char_p, _i, C.POINTER(_i), _i, _vp, _sz]),
    "xalm_cuda_host_alloc": (_vp, [_sz]),
    "xalm_cuda_host_free": (None, [_vp]),
    "xalm_cuda_shard_range": (_i, [_vp, C.c_char_p, C.POINTER(_i)]),
    "xalm_cuda_upload_tensor_shard": (_i, [_vp, C.c_char_p, _i, C.POINTER(_i), _i, C.POINTER(_i), _vp, _sz]),
    "xalm_cuda_finalize": (_i, [_vp]),
    "xalm_cuda_destroy": (None, [_vp]),
    "xalm_cuda_comm_unique_id": (_i, [_vp]),
    "xalm_cuda_comm_init": (_i, [_vp, _vp]),
    "xalm_cuda_ipc_export": (_i, [_vp, _vp]),
    "xalm_cuda_ipc_import": (_i, [_vp, _vp]),
    "xalm_cuda_set_stream": (_i, [_vp, _vp]),
    "xalm_cuda_forward": (_i, [_vp, _i, _i, _i, _vp]),
    "xalm_cuda_forward_async": (_i, [_vp, _i, _i, _i]),
    "xalm_cuda_forward_argmax": (_i, [_vp, _i, _i, C.POINTER(_i)]),
    "xalm_cuda_forward_greedy": (_i, [_vp, _i, _vp, _i, _i, _vp]),
    "xalm_cuda_sync": (_i, [_vp]),
    "xalm_cuda_logits_host": (_fp, [_vp]),
    "xalm_cuda_active_bytes": (_i, [_vp, C.c_longlong, C.POINTER(C.c_longlong)]),
    "xalm_cuda_last_launch_count": (_i, [_vp, C.POINTER(_i)]),
    "xalm_cuda_read_state": (_i, [_vp, _i, _vp, _sz]),
    "xalm_cuda_read_kv": (_i, [_vp, _i, _i, _vp, _sz]),
    "xalm_cuda_dequant": (_i, [_i, _vp, _sz, _vp]),
    "xalm_cuda_matmul": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "xalm_cuda_mha": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i]),
    "xalm_cuda_rmsnorm": (_i, [_vp, _vp, _vp, _i, _i, C.c_float]),
    "xalm_cuda_rope": (_i, [_vp, _i, _i, _i, C.c_float, _i]),
    "xalm_cuda_ffn": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i]),
    "xalm_cuda_tune": (_i, [C.c_char_p, _i]),
    "xalm_cuda_timeline": (_i, [_i, _vp, C.POINTER(_i)]),
    "xalm_cuda_bench_matvec": (_i, [_i, _i, _i, _i, _i, _i, _i, _fp]),
    "xalm_cuda_prefill": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "xalm_cuda_prefill_window": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "xalm_cuda_prefill_async": (_i, [_vp, _vp, _i, _i, _i]),
    "xalm_cuda_gemm": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i]),
    "xalm_cuda_bench_gemm": (_i, [_i, _i, _i, _i, _i, _fp]),
    "xalm_cuda_set_batch": (_i, [_vp, _i]),
    "xalm_cuda_forward_batch": (_i, [_vp, _i, _vp, _vp, _vp, _i, _vp]),
    "xalm_cuda_forward_batch_argmax": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "xalm_cuda_forward_batch_async": (_i, [_vp, _i, _vp, _vp, _vp, _i]),
    "xalm_cuda_forward_spans": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "xalm_cuda_forward_spans_argmax": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "xalm_cuda_forward_tree": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp]),
    "xalm_cuda_forward_tree_argmax": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp]),
    "xalm_cuda_tree_accept": (_i, [_vp, _i, _i, _i, _vp]),
    "xalm_cuda_select_seq": (_i, [_vp, _i]),
    "xalm_cuda_bench_matvec_batch": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, _fp]),
}

_LIB = None


def lib_path() -> str:
    return _build.LIB


def lib():
    """Load (building first if needed) libxalm_cuda.so and type every entry point."""
    global _LIB
    if _LIB is None:
        path = _build.LIB
        if not os.path.exists(path):
            _build.build_cuda()
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)          # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(status: int):
    if status != 0:
        raise XalmError(status, lib().xalm_cuda_last_error().decode("utf-8", "replace"))


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def device_count() -> int:
    n = C.c_int(0)
    check(lib().xalm_cuda_device_count(C.byref(n)))
    return n.value


def tune(key: str, value: int):
    check(lib().xalm_cuda_tune(key.encode(), int(value)))


# ---- op-level entry points -----------------------------------------------------------------------------------
def dequant(type_id: int, raw: np.ndarray, n_elems: int) -> np.ndarray:
    raw = np.ascontiguousarray(raw)
    out = np.empty(n_elems, dtype=np.float32)
    check(lib().xalm_cuda_dequant(type_id, _p(raw), n_elems, _p(out)))
    return out


def matmul(x: np.ndarray, w_raw: np.ndarray, type_id: int, n: int, d: int) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32)
    w_raw = np.ascontiguousarray(w_raw)
    out = np.empty(d, dtype=np.float32)
    check(lib().xalm_cuda_matmul(_p(out), _p(x), _p(w_raw), type_id, n, d))
    return out


def mha(q, kb, vb, head_dim, kv_len, max_seq_len, n_heads, n_kv_heads, want_att=False):
    q = np.ascontiguousarray(q, dtype=np.float32)
    kb, vb = np.ascontiguousarray(kb), np.ascontiguousarray(vb)
    out = np.empty(n_heads * head_dim, dtype=np.float32)
    att = np.zeros(n_heads * max_seq_len, dtype=np.float32) if want_att else None
    check(lib().xalm_cuda_mha(_p(out), _p(att) if want_att else None, _p(kb), _p(vb), _p(q), head_dim, kv_len, max_seq_len,
                              n_heads, n_kv_heads))
    return (out, att) if want_att else out


def rmsnorm(x, w_raw, wtype, eps):
    x = np.ascontiguousarray(x, dtype=np.float32)
    w_raw = np.ascontiguousarray(w_raw)
    out = np.empty_like(x)
    check(lib().xalm_cuda_rmsnorm(_p(out), _p(x), _p(w_raw), wtype, x.size, eps))
    return out


def rope(vec, head_dim, pos, theta, rotary_dim):
    v = np.array(vec, dtype=np.float32, copy=True)
    check(lib().xalm_cuda_rope(_p(v), v.size, head_dim, pos, theta, rotary_dim))
    return v


def ffn(x, w1, w2, w3, type_id, hidden_dim, dim, act):
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty(dim, dtype=np.float32)
    check(lib().xalm_cuda_ffn(_p(out), _p(x), _p(np.ascontiguousarray(w1)), _p(np.ascontiguousarray(w2)),
                              _p(np.ascontiguousarray(w3)), type_id, hidden_dim, dim, act))
    return out


def timeline_start(n_records: int):
    check(lib().xalm_cuda_timeline(n_records, None, None))


def timeline_stop(n_records: int) -> np.ndarray:
    out = np.zeros((n_records, 4), dtype=np.uint64)
    n = C.c_int(0)
    check(lib().xalm_cuda_timeline(n_records, _p(out), C.byref(n)))
    return out[: n.value]


def bench_matvec(type_id: int, n: int, d: int, n_buffers: int, iters: int, epi: int = 0, with_norm: bool = False) -> float:
    ms = C.c_float(0)
    check(lib().xalm_cuda_bench_matvec(type_id, n, d, epi, int(with_norm), n_buffers, iters, C.byref(ms)))
    return ms.value


def bench_matvec_batch(type_id: int, n: int, d: int, n_seqs: int, n_buffers: int, iters: int, epi: int = 0, with_norm: bool = False) -> float:
    """bench_matvec for the batched tensor-core matvec (activation quantiser + matvec) at n_seqs sequences."""
    ms = C.c_float(0)
    check(lib().xalm_cuda_bench_matvec_batch(type_id, n, d, epi, int(with_norm), n_seqs, n_buffers, iters, C.byref(ms)))
    return ms.value


def gemm(a: np.ndarray, w_raw: np.ndarray, type_id: int, K: int, N: int, split: int = 1) -> np.ndarray:
    """out(T,N) = a(T,K) . W(N,K)^T on the tensor-core path."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    T = a.shape[0]
    w_raw = np.ascontiguousarray(w_raw)
    out = np.empty((T, N), dtype=np.float32)
    check(lib().xalm_cuda_gemm(_p(out), _p(a), _p(w_raw), type_id, T, K, N, split))
    return out


def bench_gemm(T: int, N: int, K: int, split: int = 1, iters: int = 20) -> float:
    ms = C.c_float(0)
    check(lib().xalm_cuda_bench_gemm(T, N, K, split, iters, C.byref(ms)))
    return ms.value
