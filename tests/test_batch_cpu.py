"""Batched decode entry points without a GPU: argument validation, and no CPU fallback."""
import ctypes as C

import numpy as np
import pytest

from xalm_b200 import capi
from xalm_b200 import types as T


def _has_gpu():
    n = C.c_int(0)
    return capi.lib().xalm_cuda_device_count(C.byref(n)) == 0 and n.value > 0


def _ints(*v):
    return (C.c_int * len(v))(*v)


def test_batch_entry_points_refuse_a_null_handle():
    L = capi.lib()
    one = _ints(0)
    assert L.xalm_cuda_set_batch(None, 4) == 1
    assert L.xalm_cuda_select_seq(None, 0) == 1
    assert L.xalm_cuda_forward_batch(None, 1, one, one, one, 1, None) == 1
    assert L.xalm_cuda_forward_batch_async(None, 1, one, one, one, 1) == 1
    assert L.xalm_cuda_forward_batch_argmax(None, 1, one, one, one, None) == 1
    from xalm_b200.model import Model
    with pytest.raises(ValueError):
        Model._batch_args([0, 1], [5], [0, 0])       # the Python binding checks the lengths before calling in


def test_bench_matvec_batch_validates_arguments():
    L = capi.lib()
    ms = C.c_float(0)
    bad = [
        (T.Q8_0.id, 4096, 4096, 0, 0, 0, 1, 1),     # no sequences
        (T.Q8_0.id, 4096, 4096, 0, 0, 9, 1, 1),     # more than 8
        (T.Q8_0.id, 4080, 4096, 0, 0, 2, 1, 1),     # n % 32
        (T.Q8_0.id, 4096, 4096, 3, 0, 2, 1, 1),     # no QKV epilogue in the bench
        (T.Q8_0.id, 4096, 4096, 0, 0, 2, 0, 1),     # no buffers
    ]
    for args in bad:
        assert L.xalm_cuda_bench_matvec_batch(*args, C.byref(ms)) == 1, args
        if 1 <= args[5] <= 8:   # the batch-1 bench takes the same arguments without n_seqs, and checks them before the device
            assert L.xalm_cuda_bench_matvec(*args[:5], *args[6:], C.byref(ms)) == 1, args
    # formats the tensor-core kernel does not take are refused, not run another way
    for t in (T.F16, T.BF16, T.F32, T.TQ1_0, T.QI8):
        assert L.xalm_cuda_bench_matvec_batch(t.id, 4096, 4096, 0, 0, 2, 1, 1, C.byref(ms)) == 2, t.name
        assert b"batched matvec" in L.xalm_cuda_last_error()


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a box without a GPU")
def test_batch_paths_need_a_device():
    L = capi.lib()
    ms = C.c_float(0)
    assert L.xalm_cuda_bench_matvec_batch(T.Q4_0.id, 4096, 4096, 2, 1, 4, 1, 1, C.byref(ms)) == 3   # XALM_ERR_CUDA
