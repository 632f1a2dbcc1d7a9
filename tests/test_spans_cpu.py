"""Span entry points (speculative decoding) without a GPU: argument validation, and no CPU fallback."""
import ctypes as C

import pytest

from xalm_b200 import capi


def _ints(*v):
    return (C.c_int * len(v))(*v)


def test_span_entry_points_refuse_a_null_handle():
    L = capi.lib()
    one = _ints(0, 0)
    pos = _ints(3, 4)
    out = _ints(0, 0)
    assert L.xalm_cuda_forward_spans(None, 2, one, one, pos, None) == 1
    assert L.xalm_cuda_forward_spans_argmax(None, 2, one, one, pos, out) == 1
    assert b"NULL" in L.xalm_cuda_last_error()


def test_span_entry_points_refuse_null_arrays():
    L = capi.lib()
    one = _ints(0)
    assert L.xalm_cuda_forward_spans_argmax(None, 1, one, one, one, None) == 1       # no next_tokens
    assert b"next_tokens is NULL" in L.xalm_cuda_last_error()
    # NULL seqs / tokens / pos: refused before the handle is touched further (a NULL handle is reported first)
    for args in ((None, one, one), (one, None, one), (one, one, None)):
        assert L.xalm_cuda_forward_spans(None, 1, *args, None) == 1
        assert L.xalm_cuda_forward_spans_argmax(None, 1, *args, _ints(0)) == 1


def test_span_binding_checks_the_lengths():
    from xalm_b200.model import Model
    m = Model({"vocab_size": 16}, {})
    for seqs, toks, pos in (([0, 0], [5], [3, 4]), ([0, 0, 0], [5, 6, 7], [3, 4]), ([0], [5, 6], [3])):
        with pytest.raises(ValueError):
            m.forward_spans(seqs, toks, pos)
        with pytest.raises(ValueError):
            m.forward_spans_argmax(seqs, toks, pos)
