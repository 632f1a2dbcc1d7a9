"""Tree verification without a GPU: argument checks of the three entry points, the binding, and the usage errors of
`xalm_main -s k -w b`, all of which come before any device work."""
import ctypes as C
import os
import re
import subprocess

import pytest

from xalm_b200 import build, capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TARGET = os.path.join(ROOT, "tests", "golden", "tiny_q4_0.xalm")


def _ints(*v):
    return (C.c_int * len(v))(*v)


def test_symbols_are_in_the_header_and_the_binding():
    with open(os.path.join(ROOT, "include", "xalm_cuda.h")) as f:
        h = f.read()
    for name in ("xalm_cuda_forward_tree", "xalm_cuda_forward_tree_argmax", "xalm_cuda_tree_accept"):
        assert re.search(rf"\bint {name}\(", h)
        assert name in capi.SYMBOLS


def test_tree_entry_points_refuse_a_null_handle():
    L = capi.lib()
    toks, par, out = _ints(5, 6), _ints(-1, 0), _ints(0, 0)
    assert L.xalm_cuda_forward_tree(None, 0, 2, toks, par, 3, None) == 1
    assert b"NULL" in L.xalm_cuda_last_error()
    assert L.xalm_cuda_forward_tree_argmax(None, 0, 2, toks, par, 3, out) == 1
    assert b"NULL" in L.xalm_cuda_last_error()
    assert L.xalm_cuda_tree_accept(None, 0, 3, 2, _ints(0, 1)) == 1
    assert b"NULL" in L.xalm_cuda_last_error()


def test_tree_entry_points_refuse_null_arrays():
    L = capi.lib()
    toks, par = _ints(5, 6), _ints(-1, 0)
    assert L.xalm_cuda_forward_tree_argmax(None, 0, 2, toks, par, 3, None) == 1   # no next_tokens
    assert b"next_tokens is NULL" in L.xalm_cuda_last_error()
    for t, p in ((None, par), (toks, None), (None, None)):
        assert L.xalm_cuda_forward_tree(None, 0, 2, t, p, 3, None) == 1
        assert L.xalm_cuda_forward_tree_argmax(None, 0, 2, t, p, 3, _ints(0, 0)) == 1
    assert L.xalm_cuda_tree_accept(None, 0, 3, 1, None) == 1


def test_tree_binding_checks_the_lengths():
    from xalm_b200.model import Model
    m = Model({"vocab_size": 16}, {})
    for toks, parents in (([5, 6], [-1]), ([5], [-1, 0]), ([], []), ([5, 6, 7], [-1, 0])):
        with pytest.raises(ValueError):
            m.forward_tree(0, toks, parents, 3)
        with pytest.raises(ValueError):
            m.forward_tree_argmax(0, toks, parents, 3)
    with pytest.raises(ValueError):
        m.tree_accept(0, 3, [])


def _main():
    build.build_cuda()
    build.build_host()
    return build.MAIN


def test_width_usage_errors():
    exe = _main()
    for extra in (["-w", "2"],                                   # no -s
                  ["-w", "1"],
                  ["-s", "3", "-w", "4"],                        # b > k
                  ["-s", "3", "-w", "0"], ["-s", "3", "-w", "-1"], ["-s", "3", "-w", "x"],
                  ["-s", "3", "-w", "2", "-D", TARGET],          # the draft model gives one chain
                  ["-s", "3", "-w", "1", "-D", TARGET],
                  ["-s", "3", "-w", "2", "-g", "2"],             # what -s refuses
                  ["-s", "3", "-w", "2", "-m", "perplexity"], ["-s", "3", "-w", "2", "-m", "batch"],
                  ["-s", "3", "-w", "2", "-m", "passkey"],
                  ["-w", "2", "-m", "batch"], ["-w", "2", "-g", "2"]):
        r = subprocess.run([exe, TARGET, *extra], capture_output=True, text=True)
        assert r.returncode == 1 and "Usage" in r.stderr, (extra, r.stderr)
    r = subprocess.run([exe, TARGET, "-h", "x"], capture_output=True, text=True)
    assert "-w <int>" in r.stderr
