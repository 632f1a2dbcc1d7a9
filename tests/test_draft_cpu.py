"""Drafting by a model without a GPU: xalm_cuda_forward_greedy's argument checks, the binding, and the refusals of
`xalm_main -m completion -s k -D draft` that come before any device work."""
import ctypes as C
import os
import re
import subprocess

import pytest

from xalm_b200 import build, capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
TARGET = os.path.join(GOLD, "tiny_q4_0.xalm")


def _ints(*v):
    return (C.c_int * len(v))(*v)


def test_symbol_is_in_the_header_and_the_binding():
    with open(os.path.join(ROOT, "include", "xalm_cuda.h")) as f:
        assert re.search(r"\bint xalm_cuda_forward_greedy\(", f.read())
    assert "xalm_cuda_forward_greedy" in capi.SYMBOLS


def test_greedy_refuses_a_null_handle():
    L = capi.lib()
    out = _ints(*[0] * 16)
    assert L.xalm_cuda_forward_greedy(None, 1, _ints(5), 3, 4, out) == 1
    assert b"NULL" in L.xalm_cuda_last_error()
    assert L.xalm_cuda_forward_greedy(None, 0, None, -1, 0, None) == 1


def test_binding_checks_arguments_before_calling_in():
    from xalm_b200.model import Model
    m = Model({"vocab_size": 16}, {})        # no handle: any call that reached the library would fail differently
    for tokens, pos, n_out in (([], 0, 1), ([1] * 9, 0, 1), ([1], 0, 0), ([1], 0, 17), ([16], 0, 1), ([-1], 0, 1), ([1, 2], -1, 1)):
        with pytest.raises(ValueError):
            m.forward_greedy(tokens, pos, n_out)
    with pytest.raises(RuntimeError):        # valid arguments on a model that is not on a device
        m.forward_greedy([1, 2], 0, 4)


def _main():
    build.build_cuda()
    build.build_host()
    return build.MAIN


def test_draft_usage_errors():
    exe = _main()
    for extra in (["-D", TARGET], ["-D", TARGET, "-n", "4"], ["-s", "2", "-D", TARGET, "-g", "2"], ["-D", TARGET, "-g", "2"],
                  ["-s", "2", "-D", TARGET, "-m", "perplexity"], ["-s", "2", "-D", TARGET, "-m", "batch"],
                  ["-s", "2", "-D", TARGET, "-m", "passkey"], ["-D", TARGET, "-m", "perplexity"], ["-D", TARGET, "-m", "batch"],
                  ["-D", TARGET, "-m", "passkey"]):
        r = subprocess.run([exe, TARGET, *extra], capture_output=True, text=True)
        assert r.returncode == 1 and "Usage" in r.stderr, (extra, r.stderr)
    r = subprocess.run([exe, TARGET, "-h", "x"], capture_output=True, text=True)
    assert "-D <filepath>" in r.stderr


def test_draft_that_does_not_match_is_refused_before_device_work(tmp_path):
    """A draft with another vocabulary size, or the same size and other tokens, is an error naming the mismatch.  The checks run
    before any device work, so they give the same answer on a machine without a GPU."""
    exe = _main()
    other_vocab = str(tmp_path / "vocab512.xalm")
    synth.write_checkpoint(other_vocab, "tiny", "q8_0", seed=1)                # vocab 512; the golden files have 288
    r = subprocess.run([exe, TARGET, "-m", "completion", "-n", "4", "-s", "2", "-D", other_vocab], capture_output=True, text=True)
    assert r.returncode == 1
    assert "error:" in r.stderr and "vocab_size 512" in r.stderr and "288" in r.stderr, r.stderr
    other_tokens = str(tmp_path / "tokens288.xalm")
    synth.write_checkpoint(other_tokens, "tiny", "q8_0", seed=1, vocab_size=288)  # synthetic tokenizer, not the golden one
    r = subprocess.run([exe, TARGET, "-m", "completion", "-n", "4", "-s", "2", "-D", other_tokens], capture_output=True, text=True)
    assert r.returncode == 1
    assert "error:" in r.stderr and "tokenizer.tokens differ" in r.stderr, r.stderr
    r = subprocess.run([exe, TARGET, "-m", "completion", "-n", "4", "-s", "2", "-D", str(tmp_path / "missing.xalm")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "error:" in r.stderr, r.stderr
