"""xalm_main -m completion -s k: speculative greedy decoding with prompt-lookup drafts prints exactly what -m completion prints."""
import os
import re
import subprocess

import pytest

from xalm_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REPEAT = "1 2 3 1 2 3 1 2"     # 16 tokens; tiny_q4_0 accepts a draft on it inside the window


def _main():
    build.build_cuda()
    build.build_host()
    return build.MAIN


def test_spec_usage_errors():
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    for extra in (["-s", "0"], ["-s", "8"], ["-s", "-1"], ["-s", "x"], ["-s", "3", "-g", "2"], ["-s", "2", "-m", "perplexity"],
                  ["-s", "2", "-m", "batch"], ["-s", "2", "-m", "passkey"]):
        r = subprocess.run([exe, path, *extra], capture_output=True, text=True)
        assert r.returncode == 1 and "Usage" in r.stderr, extra
    r = subprocess.run([exe, path, "-h", "x"], capture_output=True, text=True)
    assert "-s <int>" in r.stderr


def _run(exe, path, prompt, n, extra=(), env=None):
    r = subprocess.run([exe, path, "-m", "completion", "-i", prompt, "-n", str(n), *extra], capture_output=True,
                       env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr.decode(errors="replace")
    out = r.stdout
    start = out.index(b"Encoding stats:")
    start = out.index(b"\n\n", start) + 2
    end = out.rindex(b"\n\nGeneration stats:")
    return out[start:end], out[end:].decode()


def _spec_line(stats):
    m = re.search(r"speculative: (\d+) passes, (\d+) drafted, (\d+) accepted, ([0-9.e+]+) tokens/pass", stats)
    assert m, stats
    return int(m.group(1)), int(m.group(2)), int(m.group(3)), float(m.group(4))


@pytest.mark.gpu
@pytest.mark.parametrize("t,env", [("q4_0", {}), ("q8_0", {"XALM_MMA": "1"})])
def test_spec_output_equals_completion(t, env):
    """q4_0 takes the tensor-core kernel in plain completion; q8_0 does with XALM_MMA=1 (else the dp4a kernel, whose sums differ
    in the last bits from the batched handle's)."""
    exe = _main()
    path = os.path.join(GOLD, f"tiny_{t}.xalm")
    for prompt in ("Q: What is the meaning of life? A:", REPEAT):
        want, stats = _run(exe, path, prompt, 48, env=env)
        assert "speculative" not in stats
        for k in (1, 3, 7):
            got, stats = _run(exe, path, prompt, 48, ["-s", str(k)])
            assert got == want, (t, prompt, k)
            passes, drafted, accepted, per = _spec_line(stats)
            assert 0 < passes <= 48 and accepted <= drafted <= k * passes


@pytest.mark.gpu
def test_spec_accepts_drafts_on_repetitive_text():
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    want, _ = _run(exe, path, REPEAT, 64)
    got, stats = _run(exe, path, REPEAT, 64, ["-s", "4"])
    assert got == want
    passes, drafted, accepted, per = _spec_line(stats)
    assert accepted > 0 and drafted > 0 and per > 1.0, stats
    assert passes < 64


@pytest.mark.gpu
def test_spec_past_the_window():
    """-T 32: spans while the sequence fits the window, plain steps on the KV ring after it; the text still matches."""
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    prompt = "Q: What is the meaning of life? A:"                # 12 tokens: 28 positions inside the window, 12 past it
    want, _ = _run(exe, path, prompt, 40, ["-T", "32"])
    got, stats = _run(exe, path, prompt, 40, ["-T", "32", "-s", "3"])
    assert got == want
    _spec_line(stats)


@pytest.mark.gpu
def test_spec_refuses_a_float_checkpoint():
    exe = _main()
    r = subprocess.run([exe, os.path.join(GOLD, "tiny_f16.xalm"), "-m", "completion", "-n", "4", "-s", "2"], capture_output=True, text=True)
    assert r.returncode == 1
    assert "batched handle" in r.stderr and ".weight" in r.stderr, r.stderr
