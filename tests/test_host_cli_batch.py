"""xalm_main -m batch: several prompts decoded together with continuous batching, each equal to -m completion's output."""
import os
import re
import subprocess

import pytest

from xalm_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
PROMPTS = ["Q: What is the meaning of life? A:", "The grass is green.", "Once upon a time", "1 2 3 4", "Hello"]


def _main():
    build.build_cuda()
    build.build_host()
    return build.MAIN


def test_batch_mode_usage_errors(tmp_path):
    exe = _main()
    f = tmp_path / "prompts.txt"
    f.write_text("\n".join(PROMPTS) + "\n")
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    for extra in (["-g", "2"], ["-n", "-1"], ["-b", "9"], ["-b", "0"]):
        r = subprocess.run([exe, path, "-m", "batch", "-f", str(f), *extra], capture_output=True, text=True)
        assert r.returncode == 1 and "Usage" in r.stderr, extra
    r = subprocess.run([exe, path, "-m", "batch"], capture_output=True, text=True)   # no prompt file
    assert r.returncode == 1 and "Usage" in r.stderr


def _completion_text(exe, path, prompt, n):
    r = subprocess.run([exe, path, "-m", "completion", "-i", prompt, "-n", str(n)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode(errors="replace")
    out = r.stdout
    start = out.index(b"Encoding stats:")
    start = out.index(b"\n\n", start) + 2
    end = out.rindex(b"\n\nGeneration stats:")
    return out[start:end]              # run_completion ends the text with "\n" + endl


@pytest.mark.gpu
def test_batch_mode_matches_completion(tmp_path):
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    f = tmp_path / "prompts.txt"
    f.write_text("\n".join(PROMPTS[:2]) + "\n\n" + "\n".join(PROMPTS[2:]) + "\n")   # empty lines are skipped
    r = subprocess.run([exe, path, "-m", "batch", "-f", str(f), "-b", "2", "-n", "16"], capture_output=True)
    assert r.returncode == 0, r.stderr.decode(errors="replace")
    out = r.stdout
    body, stats = out.split(b"\nBatch stats:\n")
    parts = re.split(rb"\[prompt (\d+)\]\n", body[body.index(b"[prompt 0]"):])
    got = {int(parts[i]): parts[i + 1][:-1] for i in range(1, len(parts), 2)}
    assert sorted(got) == list(range(len(PROMPTS)))
    for i, p in enumerate(PROMPTS):
        assert got[i] == _completion_text(exe, path, p, 16), (i, p)
    assert b"5 prompts" in stats and b"generated tokens" in stats and b"mean sequences per step" in stats
    assert b"hydrate:" in stats and b"bandwidth:" in stats and b"throughput:" in stats
