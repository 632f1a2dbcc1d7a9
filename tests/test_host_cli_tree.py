"""xalm_main -m completion -s k -w b: speculative greedy decoding that verifies up to b prompt-lookup continuations per pass as one
tree prints exactly what -m completion prints."""
import os
import re

import pytest

from test_host_cli_spec import _main, _run, _spec_line

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
TWO_WAYS = "1 2 3 4 1 2 3 5 1 2 3"                 # the repeated suffix was followed by two different continuations
BRANCHY = "the cat the dog the cat the dog the"   # tiny_q4_0 accepts more drafts on it with -w 2 than with -w 1

pytestmark = pytest.mark.gpu


def _tree_line(stats):
    m = re.search(r"tree: up to (\d+) branches, (\d+) passes verified more than one", stats)
    assert m, stats
    return int(m.group(1)), int(m.group(2))


@pytest.mark.parametrize("t,env", [("q4_0", {}), ("q8_0", {"XALM_MMA": "1"})])
def test_tree_output_equals_completion(t, env):
    exe = _main()
    path = os.path.join(GOLD, f"tiny_{t}.xalm")
    for prompt in ("Q: What is the meaning of life? A:", TWO_WAYS, BRANCHY):
        want, stats = _run(exe, path, prompt, 48, env=env)
        assert "speculative" not in stats
        for k in (3, 7):
            for b in (2, 3):
                got, stats = _run(exe, path, prompt, 48, ["-s", str(k), "-w", str(b)], env=env)
                assert got == want, (t, prompt, k, b)
                passes, drafted, accepted, per = _spec_line(stats)
                assert 0 < passes <= 48 and accepted <= drafted <= k * passes
                assert _tree_line(stats)[0] == b


@pytest.mark.parametrize("t,env", [("q4_0", {}), ("q8_0", {"XALM_MMA": "1"})])
def test_tree_past_the_window(t, env):
    """-T 32: trees while the sequence fits the window, plain steps on the KV ring after it; the text still matches."""
    exe = _main()
    path = os.path.join(GOLD, f"tiny_{t}.xalm")
    want, _ = _run(exe, path, TWO_WAYS, 48, ["-T", "32"], env=env)
    for k, b in ((3, 2), (7, 3)):
        got, stats = _run(exe, path, TWO_WAYS, 48, ["-T", "32", "-s", str(k), "-w", str(b)], env=env)
        assert got == want, (t, k, b)


def test_width_one_is_the_chain():
    """-w 1 is -s alone: the same text and the same speculative line, and no tree line."""
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    for prompt in (TWO_WAYS, BRANCHY):
        got1, s1 = _run(exe, path, prompt, 48, ["-s", "3", "-w", "1"])
        got0, s0 = _run(exe, path, prompt, 48, ["-s", "3"])
        assert got1 == got0 and _spec_line(s1)[:3] == _spec_line(s0)[:3]
        assert "tree:" not in s1


def test_two_branches_accept_more_on_branchy_text():
    exe = _main()
    path = os.path.join(GOLD, "tiny_q4_0.xalm")
    want, _ = _run(exe, path, BRANCHY, 48)
    got1, s1 = _run(exe, path, BRANCHY, 48, ["-s", "3"])
    got2, s2 = _run(exe, path, BRANCHY, 48, ["-s", "3", "-w", "2"])
    assert got1 == want and got2 == want
    a1, a2 = _spec_line(s1)[2], _spec_line(s2)[2]
    assert a2 > a1, (s1, s2)
