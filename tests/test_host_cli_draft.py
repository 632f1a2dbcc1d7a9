"""xalm_main -m completion -s k -D draft: speculative greedy decoding with a draft model prints exactly what -m completion prints,
whatever the draft."""
import os
import re

import pytest

from test_host_cli_spec import GOLD, _main, _run, _spec_line
from xalm_b200 import synth

pytestmark = pytest.mark.gpu

PROMPT = "Q: What is the meaning of life? A:"
TARGET = os.path.join(GOLD, "tiny_q4_0.xalm")


def _draft_line(stats):
    m = re.search(r"draft: (.+), (\d+) steps in (\d+) calls, ([0-9.e+-]+)s", stats)
    assert m, stats
    return int(m.group(2)), int(m.group(3))


def test_target_as_its_own_draft_accepts_every_draft():
    """The draft is the target itself (on a batch-1 handle, the same tensor-core kernel): every draft is accepted."""
    exe = _main()
    want, _ = _run(exe, TARGET, PROMPT, 48)
    for k in (1, 3, 7):
        got, stats = _run(exe, TARGET, PROMPT, 48, ["-s", str(k), "-D", TARGET])
        assert got == want, k
        passes, drafted, accepted, per = _spec_line(stats)
        assert accepted == drafted and per > 1.0, (k, stats)
        steps, calls = _draft_line(stats)
        assert calls == passes and steps >= drafted, (k, stats)


@pytest.mark.parametrize("draft", ["f16", "q8_0"])
def test_other_formats_draft_for_q4_0(draft):
    exe = _main()
    path = os.path.join(GOLD, f"tiny_{draft}.xalm")
    for prompt in (PROMPT, "1 2 3 1 2 3 1 2"):
        want, _ = _run(exe, TARGET, prompt, 48)
        for k in (1, 3, 7):
            got, stats = _run(exe, TARGET, prompt, 48, ["-s", str(k), "-D", path])
            assert got == want, (draft, prompt, k)
            passes, drafted, accepted, per = _spec_line(stats)
            assert 0 < passes <= 48 and accepted <= drafted <= k * passes
            _draft_line(stats)


def test_a_poor_draft_still_gives_the_same_text(tmp_path):
    """A synthetic target and a draft with other weights (another seed) but the same tokenizer: few drafts are accepted, the
    text is still the target's."""
    exe = _main()
    target, draft = str(tmp_path / "target.xalm"), str(tmp_path / "draft.xalm")
    synth.write_checkpoint(target, "tiny", "q4_0", seed=0, std=0.06)
    synth.write_checkpoint(draft, "tiny", "q8_0", seed=7, std=0.06)
    want, _ = _run(exe, target, PROMPT, 40)
    for k in (1, 3, 7):
        got, stats = _run(exe, target, PROMPT, 40, ["-s", str(k), "-D", draft])
        assert got == want, k
        passes, drafted, accepted, per = _spec_line(stats)
        assert accepted < drafted, (k, stats)


def test_draft_past_the_window():
    """-T 32: draft rounds while the sequence fits the window, plain steps on the KV ring after it (the draft is not called)."""
    exe = _main()
    draft = os.path.join(GOLD, "tiny_q8_0.xalm")
    want, _ = _run(exe, TARGET, PROMPT, 40, ["-T", "32"])
    for k in (1, 3, 7):
        got, stats = _run(exe, TARGET, PROMPT, 40, ["-T", "32", "-s", str(k), "-D", draft])
        assert got == want, k
        passes, drafted, accepted, per = _spec_line(stats)
        steps, calls = _draft_line(stats)
        assert 0 < calls < passes, (k, stats)
