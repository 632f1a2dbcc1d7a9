"""bench.py --dump-outputs: the dumped logits are those of the last timed step.  The oracle replays the steps bench.py runs
(same seeded weights, and the tokens and positions bench.py's own helpers give) and must end on the same logits."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import oracle
from xalm_b200 import synth
from xalm_b200 import types as T
from xalm_b200 import xalm_file as X

from gpu_util import LOGIT_TOL

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED, CTX = 0, 128


def run_bench(out, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--shape", "tiny", "--ctx", str(CTX), "--seed", str(SEED),
                        "--no-cpu-baseline", "--dump-outputs", str(out), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def tiny_oracle():
    c = synth.model_config("tiny")
    cfg = X.parse_config(synth.metadata_strings(c), CTX)
    tensors = {n: (t.id, np.ascontiguousarray(a).view(np.uint8).reshape(-1)) for n, t, a in synth.iter_tensors(c, T.Q8_0, SEED)}
    return cfg, oracle.OracleModel(cfg, tensors, acc_mode=1)


def test_dump_outputs_holds_the_last_timed_decode_step(tmp_path):
    steps, warmup = 5, 3
    run_bench(tmp_path, "--steps", str(steps), "--warmup", str(warmup), "--no-parity", "--no-prefill")
    got = np.load(tmp_path / "logits.npy")
    cfg, om = tiny_oracle()
    assert got.dtype == np.float32 and got.shape == (cfg["vocab_size"],)
    _, _, warm, timed = bench.decode_inputs(steps, warmup, CTX, cfg["vocab_size"])
    for tok, pos in warm + timed:
        lg = om.forward(tok, pos, 1)
    om.close()
    assert float(np.max(np.abs(got - lg))) <= LOGIT_TOL


def test_dump_outputs_holds_the_perplexity_step(tmp_path):
    n_tok = 64
    run_bench(tmp_path, "--workload", "perplexity", "--tokens", str(n_tok), "--steps", "2", "--warmup", "3")
    got = np.load(tmp_path / "logits_sample.npy")
    cfg, om = tiny_oracle()
    rows = bench.perplexity_sample_rows(n_tok)
    assert got.dtype == np.float32 and got.shape == (len(rows), cfg["vocab_size"])
    toks = bench.perplexity_tokens(n_tok, cfg["vocab_size"])
    ref = np.stack([om.forward(int(toks[i]), i, 1) for i in range(n_tok)])
    om.close()
    assert float(np.max(np.abs(got - ref[rows]))) <= LOGIT_TOL
