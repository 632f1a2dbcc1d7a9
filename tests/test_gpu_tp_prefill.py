"""Batched prefill on tensor-parallel models (needs >= 2 visible devices; each case skips when fewer are visible).

Each case is one torch.distributed.run of tp_prefill_worker.py, which checks on every rank: the linear and window prefill
against the CPU oracle (logits, log-probabilities, perplexity, the rank's KV shard), bit-identical sink keys against the token
loop, bit-identical logits on every rank, run-to-run determinism, greedy decode after the prefill, the logits of the unsharded
model on one GPU, and refusals that every rank makes alike without touching its cache.
"""
import os
import subprocess
import sys

import pytest

from xalm_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _ngpu():
    try:
        return capi.device_count()
    except capi.XalmError:
        return 0


# (world, wtype, shape, head_dim or None, XALM_TP_PEER, master port).  "small" keeps per-rank dimensions off the multiples of 256
# (LDG matvec, stand-alone decode exchange); head_dim 64 takes the mma.sync prefill attention; XALM_TP_PEER=0 decodes over NCCL.
CASES = [(2, "q8_0", "tp", None, "1", 29621), (2, "f16", "tp", None, "1", 29622), (2, "q4_0", "tp", None, "1", 29623),
         (2, "q8_0", "small", None, "1", 29624), (4, "q8_0", "tp", None, "1", 29625), (8, "q8_0", "tp8", None, "1", 29626),
         (8, "f16", "tp8", None, "1", 29627), (2, "q8_0", "tp", None, "0", 29628), (2, "q8_0", "tp", 64, "1", 29629)]


@pytest.mark.parametrize("world,wtype,shape,hd,peer,port", CASES,
                         ids=[f"tp{w}-{t}-{s}" + (f"-hd{h}" if h else "") + ("-nccl" if p == "0" else "") for w, t, s, h, p, _ in CASES])
def test_tp_prefill(world, wtype, shape, hd, peer, port):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    args = [wtype, shape] + ([str(hd)] if hd else [])
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "tp_prefill_worker.py"), *args],
                       capture_output=True, text=True, timeout=1200, env=dict(os.environ, XALM_TP_PEER=peer))
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "TP prefill ok" in r.stdout
