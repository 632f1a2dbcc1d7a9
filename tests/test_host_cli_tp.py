"""xalm_main -g P: tensor-parallel completion, perplexity and passkey from the C++ CLI.

The CLI forks P rank processes (csrc/host/launch.cpp).  Every test checks after every run that no process is left whose
command line names the test's checkpoint: the forked ranks carry the parent's command line.  Multi-GPU cases skip when fewer
than P devices are visible.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_host_cli import GOLD, _has_gpu, _main, _oracle_completion
from xalm_b200 import capi, synth

PROMPT = "Q: What is the meaning of life? A:"   # the CLI's default prompt
# a few hundred tokens with the synthetic byte-fallback vocabulary: hydrates past a -T 64 window in prefill_window chunks
LONG = " ".join(f"the meaning of life is {i} in the of a Q A" for i in range(12))


def _ngpu():
    try:
        return capi.device_count()
    except capi.XalmError:
        return 0


def _need(p):
    if _ngpu() < p:
        pytest.skip(f"needs {p} GPUs")


def _leftover(path):
    key = os.fsencode(path)
    left = []
    for pid in os.listdir("/proc"):
        if not pid.isdigit():
            continue
        try:
            with open(f"/proc/{pid}/cmdline", "rb") as f:
                if key in f.read():
                    left.append(int(pid))
        except OSError:
            pass
    return left


def _run(path, *args, env=None):
    r = subprocess.run([_main(), path, *args], capture_output=True, timeout=900,
                       env=dict(os.environ, **(env or {})))
    assert _leftover(path) == [], "a rank process outlived the CLI"
    return r


def _ok(r):
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-3000:]
    return r.stdout


def _ckpt(tmp_path, shape, wtype):
    path = str(tmp_path / f"{shape}_{wtype}.xalm")
    synth.write_checkpoint(path, shape, wtype, seed=1, std=0.03)
    return path


def _generated(out):
    """The completion text: after the encoding stats line, before the generation stats."""
    return out.split(b"Encoding stats:", 1)[1].split(b"\n", 1)[1].split(b"Generation stats:")[0]


def _launches(out):
    line = [l for l in out.decode(errors="replace").splitlines() if "tensor parallel:" in l]
    assert len(line) == 1, out[-800:]
    return int(line[0].split(",")[1].split()[0])


def _perplexity(out):
    line = [l for l in out.decode(errors="replace").splitlines() if "perplexity:" in l][0]
    return float(line.split("perplexity:")[1].split()[0])


# ---- without a GPU ---------------------------------------------------------------------------------------------

def test_cli_gpus_flag_usage(tmp_path):
    path = str(tmp_path / "unused.xalm")
    for g in ("0", "-1", "x", "2x"):
        r = _run(path, "-g", g)
        assert r.returncode == 1 and b"Usage" in r.stderr, (g, r.stderr)


def test_cli_verify_refuses_gpus(tmp_path):
    path = str(tmp_path / "tiny.xalm")
    shutil.copy(os.path.join(GOLD, "tiny_q8_0.xalm"), path)
    r = _run(path, "-m", "verify", "-g", "2")
    assert r.returncode == 1 and b"-m verify" in r.stderr and b"Usage" in r.stderr
    assert b"verified" not in r.stdout


def test_cli_tp_missing_file(tmp_path):
    r = _run(str(tmp_path / "missing.xalm"), "-g", "2")
    assert r.returncode == 1
    assert b"rank 0: error:" in r.stderr, r.stderr


@pytest.mark.skipif(_has_gpu(), reason="only meaningful without a GPU")
def test_cli_tp_fails_loudly_without_a_gpu(tmp_path):
    path = str(tmp_path / "tiny.xalm")
    shutil.copy(os.path.join(GOLD, "tiny_q8_0.xalm"), path)
    r = _run(path, "-g", "2", "-n", "4")
    err = r.stderr.decode(errors="replace")
    assert r.returncode == 1 and ("-g 2 needs 2 visible CUDA devices" in err or "model.cuda()" in err), err
    assert r.stdout == b""


# The launcher alone, on the CPU: launch.cpp linked with stand-ins for the three backend calls it makes before a mode function
# runs (device count, last error, NCCL id).  The mode function checks the id, swaps a handle through ipc_exchange and prints.
HARNESS = r"""
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "launch.h"
extern "C" {
int xalm_cuda_device_count(int* n) { *n = atoi(getenv("STUB_DEVICES")); return 0; }
const char* xalm_cuda_last_error(void) { return ""; }
int xalm_cuda_comm_unique_id(void* id) { memset(id, 0x5a, XALM_COMM_ID_BYTES); *(unsigned char*) id = 7; return 0; }
}
int main(int argc, char** argv) {
	const int P = atoi(argv[1]), fail = argc > 2 ? atoi(argv[2]) : -1;
	return run_tp_ranks(P, [&](const TpRank& tp) {
		const unsigned char* id = (const unsigned char*) tp.comm_id;
		if (tp.device != tp.rank || tp.size != P || id[0] != 7 || id[XALM_COMM_ID_BYTES - 1] != 0x5a) { fprintf(stderr, "bad rank\n"); return 1; }
		if (tp.rank == fail) { fprintf(stderr, "refused\n"); return 1; }
		const std::vector<uint8_t> table = tp.ipc_exchange(std::vector<uint8_t>(XALM_IPC_HANDLE_BYTES, (uint8_t) (tp.rank + 1)));
		for (int r = 0; r < P; r++)
			for (int i = 0; i < XALM_IPC_HANDLE_BYTES; i++)
				if (table[r * XALM_IPC_HANDLE_BYTES + i] != r + 1) { fprintf(stderr, "bad table\n"); return 1; }
		printf("rank %d: table of %d ok\n", tp.rank, P);
		fprintf(stderr, "done\n");
		return 0;
	});
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    from xalm_b200 import build
    d = tmp_path_factory.mktemp("launch")
    src, exe = d / "harness.cpp", str(d / "launch_harness")
    src.write_text(HARNESS)
    hdir = os.path.join(build.CSRC, "host")
    subprocess.check_call([build.GXX, "-O1", "-std=c++20", "-Wall", "-I", os.path.join(build.ROOT, "include"), "-I", hdir, str(src),
                           os.path.join(hdir, "launch.cpp"), "-o", exe])
    return exe


def _run_harness(exe, *args, devices=8):
    r = subprocess.run([exe, *args], capture_output=True, text=True, timeout=60, env=dict(os.environ, STUB_DEVICES=str(devices)))
    assert _leftover(exe) == [], "a rank process outlived the launcher"
    return r


def test_launcher_rendezvous(harness):
    for P in (2, 3, 8):
        r = _run_harness(harness, str(P))
        assert r.returncode == 0, r.stderr
        assert r.stdout == f"rank 0: table of {P} ok\n"                 # only rank 0 writes stdout
        assert sorted(r.stderr.splitlines()) == [f"rank {i}: done" for i in range(P)]


def test_launcher_one_failing_rank_ends_the_group(harness):
    r = _run_harness(harness, "3", "2")          # rank 2 fails; ranks 0 and 1 wait for its handle until they are killed
    assert r.returncode == 1 and "rank 2: refused" in r.stderr and r.stdout == "", r.stderr


def test_launcher_needs_enough_devices(harness):
    r = _run_harness(harness, "4", devices=2)
    assert r.returncode == 1 and "rank 0: error: -g 4 needs 4 visible CUDA devices, 2 found" in r.stderr, r.stderr


# ---- on P GPUs ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_cli_tp_more_ranks_than_devices(tmp_path):
    """The ranks fork before any CUDA call, so each one can still count the devices: a box with too few says so."""
    n = _ngpu()
    if not 1 <= n < 8:
        pytest.skip("needs 1 to 7 GPUs")
    path = _ckpt(tmp_path, "tp", "q8_0")
    r = _run(path, "-n", "4", "-g", str(n + 1))
    assert r.returncode == 1 and f"-g {n + 1} needs {n + 1} visible CUDA devices, {n} found".encode() in r.stderr, r.stderr


COMPLETION = [(2, "q8_0", "tp"), (2, "f16", "tp"), (2, "q4_0", "tp"), (4, "q8_0", "tp"), (8, "q8_0", "tp8")]


@pytest.mark.gpu
@pytest.mark.parametrize("P,wtype,shape", COMPLETION, ids=[f"tp{p}-{t}-{s}" for p, t, s in COMPLETION])
def test_cli_tp_completion(tmp_path, P, wtype, shape):
    _need(P)
    path = _ckpt(tmp_path, shape, wtype)
    enc, text, *_ = _oracle_completion(path, PROMPT, 24)
    one = _ok(_run(path, "-n", "24"))
    tp = _ok(_run(path, "-n", "24", "-g", str(P)))
    assert text in one, (text, one[-600:])
    assert text in tp, (text, tp[-600:])
    assert _generated(tp) == _generated(one)
    assert f"{len(enc)} tokens".encode() in tp
    assert b"tensor parallel:" not in one and f"tensor parallel: {P} GPUs".encode() in tp


@pytest.mark.gpu
def test_cli_tp_one_gpu_is_the_plain_path(tmp_path):
    _need(1)
    path = _ckpt(tmp_path, "tp", "q8_0")
    plain = _ok(_run(path, "-n", "16"))
    g1 = _ok(_run(path, "-n", "16", "-g", "1"))
    assert _generated(g1) == _generated(plain) and b"tensor parallel:" not in g1


@pytest.mark.gpu
def test_cli_tp_completion_past_the_window(tmp_path):
    _need(2)
    path = _ckpt(tmp_path, "tp", "q8_0")
    prompt = tmp_path / "prompt.txt"
    prompt.write_text(LONG)
    args = ["-n", "16", "-T", "64", "-f", str(prompt)]
    one = _ok(_run(path, *args))
    tp = _ok(_run(path, *args, "-g", "2"))
    n_tokens = int(one.split(b"Encoding stats: (")[1].split()[0])
    assert n_tokens > 64 + 2 * 62, n_tokens          # the prompt hydrate takes several prefill_window chunks
    assert _generated(tp) == _generated(one) and len(_generated(one).strip()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("context,prompt", [(0, "the meaning of life is in the the of a"), (32, LONG[:200])], ids=["linear", "window"])
def test_cli_tp_perplexity(tmp_path, context, prompt):
    from oracle import oracle
    _need(2)
    path = _ckpt(tmp_path, "tp", "q8_0")
    _, _, om, tok, cfg, f = _oracle_completion(path, prompt, 0, context)
    enc = tok.encode(prompt, True)
    s = 0.0
    for pos in range(len(enc) - 1):
        lg = om.forward(enc[pos], pos, 1)
        s += np.log(oracle.sample_prob(lg, enc[pos + 1]))
    ppl = float(np.exp(-s / (len(enc) - 1)))
    args = ["-m", "perp", "-i", prompt] + (["-T", str(context)] if context else [])
    if context:
        assert len(enc) > 2 * context
    one = _perplexity(_ok(_run(path, *args)))
    tp_out = _ok(_run(path, *args, "-g", "2"))
    tp = _perplexity(tp_out)
    assert b"tensor parallel: 2 GPUs" in tp_out
    assert abs(tp - ppl) / ppl < 2e-3, (tp, ppl)
    assert abs(tp - one) / one < 1e-3, (tp, one)


@pytest.mark.gpu
def test_cli_tp_passkey(tmp_path):
    _need(2)
    path = _ckpt(tmp_path, "tp", "q8_0")
    args = ["-m", "passkey", "-n", "3", "-T", "32", "-l", "1"]
    one = _ok(_run(path, *args))
    tp = _ok(_run(path, *args, "-g", "2"))
    suffix = b" What is the pass key? The pass key is"
    header = lambda out: out.split(b"Passkey test:")[1].split(b"\r")[0]   # prompt length and the drawn passkey
    assert header(tp) == header(one)
    assert tp.rsplit(suffix, 1)[1] == one.rsplit(suffix, 1)[1]


@pytest.mark.gpu
def test_cli_tp_fused_exchange(tmp_path):
    """The IPC handles arrive: the default decode takes the fused exchange, with fewer launches than the stand-alone one."""
    _need(2)
    path = _ckpt(tmp_path, "tp", "q8_0")
    fused = _ok(_run(path, "-n", "16", "-g", "2"))
    plain = _ok(_run(path, "-n", "16", "-g", "2", env={"XALM_TP_FUSED": "0"}))
    assert _launches(fused) < _launches(plain), (_launches(fused), _launches(plain))
    assert _generated(fused) == _generated(plain)


@pytest.mark.gpu
def test_cli_tp_standalone_exchange(tmp_path):
    """Per-rank dimensions off the multiples of 256 keep the fused exchange off; the stand-alone one still matches the oracle."""
    _need(2)
    path = _ckpt(tmp_path, "small", "q8_0")
    _, text, *_ = _oracle_completion(path, PROMPT, 16)
    out = _ok(_run(path, "-n", "16", "-g", "2"))
    plain = _ok(_run(path, "-n", "16", "-g", "2", env={"XALM_TP_FUSED": "0"}))
    assert text in out, (text, out[-600:])
    assert _launches(out) == _launches(plain)


@pytest.mark.gpu
def test_cli_tp_refuses_a_size_that_does_not_divide(tmp_path):
    _need(3)
    path = _ckpt(tmp_path, "tp", "q8_0")     # 8 heads, 4 kv heads: not in 3
    r = _run(path, "-n", "4", "-g", "3")
    assert r.returncode == 1 and b"tp_size 3 does not divide" in r.stderr, r.stderr
