"""xalm_main end to end at 1, 2, 4 and 8 GPUs (`-g P`, as many as the box has): completion and perplexity on the m7 q8_0
checkpoint, the numbers the CLI itself prints.

    python scripts/bench_cli_tp.py --out build/cli_tp

Writes the synthetic m7 q8_0 checkpoint (about 7.6 GB) to a temporary directory and deletes it at the end.  For each P:
  - `-m completion -n 256` with the default prompt: the "Generation stats" block (tokens over wall time from the start of
    the prompt hydrate, host sampler and logits copy included);
  - `-m perplexity` over a generated prompt file of --ppl-tokens tokens: the "Stats" block (batched prefill).
Each block, the launches per decode token (P > 1) and the GPU name and power limit read in the same command go into
<out>/cli_tp.json; the CLI's full stdout / stderr for each run go next to it.
"""
import argparse
import json
import os
import random
import re
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from xalm_b200 import build, capi, synth  # noqa: E402


def gpus():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    return [[s.strip() for s in l.split(",")] for l in out.stdout.strip().splitlines() if l.strip()]


def stats(stdout):
    """The key: value lines of the stats block the CLI prints last."""
    block = re.split(r"\n(?:Generation stats|Stats):\n", stdout)[-1]
    out = {}
    for line in block.splitlines():
        if ":" in line:
            k, v = line.strip().split(":", 1)
            out[k.strip()] = v.strip()
        elif line.strip():
            out.setdefault("lines", []).append(line.strip())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--model", default="m7")
    ap.add_argument("--wtype", default="q8_0")
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--ppl-tokens", type=int, default=4096)
    ap.add_argument("--sizes", default="1,2,4,8")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    exe = build.MAIN
    if not os.path.exists(exe):
        raise SystemExit(f"{exe} is missing: build first (python __graft_entry__.py)")
    cards = gpus()
    n = capi.device_count()
    sizes = [int(s) for s in args.sizes.split(",")]
    res = {"model": args.model, "wtype": args.wtype, "gpus": [{"name": c[0], "power_limit": c[1]} for c in cards], "runs": [],
           "not_measured": [p for p in sizes if p > n]}
    tmp = tempfile.mkdtemp(prefix="xalm_cli_tp_")
    try:
        ckpt = os.path.join(tmp, f"{args.model}_{args.wtype}.xalm")
        t0 = time.time()
        synth.write_checkpoint(ckpt, args.model, args.wtype, seed=0, std=0.02)
        res["checkpoint_bytes"] = os.path.getsize(ckpt)
        print(f"wrote {ckpt} ({res['checkpoint_bytes'] / 1e9:.2f} GB) in {time.time() - t0:.0f} s", flush=True)
        # exactly --ppl-tokens tokens with the BOS: none of these characters starts a multi-character token of the synthetic vocabulary
        rng = random.Random(0)
        text = "".join(rng.choice("bcdhklmpsuwxyz0123456789 .,") for _ in range(args.ppl_tokens - 1))
        prompt = os.path.join(tmp, "prompt.txt")
        with open(prompt, "w") as f:
            f.write(text)
        for p in sizes:
            if p > n:
                continue
            for mode, extra in (("completion", ["-n", str(args.steps)]), ("perplexity", ["-f", prompt])):
                cmd = [exe, ckpt, "-m", mode, *extra] + (["-g", str(p)] if p > 1 else [])
                t0 = time.time()
                r = subprocess.run(cmd, capture_output=True, text=True, errors="replace", timeout=3600)
                wall = time.time() - t0
                tag = f"{mode}_g{p}"
                with open(os.path.join(args.out, tag + ".stdout"), "w") as f:
                    f.write(r.stdout)
                with open(os.path.join(args.out, tag + ".stderr"), "w") as f:
                    f.write(r.stderr)
                run = {"mode": mode, "gpus": p, "rc": r.returncode, "process_wall_s": round(wall, 2), "command": " ".join(cmd[1:]).replace(tmp, "$TMP")}
                if r.returncode == 0:
                    run["stats"] = stats(r.stdout)
                else:
                    run["stderr_tail"] = r.stderr[-2000:]
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    res["gpus_after"] = [{"name": c[0], "power_limit": c[1]} for c in gpus()]
    with open(os.path.join(args.out, "cli_tp.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}))


if __name__ == "__main__":
    main()
