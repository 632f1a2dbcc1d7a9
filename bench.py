#!/usr/bin/env python
"""bench.py — Mistral-7B batch-1 decode throughput on N B200s (BASELINE.json metric), with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape m7] [--wtype q8_0] [--ctx 4096]
                    [--dump-outputs DIR]

A "step" is one decoded token: one pass of the hot path (embed -> 32 x [norm+QKV+rope+KV, attention, Wo+residual,
norm+W1|W3+GLU, W2+residual] -> norm+classifier).  The workload is BASELINE config[1]: Mistral-7B-v0.2 architecture,
random-init weights N(0, 0.02^2) quantised to q8_0 with the reference's own quantiser rules, batch 1, 4k context; the K
timed tokens sit at positions spread uniformly over [0, ctx) (the fp16 KV ring is fully allocated, so attention streams
kv_len rows of it exactly as a hydrated cache would).  Weights (7.5 GB) are far larger than L2 (126 MB), so every step
streams them from HBM; no L2 flush is needed between steps.

`value`  : tokens/s, device-timed (CUDA events on the launch stream, max over ranks), weights + KV resident in HBM.
`e2e`    : the same loop through the public API (Model.forward + Sampler.sample_argmax on HOST logits): every step
           copies the step's inputs (token, position: one 32-byte StepParams from pinned memory) host->device and the
           logits (vocab * 4 bytes) device->host, and is timed by the wall clock around the synchronous calls.
`--impl reference` : the reference's CPU path (oracle/ restatement; the reference C++ does not build on x86, DESIGN.md)
           on all host cores, same model, one token per step.
N > 1    : tensor parallel over N GPUs (one process per GPU, strong scaling: same model, sharded).
`--dump-outputs DIR` : after the timed steps, rank 0 writes what the timed path computed in its last step, as float32 .npy
           files: the decode workload and every --impl reference run write DIR/logits.npy, the vocab_size logits of the last
           timed token; the perplexity workload on the GPU writes DIR/logits_sample.npy, the logits of a fixed, seeded
           sample of at most 128 of its positions (perplexity_sample_rows).  Weights, tokens and positions depend only on the arguments, so two builds run with the
           same arguments can be compared output for output.  bench_outputs/ in the repository is git-ignored for this.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SMI_QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={SMI_QUERY}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs() -> tuple:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def positions_for(steps: int, ctx: int) -> list:
    if steps <= 1:
        return [ctx - 1]
    return [int(round(i * (ctx - 1) / (steps - 1))) for i in range(steps)]


def decode_inputs(steps: int, warmup: int, ctx: int, vocab_size: int) -> tuple:
    """(tokens, positions, warm-up steps, timed steps) of the decode workload, a fixed function of the arguments; each step
    is a (token, position) pair."""
    pos_list = positions_for(steps, ctx)
    toks = [int(t) for t in np.random.default_rng(123).integers(3, vocab_size, size=steps + warmup)]
    warm = [(toks[i], pos_list[min(i, len(pos_list) - 1)]) for i in range(warmup)]
    timed = [(toks[warmup + i], pos_list[i]) for i in range(steps)]
    return toks, pos_list, warm, timed


def perplexity_tokens(n_tok: int, vocab_size: int) -> np.ndarray:
    """The perplexity workload's input: n_tok tokens and the target after the last one, a fixed function of the arguments."""
    return np.random.default_rng(321).integers(3, vocab_size, size=n_tok + 1).astype(np.int32)


def perplexity_sample_rows(n_tok: int) -> np.ndarray:
    """The positions whose logits --dump-outputs keeps for the perplexity workload: a fixed, seeded sample (<= 64 MB at m7)."""
    return np.sort(np.random.default_rng(0).choice(n_tok, size=min(128, n_tok), replace=False))


def dump_outputs(d: str, **arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), np.asarray(a, dtype=np.float32))


def build_model_streaming(cfg_full: dict, cfg: dict, wtype, seed: int, keep_host: bool, std: float = 0.02, **cuda_kw):
    """Generate the synthetic checkpoint tensor by tensor and upload each as it is made (peak host RAM = one tensor
    unless keep_host, which the CPU baseline needs)."""
    import ctypes as C
    from xalm_b200 import capi, synth
    from xalm_b200.model import Model
    model = Model(cfg, {})
    L = capi.lib()
    h = C.c_void_p()
    xc = capi.XalmConfig.from_dict(cfg)
    capi.check(L.xalm_cuda_create(C.byref(xc), cuda_kw.get("device", 0), cuda_kw.get("tp_rank", 0), cuda_kw.get("tp_size", 1), C.byref(h)))
    model._h = h
    model.tp_rank, model.tp_size = cuda_kw.get("tp_rank", 0), cuda_kw.get("tp_size", 1)
    if cuda_kw.get("stream") is not None:
        capi.check(L.xalm_cuda_set_stream(h, C.c_void_p(cuda_kw["stream"])))
    if model.tp_size > 1:
        buf = (C.c_char * 128).from_buffer_copy(cuda_kw["comm_id"])
        capi.check(L.xalm_cuda_comm_init(h, buf))
        if cuda_kw.get("ipc_exchange") is not None:
            mine = (C.c_char * 64)()
            capi.check(L.xalm_cuda_ipc_export(h, mine))
            table = cuda_kw["ipc_exchange"](bytes(mine))
            tb = (C.c_char * len(table)).from_buffer_copy(table)
            capi.check(L.xalm_cuda_ipc_import(h, tb))
    from xalm_b200 import xalm_file as X
    shapes = X.expected_tensors(cfg)
    host = {}
    if model.tp_size > 1 and not keep_host:
        # shard-aware: this rank generates, quantises and uploads only the rows / columns it keeps (1/P of the host work and memory)
        for name, t, arr, rng in synth.iter_tensors(cfg_full, wtype, seed, std=std, shard_range=model.shard_range):
            model.upload_shard(name, t, shapes[name], rng, np.ascontiguousarray(arr).view(np.uint8).reshape(-1))
    else:
        for name, t, arr in synth.iter_tensors(cfg_full, wtype, seed, std=std):
            raw = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
            model.upload(name, t, shapes[name], raw)
            if keep_host:
                host[name] = (t.id, raw)
    capi.check(L.xalm_cuda_finalize(h))
    return model, host


def run_reference(args):
    """The reference's CPU implementation of the path (oracle port; DESIGN.md explains why the C++ cannot be built
    here) on all host cores.  Under torchrun only rank 0 works."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import oracle
    from xalm_b200 import synth, types as T, xalm_file as X
    cfg_full = synth.model_config(args.shape)
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    wtype = T.parse(args.wtype)
    cores = oracle.set_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: ask for every core
    synth.set_threads(cores)
    t0 = time.time()
    tensors = {name: (t.id, np.ascontiguousarray(arr).view(np.uint8).reshape(-1)) for name, t, arr in synth.iter_tensors(cfg_full, wtype, args.seed)}
    gen_s = time.time() - t0
    om = oracle.OracleModel(cfg, tensors, acc_mode=1)
    # the SAME positions as the GPU arm: spread uniformly over [0, ctx) (attention walks kv_len = pos + 1 rows of the fp16 ring)
    pos_list = positions_for(args.steps, cfg["max_seq_len"])
    tok = 1
    for i in range(args.warmup):
        lg = om.forward(tok, pos_list[min(i, len(pos_list) - 1)], 1)
        tok = oracle.sample_argmax(lg)
    t0 = time.perf_counter()
    for i in range(args.steps):
        lg = om.forward(tok, pos_list[i], 1)
        tok = oracle.sample_argmax(lg)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, logits=lg)
    tps = args.steps / dt
    sample = (f"{args.steps} tokens at positions spread uniformly over [0, {cfg['max_seq_len']}) — the GPU arm's positions — of the same "
              f"{args.shape} {args.wtype} model (full depth), wall clock")
    line = {
        "impl": "reference", "metric": "decode_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg),
        "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "notes": f"oracle/liboracle.so (restatement of src/infer.cpp), OpenMP over {cores} host cores; weights generated in {gen_s:.0f}s",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, cfg) -> dict:
    depth = f" DEPTH-REDUCED to {args.layers} layers" if getattr(args, "layers", 0) else ""
    return {"workload": (f"{args.shape} ({'Mistral-7B-v0.2' if args.shape == 'm7' else args.shape} architecture) random-init {args.wtype}, "
                         f"batch-1 decode, 4k context" if args.ctx == 4096 else f"{args.shape} {args.wtype} batch-1 decode ctx {args.ctx}") + depth,
            "n_layers": cfg["n_layers"],
            "shape": args.shape, "weight_format": args.wtype, "context": cfg["max_seq_len"], "batch": 1,
            "positions": "spread uniformly over [0, context)", "l2": "inputs larger than L2 (weights streamed from HBM every step)",
            "parallelism": f"tp{args.gpus}"}


def measured_peak_tflops() -> tuple:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["bf16_tflops"]), float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def gemm_flops(cfg: dict, T: int, with_cls: bool = True) -> float:
    """2*T*(weights that enter a GEMM): the seven per-layer contractions + the classifier (SURVEY.md 8d: 2*T*7.11e9 for m7)."""
    q_dim, kv_dim = cfg["n_heads"] * cfg["head_dim"], cfg["n_kv_heads"] * cfg["head_dim"]
    per_layer = cfg["dim"] * (q_dim + 2 * kv_dim) + q_dim * cfg["dim"] + 3 * cfg["dim"] * cfg["hidden_dim"]
    return 2.0 * T * (cfg["n_layers"] * per_layer + (cfg["vocab_size"] * cfg["dim"] if with_cls else 0))


def perplexity_summary(model, cfg, capi, n_tok: int) -> dict:
    """Device-timed tok/s of the batched perplexity pass (BASELINE config[2]) in both operand modes + its accuracy against
    the decode kernels, on the model bench.py already holds.  Full line: `bench.py --workload perplexity`."""
    import torch
    from xalm_b200.model import InferenceState
    toks = perplexity_tokens(n_tok, cfg["vocab_size"])
    out = {"tokens_per_step": n_tok, "metric": "perplexity_tokens_per_s"}
    st = InferenceState(cfg).cuda()
    for split, name in ((3, "precise_hi_lo_fp16"), (1, "plain_fp16")):
        capi.tune("prefill_split", split)
        for _ in range(2):
            model.prefill_async(toks[:-1], 0, 2)
        model.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            model.prefill_async(toks[:-1], 0, 2)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        lg_all, probs = model.prefill(toks[:-1], 0, want_logits=2, targets=toks[1:])
        worst = 0.0
        for pos in range(n_tok - 2, n_tok):
            model.forward(st, int(toks[pos]), pos, 1)
            worst = max(worst, float(np.max(np.abs(st.logits() - lg_all[pos]))))
        out[name] = {"value": n_tok / (ms / 1e3), "unit": "tok/s", "ms_per_step": ms, "gemm_tflops": gemm_flops(cfg, n_tok) / (ms / 1e3) / 1e12,
                     "max_abs_logit_diff_vs_decode_path": worst, "perplexity": float(np.exp(-np.mean(np.log(probs))))}
    capi.tune("prefill_split", 3)
    return out


def gemm_traffic(args, n_tok):
    """dram bytes of the gate|up GEMM from the committed ncu capture (profiles/kernel_traffic.json), when it is this workload"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        return d.get(f"{args.shape}_gemm_w13_T{n_tok}_bytes")
    except Exception:
        return None


def run_perplexity_workload(args):
    """BASELINE config[2]: perplexity mode on a 4k-token synthetic input.  A step = one batched pass over `--tokens` positions
    (every position's logits + softmax-at-target), weights resident.  `value` device-timed; `e2e` through Model.prefill with
    host tokens in and host probabilities out.  --impl reference: the oracle's token-at-a-time loop on a bounded sample."""
    from xalm_b200 import synth, types as T, xalm_file as X
    cfg_full = synth.model_config(args.shape)
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    wtype = T.parse(args.wtype)
    n_tok = min(args.tokens, cfg["max_seq_len"])
    toks = perplexity_tokens(n_tok, cfg["vocab_size"])
    config = {"workload": f"{args.shape} ({'Mistral-7B-v0.2' if args.shape == 'm7' else args.shape} architecture) random-init {args.wtype}, "
                          f"perplexity mode over a {n_tok}-token synthetic input (batched prefill, dequantised weights on tcgen05 GEMMs)",
              "shape": args.shape, "weight_format": args.wtype, "tokens_per_step": n_tok, "context": cfg["max_seq_len"],
              "l2": "inputs larger than L2 (7.5 GB of weights + 0.5 GB of logits per step)", "parallelism": "tp1"}
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        from oracle import oracle
        cores = oracle.set_threads(os.cpu_count() or 1)
        synth.set_threads(cores)
        tensors = {name: (t.id, np.ascontiguousarray(arr).view(np.uint8).reshape(-1)) for name, t, arr in synth.iter_tensors(cfg_full, wtype, args.seed)}
        om = oracle.OracleModel(cfg, tensors, acc_mode=1)
        n = max(1, args.steps)
        for i in range(max(1, args.warmup)):
            om.forward(int(toks[i]), i, 1)
        t0 = time.perf_counter()
        s = 0.0
        for i in range(n):
            lg = om.forward(int(toks[i]), i, 1)
            s += float(np.log(oracle.sample_prob(lg, int(toks[i + 1]))))
        dt = time.perf_counter() - t0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, logits=lg)
        tps = n / dt
        sample = f"positions 0..{n - 1} of the same input, one Model::forward + sample_prob each (main.cpp:244-254), wall clock"
        print(json.dumps({"impl": "reference", "metric": "perplexity_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": args.gpus,
                          "steps": n, "warmup": args.warmup, "ms_per_step": dt / n * 1e3, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return

    import torch
    from xalm_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the backend has no CPU fallback")
    if args.gpus != 1:
        raise SystemExit("the perplexity workload is single-GPU (the batched prefill path does not shard yet)")
    torch.cuda.set_device(0)
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    keep_host = not args.no_cpu_baseline
    synth.set_threads(os.cpu_count() or 8)
    model, host_tensors = build_model_streaming(cfg_full, cfg, wtype, args.seed, keep_host, device=0, stream=tstream.cuda_stream)
    split = args.split or 3
    capi.tune("prefill_split", split)
    steps, warm = max(1, args.steps), max(3, args.warmup)
    for _ in range(warm):
        model.prefill_async(toks[:-1], 0, 2)
    model.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            model.prefill_async(toks[:-1], 0, 2)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = model.last_launch_count() * steps
        # end to end: host tokens + targets in, host probabilities out, log + mean on the host (main.cpp:251-258)
        for _ in range(2):
            model.prefill(toks[:-1], 0, want_logits=2, targets=toks[1:], fetch_logits=False)
        t0 = time.perf_counter()
        for _ in range(steps):
            _, probs = model.prefill(toks[:-1], 0, want_logits=2, targets=toks[1:], fetch_logits=False)
            ppl = float(np.exp(-np.mean(np.log(probs))))
        e2e_s = time.perf_counter() - t0
    tps = n_tok * steps / (ms / 1e3)
    e2e_tps = n_tok * steps / e2e_s
    burst, sustained, src = measured_peak_tflops()
    # dominant kernel: the fused gate|up GEMM (2*T*2*hidden*dim flops), timed alone
    N13, K13 = 2 * cfg["hidden_dim"], cfg["dim"]
    k_ms = capi.bench_gemm(n_tok, N13, K13, split, 20)
    mmas = {1: 1, 2: 2, 3: 3}[split]
    k_tf = 2.0 * n_tok * N13 * K13 / (k_ms / 1e3) / 1e12
    step_tf = gemm_flops(cfg, n_tok) * steps / (ms / 1e3) / 1e12
    # accuracy of this mode against the token-at-a-time decode kernels on the same KV prefix (last 4 positions)
    from xalm_b200.model import InferenceState
    lg_all = model.prefill(toks[:-1], 0, want_logits=2)
    if args.dump_outputs:
        # the timed step is a pure function of (weights, tokens, position 0): this pass recomputes exactly its logits
        dump_outputs(args.dump_outputs, logits_sample=lg_all[perplexity_sample_rows(n_tok)])
    st = InferenceState(cfg).cuda()
    worst = 0.0
    for pos in range(n_tok - 4, n_tok):
        model.forward(st, int(toks[pos]), pos, 1)
        worst = max(worst, float(np.max(np.abs(st.logits() - lg_all[pos]))))
    line = {
        "metric": "perplexity_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16 operands (hi+lo pairs) / f32 accumulate" if split == 3 else "f16 operands / f32 accumulate", "data": "synthetic", "config": config,
        "e2e": {"value": e2e_tps, "unit": "tok/s", "h2d_bytes_per_step": int(2 * n_tok * 4), "d2h_bytes_per_step": int(n_tok * 4),
                "perplexity": ppl},
        "gpu_launches": launches, "clocks": clocks.summary(),
        "roofline": {"bound": "tensor", "achieved": k_tf, "peak": burst, "unit": "TFLOP/s", "frac": k_tf / burst, "traffic": gemm_traffic(args, n_tok),
                     "kernel": f"gemm_tc_kernel (tcgen05, 128x256x64 tiles) gate|up {n_tok}x{N13}x{K13}", "ms_per_launch": k_ms,
                     "mma_per_product": mmas, "issued_tflops": k_tf * mmas, "issued_frac": k_tf * mmas / burst, "peak_source": src,
                     "note": "achieved counts ALGORITHMIC flops 2*T*N*K; precision mode 3 issues 3 fp16 MMAs per product (hi.hi + lo.hi + hi.lo)"},
        "step_roofline": {"flops_per_step": gemm_flops(cfg, n_tok), "achieved": step_tf, "peak": sustained, "unit": "TFLOP/s",
                          "frac": step_tf / sustained, "note": "GEMM flops only (attention excluded) over the whole step vs the sustained cuBLAS figure"},
        "accuracy": {"max_abs_logit_diff_vs_decode_path": worst, "positions": 4, "tolerance": 1e-2, "prefill_split": split},
    }
    if keep_host:
        from oracle import oracle
        cores = oracle.set_threads(os.cpu_count() or 1)
        om = oracle.OracleModel(cfg, host_tensors, acc_mode=1)
        om.forward(int(toks[0]), 0, 1)
        n = args.cpu_tokens
        t0 = time.perf_counter()
        for i in range(n):
            lg = om.forward(int(toks[i]), i, 1)
            oracle.sample_prob(lg, int(toks[i + 1]))
        cdt = time.perf_counter() - t0
        om.close()
        line["cpu_baseline"] = {"value": n / cdt, "unit": "tok/s", "cores": cores, "kind": "port",
                                "sample": f"positions 0..{n - 1} of the same input, one forward + sample_prob each, wall clock"}
    print(json.dumps(line), flush=True)
    model.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="m7")
    ap.add_argument("--wtype", default="q8_0")
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-tokens", type=int, default=6, help="tokens the CPU baseline decodes (rank 0, N=1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the greedy-token parity check against the CPU oracle after the timed region")
    ap.add_argument("--parity-tokens", type=int, default=8)
    ap.add_argument("--layers", type=int, default=0, help="depth-reduced variant of --shape (stated in config.workload); 0 = full depth")
    ap.add_argument("--past-window", action="store_true",
                    help="also time steps at positions >= ctx: the KV ring is full (kv_len = ctx), 2 attention sinks active (infer.cpp:608-613)")
    ap.add_argument("--no-prefill", action="store_true", help="skip the perplexity-mode summary appended to the decode line at N=1")
    ap.add_argument("--workload", default="decode", choices=["decode", "perplexity"],
                    help="decode = BASELINE config[1] (the headline metric); perplexity = config[2]: batched prefill of a 4k-token input")
    ap.add_argument("--tokens", type=int, default=4096, help="perplexity workload: tokens per step")
    ap.add_argument("--split", type=int, default=0, help="perplexity workload: operand precision (0 = library default 3; 1 = plain fp16)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/*.npy (float32; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    if args.workload == "perplexity":
        run_perplexity_workload(args)
        return
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from xalm_b200 import capi, synth, types as T, xalm_file as X
    from xalm_b200.model import InferenceState, Sampler

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    from xalm_b200 import synth as _synth
    _synth.set_threads(max(1, (os.cpu_count() or 8) // world))   # torchrun exports OMP_NUM_THREADS=1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg_full = synth.model_config(args.shape, **({"n_layers": args.layers} if args.layers else {}))
    cfg = X.parse_config(synth.metadata_strings(cfg_full), args.ctx)
    wtype = T.parse(args.wtype)
    comm_id = None
    if world > 1:
        from xalm_b200.model import Model
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.frombuffer(bytearray(Model.comm_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(idt, 0)
        comm_id = bytes(idt.cpu().numpy().tobytes())
    # a dedicated (non-default) torch stream: the backend launches on it and torch.cuda.Event times it
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    keep_host = rank == 0 and not args.no_parity      # rank 0 keeps the full checkpoint: parity check at every N, CPU baseline at N = 1
    t0 = time.time()
    ipc_exchange = None
    if world > 1 and os.environ.get("XALM_TP_PEER", "1") != "0":
        from xalm_b200 import tp as _tp
        ipc_exchange = _tp.make_ipc_exchange(dist, world)
    model, host_tensors = build_model_streaming(cfg_full, cfg, wtype, args.seed, keep_host, device=local_rank, tp_rank=rank,
                                                tp_size=world, comm_id=comm_id, stream=stream, ipc_exchange=ipc_exchange)
    gen_s = time.time() - t0
    ctx = cfg["max_seq_len"]
    toks, pos_list, warm_steps, timed_steps = decode_inputs(args.steps, args.warmup, ctx, cfg["vocab_size"])

    # ---- device-timed: weights and KV resident, logits stay on the device ----
    for tok, pos in warm_steps:
        model.forward_async(tok, pos, 1)
    model.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        e0.record()
        for tok, pos in timed_steps:
            model.forward_async(tok, pos, 1)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = model.last_launch_count() * args.steps
        if args.dump_outputs and rank == 0:
            # read now: the end-to-end loops below overwrite the device logits
            dump_outputs(args.dump_outputs, logits=model.read_state(capi.S_LOGITS, cfg["vocab_size"]))
        # ---- end to end through the public API: host token in, host logits out, host sampler ----
        state = InferenceState(cfg).cuda()
        sampler = Sampler(cfg)
        tok = toks[0]
        for i in range(3):
            model.forward(state, tok, pos_list[i % len(pos_list)], 1)
            tok = sampler.sample_argmax(state)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            model.forward(state, tok, pos_list[i], 1)
            tok = sampler.sample_argmax(state)
        barrier()
        e2e_s = time.perf_counter() - t0
        # same loop with the sampler on the device: 4 bytes back per token instead of the logits
        tok = toks[0]
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            tok = model.forward_argmax(tok, pos_list[i])
        barrier()
        e2e_dev_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])
    tps = args.steps / (ms / 1e3)
    e2e_tps = args.steps / e2e_s
    past = None
    if args.past_window:
        n = min(args.steps, 64)
        for i in range(3):
            model.forward_async(toks[i], ctx + i, 1)
        model.sync()
        barrier()
        e0.record()
        for i in range(n):
            model.forward_async(toks[i], ctx + 3 + i, 1)
        e1.record()
        barrier()
        pms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([pms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pms = float(t[0])
        pb = float(model.active_bytes(ctx + 3))
        past = {"positions": f"{ctx + 3}..{ctx + 2 + n} (ring full: kv_len = {ctx}, 2 attention sinks re-rotated every step)", "steps": n,
                "value": n / (pms / 1e3), "unit": "tok/s", "ms_per_step": pms / n, "bytes_per_step_this_rank": pb,
                "achieved_gbs_this_rank": pb * n / (pms / 1e3) / 1e9}

    # ---- parity, in the record the driver keeps: the (sharded) model and the CPU oracle decode the same prompt greedily ----
    parity = None
    if not args.no_parity:
        prompt = [1] + [int(t) for t in np.random.default_rng(7).integers(3, cfg["vocab_size"], size=3)]
        pstate = InferenceState(cfg).cuda()
        psampler = Sampler(cfg)
        # The GPU ranks decode first, in lock step (a rank that stopped to run the CPU oracle between tokens would leave its peers
        # spinning in the tensor-parallel exchange until their timeout); rank 0 keeps every step's logits and replays the oracle after.
        if world > 1:
            dist.barrier()
        for p_, t_ in enumerate(prompt):
            model.forward(pstate, t_, p_, 1 if p_ + 1 == len(prompt) else 0)
        seq_g, lg_g = list(prompt), []
        for _ in range(args.parity_tokens):
            tg = psampler.sample_argmax(pstate)
            if rank == 0:
                lg_g.append(np.array(pstate.logits(), dtype=np.float32, copy=True))
            seq_g.append(tg)
            model.forward(pstate, tg, len(seq_g) - 1, 1)
        om = None
        if rank == 0:
            from oracle import oracle
            oracle.set_threads(max(1, (os.cpu_count() or 1)))
            om = oracle.OracleModel(cfg, host_tensors, acc_mode=1)
            lg_o = None
            for p_, t_ in enumerate(prompt):
                lg_o = om.forward(t_, p_, 1 if p_ + 1 == len(prompt) else 0)
            seq_o, worst = list(prompt), 0.0
            for i in range(args.parity_tokens):
                if seq_o == seq_g[: len(seq_o)]:      # same history so far: the logits are comparable
                    worst = max(worst, float(np.max(np.abs(lg_g[i] - lg_o))))
                to = oracle.sample_argmax(lg_o)
                seq_o.append(to)
                if i + 1 < args.parity_tokens:
                    lg_o = om.forward(to, len(seq_o) - 1, 1)
            seq_g = seq_g[: len(seq_o)]
        if om:
            om.close()
            parity = {"tokens_match": seq_g == seq_o, "max_abs_logit": worst, "tolerance": 1e-2, "greedy_tokens": args.parity_tokens,
                      "prompt_tokens": len(prompt), "against": "oracle/liboracle.so on rank 0 (restatement of src/infer.cpp, itself pinned to the "
                      "reference's own C++ by tests/golden/ref_fwd_*.npz), same checkpoint, full depth", "tokens": seq_g[len(prompt):]}

    # ---- roofline: whole step, and the dominant kernel (fused norm + gate|up matvec) timed alone ----
    peak, peak_src = measured_peak_gbs()
    step_bytes = float(np.mean([model.active_bytes(p) for p in pos_list]))          # this rank's shard
    step_gbs = step_bytes * args.steps / (ms / 1e3) / 1e9
    hidden_l = cfg["hidden_dim"] // world
    k_bytes = 2 * hidden_l * cfg["dim"] * wtype.bytes // wtype.block
    nbuf = max(2, int(np.ceil(600e6 / k_bytes)))
    # which matvec the MODEL runs for this format and sharding (xalm_cuda.cu: alloc_wmat): the tensor-core kernel (matvec_mma.cuh) for the
    # 4/5-bit formats and, under tensor parallelism, for the 8-bit ones; the dp4a kernel (matvec_idp.cuh) for 8-bit on one GPU
    int_fmt = args.wtype in ("q8_0", "q8", "q4_0", "q4_1", "q5_0", "q5_1")
    mma_mode = int(os.environ.get("XALM_MMA", "2"))
    mma_kernel = int_fmt and (2 * hidden_l) % 16 == 0 and (mma_mode == 1 or (mma_mode == 2 and (world > 1 or args.wtype not in ("q8_0", "q8"))))
    idp_kernel = int_fmt and not mma_kernel and cfg["dim"] % 256 == 0 and (2 * hidden_l) % 8 == 0
    if mma_kernel:
        capi.tune("mma", 1)      # the stand-alone timing takes the same kernel as the sharded model
    k_ms = capi.bench_matvec(wtype.id, cfg["dim"], hidden_l, nbuf, 200, epi=2, with_norm=True)
    if mma_kernel:
        capi.tune("mma", mma_mode)
    k_gbs = k_bytes / (k_ms / 1e3) / 1e9
    kname = "matvec_mma_kernel" if mma_kernel else "matvec_idp_kernel" if idp_kernel else "matvec_tma_kernel"
    traffic = None
    prof = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get(f"{args.shape}_{args.wtype}_w13_{kname}_tp{world}_bytes")   # null unless captured for this kernel AND shard
        except Exception:
            traffic = None

    line = {
        "metric": "decode_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": ("f32 activations and accumulation; integer weight formats multiply in int8 (" + ("mma.sync m16n8k32 u8" if mma_kernel else "dp4a") +
                  ") against 3 x int8 block-floating activation limbs") if (idp_kernel or mma_kernel) else "f32",
        "data": "synthetic", "config": workload_config(args, cfg),
        "e2e": {"value": e2e_tps, "unit": "tok/s", "h2d_bytes_per_step": 32, "d2h_bytes_per_step": cfg["vocab_size"] * 4,
                "device_sampler": {"value": args.steps / e2e_dev_s, "unit": "tok/s", "d2h_bytes_per_step": 4,
                                   "api": "xalm_cuda_forward_argmax (Sampler::sample_argmax on the device)"}},
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "roofline": {"bound": "hbm", "achieved": k_gbs, "peak": peak, "unit": "GB/s", "frac": k_gbs / peak, "traffic": traffic,
                     "kernel": f"{kname}<{args.wtype}, norm> (norm + gate|up + GLU) {2 * hidden_l}x{cfg['dim']}", "bytes_per_launch": k_bytes,
                     "ms_per_launch": k_ms, "peak_source": peak_src, "timing": "CUDA events around 200 back-to-back launches on rotating buffers > L2"},
        "step_roofline": {"bytes_per_step": step_bytes, "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                          "frac_of_8000": step_gbs / 8000.0, "formula": "Model::active_bytes(pos) (model.cpp:12-35), mean over the timed positions"},
        "notes": f"weights generated+uploaded in {gen_s:.0f}s; host cores {os.cpu_count()}",
    }
    if past:
        line["past_window"] = past
    if parity is not None:
        line["parity"] = parity

    # ---- BASELINE config[2] beside it (N = 1): the batched prefill / perplexity pass on the same resident model ----
    if world == 1 and not args.no_prefill and cfg["head_dim"] in (64, 128):
        try:
            line["perplexity_mode"] = perplexity_summary(model, cfg, capi, min(4096, ctx))
        except Exception as ex:  # never lose the decode line to the secondary measurement
            line["perplexity_mode"] = {"error": str(ex)[:200]}

    # ---- CPU baseline beside it: the oracle port on the host cores, same weights (rank 0, N = 1 only) ----
    if keep_host and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        cpu_cores = oracle.set_threads(os.cpu_count() or 1)
        om = oracle.OracleModel(cfg, host_tensors, acc_mode=1)
        tok = 1
        lg = om.forward(tok, 0, 1)          # warm-up (touches every page)
        n = args.cpu_tokens
        cpos = positions_for(n, ctx)        # spread over the context like the timed GPU steps
        t0 = time.perf_counter()
        for i in range(n):
            tok = oracle.sample_argmax(lg)
            lg = om.forward(tok, cpos[i], 1)
        cdt = time.perf_counter() - t0
        om.close()
        line["cpu_baseline"] = {"value": n / cdt, "unit": "tok/s", "cores": cpu_cores, "kind": "port",
                                "sample": f"{n} tokens at positions spread uniformly over [0, {ctx}) of the same model (full depth, same weights), wall clock"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()      # peers keep their exchange buffers mapped until rank 0 is through with the oracle replay
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
