"""GPU probe: whole-token device time of the m7 model under different tuning knobs (weights generated once)."""
import os, sys, time, json, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from xalm_b200 import capi, synth, types as T, xalm_file as X
from xalm_b200.model import Model
import bench

shape = os.environ.get("SHAPE", "m7")
wtype = T.parse(os.environ.get("WTYPE", "q8_0"))
cfg_full = synth.model_config(shape)
if os.environ.get("LAYERS"):
    cfg_full["n_layers"] = int(os.environ["LAYERS"])
cfg = X.parse_config(synth.metadata_strings(cfg_full), 4096)
torch.cuda.set_device(0)
st = torch.cuda.Stream()
t0 = time.time()
tensors = list(synth.iter_tensors(cfg_full, wtype, 0))
print(f"generated in {time.time()-t0:.0f}s", flush=True)
configs = [eval(a) for a in sys.argv[1:]] or [dict()]
K = 64
pos = bench.positions_for(K, 4096)
for kn in configs:
    for k, v in kn.items():
        capi.tune(k, v)
    model = Model.from_tensors(cfg, tensors).cuda(device=0, stream=st.cuda_stream)
    for i in range(4):
        model.forward_async(5, pos[i], 1)
    model.sync()
    res = []
    for plist, label in ((pos, "spread"), (list(range(K)), "pos0-63")):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(st)
        t0 = time.perf_counter()
        for i in range(K):
            model.forward_async(5, plist[i], 1)
        t_cpu = time.perf_counter() - t0
        e1.record(st)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        byts = np.mean([model.active_bytes(p) for p in plist])
        res.append(f"{label}: {ms/K:.3f} ms/tok {K/(ms/1e3):.0f} tok/s {byts*K/(ms/1e3)/1e9:.0f} GB/s (cpu {t_cpu/K*1e3:.3f} ms)")
    print(kn, " | ".join(res), f"launches/token {model.last_launch_count()}", flush=True)
    if os.environ.get("TIMELINE"):
        P = int(os.environ["TIMELINE"])
        capi.timeline_start(800)
        model.forward_async(5, P, 1)
        model.sync()
        tl = capi.timeline_stop(800).astype(np.int64)
        t0 = tl[:, 1].min()
        names = {100: "tma_store", 101: "tma_resid", 102: "tma_glu", 103: "tma_qkv", 200: "ldg_store", 201: "ldg_resid", 202: "ldg_glu", 203: "ldg_qkv", 300: "attn"}
        order = np.argsort(tl[:, 1])
        prev_end = None
        rows = []
        for i in order[: int(os.environ.get('TL_ROWS', 5 * 4 + 3))]:
            kid, a, b, c = tl[i]
            if kid >= 500:
                rows.append(f"      event {int(kid)} at {(a-t0)/1e3:8.2f}us")
                continue
            rows.append(f"  {str(names.get(int(kid), kid)):10s} entry {(a-t0)/1e3:8.2f}us  wait_done {(b-t0)/1e3:8.2f}  exit {(c-t0)/1e3:8.2f}  | entry->wait {(b-a)/1e3:6.2f}  work {(c-b)/1e3:6.2f}" + (f"  gap_from_prev_exit {(b-prev_end)/1e3:6.2f}" if prev_end else ""))
            prev_end = c
        print("\n".join(rows))
        tot = (tl[:, 3].max() - t0) / 1e3
        work = {}
        for kid, a, b, c in tl:
            if kid >= 500:
                continue
            work.setdefault(names.get(int(kid), kid), []).append((c - b) / 1e3)
        print(f"  token total {tot:.1f}us;", {k: (len(v), round(float(np.mean(v)), 2)) for k, v in work.items()})
    model.close()
