"""torchrun worker: the batched prefill (xalm_cuda_prefill / xalm_cuda_prefill_window) on a tensor-parallel model of WORLD_SIZE
GPUs, against the CPU oracle run token by token (rank 0), the token loop on a second TP handle set, and the unsharded model.
   python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29621 \\
       tests/tp_prefill_worker.py [wtype] [shape] [head_dim]
XALM_TP_PEER=0 runs the decode exchange through NCCL instead of the fused peer-memory path."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist

from xalm_b200 import capi, synth, tp
from xalm_b200 import types as T
from xalm_b200 import xalm_file as X
from xalm_b200.model import InferenceState, Model, Sampler

W = 256          # max_seq_len: a 200-token prompt, a second linear chunk, then window chunks over more than three windows
N_FIRST = 200
XALM_ERR_INVALID = 1  # include/xalm_cuda.h


def window_chunks(S, total):
    """Window chunk sizes covering `total` positions: mixed sizes, including 1 and the largest allowed (S = W - 2)."""
    pattern = [1, S, 17, S - 3, 5, S, 2]
    out, left, i = [], total, 0
    while left > 0:
        out.append(min(pattern[i % len(pattern)], left))
        left -= out[-1]
        i += 1
    return out


def main():
    wtype = sys.argv[1] if len(sys.argv) > 1 else "q8_0"
    shape = sys.argv[2] if len(sys.argv) > 2 else "tp"
    over = dict(head_dim=int(sys.argv[3])) if len(sys.argv) > 3 else {}
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    c = synth.model_config(shape, n_layers=2, **over)   # two layers, as the single-GPU window tests: the bounds are depth-dependent
    cfg = X.parse_config(synth.metadata_strings(c), W)
    assert cfg["max_seq_len"] == W
    V, L, hd = cfg["vocab_size"], cfg["n_layers"], cfg["head_dim"]
    kvd = cfg["n_kv_heads"] * hd
    kvl = kvd // world
    tensors = list(synth.iter_tensors(c, T.parse(wtype), seed=3, std=0.03))
    use_peer = os.environ.get("XALM_TP_PEER", "1") != "0"

    def tp_model():
        comm_id = tp.broadcast_comm_id(dist, rank, device="cuda")
        ipc = tp.make_ipc_exchange(dist, world) if use_peer else None
        return Model.from_tensors(cfg, tensors).cuda(device=local, tp_rank=rank, tp_size=world, comm_id=comm_id, ipc_exchange=ipc)

    gm = tp_model()    # batched prefill
    gm2 = tp_model()   # the token loop past the window, for the sink keys
    fails = []

    def check(ok, what):
        if not ok:
            fails.append(f"rank {rank}: {what}")

    S = W - 2
    chunks = window_chunks(S, 3 * W + 5)
    n = W + sum(chunks)
    rng = np.random.default_rng(11)
    tokens = rng.integers(3, V, size=n + 1 + 16).astype(np.int32)
    targets = tokens[1:n + 1]
    kv = lambda m: [[m.read_kv(l, w).copy() for w in (0, 1)] for l in range(L)]

    # ---- linear regime: the first chunk twice (determinism), then a second chunk at pos0 > 0 ----
    lg1, pr1 = gm.prefill(tokens[:N_FIRST], 0, want_logits=2, targets=targets[:N_FIRST])
    kv1 = kv(gm)
    lg1b, _ = gm.prefill(tokens[:N_FIRST], 0, want_logits=2, targets=targets[:N_FIRST])
    check(np.array_equal(lg1.view(np.uint32), lg1b.view(np.uint32)), "the same prefill twice gave different logits")
    check(all(np.array_equal(a, b) for x, y in zip(kv1, kv(gm)) for a, b in zip(x, y)), "the same prefill twice gave different KV shards")
    lg2, pr2 = gm.prefill(tokens[N_FIRST:W], N_FIRST, want_logits=2, targets=targets[N_FIRST:W])
    kv_lin = kv(gm)
    gm2.prefill(tokens[:N_FIRST], 0, want_logits=0)   # the second handle set hydrates [0, W) the same way
    gm2.prefill(tokens[N_FIRST:W], N_FIRST, want_logits=0)
    # ---- window regime ----
    lgs, prs, pos = [lg1, lg2], [pr1, pr2], W
    for ch in chunks:
        lg, pr = gm.prefill_window(tokens[pos:pos + ch], pos, want_logits=2, targets=targets[pos:pos + ch])
        lgs.append(lg); prs.append(pr)
        pos += ch
    got, probs = np.concatenate(lgs), np.concatenate(prs)
    kv_win = kv(gm)
    st2 = InferenceState(cfg).cuda()
    for p in range(W, n):
        gm2.forward(st2, int(tokens[p]), p, 0)
    sinks2 = kv(gm2)
    for l in range(L):
        for w in (0, 1):
            check(np.array_equal(kv_win[l][w][: 2 * kvl], sinks2[l][w][: 2 * kvl]), f"layer {l} {'kv'[w]}: sink rows differ from the token loop")

    # every rank holds the full logits, bit for bit the same
    ref_bits = torch.from_numpy(got.view(np.int32).copy()).cuda()
    dist.broadcast(ref_bits, 0)
    check(np.array_equal(ref_bits.cpu().numpy(), got.view(np.int32)), "logits differ between ranks")

    # ---- decode continues on the TP handles after the prefill ----
    state, sampler = InferenceState(cfg).cuda(), Sampler(cfg)
    state.logits()[:] = got[-1]
    seq_g, lg_dec = [], []
    for i in range(16):
        tg = sampler.sample_argmax(state)
        seq_g.append(tg)
        gm.forward(state, tg, n + i, 1)
        lg_dec.append(state.logits().copy())

    # ---- the oracle (rank 0) and the unsharded model on rank 0's GPU ----
    o_kv_lin = np.zeros((L, 2, W, kvd), dtype=np.float32)
    o_kv_win = np.zeros_like(o_kv_lin)
    if rank == 0:
        from oracle import oracle
        om = oracle.OracleModel(cfg, {nm: (t.id, np.ascontiguousarray(a).view(np.uint8).reshape(-1)) for nm, t, a in tensors})
        ref = np.empty((n, V), dtype=np.float32)
        okv = lambda: np.stack([np.stack([om.kv(l, w).view(np.float16).astype(np.float32)[: W * kvd].reshape(W, kvd) for w in (0, 1)])
                                for l in range(L)])
        for p in range(n):
            ref[p] = om.forward(int(tokens[p]), p, 1)
            if p == W - 1:
                o_kv_lin = okv()
        o_kv_win = okv()
        diff_lin = float(np.max(np.abs(got[:W] - ref[:W])))
        diff_win = float(np.max(np.abs(got[W:] - ref[W:])))
        # the project's 1e-2 contract: on these shapes the one-GPU prefill itself measured up to 2.3e-3 (linear) and 6.5e-3 (window)
        # from the oracle on a B200; what sharding adds is held to 1e-3 against the one-GPU prefill below
        check(diff_lin <= 1e-2, f"linear prefill logits differ from the oracle by {diff_lin:.2e}")
        check(diff_win <= 1e-2, f"window prefill logits differ from the oracle by {diff_win:.2e}")
        ref_lp = np.log([oracle.sample_prob(ref[p], int(targets[p])) for p in range(n)])
        lp = np.log(probs)
        dlp = float(np.max(np.abs(lp - ref_lp)))
        ppl_ref, ppl = np.exp(-np.mean(ref_lp)), np.exp(-np.mean(lp))
        check(dlp <= 2e-2, f"log-probabilities differ from the oracle by {dlp:.2e}")
        check(abs(ppl - ppl_ref) <= 2e-3 * ppl_ref, f"perplexity {ppl} vs {ppl_ref}")
        seq_o, lg_o, dmax = [], ref[-1], 0.0
        for i in range(16):
            to = oracle.sample_argmax(lg_o)
            seq_o.append(to)
            lg_o = om.forward(to, n + i, 1)
            if seq_o == seq_g[: i + 1]:
                dmax = max(dmax, float(np.max(np.abs(lg_dec[i] - lg_o))))
        check(seq_o == seq_g, "decode after the prefill diverges from the oracle")
        check(dmax <= 1e-2, f"decode logits after the prefill differ from the oracle by {dmax:.2e}")
        om.close()
        one = Model.from_tensors(cfg, tensors).cuda(device=local)
        one_lg = [one.prefill(tokens[:N_FIRST], 0, want_logits=2), one.prefill(tokens[N_FIRST:W], N_FIRST, want_logits=2)]
        pos = W
        for ch in chunks:
            one_lg.append(one.prefill_window(tokens[pos:pos + ch], pos, want_logits=2))
            pos += ch
        diff_one = float(np.max(np.abs(got - np.concatenate(one_lg))))
        check(diff_one <= 1e-3, f"TP logits differ from the one-GPU prefill by {diff_one:.2e}")
        one.close()
        print(f"TP{world} {wtype} {shape} hd{hd}: oracle linear {diff_lin:.2e} window {diff_win:.2e} logprob {dlp:.2e} "
              f"ppl {ppl:.4f}/{ppl_ref:.4f} decode {dmax:.2e} vs one GPU {diff_one:.2e}")

    # ---- each rank's KV shard against the oracle's columns for its kv heads (data slots; the sinks are checked above) ----
    okv_t = torch.from_numpy(np.stack([o_kv_lin, o_kv_win])).cuda()
    dist.broadcast(okv_t, 0)
    okv_all = okv_t.cpu().numpy()
    cols = slice(rank * kvl, (rank + 1) * kvl)
    for phase, mine in ((0, kv_lin), (1, kv_win)):
        for l in range(L):
            for w in (0, 1):
                a = mine[l][w].view(np.float16).astype(np.float32).reshape(W, kvl)
                b = okv_all[phase, l, w][:, cols]
                r0 = 0 if phase == 0 else 2
                tol = 1e-2 * max(1.0, float(np.abs(b[r0:]).max()))
                check(np.max(np.abs(a[r0:] - b[r0:])) <= tol, f"{('linear', 'window')[phase]} KV layer {l} {'kv'[w]} differs from the oracle")

    # ---- refusals: every rank refuses alike, the cache is untouched, the next valid call succeeds ----
    before = kv(gm)
    p_next = n + 16
    bad = [("prefill", np.array([5, V, 7], dtype=np.int32), 0),           # token out of range
           ("prefill_window", tokens[: S + 1], p_next),                  # n past the ring
           ("prefill_window", tokens[:1], W - 1)]                        # pos0 below the window
    for which, toks, pos0 in bad:
        try:
            getattr(gm, which)(toks, pos0, want_logits=2)
            check(False, f"{which} at {pos0} with {toks.size} tokens was not refused")
        except capi.XalmError as e:
            check(e.status == XALM_ERR_INVALID, f"{which}: {e}")
    after = kv(gm)
    check(all(np.array_equal(a, b) for x, y in zip(before, after) for a, b in zip(x, y)), "a refused call changed the KV cache")
    lg_next = gm.prefill_window(tokens[:4], p_next, want_logits=1)
    check(lg_next.shape == (V,) and np.all(np.isfinite(lg_next)), "the call after the refusals failed")

    ok = torch.tensor([0 if fails else 1], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    for f in fails:
        print(f, flush=True)
    if rank == 0 and int(ok[0]) == 1:
        print("TP prefill ok", flush=True)
    gm.close(); gm2.close()
    dist.destroy_process_group()
    sys.exit(0 if int(ok[0]) == 1 else 1)


if __name__ == "__main__":
    main()
