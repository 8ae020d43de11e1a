"""Row-range sharded exact dense search (dense.ShardedIndexFlatL2) over the wiki-sized embedding matrix on the GPUs of
one box: one JSON line per (G, k, batch), G = 1, 2, 4, 8 GPUs measured in the same run.

    torchrun --nproc-per-node 8 tools/bench_dense_sharded.py [--n 21015324] [--d 768] [--ks 5,10]
                                                             [--batches 1,8,64,512] [--gpus 1,2,4,8] [--out FILE]

The workload is tools/bench_dense.py's: synthetic clustered rows (synth.dense_rows), queries perturbed copies of random
rows (synth.dense_queries).  For each G the first G ranks build only their own rows, sharding.shard_range(n, rank, G),
and the same query batches from the shape alone (synth.dense_queries_of); the other ranks wait.  Per setting:
warm-up calls, then CUDA events around --iters calls ending in a synchronise, on every rank; the line reports the
largest time over the ranks.  Two windows are timed:
  call_ms      ShardedIndexFlatL2.search: local search + all-gather of the [B, k] lists + pr_flat_merge
  local_ms     the local IndexFlatL2.search alone, so the gather + merge share is call_ms - local_ms
Bytes per shard are computed as tools/bench_dense.py computes them for the largest shard: the bf16 copy and the norms
once per block of <= 256 queries, plus the candidates' fp32 rows.
parity_checked: 16 queries of the merged result against the oracle's order -- every rank evaluates the oracle's exact
distances (oracle.flat_oracle, torch form, on the device) over its own rows, the per-rank lists are all-gathered and
merged with the CPU restatement of the merge (tests/flat_merge_oracle.py), and must equal the GPU result.
result_digest: sha256 of the merged (D, I) of the timed batch; identical for every G when sharding changes nothing.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), HERE]

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from bench_dense import card, peaks  # noqa: E402
from flat_merge_oracle import merge_canonical  # noqa: E402
from oracle import flat_oracle as fo  # noqa: E402
from probing_rag_b200 import IndexFlatL2, ShardedIndexFlatL2, sharding, synth  # noqa: E402


def local_oracle(Q, X, k, chunk=1 << 21):
    """(D, I) [B, k] of the oracle's exact distances over this rank's rows X (local ids), (FLT_MAX, -1) padded."""
    B = Q.shape[0]
    D = torch.full((B, k), float(fo.FLT_MAX), dtype=torch.float32, device=Q.device)
    I = torch.full((B, k), -1, dtype=torch.int64, device=Q.device)
    for b in range(B):
        best_d = torch.empty(0, dtype=torch.float32, device=Q.device)
        best_i = torch.empty(0, dtype=torch.int64, device=Q.device)
        for a in range(0, X.shape[0], chunk):
            dist_ = fo.exact_distances_torch(Q[b], X[a:a + chunk])
            cd = torch.cat([best_d, dist_])
            ci = torch.cat([best_i, torch.arange(a, a + dist_.numel(), device=Q.device)])
            s, o = torch.sort(cd, stable=True)      # ci ascending within equal distances: canonical order
            best_d, best_i = s[:k], ci[o[:k]]
        D[b, :best_d.numel()] = best_d
        I[b, :best_i.numel()] = best_i
    return D, I


def timed(fn, iters, warmup, group, dev):
    """Milliseconds per call, the largest over the ranks of `group`."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    dist.barrier(group=group)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=group)
    return float(ms.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=synth.N_DOCS_WIKI)
    ap.add_argument("--d", type=int, default=768)
    ap.add_argument("--ks", default="5,10")
    ap.add_argument("--batches", default="1,8,64,512")
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_dense_sharded.py measures on CUDA devices"
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    Gs = [g for g in (int(s) for s in args.gpus.split(",")) if g <= world]
    groups = {G: dist.new_group(list(range(G))) for G in Gs}
    cards = [None] * world
    dist.all_gather_object(cards, card())
    hbm, tf, peak_src = peaks()
    N, d = args.n, args.d
    ks = [int(s) for s in args.ks.split(",")]
    batches = [int(s) for s in args.batches.split(",")]
    out = open(args.out, "a") if (args.out and rank == 0) else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    Qs = {B: synth.dense_queries_of(N, d, B, device=dev) for B in batches}
    Qp = synth.dense_queries_of(N, d, 16, device=dev, seed=99)
    base_ms = {}
    for G in Gs:
        grp = groups[G]
        if rank < G:
            t0 = time.perf_counter()
            lo, hi = sharding.shard_range(N, rank, G)
            shard = IndexFlatL2(d, dev)
            shard.add(synth.dense_rows(N, d, device=dev, row_lo=lo, row_hi=hi))
            ix = ShardedIndexFlatL2(shard, lo, grp)
            ix.search(Qs[batches[0]], 1)                                  # builds the bf16 copy and the norms
            torch.cuda.synchronize()
            build_s = time.perf_counter() - t0
            # parity: the merged lists against the oracle's order, evaluated shard by shard and merged on the host
            D, I = ix.search(Qp, 10)
            Do, Io = local_oracle(Qp, shard.rows(), 10)
            gd, gi = sharding.gather_lists(Do, Io, grp)
            Dw, Iw = merge_canonical(gd.cpu().numpy(), gi.cpu().numpy(), ix.bases, 10)
            ok = torch.tensor([int(np.array_equal(D.cpu().numpy(), Dw) and np.array_equal(I.cpu().numpy(), Iw))],
                              dtype=torch.int64, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=grp)
            checked = bool(ok.item())
            n_shard = -(-N // G)                                          # the largest shard
            for k in ks:
                for B in batches:
                    Q = Qs[B]
                    call_ms = timed(lambda: ix.search(Q, k), args.iters, args.warmup, grp, dev)
                    D, I = ix.search(Q, k)
                    digest = hashlib.sha256(D.cpu().numpy().tobytes() + I.cpu().numpy().tobytes()).hexdigest()
                    local_ms = timed(lambda: shard.search(Q, k), args.iters, args.warmup, grp, dev)
                    st = shard.last_stats()
                    mine = torch.tensor([st["candidates"], st["fallback_queries"], st["chunks"]], dtype=torch.int64,
                                        device=dev)
                    every = torch.empty((G, 3), dtype=torch.int64, device=dev)
                    dist.all_gather_into_tensor(every.view(-1), mine, group=grp)
                    every = every.cpu().tolist()
                    if rank != 0:
                        continue
                    if G == Gs[0]:
                        base_ms[(k, B)] = (G, call_ms)
                    g0, ms0 = base_ms[(k, B)]
                    n_qb = (B + 255) // 256
                    cand_max = max(c for c, _, _ in every)
                    moved = n_qb * n_shard * (d * 2 + 8) + cand_max * d * 4
                    t_mem, t_tc = moved / (hbm * 1e9), 2 * B * n_shard * d / (tf * 1e12)
                    emit({
                        "metric": "dense_flat_l2_search_sharded", "n": N, "d": d, "gpus": G, "k": k, "batch": B,
                        "rows_per_shard": n_shard, "call_ms": round(call_ms, 4), "local_ms": round(local_ms, 4),
                        "gather_merge_ms": round(call_ms - local_ms, 4),
                        "queries_per_s": round(B / (call_ms * 1e-3), 1),
                        "speedup_vs_1gpu": round(ms0 / call_ms, 3) if g0 == 1 else None,
                        "frac_of_linear": round(ms0 / call_ms / G, 3) if g0 == 1 else None,
                        "moved_bytes_per_shard": moved, "bound": "hbm" if t_mem >= t_tc else "bf16 tensor",
                        "share_of_bound_per_gpu": round(max(t_mem, t_tc) / (call_ms * 1e-3), 4),
                        "share_of_bound_local_search": round(max(t_mem, t_tc) / (local_ms * 1e-3), 4),
                        "candidates_per_query_per_shard": [round(c / B, 1) for c, _, _ in every],
                        "fallback_query_chunks_per_shard": [f for _, f, _ in every],
                        "chunks_per_shard": [c for _, _, c in every],
                        "result_digest": digest, "parity_checked": checked, "parity_queries": 16,
                        "index_build_s": round(build_s, 1), "hbm_gbs_peak": hbm, "bf16_tflops_peak": tf,
                        "peak_source": peak_src, "gpu": cards[0][0],
                        "power_limit": sorted({c[1] for c in cards[:G]}),
                        "timing": f"CUDA events, {args.warmup} warm-up + {args.iters} calls, max over ranks",
                    })
            del ix, shard, D, I, Do, Io, gd, gi
            torch.cuda.empty_cache()
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
