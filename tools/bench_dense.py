"""Exact dense search (IndexFlatL2 / IndexFlatIP drop-ins) over the wiki-sized embedding matrix: one JSON line per
(k, batch).

    python tools/bench_dense.py [--metric l2|ip] [--n 21015324] [--d 768] [--ks 5,10] [--batches 1,8,64,512] [--out FILE]

Rows are synthetic clustered embeddings generated on the device (synth.dense_rows), queries perturbed copies of
random rows.  Each setting: warm-up calls, then CUDA events around --iters calls ending in a synchronise.  Bytes and
flops are computed from shapes:
  alg_bytes      N d 4      what an exact fp32 scan (faiss IndexFlatL2) reads per call
  moved_bytes    what this design reads: the bf16 copy (N d 2) and the row norms (N 8; ip: N 4) once per query block of
                 <= 256 queries, plus the candidates' fp32 rows (4 d per candidate)
  flops          2 B N d
The share of peak is the larger of the two bounds (HBM bytes, bf16 dense tensor rate) over the measured time, naming
which applies; since the bf16 copy is half the fp32 bytes, the share against alg_bytes can exceed 1.0.
parity_checked: 16 queries at full size against the oracle's evaluation order (oracle.flat_oracle, its torch form:
the same IEEE float64 operations, run on the device over row chunks so the 64 GB matrix is never copied).
A CPU baseline (the faiss BLAS restatement on a 1M-row slice, numpy on this host) is reported at its own size.
--metric ip measures IndexFlatIP on the same rows (metric names dense_flat_ip_*); l2, the default, is unchanged.

Range mode, --radius-ranks 10,100 (and/or --radius-values): range_search instead of search, one JSON line per (radius,
batch).  The radius of rank R is the median over the batch of the exact R-th nearest distance (ip: R-th largest
score), from the index's own search; --radius-values gives radii directly.  Each line has the time per call (CUDA
events after warm-up; a call includes its host synchronise), hits and candidates per query, overflow fallbacks, how
many of the timed calls needed the second pass, and parity_checked: 4 queries of the batch against the fast reference
(tests/flat_range_fast_oracle.py, bit for bit) when the rows are finite.

--storage fp16: IndexScalarQuantizer(QT_fp16) beside the IndexFlat of --metric over the same rows (the IndexFlat
holds the generated rows without a copy, so both fit at once).  Three rounds alternate the two over every (k, batch),
one JSON line per index, round, k and batch: time per call, candidates per query, fallbacks, the index's bytes on the
device and parity_checked (16 queries of the fp16 index bit for bit against the oracle's evaluation order over the
fp16-decoded rows, decoded chunk by chunk; the IndexFlat as in the default mode).  --storage f32, the default, keeps the
output above.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import flat_oracle as fo  # noqa: E402
from oracle import flat_ip_oracle as fio  # noqa: E402
from probing_rag_b200 import IndexFlatIP, IndexFlatL2, IndexScalarQuantizer, ScalarQuantizer, synth  # noqa: E402

DATASHEET_HBM_GBS = 7700.0
DATASHEET_BF16_TFLOPS = 2250.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.strip().split(",")[:2]]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def peaks():
    p = {}
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(p.get("hbm_gbs", DATASHEET_HBM_GBS))
    tf = float(p.get("bf16_tflops", DATASHEET_BF16_TFLOPS))
    src = {"hbm_gbs": "MEASURED_PEAKS.json" if "hbm_gbs" in p else "data sheet",
           "bf16_tflops": "MEASURED_PEAKS.json" if "bf16_tflops" in p else "data sheet (dense bf16)"}
    return hbm, tf, src


def parity(index, Q, k, chunk=1 << 21, ip=False):
    """Bit-exact check of (D, I) against the oracle's evaluation order, the rows streamed in chunks (ip: the inner
    products, ranked by their key, compared as keys so that a NaN equals itself).  An IndexScalarQuantizer is checked
    against its decoded rows, decoded one chunk at a time."""
    D, I = index.search(Q, k)
    X = index.codes() if isinstance(index, IndexScalarQuantizer) else index.rows()
    ok = True
    for b in range(Q.shape[0]):
        best_d = torch.empty(0, dtype=torch.int64 if ip else torch.float32, device=X.device)
        best_i = torch.empty(0, dtype=torch.int64, device=X.device)
        for a in range(0, X.shape[0], chunk):
            Xc = X[a:a + chunk].float()
            if ip:
                dist = fio.ip_key_torch(fio.exact_inner_products_torch(Q[b], Xc))
            else:
                dist = fo.exact_distances_torch(Q[b], Xc)
            cd = torch.cat([best_d, dist])
            ci = torch.cat([best_i, torch.arange(a, a + dist.numel(), device=X.device)])
            s, o = torch.sort(cd, stable=True)      # ci ascending within equal distances: canonical order
            best_d, best_i = s[:k], ci[o[:k]]
        got = fio.ip_key_torch(D[b]) if ip else D[b]
        ok &= bool(torch.equal(best_d, got) and torch.equal(best_i, I[b]))
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--metric", default="l2", choices=("l2", "ip"))
    ap.add_argument("--n", type=int, default=synth.N_DOCS_WIKI)
    ap.add_argument("--d", type=int, default=768)
    ap.add_argument("--ks", default="5,10")
    ap.add_argument("--batches", default="1,8,64,512")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kind", default="clustered", choices=("clustered", "isotropic"))
    ap.add_argument("--cpu-rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--radius-ranks", default="")
    ap.add_argument("--radius-values", default="")
    ap.add_argument("--storage", default="f32", choices=("f32", "fp16"))
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_dense.py measures on a CUDA device"
    torch.cuda.set_device(0)
    name, power = card()
    hbm, tf, peak_src = peaks()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    if args.storage == "fp16":
        return bench_fp16(args, emit, name, power)
    t0 = time.perf_counter()
    ip = args.metric == "ip"
    index = (IndexFlatIP if ip else IndexFlatL2)(args.d)
    index.add(synth.dense_rows(args.n, args.d, kind=args.kind))
    index.search(synth.dense_queries(index.rows(), 1), 1)       # builds the bf16 copy and the norms
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    if args.radius_ranks or args.radius_values:
        return bench_range(args, index, emit, name, power, build_s)
    checked = parity(index, synth.dense_queries(index.rows(), 16, seed=99), 10, ip=ip)
    N, d = args.n, args.d
    for k in [int(s) for s in args.ks.split(",")]:
        for B in [int(s) for s in args.batches.split(",")]:
            Q = synth.dense_queries(index.rows(), B)
            for _ in range(args.warmup):
                index.search(Q, k)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                index.search(Q, k)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.iters
            st = index.last_stats()
            n_qb = (B + 255) // 256
            alg_bytes = N * d * 4
            moved = n_qb * N * (d * 2 + (4 if ip else 8)) + st["candidates"] * d * 4
            flops = 2 * B * N * d
            t_mem, t_tc = moved / (hbm * 1e9), flops / (tf * 1e12)
            bound = "hbm" if t_mem >= t_tc else "bf16 tensor"
            emit({
                "metric": f"dense_flat_{args.metric}_search", "n": N, "d": d, "k": k, "batch": B, "data": args.kind,
                "ms_per_call": round(ms, 4), "queries_per_s": round(B / (ms * 1e-3), 1),
                "alg_bytes": alg_bytes, "frac_vs_fp32_scan_bytes": round(alg_bytes / (ms * 1e-3) / (hbm * 1e9), 4),
                "frac_note": "exact fp32 scan bytes (N d 4) over the time at HBM peak; the scan reads a bf16 copy, "
                             "so the fraction can exceed 1.0",
                "moved_bytes": moved, "flops": flops, "tflops": round(flops / (ms * 1e-3) / 1e12, 2),
                "share_of_bound": round(max(t_mem, t_tc) / (ms * 1e-3), 4), "bound": bound,
                "hbm_gbs_peak": hbm, "bf16_tflops_peak": tf, "peak_source": peak_src,
                "candidates_mean_per_query": round(st["candidates"] / B, 1),
                "candidates_max_query_chunk": st["max_candidates"], "fallback_query_chunks": st["fallback_queries"],
                "chunks": st["chunks"], "launches": st["launches"],
                "parity_checked": checked, "parity_queries": 16, "index_build_s": round(build_s, 1),
                "gpu": name, "power_limit": power, "timing": f"CUDA events, {args.warmup} warm-up + {args.iters} calls",
            })
    # CPU baseline: the faiss BLAS restatement on a slice, not extrapolated
    Xc = index.rows()[:args.cpu_rows].cpu().numpy()
    for B in (1, 8, 64):
        Qc = synth.dense_queries(index.rows(), B).cpu().numpy()
        cpu_search = fio.faiss_blas_search_ip if ip else fo.faiss_blas_search
        cpu_search(Qc, Xc, 10)
        t = time.perf_counter()
        cpu_search(Qc, Xc, 10)
        s = time.perf_counter() - t
        emit({"metric": f"dense_flat_{args.metric}_cpu_baseline", "impl": "numpy restatement of faiss BLAS flat search",
              "n": Xc.shape[0], "d": d, "k": 10, "batch": B, "ms_per_call": round(s * 1e3, 2),
              "host_threads": torch.get_num_threads(), "note": "slice of the index; not extrapolated to the full size"})


def time_search(index, Q, k, warmup, iters):
    for _ in range(warmup):
        index.search(Q, k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        index.search(Q, k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def bench_fp16(args, emit, name, power):
    ip = args.metric == "ip"
    t0 = time.perf_counter()
    rows = synth.dense_rows(args.n, args.d, kind=args.kind)
    sq = IndexScalarQuantizer(args.d, ScalarQuantizer.QT_fp16, 0 if ip else 1)
    sq.add(rows)
    flat = (IndexFlatIP if ip else IndexFlatL2)(args.d)
    flat._set_rows(rows)                                        # the generated rows themselves, no second copy
    del rows
    Q1 = synth.dense_queries(flat.rows(), 1)
    for index in (flat, sq):
        index.search(Q1, 1)                                     # builds the aux (bf16 copy and norms / norms only)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    Qp = synth.dense_queries(flat.rows(), 16, seed=99)
    checked = {"f32": parity(flat, Qp, 10, ip=ip), "fp16": parity(sq, Qp, 10, ip=ip)}
    dev_bytes = {"f32": flat.rows().numel() * 4 + flat._aux.numel(), "fp16": sq.codes().numel() * 2 + sq._aux.numel()}
    for rnd in range(args.rounds):
        for k in [int(s) for s in args.ks.split(",")]:
            for B in [int(s) for s in args.batches.split(",")]:
                Q = synth.dense_queries(flat.rows(), B)
                for storage, index in (("f32", flat), ("fp16", sq)):
                    ms = time_search(index, Q, k, args.warmup, args.iters)
                    st = index.last_stats()
                    emit({
                        "metric": f"dense_{'sq_fp16' if storage == 'fp16' else 'flat'}_{args.metric}_search",
                        "storage": storage, "round": rnd, "n": args.n, "d": args.d, "k": k, "batch": B,
                        "data": args.kind, "ms_per_call": round(ms, 4), "queries_per_s": round(B / (ms * 1e-3), 1),
                        "candidates_mean_per_query": round(st["candidates"] / B, 1),
                        "candidates_max_query_chunk": st["max_candidates"],
                        "fallback_query_chunks": st["fallback_queries"], "chunks": st["chunks"],
                        "index_device_bytes": dev_bytes[storage], "parity_checked": checked[storage],
                        "parity_queries": 16, "parity_reference": "oracle evaluation order over the "
                        + ("fp16-decoded rows" if storage == "fp16" else "f32 rows"),
                        "index_build_s": round(build_s, 1), "gpu": name, "power_limit": power,
                        "timing": f"CUDA events, {args.warmup} warm-up + {args.iters} calls; f32 and fp16 alternate "
                                  f"per (k, batch) in each of {args.rounds} rounds",
                    })


def bench_range(args, index, emit, name, power, build_s):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from flat_range_fast_oracle import range_search_fast
    ip = args.metric == "ip"
    for B in [int(s) for s in args.batches.split(",")]:
        Q = synth.dense_queries(index.rows(), B)
        radii = []
        for R in [int(s) for s in args.radius_ranks.split(",") if s]:
            Dk, _ = index.search(Q, R)
            radii.append((f"rank {R}", float(torch.median(Dk[:, R - 1]))))
        radii += [("value", float(s)) for s in args.radius_values.split(",") if s]
        for how, r in radii:
            index._range_cap = 1024                          # every setting starts from the default staging size
            passes = []
            for _ in range(args.warmup):
                index.range_search(Q, r)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                cap = index._range_cap
                lims, D, I = index.range_search(Q, r)
                passes.append(int((lims[1:] - lims[:-1]).max()) > min(cap, index.ntotal) if B else False)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.iters
            st = index.last_stats()
            hits = (lims[1:] - lims[:-1]).double()
            sel = torch.arange(min(4, B), device=Q.device)
            checked = None                                   # not checked: the reference would copy every hit row
            if int(lims[len(sel)]) <= 1 << 20:
                want = range_search_fast(Q[sel], index.rows(), r, args.metric)
                got = (lims[:len(sel) + 1].cpu().numpy(), D[:int(lims[len(sel)])].cpu().numpy(),
                       I[:int(lims[len(sel)])].cpu().numpy())
                checked = bool(np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2]) and
                               np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)))
            emit({
                "metric": f"dense_flat_{args.metric}_range_search", "n": args.n, "d": args.d, "batch": B,
                "data": args.kind, "radius": r, "radius_from": how + (" (median over the batch)" if how != "value" else ""),
                "ms_per_call": round(ms, 4), "queries_per_s": round(B / (ms * 1e-3), 1),
                "hits_mean_per_query": round(float(hits.mean()), 1), "hits_max_per_query": int(hits.max()),
                "candidates_mean_per_query": round(st["candidates"] / B, 1),
                "candidates_max_query_chunk": st["max_candidates"], "fallback_query_chunks": st["fallback_queries"],
                "chunks": st["chunks"], "launches": st["launches"],
                "calls_with_second_pass": sum(passes), "timed_calls": args.iters,
                "parity_checked": checked, "parity_queries": len(sel), "index_build_s": round(build_s, 1),
                "gpu": name, "power_limit": power,
                "timing": f"CUDA events, {args.warmup} warm-up + {args.iters} calls, each ending in a host synchronise",
            })


if __name__ == "__main__":
    main()
