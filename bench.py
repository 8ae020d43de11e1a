"""bench.py -- BM25 top-10 queries/sec over a 21M-passage corpus on N B200s (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch: all n_queries synthetic queries scored
against the whole (doc-sharded for N>1) synthetic corpus and reduced to top-k, including for
N>1 the NCCL all-gather of the per-shard lists and the merge.  Prints ONE JSON line.

  value          queries/s, inputs resident in HBM, CUDA events, max over ranks
  e2e            same through the host-buffer API (pinned H2D of the query batch, D2H of the lists)
  roofline       scoring kernel: algorithmic bytes (SURVEY 8d) / its summed device time; next to the contractual
                 HBM fraction, the kernel's real limiter and real DRAM fraction from the committed ncu capture
  result_digest  sha256 of the final [B,k] (doc ids, scores) of the timed configuration: identical at N = 1, 2, 4, 8
  sample_digest  sha256 of the lists of the first 32 queries -- printed by BOTH arms (the reference arm computes
                 them with the CPU oracle in the canonical order), so the driver can see the two arms agree
  parity_checked queries whose GPU lists were compared (bit-equal ids and scores) with the CPU oracle in this run
  cpu_baseline   the reference's CPU algorithm on a bounded sample: NumPy port on a thread pool (bm25s n_threads),
                 plus labelled variants (1 thread = what llama-index runs; threaded C restatement)
  secondary      BASELINE configs 4 and 5 on the same index (N = 1): prober-gated batch, batch x k x round sweep
  --impl reference   times only the CPU path (all host threads), never loads libprobingrag.so, same line shape
  --dump-outputs DIR the ranked lists of the last timed step as DIR/{scores,doc_ids,query_rows}.npy (see dump_outputs):
                     the inputs are seeded, so two builds run with the same arguments can be compared list for list
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

from probing_rag_b200 import synth  # noqa: E402

METRIC = "bm25_top10_queries_per_sec"
UNIT = "queries/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- workload
from probing_rag_b200.sharding import gather_lists, global_stats, shard_range  # noqa: E402


def build_arrays(n_docs: int, vocab: int, device, rank: int = 0, world: int = 1):
    """Synthetic Zipf-Mandelbrot corpus shard [lo, hi) as bm25s-style index arrays on `device`
    (indptr i64[V+1], doc ids i32[nnz], weights f32[nnz]) with GLOBAL N / avgdl / df (SURVEY 8d-8e).
    torch library ops only: the reference arm builds its arrays here without touching libprobingrag.so."""
    lo, hi = shard_range(n_docs, rank, world)
    cdf = torch.from_numpy(synth.zipf_mandelbrot_cdf(vocab)).to(device)
    toks, lens = [], []
    t0 = time.time()
    for blk in range(lo // synth.DOC_BLOCK, (max(hi, 1) - 1) // synth.DOC_BLOCK + 1):
        t, l = synth.corpus_block_torch(blk, n_docs, cdf)
        b_lo = blk * synth.DOC_BLOCK
        s, e = max(lo - b_lo, 0), min(hi - b_lo, l.numel())
        if e <= s:
            continue
        if s > 0 or e < l.numel():
            off = torch.zeros(l.numel() + 1, dtype=torch.int64, device=device)
            torch.cumsum(l.long(), 0, out=off[1:])
            t = t[int(off[s]):int(off[e])]
            l = l[s:e]
        toks.append(t)
        lens.append(l)
    tokens = torch.cat(toks) if toks else torch.zeros(0, dtype=torch.int32, device=device)
    doc_lens = torch.cat(lens) if lens else torch.zeros(0, dtype=torch.int32, device=device)
    del toks, lens
    n_tok_local = tokens.numel()
    # global statistics
    from probing_rag_b200.index import bm25_weights, count_postings, idf_lucene_table
    term, doc, tf, df_local = count_postings(tokens, doc_lens, vocab)
    del tokens
    df, avgdl = global_stats(df_local, n_tok_local, n_docs)
    df_host = df.cpu().numpy()
    idf = torch.from_numpy(idf_lucene_table(df_host, n_docs)).to(device)
    w = bm25_weights(term, doc, tf, doc_lens, idf, avgdl)
    del tf, term
    indptr = torch.zeros(vocab + 1, dtype=torch.int64, device=device)
    torch.cumsum(df_local, 0, out=indptr[1:])
    torch.cuda.synchronize(device)
    log(f"[bench] rank {rank}: shard docs [{lo},{hi}) nnz={doc.numel():,} avgdl={avgdl:.3f} arrays built in {time.time() - t0:.1f}s")
    return {"indptr": indptr, "doc_ids": doc, "weights": w, "n_docs": hi - lo, "doc_id_base": lo, "avgdl": avgdl,
            "df_host": df_host}


def build_workload(n_docs: int, vocab: int, n_queries: int, device, rank: int = 0, world: int = 1,
                   query_kind: str = "round0"):
    """The shard as a BM25Index on `device` + the seeded query batch (host CSR)."""
    from probing_rag_b200 import BM25Index
    a = build_arrays(n_docs, vocab, device, rank, world)
    gi = BM25Index(a["indptr"], a["doc_ids"], a["weights"], a["n_docs"], n_docs, a["doc_id_base"], meta={"avgdl": a["avgdl"]})
    torch.cuda.synchronize(device)
    q_indptr, q_terms = synth.queries_np(n_queries, vocab, a["df_host"], kind=query_kind)
    gi.df_host = a["df_host"]
    return gi, q_indptr, q_terms


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU baseline
N_SAMPLE_DIGEST = 32


def digest(ids: np.ndarray, scores: np.ndarray) -> str:
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(ids, dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(scores, dtype=np.float32).tobytes())
    return h.hexdigest()


DUMP_MAX_BYTES = 64_000_000
DUMP_SEED = 2024


def dump_outputs(out_dir: str, scores: np.ndarray, ids: np.ndarray) -> int:
    """Write the [B, k] lists a caller of the timed path receives as out_dir/scores.npy (float32), doc_ids.npy (float64:
    exact for every int32 id) and query_rows.npy (float64: the batch row of each dumped list).  A batch whose lists
    would exceed DUMP_MAX_BYTES keeps a seeded sample of rows, the same rows for the same batch size.  Returns the
    number of rows written."""
    nq, k = scores.shape
    row_bytes = 4 * k + 8 * k + 8
    max_rows = (DUMP_MAX_BYTES - 3 * 4096) // row_bytes            # headroom for the three .npy headers
    rows = np.arange(nq, dtype=np.int64)
    if nq > max_rows:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(nq, size=max_rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), np.ascontiguousarray(scores[rows], dtype=np.float32))
    np.save(os.path.join(out_dir, "doc_ids.npy"), np.ascontiguousarray(ids[rows], dtype=np.float64))
    np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    log(f"[bench] wrote the lists of {len(rows)} of {nq} queries (top-{k}) to {out_dir}")
    return len(rows)


def timed_cpu(fn, host_index, q_indptr, q_terms, k, budget_s, max_queries, n_threads, **kw):
    """queries/s of `fn(index, q_indptr[:n+1], q_terms, k, n_threads=..)` on as many of the first queries as fit
    `budget_s` (probed with a few queries first).  Returns (queries/s, n, last result)."""
    nq = len(q_indptr) - 1
    n_probe = max(1, min(max(n_threads, 2), nq, max_queries))
    t0 = time.perf_counter()
    fn(host_index, q_indptr[:n_probe + 1], q_terms, k, n_threads=n_threads, **kw)
    dt = time.perf_counter() - t0
    n = int(min(max_queries, nq, max(n_probe, budget_s / max(dt / n_probe, 1e-9))))
    t0 = time.perf_counter()
    res = fn(host_index, q_indptr[:n + 1], q_terms, k, n_threads=n_threads, **kw)
    dt = time.perf_counter() - t0
    return n / dt, n, res


def cpu_baselines(host_index: dict, q_indptr, q_terms, k: int, budget_s: float, cores: int, nq_total: int):
    """The reference's CPU algorithm (bm25s NumPy path, SURVEY App. A.5-A.6: dense f32 accumulator, np.add.at
    per query token, argpartition + argsort) as the oracle restates it, three ways:
      numpy_pool   thread pool over queries, n_threads = cores   (bm25s's own multi-thread mechanism)  <- headline
      numpy_1t     one thread                                     (bm25s default n_threads=0: what llama-index runs)
      c_threads    the plain-C restatement of the same loop, one thread per core (no GIL, no NumPy dispatch)
    Also returns the canonical oracle lists of the first N_SAMPLE_DIGEST queries (C oracle)."""
    from oracle import bm25_oracle as bo
    from oracle import c_oracle as co
    v_pool, n_pool, _ = timed_cpu(bo.retrieve_batch, host_index, q_indptr, q_terms, k, budget_s * 0.5, 512, cores, canonical=False)
    v_1t, n_1t, _ = timed_cpu(bo.retrieve_batch, host_index, q_indptr, q_terms, k, budget_s * 0.2, 64, 1, canonical=False)
    v_c, n_c, _ = timed_cpu(co.retrieve_batch, host_index, q_indptr, q_terms, k, budget_s * 0.3, 2048, cores)
    ns = min(N_SAMPLE_DIGEST, len(q_indptr) - 1)
    s_s, s_d = co.retrieve_batch(host_index, q_indptr[:ns + 1], q_terms, k, n_threads=cores)
    what = "of %d queries (first queries of the seeded batch, whole corpus)" % nq_total
    variants = [
        {"name": "numpy_pool", "value": v_pool, "unit": UNIT, "cores": cores, "sample": f"{n_pool} {what}",
         "what": f"NumPy oracle port, thread pool over queries like bm25s n_threads={cores}"},
        {"name": "numpy_1t", "value": v_1t, "unit": UNIT, "cores": 1, "sample": f"{n_1t} {what}",
         "what": "NumPy oracle port, one thread: bm25s default n_threads=0, what llama-index's BM25Retriever runs"},
        {"name": "c_threads", "value": v_c, "unit": UNIT, "cores": cores, "sample": f"{n_c} {what}",
         "what": "plain-C restatement of the same dense-accumulator loop, one thread per core"},
    ]
    base = {"value": v_pool, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_pool} {what}, NumPy oracle port, thread pool over queries like bm25s n_threads={cores}",
            "variants": variants}
    return base, (s_s, s_d)


def host_arrays(a: dict) -> dict:
    return {"data": a["weights"].cpu().numpy(), "indices": a["doc_ids"].cpu().numpy(),
            "indptr": a["indptr"].cpu().numpy(), "num_docs": a["n_docs"], "doc_id_base": a["doc_id_base"]}


def make_config(args, world: int, nnz_total: int) -> dict:
    """The workload description -- the same dict in both arms."""
    workload = (f"BM25 top-{args.k} over {args.n_docs:,}-passage DPR-Wikipedia-shaped synthetic corpus, "
                f"{args.n_queries:,} queries" + (f", doc-sharded over {world} GPUs" if world > 1 else ", 1xB200"))
    return {"workload": workload, "k": args.k, "n_docs": args.n_docs, "n_queries": args.n_queries, "vocab": args.vocab,
            "nnz": int(nnz_total), "l2": "inputs (postings of %.1f GB) larger than L2" % (nnz_total * 8 / 1e9),
            "parallelism": f"doc-shard x{world}" if world > 1 else "single"}


# ----------------------------------------------------------------------------- secondary: BASELINE configs 4 and 5
def dev_time(fn, reps: int, warm: int = 2) -> float:
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def secondary_block(gi, qi, qt, device, vocab: int, peaks: dict) -> dict:
    """BASELINE configs 4 (prober-gated batch of 16,384 questions) and 5 (batch x depth x round sweep, the
    reference's own regime: small batches, later rounds search with the decoded transcript, exp_rag.py:428)
    on the index the headline ran on.  Device-timed, inputs resident; a compact table -- the full sweep is
    committed under profiles/."""
    from probing_rag_b200.prober import ProberGate, gate_and_retrieve
    from probing_rag_b200.retriever import BM25Retriever
    out = {}
    # ---- config 4
    rows = 16384
    sds = [synth.make_prober_state(l) for l in synth.PROBE_LAYERS]
    gate = ProberGate(sds, device=device)
    x = synth.make_hidden_states(rows, seed=4).to(device)
    d_qi = torch.from_numpy(qi[:rows + 1]).to(device)
    d_qt = torch.from_numpy(qt[:qi[rows]]).to(device)
    retr = BM25Retriever(None, 10, index=gi)
    ms_gate = dev_time(lambda: gate(x, sync=False), 10)
    res = gate_and_retrieve(gate, retr, x, d_qi, d_qt, k=10)
    n_ret = int(res[0].retrieve.sum().item())
    ms_all = dev_time(lambda: gate_and_retrieve(gate, retr, x, d_qi, d_qt, k=10), 3, 1)
    flops = gate.flops(rows)
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    out["config4_prober_gated_batch"] = {
        "rows": rows, "retrieve_rows": n_ret, "prober_ms": ms_gate, "prober_rows_per_s": rows / ms_gate * 1e3,
        "prober_tflops_algorithmic": flops / ms_gate / 1e9, "prober_frac_of_bf16_peak": flops / ms_gate / 1e9 / peak_tf,
        "prober_peak_tflops": peak_tf, "prober_dtype": "bf16x3 operands, f32 accumulate (tcgen05)",
        "gate_plus_bm25_top10_ms": ms_all, "questions_per_s": rows / ms_all * 1e3}
    # ---- config 5
    sweep = []
    # one query per call (the reference's call shape): the mean over 64 different queries, one call each
    singles = [(torch.from_numpy(qi[c:c + 2] - qi[c]).to(device), d_qt[int(qi[c]):int(qi[c + 1])]) for c in range(64)]

    def single_pass(k):
        for sq, st in singles:
            gi.topk(sq, st, k, check_status=False)
    for b in (1, 8, 64, 512, 4096):
        for k in (1, 10, 100):
            if b == 1:
                ms = dev_time(lambda: single_pass(k), 5, 1) / len(singles)
                alg = gi.algorithmic_bytes(qi[:len(singles) + 1], qt[:qi[len(singles)]], k) / len(singles)
            else:
                bq, bt = d_qi[:b + 1], d_qt[:int(qi[b])]
                ms = dev_time(lambda: gi.topk(bq, bt, k, check_status=False), 20 if b <= 512 else 3)
                alg = gi.algorithmic_bytes(qi[:b + 1], qt[:qi[b]], k)
            sweep.append({"round": 0, "batch": b, "k": k, "ms": ms, "qps": b / ms * 1e3, "alg_gbs": alg / ms / 1e6})
    lqi, lqt = synth.queries_np(64, vocab, gi.df_host, kind="later")       # rounds 1-3: transcript-sized queries
    d_lqi, d_lqt = torch.from_numpy(lqi).to(device), torch.from_numpy(lqt).to(device)
    for b in (1, 8, 64):
        bq, bt = d_lqi[:b + 1], d_lqt[:int(lqi[b])]
        ms = dev_time(lambda: gi.topk(bq, bt, 10, check_status=False), 5, 1)
        sweep.append({"round": "1-3 (transcript, %.0f terms/query)" % (lqi[b] / b), "batch": b, "k": 10, "ms": ms, "qps": b / ms * 1e3,
                      "alg_gbs": gi.algorithmic_bytes(lqi[:b + 1], lqt[:lqi[b]], 10) / ms / 1e6})
    out["config5_sweep"] = sweep
    return out


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-docs", type=int, default=synth.N_DOCS_WIKI)
    ap.add_argument("--vocab", type=int, default=1 << 22)
    ap.add_argument("--n-queries", type=int, default=65536)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--cpu-budget-s", type=float, default=25.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "allreduce", "none"],
                    help="N > 1: how the shards share score bounds (p2p = live over NVLink peer memory)")
    ap.add_argument("--list-rounds", type=int, default=4,
                    help="N > 1, p2p: launches of a call behind which the shards' running lists are all-gathered (union bound)")
    ap.add_argument("--tune", default="", help="comma list key=value for pr_bm25_tuning_t")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ranked lists of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return                                        # rank 0 alone runs the CPU arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    cores = os.cpu_count() or 1
    nq, k = args.n_queries, args.k

    if args.impl == "reference":
        # the whole corpus as host arrays (built with torch library ops on the GPU, then dropped from it); the
        # product library is never loaded in this process
        a = build_arrays(args.n_docs, args.vocab, device)
        host = host_arrays(a)
        nnz = int(a["doc_ids"].numel())
        qi, qt = synth.queries_np(nq, args.vocab, a["df_host"])
        del a
        torch.cuda.empty_cache()
        from oracle import bm25_oracle as bo
        from oracle import c_oracle as co
        per_step_budget = max(5.0, min(40.0, 120.0 / max(args.steps + args.warmup, 1)))
        vals, n, last = [], 0, None
        for i in range(args.warmup + args.steps):
            v, n, last = timed_cpu(bo.retrieve_batch, host, qi, qt, k, per_step_budget, 512, cores, canonical=False)
            if i >= args.warmup:
                vals.append(v)
        v = float(np.mean(vals))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *last)                 # the first n queries of the batch
        base, (s_s, s_d) = cpu_baselines(host, qi, qt, k, 20.0, cores, nq)
        base = dict(base, value=v, sample=f"{n} of {nq} queries per step (first queries of the seeded batch, whole corpus), "
                                           f"NumPy oracle port, thread pool over queries like bm25s n_threads={cores}")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * n / v,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, args.gpus, nnz),
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "sample_digest": digest(s_d, s_s), "sample_queries": int(s_d.shape[0]),
            "native_library_loaded": "libprobingrag" in open("/proc/self/maps").read(),
            "gpu_launches": 0}))
        return

    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from probing_rag_b200.sharding import ShardedBM25
    gi, qi, qt = build_workload(args.n_docs, args.vocab, nq, device, rank, world)
    if args.tune:
        gi.set_tuning(**{kv.split("=")[0]: int(kv.split("=")[1]) for kv in args.tune.split(",")})
    sharded, exchange_used = None, None
    if world > 1:
        exchange_used = None if args.exchange == "none" else args.exchange
        if exchange_used == "p2p":
            # peer memory needs CUDA IPC between the ranks' GPUs; if this box cannot provide it, say so and use the
            # all-reduce form of the same exchange (every rank takes the same branch: the failure is collective)
            ok = torch.ones(1, device=device)
            try:
                sharded = ShardedBM25(gi, exchange="p2p", max_queries=nq, list_rounds=args.list_rounds)
            except Exception as ex:
                log(f"[bench] rank {rank}: peer-memory thresholds unavailable ({ex!r})")
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() == 0:
                if sharded is not None:
                    sharded.close()
                sharded, exchange_used = None, "allreduce"
        if sharded is None:
            sharded = ShardedBM25(gi, exchange=exchange_used)
    d_qi = torch.from_numpy(qi).to(device)
    d_qt = torch.from_numpy(qt).to(device)
    out = (torch.empty((nq, k), dtype=torch.float32, device=device),
           torch.empty((nq, k), dtype=torch.int32, device=device))

    def step_device():
        if world > 1:
            return sharded.topk(d_qi, d_qt, k, check_status=False)
        return gi.topk(d_qi, d_qt, k, out=out, check_status=False)

    def step_host():
        return (sharded if world > 1 else gi).topk_host(qi, qt, k)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = None
        for _ in range(steps):
            r = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), r

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, res = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    n_score_launches = gi.num_launches(nq, k)
    # kernels of ours per step: init + (score + merge) per launch; N > 1: + the merge of the gathered lists
    launches_per_step = gi.last_launches + (1 if world > 1 else 0)
    res_s, res_d = res[0].cpu().numpy(), res[1].cpu().numpy()

    # scoring-kernel device time for the roofline (events around its launches)
    gi.set_profiling(True)
    barrier()
    step_device()
    torch.cuda.synchronize(device)
    score_ms, score_launches = gi.profile()
    gi.set_profiling(False)
    alg_bytes = gi.algorithmic_bytes(qi, qt, k)

    # end to end through the host-buffer API
    for _ in range(2):
        step_host()
    ms_e2e, last = timed(step_host, args.steps)
    e2e_s, e2e_d, h2d, d2h = last
    assert np.array_equal(e2e_d, res_d) and np.array_equal(e2e_s, res_s), "host-buffer path returned different lists"

    # size-independent properties of the measured output: ranked, canonical tie order, ids in range
    assert bool((res_s[:, :-1] >= res_s[:, 1:]).all()), "ranked lists not score-descending"
    tie = res_s[:, :-1] == res_s[:, 1:]
    assert bool((res_d[:, :-1][tie] < res_d[:, 1:][tie]).all()), "ties not in ascending doc id order"
    assert int(res_d.min()) >= 0 and int(res_d.max()) < args.n_docs

    t = torch.tensor([float(alg_bytes), float(gi.nnz)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t)                       # total algorithmic bytes / postings over the shards
    alg_total, nnz_total = float(t[0].item()), int(t[1].item())

    if world > 1:
        sharded.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res_s, res_d)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    kernel = "bm25_lean_kernel"
    # what the committed `ncu --set full` capture of that kernel says (profiles/): DRAM bytes, real limiter
    cap = {}
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if cap.get("kernel") != kernel:
            cap = {}
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    achieved = alg_bytes / (score_ms * 1e-3) / 1e9 if score_ms > 0 else 0.0
    value = nq * args.steps / (ms_dev * 1e-3)
    e2e = nq * args.steps / (ms_e2e * 1e-3)
    traffic = int(cap["dram_bytes_per_launch"]) if "dram_bytes_per_launch" in cap else None
    dram_frac = None
    if traffic and cap.get("captured_launch_ms"):
        dram_frac = traffic / (cap["captured_launch_ms"] * 1e-3) / 1e9 / peak

    cpu_base, parity = None, {"parity_checked": 0}
    sample_dig = None
    if world == 1 and not args.no_cpu_baseline:
        host = {"data": gi.weights.cpu().numpy(), "indices": gi.doc_ids.cpu().numpy(), "indptr": gi.indptr.cpu().numpy(),
                "num_docs": gi.n_docs, "doc_id_base": gi.doc_id_base}
        cpu_base, (o_s, o_d) = cpu_baselines(host, qi, qt, k, args.cpu_budget_s, cores, nq)
        ns = o_d.shape[0]
        ok = bool(np.array_equal(o_d, res_d[:ns]) and np.array_equal(o_s, res_s[:ns]))
        parity = {"parity_checked": int(ns), "parity_ok": ok,
                  "parity_what": "GPU lists of the first queries == CPU oracle (C restatement, canonical order): ids and f32 scores bit-equal"}
        assert ok, "GPU lists differ from the CPU oracle on the checked sample"
        del host
    ns = min(N_SAMPLE_DIGEST, nq)
    sample_dig = digest(res_d[:ns], res_s[:ns])

    secondary = None
    if world == 1 and not args.no_secondary:
        try:
            secondary = secondary_block(gi, qi, qt, device, args.vocab, peaks)
        except Exception as ex:                               # the headline line must not die on the side table
            secondary = {"error": repr(ex)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args, world, nnz_total),
        "plan": {"tuning": gi.get_tuning(), "scoring_launches_per_step": n_score_launches, "nnz_shard0": gi.nnz,
                 "threshold_exchange": exchange_used,
                 "union_bound_rounds": sharded.list_rounds if sharded is not None else 0},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches_per_step * args.steps),
        "result_digest": digest(res_d, res_s), "sample_digest": sample_dig, "sample_queries": int(ns),
        **parity,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "frac_of_8000_nominal": achieved / 8000.0, "traffic": traffic,
                     "traffic_unit": "DRAM bytes (read + write) per launch, ncu", "traffic_source": cap.get("source"),
                     "bound_note": "contractual accounting (algorithmic posting bytes / kernel time vs copy bandwidth); a 64k-query "
                                   "batch re-reads each launch's posting slice from L2, so the chip-level limiter is not DRAM",
                     "limiter": cap.get("limiter"), "dram_frac": dram_frac,
                     "peak_source": peak_src, "kernel": kernel,
                     "algorithmic_bytes_per_launch": int(alg_bytes / max(score_launches, 1)),
                     "algorithmic_bytes_per_step_rank0": int(alg_bytes),
                     "algorithmic_bytes_per_step_all_ranks": int(alg_total),
                     "kernel_ms_per_step": score_ms, "kernel_launches_per_step": score_launches,
                     "kernel_share_of_step": score_ms / (ms_dev / args.steps)},
        "cpu_baseline": cpu_base,
        "secondary": secondary,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
