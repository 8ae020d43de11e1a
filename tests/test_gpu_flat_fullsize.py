"""Exact dense search at the size bench_dense.py measures -- 21,015,324 x 768 rows -- against the batched reference
(tests/flat_fast_oracle.py, pinned bit for bit to the canonical restatements), ids and distance or score bits, on one
GPU and row-sharded over 2, 4 and 8 GPUs.  Needs a B200 (and, for the sharded tests, as many GPUs as the world).

One index is resident at a time: an L2 or IP index of the 21M rows holds 64.5 GB of rows and 32 GB of bf16 copy, so
the current one is freed before the next is built.

PR_SKIP_FULL=1 skips the file.  The reference lists are computed for a seeded sample of 1,024 of the 4,096 queries of
the batch (the first 256 and the last 64 among them); PR_FULL_ORACLE_ALL=1 computes them for all 4,096.
"""
import gc
import os
import socket
import time

import numpy as np
import pytest
import torch

import flat_fast_oracle as ffo
from probing_rag_b200 import IndexFlatIP, IndexFlatL2, ShardedIndexFlatIP, ShardedIndexFlatL2, sharding, synth

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(os.environ.get("PR_SKIP_FULL") == "1", reason="PR_SKIP_FULL=1")]

N_ROWS, D = synth.N_DOCS_WIKI, 768
NQ, N_SAMPLE, K_MAX = 4096, 1024, 128
CLS = {"l2": IndexFlatL2, "ip": IndexFlatIP}
SHARDED = {"l2": ShardedIndexFlatL2, "ip": ShardedIndexFlatIP}


def log(msg):
    print(f"[flat fullsize] {msg}", flush=True)


def sample_rows(nq, n, seed):
    if os.environ.get("PR_FULL_ORACLE_ALL") == "1" or n >= nq:
        return np.arange(nq)
    must = np.concatenate([np.arange(256), np.arange(nq - 64, nq)])
    rest = np.setdiff1d(np.arange(nq), must)
    extra = np.random.default_rng(seed).choice(rest, size=n - len(must), replace=False)
    return np.sort(np.concatenate([must, extra]))


def _bits(D_):
    return np.ascontiguousarray(D_.cpu().numpy() if isinstance(D_, torch.Tensor) else D_).view(np.uint32)


_resident = {}


def _free():
    _resident.clear()
    gc.collect()
    torch.cuda.empty_cache()


def resident(metric, kind="clustered"):
    """The index of `metric` over dense_rows(21M, 768, kind), its 4,096-query batch, and the reference lists (top-128)
    of the sampled rows of the batch.  Builds it after freeing whatever index was resident."""
    key = (metric, kind)
    if _resident.get("key") != key:
        _free()
        t0 = time.perf_counter()
        rows = synth.dense_rows(N_ROWS, D, kind=kind)
        index = CLS[metric](D)
        index.add(rows)
        del rows
        torch.cuda.empty_cache()
        Q = synth.dense_queries(index.rows(), NQ)
        torch.cuda.synchronize()
        log(f"{metric} {kind}: rows and index built in {time.perf_counter() - t0:.1f} s")
        sel = sample_rows(NQ, N_SAMPLE, 1) if kind == "clustered" else np.arange(256)
        t0 = time.perf_counter()
        st = {}
        ref = ffo.search_fast(Q[torch.from_numpy(sel).cuda()], index.rows(), K_MAX, metric, stats=st)
        log(f"{metric} {kind}: reference lists of {len(sel)} queries (top-{K_MAX}) in "
            f"{time.perf_counter() - t0:.1f} s; survivors per query mean {np.mean(st['survivors']):.1f}, "
            f"max {max(st['survivors'])}, chunks re-estimated {st['redone_pairs']}")
        _resident.update(key=key, index=index, Q=Q, sel=sel, ref=ref)
    return _resident


def check_rows(got, r, k, what, first=0):
    """got: lists [B, k] of the batch rows [first, first + B); compared where the sample reaches."""
    D_, I_ = (x.cpu().numpy() for x in got)
    sel = r["sel"]
    pick = (sel >= first) & (sel < first + D_.shape[0])
    assert pick.any(), what
    rows = sel[pick] - first
    assert np.array_equal(I_[rows], r["ref"][1][pick, :k]), f"{what}: ids differ"
    assert np.array_equal(_bits(D_[rows]), _bits(r["ref"][0][pick, :k])), f"{what}: distance / score bits differ"
    return int(pick.sum())


METRICS = ["l2", "ip"]


@pytest.fixture(scope="module", params=METRICS)
def metric(request):
    """Module-scoped, so that pytest runs every test of one metric before the other's (one build each)."""
    return request.param


def test_sampled_batch_at_every_k(metric):
    r = resident(metric)
    index = r["index"]
    index.set_tuning()
    for k in (1, 10, 100, 128):
        t0 = time.perf_counter()
        got = index.search(r["Q"], k)
        torch.cuda.synchronize()
        n = check_rows(got, r, k, f"{metric} B={NQ} k={k}")
        st = index.last_stats()
        log(f"{metric} B={NQ} k={k}: {n} queries compared; search {time.perf_counter() - t0:.2f} s; "
            f"candidates {st['candidates']:,}, fallbacks {st['fallback_queries']}, chunks {st['chunks']}")
        assert st["chunks"] == 8


def test_batch_slices_equal_the_full_batch(metric):
    """Batches of 1 to 512 queries (one query block of nq = 32 to 256, or two) cut from the front and the back of the
    batch: each query's list does not depend on the batch it came in."""
    r = resident(metric)
    index, Q = r["index"], r["Q"]
    index.set_tuning()
    for k in (10, 128):
        Dall, Iall = index.search(Q, k)
        for B in (1, 8, 64, 96, 128, 192, 224, 512):
            for a in (0, NQ - B):
                D_, I_ = index.search(Q[a:a + B], k)
                assert torch.equal(I_, Iall[a:a + B]), f"B={B} at {a} k={k}: ids differ"
                assert np.array_equal(_bits(D_), _bits(Dall[a:a + B])), f"B={B} at {a} k={k}: bits differ"
        check_rows((Dall, Iall), r, k, f"{metric} k={k}")


PLANS = [dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2), dict(cand_capacity=1)]


@pytest.mark.parametrize("plan", PLANS, ids=["one-chunk", "128-x2", "cap1-fallback"])
def test_launch_plans(metric, plan):
    """One chunk of 21M rows; 128 rows growing x2 (18 chunks); a capacity of one candidate, so that every chunk with
    two or more candidates of a query, the largest ones included, is evaluated in full by the exact fallback."""
    r = resident(metric)
    index = r["index"]
    index.set_tuning(**plan)
    try:
        for k in ((128,) if "cand_capacity" in plan else (10, 128)):
            t0 = time.perf_counter()
            got = index.search(r["Q"][:64], k)
            torch.cuda.synchronize()
            check_rows(got, r, k, f"{metric} {plan} k={k}")
            st = index.last_stats()
            log(f"{metric} {plan} B=64 k={k}: {time.perf_counter() - t0:.2f} s, chunks {st['chunks']}, "
                f"candidates {st['candidates']:,}, fallbacks {st['fallback_queries']}")
            if plan.get("first_chunk_rows") == 1 << 30:
                assert st["chunks"] == 1
            if plan.get("growth") == 2:
                assert st["chunks"] == 18
            if "cand_capacity" in plan:
                assert st["fallback_queries"] > 64            # more than the first chunk's 64
    finally:
        index.set_tuning()


def test_isotropic_rows(metric):
    """N(0, 1/d) rows, the filter's worst case (distances concentrate), at B = 256.  The candidate and fallback counts
    are printed, not asserted."""
    r = resident(metric, "isotropic")
    index = r["index"]
    index.set_tuning()
    for k in (10, 128):
        t0 = time.perf_counter()
        got = index.search(r["Q"][:256], k)
        torch.cuda.synchronize()
        check_rows(got, r, k, f"{metric} isotropic k={k}")
        st = index.last_stats()
        log(f"{metric} isotropic B=256 k={k}: {time.perf_counter() - t0:.2f} s; candidates {st['candidates']:,} "
            f"({st['candidates'] / 256:,.0f} per query), max per query and chunk {st['max_candidates']:,}, "
            f"fallbacks {st['fallback_queries']}")


# ----------------------------------------------------------------------------- row shards over NCCL
# (batch size, k) of the calls each rank makes, in order
CALLS = [(NQ, 10), (64, 128), (1, 1), (512, 100)]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        lo, hi = sharding.shard_range(N_ROWS, rank, world)
        Q = synth.dense_queries_of(N_ROWS, D, NQ, device=dev)
        res = {}
        for metric in METRICS:
            shard = CLS[metric](D, dev)
            rows = synth.dense_rows(N_ROWS, D, device=dev, row_lo=lo, row_hi=hi)
            shard.add(rows)
            del rows
            sx = SHARDED[metric](shard, lo)
            for B, k in CALLS:
                D_, I_ = sx.search(Q[:B], k)
                res[f"{metric}_{B}_{k}_D"], res[f"{metric}_{B}_{k}_I"] = D_.cpu().numpy(), I_.cpu().numpy()
            del sx, shard
            gc.collect()
            torch.cuda.empty_cache()
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def single_lists(tmp_path_factory):
    """The single-GPU lists of CALLS for both metrics, checked against the reference where the sample reaches; the
    device is freed afterwards, so that the ranks have it to themselves."""
    out = {}
    for metric in METRICS:
        r = resident(metric)
        r["index"].set_tuning()
        for B, k in CALLS:
            D_, I_ = r["index"].search(r["Q"][:B], k)
            check_rows((D_, I_), r, k, f"{metric} B={B} k={k}")
            out[f"{metric}_{B}_{k}_D"], out[f"{metric}_{B}_{k}_I"] = D_.cpu().numpy(), I_.cpu().numpy()
    _free()
    return out


@pytest.mark.timeout(3000)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_shards_over_nccl_equal_the_single_gpu_lists(world, tmp_path, request):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp
    single = request.getfixturevalue("single_lists")
    t0 = time.perf_counter()
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    log(f"world {world}: {time.perf_counter() - t0:.1f} s")
    for rank in range(world):
        got = np.load(tmp_path / f"r{rank}.npz")
        for name, want in single.items():
            if name.endswith("_I"):
                assert np.array_equal(got[name], want), f"rank {rank} {name}: ids differ"
            else:
                assert np.array_equal(got[name].view(np.uint32), want.view(np.uint32)), f"rank {rank} {name}: bits differ"
