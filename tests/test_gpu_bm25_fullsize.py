"""BM25 top-k at the size bench.py measures -- 21,015,324 documents, 65,536 queries -- against the torch restatement of
the oracle (tests/bm25_torch_oracle.py), ids and score bits, on one GPU and doc-sharded over 2, 4 and 8 GPUs.  Needs a
B200 (and, for the sharded tests, as many GPUs as the world).

PR_SKIP_FULL=1 skips the file.  The reference lists are computed for a seeded sample of 4,096 queries of the batch
(the first 512 and the last 64 among them); PR_FULL_ORACLE_ALL=1 computes them for all 65,536.
"""
import hashlib
import os
import socket
import time

import numpy as np
import pytest
import torch

import bm25_torch_oracle as tor
from oracle import c_oracle as co
from probing_rag_b200 import synth

from test_gpu_bm25 import assert_parity, to_dev, tune

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(os.environ.get("PR_SKIP_FULL") == "1", reason="PR_SKIP_FULL=1")]

N_DOCS, VOCAB, NQ = synth.N_DOCS_WIKI, 1 << 22, 65536
K_MAX = 128
N_SAMPLE = 4096


def log(msg):
    print(f"[fullsize] {msg}", flush=True)


def sample_rows(nq, n, seed):
    if os.environ.get("PR_FULL_ORACLE_ALL") == "1" or n >= nq:
        return np.arange(nq)
    must = np.concatenate([np.arange(min(512, nq)), np.arange(nq - 64, nq)])
    rest = np.setdiff1d(np.arange(nq), must)
    extra = np.random.default_rng(seed).choice(rest, size=n - len(must), replace=False)
    return np.sort(np.concatenate([must, extra]))


def reference(gi, qi, qt, rows, k=K_MAX):
    """Canonical top-k lists of `rows` of the batch (k = 128: every shallower list is a prefix of it)."""
    t0 = time.perf_counter()
    s, d = tor.retrieve_batch(gi.indptr, gi.doc_ids, gi.weights, gi.n_docs, qi, qt, k, gi.doc_id_base, rows=rows)
    torch.cuda.synchronize()
    log(f"reference lists of {len(rows)} queries (top-{k}) in {time.perf_counter() - t0:.1f} s")
    return s, d


def check_rows(got, ref, rows, k, what):
    """got: GPU lists [B, k] of the batch's first B queries; ref: reference [len(rows), 128] of `rows`."""
    gs, gd = (x.cpu().numpy() if torch.is_tensor(x) else x for x in got)
    sel = rows < gs.shape[0]
    assert sel.any(), what
    assert_parity(gs[rows[sel]], gd[rows[sel]], ref[0][sel, :k], ref[1][sel, :k])
    return int(sel.sum())


@pytest.fixture(scope="module")
def full():
    import bench
    t0 = time.perf_counter()
    gi, qi, qt = bench.build_workload(N_DOCS, VOCAB, NQ, torch.device("cuda"))
    log(f"workload built in {time.perf_counter() - t0:.1f} s, nnz {gi.nnz:,}")
    rows = sample_rows(NQ, N_SAMPLE, 1)
    return {"gi": gi, "qi": qi, "qt": qt, "rows": rows, "ref": reference(gi, qi, qt, rows)}


def test_reference_restatement_equals_the_c_oracle_at_full_size(full):
    gi, qi, qt = full["gi"], full["qi"], full["qt"]
    host = {"data": gi.weights.cpu().numpy(), "indices": gi.doc_ids.cpu().numpy(), "indptr": gi.indptr.cpu().numpy(),
            "num_docs": gi.n_docs}
    want_s, want_d = co.retrieve_batch(host, qi[:25], qt, K_MAX, n_threads=min(24, os.cpu_count() or 1))
    assert np.array_equal(full["rows"][:24], np.arange(24))
    assert_parity(full["ref"][0][:24], full["ref"][1][:24], want_s, want_d)


def test_full_batch_top10_default_plan(full):
    """What bench.py times: 65,536 queries, top-10, the default tuning."""
    gi = full["gi"]
    tune(gi)
    d_qi, d_qt = to_dev(gi, full["qi"], full["qt"])
    n = check_rows(gi.topk(d_qi, d_qt, 10), full["ref"], full["rows"], 10, "k=10")
    log(f"top-10, default plan: {n} of {NQ} queries compared")


@pytest.mark.parametrize("plan", [dict(), dict(subs_per_item=12, warps_per_cta=8, docs_per_launch=98304, min_items=2048),
                                  dict(batch_variant=2, tile_epochs=2)], ids=["default", "subs12", "bv2-te2"])
@pytest.mark.parametrize("k", [100, 128])
def test_full_batch_deep_lists(full, k, plan):
    gi = full["gi"]
    tune(gi, **plan)
    d_qi, d_qt = to_dev(gi, full["qi"], full["qt"])
    n = check_rows(gi.topk(d_qi, d_qt, k), full["ref"], full["rows"], k, f"k={k}")
    log(f"top-{k}, {plan or 'default'}: {n} queries compared")
    tune(gi)


@pytest.mark.parametrize("k", [1, 10, 100])
def test_config5_batches(full, k):
    """Small-batch calls: one launch, the REFRESH variant, the wide merge over thousands of lists per query."""
    gi, qi, qt = full["gi"], full["qi"], full["qt"]
    tune(gi)
    d_qi, d_qt = to_dev(gi, qi, qt)
    for b in (8, 64, 512, 4096):
        got = gi.topk(d_qi[:b + 1], d_qt[:int(qi[b])], k)
        n = check_rows(got, full["ref"], full["rows"], k, f"b={b}")
        log(f"batch {b}, top-{k}: {n} queries compared")
    if k == 10:
        assert gi.num_launches(64, k) == 1
    singles = [gi.topk(d_qi[c:c + 2] - d_qi[c], d_qt[int(qi[c]):int(qi[c + 1])], k) for c in range(64)]
    got = (torch.cat([s for s, _ in singles]), torch.cat([d for _, d in singles]))
    check_rows(got, full["ref"], full["rows"], k, "b=1")


def test_transcript_and_very_long_queries(full):
    """Rounds 1-3 search with LM transcripts: a kind="later" batch, and queries of 1,025-4,096 terms (concatenated
    later-round queries: no cursor scratch, every sub-tile searched again) over the full index."""
    gi = full["gi"]
    lqi, lqt = synth.queries_np(256, VOCAB, gi.df_host, kind="later", seed=77)
    rng = np.random.default_rng(78)
    parts, lens = [], []
    for _ in range(24):
        want, q = int(rng.integers(1025, 4097)), []
        while len(q) < want:
            j = int(rng.integers(0, 256))
            q.extend(lqt[lqi[j]:lqi[j + 1]].tolist())
        parts.append(q[:want])
        lens.append(want)
    vqi = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    vqt = np.array([t for q in parts for t in q], np.int32)
    for q_i, q_t, what in ((lqi, lqt, "transcripts"), (vqi, vqt, "1,025-4,096 terms")):
        rows = np.arange(len(q_i) - 1)
        ref = reference(gi, q_i, q_t, rows, 100)
        for plan in (dict(), dict(batch_variant=2), dict(batch_variant=2, tile_epochs=2)):
            tune(gi, **plan)
            for k in (10, 100):
                check_rows(gi.topk(*to_dev(gi, q_i, q_t), k), ref, rows, k, what)
        log(f"{what}: {len(rows)} queries compared")
    tune(gi)


def test_second_batch_on_the_same_index_and_workspace(full):
    gi = full["gi"]
    tune(gi)
    gi.topk(*to_dev(gi, full["qi"], full["qt"]), 10)
    qi2, qt2 = synth.queries_np(NQ, VOCAB, gi.df_host, seed=synth.QUERY_SEED + 1)
    got = gi.topk(*to_dev(gi, qi2, qt2), 10)
    rows = sample_rows(NQ, 1024, 2)
    n = check_rows(got, reference(gi, qi2, qt2, rows), rows, 10, "second batch")
    log(f"second batch: {n} queries compared")


# ----------------------------------------------------------------------------- doc-sharded over NCCL
def first_terms(qi, qt):
    """Every query cut to its first term: no query scores higher than in the full batch, most score lower -- bounds
    of the full batch left over in a later call would cut documents."""
    lens = np.minimum(np.diff(qi), 1)
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), qt[qi[:-1][lens > 0]].astype(np.int32)


# (name, batch, size, k): the third call follows the first, of a different batch with higher bounds, two calls later
# (the other half of the peer-shared threshold arrays)
CALLS = [("a65536k10", "a", NQ, 10), ("b4096k100", "b", 4096, 100), ("b65536k10", "b", NQ, 10), ("b1k10", "b", 1, 10),
         ("a64k128", "a", 64, 128)]


def cut(q, n):
    qi, qt = q
    return qi[:n + 1], qt[:qi[n]]


def shard_digests(gi, lo, hi):
    """SHA-256 of (indptr, doc ids, weights) of the cut [lo, hi) of an index, made as BM25Index.load(doc_range) does."""
    keep = (gi.doc_ids >= lo) & (gi.doc_ids < hi)
    run = torch.zeros(gi.doc_ids.numel() + 1, dtype=torch.int64, device=gi.device)
    torch.cumsum(keep, 0, out=run[1:])
    out = [run[gi.indptr], (gi.doc_ids[keep] - lo).to(torch.int32), gi.weights[keep]]
    del run, keep
    return [hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest() for t in out]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import bench
        from probing_rag_b200.sharding import ShardedBM25
        dev = torch.device("cuda", rank)
        gi, qi, qt = bench.build_workload(N_DOCS, VOCAB, NQ, dev, rank, world)
        want = np.load(os.path.join(out_dir, "digests.npy"), allow_pickle=True)[rank]
        got = [hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest() for t in (gi.indptr, gi.doc_ids, gi.weights)]
        assert got == list(want), f"rank {rank}: shard arrays differ from the cut of the single index"
        batches = {"a": (qi, qt), "b": first_terms(qi, qt)}
        res = {}
        for mode, list_rounds in (("p2p", 4), ("p2p", 0), ("allreduce", 0), (None, 0)):
            sb = ShardedBM25(gi, exchange=mode, max_queries=NQ, list_rounds=list_rounds)
            assert sb.exchange == mode
            for name, b, n, k in CALLS:
                q_i, q_t = cut(batches[b], n)
                s, d = sb.topk(torch.from_numpy(q_i).to(dev), torch.from_numpy(q_t).to(dev), k)
                torch.cuda.synchronize()
                res[f"{mode}{list_rounds}_{name}_s"], res[f"{mode}{list_rounds}_{name}_d"] = s.cpu().numpy(), d.cpu().numpy()
            sb.close()
        if rank == 0:
            np.savez(os.path.join(out_dir, "r0.npz"), **res)
        dig = hashlib.sha256(b"".join(v.tobytes() for _, v in sorted(res.items()))).hexdigest()
        with open(os.path.join(out_dir, f"digest{rank}"), "w") as f:
            f.write(dig)
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def single_lists(full):
    """The single-GPU lists of the call sequence, each checked against the reference where the sample reaches."""
    gi = full["gi"]
    tune(gi)
    batches = {"a": (full["qi"], full["qt"]), "b": first_terms(full["qi"], full["qt"])}
    rows = full["rows"]
    ref = {"a": full["ref"], "b": reference(gi, *batches["b"], rows)}
    out = {}
    for name, b, n, k in CALLS:
        s, d = gi.topk(*to_dev(gi, *cut(batches[b], n)), k)
        s, d = s.cpu().numpy(), d.cpu().numpy()
        check_rows((s, d), ref[b], rows, k, name)
        out[name] = (s, d)
    return out


@pytest.mark.timeout(3000)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_doc_shards_over_nccl_equal_the_single_gpu_lists(full, single_lists, tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp

    from probing_rag_b200.sharding import shard_range
    gi = full["gi"]
    dig = np.empty(world, dtype=object)
    for r in range(world):
        dig[r] = shard_digests(gi, *shard_range(N_DOCS, r, world))
    np.save(tmp_path / "digests.npy", dig, allow_pickle=True)
    t0 = time.perf_counter()
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    log(f"world {world}: {time.perf_counter() - t0:.1f} s")
    got = np.load(tmp_path / "r0.npz")
    digs = {open(tmp_path / f"digest{r}").read() for r in range(world)}
    assert len(digs) == 1, "ranks returned different merged lists"
    for mode in ("p2p4", "p2p0", "allreduce0", "None0"):
        for name, (s, d) in single_lists.items():
            assert_parity(got[f"{mode}_{name}_s"], got[f"{mode}_{name}_d"], s, d)
