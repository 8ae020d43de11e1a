"""Exact flat range search on the GPU (pr_flat_range_search through IndexFlatL2 / IndexFlatIP.range_search): lims,
ids and value bits equal to the canonical oracle (oracle/flat_range_oracle.py) for both metrics, at the radius and
a few ulp around it, on non-finite values, under every launch plan and staging size, against search, over simulated
and NCCL row shards, and at the full 21,015,324 x 768 size against the fast reference."""
import os
import socket

import numpy as np
import pytest
import torch

from flat_range_fast_oracle import range_search_fast
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from oracle import flat_range_oracle as fro
from probing_rag_b200 import IndexFlatIP, IndexFlatL2, ShardedIndexFlatIP, ShardedIndexFlatL2, sharding, synth
from test_gpu_flat import SHAPES

pytestmark = pytest.mark.gpu

CLS = {"l2": IndexFlatL2, "ip": IndexFlatIP}
SHARDED = {"l2": ShardedIndexFlatL2, "ip": ShardedIndexFlatIP}
INF, NAN = float("inf"), float("nan")
FMAX = float(np.finfo(np.float32).max)


def _index(X, metric, **plan):
    ix = CLS[metric](X.shape[1])
    ix.add(X)
    if plan:
        ix.set_tuning(**plan)
    return ix


def _np(res):
    return tuple(x.cpu().numpy() if isinstance(x, torch.Tensor) else x for x in res)


def _same(a, b):
    (la, Da, Ia), (lb, Db, Ib) = _np(a), _np(b)
    return (np.array_equal(la.astype(np.int64), lb.astype(np.int64)) and np.array_equal(Ia, Ib)
            and np.array_equal(Da.view(np.uint32), Db.view(np.uint32)))


def _check(ix, Q, radius, metric):
    got = ix.range_search(Q, radius)
    assert got[0].dtype == torch.int64 and got[0].is_cuda and got[1].is_cuda and got[2].dtype == torch.int64
    want = fro.range_search_canonical_torch(Q, ix.rows(), radius, metric)
    assert _same(got, want), f"{metric} radius {radius!r}: differs from the oracle"
    return got


def _values(Q, X, metric):
    f = fo.exact_distances_torch if metric == "l2" else fio.exact_inner_products_torch
    return torch.stack([f(q, X) for q in Q])


def _toward(v, metric):
    """The next f32 after v toward the inside of the ball: a radius that includes v."""
    return float(np.nextafter(np.float32(v), np.float32(INF if metric == "l2" else -INF)))


def _radii(Q, X, metric):
    """The 1st, 10th and 100th value of query 0 (excluded) and their nextafter (included), 0, a negative radius,
    +-inf and NaN."""
    v = _values(Q[:1], X, metric)[0]
    s = torch.sort(v, descending=metric == "ip").values.cpu().numpy()
    out = []
    for j in (0, 9, 99):
        if j < len(s):
            out += [float(s[j]), _toward(s[j], metric)]
    return out + [0.0, -1.5, INF, -INF, NAN]


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_shapes_at_radii_from_the_exact_values(n, d, B, k, metric):
    rows = synth.dense_rows(n, d)
    ix = _index(rows, metric)
    Q = synth.dense_queries(rows, min(B, 64))
    for r in _radii(Q, rows, metric):
        if n * min(B, 64) > 2_000_000 and abs(r) == INF:
            continue                                    # every row a result: covered by test_many_hits
        _check(ix, Q, r, metric)


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_near_radius_shells(metric):
    """Rows whose values lie a few ulp apart around the radius: only the margin keeps the ones inside."""
    g = torch.Generator(device="cuda").manual_seed(61)
    d = 768
    q = torch.randn(d, generator=g, device="cuda")
    u = torch.randn((20_000, d), generator=g, device="cuda")
    u = u / u.norm(dim=1, keepdim=True)
    r = 1.0 + torch.randint(0, 8, (20_000, 1), generator=g, device="cuda") * 2.0 ** -22
    X = torch.cat([synth.dense_rows(30_000, d) * 10, q[None, :] + u * r, synth.dense_rows(20_000, d) * 10])
    ix = _index(X, metric)
    Q = torch.stack([q, q + 1e-7 * torch.randn(d, generator=g, device="cuda")])
    v = torch.unique(_values(Q[:1], X[30_000:50_000], metric)[0]).cpu().numpy()
    picks = v[len(v) // 2 - 3: len(v) // 2 + 3]
    for a in picks:
        for r in (float(a), _toward(a, metric)):
            _check(ix, Q, r, metric)


def test_bf16_rounding_bias_needs_the_whole_margin():
    """The all-one-sign bf16 rounding case of test_gpu_flat_ip: the targets' bf16 products fall short of their exact
    scores by ~2u |q||x|; a radius just below the targets' score keeps them only with the filter's whole margin."""
    d = 768
    c = np.float32(1 + 2.0 ** -8 - 2.0 ** -20)
    q = torch.full((1, d), float(c), device="cuda")
    X = torch.zeros((30_000, d), device="cuda")
    X[:4096] = 1.0
    X[:4096, : d // 4] = 1 + 2.0 ** -7
    targets = [7_000, 12_345, 29_999]
    X[targets] = float(c)
    ix = _index(X, "ip")
    s = float(fio.exact_inner_products_torch(q[0], X[targets[:1]])[0])
    filler = float(fio.exact_inner_products_torch(q[0], X[:1])[0])
    assert filler < s
    for r in (float(np.nextafter(np.float32(s), np.float32(-INF))), (filler + s) / 2):
        lims, D, I = _check(ix, q, r, "ip")
        assert I.tolist() == targets


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_special_values_in_the_first_and_later_chunks(metric):
    g = torch.Generator(device="cuda").manual_seed(62)
    d = 64
    X = torch.randn((40_000, d), generator=g, device="cuda")
    for base in (5, 1_000, 20_000, 39_990):             # the first chunk, and chunks reached through the filter
        X[base, 0] = NAN
        X[base + 1, 1] = INF
        X[base + 2, 2] = -INF
        X[base + 3] = 0.0
        X[base + 4] = 3e38
        X[base + 5] = -3e38
    Q = torch.cat([X[100:102], torch.zeros((1, d), device="cuda"), torch.rand((1, d), generator=g, device="cuda") + 0.5])
    for plan in ({}, dict(first_chunk_rows=128, growth=2)):
        ix = _index(X, metric, **plan)
        for r in [1.0, 50.0, 128.0, FMAX, INF, -INF, 0.0, -5.0, NAN]:
            _check(ix, Q, r, metric)


PLANS = [dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2), dict(cand_capacity=1), {}]


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_launch_plans_and_staging_sizes_give_identical_output(metric):
    rows = synth.dense_rows(100_003, 256)
    Q = synth.dense_queries(rows, 257)
    v = torch.sort(_values(Q[:1], rows, metric)[0], descending=metric == "ip").values.cpu().numpy()
    for r in (float(v[9]), _toward(v[499], metric)):
        ref = fro.range_search_canonical_torch(Q, rows, r, metric)
        for plan in PLANS:
            ix = _index(rows, metric, **plan)
            assert _same(ix.range_search(Q, r), ref), plan
            st = ix.last_stats()
            assert st["launches"] == 2 * st["chunks"] + 2, plan
            if plan.get("first_chunk_rows") == 1 << 30:
                assert st["chunks"] == 1
            if plan.get("cand_capacity") == 1:
                assert st["fallback_queries"] > 0
            if plan.get("growth") == 2:
                assert st["chunks"] >= 8
        ix = _index(rows, metric)
        ix._range_cap_forced = 1                            # every query overflows the staging: the second pass
        assert _same(ix.range_search(Q, r), ref)
        ix._range_cap_forced = None
        assert _same(ix.range_search(Q, r), ref) and ix._range_cap >= int(np.diff(ref[0]).max())
        lims, D, I = ix.range_search(Q.cpu().numpy(), r)     # NumPy in -> NumPy out, lims as faiss's size_t
        assert lims.dtype == np.uint64 and isinstance(D, np.ndarray) and _same((lims, D, I), ref)


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_many_hits(metric):
    """Every finite row of 100,003 is a result of a few queries: one CTA per query scans every chunk."""
    rows = synth.dense_rows(100_003, 768)
    rows[777, 5] = NAN
    Q = synth.dense_queries(rows, 3)
    ix = _index(rows, metric)
    lims, D, I = _check(ix, Q, INF if metric == "l2" else -INF, metric)
    assert lims.tolist() == [0, 100_002, 200_004, 300_006] and 777 not in I[:100_002].tolist()


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_first_k_results_equal_search(metric):
    rows = synth.dense_rows(50_000, 768)
    rows[1000:1010] = rows[2000:2010]                    # exact ties
    Q = torch.cat([synth.dense_queries(rows, 16), rows[2000:2002]])
    ix = _index(rows, metric)
    for k in (1, 10, 100):
        Ds, Is = ix.search(Q, k)
        for b in range(Q.shape[0]):
            r = _toward(Ds[b, k - 1].item(), metric)
            lims, D, I = ix.range_search(Q[b:b + 1], r)
            key = D.view(torch.int32).to(torch.int64) if metric == "l2" else fio.ip_key_torch(D)
            o = np.lexsort((I.cpu().numpy(), key.cpu().numpy()))[:k]
            assert torch.equal(I[o], Is[b]) and torch.equal(D[o].view(torch.int32), Ds[b].view(torch.int32)), (k, b)


def _concat_shards(parts, bases, B):
    """Per query, the shards' results in shard order with ids + base."""
    lims, Ds, Is = [0], [], []
    for b in range(B):
        for (l, D, I), base in zip(parts, bases):
            Ds.append(D[l[b]:l[b + 1]])
            Is.append(I[l[b]:l[b + 1]] + base)
        lims.append(lims[-1] + sum(int(p[0][b + 1] - p[0][b]) for p in parts))
    return np.array(lims), np.concatenate(Ds), np.concatenate(Is)


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("parts", [2, 3, 8])
def test_simulated_shards_equal_one_index(metric, parts):
    rows = synth.dense_rows(100_003, 768)
    rows[50_000:50_010] = rows[10:20]
    Q = synth.dense_queries(rows, 65)
    one = _index(rows, metric)
    v = torch.sort(_values(Q[:1], rows, metric)[0], descending=metric == "ip").values.cpu().numpy()
    cuts = [sharding.shard_range(len(rows), p, parts) for p in range(parts)] + [(len(rows), len(rows))]   # + an empty one
    shards = [_index(rows[lo:hi], metric) for lo, hi in cuts]
    for r in (float(v[9]), _toward(v[99], metric), INF if metric == "l2" else -INF):
        want = one.range_search(Q, r)
        got = _concat_shards([_np(s.range_search(Q, r)) for s in shards], [lo for lo, _ in cuts], Q.shape[0])
        assert _same(got, want)


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
        res = {}
        rows = synth.dense_rows(100_003, 768, device=dev)
        Q = synth.dense_queries(rows, 33)
        radii = np.load(os.path.join(out_dir, "radii.npz"))
        for metric in ("l2", "ip"):
            lo, hi = sharding.shard_range(len(rows), rank, world)
            ix = SHARDED[metric](_index(rows[lo:hi], metric), lo)
            for j, r in enumerate(radii[metric]):
                lims, D, I = ix.range_search(Q, float(r))
                ln, Dn, In = ix.range_search(Q.cpu().numpy(), float(r))
                assert ln.dtype == np.uint64 and _same((ln, Dn, In), (lims, D, I))
                res[f"{metric}{j}_l"], res[f"{metric}{j}_D"], res[f"{metric}{j}_I"] = _np((lims, D, I))
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 4])
def test_nccl_row_shards_equal_one_index(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp
    rows = synth.dense_rows(100_003, 768)
    Q = synth.dense_queries(rows, 33)
    radii, want = {}, {}
    for metric in ("l2", "ip"):
        v = torch.sort(_values(Q[:1], rows, metric)[0], descending=metric == "ip").values.cpu().numpy()
        radii[metric] = np.array([v[9], _toward(v[99], metric), INF if metric == "l2" else -INF], np.float64)
        one = _index(rows, metric)
        want[metric] = [one.range_search(Q, float(r)) for r in radii[metric]]
    np.savez(tmp_path / "radii.npz", **radii)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        got = np.load(tmp_path / f"r{rank}.npz")
        for metric in ("l2", "ip"):
            for j in range(3):
                assert _same((got[f"{metric}{j}_l"], got[f"{metric}{j}_D"], got[f"{metric}{j}_I"]), want[metric][j])


# ---------------------------------------------------------------------------------------------- full size
@pytest.mark.skipif(os.environ.get("PR_SKIP_FULL") == "1", reason="PR_SKIP_FULL=1")
@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_full_size_against_the_fast_reference(metric):
    """21,015,324 x 768 clustered rows, 48 sampled queries of the 4,096-query batch, radii giving about 10 and 1,000
    hits per query (the median over the sample of the f64-estimated 10th and 1,000th value), under three plans.  The
    index is test_gpu_flat_fullsize's resident one, so that one 21M-row index is on the device at a time (64.5 GB of
    rows and 32 GB of bf16 copy); the chunks of the reference are bounded at 1M rows (6.4 GB in f64)."""
    import test_gpu_flat_fullsize as fs
    res = fs.resident(metric)
    ix = res["index"]
    X = ix.rows()
    sel = np.sort(np.random.default_rng(7).choice(res["Q"].shape[0], 48, replace=False))
    Q = res["Q"][torch.from_numpy(sel).cuda()].contiguous()
    Q64 = Q.to(torch.float64)
    best = []
    for a in range(0, X.shape[0], 1 << 20):
        Xc = X[a:a + (1 << 20)].to(torch.float64)
        e = (Xc * Xc).sum(1)[None, :] - 2.0 * Q64 @ Xc.T if metric == "l2" else -(Q64 @ Xc.T)
        best.append(torch.topk(e, 1000, dim=1, largest=False).values)
        del Xc, e
    best = torch.topk(torch.cat(best, 1), 1000, dim=1, largest=False).values
    best = best + (Q64 * Q64).sum(1)[:, None] if metric == "l2" else -best
    try:
        for j in (9, 999):
            r = float(torch.median(best[:, j]))
            want = range_search_fast(Q, X, r, metric)
            hits = np.diff(want[0])
            assert 1 <= np.median(hits) <= 3 * (j + 1)
            for plan in ({}, dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2)):
                ix.set_tuning(**plan)
                assert _same(ix.range_search(Q, r), want), (j, plan)
    finally:
        ix.set_tuning()
