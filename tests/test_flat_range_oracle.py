"""Exact flat range search without a GPU: the oracle's semantics at the radius and on non-finite values, the fast
reference against it, C-ABI argument errors, the range refine's SASS and the filter's unchanged resources, row-range
shards over gloo, and faiss's own range_search where faiss is installed."""
import ctypes
import os
import re
import shutil
import socket
import subprocess
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from flat_range_fast_oracle import range_search_fast
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from oracle import flat_range_oracle as fro
from probing_rag_b200 import _lib, build, dense, sharding

INF, NAN = float("inf"), float("nan")


def _values(Q, X, metric):
    f = fo.exact_distances if metric == "l2" else fio.exact_inner_products
    return np.stack([f(q, X) for q in Q]) if len(X) and len(Q) else np.zeros((len(Q), len(X)), np.float32)


def _brute(Q, X, radius, metric):
    """The contract restated per (query, row) in plain Python."""
    r = np.float32(radius)
    lims, D, I = [0], [], []
    V = _values(Q, X, metric)
    for b in range(len(Q)):
        for i in range(len(X)):
            v = V[b, i]
            if (v < r) if metric == "l2" else (v > r):
                D.append(v)
                I.append(i)
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D, np.float32), np.array(I, np.int64)


def _same(a, b):
    la, Da, Ia = a
    lb, Db, Ib = b
    return (np.array_equal(np.asarray(la, np.int64), np.asarray(lb, np.int64)) and np.array_equal(Ia, Ib)
            and np.array_equal(np.asarray(Da, np.float32).view(np.uint32), np.asarray(Db, np.float32).view(np.uint32)))


def _both(Q, X, radius, metric):
    """The NumPy oracle, checked against its torch form and the per-pair restatement."""
    got = fro.range_search_canonical(Q, X, radius, metric)
    assert _same(got, fro.range_search_canonical_torch(torch.from_numpy(Q), torch.from_numpy(X), radius, metric))
    assert _same(got, _brute(Q, X, radius, metric))
    return got


def _rows(seed=0, n=60, d=64):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d)).astype(np.float32)
    Q = np.concatenate([X[:3] + 0.1 * rng.standard_normal((3, d)).astype(np.float32),
                        rng.standard_normal((2, d)).astype(np.float32)])
    return Q, X


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_a_row_at_the_radius_is_excluded_and_one_ulp_inside_included(metric):
    Q, X = _rows(1)
    X = np.concatenate([X, X[7:8], X[7:8]])            # rows 7, 60, 61 tie exactly
    V = _values(Q[:1], X, metric)[0]
    v = V[7]
    inside = np.nextafter(v, np.float32(INF if metric == "l2" else -INF))
    lims, D, I = _both(Q[:1], X, v, metric)
    assert 7 not in I and 60 not in I and 61 not in I
    lims2, D2, I2 = _both(Q[:1], X, inside, metric)
    assert {7, 60, 61} <= set(I2.tolist())
    assert len(I2) == len(I) + 3 + int(np.sum(V == inside))
    assert np.all(np.diff(I2) > 0) and np.all(D2 == V[I2])


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_a_python_float_radius_is_rounded_to_f32_first(metric):
    Q, X = _rows(2)
    v = _values(Q[:1], X, metric)[0][5]
    ulp = float(np.spacing(v))
    above = float(v) + 0.25 * ulp if metric == "l2" else float(v) - 0.25 * ulp   # rounds back to v
    assert np.float32(above) == v
    _, _, I = _both(Q[:1], X, above, metric)
    assert 5 not in I                                   # an f64 comparison would have kept row 5


def _special():
    rng = np.random.default_rng(3)
    X = rng.standard_normal((40, 64)).astype(np.float32)
    X[3, 0] = NAN
    X[4, 1] = INF
    X[5, 2] = -INF
    X[6] = 0.0
    X[7, :] = 3e38                                       # distance and score overflow to inf
    Q = np.concatenate([X[10:12], np.zeros((1, 64), np.float32), -np.abs(X[12:13])])
    Qs = Q.copy()
    Qs[0, 5] = NAN
    Qs[1, 6] = INF
    return Q, Qs, X


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("radius", [0.0, -1.0, 1.0, 100.0, 1e30, INF, -INF, NAN])
def test_non_finite_rows_queries_and_radii(metric, radius):
    Q, Qs, X = _special()
    for QQ in (Q, Qs):
        lims, D, I = _both(QQ, X, radius, metric)
        V = _values(QQ, X, metric)
        assert not np.any(np.isnan(D))
        if radius != radius:
            assert lims[-1] == 0
        if metric == "l2":
            assert np.all(D >= 0)
            if radius <= 0:
                assert lims[-1] == 0
            if radius == INF:                              # every row with a finite distance
                assert lims[-1] == int(np.isfinite(V).sum())
        elif radius == -INF:                               # every row scoring other than -inf and NaN
            assert lims[-1] == int((~np.isnan(V) & (V != -INF)).sum())
        for b in range(len(QQ)):
            assert np.all(np.diff(I[lims[b]:lims[b + 1]]) > 0)


def test_ip_scores_are_never_negative_zero():
    Q = np.zeros((2, 64), np.float32)
    Q[1, 0] = 1e-30
    X = -np.ones((5, 64), np.float32)
    X[:, 0] = -1e-30                                       # q.x underflows f32 from below
    lims, D, I = _both(Q, X, -1.0, "ip")
    assert lims[-1] == 10 and np.all(D.view(np.uint32) == 0)


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_empty_batch_and_empty_index(metric):
    Q, X = _rows(4)
    lims, D, I = _both(Q[:0], X, 1.0, metric)
    assert lims.tolist() == [0] and len(D) == len(I) == 0
    lims, D, I = _both(Q, X[:0], INF if metric == "l2" else -INF, metric)
    assert lims.tolist() == [0] * (len(Q) + 1) and len(D) == len(I) == 0
    for bad in ("cos", None):
        with pytest.raises(ValueError):
            fro.range_search_canonical(Q, X, 1.0, bad)


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_fast_reference_equals_the_canonical_one(metric):
    rng = np.random.default_rng(5)
    base = rng.standard_normal((500, 128)).astype(np.float32)
    X = np.concatenate([base, base[:50], rng.standard_normal((3000, 128)).astype(np.float32) * 3])
    Q = np.concatenate([base[:6] + 0.05 * rng.standard_normal((6, 128)).astype(np.float32), np.zeros((1, 128), np.float32)])
    Qt, Xt = torch.from_numpy(Q), torch.from_numpy(X)
    V = _values(Q, X, metric)
    srt = np.sort(V, axis=1) if metric == "l2" else -np.sort(-V, axis=1)
    radii = [srt[0, 0], srt[0, 9], np.nextafter(srt[0, 9], np.float32(INF if metric == "l2" else -INF)),
             float(np.median(srt[:, 99])), float(np.median(srt[:, 1999])), 0.0, -3.0, INF, -INF, NAN]
    for r in radii:
        ref = fro.range_search_canonical(Q, X, r, metric)
        st = {}
        got = range_search_fast(Qt, Xt, r, metric, chunk_rows=1000, stats=st)
        assert _same(got, ref), r
        if r == r:
            assert all(s >= c for s, c in zip(st["survivors"], np.diff(ref[0])))
    with pytest.raises(ValueError):
        Xb = X.copy()
        Xb[3, 3] = INF
        range_search_fast(Qt, torch.from_numpy(Xb), 1.0, metric)


# ---------------------------------------------------------------------------------------------- C ABI
class _FakeFlat(ctypes.Structure):
    """struct pr_flat of csrc/flat.cu, field for field: a handle built without a device, for the checks that
    pr_flat_range_search makes before it touches one."""
    _fields_ = [("device", ctypes.c_int), ("n_sm", ctypes.c_int), ("n", ctypes.c_int64), ("d", ctypes.c_int32),
                ("rows", ctypes.c_void_p), ("rows_bf", ctypes.c_void_p), ("norm2", ctypes.c_void_p),
                ("norm", ctypes.c_void_p), ("metric", ctypes.c_int), ("tun", _lib.FlatTuning),
                ("last_launches", ctypes.c_int64), ("last_chunks", ctypes.c_int64)]


def test_range_capi_argument_errors_without_gpu():
    L = _lib.lib()
    p = ctypes.c_void_p(0x10000)
    ws = ctypes.c_void_p(0x100000)
    assert L.pr_flat_range_workspace_bytes(None, 4) == 0
    assert L.pr_flat_range_search(None, 1, p, 1.0, p, p, p, p, ws, 1 << 20, None) == _lib.PR_EINVAL
    for metric in (dense.METRIC_L2, dense.METRIC_INNER_PRODUCT):
        fake = _FakeFlat(device=0, n_sm=148, n=1000, d=64, rows=0x10000, metric=metric)
        h = ctypes.cast(ctypes.pointer(fake), ctypes.c_void_p)
        assert L.pr_flat_range_workspace_bytes(h, 0) == 0
        need = L.pr_flat_range_workspace_bytes(h, 4)
        assert need == L.pr_flat_workspace_bytes(h, 4, 1) > 0
        args = lambda **kw: [kw.get(n, v) for n, v in (("h", h), ("B", 4), ("q", p), ("r", 1.0), ("lims", p),
                                                         ("count", p), ("D", p), ("I", p), ("ws", ws),
                                                         ("nb", need), ("st", None))]
        assert L.pr_flat_range_search(*args(B=-1)) == _lib.PR_EINVAL
        assert b"negative batch" in L.pr_last_error()
        for name in ("q", "lims", "count", "D", "I", "ws"):
            assert L.pr_flat_range_search(*args(**{name: None})) == _lib.PR_EINVAL, name
        assert L.pr_flat_range_search(*args()) == _lib.PR_EINVAL          # pr_flat_build_aux not called
        assert b"pr_flat_build_aux" in L.pr_last_error()
        fake.rows_bf, fake.norm2, fake.norm = 0x200000, 0x300000, 0x400000
        for name, bad in (("q", 0x10004), ("ws", 0x100100), ("lims", 0x10004), ("count", 0x10004), ("I", 0x10004),
                          ("D", 0x10002)):
            assert L.pr_flat_range_search(*args(**{name: ctypes.c_void_p(bad)})) == _lib.PR_EINVAL, name
            assert b"aligned" in L.pr_last_error()
        assert L.pr_flat_range_search(*args(nb=need - 1)) == _lib.PR_EWORKSPACE
        assert b"workspace" in L.pr_last_error()
        assert L.pr_flat_range_search(*args(B=0, q=None, lims=None, count=None, D=None, I=None, ws=None)) == _lib.PR_OK
        assert fake.last_launches == 0 and fake.last_chunks == 0


def _res_usage(lib):
    res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout.splitlines()
    return {re.search(r"\d(flat\w*?_kernel)", l).group(1): (re.search(r"(_Z\w+)", l).group(1), res[i + 1])
            for i, l in enumerate(res) if re.search(r"\dflat\w*?_kernel", l) and i + 1 < len(res)}


def test_range_refine_sass_and_filter_resources():
    """Both range refine kernels are compiled for sm_100a without local memory; the filter kernels they run behind keep
    the registers and stack of exact top-k search (79 and 76 registers, no stack)."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = build.build()
    use = _res_usage(lib)
    for kern in ("flat_range_refine_kernel", "flat_ip_range_refine_kernel"):
        name, line = use[kern]
        m = re.search(r"REG:(\d+) STACK:(\d+)", line)
        assert m and int(m.group(2)) == 0 and "LOCAL:0" in line, line
        out = subprocess.run(["cuobjdump", "-sass", "-fun", name, lib], capture_output=True, text=True).stdout
        sass = next(part for part in out.split("Fatbin elf code") if "Function : " + name in part)
        assert "arch = sm_100a" in sass
        assert "DFMA" not in sass and "DADD" in sass and "DMUL" in sass            # the exact f64 evaluation
        assert "LDL" not in sass and "STL" not in sass
    for kern, regs in (("flat_filter_kernel", 79), ("flat_ip_filter_kernel", 76)):
        m = re.search(r"REG:(\d+) STACK:(\d+)", use[kern][1])
        assert m and (int(m.group(1)), int(m.group(2))) == (regs, 0), use[kern]


# ---------------------------------------------------------------------------------------------- shards over gloo
D_ = 64


def _matrix():
    """Rows twice and three times (exact ties across shard boundaries), zero rows, and a NaN row."""
    rng = np.random.default_rng(26)
    base = rng.standard_normal((100, D_)).astype(np.float32)
    X = np.concatenate([base, base, np.zeros((20, D_), np.float32), base[:5]])
    X[150, 3] = NAN
    Q = np.concatenate([base[:6], np.zeros((1, D_), np.float32), rng.standard_normal((3, D_)).astype(np.float32)])
    return X, Q


RADII = {"l2": [0.0, 60.0, 128.0, INF, NAN], "ip": [-INF, -5.0, 0.0, 30.0, INF]}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded(X, rank, world, metric):
    lo, hi = sharding.shard_range(len(X), rank, world)
    Xl = X[lo:hi]

    def local_range(q, radius):
        return tuple(torch.from_numpy(a) for a in fro.range_search_canonical(q.numpy(), Xl, radius, metric))

    shard = types.SimpleNamespace(d=D_, ntotal=hi - lo)
    cls = dense.ShardedIndexFlatL2 if metric == "l2" else dense.ShardedIndexFlatIP
    return cls(shard, lo, local_range=local_range)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, Q = _matrix()
        res = {}
        for metric in ("l2", "ip"):
            for name, rows in (("full", X), ("tiny", X[:2])):      # tiny: the last ranks hold no rows
                ix = _sharded(rows, rank, world, metric)
                for j, r in enumerate(RADII[metric]):
                    lims, D, I = ix.range_search(Q, r)
                    assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
                    lt, Dt, It = ix.range_search(torch.from_numpy(Q), r)
                    assert lt.dtype == torch.int64 and np.array_equal(lt.numpy(), lims.astype(np.int64))
                    assert np.array_equal(It.numpy(), I) and np.array_equal(Dt.numpy().view(np.uint32), D.view(np.uint32))
                    res[f"{metric}_{name}_{j}_l"], res[f"{metric}_{name}_{j}_D"], res[f"{metric}_{name}_{j}_I"] = lims, D, I
                lims, D, I = ix.range_search(Q[:0], 1.0)
                assert lims.tolist() == [0] and len(D) == 0
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_range_row_shards_equal_single_index(tmp_path, world):
    X, Q = _matrix()
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for metric in ("l2", "ip"):
        for name, rows in (("full", X), ("tiny", X[:2])):
            for j, r in enumerate(RADII[metric]):
                want = fro.range_search_canonical(Q, rows, r, metric)
                for rank in range(world):
                    got = np.load(tmp_path / f"r{rank}.npz")
                    key = f"{metric}_{name}_{j}"
                    assert _same((got[key + "_l"], got[key + "_D"], got[key + "_I"]), want), (rank, key)


def test_sharded_range_search_of_one_rank_equals_the_index():
    X, Q = _matrix()
    for metric in ("l2", "ip"):
        ix = _sharded(X, 0, 1, metric)
        for r in RADII[metric]:
            assert _same(ix.range_search(Q, r), fro.range_search_canonical(Q, X, r, metric))


# ---------------------------------------------------------------------------------------------- real faiss
@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_against_faiss_range_search(metric):
    """faiss's own range_search agrees with the oracle except for rows within 1e-5 relative of the radius, and its
    lims are uint64 (RangeSearchResult.lims is size_t), as range_search returns them for NumPy input."""
    faiss = pytest.importorskip("faiss")
    rng = np.random.default_rng(28)
    X = rng.standard_normal((5000, 768)).astype(np.float32)
    Q = (X[:16] + 0.5 * rng.standard_normal((16, 768))).astype(np.float32)
    ref = (faiss.IndexFlatL2 if metric == "l2" else faiss.IndexFlatIP)(768)
    ref.add(X)
    V = _values(Q, X, metric)
    radius = float(np.median(np.sort(V, 1)[:, 20] if metric == "l2" else -np.sort(-V, 1)[:, 20]))
    lf, Df, If = ref.range_search(Q, radius)
    assert lf.dtype == np.uint64 and Df.dtype == np.float32 and If.dtype == np.int64
    lims, D, I = fro.range_search_canonical(Q, X, radius, metric)
    for b in range(len(Q)):
        a, f = set(I[lims[b]:lims[b + 1]].tolist()), set(If[lf[b]:lf[b + 1]].tolist())
        for i in a ^ f:
            assert abs(float(V[b, i]) - radius) <= 1e-5 * abs(radius), (b, i)
    if torch.cuda.is_available():
        gi = (dense.IndexFlatL2 if metric == "l2" else dense.IndexFlatIP)(768)
        gi.add(X)
        got = gi.range_search(Q, radius)
        assert got[0].dtype == np.uint64 and _same(got, (lims, D, I))
