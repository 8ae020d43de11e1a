"""Exact flat inner-product search without a GPU: the oracle's evaluation order and ranking rules (ties, never -0,
NaN after -inf, (-FLT_MAX, -1) padding), the IndexFlatIP file layout and read_index's dispatch on it, the filter's
upper bound against emulated bf16 products, C-ABI argument errors, the IP filter kernel's SASS, and
ShardedIndexFlatIP's host logic over two and three gloo ranks with the oracle standing in."""
import ctypes
import os
import re
import shutil
import socket
import struct
import subprocess
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from flat_ip_merge_oracle import merge_canonical_ip
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from probing_rag_b200 import _lib, build, dense, sharding

IP = dense.METRIC_INNER_PRODUCT
FMAX = fo.FLT_MAX


# ---------------------------------------------------------------------------------------------- oracle
def test_exact_inner_products_follow_the_documented_order():
    rng = np.random.default_rng(21)
    q = (rng.standard_normal(128) * np.logspace(-3, 3, 128)).astype(np.float32)
    X = (rng.standard_normal((5, 128)) * np.logspace(3, -3, 128)).astype(np.float32)
    for r in range(5):
        lanes = [0.0] * 32
        for j in range(128):
            lanes[j % 32] = lanes[j % 32] + float(q[j]) * float(X[r, j])
        for o in (16, 8, 4, 2, 1):
            lanes = [lanes[l] + lanes[l ^ o] for l in range(32)]
        assert fio.exact_inner_products(q, X[r:r + 1])[0] == np.float32(lanes[0])
    assert np.array_equal(fio.exact_inner_products_torch(torch.from_numpy(q), torch.from_numpy(X)).numpy(),
                          fio.exact_inner_products(q, X))


def test_score_is_never_negative_zero():
    q = np.zeros(64, np.float32)
    q[0], q[1] = 2.0 ** -100, -(2.0 ** -100)
    X = np.zeros((3, 64), np.float32)
    X[0, 0] = 2.0 ** -60           # -2^-160 after the f64 sum would round to -0 in f32
    X[0, 1] = 2.0 ** -60 * 1.5
    X[1, 0] = -0.0                  # (-0) products added to +0.0
    for s in (fio.exact_inner_products(q, X), fio.exact_inner_products_torch(torch.from_numpy(q), torch.from_numpy(X)).numpy()):
        assert np.all(s == 0) and not np.any(np.signbit(s))


def _special_rows():
    """Rows whose inner product with e_0 is each special value, some twice (exact ties)."""
    vals = [1.0, np.inf, -FMAX, 0.0, np.nan, -np.inf, FMAX, 1.0, -1.0, np.nan, -FMAX, -np.inf, 0.0]
    X = np.zeros((len(vals), 64), np.float32)
    X[:, 0] = np.array(vals, np.float32)
    q = np.zeros((1, 64), np.float32)
    q[0, 0] = 1.0
    return q, X


def test_canonical_ip_order_nan_and_padding():
    q, X = _special_rows()
    D, I = fio.search_canonical_ip(q, X, 16)
    # +inf, FLT_MAX, the two 1.0 by id, the two +0 by id, -1, the two -FLT_MAX, the two -inf, the two NaN, padding
    assert I[0].tolist() == [1, 6, 0, 7, 3, 12, 8, 2, 10, 5, 11, 4, 9, -1, -1, -1]
    assert np.all(np.isnan(D[0, 11:13])) and np.all(D[0, 11:13].view(np.uint32) == 0xFFFFFFFF)
    assert D[0, :11].tolist() == [np.inf, FMAX, 1, 1, 0, 0, -1, -FMAX, -FMAX, -np.inf, -np.inf]
    assert np.all(D[0, 13:] == -FMAX) and not np.any(np.signbit(D[0, 4:6]))
    D2, I2 = fio.search_canonical_ip_torch(torch.from_numpy(q), torch.from_numpy(X), 16)
    assert np.array_equal(I, I2) and np.array_equal(D.view(np.uint32), D2.view(np.uint32))
    D3, I3 = fio.search_canonical_ip(q, X, 16, rows_per_block=5)       # blockwise == whole
    assert np.array_equal(I, I3) and np.array_equal(D.view(np.uint32), D3.view(np.uint32))


def test_canonical_ip_ties_and_zero_query():
    rng = np.random.default_rng(22)
    base = rng.standard_normal((4, 64)).astype(np.float32)
    X = np.concatenate([base, base[::-1], np.zeros((2, 64), np.float32)])
    Q = np.concatenate([base[:1], np.zeros((1, 64), np.float32)])
    D, I = fio.search_canonical_ip(Q, X, 12)
    assert I[0, 0] == 0 and I[0, 1] == 7 and D[0, 0] == D[0, 1]                # equal scores: ascending ids
    keys = list(zip(fio.ip_key(D[0, :10]).tolist(), I[0, :10].tolist()))
    assert keys == sorted(keys)
    assert I[1, :10].tolist() == list(range(10)) and np.all(D[1, :10] == 0)    # zero query: pure id order
    assert I[0, 10:].tolist() == [-1, -1] and np.all(D[:, 10:] == -FMAX)
    D2, I2 = fio.search_canonical_ip_torch(torch.from_numpy(Q), torch.from_numpy(X), 12)
    assert np.array_equal(D, D2) and np.array_equal(I, I2)


def test_faiss_blas_ip_restatement_agrees_modulo_near_ties():
    rng = np.random.default_rng(23)
    X = rng.standard_normal((3000, 128)).astype(np.float32)
    Q = (X[:8] + 0.1 * rng.standard_normal((8, 128))).astype(np.float32)
    D, I = fio.search_canonical_ip(Q, X, 10)
    Db, Ib = fio.faiss_blas_search_ip(Q, X, 10)
    atol = 1e-6 * float(np.max(np.linalg.norm(Q, axis=1))) * float(np.max(np.linalg.norm(X, axis=1)))
    assert fo.agree_modulo_near_ties(D, I, Db, Ib, atol=atol)
    assert not fo.agree_modulo_near_ties(D, I, Db, Ib[:, ::-1], atol=atol)
    Ds, Is = fio.faiss_blas_search_ip(Q[:1], X[:3], 5)
    assert Is[0, 3:].tolist() == [-1, -1] and np.all(Ds[0, 3:] == -FMAX)


def test_merge_restatement_order_padding_and_bases():
    inf, nan = np.float32(np.inf), np.float32(np.nan)
    D = np.array([[[7.0, 1.0, -FMAX]], [[7.0, -inf, 0.0]], [[inf, nan, 2.0]]], np.float32)
    I = np.array([[[3, 1, -1]], [[0, 2, -1]], [[-1, 4, -1]]], np.int64)
    Dm, Im = merge_canonical_ip(D, I, [0, 2 ** 33, 10], 6)
    assert Im.tolist() == [[3, 2 ** 33, 1, 2 ** 33 + 2, 14, -1]]
    assert Dm[0, :4].tolist() == [7.0, 7.0, 1.0, -np.inf] and np.isnan(Dm[0, 4]) and Dm[0, 5] == -FMAX


# ---------------------------------------------------------------------------------------------- file layout
def test_ip_index_file_round_trip_and_layout(tmp_path):
    rng = np.random.default_rng(24)
    X = rng.standard_normal((37, 64)).astype(np.float32)
    p = str(tmp_path / "flat_ip.index")
    dense.write_rows(p, X, 64, IP)
    raw = open(p, "rb").read()
    assert raw[:4] == b"IxFI" and len(raw) == 45 + X.nbytes
    assert struct.unpack_from("<iqqqBiQ", raw, 4) == (64, 37, 1 << 20, 1 << 20, 1, 0, 37 * 64)
    mm = dense.read_rows(p, IP)
    assert isinstance(mm, np.memmap) and np.array_equal(np.asarray(mm), X)
    base, part = dense.read_shard_rows(p, metric=IP)
    assert base == 0 and np.array_equal(np.asarray(part), X)
    dense.write_rows(p, X[:0], 64, IP)
    assert dense.read_rows(p, IP).shape == (0, 64)
    with pytest.raises(ValueError):
        dense.write_rows(p, X, 64, 2)


@pytest.mark.parametrize("fourcc, metric_field, read_as, msg", [
    (b"IxFI", 1, IP, "metric_type 1"), (b"IxF2", 0, IP, "IxF2"), (b"IxFI", 0, dense.METRIC_L2, "IxFI"),
    (b"IxF2", 0, dense.METRIC_L2, "metric_type 0")])
def test_mismatched_fourcc_and_metric_are_rejected(tmp_path, fourcc, metric_field, read_as, msg):
    p = str(tmp_path / "flat.index")
    dense.write_rows(p, np.zeros((3, 64), np.float32), 64)
    raw = bytearray(open(p, "rb").read())
    raw[0:4] = fourcc
    raw[4 + 4 + 24 + 1:4 + 4 + 24 + 5] = struct.pack("<i", metric_field)
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=msg):
        dense.read_rows(p, read_as)


class _FakeIndex:
    """Stands in for IndexFlatL2 / IndexFlatIP in read_index (no device needed)."""

    def __init__(self, d, device):
        self.d, self.device, self.rows = d, torch.device("cpu"), None

    def _set_rows(self, rows):
        self.rows = rows


def test_read_index_dispatches_on_the_fourcc(tmp_path, monkeypatch):
    fakes = {name: type(name, (_FakeIndex,), {}) for name in ("IndexFlatL2", "IndexFlatIP")}
    for name, cls in fakes.items():
        monkeypatch.setattr(dense, name, cls)
    X = np.random.default_rng(25).standard_normal((10, 64)).astype(np.float32)
    for metric, name in ((IP, "IndexFlatIP"), (dense.METRIC_L2, "IndexFlatL2")):
        p = str(tmp_path / f"{name}.index")
        dense.write_rows(p, X, 64, metric)
        ix = dense.read_index(p)
        assert type(ix) is fakes[name] and torch.equal(ix.rows, torch.from_numpy(X))
    p = str(tmp_path / "other.index")
    dense.write_rows(p, X, 64)
    raw = bytearray(open(p, "rb").read())
    raw[0:4] = b"IxHF"
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="IxF2.*IxFI"):
        dense.read_index(p)


# ---------------------------------------------------------------------------------------------- margin
def _ip_upper_bound(q, x, c1_scale=1.0):
    """The filter's upper bound restated in f32 with the kernel's constants (csrc/flat.cu margin_c1ip), the dot
    product from bf16-rounded operands accumulated in f32 (one of the accumulation orders the margin allows)."""
    d = q.shape[0]
    u = 2.0 ** -8
    c1 = np.nextafter(np.float32(((2 * u + u * u) + d * 2.0 ** -22 * (1 + u) ** 2 + (d + 5) * 2.0 ** -53 + 2.0 ** -22)
                                 * (1 + 2.0 ** -10)), np.float32(np.inf))
    c1 = np.float32(c1 * c1_scale)
    c3 = np.float32(2.0 ** -100)
    qb = torch.from_numpy(q).bfloat16().float().numpy()
    xb = torch.from_numpy(x).bfloat16().float().numpy()
    acc = np.float32(0)
    for p in (qb * xb):
        acc = np.float32(acc + p)
    nrm = lambda v: np.float32(np.sqrt(np.dot(v.astype(np.float64), v.astype(np.float64))))
    qn, xn = nrm(q), nrm(x)
    margin = np.float32(np.float32(c1 * qn) * xn + np.float32(c3 * np.float32(np.float32(1 + qn) + xn)))
    return np.float32(acc + margin)


def _bf16_biased(d, rng):
    """q and x whose every element rounds down to bf16 by almost u: the bf16 dot product is short of q.x by almost
    2u |q||x|, all of it one-signed (the case the factor 2u + u^2 of c1ip exists for)."""
    c = np.float32(1 + 2.0 ** -8 - 2.0 ** -20)
    s = rng.choice([-1.0, 1.0], d) if rng.random() < 0.5 else np.ones(d)
    q = (c * s).astype(np.float32)
    return q, q.copy()


@pytest.mark.parametrize("case", ["dynamic_range", "cancellation", "near_duplicate", "d1024", "tiny", "negative",
                                  "mixed_sign", "bf16_biased"])
def test_ip_margin_is_an_upper_bound_on_adversarial_vectors(case):
    rng = np.random.default_rng(sum(map(ord, case)))
    d = 1024 if case == "d1024" else 768 if case == "bf16_biased" else 256
    for _ in range(20):
        q = rng.standard_normal(d)
        if case == "dynamic_range":
            q *= np.exp(rng.uniform(-30, 30, d))
            x = q * (1 + rng.uniform(-1e-2, 1e-2, d))
        elif case == "cancellation":
            r = rng.standard_normal(d)
            x = r - (r @ q) / (q @ q) * q + rng.standard_normal(d) * 1e-4     # q.x tiny against |q||x|
        elif case == "near_duplicate":
            x = q.copy()
            x[rng.integers(d)] *= 1 + 2.0 ** -20
        elif case == "tiny":
            q *= 1e-19
            x = q + rng.standard_normal(d) * 1e-21
        elif case == "negative":
            x = -q * rng.uniform(0.5, 2, d)
        elif case == "mixed_sign":
            x = rng.standard_normal(d) * np.exp(rng.uniform(-5, 5, d)) + 0.3 * q
        elif case == "bf16_biased":
            q, x = _bf16_biased(d, rng)
        else:
            x = rng.standard_normal(d) + 3 * q
        q, x = q.astype(np.float32), x.astype(np.float32)
        exact = fio.exact_inner_products(q, x[None, :])[0]
        assert np.isfinite(exact) and _ip_upper_bound(q, x) >= exact, case
        if case == "bf16_biased":                  # half the margin would not be a bound
            assert _ip_upper_bound(q, x, 0.5) < exact


# ---------------------------------------------------------------------------------------------- C ABI
def test_flat_metric_capi_argument_errors_without_gpu():
    L = _lib.lib()
    h = ctypes.c_void_p()
    rows = ctypes.c_void_p(0x10000)
    assert L.pr_flat_create_metric(None, 0, rows, 10, 64, IP) == _lib.PR_EINVAL
    assert L.pr_flat_create_metric(ctypes.byref(h), 0, None, 10, 64, IP) == _lib.PR_EINVAL
    assert L.pr_flat_create_metric(ctypes.byref(h), 0, rows, -1, 64, IP) == _lib.PR_EINVAL
    for metric in (2, -1, 23):
        assert L.pr_flat_create_metric(ctypes.byref(h), 0, rows, 10, 64, metric) == _lib.PR_EUNSUPPORTED
        assert b"metric" in L.pr_last_error() and not h.value
    assert L.pr_flat_create_metric(ctypes.byref(h), 0, rows, 10, 96, IP) == _lib.PR_EUNSUPPORTED
    assert b"multiple of 64" in L.pr_last_error()
    assert L.pr_flat_create_metric(ctypes.byref(h), 0, rows, 2 ** 31, 64, IP) == _lib.PR_EUNSUPPORTED
    assert L.pr_flat_create_metric(ctypes.byref(h), 0, ctypes.c_void_p(0x10004), 10, 64, IP) == _lib.PR_EINVAL
    p = ctypes.c_void_p(0x10000)
    base = (ctypes.c_int64 * 33)(*([0] * 33))
    for metric in (IP, dense.METRIC_L2):
        assert L.pr_flat_merge_metric(-1, 5, 2, p, p, base, p, p, None, metric) == _lib.PR_EINVAL
        assert L.pr_flat_merge_metric(4, 5, 33, p, p, base, p, p, None, metric) == _lib.PR_EINVAL
        assert b"n_lists" in L.pr_last_error()
        assert L.pr_flat_merge_metric(4, 129, 2, p, p, base, p, p, None, metric) == _lib.PR_EINVAL
        assert L.pr_flat_merge_metric(4, 5, 2, p, None, base, p, p, None, metric) == _lib.PR_EINVAL
        neg = (ctypes.c_int64 * 2)(0, -5)
        assert L.pr_flat_merge_metric(4, 5, 2, p, p, neg, p, p, None, metric) == _lib.PR_EINVAL
        assert b"negative" in L.pr_last_error()
        assert L.pr_flat_merge_metric(0, 5, 2, None, None, base, None, None, None, metric) == _lib.PR_OK
    assert L.pr_flat_merge_metric(4, 5, 2, p, p, base, p, p, None, 2) == _lib.PR_EUNSUPPORTED
    assert b"metric" in L.pr_last_error()


def test_ip_filter_kernel_sass():
    """The IP filter is the same tcgen05 GEMM fed by TMA with its accumulator read from TMEM, and nothing spills."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = build.build()
    res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout.splitlines()
    hit = [(l, res[i + 1]) for i, l in enumerate(res) if "flat_ip_filter_kernel" in l and i + 1 < len(res)]
    assert len(hit) == 1, hit
    m = re.search(r"REG:(\d+) STACK:(\d+)", hit[0][1])
    assert m and int(m.group(2)) == 0, hit[0]
    name = re.search(r"(_Z\w*flat_ip_filter_kernel\w*)", hit[0][0]).group(1)
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", name, lib], capture_output=True, text=True).stdout
    assert re.search(r"UTC[HQ]MMA", sass) and "UTMALDG" in sass and "LDTM" in sass
    assert "LDL" not in sass and "STL" not in sass


# ---------------------------------------------------------------------------------------------- shards over gloo
D_ = 64


def _matrix():
    """Every base row twice and a few three times, a block of zero rows: exact ties, across shard boundaries too;
    queries include zero queries (every score +0) and negated rows (negative scores)."""
    rng = np.random.default_rng(26)
    base = rng.standard_normal((100, D_)).astype(np.float32)
    X = np.concatenate([base, base, np.zeros((20, D_), np.float32), base[:5]])
    Q = np.concatenate([base[:30], np.zeros((2, D_), np.float32), -base[30:34],
                        rng.standard_normal((4, D_)).astype(np.float32)])
    return X, Q


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded(X, rank, world, metric_type=IP):
    lo, hi = sharding.shard_range(len(X), rank, world)
    Xl = X[lo:hi]

    def local_search(q, k):
        Dl, Il = fio.search_canonical_ip(q.numpy(), Xl, k)
        return torch.from_numpy(Dl), torch.from_numpy(Il)

    def merge(gd, gi, bases):
        Dm, Im = merge_canonical_ip(gd.numpy(), gi.numpy(), bases, gd.shape[2])
        return torch.from_numpy(Dm), torch.from_numpy(Im)

    shard = types.SimpleNamespace(d=D_, ntotal=hi - lo)
    if metric_type is not None:
        shard.metric_type = metric_type
    return dense.ShardedIndexFlatIP(shard, lo, local_search=local_search, merge=merge)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, Q = _matrix()
        res = {}
        for name, rows in (("full", X), ("tiny", X[:4])):        # tiny: the last of three ranks holds no rows
            ix = _sharded(rows, rank, world, metric_type=IP if rank else None)   # a shard with only d and ntotal
            assert ix.ntotal == len(rows) and ix.d == D_ and ix.is_trained and ix.metric_type == 0
            for k in (5, 64):
                Dn, In = ix.search(Q, k)
                assert isinstance(Dn, np.ndarray) and Dn.dtype == np.float32 and In.dtype == np.int64
                Dt, It = ix.search(torch.from_numpy(Q), k)
                assert isinstance(Dt, torch.Tensor) and np.array_equal(Dt.numpy(), Dn) and np.array_equal(It.numpy(), In)
                res[f"{name}_D{k}"], res[f"{name}_I{k}"] = Dn, In
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_ip_row_shards_equal_single_index(tmp_path, world):
    X, Q = _matrix()
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for name, rows in (("full", X), ("tiny", X[:4])):
        for k in (5, 64):
            Dw, Iw = fio.search_canonical_ip(Q, rows, k)
            for r in range(world):
                got = np.load(tmp_path / f"r{r}.npz")
                assert np.array_equal(got[f"{name}_I{k}"], Iw), f"rank {r} {name} k={k}: merged ids differ"
                assert np.array_equal(got[f"{name}_D{k}"], Dw), f"rank {r} {name} k={k}: merged scores differ"
    assert np.all(Iw[:, 4:] == -1) and np.all(Dw[:, 4:] == -FMAX)
    assert Iw[30].tolist()[:4] == [0, 1, 2, 3]                    # zero query: every score +0, pure id order


def test_sharded_classes_reject_a_shard_of_the_other_metric():
    X, Q = _matrix()
    with pytest.raises(ValueError, match="metric"):
        _sharded(X, 0, 1, metric_type=dense.METRIC_L2)
    with pytest.raises(ValueError, match="metric"):
        dense.ShardedIndexFlatL2(types.SimpleNamespace(d=D_, ntotal=4, metric_type=IP), 0,
                                 local_search=lambda q, k: None, merge=lambda *a: None)
    ix = _sharded(X, 0, 1)
    D, I = ix.search(Q, 10)
    Dw, Iw = fio.search_canonical_ip(Q, X, 10)
    assert np.array_equal(D, Dw) and np.array_equal(I, Iw)


# ---------------------------------------------------------------------------------------------- real faiss
def test_against_an_ip_file_written_by_faiss(tmp_path):
    """faiss writes an IndexFlatIP file, this package reads it; the search agrees with faiss's own modulo near-ties
    (the faiss part runs wherever faiss is installed; the GPU part where a device is present)."""
    faiss = pytest.importorskip("faiss")
    rng = np.random.default_rng(27)
    X = rng.standard_normal((5000, 768)).astype(np.float32)
    Q = (X[:16] + 0.05 * rng.standard_normal((16, 768))).astype(np.float32)
    ref = faiss.IndexFlatIP(768)
    ref.add(X)
    p = str(tmp_path / "faiss_ip.index")
    faiss.write_index(ref, p)
    assert open(p, "rb").read(4) == b"IxFI"
    assert np.array_equal(np.asarray(dense.read_rows(p, IP)), X)
    Df, If = ref.search(Q, 5)
    D, I = fio.search_canonical_ip(Q, X, 5)
    atol = 1e-6 * float(np.max(np.linalg.norm(Q, axis=1))) * float(np.max(np.linalg.norm(X, axis=1)))
    assert fo.agree_modulo_near_ties(D, I, Df, If, atol=atol)
    small = faiss.IndexFlatIP(768)                  # padding of k > ntotal: faiss's min-heap leaves (-FLT_MAX, -1)
    small.add(X[:3])
    Ds, Is = small.search(Q[:1], 5)
    assert list(Is[0, 3:]) == [-1, -1] and np.all(Ds[0, 3:] == -FMAX)
    if torch.cuda.is_available():
        gi = dense.read_index(p)
        assert isinstance(gi, dense.IndexFlatIP)
        Dg, Ig = gi.search(Q, 5)
        assert np.array_equal(Dg, D) and np.array_equal(Ig, I)
