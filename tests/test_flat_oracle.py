"""Exact flat L2 search without a GPU: the oracle's order and ties, the IndexFlatL2 file layout, the filter's margin
against emulated bf16 products, C-ABI argument errors and the filter kernel's SASS."""
import ctypes
import os
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest
import torch

from oracle import flat_oracle as fo
from probing_rag_b200 import _lib, build, dense


def test_exact_distances_follow_the_documented_order():
    rng = np.random.default_rng(1)
    q = rng.standard_normal(128).astype(np.float32)
    X = (rng.standard_normal((5, 128)) * np.logspace(-3, 3, 128)).astype(np.float32)
    for r in range(5):
        lanes = [0.0] * 32
        for j in range(128):
            df = float(q[j]) - float(X[r, j])
            lanes[j % 32] = lanes[j % 32] + df * df
        for o in (16, 8, 4, 2, 1):
            lanes = [lanes[l] + lanes[l ^ o] for l in range(32)]
        assert fo.exact_distances(q, X[r:r + 1])[0] == np.float32(lanes[0])
    assert np.array_equal(fo.exact_distances_torch(torch.from_numpy(q), torch.from_numpy(X)).numpy(),
                          fo.exact_distances(q, X))


def test_canonical_order_ties_and_padding():
    rng = np.random.default_rng(2)
    base = rng.standard_normal((4, 64)).astype(np.float32)
    X = np.concatenate([base, base[::-1], np.zeros((2, 64), np.float32)])   # every row twice, two zero rows
    D, I = fo.search_canonical(base[:1], X, 12)
    assert I[0, 0] == 0 and I[0, 1] == 7 and D[0, 0] == D[0, 1] == 0.0     # equal distances: ascending ids
    for a in range(9):
        assert (D[0, a], I[0, a]) <= (D[0, a + 1], I[0, a + 1])
    assert list(I[0, 10:]) == [-1, -1] and np.all(D[0, 10:] == fo.FLT_MAX)  # k > n: (FLT_MAX, -1)
    D2, I2 = fo.search_canonical_torch(torch.from_numpy(base[:1]), torch.from_numpy(X), 12)
    assert np.array_equal(D, D2) and np.array_equal(I, I2)


def test_faiss_blas_restatement_agrees_modulo_near_ties():
    rng = np.random.default_rng(3)
    X = rng.standard_normal((3000, 128)).astype(np.float32)
    Q = (X[:8] + 0.1 * rng.standard_normal((8, 128))).astype(np.float32)
    D, I = fo.search_canonical(Q, X, 10)
    Db, Ib = fo.faiss_blas_search(Q, X, 10)
    atol = 1e-6 * 2 * float(np.max(np.sum(X * X, 1)))
    assert fo.agree_modulo_near_ties(D, I, Db, Ib, atol=atol)
    assert not fo.agree_modulo_near_ties(D, I, Db, Ib[:, ::-1], atol=atol)


def test_index_file_round_trip_and_layout(tmp_path):
    rng = np.random.default_rng(4)
    X = rng.standard_normal((37, 64)).astype(np.float32)
    p = str(tmp_path / "flat.index")
    dense.write_rows(p, X, 64)
    raw = open(p, "rb").read()
    assert raw[:4] == b"IxF2" and len(raw) == 45 + X.nbytes
    assert struct.unpack_from("<iqqqBiQ", raw, 4) == (64, 37, 1 << 20, 1 << 20, 1, 1, 37 * 64)
    mm = dense.read_rows(p)
    assert isinstance(mm, np.memmap) and np.array_equal(np.asarray(mm), X)
    dense.write_rows(p, X[:0], 64)
    assert dense.read_rows(p).shape == (0, 64)


@pytest.mark.parametrize("patch, msg", [((0, b"IxFI"), "IxFI"), ((4 + 4 + 24 + 1, struct.pack("<i", 0)), "metric_type 0")])
def test_index_file_other_types_are_rejected(tmp_path, patch, msg):
    p = str(tmp_path / "flat.index")
    dense.write_rows(p, np.zeros((3, 64), np.float32), 64)
    raw = bytearray(open(p, "rb").read())
    off, b = patch
    raw[off:off + len(b)] = b
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=msg):
        dense.read_rows(p)


def _margin_lower_bound(q, x):
    """The filter's lower bound restated in f32 with the kernel's constants (csrc/flat.cu), the dot product from
    bf16-rounded operands accumulated in f32 (one of the accumulation orders the margin allows)."""
    d = q.shape[0]
    u = 2.0 ** -8
    c1 = np.nextafter(np.float32(2 * ((2 * u + u * u) + d * 2.0 ** -22 * (1 + u) ** 2) * (1 + 2.0 ** -10)), np.float32(np.inf))
    c2, c3 = np.float32(2.0 ** -17), np.float32(2.0 ** -100)
    qb = torch.from_numpy(q).bfloat16().float().numpy()
    xb = torch.from_numpy(x).bfloat16().float().numpy()
    acc = np.float32(0)
    for p in (qb * xb):
        acc = np.float32(acc + p)
    n2 = lambda v: np.float32(np.dot(v.astype(np.float64), v.astype(np.float64)))
    qn2, xn2 = n2(q), n2(x)
    qn, xn = np.float32(np.sqrt(np.float64(qn2))), np.float32(np.sqrt(np.float64(xn2)))
    s2 = np.float32(qn2 + xn2)
    margin = np.float32(np.float32(c1 * qn) * xn + np.float32(c2 * s2 + np.float32(c3 * np.float32(np.float32(1 + qn) + xn))))
    return np.float32(np.float32(s2 - np.float32(2) * acc) - margin)


@pytest.mark.parametrize("case", ["dynamic_range", "cancellation", "near_duplicate", "d1024", "tiny"])
def test_margin_is_a_lower_bound_on_adversarial_vectors(case):
    rng = np.random.default_rng(hash(case) % 2 ** 32)
    d = 1024 if case == "d1024" else 256
    for _ in range(20):
        q = rng.standard_normal(d)
        if case == "dynamic_range":
            q *= np.exp(rng.uniform(-30, 30, d))
            x = q * (1 + rng.uniform(-1e-2, 1e-2, d))
        elif case == "cancellation":
            x = q + rng.standard_normal(d) * 1e-4          # distance tiny against the norms
        elif case == "near_duplicate":
            x = q.copy()
            x[rng.integers(d)] *= 1 + 2.0 ** -20
        elif case == "tiny":
            q *= 1e-19
            x = q + rng.standard_normal(d) * 1e-21
        else:
            x = rng.standard_normal(d) + 3 * q
        q, x = q.astype(np.float32), x.astype(np.float32)
        exact = fo.exact_distances(q, x[None, :])[0]
        assert np.isfinite(exact) and _margin_lower_bound(q, x) <= exact, case


def test_flat_capi_argument_errors_without_gpu():
    L = _lib.lib()
    h = ctypes.c_void_p()
    rows = ctypes.c_void_p(0x10000)
    assert L.pr_flat_create(None, 0, rows, 10, 64) == _lib.PR_EINVAL
    assert L.pr_flat_create(ctypes.byref(h), 0, None, 10, 64) == _lib.PR_EINVAL
    assert L.pr_flat_create(ctypes.byref(h), 0, rows, -1, 64) == _lib.PR_EINVAL
    assert L.pr_flat_create(ctypes.byref(h), 0, rows, 10, 96) == _lib.PR_EUNSUPPORTED
    assert b"multiple of 64" in L.pr_last_error()
    assert L.pr_flat_create(ctypes.byref(h), 0, rows, 10, 2048) == _lib.PR_EUNSUPPORTED
    assert L.pr_flat_create(ctypes.byref(h), 0, rows, 2 ** 31, 64) == _lib.PR_EUNSUPPORTED
    assert L.pr_flat_create(ctypes.byref(h), 0, ctypes.c_void_p(0x10004), 10, 64) == _lib.PR_EINVAL   # alignment
    assert L.pr_flat_aux_bytes(None) == 0 and L.pr_flat_workspace_bytes(None, 4, 5) == 0
    assert L.pr_flat_build_aux(None, None, 0, None) == _lib.PR_EINVAL
    assert L.pr_flat_search(None, 1, None, 5, None, None, None, 0, None) == _lib.PR_EINVAL
    t = _lib.FlatTuning()
    assert L.pr_flat_set_tuning(None, ctypes.byref(t)) == _lib.PR_EINVAL
    assert L.pr_flat_get_tuning(None, ctypes.byref(t)) == _lib.PR_EINVAL
    s = _lib.FlatStats()
    assert L.pr_flat_last_stats(None, None, 1, 5, ctypes.byref(s), None) == _lib.PR_EINVAL
    assert L.pr_flat_destroy(None) == _lib.PR_OK


def test_index_rejects_unsupported_d_without_gpu():
    for d in (0, 32, 100, 2048, 768.0):
        with pytest.raises(ValueError):
            dense.IndexFlatL2(d)
    with pytest.raises(ValueError, match="CUDA"):
        dense.IndexFlatL2(768, device="cpu")


def test_filter_kernel_sass():
    """The filter is a tcgen05 GEMM fed by TMA with its accumulator read from TMEM, and nothing spills."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = build.build()
    res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout.splitlines()
    hit = [res[i + 1] for i, l in enumerate(res) if "flat_filter_kernel" in l and i + 1 < len(res)]
    assert len(hit) == 1, hit
    m = re.search(r"REG:(\d+) STACK:(\d+)", hit[0])
    assert m and int(m.group(2)) == 0, hit[0]
    name = re.search(r"(_Z\w*flat_filter_kernel\w*)", next(l for l in res if "flat_filter_kernel" in l)).group(1)
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", name, lib], capture_output=True, text=True).stdout
    assert re.search(r"UTC[HQ]MMA", sass) and "UTMALDG" in sass and "LDTM" in sass
    assert "LDL" not in sass and "STL" not in sass


def test_against_a_file_written_by_faiss(tmp_path):
    """faiss writes the file, this package reads it; the search agrees with faiss's own modulo near-ties (the faiss
    part runs wherever faiss is installed; the GPU part where a device is present)."""
    faiss = pytest.importorskip("faiss")
    rng = np.random.default_rng(5)
    X = rng.standard_normal((5000, 768)).astype(np.float32)
    Q = (X[:16] + 0.05 * rng.standard_normal((16, 768))).astype(np.float32)
    ref = faiss.IndexFlatL2(768)
    ref.add(X)
    p = str(tmp_path / "faiss.index")
    faiss.write_index(ref, p)
    assert np.array_equal(np.asarray(dense.read_rows(p)), X)
    Df, If = ref.search(Q, 5)
    D, I = fo.search_canonical(Q, X, 5)
    assert fo.agree_modulo_near_ties(D, I, Df, If, atol=1e-6 * 2 * float(np.max(np.sum(X * X, 1))))
    # padding of k > ntotal: faiss's max-heap leaves (FLT_MAX, -1)
    small = faiss.IndexFlatL2(768)
    small.add(X[:3])
    Ds, Is = small.search(Q[:1], 5)
    assert list(Is[0, 3:]) == [-1, -1] and np.all(Ds[0, 3:] == fo.FLT_MAX)
    if torch.cuda.is_available():
        gi = dense.read_index(p)
        Dg, Ig = gi.search(Q, 5)
        assert np.array_equal(Dg, D) and np.array_equal(Ig, I)
