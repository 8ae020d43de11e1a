"""IndexScalarQuantizer(QT_fp16) without a GPU: the 'IxSQ' file layout, round trip and read_index dispatch, the errors
of bad qtypes, metrics and sizes, C-ABI argument errors of pr_flat_create_fp16, the fp16 encoding torch performs,
the restated fp16 margin against emulated fp16 products, the fp16 kernels' SASS, and files of real faiss."""
import ctypes
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest
import torch

import flat_sq_margin as sqm
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from probing_rag_b200 import _lib, build, dense

IP, L2 = dense.METRIC_INNER_PRODUCT, dense.METRIC_L2
QT = dense.ScalarQuantizer.QT_fp16


# ---------------------------------------------------------------------------------------------- files
def _codes(n=37, d=64, seed=51):
    return np.random.default_rng(seed).standard_normal((n, d)).astype(np.float16)


@pytest.mark.parametrize("metric", [L2, IP])
def test_sq_file_layout_and_round_trip(tmp_path, metric):
    C = _codes()
    p = str(tmp_path / "sq.index")
    dense.write_codes(p, C, 64, metric)
    raw = open(p, "rb").read()
    assert raw[:4] == b"IxSQ" and len(raw) == 81 + C.nbytes
    assert struct.unpack_from("<iqqqBi", raw, 4) == (64, 37, 1 << 20, 1 << 20, 1, metric)
    assert struct.unpack_from("<iifQQQQ", raw, 37) == (QT, 0, 0.0, 64, 128, 0, C.nbytes)
    assert raw[81:] == C.astype("<f2").tobytes()
    mm, m = dense.read_codes(p)
    assert m == metric and isinstance(mm, np.memmap) and np.array_equal(np.asarray(mm), C)
    dense.write_codes(p, C[:0], 64, metric)
    assert dense.read_codes(p)[0].shape == (0, 64)
    with pytest.raises(ValueError):
        dense.write_codes(p, C, 64, 2)
    with pytest.raises(ValueError, match="float16"):
        dense.write_codes(p, C.astype(np.float32), 64, metric)


@pytest.mark.parametrize("field, value, msg", [
    (37, struct.pack("<i", 0), "qtype 0"), (37, struct.pack("<i", 7), "qtype 7"), (33, struct.pack("<i", 2), "metric"),
    (49, struct.pack("<Q", 65), "ScalarQuantizer d"), (57, struct.pack("<Q", 64), "code_size"),
    (73, struct.pack("<Q", 10), "code bytes"), (4, struct.pack("<i", 96), "d = 96")])
def test_bad_qtype_metric_and_sizes_are_rejected(tmp_path, field, value, msg):
    p = str(tmp_path / "sq.index")
    dense.write_codes(p, _codes(), 64)
    raw = bytearray(open(p, "rb").read())
    raw[field:field + len(value)] = value
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=msg):
        dense.read_codes(p)


def test_truncated_files_are_rejected(tmp_path):
    p = str(tmp_path / "sq.index")
    dense.write_codes(p, _codes(), 64)
    raw = open(p, "rb").read()
    for cut in (10, 80, len(raw) - 1):
        open(p, "wb").write(raw[:cut])
        with pytest.raises(ValueError, match="truncated"):
            dense.read_codes(p)


def test_index_constructor_errors_without_gpu():
    for qtype in (0, 1, 2, 3, 5, 6, 7, 8, 99):
        with pytest.raises(ValueError, match="qtype"):
            dense.IndexScalarQuantizer(64, qtype)
    for metric in (2, -1, 23):
        with pytest.raises(ValueError, match="metric"):
            dense.IndexScalarQuantizer(64, QT, metric)
    with pytest.raises(ValueError, match="multiple of 64"):
        dense.IndexScalarQuantizer(96, QT)
    with pytest.raises(ValueError, match="CUDA"):
        dense.IndexScalarQuantizer(64, QT, device="cpu")
    assert dense.ScalarQuantizer.QT_fp16 == 4 and dense.ScalarQuantizer.QT_bf16 == 7


class _FakeIndex:
    """Stands in for the index classes in read_index (no device needed)."""

    def __init__(self, d, *args):
        self.d, self.device, self.rows, self.args = d, torch.device("cpu"), None, args
        self.metric_type = args[1] if len(args) > 1 else None

    def _set_rows(self, rows):
        self.rows = rows
        self.ntotal = rows.shape[0]


def test_read_index_dispatches_on_the_fourcc(tmp_path, monkeypatch):
    fakes = {name: type(name, (_FakeIndex,), {}) for name in ("IndexFlatL2", "IndexFlatIP", "IndexScalarQuantizer")}
    for name, cls in fakes.items():
        monkeypatch.setattr(dense, name, cls)
    C = _codes(10)
    for metric in (L2, IP):
        p = str(tmp_path / f"sq{metric}.index")
        dense.write_codes(p, C, 64, metric)
        ix = dense.read_index(p)
        assert type(ix) is fakes["IndexScalarQuantizer"] and ix.args[:2] == (QT, metric)
        assert ix.rows.dtype == torch.float16 and torch.equal(ix.rows, torch.from_numpy(C))
        sx = dense.read_index(p, sharded=True)                       # one process: the whole file, row_base 0
        assert type(sx) is (dense.ShardedIndexFlatL2 if metric == L2 else dense.ShardedIndexFlatIP)
        assert sx.ntotal == 10 and sx.row_base == 0 and torch.equal(sx.shard.rows, torch.from_numpy(C))
    X = C.astype(np.float32)
    p = str(tmp_path / "flat.index")
    dense.write_rows(p, X, 64)
    assert type(dense.read_index(p)) is fakes["IndexFlatL2"]
    raw = bytearray(open(p, "rb").read())
    raw[0:4] = b"IxHF"
    open(p, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="IxF2.*IxFI.*IxSQ"):
        dense.read_index(p)


# ---------------------------------------------------------------------------------------------- C ABI
def test_create_fp16_capi_argument_errors_without_gpu():
    L = _lib.lib()
    h = ctypes.c_void_p()
    codes = ctypes.c_void_p(0x10000)
    assert L.pr_flat_create_fp16(None, 0, codes, 10, 64, L2) == _lib.PR_EINVAL
    assert L.pr_flat_create_fp16(ctypes.byref(h), 0, None, 10, 64, L2) == _lib.PR_EINVAL
    assert L.pr_flat_create_fp16(ctypes.byref(h), 0, codes, -1, 64, IP) == _lib.PR_EINVAL
    for metric in (2, -1, 23):
        assert L.pr_flat_create_fp16(ctypes.byref(h), 0, codes, 10, 64, metric) == _lib.PR_EUNSUPPORTED
        assert b"metric" in L.pr_last_error() and not h.value
    for d in (96, 2048, 0):
        assert L.pr_flat_create_fp16(ctypes.byref(h), 0, codes, 10, d, L2) == _lib.PR_EUNSUPPORTED
        assert b"multiple of 64" in L.pr_last_error()
    assert L.pr_flat_create_fp16(ctypes.byref(h), 0, codes, 2 ** 31, 64, IP) == _lib.PR_EUNSUPPORTED
    assert L.pr_flat_create_fp16(ctypes.byref(h), 0, ctypes.c_void_p(0x10008), 10, 64, L2) == _lib.PR_EINVAL
    assert b"16-byte" in L.pr_last_error()


# ---------------------------------------------------------------------------------------------- encoding
def _encoding_pins():
    vals = []
    for e in range(-24, 16):                           # a tie, both neighbours of one, at every exponent
        ulp = 2.0 ** (max(e, -14) - 10)
        for m in (1.0, 1.5, 1.0 + 2 ** -10):
            v = m * 2.0 ** e
            vals += [v + ulp / 2, v + 1.5 * ulp, v + ulp / 2 * (1 - 2 ** -12), v + ulp / 2 * (1 + 2 ** -12)]
    vals += [65504.0, 65519.99, 65520.0, 1e6, (1023 / 1024) * 2.0 ** -14, 2.0 ** -25, 2.0 ** -25 * (1 + 2 ** -20),
             2.0 ** -26, 3 * 2.0 ** -26, 0.0, float("inf")]
    return np.array(vals + [-v for v in vals], np.float32)


@np.errstate(over="ignore")
def test_torch_cpu_encoding_equals_numpy_and_pins():
    x = _encoding_pins()
    want = x.astype(np.float16)
    assert np.array_equal(torch.from_numpy(x).to(torch.float16).numpy().view(np.uint16), want.view(np.uint16))
    h = lambda v: int(np.array([v], np.float32).astype(np.float16).view(np.uint16)[0])
    assert h(65504.0) == 0x7BFF and h(65519.99) == 0x7BFF and h(65520.0) == 0x7C00 and h(-65520.0) == 0xFC00
    assert h(2.0 ** -25) == 0 and h(2.0 ** -25 * (1 + 2 ** -20)) == 1 and h(3 * 2.0 ** -26) == 1 and h(2.0 ** -24) == 1
    assert h((1023 / 1024) * 2.0 ** -14) == 0x03FF and h(1 + 2 ** -11) == 0x3C00 and h(1 + 3 * 2 ** -11) == 0x3C02
    assert np.isnan(np.array([np.nan], np.float32).astype(np.float16)[0])


# ---------------------------------------------------------------------------------------------- margin
def _fp16_biased(d, rng):
    """A query whose every element rounds down to fp16 by almost 2^-11 after scaling, over exact fp16 rows: the
    filter's dot product is short of q.x by almost 2^-11 |q||x|, all of it one-signed."""
    c = np.float32(1 + 2.0 ** -11 - 2.0 ** -23)
    s = rng.choice([-1.0, 1.0], d) if rng.random() < 0.5 else np.ones(d)
    return (c * s).astype(np.float32), s.astype(np.float32)


CASES = ["dynamic_range", "cancellation", "near_duplicate", "d1024", "tiny", "huge", "mixed_query", "negative",
         "subnormal_rows", "fp16_biased"]


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("case", CASES)
def test_fp16_margin_is_a_bound_on_adversarial_vectors(case, metric):
    rng = np.random.default_rng(sum(map(ord, case + metric)))
    d = 1024 if case == "d1024" else 768 if case == "fp16_biased" else 256
    for _ in range(10):
        q = rng.standard_normal(d)
        if case == "dynamic_range":
            q *= np.exp(rng.uniform(-8, 8, d))
            x = q * (1 + rng.uniform(-1e-2, 1e-2, d))
        elif case == "cancellation":
            r = rng.standard_normal(d)
            x = r - (r @ q) / (q @ q) * q + rng.standard_normal(d) * 1e-3
        elif case == "near_duplicate":
            x = q.copy()
        elif case == "tiny":
            q *= 1e-30
            x = rng.standard_normal(d)
        elif case == "huge":
            q *= 1e8
            x = rng.standard_normal(d) + q * 1e-8
        elif case == "mixed_query":
            q = np.where(rng.random(d) < 0.5, 1e4, 1e-6) * np.sign(q)
            x = rng.standard_normal(d)
        elif case == "negative":
            x = -q * rng.uniform(0.5, 2, d)
        elif case == "subnormal_rows":
            x = np.abs(rng.standard_normal(d)) * 2.0 ** -16
            x[:8] = 1e-3
            q = np.abs(q)
        elif case == "fp16_biased":
            q, x = _fp16_biased(d, rng)
        else:
            x = rng.standard_normal(d) + 3 * q
        q = q.astype(np.float32)
        x = x.astype(np.float32).astype(np.float16).astype(np.float32)     # the decoded row
        for flush in (False, True):
            b = sqm.bound(q, x, metric, flush=flush)
            if metric == "l2":
                exact = fo.exact_distances(q, x[None, :])[0]
                assert np.isfinite(exact) and b <= exact, (case, flush)
            else:
                exact = fio.exact_inner_products(q, x[None, :])[0]
                assert np.isfinite(exact) and b >= exact, (case, flush)
        if case == "fp16_biased" and np.all(x > 0):            # half of c1 would not be a bound
            half = sqm.bound(q, x, metric, c1_scale=0.5)
            assert (half > exact) if metric == "l2" else (half < exact)
        if case == "subnormal_rows" and metric == "ip":        # nor half of csub, were subnormals flushed (the L2
            half = sqm.bound(q, x, metric, csub_scale=0.5, flush=True)   # case: tests/test_gpu_flat_sq.py)
            assert half < exact


def test_margin_constants():
    c1, cs = sqm.constants(768, "l2")
    c1ip, csip = sqm.constants(768, "ip")
    assert 0.00134 < c1 < 0.00135 and 0.000672 < c1ip < 0.000673 and 2.0 < cs < 2.005 and 1.0 < csip < 1.0025


# ---------------------------------------------------------------------------------------------- SASS
def test_fp16_kernels_sass():
    """The fp16 filters are the tcgen05 GEMM fed by TMA with the accumulator read from TMEM; the refines evaluate in
    f64 without contraction; nothing spills and no kernel has a stack."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = build.build()
    res = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout.splitlines()
    names = {}
    for i, line in enumerate(res):
        m = re.search(r"(_Z\w*(flat_fp16_\w*kernel)\w*)", line)
        if m and i + 1 < len(res):
            names[m.group(2)] = m.group(1)
            assert re.search(r"STACK:0\b", res[i + 1]), (line, res[i + 1])
    assert set(names) == {"flat_fp16_prep_kernel", "flat_fp16_query_prep_kernel", "flat_fp16_filter_kernel",
                          "flat_fp16_ip_filter_kernel", "flat_fp16_refine_kernel", "flat_fp16_ip_refine_kernel",
                          "flat_fp16_range_refine_kernel", "flat_fp16_ip_range_refine_kernel"}, names
    for short, name in names.items():
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", name, lib], capture_output=True, text=True).stdout
        assert "LDL" not in sass and "STL" not in sass, short
        if "filter" in short:
            assert re.search(r"UTC[HQ]MMA", sass) and "UTMALDG" in sass and "LDTM" in sass, short
        if "refine" in short:
            assert "DFMA" not in sass and "DADD" in sass and "DMUL" in sass, short


# ---------------------------------------------------------------------------------------------- real faiss
@pytest.mark.parametrize("metric", [L2, IP])
def test_against_files_of_faiss(tmp_path, metric):
    """faiss writes an IndexScalarQuantizer(QT_fp16) file that this package reads, and reads the one it writes; the
    exact search over the decoded rows agrees with faiss's own modulo near-ties."""
    faiss = pytest.importorskip("faiss")
    rng = np.random.default_rng(52)
    X = rng.standard_normal((3000, 128)).astype(np.float32)
    Q = (X[:8] + 0.05 * rng.standard_normal((8, 128))).astype(np.float32)
    ref = faiss.IndexScalarQuantizer(128, faiss.ScalarQuantizer.QT_fp16, metric)
    ref.add(X)
    p = str(tmp_path / "faiss_sq.index")
    faiss.write_index(ref, p)
    assert open(p, "rb").read(4) == b"IxSQ"
    codes, m = dense.read_codes(p)
    assert m == metric and np.array_equal(np.asarray(codes), X.astype(np.float16))
    q2 = str(tmp_path / "ours_sq.index")
    dense.write_codes(q2, X.astype(np.float16), 128, metric)
    back = faiss.read_index(q2)
    assert back.ntotal == 3000 and back.metric_type == metric
    assert np.array_equal(back.sa_decode(back.sa_encode(X[:4])), ref.sa_decode(ref.sa_encode(X[:4])))
    Df, If = ref.search(Q, 5)
    Xd = X.astype(np.float16).astype(np.float32)
    D, I = (fo.search_canonical if metric == L2 else fio.search_canonical_ip)(Q, Xd, 5)
    assert fo.agree_modulo_near_ties(D, I, Df, If, atol=1e-3)
    Db, Ib = back.search(Q, 5)
    assert np.array_equal(Ib, If)
    if torch.cuda.is_available():
        gi = dense.read_index(p)
        Dg, Ig = gi.search(Q, 5)
        assert np.array_equal(Dg, D) and np.array_equal(Ig, I)
