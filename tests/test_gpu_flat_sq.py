"""Exact flat search over fp16 rows on the GPU (pr_flat_create_fp16 through dense.IndexScalarQuantizer): search and
range_search equal, in lims, ids and value bits, an IndexFlatL2 / IndexFlatIP built from the fp16-decoded rows and the
canonical oracles over those rows, for both metrics, on every launch plan and sharding, on queries and rows across the
whole f32 / fp16 range, and on the cases where the filter needs its whole fp16 margin."""
import os
import socket

import numpy as np
import pytest
import torch

import flat_sq_margin as sqm
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from oracle import flat_range_oracle as fro
from probing_rag_b200 import (METRIC_INNER_PRODUCT, METRIC_L2, IndexFlatIP, IndexFlatL2, IndexScalarQuantizer,
                              ScalarQuantizer, ShardedIndexFlatIP, ShardedIndexFlatL2, _lib, dense, read_index,
                              sharding, synth, write_index)
from test_gpu_flat import SHAPES

pytestmark = pytest.mark.gpu

METRIC = {"l2": METRIC_L2, "ip": METRIC_INNER_PRODUCT}
FLAT = {"l2": IndexFlatL2, "ip": IndexFlatIP}
SHARDED = {"l2": ShardedIndexFlatL2, "ip": ShardedIndexFlatIP}
INF, NAN = float("inf"), float("nan")
METRICS = ["l2", "ip"]


def _bits(D):
    return np.ascontiguousarray(D.cpu().numpy() if isinstance(D, torch.Tensor) else D).view(np.uint32)


def _sq(X, metric, **plan):
    ix = IndexScalarQuantizer(X.shape[1], ScalarQuantizer.QT_fp16, METRIC[metric])
    ix.add(X)
    if plan:
        ix.set_tuning(**plan)
    return ix


def _oracle(Q, X, k, metric):
    return (fo.search_canonical_torch if metric == "l2" else fio.search_canonical_ip_torch)(Q, X, k)


def _check(ix, Q, k, metric, flat=True):
    """ix.search against the oracle over the decoded rows and (flat=True) an IndexFlat over them, same plan."""
    D, I = ix.search(Q, k)
    X = ix.rows()
    Dr, Ir = _oracle(Q, X, k, metric)
    assert np.array_equal(I.cpu().numpy(), Ir), f"{metric}: ids differ from the oracle"
    assert np.array_equal(_bits(D), _bits(Dr)), f"{metric}: value bits differ from the oracle"
    if flat:
        ref = FLAT[metric](X.shape[1])
        ref.add(X)
        ref.set_tuning(**{f: v for f, v in ix.get_tuning().items()})
        Df, If = ref.search(Q, k)
        assert torch.equal(I, If) and np.array_equal(_bits(D), _bits(Df)), f"{metric}: differs from IndexFlat"
    return D, I


def _same_range(a, b):
    (la, Da, Ia), (lb, Db, Ib) = [tuple(x.cpu().numpy() if isinstance(x, torch.Tensor) else x for x in r)
                                  for r in (a, b)]
    return (np.array_equal(la.astype(np.int64), lb.astype(np.int64)) and np.array_equal(Ia, Ib)
            and np.array_equal(Da.view(np.uint32), Db.view(np.uint32)))


def _check_range(ix, Q, radius, metric):
    got = ix.range_search(Q, radius)
    X = ix.rows()
    assert _same_range(got, fro.range_search_canonical_torch(Q, X, radius, metric)), f"{metric} {radius}: oracle"
    ref = FLAT[metric](X.shape[1])
    ref.add(X)
    assert _same_range(got, ref.range_search(Q, radius)), f"{metric} {radius}: IndexFlat"
    return got


# ---------------------------------------------------------------------------------------------- shapes and plans
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_parity(n, d, B, k, metric):
    rows = synth.dense_rows(n, d)
    ix = _sq(rows, metric)
    _check(ix, synth.dense_queries(rows, B), k, metric)
    assert ix.ntotal == n and ix.code_size == 2 * d and ix.codes().dtype == torch.float16


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("plan", [dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2),
                                  dict(cand_capacity=16), dict(first_chunk_rows=128, growth=2, cand_capacity=4)])
def test_launch_plans_and_overflow_fallback(plan, metric):
    rows = synth.dense_rows(100_003, 256)
    ix = _sq(rows, metric, **plan)
    _check(ix, synth.dense_queries(rows, 257), 100, metric)
    st = ix.last_stats()
    assert st["launches"] == 2 * st["chunks"] + 3
    if plan.get("first_chunk_rows") == 1 << 30:
        assert st["chunks"] == 1
    if "cand_capacity" in plan:
        assert st["fallback_queries"] > 0
    if plan.get("growth") == 2:
        assert st["chunks"] >= 8


@pytest.mark.parametrize("metric", METRICS)
def test_range_search_plans_and_second_pass(metric):
    rows = synth.dense_rows(60_001, 256)
    Q = synth.dense_queries(rows, 33)
    ix = _sq(rows, metric)
    D, _ = ix.search(Q, 50)
    radius = float(D[:, 49].max()) if metric == "l2" else float(D[:, 49].min())
    _check_range(ix, Q, radius, metric)
    ix._range_cap_forced = 3                                         # every query overflows the staging: pass two
    _check_range(ix, Q, radius, metric)
    ix._range_cap_forced = None
    for plan in (dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2, cand_capacity=4)):
        ix.set_tuning(**plan)
        _check_range(ix, Q, radius, metric)
        st = ix.last_stats()
        assert st["launches"] == 2 * st["chunks"] + 2, plan


# ---------------------------------------------------------------------------------------------- hazards
@pytest.mark.parametrize("metric", METRICS)
def test_queries_across_the_f32_range(metric):
    """Elements beyond fp16's 65504, a largest element near 1e-30 and below f32's normal range, 1e4 and 1e-6 in one
    vector, all-zero queries and queries holding NaN or +-inf: the per-query scale keeps every result exact."""
    g = torch.Generator(device="cuda").manual_seed(41)
    rows = synth.dense_rows(50_000, 256)
    base = rows[torch.randint(0, 50_000, (4,), generator=g, device="cuda")]
    mixed = torch.where(torch.rand((2, 256), generator=g, device="cuda") < 0.5, 1e4, 1e-6) * \
        torch.sign(torch.randn((2, 256), generator=g, device="cuda"))
    special = torch.zeros((4, 256), device="cuda")
    special[1, 5], special[2, 7], special[3, 9] = NAN, INF, -INF
    special[1:] += base[:3]
    Q = torch.cat([base * 1e5, base * 1e-30, base * 1e-40, mixed, torch.zeros((2, 256), device="cuda"), special])
    ix = _sq(rows, metric)
    for k in (1, 10, 128):
        _check(ix, Q, k, metric)


@pytest.mark.parametrize("metric", METRICS)
def test_rows_overflow_subnormal_and_nan(metric):
    """Rows that overflow fp16 at add (65504 stays finite, 65520 is inf), rows made mostly of fp16 subnormals and
    NaN rows, in the first chunk and in later ones."""
    g = torch.Generator(device="cuda").manual_seed(42)
    d = 128
    X = torch.randn((40_000, d), generator=g, device="cuda")
    sub = torch.rand((4, d), generator=g, device="cuda") * 2.0 ** -15                 # below 2^-14: subnormal
    for r, row in zip((10, 1000, 20_000, 39_999), sub):
        X[r] = row
        X[r, :4] = 2.0 ** -13                                                           # a few normal elements
    X[50, 0], X[25_000, 1] = 65504.0, 65519.99
    X[60, 2], X[30_000, 3] = 65520.0, -70000.0
    X[70, 4], X[35_000, 5] = NAN, NAN
    ix = _sq(X, metric)
    codes = ix.codes()
    assert float(codes[50, 0]) == 65504.0 and float(codes[25_000, 1]) == 65504.0
    assert float(codes[60, 2]) == INF and float(codes[30_000, 3]) == -INF
    Q = torch.cat([X[[10, 20_000, 39_999]].abs() + 2.0 ** -16, X[[0, 5, 50]], torch.ones((1, d), device="cuda")])
    for k in (1, 5, 128):
        _check(ix, Q, k, metric)
    _check_range(ix, Q[:3], 1e-6 if metric == "l2" else 1e-6, metric)


def test_fp16_rounding_bias_needs_the_whole_margin_ip():
    """q rounds down to fp16 by almost 2^-11 in every element (the rows are exact): the filter's dot product with the
    all-ones targets is short of the exact score by ~2^-11 |q||x|, all one-signed.  Filler rows of the first chunk
    set the bound between that dot product plus half the margin and the exact score: a filter with half of c1 drops
    the targets, which sit in later chunks."""
    d = 768
    c = np.float32(1 + 2.0 ** -11 - 2.0 ** -23)
    q = torch.full((1, d), float(c), device="cuda")
    X = torch.zeros((30_000, d), device="cuda")
    X[:4096] = 1.0
    X[:4096, : d // 4] = 1 - 2.0 ** -11                                  # fillers: score just below the targets'
    targets = [7_000, 12_345, 29_999]
    X[targets] = 1.0
    qn, xt, xf = q[0].cpu().numpy(), X[7_000].cpu().numpy(), X[0].cpu().numpy()
    theta = fio.exact_inner_products(qn, xf[None])[0]
    assert sqm.bound(qn, xt, "ip", c1_scale=0.5) < theta < fio.exact_inner_products(qn, xt[None])[0]
    for k in (1, 3, 5):
        D, I = _check(_sq(X, "ip"), q, k, "ip")
        assert I[0, :min(k, 3)].tolist() == targets[:k]


def test_fp16_rounding_bias_needs_the_whole_margin_l2():
    """The L2 form: the targets' bound from the fp16 dot product overestimates their distance by ~2 2^-11 |q||x|;
    fillers at a distance between the exact one and the bound with half of c1 set theta."""
    d = 768
    c = np.float32(1 + 2.0 ** -11 - 2.0 ** -23)
    q = torch.full((1, d), float(c), device="cuda")
    X = torch.zeros((30_000, d), device="cuda")
    X[:4096] = 1.0
    X[:4096, :8] = 1.125
    targets = [7_000, 12_345, 29_999]
    X[targets] = 1.0
    qn, xt, xf = q[0].cpu().numpy(), X[7_000].cpu().numpy(), X[0].cpu().numpy()
    theta = fo.exact_distances(qn, xf[None])[0]
    assert fo.exact_distances(qn, xt[None])[0] < theta < sqm.bound(qn, xt, "l2", c1_scale=0.5)
    for k in (1, 3, 5):
        D, I = _check(_sq(X, "l2"), q, k, "l2")
        assert I[0, :min(k, 3)].tolist() == targets[:k]


@pytest.mark.parametrize("metric", METRICS)
def test_subnormal_rows_need_the_x_sub_term(metric):
    """Target rows made only of fp16 subnormals.  A tensor core that flushed them would see a dot product of 0; the
    fillers put theta where only the whole |q| ||x_sub|| term keeps the targets (half of it would drop them, as the
    restated bound with flushing shows)."""
    d = 768
    s = 2.0 ** -15
    X = torch.zeros((30_000, d), device="cuda")
    targets = [7_000, 12_345, 29_999]
    if metric == "ip":
        q = torch.ones((1, d), device="cuda")
        X[:4096] = 0.75 * s
        X[targets] = s
    else:
        q = torch.full((1, d), s, device="cuda")
        X[:4096] = s + 2.0 ** -17
        X[targets] = s
    qn, xt, xf = q[0].cpu().numpy(), X[7_000].cpu().numpy(), X[0].cpu().numpy()
    if metric == "ip":
        theta = fio.exact_inner_products(qn, xf[None])[0]
        assert sqm.bound(qn, xt, "ip", csub_scale=0.5, flush=True) < theta
        assert sqm.bound(qn, xt, "ip", flush=True) >= fio.exact_inner_products(qn, xt[None])[0]
    else:
        theta = fo.exact_distances(qn, xf[None])[0]
        assert sqm.bound(qn, xt, "l2", csub_scale=0.5, flush=True) > theta
        assert sqm.bound(qn, xt, "l2", flush=True) <= fo.exact_distances(qn, xt[None])[0]
    for k in (1, 3, 5):
        D, I = _check(_sq(X, metric), q, k, metric)
        assert I[0, :min(k, 3)].tolist() == targets[:k]


def test_device_encoding_equals_numpy():
    """torch's device conversion (what add runs) equals numpy's astype(float16) bit for bit: ties at every exponent,
    65504 / 65519.99 / 65520, the largest subnormal, 2^-25 and its neighbours, and random values."""
    vals = []
    for e in range(-24, 16):
        ulp = 2.0 ** (max(e, -14) - 10)
        for m in (1.0, 1.5, 1.25):
            v = m * 2.0 ** e
            vals += [v + ulp / 2, v + 1.5 * ulp, v - ulp / 4, v + ulp / 2 * (1 + 2 ** -12)]
    vals += [65504.0, 65519.99, 65520.0, 1e6, (1023 / 1024) * 2.0 ** -14, 2.0 ** -25, 2.0 ** -25 * (1 + 2 ** -20),
             2.0 ** -26, 3 * 2.0 ** -26, 0.0, -0.0, INF, -INF, NAN]
    x = np.array(vals + [-v for v in vals], np.float32)
    x = np.concatenate([x, np.random.default_rng(43).standard_normal(100_000).astype(np.float32)
                        * np.exp2(np.random.default_rng(44).uniform(-30, 18, 100_000)).astype(np.float32)])
    dev = torch.from_numpy(x).cuda().to(torch.float16).cpu().numpy().view(np.uint16)
    want = x.astype(np.float16).view(np.uint16)
    nan = np.isnan(x)
    assert np.array_equal(dev[~nan], want[~nan]) and np.all((dev[nan] & 0x7C00) == 0x7C00)
    ix = IndexScalarQuantizer(64, ScalarQuantizer.QT_fp16)
    ix.add(x[:len(x) // 64 * 64].reshape(-1, 64))
    got = ix.codes().cpu().numpy().reshape(-1).view(np.uint16)
    n = len(got)
    assert np.array_equal(got[~nan[:n]], want[:n][~nan[:n]])


# ---------------------------------------------------------------------------------------------- surface
@pytest.mark.parametrize("metric", METRICS)
def test_interfaces_file_round_trip_and_memory(tmp_path, metric):
    rows = synth.dense_rows(5000, 768)
    Q = synth.dense_queries(rows, 9)
    ix = IndexScalarQuantizer(768, ScalarQuantizer.QT_fp16, METRIC[metric])
    ix.train(rows)
    ix.add(rows[:3000].cpu().numpy())
    ix.add(rows[3000:])
    assert ix.ntotal == 5000 and ix.is_trained and ix.metric_type == METRIC[metric] and ix.d == 768
    assert torch.equal(ix.codes(), rows.to(torch.float16))
    D, I = ix.search(Q.cpu().numpy(), 5)
    assert isinstance(D, np.ndarray) and D.dtype == np.float32 and I.dtype == np.int64
    Dt, It = ix.search(Q, 5)
    assert np.array_equal(Dt.cpu().numpy(), D) and np.array_equal(It.cpu().numpy(), I)
    p = str(tmp_path / "sq.index")
    write_index(ix, p)
    assert open(p, "rb").read(4) == b"IxSQ"
    again = read_index(p)
    assert isinstance(again, IndexScalarQuantizer) and again.metric_type == METRIC[metric]
    assert torch.equal(again.codes(), ix.codes())
    D2, I2 = again.search(Q.cpu().numpy(), 5)
    assert np.array_equal(D2, D) and np.array_equal(I2, I)
    L = _lib.lib()
    h = ix._handle()
    assert L.pr_flat_aux_bytes(h) <= 16 * 5000 + 1024          # norms only: no copy of the rows
    for B, k in ((1, 1), (9, 5), (300, 128)):                    # the f32 layout plus the per-query scales
        flat = IndexFlatL2(768)
        flat.add(rows)
        nq = (B + (B + 255) // 256 - 1) // ((B + 255) // 256)
        b_pad = (B + 255) // 256 * ((nq + 31) // 32 * 32)
        up = lambda v: (v + 255) // 256 * 256
        f32 = 0
        for size in (b_pad * 768 * 2, b_pad * 4, b_pad * 4, B * 4, B * 4, B * 8192 * 4, B * k * 8, 32):
            f32 = up(f32 + size)
        assert L.pr_flat_workspace_bytes(flat._handle(), B, k) == f32
        assert L.pr_flat_workspace_bytes(h, B, k) == f32 + up(b_pad * 4)
    ix.reset()
    assert ix.ntotal == 0
    D, I = ix.search(Q, 4)
    assert torch.all(I == -1)
    with pytest.raises(ValueError):
        ix.search(np.zeros((2, 768), np.float16), 5)
    with pytest.raises(ValueError):
        ix.add(np.zeros((2, 768), np.float64))


# ---------------------------------------------------------------------------------------------- shards
def _split(n, parts):
    r = [sharding.shard_range(n, i, parts) for i in range(parts)]
    return [r[0], (r[0][1], r[0][1])] + r[1:]


@pytest.mark.parametrize("metric", METRICS)
def test_simulated_shards_equal_single_index(metric):
    rows = synth.dense_rows(100_003, 256)
    Q = synth.dense_queries(rows, 64)
    single = _sq(rows, metric)
    for k in (5, 128):
        Ds, Is = _check(single, Q, k, metric, flat=False)
        for parts in (2, 3, 8):
            ranges = _split(rows.shape[0], parts)
            Dl, Il = zip(*[_sq(rows[lo:hi], metric).search(Q, k) for lo, hi in ranges])
            D, I = dense.merge_lists(torch.stack(Dl), torch.stack(Il), [lo for lo, _ in ranges], METRIC[metric])
            assert torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds)), f"{parts} shards differ"
    sx = SHARDED[metric](single, 0)
    D, I = sx.search(Q, 10)
    Ds, Is = single.search(Q, 10)
    assert torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds))
    assert _same_range(sx.range_search(Q, float(Ds[:, -1].max() if metric == "l2" else Ds[:, -1].min())),
                       single.range_search(Q, float(Ds[:, -1].max() if metric == "l2" else Ds[:, -1].min())))


N_FILE, D_FILE, B_FILE = 50_003, 768, 16


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir, metric):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        Q = np.load(os.path.join(out_dir, "q.npy"))
        for name in ("big", "small"):
            ix = read_index(os.path.join(out_dir, f"{name}.index"), device=dev, sharded=True)
            assert isinstance(ix, SHARDED[metric]) and isinstance(ix.shard, IndexScalarQuantizer)
            for k in (5, 128):
                res[f"{name}_D{k}"], res[f"{name}_I{k}"] = ix.search(Q, k)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("world", [2, 4])
def test_nccl_row_shards_equal_single_index(tmp_path, world, metric):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp
    rows = synth.dense_rows(N_FILE, D_FILE)
    Q = synth.dense_queries(rows, B_FILE)
    single, tiny = _sq(rows, metric), _sq(rows[:world - 1], metric)
    write_index(single, str(tmp_path / "big.index"))
    write_index(tiny, str(tmp_path / "small.index"))
    np.save(tmp_path / "q.npy", Q.cpu().numpy())
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), metric), nprocs=world, join=True)
    for name, ix in (("big", single), ("small", tiny)):
        for k in (5, 128):
            Ds, Is = _check(ix, Q, k, metric, flat=False)
            for r in range(world):
                got = np.load(tmp_path / f"r{r}.npz")
                assert np.array_equal(got[f"{name}_I{k}"], Is.cpu().numpy()), f"rank {r} {name} k={k}: ids differ"
                assert np.array_equal(_bits(got[f"{name}_D{k}"]), _bits(Ds)), f"rank {r} {name} k={k}: values"
