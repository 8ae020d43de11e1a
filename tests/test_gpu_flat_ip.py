"""Exact flat inner-product search on the GPU (csrc/flat.cu through dense.IndexFlatIP, pr_flat_merge_metric and
ShardedIndexFlatIP): ids AND score bit patterns identical to the oracle's documented evaluation order and ranking
(NaN after -inf, (-FLT_MAX, -1) padding), whatever the launch plan, the chunking or the sharding."""
import os
import socket

import numpy as np
import pytest
import torch

from flat_ip_merge_oracle import merge_canonical_ip
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from probing_rag_b200 import (METRIC_INNER_PRODUCT, IndexFlatIP, IndexFlatL2, ShardedIndexFlatIP, dense, read_index,
                              sharding, synth, write_index)
from test_gpu_flat import SHAPES

pytestmark = pytest.mark.gpu

FMAX = float(np.finfo(np.float32).max)


def _bits(D):
    return np.ascontiguousarray(D.cpu().numpy() if isinstance(D, torch.Tensor) else D).view(np.uint32)


def _check(index, Q, k, X=None):
    X = index.rows() if X is None else X
    D, I = index.search(Q, k)
    Dr, Ir = fio.search_canonical_ip_torch(Q, X, k)
    assert np.array_equal(I.cpu().numpy(), Ir)
    assert np.array_equal(_bits(D), _bits(Dr))          # bit patterns: +0 vs -0 and the NaN's bits too
    return D, I


def _index(X):
    index = IndexFlatIP(X.shape[1])
    index.add(X)
    return index


@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_parity(n, d, B, k):
    rows = synth.dense_rows(n, d)
    index = _index(rows)
    _check(index, synth.dense_queries(rows, B), k)
    assert index.last_stats()["fallback_queries"] >= 0


def test_isotropic_rows_and_stats():
    rows = synth.dense_rows(100_003, 768, kind="isotropic")
    index = _index(rows)
    _check(index, synth.dense_queries(rows, 64), 10)
    st = index.last_stats()
    assert st["chunks"] >= 2 and st["launches"] == 2 * st["chunks"] + 3 and st["candidates"] >= 64 * 10


def test_duplicates_zero_rows_zero_query_and_padding():
    g = torch.Generator(device="cuda").manual_seed(31)
    base = torch.randn((300, 128), generator=g, device="cuda")
    X = torch.cat([base, base, torch.zeros((40, 128), device="cuda"), base[:5]])   # rows 3x, 2x; exact ties
    index = _index(X)
    Q = torch.cat([base[:20], torch.zeros((3, 128), device="cuda")])
    D, I = _check(index, Q, 64)
    assert torch.all(I[20:] == torch.arange(64, device="cuda")) and not np.any(_bits(D[20:]))   # all +0: id order
    small = _index(X[:3])
    D, I = _check(small, Q, 8)
    assert torch.all(I[:, 3:] == -1) and torch.all(D[:, 3:] == -FMAX)
    D, I = IndexFlatIP(128).search(Q, 4)
    assert torch.all(I == -1) and torch.all(D == -FMAX)


def test_negative_only_and_mixed_sign_scores():
    g = torch.Generator(device="cuda").manual_seed(32)
    q = torch.rand((8, 256), generator=g, device="cuda") + 0.1
    neg = -torch.rand((50_000, 256), generator=g, device="cuda")             # every score negative
    D, _ = _check(_index(neg), q, 100)
    assert torch.all(D < 0)
    mixed = torch.randn((50_000, 256), generator=g, device="cuda") * torch.rand((50_000, 1), generator=g, device="cuda")
    D, _ = _check(_index(mixed), torch.randn((8, 256), generator=g, device="cuda"), 128)
    assert torch.all(D[:, 0] > 0)


def test_rows_of_very_different_norms():
    """A large-norm row beats a near-duplicate of the query: the inner product is not a similarity of directions."""
    g = torch.Generator(device="cuda").manual_seed(33)
    d = 768
    u = torch.randn((60_000, d), generator=g, device="cuda")
    X = u / u.norm(dim=1, keepdim=True) * torch.logspace(-3, 3, 60_000, device="cuda")[torch.randperm(60_000, generator=g, device="cuda")][:, None]
    q = X[5000] / X[5000].norm()
    X[40_000] = q + 1e-3 * torch.randn(d, generator=g, device="cuda")       # near-duplicate, norm 1, score ~1
    D, I = _check(_index(X), torch.stack([q, -q]), 10)
    assert int(I[0, 0]) != 40_000 and float(X[int(I[0, 0])].norm()) > 10


def test_near_tie_sets():
    """Rows whose scores lie a few ulp apart around the k-th, with a large orthogonal part so that the margin (relative
    to |q||x|) is far wider than the spread: the bf16 filter cannot order them, only the margin keeps every one that
    belongs to the top-k."""
    g = torch.Generator(device="cuda").manual_seed(34)
    d = 768
    q = torch.randn(d, generator=g, device="cuda")
    qh = q / q.norm()
    o = torch.randn((5_000, d), generator=g, device="cuda")
    o = o - (o @ qh)[:, None] * qh[None, :]
    s = 10.0 * (1 + torch.randint(0, 8, (5_000, 1), generator=g, device="cuda") * 2.0 ** -22)
    X = s * qh[None, :] + o
    far = synth.dense_rows(50_000, d) - 3 * qh[None, :]
    X = torch.cat([far[:25_000], X, far[25_000:]])
    Q = torch.stack([q, q + 1e-7 * torch.randn(d, generator=g, device="cuda")])
    for k in (1, 10, 128):
        _check(_index(X), Q, k)


def test_bf16_rounding_bias_needs_the_whole_margin():
    """q and the target rows round down to bf16 by almost u in every element, so their bf16 dot product is short of the
    exact score by ~2u |q||x|, all one-signed.  Filler rows in the first chunk set the bound between the bf16 dot
    product plus half the margin and the exact score: a filter with half of c1ip drops the targets."""
    d = 768
    c = np.float32(1 + 2.0 ** -8 - 2.0 ** -20)
    q = torch.full((1, d), float(c), device="cuda")
    X = torch.zeros((30_000, d), device="cuda")                              # score 0, far below
    X[:4096] = 1.0
    X[:4096, : d // 4] = 1 + 2.0 ** -7                                      # fillers: d c (1 + 2^-9), exact in bf16
    targets = [7_000, 12_345, 29_999]
    X[targets] = float(c)                                                   # score ~ d c^2 > filler's
    for k in (1, 3, 5):
        D, I = _check(_index(X), q, k)
        assert I[0, :min(k, 3)].tolist() == targets[:k]


def test_special_values_nan_inf_and_padding():
    """NaN and +-inf rows, rows whose score is exactly -FLT_MAX / FLT_MAX / +-inf, in the first chunk (every row a
    candidate) and in later chunks (through the filter's bound)."""
    g = torch.Generator(device="cuda").manual_seed(35)
    d = 64
    q = torch.zeros((2, d), device="cuda")
    q[0, 0] = 1.0
    q[1] = torch.rand(d, generator=g, device="cuda") + 0.5                   # positive: an +inf element gives +inf
    vals = [1.0, float("inf"), -FMAX, 0.0, float("nan"), float("-inf"), FMAX, 1.0, -1.0, float("nan"), -FMAX,
            float("-inf"), 0.0]
    X = torch.zeros((len(vals), d), device="cuda")
    X[:, 0] = torch.tensor(vals)
    D, I = _check(_index(X), q[:1], 16)                                      # k > n: padding after the NaN rows
    assert I[0].tolist() == [1, 6, 0, 7, 3, 12, 8, 2, 10, 5, 11, 4, 9, -1, -1, -1]
    assert np.all(_bits(D[0, 11:13]) == 0xFFFFFFFF) and torch.all(D[0, 13:] == -FMAX)
    big = torch.randn((60_000, d), generator=g, device="cuda")
    for row, v in ((30_000, float("inf")), (31_000, float("nan")), (32_000, float("-inf")), (50_000, float("inf"))):
        big[row, 3] = v
    big[40_000] = 3e38                                                       # finite; q[1]'s score +inf in f32
    for k in (1, 5, 128):
        D, I = _check(_index(big), q, k)


def test_infinite_k_th_score_keeps_infinite_bounds_as_candidates():
    """Every score is +inf (finite rows whose q.x overflows f32).  The k-th score is +inf after the first chunk, and
    a pair is a candidate iff !(bound < theta): every later row, whose bound is +inf, still is."""
    q = torch.full((2, 64), 1e20, device="cuda")
    X = torch.full((10_000, 64), 1e20, device="cuda")
    index = _index(X)
    D, I = _check(index, q, 5)
    assert torch.all(torch.isinf(D)) and torch.all(I == torch.arange(5, device="cuda"))
    assert index.last_stats()["candidates"] == 2 * 10_000


@pytest.mark.parametrize("plan", [dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2),
                                  dict(cand_capacity=16), dict(first_chunk_rows=128, growth=2, cand_capacity=4)])
def test_launch_plans_and_overflow_fallback(plan):
    rows = synth.dense_rows(100_003, 256)
    index = _index(rows)
    Q = synth.dense_queries(rows, 257)
    index.set_tuning(**plan)
    _check(index, Q, 100)
    st = index.last_stats()
    if plan.get("first_chunk_rows") == 1 << 30:
        assert st["chunks"] == 1
    if "cand_capacity" in plan:
        assert st["fallback_queries"] > 0
    if plan.get("growth") == 2:
        assert st["chunks"] >= 8
    assert index.get_tuning()["first_chunk_rows"] == plan.get("first_chunk_rows", 2048)


def test_numpy_and_cuda_interfaces_and_file(tmp_path):
    rows = synth.dense_rows(5000, 768)
    Q = synth.dense_queries(rows, 9)
    index = IndexFlatIP(768)
    index.add(rows[:3000].cpu().numpy())
    index.add(rows[3000:])
    assert index.ntotal == 5000 and index.is_trained and index.metric_type == 0 and index.d == 768
    D, I = index.search(Q.cpu().numpy(), 5)
    assert isinstance(D, np.ndarray) and D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (9, 5)
    Dt, It = index.search(Q, 5)
    assert Dt.is_cuda and It.is_cuda and np.array_equal(Dt.cpu().numpy(), D) and np.array_equal(It.cpu().numpy(), I)
    Dr, Ir = fio.search_canonical_ip(Q.cpu().numpy(), rows.cpu().numpy(), 5)
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir)
    p = str(tmp_path / "flat_ip.index")
    write_index(index, p)
    assert open(p, "rb").read(4) == b"IxFI"
    again = read_index(p)
    assert isinstance(again, IndexFlatIP) and again.ntotal == 5000 and torch.equal(again.rows(), rows)
    D2, I2 = again.search(Q.cpu().numpy(), 5)
    assert np.array_equal(D2, D) and np.array_equal(I2, I)
    index.reset()
    assert index.ntotal == 0
    with pytest.raises(ValueError):
        index.search(np.zeros((2, 768), np.float64), 5)


def test_l2_and_ip_over_the_same_rows():
    rows = synth.dense_rows(100_003, 768)
    Q = synth.dense_queries(rows, 33)
    l2, ip = IndexFlatL2(768), IndexFlatIP(768)
    l2.add(rows)
    ip.add(rows)
    Dl, Il = l2.search(Q, 10)
    Dr, Ir = fo.search_canonical_torch(Q, rows, 10)
    assert np.array_equal(Il.cpu().numpy(), Ir) and np.array_equal(Dl.cpu().numpy(), Dr)
    _check(ip, Q, 10)
    Dl2, Il2 = l2.search(Q, 10)                                     # interleaved calls do not disturb each other
    assert torch.equal(Dl, Dl2) and torch.equal(Il, Il2)


# ---------------------------------------------------------------------------------------------- merge
def _ip_lists(rng, L, B, k, short="some", empty_list=False):
    """[L, B, k] ranked lists as pr_flat_search writes them for IP: scores from a small set (exact ties within and
    across lists, -FLT_MAX, -inf, NaN, +inf), distinct local ids, (ip_key, id) ascending, padded tails whose score is
    arbitrary."""
    values = np.array([3.0, 1.0, 1.0 + 2 ** -23, 0.0, -0.5, -FMAX, -np.inf, np.nan, np.inf], np.float32)
    sc = rng.choice(values, size=(L, B, k)).astype(np.float32)
    ids = np.argsort(rng.random((L, B, 3 * k)), axis=-1)[:, :, :k].astype(np.int64)
    m = rng.integers(0, k + 1, size=(L, B)) if short == "some" else \
        (rng.integers(0, k, size=(L, B)) if short == "all" else np.full((L, B), k))
    if empty_list:
        m[0] = 0
    pad = np.arange(k)[None, None, :] >= m[:, :, None]
    key = (fio.ip_key(sc).astype(np.uint64) << np.uint64(32)) | ids.astype(np.uint64)
    key[pad] = np.iinfo(np.uint64).max
    key.sort(axis=-1)
    pad = key == np.iinfo(np.uint64).max
    sc = fio.ip_score((key >> np.uint64(32)).astype(np.uint32))
    ids = (key & np.uint64(0xFFFFFFFF)).astype(np.int64)
    sc[pad] = rng.choice(np.array([-FMAX, 0.0, 2.0, np.nan], np.float32), size=int(pad.sum()))
    ids[pad] = -1
    return sc, ids


MERGE_CASES = [  # (lists, k, B, rows short of k, an all-padding list, bases)
    (1, 1, 1, "some", False, "big"), (1, 128, 64, "none", False, "big"), (2, 5, 65536, "some", False, "big"),
    (3, 100, 257, "all", False, "big"), (8, 128, 1000, "some", True, "big"), (32, 128, 300, "some", False, "big"),
    (32, 1, 513, "none", True, "big"), (16, 5, 4096, "all", False, "zero"), (5, 10, 2000, "some", True, "zero"),
]


@pytest.mark.parametrize("L, k, B, short, empty_list, bases", MERGE_CASES)
def test_ip_merge_against_oracle(L, k, B, short, empty_list, bases):
    rng = np.random.default_rng(L * 1000 + k * 7 + B + 1)
    Dl, Il = _ip_lists(rng, L, B, k, short, empty_list)
    base = [int(b) for b in np.sort(rng.integers(0, 2 ** 40, size=L)) + 2 ** 32] if bases == "big" else [0] * L
    D, I = dense.merge_lists(torch.from_numpy(Dl).cuda(), torch.from_numpy(Il).cuda(), base, METRIC_INNER_PRODUCT)
    Dw, Iw = merge_canonical_ip(Dl, Il, base, k)
    assert np.array_equal(I.cpu().numpy(), Iw)
    assert np.array_equal(_bits(D), _bits(Dw))


# ---------------------------------------------------------------------------------------------- simulated shards
def _split(n, parts):
    r = [sharding.shard_range(n, i, parts) for i in range(parts)]
    return [r[0], (r[0][1], r[0][1])] + r[1:]


def _check_shards(rows, Q, k):
    single = _index(rows)
    Ds, Is = single.search(Q, k)
    for parts in (2, 3, 8):
        ranges = _split(rows.shape[0], parts)
        Dl, Il = [], []
        for lo, hi in ranges:
            d, i = _index(rows[lo:hi]).search(Q, k)
            Dl.append(d)
            Il.append(i)
        D, I = dense.merge_lists(torch.stack(Dl), torch.stack(Il), [lo for lo, _ in ranges], METRIC_INNER_PRODUCT)
        assert torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds)), f"{parts} shards differ from the single index"
    sx = ShardedIndexFlatIP(single, 0)
    D, I = sx.search(Q, k)
    assert sx.ntotal == rows.shape[0] and torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds))
    with pytest.raises(ValueError, match="metric"):
        dense.ShardedIndexFlatL2(single, 0)
    return Ds, Is


@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_simulated_shards_equal_single_index(n, d, B, k):
    rows = synth.dense_rows(n, d)
    _check_shards(rows, synth.dense_queries(rows, B), k)


def test_simulated_shards_ties_and_special_values():
    g = torch.Generator(device="cuda").manual_seed(36)
    base = torch.randn((300, 128), generator=g, device="cuda")
    X = torch.cat([base, base, torch.zeros((40, 128), device="cuda"), base[:5]])   # exact ties across every cut
    X[7, 0], X[400, 1], X[500, 2] = float("nan"), float("-inf"), float("inf")
    Q = torch.cat([base[:20], torch.zeros((3, 128), device="cuda")])
    D, I = _check_shards(X, Q, 128)
    Dr, Ir = fio.search_canonical_ip_torch(Q, X, 128)
    assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(_bits(D), _bits(Dr))


# ---------------------------------------------------------------------------------------------- NCCL, one process per GPU
N_FILE, D_FILE, B_FILE = 50_003, 768, 16


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
        Q = np.load(os.path.join(out_dir, "q.npy"))
        for name in ("big", "small"):
            ix = read_index(os.path.join(out_dir, f"{name}.index"), device=dev, sharded=True)
            lo, hi = sharding.shard_range(ix.ntotal, rank, world)
            assert isinstance(ix, ShardedIndexFlatIP) and ix.shard.ntotal == hi - lo and ix.row_base == lo
            for k in (5, 128):
                Dn, In = ix.search(Q, k)
                Dt, It = ix.search(torch.from_numpy(Q).to(dev), k)
                assert isinstance(Dn, np.ndarray) and Dt.device == dev
                assert np.array_equal(Dt.cpu().numpy(), Dn) and np.array_equal(It.cpu().numpy(), In)
                res[f"{name}_D{k}"], res[f"{name}_I{k}"] = Dn, In
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 4])
def test_nccl_row_shards_equal_single_index_and_oracle(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp
    rows = synth.dense_rows(N_FILE, D_FILE)
    Q = synth.dense_queries(rows, B_FILE)
    single = _index(rows)
    write_index(single, str(tmp_path / "big.index"))
    tiny = _index(rows[:world - 1])                          # more ranks than rows: the last rank holds none
    write_index(tiny, str(tmp_path / "small.index"))
    np.save(tmp_path / "q.npy", Q.cpu().numpy())
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for name, ix in (("big", single), ("small", tiny)):
        for k in (5, 128):
            Ds, Is = ix.search(Q, k)
            Dr, Ir = fio.search_canonical_ip_torch(Q, ix.rows(), k)
            assert np.array_equal(Is.cpu().numpy(), Ir) and np.array_equal(_bits(Ds), _bits(Dr))
            for r in range(world):
                got = np.load(tmp_path / f"r{r}.npz")
                assert np.array_equal(got[f"{name}_I{k}"], Ir), f"rank {r} {name} k={k}: ids differ"
                assert np.array_equal(_bits(got[f"{name}_D{k}"]), _bits(Dr)), f"rank {r} {name} k={k}: scores differ"
