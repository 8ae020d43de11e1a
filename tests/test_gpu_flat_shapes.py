"""Exact flat search (csrc/flat.cu) at every shape its pipeline takes, and L2 on non-finite input: ids and distance or
score bit patterns against the oracle.

  - every d = 64..1024 (1 to 16 K-blocks of 64) against every query-tile width nq = 32..256 (ring depths 8, 6, 5, 4;
    UMMA N = 32..256), with several chunks and row tiles per call;
  - batches of 2 to 16 query blocks, rows at the tile and chunk edges, the empty batch;
  - L2 on NaN rows of either sign and other payloads, +-inf rows, rows that are finite in f32 but infinite in bf16 or
    in ||x||^2, NaN / inf / overflowing queries, an all-+inf top-k; in the first chunk and in later ones;
  - the L2 margin where every bf16 rounding errs one way (the L2 counterpart of the IP margin test), and far rows seen
    from a tiny query, where only the c2 (|q|^2 + |x|^2) term covers the f32 rounding of the bound.

The L2 contract on non-finite input: a NaN distance ranks after +inf, NaN distances among themselves by row id, and
comes back as the NaN 0x7FFFFFFF whatever NaN the input held.
"""
import functools

import numpy as np
import pytest
import torch

import flat_fast_oracle as ffo
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from probing_rag_b200 import IndexFlatIP, IndexFlatL2, ShardedIndexFlatL2, dense, sharding, synth

pytestmark = pytest.mark.gpu

FMAX = float(np.finfo(np.float32).max)
CLS = {"l2": IndexFlatL2, "ip": IndexFlatIP}


def _bits(D):
    return np.ascontiguousarray(D.cpu().numpy() if isinstance(D, torch.Tensor) else D).view(np.uint32)


def l2_canonical(Q, X, k):
    """The L2 contract restated: exact distances (fo.exact_distances_torch), every NaN as 0x7FFFFFFF, ranked by
    (bits, id) ascending; rows short of k (FLT_MAX, -1)."""
    B, n = Q.shape[0], X.shape[0]
    D = np.full((B, k), FMAX, dtype=np.float32)
    I = np.full((B, k), -1, dtype=np.int64)
    m = min(k, n)
    for b in range(B):
        bits = fo.exact_distances_torch(Q[b], X).view(torch.int32).to(torch.int64) & 0xFFFFFFFF
        key = torch.where((bits & 0x7FFFFFFF) > 0x7F800000, torch.full_like(bits, 0x7FFFFFFF), bits)
        s, o = torch.sort(key, stable=True)
        D[b, :m] = s[:m].to(torch.int32).view(torch.float32).cpu().numpy()
        I[b, :m] = o[:m].cpu().numpy()
    return D, I


def reference(Q, X, k, metric):
    return l2_canonical(Q, X, k) if metric == "l2" else fio.search_canonical_ip_torch(Q, X, k)


def check(index, Q, k, metric, ref=None):
    D, I = index.search(Q, k)
    Dr, Ir = reference(Q, index.rows(), k, metric) if ref is None else ref
    assert np.array_equal(I.cpu().numpy(), Ir), f"{metric}: ids differ"
    assert np.array_equal(_bits(D), _bits(Dr)), f"{metric}: distance / score bits differ"
    return D, I


def make(metric, X, **plan):
    index = CLS[metric](X.shape[1])
    index.add(X)
    if plan:
        index.set_tuning(**plan)
    return index


# ---------------------------------------------------------------------------------------------- d x nq grid
D_GRID = list(range(64, 1025, 64))                     # 1..16 K-blocks
B_GRID = [1, 33, 65, 97, 129, 161, 193, 225]           # nq = 32, 64, 96, ..., 256: one query block each
N_GRID = 3000                                          # chunks 128, 512, 2048, 312 under first_chunk_rows = 128


@functools.lru_cache(maxsize=2)
def _grid_index(metric, d):
    return make(metric, synth.dense_rows(N_GRID, d), first_chunk_rows=128)


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("d", D_GRID)
@pytest.mark.parametrize("B", B_GRID)
def test_every_k_block_count_and_query_tile_width(metric, d, B):
    index = _grid_index(metric, d)
    Q = synth.dense_queries(index.rows(), B)
    check(index, Q, 10, metric)
    if D_GRID.index(d) % len(B_GRID) == B_GRID.index(B):          # a diagonal of the grid, twice over d
        check(index, Q, 128, metric)
    assert index.last_stats()["chunks"] == 4


# ---------------------------------------------------------------------------------------------- batches, rows
@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_multi_block_batches(metric):
    """flat_layout cuts a batch of B > 256 into ceil(B / 256) equal query blocks of nq columns:
    B = 257 -> 2 x 160, 448 -> 2 x 224, 449 -> 2 x 256, 513 -> 3 x 192, 769 -> 4 x 224, 1025 -> 5 x 224,
    4096 -> 16 x 256 (the last block's tail columns are padding queries)."""
    rows = synth.dense_rows(20_000, 384)
    index = make(metric, rows, first_chunk_rows=128)
    Q = synth.dense_queries(rows, 4096)
    ref = ffo.search_fast(Q, rows, 128, metric)
    for B in (257, 448, 449, 513, 769, 1025, 4096):
        for k in (10, 128):
            D, I = index.search(Q[:B], k)
            assert np.array_equal(I.cpu().numpy(), ref[1][:B, :k]), f"B={B} k={k}"
            assert np.array_equal(_bits(D), _bits(ref[0][:B, :k])), f"B={B} k={k}"


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 2047, 2048, 2049, 10240, 10241])
def test_rows_at_tile_and_chunk_edges(metric, n):
    """Row counts around a 128-row tile and around the default plan's chunk ends (2048, then 2048 + 8192 = 10240)."""
    rows = synth.dense_rows(n, 256)
    index = make(metric, rows)
    Q = synth.dense_queries(rows, 65)
    for k in (1, 10, 128):
        check(index, Q, k, metric)


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_empty_batch(metric):
    rows = synth.dense_rows(1000, 128)
    index = make(metric, rows)
    for k in (1, 128):
        D, I = index.search(torch.empty((0, 128), device="cuda"), k)
        assert D.shape == (0, k) and I.shape == (0, k) and D.dtype == torch.float32 and I.dtype == torch.int64
        D, I = index.search(np.zeros((0, 128), np.float32), k)
        assert isinstance(D, np.ndarray) and D.shape == (0, k) and I.shape == (0, k)


def test_reference_equals_the_canonical_restatements_on_the_gpu():
    """The full-size reference pinned to the canonical lists at 100,003 rows x 1,000 queries, k = 1, 10, 128."""
    rows = synth.dense_rows(100_003, 768)
    Q = synth.dense_queries(rows, 1000)
    for metric in ("l2", "ip"):
        Dr, Ir = fo.search_canonical_torch(Q, rows, 128) if metric == "l2" else fio.search_canonical_ip_torch(Q, rows, 128)
        for k in (1, 10, 128):
            D, I = ffo.search_fast(Q, rows, k, metric, chunk_rows=1 << 15)
            assert np.array_equal(I, Ir[:, :k]) and np.array_equal(_bits(D), _bits(Dr[:, :k])), f"{metric} k={k}"


# ---------------------------------------------------------------------------------------------- L2, non-finite input
def _f32(bits):
    return torch.tensor([bits], dtype=torch.int64).to(torch.int32).view(torch.float32).item()


NANS = [float("nan"), -float("nan"), _f32(0x7FC0BEEF), _f32(0xFFC01234), _f32(0x7F800001), _f32(0xFFFFFFFF)]
BF16_INF = 3.3961e38                                   # finite in f32, rounds to inf in bf16


def _special_rows(d):
    """[18, d] rows: finite, NaN of six bit patterns (element 0), +-inf, bf16-infinite, ||x||^2 beyond FLT_MAX."""
    X = torch.zeros((18, d), device="cuda")
    X[0, 0] = 1.0
    for i, v in enumerate(NANS):
        X[1 + 2 * i, 0] = v                            # rows 1, 3, 5, 7, 9, 11
    X[2, 1] = float("inf")
    X[4, 2] = -float("inf")
    X[6, 3] = BF16_INF
    X[8] = 3e19                                        # ||x||^2 = d 9e38 > FLT_MAX, every element finite in bf16
    X[10, 0] = -1.0
    X[12] = 1e-3
    X[13, 5] = FMAX
    X[14, :] = -2.0
    X[15, 7] = 0.5
    X[16, 0] = float("inf")
    X[17, 0] = float("nan")
    return X


def _special_queries(d):
    g = torch.Generator(device="cuda").manual_seed(41)
    Q = torch.zeros((6, d), device="cuda")
    Q[0, 0] = 1.0
    Q[1] = torch.randn(d, generator=g, device="cuda")
    Q[2, 3] = float("nan")                             # every distance NaN
    Q[3, 1] = float("inf")
    Q[4] = 1e20                                        # ||q||^2 overflows f32
    Q[5] = -torch.rand(d, generator=g, device="cuda")
    return Q


def test_l2_special_values_in_the_first_chunk():
    """k above n: every row is ranked, so the order of +inf and NaN distances and the padding after them show."""
    d = 64
    X = _special_rows(d)
    index = make("l2", X)
    Q = _special_queries(d)
    D, I = check(index, Q, 24, "l2")
    bits = _bits(D)
    for b in range(Q.shape[0]):
        nan = np.isnan(D[b].cpu().numpy())
        inf = np.isinf(D[b].cpu().numpy())
        n_nan = int(nan.sum())
        assert np.all(bits[b][nan] == 0x7FFFFFFF)
        assert np.all(nan[18 - n_nan:18]) and not np.any(inf[18:]), "NaN after +inf, before the padding"
        assert np.all(np.diff(I[b, 18 - n_nan:18].cpu().numpy()) > 0), "NaN distances rank by id"
        assert torch.all(I[b, 18:] == -1) and torch.all(D[b, 18:] == FMAX)
    assert torch.all(I[2, :18] == torch.arange(18, device="cuda"))   # a NaN query: every distance NaN, id order


def test_l2_special_values_in_later_chunks():
    """The special rows scattered over a 12,000-row index whose other rows are NaN (of every bit pattern in turn), so
    that the ranked lists reach deep into the NaN distances: through the filter's bound after the first chunk, and
    with the one-chunk plan."""
    d = 64
    n = 12_000
    X = torch.zeros((n, d), device="cuda")
    X[:, 0] = torch.tensor(NANS, device="cuda").repeat(n // len(NANS))
    special = _special_rows(d)
    at = [5, 100, 200, 2047, 2048, 2500, 3000, 5000, 7000, 8000, 9000, 10000, 10239, 10240, 11000, 11500, 11998, 11999]
    X[at] = special
    Q = _special_queries(d)
    for plan in (dict(), dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2, cand_capacity=64)):
        index = make("l2", X, **plan)
        for k in (1, 16, 128):
            D, I = check(index, Q, k, "l2")
            assert np.all(_bits(D)[np.isnan(D.cpu().numpy())] == 0x7FFFFFFF)


def test_l2_simulated_shards_with_nan_distances():
    """The same index cut into row-range shards and merged: the merge ranks NaN distances as the search does."""
    d = 64
    X = torch.randn((5000, d), device="cuda")
    X[::3, 0] = torch.tensor(NANS, device="cuda").repeat(5000 // 3 // len(NANS) + 1)[:len(range(0, 5000, 3))]
    X[[10, 2600, 4999], 1] = float("inf")
    Q = _special_queries(d)
    Ds, Is = check(make("l2", X), Q, 128, "l2")
    for parts in (2, 3, 8):
        ranges = [sharding.shard_range(5000, i, parts) for i in range(parts)]
        lists = [make("l2", X[lo:hi]).search(Q, 128) for lo, hi in ranges]
        D, I = dense.merge_lists(torch.stack([a for a, _ in lists]), torch.stack([b for _, b in lists]),
                                 [lo for lo, _ in ranges])
        assert torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds)), f"{parts} shards"
    D, I = ShardedIndexFlatL2(make("l2", X), 0).search(Q, 128)
    assert torch.equal(I, Is) and np.array_equal(_bits(D), _bits(Ds))


def test_l2_infinite_k_th_distance_keeps_every_later_row_a_candidate():
    """Every distance is +inf (finite rows whose distance overflows f32).  theta is +inf after the first chunk, and a
    pair is a candidate iff !(bound > theta): every later row, whose bound is NaN or +-inf, still is."""
    q = torch.full((2, 64), -1e20, device="cuda")
    X = torch.full((10_000, 64), 1e20, device="cuda")
    index = make("l2", X)
    D, I = check(index, q, 5, "l2")
    assert torch.all(torch.isinf(D)) and torch.all(I == torch.arange(5, device="cuda"))
    assert index.last_stats()["candidates"] == 2 * 10_000


# ---------------------------------------------------------------------------------------------- L2 margin
def test_l2_bf16_rounding_bias_needs_the_whole_margin():
    """q and the target rows (copies of q) round down to bf16 by almost u in every element, so the bf16 dot product
    is short of q.x by ~2u |q||x| and the bound ||q||^2 + ||x||^2 - 2 dot exceeds the distance 0 by ~4u |q||x|.  The
    fillers of the first chunk put theta at ~0.012, between the distance and the bound with half of c1: a filter with
    half the margin drops the targets, which sit in later chunks."""
    d = 768
    c = np.float32(1 + 2.0 ** -8 - 2.0 ** -20)
    q = torch.full((1, d), float(c), device="cuda")
    X = torch.zeros((30_000, d), device="cuda")                              # distance ||q||^2, far above
    X[:4096] = 1.0
    X[:4096, : d // 4] = 1 + 2.0 ** -7                                      # fillers: exact in bf16
    targets = [7_000, 12_345, 29_999]
    X[targets] = float(c)
    for k in (1, 3, 5):
        D, I = check(make("l2", X), q, k, "l2")
        assert I[0, :min(k, 3)].tolist() == targets[:k] and float(D[0, 0]) == 0.0


def test_l2_far_rows_seen_from_a_tiny_query():
    """Rows of norm ~1000 around a query of norm ~0.001: every distance is ~10^6 and the rows differ by a few ulp of
    it, while c1 |q||x| is ~0.016, a quarter of an ulp.  Only the c2 (|q|^2 + |x|^2) term covers the f32 rounding of
    the stored norm and of the bound."""
    g = torch.Generator(device="cuda").manual_seed(42)
    d = 256
    u = torch.randn((40_000, d), generator=g, device="cuda")
    r = 1000.0 * (1 + torch.randint(-4, 5, (40_000, 1), generator=g, device="cuda") * 2.0 ** -24)
    X = u / u.norm(dim=1, keepdim=True) * r
    Q = torch.randn((8, d), generator=g, device="cuda") * 1e-3 / d ** 0.5
    for k in (1, 10, 128):
        check(make("l2", X), Q, k, "l2")
