"""Exact flat L2 search on the GPU (csrc/flat.cu through dense.IndexFlatL2): ids AND distances bit-identical to the
oracle's documented evaluation order, whatever the launch plan."""
import numpy as np
import pytest
import torch

from oracle import flat_oracle as fo
from probing_rag_b200 import IndexFlatL2, read_index, synth, write_index

pytestmark = pytest.mark.gpu


def _check(index, Q, k, X=None):
    X = index.rows() if X is None else X
    D, I = index.search(Q, k)
    Dr, Ir = fo.search_canonical_torch(Q, X, k)
    assert np.array_equal(I.cpu().numpy(), Ir)
    assert np.array_equal(D.cpu().numpy(), Dr)
    return D, I


# (N, d, B, k): every size of the issue's grid appears at least once
SHAPES = [(1, 64, 1, 1), (1, 64, 7, 5), (127, 768, 7, 10), (128, 768, 1, 128), (129, 1024, 257, 100),
          (129, 64, 1000, 128), (100_003, 768, 256, 10), (100_003, 64, 1000, 5), (100_003, 1024, 1, 128),
          (100_003, 768, 257, 100)]


@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_parity(n, d, B, k):
    rows = synth.dense_rows(n, d)
    index = IndexFlatL2(d)
    index.add(rows)
    Q = synth.dense_queries(rows, B)
    _check(index, Q, k)
    assert index.last_stats()["fallback_queries"] >= 0


def test_isotropic_rows_and_stats():
    rows = synth.dense_rows(100_003, 768, kind="isotropic")
    index = IndexFlatL2(768)
    index.add(rows)
    Q = synth.dense_queries(rows, 64)
    _check(index, Q, 10)
    st = index.last_stats()
    assert st["chunks"] >= 2 and st["launches"] == 2 * st["chunks"] + 3 and st["candidates"] >= 64 * 10


def test_duplicates_ties_zero_rows_and_padding():
    g = torch.Generator(device="cuda").manual_seed(5)
    base = torch.randn((300, 128), generator=g, device="cuda")
    X = torch.cat([base, base, torch.zeros((40, 128), device="cuda"), base[:5]])   # rows 3x, 2x; exact ties
    index = IndexFlatL2(128)
    index.add(X)
    Q = torch.cat([base[:20], torch.zeros((3, 128), device="cuda")])
    D, I = _check(index, Q, 64)
    assert torch.all(D[:20, 0] == 0) and torch.all(I[:5, :3] == torch.stack([torch.arange(5), torch.arange(300, 305),
                                                                               torch.arange(640, 645)], 1).cuda())
    small = IndexFlatL2(128)
    small.add(X[:3])
    D, I = _check(small, Q, 8)
    assert torch.all(I[:, 3:] == -1) and torch.all(D[:, 3:] == torch.finfo(torch.float32).max)
    empty = IndexFlatL2(128)
    D, I = empty.search(Q, 4)
    assert torch.all(I == -1) and torch.all(D == torch.finfo(torch.float32).max)
    assert empty.last_stats()["launches"] == 2                    # init and output
    lims, D, I = empty.range_search(Q, 1.0)
    assert torch.all(lims == 0) and D.numel() == 0 and empty.last_stats()["launches"] == 1    # init


def test_near_tie_shells():
    """Rows on shells around the query whose distances lie a few ulp apart: the bf16 filter cannot tell them apart,
    only the margin keeps every one that belongs to the top-k."""
    g = torch.Generator(device="cuda").manual_seed(6)
    d = 768
    q = torch.randn(d, generator=g, device="cuda")
    u = torch.randn((20_000, d), generator=g, device="cuda")
    u = u / u.norm(dim=1, keepdim=True)
    r = 1.0 + torch.randint(0, 8, (20_000, 1), generator=g, device="cuda") * 2.0 ** -22
    X = q[None, :] + u * r
    far = synth.dense_rows(50_000, d) * 10
    X = torch.cat([far[:25_000], X, far[25_000:]])
    index = IndexFlatL2(d)
    index.add(X)
    Q = torch.stack([q, q + 1e-7 * torch.randn(d, generator=g, device="cuda")])
    for k in (1, 10, 128):
        _check(index, Q, k)


@pytest.mark.parametrize("plan", [dict(first_chunk_rows=1 << 30), dict(first_chunk_rows=128, growth=2),
                                  dict(cand_capacity=16), dict(first_chunk_rows=128, growth=2, cand_capacity=4)])
def test_launch_plans_and_overflow_fallback(plan):
    rows = synth.dense_rows(100_003, 256)
    index = IndexFlatL2(256)
    index.add(rows)
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


def test_numpy_and_cuda_interfaces(tmp_path):
    rows = synth.dense_rows(5000, 768)
    Q = synth.dense_queries(rows, 9)
    index = IndexFlatL2(768)
    index.add(rows[:3000].cpu().numpy())
    index.add(rows[3000:])
    assert index.ntotal == 5000 and index.is_trained and index.metric_type == 1 and index.d == 768
    D, I = index.search(Q.cpu().numpy(), 5)
    assert isinstance(D, np.ndarray) and D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (9, 5)
    Dt, It = index.search(Q, 5)
    assert Dt.is_cuda and It.is_cuda and np.array_equal(Dt.cpu().numpy(), D) and np.array_equal(It.cpu().numpy(), I)
    Dr, Ir = fo.search_canonical(Q.cpu().numpy(), rows.cpu().numpy(), 5)
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir)
    p = str(tmp_path / "flat.index")
    write_index(index, p)
    again = read_index(p)
    assert again.ntotal == 5000 and torch.equal(again.rows(), rows)
    D2, I2 = again.search(Q.cpu().numpy(), 5)
    assert np.array_equal(D2, D) and np.array_equal(I2, I)
    index.reset()
    assert index.ntotal == 0


def test_value_errors():
    index = IndexFlatL2(64)
    index.add(np.zeros((10, 64), np.float32))
    q = np.zeros((2, 64), np.float32)
    for bad_k in (0, 129, -1, 2.0):
        with pytest.raises(ValueError):
            index.search(q, bad_k)
    with pytest.raises(ValueError):
        index.search(np.zeros((2, 128), np.float32), 5)            # wrong d
    with pytest.raises(ValueError):
        index.search(np.zeros((2, 64), np.float64), 5)             # dtype
    with pytest.raises(ValueError):
        index.search(np.zeros(64, np.float32), 5)                  # rank
    with pytest.raises(ValueError):
        index.search(torch.zeros((2, 64)), 5)                      # device
    with pytest.raises(ValueError):
        index.search(torch.zeros((2, 64), dtype=torch.float16, device="cuda"), 5)
    with pytest.raises(ValueError):
        index.add(np.zeros((2, 65), np.float32))
