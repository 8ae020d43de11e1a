"""The batched full-size reference (tests/flat_fast_oracle.py) against the canonical restatements, bit for bit, on the
CPU: random, clustered and tied rows, near-tie shells whose distances lie a few ulp apart, the one-signed bf16-bias
vectors, k above n, and per-chunk cuts small enough that the window check has to re-estimate chunks."""
import numpy as np
import pytest
import torch

import flat_fast_oracle as ffo
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo


def _canonical(Q, X, k, metric):
    return fo.search_canonical_torch(Q, X, k) if metric == "l2" else fio.search_canonical_ip_torch(Q, X, k)


def _pin(Q, X, k, metric, **kw):
    stats = {}
    D, I = ffo.search_fast(Q, X, k, metric, stats=stats, **kw)
    Dr, Ir = _canonical(Q, X, k, metric)
    assert np.array_equal(I, Ir), metric
    assert np.array_equal(D.view(np.uint32), Dr.view(np.uint32)), metric
    return stats


def _clustered(g, n, d, n_cent=16):
    cent = torch.randn((n_cent, d), generator=g, dtype=torch.float32) * 1.5 / d ** 0.5
    c = torch.randint(0, n_cent, (n,), generator=g)
    return cent[c] + torch.randn((n, d), generator=g) * 0.6 / d ** 0.5


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("k", [1, 10, 128])
def test_random_and_clustered_rows(metric, k):
    g = torch.Generator().manual_seed(11 + k)
    for X in (torch.randn((3000, 64), generator=g), _clustered(g, 3000, 128)):
        Q = torch.cat([X[:5] + 0.01 * torch.randn((5, X.shape[1]), generator=g),
                       torch.randn((4, X.shape[1]), generator=g)])
        _pin(Q, X, k, metric)
        st = _pin(Q, X, k, metric, chunk_rows=700, keep=k)       # cuts of exactly k: chunks get re-estimated
        assert min(st["survivors"]) >= k


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_exact_ties_duplicates_and_k_above_n(metric):
    g = torch.Generator().manual_seed(3)
    base = torch.randn((100, 64), generator=g)
    X = torch.cat([base, base, torch.zeros((30, 64)), base[:5]])
    Q = torch.cat([base[:6], torch.zeros((2, 64))])
    for k in (1, 64, 128):
        _pin(Q, X, k, metric, chunk_rows=50, keep=8)
    _pin(Q, X[:3], 8, metric)                                      # k > n: padding
    D, I = ffo.search_fast(Q, X[:0], 4, metric)
    assert np.all(I == -1)


def test_near_tie_shells():
    """Rows on shells around the query (L2) and rows of one score up to a few ulp (IP): thousands of rows inside the
    window, far more than a chunk's cut keeps."""
    g = torch.Generator().manual_seed(6)
    d = 128
    q = torch.randn(d, generator=g)
    u = torch.randn((2000, d), generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    r = 1.0 + torch.randint(0, 8, (2000, 1), generator=g) * 2.0 ** -22
    far = torch.randn((3000, d), generator=g) * 3
    X = torch.cat([far[:1500], q[None, :] + u * r, far[1500:]])
    Q = torch.stack([q, q + 1e-7 * torch.randn(d, generator=g)])
    for k in (1, 10, 128):
        st = _pin(Q, X, k, "l2", chunk_rows=1000, keep=k)
        assert st["redone_pairs"] > 0
    qh = q / q.norm()
    o = torch.randn((2000, d), generator=g)
    o = o - (o @ qh)[:, None] * qh[None, :]
    s = 10.0 * (1 + torch.randint(0, 8, (2000, 1), generator=g) * 2.0 ** -22)
    X = torch.cat([far[:1500] - 3 * qh, s * qh[None, :] + o, far[1500:] - 3 * qh])
    for k in (1, 10, 128):
        st = _pin(Q, X, k, "ip", chunk_rows=1000, keep=k)
        assert st["redone_pairs"] > 0


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_bf16_biased_vectors(metric):
    """The one-signed bf16-bias vectors of test_flat_ip_oracle, with fillers scoring between them, in one or both
    signs."""
    d = 768
    rng = np.random.default_rng(9)
    c = np.float32(1 + 2.0 ** -8 - 2.0 ** -20)
    rows = []
    for _ in range(300):
        s = rng.choice([-1.0, 1.0], d) if rng.random() < 0.5 else np.ones(d)
        rows.append((c * s).astype(np.float32))
    X = np.stack(rows)
    fill = np.ones((200, d), np.float32)
    fill[:, : d // 4] = 1 + 2.0 ** -7
    X = torch.from_numpy(np.concatenate([fill, X, np.zeros((100, d), np.float32)]))
    Q = torch.stack([X[200], X[201], torch.full((d,), float(c))])
    for k in (1, 10, 128):
        _pin(Q, X, k, metric, chunk_rows=128, keep=k)


def test_non_finite_input_is_refused():
    X = torch.randn((10, 64))
    X[3, 5] = float("nan")
    for metric in ("l2", "ip"):
        with pytest.raises(ValueError, match="finite"):
            ffo.search_fast(torch.randn((2, 64)), X, 3, metric)
    with pytest.raises(ValueError, match="finite"):
        ffo.search_fast(torch.full((1, 64), 1e30), torch.full((4, 64), 1e30), 3, "l2")
