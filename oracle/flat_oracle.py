"""CPU oracle of the exact flat L2 search (csrc/flat.cu) -- TEST INFRASTRUCTURE ONLY.

  exact_distances     ||q - x||^2 in the documented order (DESIGN §3): lane l of a warp sums (q_j - x_j)^2 over
                      j = l, l+32, ... in increasing j, each difference, square and add a separately rounded float64
                      operation; then an xor butterfly over the 32 lanes (offsets 16, 8, 4, 2, 1); rounded once to f32
  search_canonical    top-k in (distance asc, id asc) order, (FLT_MAX, -1) padding when k > n
  faiss_blas_search   a restatement of faiss's BLAS flat search (||x||^2 + ||q||^2 - 2 X q in float32, argpartition):
                      the CPU baseline and the comparison "modulo near-ties" against faiss itself
"""
from __future__ import annotations

import numpy as np

FLT_MAX = np.float32(np.finfo(np.float32).max)


def exact_distances(q: np.ndarray, X: np.ndarray) -> np.ndarray:
    """f32 [n] distances of one query q [d] to the rows X [n, d] (float32 inputs, d a multiple of 32)."""
    q = np.asarray(q, dtype=np.float32).astype(np.float64)
    X = np.asarray(X, dtype=np.float32)
    n, d = X.shape
    lanes = np.zeros((n, 32), dtype=np.float64)
    for t in range(d // 32):
        diff = q[t * 32:(t + 1) * 32][None, :] - X[:, t * 32:(t + 1) * 32].astype(np.float64)
        lanes += diff * diff
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, np.arange(32) ^ o]
    return lanes[:, 0].astype(np.float32)


def search_canonical(Q: np.ndarray, X: np.ndarray, k: int, rows_per_block: int = 1 << 16):
    """(D f32 [B, k], I i64 [B, k]) of the exact distances, ascending, ties by row id."""
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float32))
    X = np.asarray(X, dtype=np.float32)
    n = X.shape[0]
    D = np.full((Q.shape[0], k), FLT_MAX, dtype=np.float32)
    I = np.full((Q.shape[0], k), -1, dtype=np.int64)
    for b, q in enumerate(Q):
        best_d = np.zeros(0, np.float32)
        best_i = np.zeros(0, np.int64)
        for a in range(0, n, rows_per_block):
            dist = exact_distances(q, X[a:a + rows_per_block])
            cd = np.concatenate([best_d, dist])
            ci = np.concatenate([best_i, np.arange(a, a + len(dist), dtype=np.int64)])
            o = np.lexsort((ci, cd))[:k]
            best_d, best_i = cd[o], ci[o]
        D[b, :len(best_d)] = best_d
        I[b, :len(best_i)] = best_i
    return D, I


def faiss_blas_search(Q: np.ndarray, X: np.ndarray, k: int):
    """faiss's exhaustive_L2sqr_blas restated: ip = Q X^T in float32 BLAS, dis = ||q||^2 + ||x||^2 - 2 ip (float32),
    the k smallest by argpartition then sorted.  Rounding differs from the exact distances in the low bits."""
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float32))
    X = np.asarray(X, dtype=np.float32)
    xn = np.einsum("ij,ij->i", X, X)
    qn = np.einsum("ij,ij->i", Q, Q)
    dis = qn[:, None] + xn[None, :] - np.float32(2) * (Q @ X.T)
    np.maximum(dis, 0, out=dis)
    kk = min(k, X.shape[0])
    part = np.argpartition(dis, kk - 1, axis=1)[:, :kk] if kk < X.shape[0] else np.tile(np.arange(X.shape[0]), (len(Q), 1))
    pd = np.take_along_axis(dis, part, 1)
    o = np.argsort(pd, axis=1, kind="stable")
    D = np.full((len(Q), k), FLT_MAX, dtype=np.float32)
    I = np.full((len(Q), k), -1, dtype=np.int64)
    D[:, :kk] = np.take_along_axis(pd, o, 1)
    I[:, :kk] = np.take_along_axis(part, o, 1)
    return D, I


def agree_modulo_near_ties(D_ref: np.ndarray, I_ref: np.ndarray, D: np.ndarray, I: np.ndarray, rel: float = 1e-5,
                           atol: float = 0.0) -> bool:
    """Two ranked lists agree modulo near-ties: position by position the distances lie within rel * |D| + atol of each
    other, a row ranked differently has a near-equal distance, and an id found in only one of the two lists has a distance that close to that list's k-th distance (which
    of several near-equal rows fills the last slots).  An fp32 BLAS distance ||q||^2 + ||x||^2 - 2 q.x carries an
    error relative to the norms, not to the distance: pass atol ~ 1e-6 (||q||^2 + ||x||^2) for it."""
    if D_ref.shape != D.shape:
        return False
    D_ref64, D64 = D_ref.astype(np.float64), D.astype(np.float64)
    if not np.all(np.abs(D_ref64 - D64) <= rel * np.abs(D_ref64) + atol):
        return False
    for b in range(len(I)):
        for ids, dist, other in ((I_ref[b], D_ref64[b], I[b]), (I[b], D64[b], I_ref[b])):
            only = ~np.isin(ids, other)
            if np.any(np.abs(dist[only] - dist[-1]) > rel * abs(dist[-1]) + atol):
                return False
        pos = {int(i): j for j, i in enumerate(I_ref[b])}
        for a in np.nonzero(I_ref[b] != I[b])[0]:      # a swapped pair must be a near-tie
            j = pos.get(int(I[b, a]))
            if j is not None and abs(D_ref64[b, j] - D_ref64[b, a]) > rel * abs(D_ref64[b, a]) + atol:
                return False
    return True


def exact_distances_torch(q, X):
    """exact_distances with torch float64 tensors (same IEEE operations in the same order, so bit-identical; fast
    on a GPU for the large parity tests)."""
    import torch
    q = q.to(torch.float64)
    n, d = X.shape
    lanes = torch.zeros((n, 32), dtype=torch.float64, device=X.device)
    for t in range(d // 32):
        diff = q[t * 32:(t + 1) * 32][None, :] - X[:, t * 32:(t + 1) * 32].to(torch.float64)
        lanes = lanes + diff * diff
    idx = torch.arange(32, device=X.device)
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, idx ^ o]
    return lanes[:, 0].to(torch.float32)


def search_canonical_torch(Q, X, k: int):
    """search_canonical on torch tensors (stable sort: equal distances keep ascending row ids)."""
    import torch
    B, n = Q.shape[0], X.shape[0]
    D = torch.full((B, k), float(FLT_MAX), dtype=torch.float32)
    I = torch.full((B, k), -1, dtype=torch.int64)
    for b in range(B):
        dist = exact_distances_torch(Q[b], X)
        s, o = torch.sort(dist, stable=True)
        m = min(k, n)
        D[b, :m] = s[:m].cpu()
        I[b, :m] = o[:m].cpu()
    return D.numpy(), I.numpy()
