"""Batched reference of the exact flat search, fast enough for the 21M-row index -- TEST INFRASTRUCTURE ONLY.

  search_fast(Q, X, k, metric)   the lists of flat_oracle.search_canonical_torch (L2) or
                                 flat_ip_oracle.search_canonical_ip_torch (IP), bit for bit, for finite inputs

The canonical restatements evaluate every (query, row) pair exactly, one query at a time; at 21M rows that is minutes
per query.  This reference does the same in two passes:

  prefilter   an f64 GEMM estimate of every (query, row), smaller is better:
                  L2  e = ||x||^2_64 - 2 (q.x)_64          (the distance minus the constant ||q||^2)
                  IP  e = -(q.x)_64                         (minus the score)
              kept per row chunk: the `keep` smallest per query.  The survivors of a query are the rows with
              e <= e_k + tau, e_k the query's k-th smallest estimate, with
                  L2  tau = 2^-18 (||q||^2 + max ||x||^2) + 2^-140
                  IP  tau = 2^-18 ||q|| max ||x||          + 2^-140
  exact pass  the survivors' exact distances (fo.exact_distances_torch) or scores (fio.exact_inner_products_torch),
              ranked canonically: (distance, id) ascending, or (ip_key of the score, id) ascending.

Why tau keeps every row of the true top-k.  Let v(r) be the ranked value the exact pass computes (the f32 distance,
or minus the f32 score) and c the constant ||q||^2 (L2) or 0 (IP).  With u = 2^-53 and any summation order:
  - the f64 GEMM error: an f64 sum of d products, in any order or blocking, is within (d - 1) u sum |q_i x_i| <=
    d u ||q|| ||x|| of q.x, and ||x||^2_64 within d u ||x||^2 of ||x||^2; with the final subtraction's rounding,
    |e(r) - (||q - x||^2 - c)| <= 3 d u (||q||^2 + ||x||^2) for L2 and |e(r) + q.x| <= d u ||q|| ||x|| for IP;
  - the gap to the f32-rounded exact value: the lane-order f64 sum of the exact pass is within (d + 5) u of the real
    value relative to ||q - x||^2 <= 2 (||q||^2 + ||x||^2) (L2) or to sum |q_i x_i| <= ||q|| ||x|| (IP), and its
    rounding to f32 adds 2^-24 relative (2^-150 absolute below the normal range).
For d <= 1024 the two together are below 2^-22 (||q||^2 + ||x||^2) for L2 and 2^-23 ||q|| ||x|| for IP, plus
2^-150: so |e(r) - (v(r) - c)| <= tau / 2 for every row, with 16x to spare for the f64 rounding of tau and e_k + tau.
Then for a row r of the true top-k, v(r) <= v_k (the k-th ranked value); the k rows of smallest estimate all have
v <= e_k + c + tau / 2, so v_k <= e_k + c + tau / 2, and e(r) <= v(r) - c + tau / 2 <= e_k + tau: r survives.  Rows
outside the top-k that survive only cost exact evaluations.

Self-check.  e_k is exact over the per-chunk cuts when keep >= k (the k smallest estimates lie in their chunks' cuts).
A chunk's cut may have dropped a row of the window only if the chunk holds more than `keep` rows and its keep-th
estimate is <= e_k + tau; such (query, chunk) pairs are estimated again, one query over the whole chunk, and every row
of the window is kept.  Nothing is returned from a truncated window.

Finite inputs only, with ||q||^2 + ||x||^2 <= 2^125 so that no distance or score overflows f32 (what the full-size and
shape tests feed it); other inputs raise ValueError.  Non-finite rows and queries are for the canonical restatements.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo

FLT_MAX = float(np.finfo(np.float32).max)
TAU_REL = 2.0 ** -18
TAU_ABS = 2.0 ** -140


def _estimates(Q64, Xc, xn2c, l2: bool):
    """[B, rows] f64 estimates of the chunk Xc (f32) for the f64 queries Q64; smaller is better."""
    ip = Q64 @ Xc.to(torch.float64).T
    return xn2c[None, :] - 2.0 * ip if l2 else -ip


def search_fast(Q, X, k: int, metric: str = "l2", chunk_rows: int = 1 << 20, keep: int = 256, stats: dict | None = None):
    """(D f32 [B, k], I i64 [B, k]) NumPy, equal to search_canonical_torch (metric "l2") or search_canonical_ip_torch
    ("ip") of the f32 tensors Q [B, d] and X [n, d] (on one device).  `stats`, when given, receives the survivor
    counts and the number of re-estimated (query, chunk) pairs."""
    if metric not in ("l2", "ip"):
        raise ValueError(metric)
    l2 = metric == "l2"
    B, n = Q.shape[0], X.shape[0]
    keep = max(keep, k)
    D = np.full((B, k), FLT_MAX if l2 else -FLT_MAX, dtype=np.float32)
    I = np.full((B, k), -1, dtype=np.int64)
    if B == 0 or n == 0:
        return D, I
    kk = min(k, n)
    Q64 = Q.to(torch.float64)
    xn2 = torch.empty(n, dtype=torch.float64, device=X.device)
    for a in range(0, n, chunk_rows):
        xc = X[a:a + chunk_rows].to(torch.float64)
        xn2[a:a + chunk_rows] = (xc * xc).sum(1)
        del xc
    if not bool(torch.isfinite(xn2).all()) or not bool(torch.isfinite(Q64).all()):
        raise ValueError("search_fast takes finite rows and queries only")
    qn2 = (Q64 * Q64).sum(1)
    xmax2 = xn2.max()
    if float(qn2.max() + xmax2) > 2.0 ** 125:      # ||q - x||^2 <= 2 (||q||^2 + ||x||^2) and q.x stay below FLT_MAX
        raise ValueError("search_fast: a distance or score could overflow f32 (finite, bounded inputs only)")
    tau = TAU_REL * (qn2 + xmax2 if l2 else torch.sqrt(qn2) * torch.sqrt(xmax2)) + TAU_ABS

    vals, idx, last, bounds = [], [], [], []
    for a in range(0, n, chunk_rows):
        b = min(n, a + chunk_rows)
        e = _estimates(Q64, X[a:b], xn2[a:b], l2)
        if not bool(torch.isfinite(e).all()):
            raise ValueError("search_fast: a non-finite estimate (finite inputs only)")
        m = min(keep, b - a)
        v, i = torch.topk(e, m, dim=1, largest=False, sorted=True)
        vals.append(v)
        idx.append(i + a)
        last.append(v[:, -1] if m < b - a else torch.full((B,), float("inf"), dtype=torch.float64, device=X.device))
        bounds.append((a, b))
        del e
    vals, idx = torch.cat(vals, 1), torch.cat(idx, 1)
    e_k = torch.topk(vals, kk, dim=1, largest=False, sorted=True).values[:, -1]
    limit = e_k + tau
    redo = torch.stack(last, 1) <= limit[:, None]                # [B, chunks]: the cut may have dropped window rows
    redo_pairs = torch.nonzero(redo).tolist()
    redo_of = {}
    for b_, c in redo_pairs:
        a, b = bounds[c]
        e = _estimates(Q64[b_:b_ + 1], X[a:b], xn2[a:b], l2)[0]
        redo_of.setdefault(b_, []).append((a, b, torch.nonzero(e <= limit[b_]).flatten() + a))
    n_surv = []
    for b_ in range(B):
        own = idx[b_][vals[b_] <= limit[b_]]
        for a, b, extra in redo_of.get(b_, []):
            own = torch.cat([own[(own < a) | (own >= b)], extra])
        own = torch.sort(own).values                            # ascending ids: a stable sort keeps them for ties
        n_surv.append(int(own.numel()))
        Xs = X[own]
        if l2:
            key = fo.exact_distances_torch(Q[b_], Xs)
        else:
            key = fio.ip_key_torch(fio.exact_inner_products_torch(Q[b_], Xs))
        s, o = torch.sort(key, stable=True)
        D[b_, :kk] = (s[:kk] if l2 else fio.ip_score_torch(s[:kk])).cpu().numpy()
        I[b_, :kk] = own[o[:kk]].cpu().numpy()
    if stats is not None:
        stats.update(survivors=n_surv, redone_pairs=len(redo_pairs), tau_max=float(tau.max()))
    return D, I
