"""Batched reference of the exact flat range search, fast enough for the 21M-row index -- TEST INFRASTRUCTURE ONLY.

  range_search_fast(Q, X, radius, metric)   the result of flat_range_oracle.range_search_canonical_torch, bit for bit,
                                            for finite inputs

It rests on the prefilter argument of flat_fast_oracle (read it there): with the f64 GEMM estimate
    L2  e = ||x||^2_64 - 2 (q.x)_64        IP  e = -(q.x)_64
the ranked value v of the exact pass (the f32 distance, or minus the f32 score) and c = ||q||^2 (L2) or 0 (IP),
|e - (v - c)| <= tau / 2 with the same tau.  A result has v < radius (L2) or v = -S < -radius (IP), so
    L2  e <= v - c + tau / 2 < radius - ||q||^2 + tau        IP  e < -radius + tau
and every row with e <= radius - ||q||^2 + tau (IP: e <= -radius + tau) is kept; the survivors are evaluated exactly
and those with D < radius (S > radius) returned in ascending row id.  The f64 rounding of the limit is covered by the
factor 16 of slack in tau.  The radius is rounded to f32 first, as the index rounds it.
"""
from __future__ import annotations

import numpy as np
import torch

from flat_fast_oracle import TAU_ABS, TAU_REL, _estimates
from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo


def range_search_fast(Q, X, radius, metric: str = "l2", chunk_rows: int = 1 << 20, stats: dict | None = None):
    """(lims i64 [B + 1], D f32, I i64) NumPy of the f32 tensors Q [B, d], X [n, d] (one device).  `stats`, when given,
    receives the survivor count per query."""
    if metric not in ("l2", "ip"):
        raise ValueError(metric)
    l2 = metric == "l2"
    r = float(np.float32(radius))
    B, n = Q.shape[0], X.shape[0]
    lims = np.zeros(B + 1, dtype=np.int64)
    if B == 0 or n == 0 or r != r:
        return lims, np.zeros(0, np.float32), np.zeros(0, np.int64)
    Q64 = Q.to(torch.float64)
    xn2 = torch.empty(n, dtype=torch.float64, device=X.device)
    for a in range(0, n, chunk_rows):
        xc = X[a:a + chunk_rows].to(torch.float64)
        xn2[a:a + chunk_rows] = (xc * xc).sum(1)
        del xc
    if not bool(torch.isfinite(xn2).all()) or not bool(torch.isfinite(Q64).all()):
        raise ValueError("range_search_fast takes finite rows and queries only")
    qn2 = (Q64 * Q64).sum(1)
    xmax2 = xn2.max()
    if float(qn2.max() + xmax2) > 2.0 ** 125:
        raise ValueError("range_search_fast: a distance or score could overflow f32 (finite, bounded inputs only)")
    tau = TAU_REL * (qn2 + xmax2 if l2 else torch.sqrt(qn2) * torch.sqrt(xmax2)) + TAU_ABS
    limit = (r - qn2 + tau) if l2 else (-r + tau)                 # [B]; +inf when r = +inf (L2) or -inf (IP)
    surv = [[] for _ in range(B)]
    for a in range(0, n, chunk_rows):
        b = min(n, a + chunk_rows)
        e = _estimates(Q64, X[a:b], xn2[a:b], l2)
        hit = e <= limit[:, None]
        qi, ri = torch.nonzero(hit, as_tuple=True)
        counts = torch.bincount(qi, minlength=B).tolist()
        rows = (ri + a).split(counts)
        for q_ in range(B):
            if counts[q_]:
                surv[q_].append(rows[q_])
        del e, hit
    Ds, Is, n_surv = [], [], []
    for q_ in range(B):
        own = torch.cat(surv[q_]) if surv[q_] else torch.zeros(0, dtype=torch.int64, device=X.device)
        n_surv.append(int(own.numel()))
        v = (fo.exact_distances_torch if l2 else fio.exact_inner_products_torch)(Q[q_], X[own])
        keep = v < r if l2 else v > r
        Ds.append(v[keep].cpu().numpy())
        Is.append(own[keep].cpu().numpy().astype(np.int64))
        lims[q_ + 1] = lims[q_] + int(keep.sum())
    if stats is not None:
        stats.update(survivors=n_surv)
    return lims, np.concatenate(Ds).astype(np.float32), np.concatenate(Is)
