"""CPU oracle of the exact flat range search (csrc/flat.cu, pr_flat_range_search) -- TEST INFRASTRUCTURE ONLY.

  range_search_canonical(Q, X, radius, metric)   (lims, D, I) in faiss's RangeSearchResult layout:
      L2  row r is a result of query q iff its exact distance (flat_oracle.exact_distances) satisfies D < radius
      IP  iff its exact score (flat_ip_oracle.exact_inner_products) satisfies S > radius
  with radius first rounded to f32 (RNE).  The comparisons are strict and false for NaN, so a NaN value is never a
  result and a NaN radius gives none.  Results of a query are in ascending row id; lims [B + 1] int64 with lims[0] = 0.
  range_search_canonical_torch   the same on torch tensors (bit-identical; fast on a GPU)
"""
from __future__ import annotations

import numpy as np

from .flat_ip_oracle import exact_inner_products, exact_inner_products_torch
from .flat_oracle import exact_distances, exact_distances_torch


def _check_metric(metric: str) -> bool:
    if metric not in ("l2", "ip"):
        raise ValueError(f"metric must be 'l2' or 'ip', got {metric!r}")
    return metric == "l2"


def range_search_canonical(Q, X, radius, metric: str = "l2", rows_per_block: int = 1 << 16):
    """(lims i64 [B + 1], D f32 [total], I i64 [total]) of the exact range search of Q [B, d] over X [n, d]."""
    l2 = _check_metric(metric)
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float32))
    X = np.asarray(X, dtype=np.float32)
    r = np.float32(radius)
    lims = np.zeros(Q.shape[0] + 1, dtype=np.int64)
    Ds, Is = [], []
    for b, q in enumerate(Q):
        for a in range(0, X.shape[0], rows_per_block):
            v = (exact_distances if l2 else exact_inner_products)(q, X[a:a + rows_per_block])
            hit = np.nonzero(v < r if l2 else v > r)[0]
            Ds.append(v[hit])
            Is.append(hit.astype(np.int64) + a)
            lims[b + 1] += len(hit)
    lims = np.cumsum(lims)
    D = np.concatenate(Ds) if Ds else np.zeros(0, np.float32)
    I = np.concatenate(Is) if Is else np.zeros(0, np.int64)
    return lims, D.astype(np.float32), I


def range_search_canonical_torch(Q, X, radius, metric: str = "l2"):
    """range_search_canonical on torch f32 tensors (Q and X on one device); NumPy results."""
    import torch
    l2 = _check_metric(metric)
    r = float(np.float32(radius))
    lims = np.zeros(Q.shape[0] + 1, dtype=np.int64)
    Ds, Is = [], []
    for b in range(Q.shape[0]):
        v = (exact_distances_torch if l2 else exact_inner_products_torch)(Q[b], X)
        hit = torch.nonzero(v < r if l2 else v > r).flatten()
        Ds.append(v[hit].cpu().numpy())
        Is.append(hit.cpu().numpy().astype(np.int64))
        lims[b + 1] = lims[b] + hit.numel()
    D = np.concatenate(Ds) if Ds else np.zeros(0, np.float32)
    I = np.concatenate(Is) if Is else np.zeros(0, np.int64)
    return lims, D.astype(np.float32), I
