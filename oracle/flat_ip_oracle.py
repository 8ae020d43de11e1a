"""CPU oracle of the exact flat inner-product search (csrc/flat.cu, IndexFlatIP) -- TEST INFRASTRUCTURE ONLY.

  exact_inner_products  q.x in the lane order of flat_oracle.exact_distances (DESIGN §3): lane l starts at +0.0 and adds
                        q_j x_j (an exact f64 product, one rounded f64 add) over j = l, l+32, ...; the xor butterfly;
                        rounded once to f32, then + 0.0 so that a score is never -0
  search_canonical_ip   top-k by ip_key (score descending, NaN after -inf), ties by id; (-FLT_MAX, -1) padding
  faiss_blas_search_ip  faiss's BLAS inner-product search restated (Q X^T in float32, argpartition): the CPU baseline
  ip_key / ip_score     the refine's key of a score (ascending as the score descends) and its inverse; *_torch forms

flat_oracle.agree_modulo_near_ties compares these lists with faiss's too (atol ~1e-6 max |q||x|).
"""
from __future__ import annotations

import numpy as np

from .flat_oracle import FLT_MAX


def ip_key(scores) -> np.ndarray:
    """uint32 key of f32 scores that ascends as the score descends, every NaN mapped to 0xFFFFFFFF (after -inf)
    (csrc/flat.cu ip_key)."""
    b = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32)
    k = np.where(b & np.uint32(0x80000000), b, b ^ np.uint32(0x7FFFFFFF))
    return np.where((b & np.uint32(0x7FFFFFFF)) > np.uint32(0x7F800000), np.uint32(0xFFFFFFFF), k).astype(np.uint32)


def ip_score(keys) -> np.ndarray:
    """The f32 scores of ip_key values (a NaN comes back as the NaN 0xFFFFFFFF)."""
    k = np.asarray(keys, dtype=np.uint32)
    return np.where(k & np.uint32(0x80000000), k, k ^ np.uint32(0x7FFFFFFF)).astype(np.uint32).view(np.float32)


def exact_inner_products(q: np.ndarray, X: np.ndarray) -> np.ndarray:
    """f32 [n] inner products of one query q [d] with the rows X [n, d] (float32 inputs, d a multiple of 32)."""
    q = np.asarray(q, dtype=np.float32).astype(np.float64)
    X = np.asarray(X, dtype=np.float32)
    n, d = X.shape
    lanes = np.zeros((n, 32), dtype=np.float64)
    for t in range(d // 32):
        lanes = lanes + q[t * 32:(t + 1) * 32][None, :] * X[:, t * 32:(t + 1) * 32].astype(np.float64)
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, np.arange(32) ^ o]
    return lanes[:, 0].astype(np.float32) + np.float32(0)


def search_canonical_ip(Q: np.ndarray, X: np.ndarray, k: int, rows_per_block: int = 1 << 16):
    """(D f32 [B, k], I i64 [B, k]) of the exact inner products, descending (NaN last, as the NaN 0xFFFFFFFF), ties by
    row id; rows short of k are (-FLT_MAX, -1)."""
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float32))
    X = np.asarray(X, dtype=np.float32)
    n = X.shape[0]
    D = np.full((Q.shape[0], k), -FLT_MAX, dtype=np.float32)
    I = np.full((Q.shape[0], k), -1, dtype=np.int64)
    for b, q in enumerate(Q):
        best_k = np.zeros(0, np.uint32)
        best_i = np.zeros(0, np.int64)
        for a in range(0, n, rows_per_block):
            ck = np.concatenate([best_k, ip_key(exact_inner_products(q, X[a:a + rows_per_block]))])
            ci = np.concatenate([best_i, np.arange(a, min(n, a + rows_per_block), dtype=np.int64)])
            o = np.lexsort((ci, ck))[:k]
            best_k, best_i = ck[o], ci[o]
        D[b, :len(best_k)] = ip_score(best_k)
        I[b, :len(best_i)] = best_i
    return D, I


def faiss_blas_search_ip(Q: np.ndarray, X: np.ndarray, k: int):
    """faiss's exhaustive_inner_product_blas restated: Q X^T in float32 BLAS, the k largest by argpartition, then
    sorted descending; rows short of k are (-FLT_MAX, -1).  Rounding differs from the exact scores in the low bits."""
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float32))
    X = np.asarray(X, dtype=np.float32)
    neg = -(Q @ X.T)
    kk = min(k, X.shape[0])
    part = np.argpartition(neg, kk - 1, axis=1)[:, :kk] if kk < X.shape[0] else np.tile(np.arange(X.shape[0]), (len(Q), 1))
    pn = np.take_along_axis(neg, part, 1)
    o = np.argsort(pn, axis=1, kind="stable")
    D = np.full((len(Q), k), -FLT_MAX, dtype=np.float32)
    I = np.full((len(Q), k), -1, dtype=np.int64)
    D[:, :kk] = -np.take_along_axis(pn, o, 1)
    I[:, :kk] = np.take_along_axis(part, o, 1)
    return D, I


def ip_key_torch(scores):
    """ip_key on a torch float32 tensor, as int64 values in [0, 2^32)."""
    import torch
    b = scores.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    k = torch.where((b & 0x80000000) != 0, b, b ^ 0x7FFFFFFF)
    return torch.where((b & 0x7FFFFFFF) > 0x7F800000, torch.full_like(b, 0xFFFFFFFF), k)


def ip_score_torch(keys):
    """The f32 scores of int64 ip_key values (the inverse of ip_key_torch; a NaN as 0xFFFFFFFF)."""
    import torch
    b = torch.where((keys & 0x80000000) != 0, keys, keys ^ 0x7FFFFFFF)
    return torch.where(b >= 2 ** 31, b - 2 ** 32, b).to(torch.int32).view(torch.float32)


def exact_inner_products_torch(q, X):
    """exact_inner_products with torch float64 tensors (same IEEE operations in the same order, so bit-identical; fast
    on a GPU for the large parity tests)."""
    import torch
    q = q.to(torch.float64)
    n, d = X.shape
    lanes = torch.zeros((n, 32), dtype=torch.float64, device=X.device)
    for t in range(d // 32):
        lanes = lanes + q[t * 32:(t + 1) * 32][None, :] * X[:, t * 32:(t + 1) * 32].to(torch.float64)
    idx = torch.arange(32, device=X.device)
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, idx ^ o]
    return lanes[:, 0].to(torch.float32) + 0.0


def search_canonical_ip_torch(Q, X, k: int):
    """search_canonical_ip on torch tensors (a stable sort of the keys: equal keys keep ascending row ids)."""
    import torch
    B, n = Q.shape[0], X.shape[0]
    D = torch.full((B, k), -float(FLT_MAX), dtype=torch.float32)
    I = torch.full((B, k), -1, dtype=torch.int64)
    for b in range(B):
        s, o = torch.sort(ip_key_torch(exact_inner_products_torch(Q[b], X)), stable=True)
        m = min(k, n)
        D[b, :m] = ip_score_torch(s[:m]).cpu()
        I[b, :m] = o[:m].cpu()
    return D.numpy(), I.numpy()

