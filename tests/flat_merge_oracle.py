"""CPU restatement of pr_flat_merge (csrc/flat.cu) -- TEST INFRASTRUCTURE ONLY.

  merge_canonical   per query, every entry of the L lists with id >= 0, its id offset by its list's base, ranked by
                    (uint32 bit pattern of the distance, every NaN as 0x7FFFFFFF; global id) ascending -- the key
                    order of the single index's lists -- and cut to k; short rows padded (FLT_MAX, -1); a NaN comes
                    back as 0x7FFFFFFF.  Entries equal in both keys keep list order.
"""
from __future__ import annotations

import numpy as np

FLT_MAX = np.float32(np.finfo(np.float32).max)
_EMPTY = np.uint64(1 << 32)          # above the bit pattern of every real distance


def merge_canonical(D: np.ndarray, I: np.ndarray, bases, k: int):
    """D f32 [L, B, kk], I i64 [L, B, kk], bases [L] -> (D f32 [B, k], I i64 [B, k])."""
    D = np.ascontiguousarray(D, dtype=np.float32)
    I = np.asarray(I, dtype=np.int64)
    L, B, kk = D.shape
    valid = I >= 0
    bits = D.view(np.uint32).astype(np.uint64)
    bits = np.where((bits & np.uint64(0x7FFFFFFF)) > np.uint64(0x7F800000), np.uint64(0x7FFFFFFF), bits)
    hi = np.where(valid, bits, _EMPTY)
    gid = np.where(valid, I + np.asarray(bases, dtype=np.int64)[:, None, None], np.iinfo(np.int64).max)
    hi = hi.transpose(1, 0, 2).reshape(B, L * kk)          # per query, list-major: equal keys keep list order
    gid = gid.transpose(1, 0, 2).reshape(B, L * kk)
    order = np.lexsort((gid, hi), axis=-1)[:, :k]
    hi, gid = np.take_along_axis(hi, order, 1), np.take_along_axis(gid, order, 1)
    out_d = np.full((B, k), FLT_MAX, dtype=np.float32)
    out_i = np.full((B, k), -1, dtype=np.int64)
    m = min(k, L * kk)
    real = hi[:, :m] != _EMPTY
    out_d[:, :m] = np.where(real, hi[:, :m].astype(np.uint32).view(np.float32), FLT_MAX)
    out_i[:, :m] = np.where(real, gid[:, :m], -1)
    return out_d, out_i
