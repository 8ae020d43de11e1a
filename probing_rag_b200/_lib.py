"""ctypes binding of libprobingrag.so (include/probing_rag.h).

There is no CPU fallback: if the CUDA library is missing or fails to load, importing the
symbols raises.  `check(rc)` turns PR_E* codes into the exceptions bm25s raises at the same
points (ValueError for k > num_docs / bad token ids, SURVEY App. A.5)."""
from __future__ import annotations

import ctypes
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PR_LIB_PATH") or os.path.join(PKG_DIR, "libprobingrag.so")   # PR_LIB_PATH: A/B builds

PR_OK, PR_EINVAL, PR_ECUDA, PR_ERANGE, PR_EWORKSPACE, PR_EUNSUPPORTED = 0, -1, -2, -3, -4, -5
PR_MAX_K = 128
PR_PROBER_MAX = 8
PR_MAX_PEERS = 15
PR_FLAT_MAX_LISTS = 32
PR_METRIC_INNER_PRODUCT, PR_METRIC_L2 = 0, 1

c_i32, c_i64, c_f32, c_vp, c_sz = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


class Tuning(ctypes.Structure):
    _fields_ = [("subs_per_item", c_i32), ("warps_per_cta", c_i32), ("docs_per_launch", c_i32),
                ("min_items", c_i32), ("items_per_warp", c_i32), ("tile_epochs", c_i32),
                ("batch_variant", c_i32)]


class AuxInfo(ctypes.Structure):
    _fields_ = [("table_rows", c_i32), ("hot_rows", c_i32), ("n_sub_tiles", c_i32),
                ("table_min_df", c_i64), ("hot_min_df", c_i64), ("hot_stream_bytes", c_i64),
                ("cold_stream_bytes", c_i64)]


class ProberSet(ctypes.Structure):
    _fields_ = [("n_probers", c_i32), ("d_model", c_i32), ("hidden", c_i32),
                ("w1_rowsum", c_vp), ("b1", c_vp),
                ("ln1_w", c_vp), ("ln1_b", c_vp), ("b2", c_vp),
                ("ln2_w", c_vp), ("ln2_b", c_vp), ("w3", c_vp), ("b3", c_vp),
                ("w1_hi", c_vp), ("w1_lo", c_vp), ("w2_hi", c_vp), ("w2_lo", c_vp)]


class FlatTuning(ctypes.Structure):
    _fields_ = [("first_chunk_rows", c_i64), ("growth", c_i32), ("cand_capacity", c_i32)]


class FlatStats(ctypes.Structure):
    _fields_ = [("launches", c_i64), ("chunks", c_i64), ("candidates", c_i64), ("max_candidates", c_i64),
                ("fallback_queries", c_i64)]


# every symbol include/probing_rag.h declares: (restype, argtypes)
SIGNATURES = {
    "pr_version": (ctypes.c_int, []),
    "pr_last_error": (ctypes.c_char_p, []),
    "pr_index_create": (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int, c_i64, c_i32, c_i32, c_i32, c_i64,
                                       c_vp, c_vp, c_vp]),
    "pr_index_destroy": (ctypes.c_int, [c_vp]),
    "pr_index_aux_bytes": (c_sz, [c_vp, c_sz]),
    "pr_index_build_aux": (ctypes.c_int, [c_vp, c_vp, c_sz, c_vp]),
    "pr_index_aux_info": (ctypes.c_int, [c_vp, ctypes.POINTER(AuxInfo)]),
    "pr_index_set_tuning": (ctypes.c_int, [c_vp, ctypes.POINTER(Tuning)]),
    "pr_index_get_tuning": (ctypes.c_int, [c_vp, ctypes.POINTER(Tuning)]),
    "pr_bm25_workspace_bytes": (c_sz, [c_vp, c_i32, c_i32]),
    "pr_bm25_topk": (ctypes.c_int, [c_vp, c_i32, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "pr_bm25_num_launches": (c_i32, [c_vp, c_i32, c_i32, c_i64]),
    "pr_bm25_theta_offset": (c_sz, [c_vp, c_i32, c_i32]),
    "pr_bm25_running_scores_offset": (c_sz, [c_vp, c_i32, c_i32]),
    "pr_bm25_raise_union_bound": (ctypes.c_int, [c_vp, c_i32, c_i32, c_vp, c_i32, c_vp, c_sz, c_vp]),
    "pr_bm25_topk_range": (ctypes.c_int, [c_vp, c_i32, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_sz, c_i32, c_i32,
                                          c_vp]),
    "pr_peer_alloc": (ctypes.c_int, [ctypes.c_int, c_sz, ctypes.POINTER(c_vp), ctypes.c_char_p]),
    "pr_peer_open": (ctypes.c_int, [ctypes.c_int, ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "pr_peer_close": (ctypes.c_int, [c_vp]),
    "pr_peer_free": (ctypes.c_int, [c_vp]),
    "pr_index_set_peer_thetas": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, ctypes.POINTER(c_vp), c_vp]),
    "pr_bm25_status": (ctypes.c_int, [c_vp, c_vp]),
    "pr_bm25_last_launches": (c_i64, [c_vp]),
    "pr_index_set_profiling": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "pr_bm25_profile": (ctypes.c_int, [c_vp, ctypes.POINTER(c_f32), ctypes.POINTER(c_i32)]),
    "pr_topk_merge": (ctypes.c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "pr_prober_workspace_bytes": (c_sz, [c_i32, c_i32, c_i32, c_i32]),
    "pr_pool_accumulate": (ctypes.c_int, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_i32, c_i64, c_i64,
                                          c_vp, c_vp]),
    "pr_prober_forward": (ctypes.c_int, [ctypes.POINTER(ProberSet), c_i32, c_vp, c_i32, ctypes.c_double, c_i32, c_vp, c_vp,
                                         c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "pr_flat_create": (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int, c_vp, c_i64, c_i32]),
    "pr_flat_create_metric": (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int, c_vp, c_i64, c_i32, ctypes.c_int]),
    "pr_flat_destroy": (ctypes.c_int, [c_vp]),
    "pr_flat_aux_bytes": (c_sz, [c_vp]),
    "pr_flat_build_aux": (ctypes.c_int, [c_vp, c_vp, c_sz, c_vp]),
    "pr_flat_set_tuning": (ctypes.c_int, [c_vp, ctypes.POINTER(FlatTuning)]),
    "pr_flat_get_tuning": (ctypes.c_int, [c_vp, ctypes.POINTER(FlatTuning)]),
    "pr_flat_workspace_bytes": (c_sz, [c_vp, c_i32, c_i32]),
    "pr_flat_search": (ctypes.c_int, [c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "pr_flat_last_stats": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i32, ctypes.POINTER(FlatStats), c_vp]),
    "pr_flat_merge": (ctypes.c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, ctypes.POINTER(c_i64), c_vp, c_vp, c_vp]),
    "pr_flat_merge_metric": (ctypes.c_int, [c_i32, c_i32, c_i32, c_vp, c_vp, ctypes.POINTER(c_i64), c_vp, c_vp, c_vp,
                                            ctypes.c_int]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load the library once; raise (never fall back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m probing_rag_b200.build` "
                "(there is no CPU fallback for the retrieval hot path)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the library lacks a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def last_error() -> str:
    return lib().pr_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc == PR_OK:
        return
    msg = last_error()
    if rc in (PR_ERANGE, PR_EINVAL):
        raise ValueError(msg)
    raise RuntimeError(f"libprobingrag error {rc}: {msg}")
