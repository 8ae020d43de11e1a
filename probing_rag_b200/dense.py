"""Exact dense retrieval: faiss ``IndexFlatL2`` and ``IndexFlatIP`` drop-ins on the GPU (include/probing_rag.h, "dense
flat L2 and inner-product search").

The reference's dense path (``exp_rag.py`` without ``--is_sparse``) builds ``faiss.IndexFlatL2(768)`` over contriever
embeddings (/root/reference/make_indexer.py:446-457), loads it with ``faiss.read_index`` (exp_rag.py:243-248) and calls
``index.search(q, 5)`` (exp_rag.py:431-438, 496; utils.py:365-380).  This module offers the same names:

    index = dense.read_index("wiki_contriever.index")     # or IndexFlatL2(768); index.add(xb)
    D, I = index.search(q, 5)                              # numpy in -> numpy out, like faiss

Under torchrun (one process per GPU), ``dense.read_index(path, sharded=True)`` gives each rank a contiguous row range
of the file and returns a ``ShardedIndexFlatL2``; its ``search`` returns, on every rank, the same lists as one index.

``D`` holds float32 squared L2 distances, ascending, ties broken by row id; ``I`` int64 row ids; rows short of k are
(FLT_MAX, -1).  ``IndexFlatIP`` (Contriever's and DPR's own indexes, fourcc 'IxFI') returns inner products q.x instead,
descending, ties by row id, NaN after -inf, rows short of k padded (-FLT_MAX, -1); ``read_index`` returns whichever class
the file holds.  ``IndexScalarQuantizer(d, ScalarQuantizer.QT_fp16, metric)`` (fourcc 'IxSQ') stores the rows as fp16
codes, a third of an IndexFlat's device memory, and returns bit for bit what IndexFlatL2 / IndexFlatIP returns over the
fp16-decoded rows.  The distances are exact (float64 evaluation in a fixed order, DESIGN §3), so they can differ from
faiss's own fp32 BLAS results in the last bits and near-ties may rank differently.  A CUDA tensor batch returns CUDA
tensors without a host copy.  There is no CPU path: search runs the sm_100a kernels of libprobingrag.so.
"""
from __future__ import annotations

import ctypes
import os
import struct

import numpy as np
import torch
import torch.distributed as dist

from . import _lib

METRIC_INNER_PRODUCT, METRIC_L2 = _lib.PR_METRIC_INNER_PRODUCT, _lib.PR_METRIC_L2     # faiss's numbering
FOURCC_FLAT_L2, FOURCC_FLAT_IP, FOURCC_SQ = b"IxF2", b"IxFI", b"IxSQ"
_FOURCC = {METRIC_L2: FOURCC_FLAT_L2, METRIC_INNER_PRODUCT: FOURCC_FLAT_IP}
_NAME = {METRIC_L2: "IndexFlatL2", METRIC_INNER_PRODUCT: "IndexFlatIP"}
_HEADER = struct.Struct("<4siqqqBiQ")     # fourcc, d, ntotal, 2 dummies, is_trained, metric_type, float count
_SQ_HEADER = struct.Struct("<4siqqqBiiifQQQ")   # IxSQ: the index header without the float count, then the
#                                                 ScalarQuantizer: qtype, rangestat, rangestat_arg, d, code_size,
#                                                 trained count (its floats follow, then the codes' byte count)
_COPY_BYTES = 256 << 20                  # host <-> device copies of rows go in pieces of this size
_RANGE_CAP0 = 1024                       # range_search's first staging size per query ...
_RANGE_STAGING_BYTES = 1 << 30           # ... and the most its staging buffers take (12 bytes a result)


def _check_d(d) -> int:
    if not isinstance(d, (int, np.integer)) or d < 64 or d > 1024 or d % 64:
        raise ValueError(f"d = {d!r} unsupported: a multiple of 64 in [64, 1024]")
    return int(d)


def _check_k(k) -> int:
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= k <= _lib.PR_MAX_K:
        raise ValueError(f"k must be an integer in [1, {_lib.PR_MAX_K}], got {k!r}")
    return int(k)


def _as_rows(x, d: int, what: str) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        if x.dtype != np.float32:
            raise ValueError(f"{what} must be float32, got {x.dtype}")
        x = torch.from_numpy(np.ascontiguousarray(x))
    elif not isinstance(x, torch.Tensor):
        raise ValueError(f"{what} must be a NumPy array or a tensor, got {type(x).__name__}")
    elif x.dtype != torch.float32:
        raise ValueError(f"{what} must be float32, got {x.dtype}")
    if x.dim() != 2 or x.shape[1] != d:
        raise ValueError(f"{what} must be [n, {d}], got {tuple(x.shape)}")
    return x


def _queries(x, d: int, device=None) -> torch.Tensor:
    """The query rows [B, d] float32 of x, a NumPy array or a tensor; a tensor must be on `device` (None: anywhere)."""
    if isinstance(x, torch.Tensor) and device is not None and x.device != device:
        raise ValueError(f"queries are on {x.device}, the index on {device}")
    return _as_rows(x, d, "queries")


def _like_queries(x, *res):
    """Results as the queries x came: tensors for a tensor; NumPy arrays for a NumPy array, with a range search's
    lims (the first of three) as uint64, faiss's size_t."""
    if not isinstance(x, np.ndarray):
        return res
    res = tuple(r.cpu().numpy() for r in res)
    return (res[0].astype(np.uint64),) + res[1:] if len(res) == 3 else res


def _aligned(nbytes: int, device) -> tuple[torch.Tensor, int]:
    """(buffer, pointer): nbytes of device memory from a 1024-byte-aligned pointer, as the C ABI takes workspaces and
    aux buffers."""
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    return buf, (buf.data_ptr() + 1023) // 1024 * 1024


class _IndexFlat:
    """A flat index of one metric (the subclass's ``metric_type``) on one GPU."""

    is_trained = True
    metric_type: int

    def __init__(self, d: int, device="cuda"):
        self.d = _check_d(d)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError(f"{type(self).__name__} needs a CUDA device, got {self.device}")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._rows = torch.empty((0, self.d), dtype=torch.float32, device=self.device)
        self._tuning = _lib.FlatTuning()
        self._h = None
        self._aux = None
        self._last = None
        self._range_cap = _RANGE_CAP0   # staging results per query of range_search: the most one query had last time
        self._range_cap_forced = None   # tests: a fixed staging size (a tiny one takes the second pass)

    # ------------------------------------------------------------------ faiss interface
    @property
    def ntotal(self) -> int:
        return int(self._rows.shape[0])

    def add(self, x) -> None:
        """Append float32 rows [n, d] (NumPy array or tensor).  The rows are copied, as faiss copies them: changing
        or reusing x afterwards leaves the index as it was."""
        x = self._as_rows(x, "x")
        if self.ntotal + x.shape[0] > 2 ** 31 - 1:
            raise ValueError(f"an {type(self).__name__} holds at most 2^31 - 1 rows")
        if self.ntotal:
            self._set_rows(torch.cat([self._rows, x.to(self.device)]))
        else:       # a contiguous float32 tensor already on the device would otherwise be stored as it is
            self._set_rows(x.to(self.device, memory_format=torch.contiguous_format, copy=True))

    def reset(self) -> None:
        self._set_rows(torch.empty((0, self.d), dtype=torch.float32, device=self.device))

    @torch.no_grad()
    def search(self, x, k: int):
        """(D, I) of the k nearest rows (L2) or the k largest inner products (IP) of every query row of x [B, d]
        float32."""
        k = _check_k(k)
        q = _queries(x, self.d, self.device).to(self.device).contiguous()
        B = q.shape[0]
        D = torch.empty((B, k), dtype=torch.float32, device=self.device)
        I = torch.empty((B, k), dtype=torch.int64, device=self.device)
        if B:
            L = _lib.lib()
            h = self._handle()
            nbytes = int(L.pr_flat_workspace_bytes(h, B, k))
            ws, ws_ptr = _aligned(nbytes, self.device)
            with torch.cuda.device(self.device):
                _lib.check(L.pr_flat_search(h, B, q.data_ptr(), k, D.data_ptr(), I.data_ptr(), ws_ptr,
                                            nbytes, torch.cuda.current_stream(self.device).cuda_stream))
            self._last = (ws, ws_ptr, B, k)
        return _like_queries(x, D, I)

    @torch.no_grad()
    def range_search(self, x, radius):
        """(lims, D, I): every row with exact distance D < radius (L2) or score S > radius (IP) for each query row of
        x [B, d] float32; query q's results are D[lims[q]:lims[q + 1]], I[...], in ascending row id.  The radius is
        rounded to float32 first; NaN values are never results.  NumPy in -> NumPy out with lims uint64 (faiss's
        size_t), a CUDA tensor in -> CUDA tensors out with lims int64.  Synchronises the device once (twice when some
        query has more results than the staging segments hold)."""
        radius = float(np.float32(radius))
        q = _queries(x, self.d, self.device).to(self.device).contiguous()
        B = q.shape[0]
        lims = torch.zeros(B + 1, dtype=torch.int64, device=self.device)
        D = torch.empty(0, dtype=torch.float32, device=self.device)
        I = torch.empty(0, dtype=torch.int64, device=self.device)
        if B:
            cap = self._range_cap_forced or max(1, min(self._range_cap, self.ntotal, _RANGE_STAGING_BYTES // (12 * B)))
            count = torch.empty(B, dtype=torch.int64, device=self.device)
            Ds = torch.empty(B * cap, dtype=torch.float32, device=self.device)
            Is = torch.empty(B * cap, dtype=torch.int64, device=self.device)
            self._range_call(q, radius, torch.arange(B + 1, device=self.device) * cap, count, Ds, Is)
            torch.cumsum(count, 0, out=lims[1:])
            most = int(count.max())
            if most <= cap:
                keep = torch.arange(cap, device=self.device)[None, :] < count[:, None]
                D, I = Ds.view(B, cap)[keep], Is.view(B, cap)[keep]
            else:                           # the same rows again, written straight to their final places
                total = int(lims[-1])
                D = torch.empty(total, dtype=torch.float32, device=self.device)
                I = torch.empty(total, dtype=torch.int64, device=self.device)
                self._range_call(q, radius, lims, count, D, I)
            self._range_cap = max(_RANGE_CAP0, most)
        return _like_queries(x, lims, D, I)

    # ------------------------------------------------------------------ project extras
    def set_tuning(self, first_chunk_rows: int = 0, growth: int = 0, cand_capacity: int = 0) -> None:
        """Launch plan of the search (0 = default); tests force the one-chunk, many-chunk and overflow paths."""
        self._tuning = _lib.FlatTuning(first_chunk_rows, growth, cand_capacity)
        if self._h is not None:
            _lib.check(_lib.lib().pr_flat_set_tuning(self._h, ctypes.byref(self._tuning)))

    def get_tuning(self) -> dict:
        t = _lib.FlatTuning()
        _lib.check(_lib.lib().pr_flat_get_tuning(self._handle(), ctypes.byref(t)))
        return {f: getattr(t, f) for f, _ in _lib.FlatTuning._fields_}

    def last_stats(self) -> dict:
        """Launches, chunks, candidates (sum and max per query and chunk) and overflow fallbacks of the last search or
        of the last pass of the last range_search (synchronises the device)."""
        if self._last is None:
            raise ValueError("no search has run on this index")
        _ws, ws_ptr, B, k = self._last
        s = _lib.FlatStats()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().pr_flat_last_stats(self._handle(), ws_ptr, B, k, ctypes.byref(s),
                                                     torch.cuda.current_stream(self.device).cuda_stream))
        return {f: getattr(s, f) for f, _ in _lib.FlatStats._fields_}

    def rows(self) -> torch.Tensor:
        """The float32 rows [ntotal, d] on the device (not a copy)."""
        return self._rows

    # ------------------------------------------------------------------ internals
    def _as_rows(self, x, what: str) -> torch.Tensor:
        return _as_rows(x, self.d, what)

    def _range_call(self, q, radius: float, lims_in, count, D, I) -> None:
        """One pr_flat_range_search: hits of query b into D, I at [lims_in[b], lims_in[b + 1]), all counts in count."""
        L = _lib.lib()
        h = self._handle()
        B = q.shape[0]
        nbytes = int(L.pr_flat_range_workspace_bytes(h, B))
        ws, ws_ptr = _aligned(nbytes, self.device)
        with torch.cuda.device(self.device):
            _lib.check(L.pr_flat_range_search(h, B, q.data_ptr(), radius, lims_in.data_ptr(), count.data_ptr(),
                                              D.data_ptr(), I.data_ptr(), ws_ptr, nbytes,
                                              torch.cuda.current_stream(self.device).cuda_stream))
        self._last = (ws, ws_ptr, B, 1)

    def _set_rows(self, rows: torch.Tensor) -> None:
        self._release()
        self._rows = rows

    def _release(self) -> None:
        if self._h is not None:
            _lib.lib().pr_flat_destroy(self._h)
        self._h, self._aux, self._last = None, None, None

    def _handle(self):
        if self._h is None:
            L = _lib.lib()
            h = ctypes.c_void_p()
            n = self.ntotal
            _lib.check(self._create(L, h, n))
            try:
                _lib.check(L.pr_flat_set_tuning(h, ctypes.byref(self._tuning)))
                nbytes = int(L.pr_flat_aux_bytes(h))
                aux, aux_ptr = _aligned(nbytes, self.device)
                with torch.cuda.device(self.device):
                    _lib.check(L.pr_flat_build_aux(h, aux_ptr, nbytes,
                                                   torch.cuda.current_stream(self.device).cuda_stream))
            except Exception:
                L.pr_flat_destroy(h)
                raise
            self._h, self._aux = h, aux
        return self._h

    def _create(self, L, h, n: int) -> int:
        return L.pr_flat_create_metric(ctypes.byref(h), self.device.index, self._rows.data_ptr() if n else None, n,
                                       self.d, self.metric_type)

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass


class IndexFlatL2(_IndexFlat):
    """faiss.IndexFlatL2 on one GPU: ``d``, ``ntotal``, ``is_trained``, ``metric_type``, ``add``, ``reset``,
    ``search``.  The float32 rows live on ``device``; a bf16 copy and the row norms (half the rows' size again) are
    built on the first search after an ``add``."""

    metric_type = METRIC_L2


class IndexFlatIP(_IndexFlat):
    """faiss.IndexFlatIP on one GPU, with the surface of IndexFlatL2.  ``search`` returns exact inner products q.x,
    descending, ties by row id, NaN after -inf; rows short of k are (-FLT_MAX, -1)."""

    metric_type = METRIC_INNER_PRODUCT


class ScalarQuantizer:
    """faiss.ScalarQuantizer's qtype numbering.  Only QT_fp16 is built; IndexScalarQuantizer raises for the others."""
    QT_8bit, QT_4bit, QT_8bit_uniform, QT_4bit_uniform, QT_fp16, QT_8bit_direct, QT_6bit, QT_bf16, \
        QT_8bit_direct_signed = range(9)


class IndexScalarQuantizer(_IndexFlat):
    """faiss.IndexScalarQuantizer(d, ScalarQuantizer.QT_fp16, metric) on one GPU: ``d``, ``ntotal``, ``is_trained``,
    ``metric_type``, ``code_size`` (2 d), ``train`` (nothing to learn for fp16), ``add``, ``reset``, ``search``,
    ``range_search``.  ``add`` encodes float32 rows to IEEE binary16 (round to nearest even, overflow to +-inf, as
    numpy's astype(float16) and faiss's F16C encoder); only the codes (2 d bytes a row) and 12 bytes of norms a row
    stay on the device.  Results are bit for bit those of IndexFlatL2 / IndexFlatIP over the decoded rows
    ``codes().float()``; the tensor-core filter reads the codes themselves."""

    def __init__(self, d: int, qtype: int, metric: int = METRIC_L2, device="cuda"):
        if qtype != ScalarQuantizer.QT_fp16:
            raise ValueError(f"qtype {qtype!r} unsupported: only ScalarQuantizer.QT_fp16 = {ScalarQuantizer.QT_fp16}")
        if metric not in _FOURCC:
            raise ValueError(f"metric {metric!r} unsupported (METRIC_L2 = 1 or METRIC_INNER_PRODUCT = 0)")
        self.metric_type = int(metric)
        self.qtype = int(qtype)
        super().__init__(d, device)
        self._rows = torch.empty((0, self.d), dtype=torch.float16, device=self.device)

    @property
    def code_size(self) -> int:
        return 2 * self.d

    def train(self, x) -> None:
        """fp16 has no trained parameters: checks x as faiss would accept it and does nothing."""
        self._as_rows(x, "x")

    def add(self, x) -> None:
        """Append float32 rows [n, d] (NumPy array or tensor), encoded to fp16 on the device in pieces, so that no
        float32 copy of the whole input is made there."""
        x = self._as_rows(x, "x")
        n = x.shape[0]
        if self.ntotal + n > 2 ** 31 - 1:
            raise ValueError("an IndexScalarQuantizer holds at most 2^31 - 1 rows")
        codes = torch.empty((self.ntotal + n, self.d), dtype=torch.float16, device=self.device)
        codes[:self.ntotal].copy_(self._rows)
        step = max(1, _COPY_BYTES // (4 * self.d))
        for a in range(0, n, step):
            codes[self.ntotal + a:self.ntotal + a + step].copy_(x[a:a + step].to(self.device).to(torch.float16))
        self._set_rows(codes)

    def reset(self) -> None:
        self._set_rows(torch.empty((0, self.d), dtype=torch.float16, device=self.device))

    def codes(self) -> torch.Tensor:
        """The fp16 codes [ntotal, d] on the device (not a copy)."""
        return self._rows

    def rows(self) -> torch.Tensor:
        """The decoded rows [ntotal, d] as a new float32 tensor on the device (4 d bytes a row)."""
        return self._rows.float()

    def _create(self, L, h, n: int) -> int:
        return L.pr_flat_create_fp16(ctypes.byref(h), self.device.index, self._rows.data_ptr() if n else None, n,
                                     self.d, self.metric_type)


# ---------------------------------------------------------------------- row-range shards over the GPUs of one box
def merge_lists(dist_lists: torch.Tensor, id_lists: torch.Tensor, bases,
                metric: int = METRIC_L2) -> tuple[torch.Tensor, torch.Tensor]:
    """pr_flat_merge_metric: ranked lists f32 / i64 [L, B, k] on one device, list l's ids offset by bases[l] -> the
    merged (D [B, k], I [B, k]) in the order of the metric's search: (distance bits, global id), short rows
    (FLT_MAX, -1); METRIC_INNER_PRODUCT: (score descending with NaN last, global id), short rows (-FLT_MAX, -1)."""
    L_, B, k = dist_lists.shape
    if tuple(id_lists.shape) != (L_, B, k) or len(bases) != L_:
        raise ValueError(f"lists {tuple(dist_lists.shape)} / {tuple(id_lists.shape)} with {len(bases)} bases")
    if dist_lists.dtype != torch.float32 or id_lists.dtype != torch.int64 or not dist_lists.is_cuda \
            or id_lists.device != dist_lists.device:
        raise ValueError("merge_lists takes float32 distances and int64 ids on one CUDA device")
    dev = dist_lists.device
    D = torch.empty((B, k), dtype=torch.float32, device=dev)
    I = torch.empty((B, k), dtype=torch.int64, device=dev)
    if B:
        base = (ctypes.c_int64 * L_)(*[int(b) for b in bases])
        dl, il = dist_lists.contiguous(), id_lists.contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().pr_flat_merge_metric(B, k, L_, dl.data_ptr(), il.data_ptr(), base, D.data_ptr(),
                                                       I.data_ptr(), torch.cuda.current_stream(dev).cuda_stream,
                                                       metric))
    return D, I


class _ShardedIndexFlat:
    """One rank's share of a row-range sharded flat index: ``shard`` (an index of the class's metric) holds the global
    rows [row_base, row_base + shard.ntotal).  One process per GPU (torchrun); every rank passes the same batch to
    ``search`` and gets the same global (D, I), equal bit for bit to one index over all rows:

        local search     pr_flat_search over this rank's rows                 [B, k] local ids
        all-gather       sharding.gather_lists                               [G, B, k], rank-major
        merge            pr_flat_merge_metric with every rank's row_base       global ids, the single index's order

    Each row is evaluated on exactly one rank, by the same exact distance or score as the single index, and the merge
    uses the single index's key order, so ties (equal values, even across shard boundaries) rank by global row id.
    ``local_search(q, k) -> (D, I)``, ``merge(D [G,B,k], I [G,B,k], bases) -> (D, I)`` and
    ``local_range(q, radius) -> (lims, D, I)`` (tensors) can be injected (the host logic is then testable on CPU with an
    oracle standing in); with them, ``shard`` only needs ``d`` and ``ntotal``.
    ``range_search`` gathers every rank's per-query counts and results and concatenates them per query in rank order
    with global ids: the ranks hold ascending contiguous row ranges, so the result is in ascending global id and equals
    one index's bit for bit.
    A shard whose ``metric_type`` is the other metric raises ValueError.
    Not supported: appending rows (``add``), writing the sharded index, one process driving several GPUs, multi-node."""

    is_trained = True
    metric_type: int

    def __init__(self, shard, row_base: int, group=None, local_search=None, merge=None, local_range=None):
        from . import sharding
        m = getattr(shard, "metric_type", self.metric_type)
        if m != self.metric_type:
            raise ValueError(f"{type(self).__name__} needs shards of metric {self.metric_type} "
                             f"({_NAME[self.metric_type]}), got a shard of metric {m}")
        self.shard, self.group = shard, group
        self.d = int(shard.d)
        self._local, self._merge, self._local_range = local_search, merge, local_range
        self._gath = {}
        self.device = getattr(shard, "device", torch.device("cpu"))
        world = sharding._world(group)
        if world > _lib.PR_FLAT_MAX_LISTS:
            raise ValueError(f"at most {_lib.PR_FLAT_MAX_LISTS} ranks can share a dense index, got {world}")
        mine = torch.tensor([int(row_base), int(shard.ntotal), self.d], dtype=torch.int64, device=self.device)
        if world > 1:
            every = torch.empty((world, 3), dtype=torch.int64, device=self.device)
            dist.all_gather_into_tensor(every.view(-1), mine, group=group)
            every = every.cpu().tolist()
        else:
            every = [mine.cpu().tolist()]
        expect = 0
        for r, (base, n, d) in enumerate(every):
            if base != expect or n < 0:
                raise ValueError(f"rank {r} holds rows [{base}, {base + n}), expected them to start at {expect}: "
                                 f"the ranks' row ranges must be contiguous, in rank order, from 0 "
                                 f"(ranges {[(b, b + m) for b, m, _ in every]})")
            if d != self.d:
                raise ValueError(f"rank {r} has d = {d}, this rank d = {self.d}")
            expect += n
        self.bases = [b for b, _, _ in every]
        self.row_base = int(row_base)
        self.ntotal = expect

    # ------------------------------------------------------------------ faiss interface
    def add(self, x) -> None:
        raise ValueError("a sharded index is read-only: appending rows would break the contiguous row ranges")

    def reset(self) -> None:
        raise ValueError("a sharded index is read-only: build a new one instead of resetting it")

    @torch.no_grad()
    def search(self, x, k: int):
        """(D, I) of the k nearest rows among ALL ranks' rows for every query of x [B, d] float32 (the same batch on
        every rank); NumPy in -> NumPy out, a CUDA tensor in -> CUDA tensors out."""
        from . import sharding
        k = _check_k(k)
        q = _queries(x, self.d, self.device if self._local is None else None)
        Dl, Il = self.shard.search(q.to(self.device), k) if self._local is None else self._local(q, k)
        B = q.shape[0]
        if B:
            key = (B, k)
            gd, gi = self._gath[key] = sharding.gather_lists(Dl, Il, self.group, self._gath.get(key))
            if len(self._gath) > 16:
                self._gath = {key: (gd, gi)}
            D, I = self._merge(gd, gi, self.bases) if self._merge else \
                merge_lists(gd, gi, self.bases, self.metric_type)
        else:
            D, I = Dl, Il
        return _like_queries(x, D, I)

    @torch.no_grad()
    def range_search(self, x, radius):
        """(lims, D, I) of IndexFlatL2.range_search over ALL ranks' rows (the same batch and radius on every rank),
        ids global and ascending per query; NumPy in -> NumPy out (lims uint64), a CUDA tensor in -> CUDA tensors
        out (lims int64)."""
        from . import sharding
        q = _queries(x, self.d, self.device if self._local_range is None else None)
        lims_l, Dl, Il = self.shard.range_search(q.to(self.device), radius) if self._local_range is None else \
            self._local_range(q, radius)
        B, dev = q.shape[0], lims_l.device
        if B == 0:
            return _like_queries(x, lims_l, Dl, Il)
        world = sharding._world(self.group)
        counts = (lims_l[1:] - lims_l[:-1]).contiguous()
        if world > 1:
            every = torch.empty((world, B), dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(every.view(-1), counts, group=self.group)
        else:
            every = counts[None]
        totals = every.sum(1)
        width = max(1, int(totals.max()))                       # every rank's results, padded to the largest
        pad_d = torch.zeros(width, dtype=torch.float32, device=dev)
        pad_i = torch.zeros(width, dtype=torch.int64, device=dev)
        pad_d[:Dl.numel()], pad_i[:Il.numel()] = Dl, Il
        gd, gi = sharding.gather_lists(pad_d[None], pad_i[None], self.group)
        gd, gi = gd.view(world, width), gi.view(world, width)
        # the results of rank g, query b go to lims[b] + (the results of ranks < g for query b)
        flat = every.reshape(-1)                                                   # (g, b) rank-major
        start_gb = torch.cumsum(flat, 0) - flat                                    # their place in the gathered order
        by_b = every.T.reshape(-1)                                                 # (b, g) query-major
        out_bg = (torch.cumsum(by_b, 0) - by_b).view(B, world).T.reshape(-1)      # their place in the output, (g, b)
        seg = torch.repeat_interleave(torch.arange(world * B, device=dev), flat)
        pos = out_bg[seg] + torch.arange(seg.numel(), device=dev) - start_gb[seg]
        keep = torch.arange(width, device=dev)[None, :] < totals[:, None]
        bases = torch.tensor(self.bases, dtype=torch.int64, device=dev)
        D = torch.empty(seg.numel(), dtype=torch.float32, device=dev)
        I = torch.empty(seg.numel(), dtype=torch.int64, device=dev)
        D[pos] = gd[keep]
        I[pos] = (gi + bases[:, None])[keep]
        lims = torch.zeros(B + 1, dtype=torch.int64, device=dev)
        torch.cumsum(every.sum(0), 0, out=lims[1:])
        return _like_queries(x, lims, D, I)

    # ------------------------------------------------------------------ project extras (this rank's shard)
    def set_tuning(self, first_chunk_rows: int = 0, growth: int = 0, cand_capacity: int = 0) -> None:
        self.shard.set_tuning(first_chunk_rows, growth, cand_capacity)

    def last_stats(self) -> dict:
        """Counters of this rank's local search in the last call (IndexFlatL2.last_stats)."""
        return self.shard.last_stats()


class ShardedIndexFlatL2(_ShardedIndexFlat):
    """Row-range shards of an IndexFlatL2 (see _ShardedIndexFlat): (distance asc, global id) order."""
    metric_type = METRIC_L2


class ShardedIndexFlatIP(_ShardedIndexFlat):
    """Row-range shards of an IndexFlatIP (see _ShardedIndexFlat): (score desc with NaN last, global id) order."""
    metric_type = METRIC_INNER_PRODUCT


# ---------------------------------------------------------------------- persistence (faiss index_write.cpp layout)
def _fourcc(path: str) -> bytes:
    with open(path, "rb") as f:
        head = f.read(4)
    if len(head) < 4:
        raise ValueError(f"{path}: not a faiss index file")
    return head


def _metric_of(path: str) -> int:
    """The metric of a flat index file from its fourcc; ValueError for any other index type."""
    head = _fourcc(path)
    for metric, fourcc in _FOURCC.items():
        if head == fourcc:
            return metric
    raise ValueError(f"{path}: index type {head!r} is not supported (only IndexFlatL2, fourcc 'IxF2', "
                     f"IndexFlatIP, fourcc 'IxFI', and IndexScalarQuantizer with QT_fp16, fourcc 'IxSQ')")


def _read_sq_header(path: str):
    """(d, ntotal, metric, codes offset) of an IndexScalarQuantizer file (faiss index_write.cpp: the index header, the
    ScalarQuantizer, the codes); ValueError unless it holds QT_fp16 codes of a supported d and metric."""
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        head = f.read(_SQ_HEADER.size)
        if len(head) < _SQ_HEADER.size:
            raise ValueError(f"{path}: truncated header")
        fourcc, d, ntotal, _, _, _, metric, qtype, _, _, sq_d, code_size, n_trained = _SQ_HEADER.unpack(head)
        if fourcc != FOURCC_SQ:
            raise ValueError(f"{path}: index type {fourcc!r} is not an IndexScalarQuantizer (fourcc 'IxSQ')")
        if qtype != ScalarQuantizer.QT_fp16:
            raise ValueError(f"{path}: qtype {qtype} is not supported (only QT_fp16 = {ScalarQuantizer.QT_fp16})")
        if metric not in _FOURCC:
            raise ValueError(f"{path}: metric_type {metric} is not supported (METRIC_L2 = 1 or METRIC_INNER_PRODUCT = 0)")
        _check_d(d)
        if sq_d != d or code_size != 2 * d or ntotal < 0:
            raise ValueError(f"{path}: ScalarQuantizer d = {sq_d}, code_size = {code_size} for an index of d = {d}")
        off = _SQ_HEADER.size + 4 * n_trained
        f.seek(off)
        raw = f.read(8)
        if len(raw) < 8:
            raise ValueError(f"{path}: truncated header")
        (nbytes,) = struct.unpack("<Q", raw)
    if nbytes != ntotal * code_size:
        raise ValueError(f"{path}: {nbytes} code bytes stored for ntotal = {ntotal}, code_size = {code_size}")
    if size < off + 8 + nbytes:
        raise ValueError(f"{path}: truncated payload")
    return d, ntotal, metric, off + 8


def read_codes(path: str) -> tuple[np.ndarray, int]:
    """(codes, metric) of an IndexScalarQuantizer(QT_fp16) file: the codes as a read-only float16 memory map
    [ntotal, d] (nothing is read yet)."""
    d, ntotal, metric, off = _read_sq_header(path)
    if ntotal == 0:
        return np.zeros((0, d), dtype=np.float16), metric
    return np.memmap(path, dtype="<f2", mode="r", offset=off, shape=(ntotal, d)), metric


def _read_header(path: str, metric: int = METRIC_L2):
    """(d, ntotal, payload offset) of a flat index file of `metric`; ValueError for any other index type or metric."""
    fourcc = _FOURCC[metric]
    head = _fourcc(path)
    if head != fourcc:
        raise ValueError(f"{path}: index type {head!r} is not supported here (only {_NAME[metric]}, "
                         f"fourcc {fourcc.decode()!r})")
    with open(path, "rb") as f:
        head = f.read(_HEADER.size)
    if len(head) < _HEADER.size:
        raise ValueError(f"{path}: truncated header")
    _, d, ntotal, _, _, _, m, count = _HEADER.unpack(head)
    if m != metric:
        raise ValueError(f"{path}: metric_type {m} is not supported in an {_NAME[metric]} file (only {metric})")
    if ntotal < 0 or count != ntotal * d:
        raise ValueError(f"{path}: {count} floats stored for ntotal = {ntotal}, d = {d}")
    if os.path.getsize(path) < _HEADER.size + 4 * count:
        raise ValueError(f"{path}: truncated payload")
    return d, ntotal, _HEADER.size


def read_rows(path: str, metric: int = METRIC_L2) -> np.ndarray:
    """The rows of an IndexFlatL2 file (an IndexFlatIP file with metric=METRIC_INNER_PRODUCT) as a read-only memory
    map [ntotal, d] (nothing is read yet)."""
    d, ntotal, off = _read_header(path, metric)
    if ntotal == 0:
        return np.zeros((0, d), dtype=np.float32)
    return np.memmap(path, dtype="<f4", mode="r", offset=off, shape=(ntotal, d))


def _my_rows(n: int, group) -> tuple[int, int]:
    """This rank's row range [lo, hi) of n rows: sharding.shard_range(n, rank, world)."""
    from . import sharding
    world = sharding._world(group)
    return sharding.shard_range(n, dist.get_rank(group) if world > 1 else 0, world)


def read_shard_rows(path: str, group=None, metric: int = METRIC_L2):
    """(row_base, rows): this rank's row range sharding.shard_range(ntotal, rank, world) of a flat index file of
    `metric`, as a read-only memory map (nothing is read yet)."""
    rows_mm = read_rows(path, metric)
    lo, hi = _my_rows(rows_mm.shape[0], group)
    return lo, rows_mm[lo:hi]


def _to_device(mm: np.ndarray, device) -> torch.Tensor:
    """A new tensor on `device` holding mm [n, d] (a memory map of float32 rows or fp16 codes), copied in pieces of
    _COPY_BYTES so that the file is never held in host RAM."""
    n, d = mm.shape
    native = mm.dtype.newbyteorder("=")
    out = torch.empty((n, d), dtype=torch.from_numpy(np.empty(0, native)).dtype, device=device)
    step = max(1, _COPY_BYTES // (native.itemsize * d))
    for a in range(0, n, step):
        out[a:a + step].copy_(torch.from_numpy(np.array(mm[a:a + step], dtype=native)))
    return out


def read_index(path: str, device="cuda", sharded: bool = False, group=None):
    """faiss.read_index for IndexFlatL2, IndexFlatIP and IndexScalarQuantizer(QT_fp16) files (the fourcc picks the
    class; the sharded classes take IndexScalarQuantizer shards of their metric): the payload is
    memory-mapped and copied to the device in pieces, so a 64 GB index is never held in host RAM (not even once).
    sharded=True (one process per GPU, torch.distributed initialised, every rank of `group` calling): each rank copies
    only its row range (read_shard_rows) and gets a ShardedIndexFlatL2 / ShardedIndexFlatIP whose search covers the
    whole file."""
    sq = _fourcc(path) == FOURCC_SQ
    if sq:
        mm, metric = read_codes(path)
    else:
        metric = _metric_of(path)
        mm = read_rows(path, metric)
    row_base, hi = _my_rows(mm.shape[0], group) if sharded else (0, mm.shape[0])
    mm = mm[row_base:hi]
    if sq:
        index = IndexScalarQuantizer(mm.shape[1], ScalarQuantizer.QT_fp16, metric, device)
    else:
        index = (IndexFlatL2 if metric == METRIC_L2 else IndexFlatIP)(mm.shape[1], device)
    index._set_rows(_to_device(mm, index.device))
    if not sharded:
        return index
    return (ShardedIndexFlatL2 if metric == METRIC_L2 else ShardedIndexFlatIP)(index, row_base, group)


def _write_pieces(f, a, dtype: str, d: int) -> None:
    """Append a [n, d] (a NumPy array, or a tensor copied to the host piece by piece) to f as `dtype`, '<f4' or '<f2',
    in pieces of _COPY_BYTES; '<f2' takes float16 input only."""
    step = max(1, _COPY_BYTES // (np.dtype(dtype).itemsize * d))
    for i in range(0, int(a.shape[0]), step):
        piece = a[i:i + step]
        if isinstance(piece, torch.Tensor):
            piece = piece.cpu().numpy()
        if dtype == "<f2" and piece.dtype != np.float16:
            raise ValueError(f"codes must be float16, got {piece.dtype}")
        f.write(np.ascontiguousarray(piece, dtype=dtype).tobytes())


def write_codes(path: str, codes, d: int, metric: int = METRIC_L2) -> None:
    """Write fp16 codes [n, d] (a float16 NumPy array, or a tensor copied to the host piece by piece) as an
    IndexScalarQuantizer(d, QT_fp16, metric) file readable by faiss.read_index."""
    if metric not in _FOURCC:
        raise ValueError(f"metric {metric!r} unsupported (METRIC_L2 = 1 or METRIC_INNER_PRODUCT = 0)")
    n = int(codes.shape[0])
    with open(path, "wb") as f:
        f.write(_SQ_HEADER.pack(FOURCC_SQ, d, n, 1 << 20, 1 << 20, 1, metric, ScalarQuantizer.QT_fp16, 0, 0.0, d,
                                2 * d, 0))
        f.write(struct.pack("<Q", n * 2 * d))
        _write_pieces(f, codes, "<f2", d)


def write_rows(path: str, rows, d: int, metric: int = METRIC_L2) -> None:
    """Write float32 rows [n, d] (NumPy array, or a tensor copied to the host piece by piece) as an IndexFlatL2 file
    (metric=METRIC_INNER_PRODUCT: an IndexFlatIP file) readable by faiss.read_index."""
    if metric not in _FOURCC:
        raise ValueError(f"metric {metric!r} unsupported (METRIC_L2 = 1 or METRIC_INNER_PRODUCT = 0)")
    n = int(rows.shape[0])
    with open(path, "wb") as f:
        f.write(_HEADER.pack(_FOURCC[metric], d, n, 1 << 20, 1 << 20, 1, metric, n * d))
        _write_pieces(f, rows, "<f4", d)


def write_index(index, path: str) -> None:
    """faiss.write_index for an IndexFlatL2, an IndexFlatIP or an IndexScalarQuantizer (QT_fp16)."""
    if isinstance(index, IndexScalarQuantizer):
        write_codes(path, index.codes(), index.d, index.metric_type)
        return
    if not isinstance(index, _IndexFlat):
        raise ValueError(f"write_index writes IndexFlatL2, IndexFlatIP and IndexScalarQuantizer only, "
                         f"got {type(index).__name__}")
    write_rows(path, index.rows(), index.d, index.metric_type)
