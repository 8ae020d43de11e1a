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
the file holds.  The distances are exact (float64 evaluation in a fixed order, DESIGN §3), so they can differ from
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
FOURCC_FLAT_L2, FOURCC_FLAT_IP = b"IxF2", b"IxFI"
_FOURCC = {METRIC_L2: FOURCC_FLAT_L2, METRIC_INNER_PRODUCT: FOURCC_FLAT_IP}
_NAME = {METRIC_L2: "IndexFlatL2", METRIC_INNER_PRODUCT: "IndexFlatIP"}
_HEADER = struct.Struct("<4siqqqBiQ")     # fourcc, d, ntotal, 2 dummies, is_trained, metric_type, float count
_COPY_BYTES = 256 << 20                  # host <-> device copies of rows go in pieces of this size


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
        as_numpy = isinstance(x, np.ndarray)
        if not as_numpy:
            if not isinstance(x, torch.Tensor):
                raise ValueError(f"queries must be a NumPy array or a CUDA tensor, got {type(x).__name__}")
            if x.device != self.device:
                raise ValueError(f"queries are on {x.device}, the index on {self.device}")
        q = self._as_rows(x, "queries").to(self.device).contiguous()
        B = q.shape[0]
        D = torch.empty((B, k), dtype=torch.float32, device=self.device)
        I = torch.empty((B, k), dtype=torch.int64, device=self.device)
        if B:
            L = _lib.lib()
            h = self._handle()
            nbytes = int(L.pr_flat_workspace_bytes(h, B, k))
            ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
            ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
            with torch.cuda.device(self.device):
                _lib.check(L.pr_flat_search(h, B, q.data_ptr(), k, D.data_ptr(), I.data_ptr(), ws_ptr,
                                            nbytes, torch.cuda.current_stream(self.device).cuda_stream))
            self._last = (ws, ws_ptr, B, k)
        if as_numpy:
            return D.cpu().numpy(), I.cpu().numpy()
        return D, I

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
        """Launches, chunks, candidates (sum and max per query and chunk) and overflow fallbacks of the last search
        (synchronises the device)."""
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
            _lib.check(L.pr_flat_create_metric(ctypes.byref(h), self.device.index,
                                               self._rows.data_ptr() if n else None, n, self.d, self.metric_type))
            try:
                _lib.check(L.pr_flat_set_tuning(h, ctypes.byref(self._tuning)))
                nbytes = int(L.pr_flat_aux_bytes(h))
                aux = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
                aux_ptr = (aux.data_ptr() + 1023) // 1024 * 1024
                with torch.cuda.device(self.device):
                    _lib.check(L.pr_flat_build_aux(h, aux_ptr, nbytes,
                                                   torch.cuda.current_stream(self.device).cuda_stream))
            except Exception:
                L.pr_flat_destroy(h)
                raise
            self._h, self._aux = h, aux
        return self._h

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
    ``local_search(q, k) -> (D, I)`` and ``merge(D [G,B,k], I [G,B,k], bases) -> (D, I)`` can be injected (the host
    logic is then testable on CPU with an oracle standing in); with them, ``shard`` only needs ``d`` and ``ntotal``.
    A shard whose ``metric_type`` is the other metric raises ValueError.
    Not supported: appending rows (``add``), writing the sharded index, one process driving several GPUs, multi-node."""

    is_trained = True
    metric_type: int

    def __init__(self, shard, row_base: int, group=None, local_search=None, merge=None):
        from . import sharding
        m = getattr(shard, "metric_type", self.metric_type)
        if m != self.metric_type:
            raise ValueError(f"{type(self).__name__} needs shards of metric {self.metric_type} "
                             f"({_NAME[self.metric_type]}), got a shard of metric {m}")
        self.shard, self.group = shard, group
        self.d = int(shard.d)
        self._local, self._merge = local_search, merge
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
        as_numpy = isinstance(x, np.ndarray)
        q = _as_rows(x, self.d, "queries")
        if self._local is not None:
            Dl, Il = self._local(q, k)
        else:
            if not as_numpy and q.device != self.device:
                raise ValueError(f"queries are on {q.device}, the index on {self.device}")
            Dl, Il = self.shard.search(q.to(self.device), k)
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
        if as_numpy:
            return D.cpu().numpy(), I.cpu().numpy()
        return D, I

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
    raise ValueError(f"{path}: index type {head!r} is not supported (only IndexFlatL2, fourcc 'IxF2', and "
                     f"IndexFlatIP, fourcc 'IxFI')")


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


def read_shard_rows(path: str, group=None, metric: int = METRIC_L2):
    """(row_base, rows): this rank's row range sharding.shard_range(ntotal, rank, world) of a flat index file of
    `metric`, as a read-only memory map (nothing is read yet)."""
    from . import sharding
    rows_mm = read_rows(path, metric)
    rank = dist.get_rank(group) if sharding._world(group) > 1 else 0
    lo, hi = sharding.shard_range(rows_mm.shape[0], rank, sharding._world(group))
    return lo, rows_mm[lo:hi]


def read_index(path: str, device="cuda", sharded: bool = False, group=None):
    """faiss.read_index for IndexFlatL2 and IndexFlatIP files (the fourcc picks the class): the payload is
    memory-mapped and copied to the device in pieces, so a 64 GB index is never held in host RAM (not even once).
    sharded=True (one process per GPU, torch.distributed initialised, every rank of `group` calling): each rank copies
    only its row range (read_shard_rows) and gets a ShardedIndexFlatL2 / ShardedIndexFlatIP whose search covers the
    whole file."""
    metric = _metric_of(path)
    if sharded:
        row_base, rows_mm = read_shard_rows(path, group, metric)
    else:
        row_base, rows_mm = 0, read_rows(path, metric)
    cls, sharded_cls = (IndexFlatL2, ShardedIndexFlatL2) if metric == METRIC_L2 else (IndexFlatIP, ShardedIndexFlatIP)
    index = cls(rows_mm.shape[1], device)
    n, d = rows_mm.shape
    rows = torch.empty((n, d), dtype=torch.float32, device=index.device)
    step = max(1, _COPY_BYTES // (4 * d))
    for a in range(0, n, step):
        rows[a:a + step].copy_(torch.from_numpy(np.array(rows_mm[a:a + step], dtype=np.float32)))
    index._set_rows(rows)
    return sharded_cls(index, row_base, group) if sharded else index


def write_rows(path: str, rows, d: int, metric: int = METRIC_L2) -> None:
    """Write float32 rows [n, d] (NumPy array, or a tensor copied to the host piece by piece) as an IndexFlatL2 file
    (metric=METRIC_INNER_PRODUCT: an IndexFlatIP file) readable by faiss.read_index."""
    if metric not in _FOURCC:
        raise ValueError(f"metric {metric!r} unsupported (METRIC_L2 = 1 or METRIC_INNER_PRODUCT = 0)")
    n = int(rows.shape[0])
    with open(path, "wb") as f:
        f.write(_HEADER.pack(_FOURCC[metric], d, n, 1 << 20, 1 << 20, 1, metric, n * d))
        step = max(1, _COPY_BYTES // (4 * d))
        for a in range(0, n, step):
            piece = rows[a:a + step]
            if isinstance(piece, torch.Tensor):
                piece = piece.cpu().numpy()
            f.write(np.ascontiguousarray(piece, dtype="<f4").tobytes())


def write_index(index, path: str) -> None:
    """faiss.write_index for an IndexFlatL2 or an IndexFlatIP."""
    if not isinstance(index, _IndexFlat):
        raise ValueError(f"write_index writes IndexFlatL2 and IndexFlatIP only, got {type(index).__name__}")
    write_rows(path, index.rows(), index.d, index.metric_type)
