"""`oracle.bm25_oracle.score_query` + `topk_canonical` restated in torch, so that the reference lists of a
21M-document index can be computed on the GPU (the C oracle does a few hundred queries per second on a host).

Scoring: one dense f32 accumulator row per query.  The queries of a row chunk are batched by token position: at
position j every query whose length exceeds j adds the postings of its j-th term to its own row, in query order,
duplicates counted each time.  Inside one position the flat targets row * n_docs + doc are distinct (one term's
postings name distinct documents, each query owns its row), so `index_add_` performs exactly one rounded f32 add per
element -- the oracle's `np.add.at` order, bit for bit.

Selection: scores are >= +0, so the int64 key (score_bits << 32) | (0xFFFFFFFF - doc) orders by score descending,
then doc id ascending, and a row with fewer than k positive scores is filled with the lowest-id zero-score documents:
`torch.topk` of the key is the canonical order exactly.

Peak memory: 12 bytes per (row, document) for the accumulator and the keys (at most `mem_bytes`, see `rows_per_chunk`)
plus about 40 bytes per gathered posting, at most `POSTING_CHUNK` postings at a time (~1.3 GB).
"""
from __future__ import annotations

import numpy as np
import torch

POSTING_CHUNK = 1 << 25
MEM_BYTES = 16 << 30


def rows_per_chunk(n_docs: int, mem_bytes: int = MEM_BYTES) -> int:
    return max(1, int(mem_bytes // (12 * max(n_docs, 1))))


def score_rows(indptr: torch.Tensor, doc_ids: torch.Tensor, weights: torch.Tensor, n_docs: int,
               q_indptr: torch.Tensor, q_terms: torch.Tensor) -> torch.Tensor:
    """Dense f32 scores [B, n_docs] of the B queries of the CSR batch (q_indptr int64[B+1], q_terms)."""
    dev = weights.device
    q_indptr = q_indptr.to(dev, torch.int64)
    q_terms = q_terms.to(dev, torch.int64)
    nq = q_indptr.numel() - 1
    acc = torch.zeros((nq, n_docs), dtype=torch.float32, device=dev)
    flat = acc.view(-1)
    starts, lens = q_indptr[:-1], q_indptr[1:] - q_indptr[:-1]
    n_terms = indptr.numel() - 1
    if q_terms.numel() and (int(q_terms.min()) < 0 or int(q_terms.max()) >= n_terms):
        raise ValueError(f"query token id out of range [0, {n_terms})")
    max_len = int(lens.max()) if nq else 0
    rows_all = torch.arange(nq, device=dev)
    for j in range(max_len):
        act = rows_all[lens > j]
        t = q_terms[starts[act] + j]
        p0, cnt = indptr[t], indptr[t + 1] - indptr[t]
        # split the position's queries into groups of at most POSTING_CHUNK postings (one query never splits: its
        # postings alone may exceed the bound, which only costs memory)
        csum = torch.cumsum(cnt, 0)
        bounds = [0]
        total = int(csum[-1]) if csum.numel() else 0
        if total > POSTING_CHUNK:
            cuts = torch.searchsorted(csum, torch.arange(POSTING_CHUNK, total, POSTING_CHUNK, device=dev), right=True)
            bounds += sorted(set(int(c) for c in cuts.tolist()) - {0})
        bounds.append(act.numel())
        for a, b in zip(bounds[:-1], bounds[1:]):
            if b <= a:
                continue
            c = cnt[a:b]
            n = int(c.sum())
            if n == 0:
                continue
            first = torch.repeat_interleave(torch.cumsum(c, 0) - c, c)
            pos = torch.arange(n, device=dev) - first + torch.repeat_interleave(p0[a:b], c)
            tgt = torch.repeat_interleave(act[a:b], c) * n_docs + doc_ids[pos].to(torch.int64)
            flat.index_add_(0, tgt, weights[pos])
    return acc


def topk_rows(scores: torch.Tensor, k: int, doc_id_base: int = 0):
    """Canonical top-k of every row of a dense [B, n] f32 score matrix -> (scores f32[B,k], ids i32[B,k])."""
    n = scores.shape[1]
    if k > n:
        raise ValueError(f"k of {k} is larger than the number of documents {n}")
    key = scores.view(torch.int32).to(torch.int64) << 32
    key |= 0xFFFFFFFF - torch.arange(n, dtype=torch.int64, device=scores.device)
    top = torch.topk(key, k, dim=1, sorted=True).values
    del key
    s = (top >> 32).to(torch.int32).view(torch.float32)
    d = (0xFFFFFFFF - (top & 0xFFFFFFFF) + doc_id_base).to(torch.int32)
    return s, d


def retrieve_batch(indptr, doc_ids, weights, n_docs: int, q_indptr, q_terms, k: int, doc_id_base: int = 0,
                   rows=None, mem_bytes: int = MEM_BYTES):
    """Canonical top-k lists of the queries `rows` (default: all) of a host CSR batch, as host arrays
    (scores f32[R,k], ids i32[R,k]); same contract as `oracle.c_oracle.retrieve_batch`.  The index arrays are
    torch tensors on the device the reference runs on."""
    q_indptr = np.asarray(q_indptr, dtype=np.int64)
    q_terms = np.asarray(q_terms, dtype=np.int32)
    nq = len(q_indptr) - 1
    rows = np.arange(nq) if rows is None else np.asarray(rows, dtype=np.int64)
    if k > n_docs:
        raise ValueError(f"k of {k} is larger than the number of documents {n_docs}")
    out_s = np.zeros((len(rows), k), np.float32)
    out_d = np.zeros((len(rows), k), np.int32)
    step = rows_per_chunk(n_docs, mem_bytes)
    for c0 in range(0, len(rows), step):
        sel = rows[c0:c0 + step]
        lens = q_indptr[sel + 1] - q_indptr[sel]
        qi = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        qt = np.concatenate([q_terms[q_indptr[r]:q_indptr[r + 1]] for r in sel]) if len(sel) else np.zeros(0, np.int32)
        acc = score_rows(indptr, doc_ids, weights, n_docs, torch.from_numpy(qi), torch.from_numpy(qt.astype(np.int32)))
        s, d = topk_rows(acc, k, doc_id_base)
        del acc
        out_s[c0:c0 + len(sel)] = s.cpu().numpy()
        out_d[c0:c0 + len(sel)] = d.cpu().numpy()
    return out_s, out_d


def retrieve_index(index: dict, q_indptr, q_terms, k: int, device="cpu", **kw):
    """`retrieve_batch` over an oracle index dict (data / indices / indptr / num_docs / doc_id_base)."""
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(device)
    return retrieve_batch(t(index["indptr"], np.int64), t(index["indices"], np.int32), t(index["data"], np.float32),
                          int(index["num_docs"]), q_indptr, q_terms, k, int(index.get("doc_id_base", 0)), **kw)
