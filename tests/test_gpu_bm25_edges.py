"""Edges of the BM25 scoring kernel and of the shard merge, against the C oracle bit for bit.  Needs a B200.

- live peer bounds (pr_index_set_peer_thetas) between G doc-range shards on ONE device, racing on their own streams,
  over call sequences whose batches change from call to call (a bound left over from an earlier call must never
  survive into a later one);
- query lengths around the warp's cursor scratch (kCursorCap = 1024 terms) and far beyond;
- weights on either side of the range in which large batches run the four-epoch variant, and queries on either side
  of the term-count limit of that variant;
- pr_topk_merge against oracle.bm25_oracle.merge_topk.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import bm25_oracle as bo
from oracle import c_oracle as co
from probing_rag_b200 import synth

from test_gpu_bm25 import assert_parity, gpu_index, run_gpu, to_dev, tune

pytestmark = pytest.mark.gpu

# one plan per family: small-batch (REFRESH) and large-batch two- and four-epoch variants, one launch and many
PLANS = [
    dict(),
    dict(batch_variant=1, subs_per_item=24, docs_per_launch=49152, min_items=1),
    dict(batch_variant=1, subs_per_item=5, warps_per_cta=12, docs_per_launch=1000000, min_items=100000),
    dict(batch_variant=2, tile_epochs=2, subs_per_item=4, docs_per_launch=16384, min_items=1),
    dict(batch_variant=2, tile_epochs=2, docs_per_launch=1000000, min_items=100000),
    dict(batch_variant=2, subs_per_item=3, docs_per_launch=16384, min_items=1),
    dict(batch_variant=2, subs_per_item=24, warps_per_cta=8, docs_per_launch=1000000, min_items=100000),
]


def csr(queries):
    qi = np.zeros(len(queries) + 1, np.int64)
    qi[1:] = np.cumsum([len(q) for q in queries])
    qt = np.array([t for q in queries for t in q], dtype=np.int32) if len(queries) else np.zeros(0, np.int32)
    return qi, qt


def lean_variants(gi, qi, qt, k):
    """The VAR template argument of every scoring kernel one call launches (bm25_lean_kernel<NW, E, VAR>)."""
    from torch.profiler import ProfilerActivity, profile
    d_qi, d_qt = to_dev(gi, qi, qt)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gi.topk(d_qi, d_qt, k)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "bm25_lean_kernel<" in e.name}
    assert names, "no scoring kernel in the profile"
    return {int(n.split("bm25_lean_kernel<")[1].split(">")[0].split(",")[2]) for n in names}


# ----------------------------------------------------------------------------- live peer bounds on one device
def shard_cuts(n_docs, g, rng):
    """g unequal doc ranges covering [0, n_docs), one of them empty."""
    inner = np.sort(rng.choice(np.arange(1, n_docs), size=g - 2, replace=False))
    empty_at = int(rng.integers(0, g - 1))
    cuts = np.concatenate([[0], inner[:empty_at], [inner[empty_at - 1] if empty_at else 0], inner[empty_at:], [n_docs]])
    return [(int(cuts[i]), int(cuts[i + 1])) for i in range(g)]


def build_range_shards(small_corpus, ranges):
    idx, toks, lens = small_corpus["index"], small_corpus["tokens"], small_corpus["doc_lens"]
    off = np.concatenate([[0], np.cumsum(lens, dtype=np.int64)])
    n_docs = len(lens)
    out = []
    for lo, hi in ranges:
        sh = bo.build_index(toks[off[lo]:off[hi]], lens[lo:hi], small_corpus["vocab"], n_docs_global=n_docs,
                            avgdl_global=idx["avgdl"], df_global=idx["df"], doc_id_base=lo)
        out.append(gpu_index(sh, n_docs_global=n_docs, doc_id_base=lo))
    return out


class PeerShards:
    """G shards on one device sharing live bounds: each owns a 2 x capacity float array from torch and raises the
    others' arrays (plain device pointers: the raise is a red.sys on an address)."""

    def __init__(self, shards, capacity):
        from probing_rag_b200 import _lib
        self.L, self.shards, self.capacity = _lib.lib(), shards, capacity
        self.local = [torch.empty(2 * capacity, dtype=torch.float32, device="cuda") for _ in shards]
        self.tables = [torch.zeros(2 * _lib.PR_MAX_PEERS, dtype=torch.int64, device="cuda") for _ in shards]
        self.streams = [torch.cuda.Stream() for _ in shards]
        for i, gi in enumerate(shards):
            peers = [self.local[j].data_ptr() for j in range(len(shards)) if j != i]
            bases = (ctypes.c_void_p * max(len(peers), 1))(*peers)
            _lib.check(self.L.pr_index_set_peer_thetas(gi._handle, self.local[i].data_ptr(), capacity, len(peers), bases,
                                                       self.tables[i].data_ptr()))

    def close(self):
        torch.cuda.synchronize()
        for gi in self.shards:
            self.L.pr_index_set_peer_thetas(gi._handle, None, 0, 0, None, None)

    def topk(self, qi, qt, k, union_rounds=0):
        """One call on every shard, each on its own stream (they race), then the merge.  With union_rounds > 0 the
        shards go launch by launch for that many launches, and behind each the running lists are stacked (the
        all-gather) and every bound raised to the k-th largest score of the union (pr_bm25_raise_union_bound)."""
        from probing_rag_b200 import _lib, merge_topk
        L, nq = self.L, len(qi) - 1
        d_qi, d_qt = to_dev(self.shards[0], qi, qt)
        torch.cuda.synchronize()
        outs, args, ws_all, n_launch = [], [], [], []
        for gi in self.shards:
            out = (torch.empty((nq, k), dtype=torch.float32, device="cuda"), torch.empty((nq, k), dtype=torch.int32, device="cuda"))
            ws = gi._workspace(nq, k)
            outs.append(out)
            ws_all.append(ws)
            n_launch.append(gi.num_launches(nq, k))
            args.append((gi._handle, nq, d_qi.data_ptr(), d_qt.data_ptr() if d_qt.numel() else None, d_qt.numel(), k,
                         out[0].data_ptr(), out[1].data_ptr(), ws.data_ptr(), ws.numel()))
        rounds = min(union_rounds, max(n_launch) - 1)
        done = [0] * len(self.shards)
        for r in range(rounds):
            for i, (gi, st) in enumerate(zip(self.shards, self.streams)):
                if done[i] < n_launch[i]:
                    _lib.check(L.pr_bm25_topk_range(*args[i], done[i], done[i] + 1, st.cuda_stream))
                    done[i] += 1
            torch.cuda.synchronize()
            runs = []
            for gi, ws in zip(self.shards, ws_all):
                off = int(L.pr_bm25_running_scores_offset(gi._handle, nq, k))
                runs.append(ws[off:off + 4 * nq * k].view(torch.float32).view(nq, k))
            gathered = torch.stack(runs).contiguous()
            for i, gi in enumerate(self.shards):
                if done[i] < n_launch[i]:
                    _lib.check(L.pr_bm25_raise_union_bound(gi._handle, nq, k, gathered.data_ptr(), len(runs), ws_all[i].data_ptr(),
                                                           ws_all[i].numel(), torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
        for i, st in enumerate(self.streams):
            if done[i] < n_launch[i]:
                _lib.check(L.pr_bm25_topk_range(*args[i], done[i], n_launch[i], st.cuda_stream))
        torch.cuda.synchronize()                     # stands in for the all-gather: every shard has finished the call
        ms, md = merge_topk(torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs]))
        torch.cuda.synchronize()
        return ms.cpu().numpy(), md.cpu().numpy()


def call_sequence(small_corpus):
    """Two batches that differ: A = transcript-sized queries (high scores, high bounds), B = round-0 queries.  The
    third call (B) follows the first (A) two calls later: a bound of A left in the other half of the peer arrays would
    cut B's documents."""
    idx, vocab = small_corpus["index"], small_corpus["vocab"]
    a = synth.queries_np(256, vocab, idx["df"], kind="later", seed=31)
    b = synth.queries_np(256, vocab, idx["df"], seed=32)

    def head(batch, n):
        qi, qt = batch
        return qi[:n + 1], qt[:qi[n]]
    return [(a, 10), (b, 100), (b, 10), (head(b, 1), 10), (head(a, 64), 128), (b, 10), (a, 33)]


@pytest.mark.parametrize("union_rounds", [0, 3])
@pytest.mark.parametrize("g", [2, 5, 16])
def test_live_peer_bounds_between_racing_shards_over_changing_batches(small_corpus, g, union_rounds):
    rng = np.random.default_rng(100 + g)
    ranges = shard_cuts(small_corpus["index"]["num_docs"], g, rng)
    sizes = [hi - lo for lo, hi in ranges]
    assert sizes.count(0) == 1 and len(set(sizes)) > min(g - 1, 2)
    shards = build_range_shards(small_corpus, ranges)
    for gi in shards:
        tune(gi, batch_variant=2, subs_per_item=2, docs_per_launch=8192, min_items=1)
    ps = PeerShards(shards, 256)
    try:
        seq = call_sequence(small_corpus)
        for (qi, qt), k in seq:
            got_s, got_d = ps.topk(qi, qt, k, union_rounds)
            want_s, want_d = co.retrieve_batch(small_corpus["index"], qi, qt, k, n_threads=8)
            assert_parity(got_s, got_d, want_s, want_d)
        # the small-batch variant (REFRESH: re-reads the bound in front of tile scans) over the same sequence
        for gi in shards:
            tune(gi, batch_variant=1, subs_per_item=4, docs_per_launch=16384, min_items=1)
        for (qi, qt), k in seq[:4]:
            got_s, got_d = ps.topk(qi, qt, k, union_rounds)
            want_s, want_d = co.retrieve_batch(small_corpus["index"], qi, qt, k, n_threads=8)
            assert_parity(got_s, got_d, want_s, want_d)
    finally:
        ps.close()


# ----------------------------------------------------------------------------- query length
def long_queries(idx, rng):
    """Queries of 32, 33, 1,023, 1,024, 1,025, 2,048 and 5,000 terms drawn from the corpus vocabulary, and queries
    of a few terms repeated many times."""
    known = np.flatnonzero(idx["df"] > 0)
    p = idx["df"][known] / idx["df"][known].sum()
    out = [rng.choice(known, size=n, p=p).astype(np.int32).tolist() for n in (32, 33, 1023, 1024, 1025, 2048, 5000)]
    few = rng.choice(known, size=3, p=p).astype(np.int32)
    out += [np.tile(few, 700).tolist(), [int(few[0])] * 1025, np.repeat(few, 400).tolist()]
    return out


def test_query_length_around_the_cursor_scratch(small_corpus):
    idx = small_corpus["index"]
    gi = gpu_index(idx)
    qi, qt = csr(long_queries(idx, np.random.default_rng(7)))
    assert {32, 33, 1023, 1024, 1025, 2048, 5000} <= set(np.diff(qi).tolist())
    for k in (10, 100):
        want_s, want_d = co.retrieve_batch(idx, qi, qt, k, n_threads=8)
        for plan in PLANS:
            tune(gi, **plan)
            got_s, got_d = run_gpu(gi, qi, qt, k)
            assert_parity(got_s, got_d, want_s, want_d)


# ----------------------------------------------------------------------------- four-epoch limits
def scaled_index(small_corpus, wmin, wmax):
    """The corpus index with its weights mapped affinely onto [wmin, wmax] (both ends taken exactly)."""
    idx = dict(small_corpus["index"])
    d = idx["data"].astype(np.float64)
    lo, hi = d.min(), d.max()
    data = (np.float64(wmin) + (d - lo) * ((np.float64(wmax) - np.float64(wmin)) / (hi - lo))).astype(np.float32)
    data[np.argmin(d)], data[np.argmax(d)] = np.float32(wmin), np.float32(wmax)
    idx["data"] = data
    return idx


@pytest.mark.parametrize("wmin,wmax,four", [
    (2.0 ** -30, 256.0, True),
    (np.float32(2.0 ** -30) * np.float32(1 - 2.0 ** -24), 256.0, False),
    (2.0 ** -30, np.float32(256.0) * np.float32(1 + 2.0 ** -23), False),
])
def test_weights_on_the_four_epoch_edges(small_corpus, wmin, wmax, four):
    idx = scaled_index(small_corpus, wmin, wmax)
    assert idx["data"].min() == np.float32(wmin) and idx["data"].max() == np.float32(wmax)
    gi = gpu_index(idx)
    qi, qt = small_corpus["q_indptr"][:129], small_corpus["q_terms"]
    lqi, lqt = synth.queries_np(24, small_corpus["vocab"], idx["df"], kind="later", seed=41)
    for plan in PLANS:
        tune(gi, **plan)
        for q_i, q_t in ((qi, qt), (lqi, lqt)):
            want_s, want_d = co.retrieve_batch(idx, q_i, q_t, 10, n_threads=8)
            got_s, got_d = run_gpu(gi, q_i, q_t, 10)
            assert_parity(got_s, got_d, want_s, want_d)
    tune(gi, batch_variant=2, subs_per_item=3, docs_per_launch=16384, min_items=1)
    assert lean_variants(gi, qi, qt, 10) == ({0, 2} if four else {0})


def epoch_corpus(n_docs=60_000, seed=3):
    """Term 0: weight 256 in one document of every sub-tile (offset 5); term 1: tiny weights (2^-30 and a few
    larger) in every document; term 2: one weight-1 posting per sub-tile at offset 5 of later sub-tiles; the other
    terms: random small weights.  A query of term 0 repeated n times gives offset-5 sums of 256 n, the stale words
    the four-epoch accumulation must shed."""
    rng = np.random.default_rng(seed)
    n_sub = -(-n_docs // 2048)
    cols = {0: (np.arange(n_sub) * 2048 + 5, np.full(n_sub, 256.0)),
            1: (np.arange(n_docs), np.where(rng.random(n_docs) < 0.9, 2.0 ** -30, rng.uniform(2.0 ** -20, 1.0, n_docs))),
            2: (np.arange(1, n_sub, 3) * 2048 + 5, np.ones(len(range(1, n_sub, 3))))}
    for t in range(3, 40):
        docs = np.sort(rng.choice(n_docs, size=int(rng.integers(50, 3000)), replace=False))
        cols[t] = (docs, rng.uniform(0.5, 8.0, len(docs)))
    indptr = np.zeros(41, np.int64)
    indptr[1:] = np.cumsum([len(cols[t][0]) if t in cols else 0 for t in range(40)])
    indices = np.concatenate([cols[t][0] for t in range(40)]).astype(np.int32)
    data = np.concatenate([cols[t][1] for t in range(40)]).astype(np.float32)
    data[indptr[1]] = np.float32(2.0 ** -30)
    return {"data": data, "indices": indices, "indptr": indptr, "num_docs": n_docs}


def test_queries_on_either_side_of_the_four_epoch_term_limit():
    """At max weight 256 a query of 65,535 terms still runs four epochs, 65,536 run two.  One weight-256 term repeated
    that often builds stale tile words close to 2^24; tiny weights land on top of them in the scaled epochs."""
    idx = epoch_corpus()
    gi = gpu_index(idx)
    rng = np.random.default_rng(5)
    queries = []
    for n in (65_535, 65_536, 40_000):
        q = [0] * n
        for t, pos in ((1, n // 3), (2, n // 2), (int(rng.integers(3, 40)), 7)):
            q[pos] = t
        queries.append(q)
    queries += [[1, 2] + list(rng.integers(3, 40, size=30)) for _ in range(40)]       # short queries beside them
    qi, qt = csr(queries)
    for k in (1, 10, 100):
        want_s, want_d = co.retrieve_batch(idx, qi, qt, k, n_threads=8)
        for plan in PLANS:
            tune(gi, **plan)
            got_s, got_d = run_gpu(gi, qi, qt, k)
            assert_parity(got_s, got_d, want_s, want_d)
    tune(gi, batch_variant=2, subs_per_item=3, docs_per_launch=16384, min_items=1)
    assert 2 in lean_variants(gi, qi, qt, 10)


def test_zero_score_tail_in_four_epoch_items():
    """Queries with fewer than k positive documents in items that ran four epochs behind a skipped sub-tile: the
    zero-score tail is the lowest ids, never a document holding dust of an earlier sub-tile's sums."""
    idx = epoch_corpus()
    gi = gpu_index(idx)
    few = np.flatnonzero(np.diff(idx["indptr"]) <= 60)
    queries = [[0] * 4096 + [int(t)] for t in few] + [[2] * 3, [0] * 30_000, [2, 0, 2]]
    queries += [[int(t)] for t in range(3, 40)]
    qi, qt = csr(queries)
    for k in (10, 100, 128):
        want_s, want_d = co.retrieve_batch(idx, qi, qt, k, n_threads=8)
        assert k == 10 or (want_s == 0).any(axis=1).sum() >= 5            # zero-score tails behind few positives
        for plan in PLANS:
            tune(gi, **plan)
            got_s, got_d = run_gpu(gi, qi, qt, k)
            assert_parity(got_s, got_d, want_s, want_d)


# ----------------------------------------------------------------------------- pr_topk_merge
def shard_like_lists(rng, g, nq, k, n_docs=1 << 20):
    """[g, nq, k] ranked lists as doc-range shards return them: each list in canonical order over its own id range,
    scores from a small set (exact ties across lists), zero-score tails, padding (-1, -1) or (-inf, -1) at the end,
    and at least k valid entries per query over all lists."""
    per = n_docs // g
    levels = np.array([0.0, 0.5, 1.0, 1.25, 3.0, 7.5, 1e-30, 2.0 ** -30], np.float32)
    s = np.full((g, nq, k), -1.0, np.float32)
    d = np.full((g, nq, k), -1, np.int32)
    n_valid = rng.integers(0, k + 1, size=(g, nq))
    short = n_valid.sum(axis=0) < k
    n_valid[0, short] = k
    for gi_ in range(g):
        for q in range(nq):
            n = int(n_valid[gi_, q])
            if n == 0:
                continue
            sc = np.sort(levels[rng.integers(0, len(levels), size=n)])[::-1]
            ids = np.sort(rng.choice(per, size=n, replace=False)) + gi_ * per
            o = np.lexsort((ids, -sc.astype(np.float64)))
            s[gi_, q, :n], d[gi_, q, :n] = sc[o], ids[o]
            if rng.random() < 0.3:
                s[gi_, q, n:] = -np.inf
    return s, d


@pytest.mark.parametrize("g", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("k", [1, 10, 32, 33, 100, 128])
def test_topk_merge_against_the_oracle_merge(g, k):
    from probing_rag_b200 import merge_topk
    rng = np.random.default_rng(g * 1000 + k)
    s, d = shard_like_lists(rng, g, 300, k)
    want_s, want_d = bo.merge_topk(s, d, k)
    got_s, got_d = merge_topk(torch.from_numpy(s).cuda(), torch.from_numpy(d).cuda())
    torch.cuda.synchronize()
    assert_parity(got_s.cpu().numpy(), got_d.cpu().numpy(), want_s, want_d)


def test_topk_merge_of_a_full_size_batch():
    from probing_rag_b200 import merge_topk
    rng = np.random.default_rng(77)
    for g, nq, k in ((4, 65536, 10), (16, 4096, 128)):
        s, d = shard_like_lists(rng, g, nq, k)
        want_s, want_d = bo.merge_topk(s, d, k)
        got_s, got_d = merge_topk(torch.from_numpy(s).cuda(), torch.from_numpy(d).cuda())
        torch.cuda.synchronize()
        assert_parity(got_s.cpu().numpy(), got_d.cpu().numpy(), want_s, want_d)
