"""The torch restatement of the BM25 oracle (tests/bm25_torch_oracle.py), run on the CPU, against the C oracle bit
for bit: the GPU tests use it as the reference at 21M documents, where the C oracle is too slow."""
import numpy as np
import pytest
import torch

import bm25_torch_oracle as tor
from oracle import bm25_oracle as bo
from oracle import c_oracle as co
from probing_rag_b200 import synth


def csr(queries):
    qi = np.zeros(len(queries) + 1, np.int64)
    qi[1:] = np.cumsum([len(q) for q in queries])
    qt = np.array([t for q in queries for t in q], dtype=np.int32)
    return qi, qt


def check(idx, qi, qt, k, **kw):
    want_s, want_d = co.retrieve_batch(idx, qi, qt, k)
    got_s, got_d = tor.retrieve_index(idx, qi, qt, k, **kw)
    assert np.array_equal(got_d, want_d), f"ids differ in rows {np.flatnonzero((got_d != want_d).any(axis=1))[:8]}"
    assert np.array_equal(got_s.view(np.uint32), want_s.view(np.uint32)), "scores not bit-identical"
    return got_s, got_d


@pytest.fixture(scope="module")
def corpus():
    n_docs, vocab = 20_000, 1 << 14
    toks, lens = synth.corpus_np(n_docs, vocab, seed=5)
    return bo.build_index(toks, lens, vocab), vocab


@pytest.mark.parametrize("k", [1, 10, 33, 128])
def test_zipf_queries_and_transcripts(corpus, k):
    idx, vocab = corpus
    qi, qt = synth.queries_np(200, vocab, idx["df"], seed=3)
    check(idx, qi, qt, k)
    lqi, lqt = synth.queries_np(6, vocab, idx["df"], kind="later", seed=4)
    check(idx, lqi, lqt, k)


def test_small_row_and_posting_chunks(corpus, monkeypatch):
    """Row chunks of a few queries and posting chunks smaller than one term's list give the same bits."""
    idx, vocab = corpus
    qi, qt = synth.queries_np(50, vocab, idx["df"], seed=8)
    monkeypatch.setattr(tor, "POSTING_CHUNK", 1000)
    check(idx, qi, qt, 10, mem_bytes=12 * idx["num_docs"] * 7)


def test_edges():
    """Ties at the k-th score, fewer than k positive scores, empty queries, duplicate terms, k = 1 and k = PR_MAX_K."""
    rng = np.random.default_rng(1)
    base = [rng.integers(0, 12, size=int(rng.integers(2, 6))).astype(np.int32) for _ in range(6)]
    docs = [base[int(rng.integers(0, 6))].copy() for _ in range(400)]      # identical documents: exact score ties
    idx = bo.build_index(np.concatenate(docs), np.array([len(d) for d in docs]), 16)
    df = idx["df"]
    rare = int(np.flatnonzero(df > 0)[np.argmin(df[df > 0])])
    queries = [[], [rare], [rare, rare, rare], [0], [0, 0, 5, 0], [3, 7, 11, 3], list(range(12)), [15], [15, rare]]
    qi, qt = csr(queries)
    for k in (1, 7, 10, 128, 400):
        s, d = check(idx, qi, qt, k)
        assert d[0].tolist() == list(range(k)) and not s[0].any()        # empty query: the lowest ids, score 0
    assert (s[1] > 0).sum() < 128 and (s[1] > 0).sum() > 0                  # a zero-score tail behind the positives
    tie = s[:, :-1] == s[:, 1:]
    assert tie[:, :9].any()                                                # ties at the cut are really exercised


def test_doc_id_base_on_a_shard(corpus):
    idx, vocab = corpus
    toks, lens = synth.corpus_np(idx["num_docs"], vocab, seed=5)
    off = np.concatenate([[0], np.cumsum(lens, dtype=np.int64)])
    lo, hi = 7_000, 13_500
    sh = bo.build_index(toks[off[lo]:off[hi]], lens[lo:hi], vocab, n_docs_global=idx["num_docs"],
                        avgdl_global=idx["avgdl"], df_global=idx["df"], doc_id_base=lo)
    qi, qt = synth.queries_np(64, vocab, idx["df"], seed=9)
    qi, qt = np.concatenate([[0, 0], qi[1:]]), qt                          # an empty first query: tail from lo
    s, d = check(sh, qi, qt, 10)
    assert d[0].tolist() == list(range(lo, lo + 10))


def test_out_of_range_term_raises(corpus):
    idx, vocab = corpus
    with pytest.raises(ValueError):
        tor.retrieve_index(idx, np.array([0, 1], np.int64), np.array([vocab], np.int32), 10)
    with pytest.raises(ValueError):
        tor.retrieve_index(idx, np.array([0, 1], np.int64), np.array([1], np.int32), idx["num_docs"] + 1)


def test_dense_scores_equal_the_numpy_oracle(corpus):
    """The dense accumulator itself, bit for bit, including duplicate terms (one rounded add per occurrence)."""
    idx, vocab = corpus
    qi, qt = synth.queries_np(20, vocab, idx["df"], seed=12)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt))
    acc = tor.score_rows(t(idx["indptr"], np.int64), t(idx["indices"], np.int32), t(idx["data"], np.float32),
                         idx["num_docs"], t(qi, np.int64), t(qt, np.int32)).numpy()
    for r in range(20):
        want = bo.score_query(idx, qt[qi[r]:qi[r + 1]])
        assert np.array_equal(acc[r].view(np.uint32), want.view(np.uint32))
