"""Seeded synthetic "DPR-Wikipedia-shaped" corpus and query generator (SURVEY 8d).

No dataset can be downloaded here, so the benchmark and the parity tests run on a
Zipf-Mandelbrot corpus of the named shape:

  docs      N = 100,000 (config 1) or 21,015,324 (= DPR psgs_w100, download/download.sh:20)
  length    clip(round(Normal(70, 12)), 8, 128) post-stop-word tokens
  vocab     V = 2^20 (config 1) / 2^22; token rank r ~ p(r) ∝ (r + 30)^-1.1, term id = rank
  queries   round 0: clip(1 + Poisson(5), 1, 32) terms iid from p(r), df==0 terms dropped,
            duplicates kept (bm25s query semantics, SURVEY App. A.5);
            later rounds: clip(Normal(350, 100), 64, 1024) terms (LM transcript, exp_rag.py:457)

Everything is generated in fixed blocks of DOC_BLOCK documents, each with its own seed,
so a doc-range shard holds exactly the documents the single index holds for that range.
"""
from __future__ import annotations

import functools

import numpy as np
import torch

N_DOCS_WIKI = 21_015_324
ZM_Q = 30.0
ZM_S = 1.1
DOC_LEN_MEAN, DOC_LEN_STD, DOC_LEN_MIN, DOC_LEN_MAX = 70.0, 12.0, 8, 128
DOC_BLOCK = 1 << 18
CORPUS_SEED = 1234
QUERY_SEED = 4321


@functools.lru_cache(maxsize=4)
def zipf_mandelbrot_cdf(vocab: int) -> np.ndarray:
    r = np.arange(vocab, dtype=np.float64)
    p = (r + ZM_Q) ** (-ZM_S)
    cdf = np.cumsum(p)
    cdf /= cdf[-1]
    cdf[-1] = 1.0
    return cdf


# ----------------------------------------------------------------------------- numpy (CPU)
def corpus_block_np(block: int, n_docs_total: int, cdf: np.ndarray, seed: int = CORPUS_SEED):
    """Token ids and doc lengths of docs [block*DOC_BLOCK, min((block+1)*DOC_BLOCK, N))."""
    lo = block * DOC_BLOCK
    n = max(0, min(DOC_BLOCK, n_docs_total - lo))
    rng = np.random.default_rng([seed, block])
    lens = np.clip(np.rint(rng.normal(DOC_LEN_MEAN, DOC_LEN_STD, size=n)), DOC_LEN_MIN, DOC_LEN_MAX)
    lens = lens.astype(np.int32)
    u = rng.random(int(lens.sum()))
    tokens = np.searchsorted(cdf, u, side="right").astype(np.int32)
    np.minimum(tokens, len(cdf) - 1, out=tokens)
    return tokens, lens


def corpus_np(n_docs: int, vocab: int, seed: int = CORPUS_SEED, doc_lo: int = 0, doc_hi: int | None = None):
    """(tokens, doc_lens) for docs [doc_lo, doc_hi) of the n_docs-document corpus."""
    doc_hi = n_docs if doc_hi is None else doc_hi
    cdf = zipf_mandelbrot_cdf(vocab)
    toks, lens = [], []
    for blk in range(doc_lo // DOC_BLOCK, (max(doc_hi, 1) - 1) // DOC_BLOCK + 1):
        t, l = corpus_block_np(blk, n_docs, cdf, seed)
        b_lo = blk * DOC_BLOCK
        s, e = max(doc_lo - b_lo, 0), min(doc_hi - b_lo, len(l))
        if e <= s:
            continue
        off = np.concatenate([[0], np.cumsum(l, dtype=np.int64)])
        toks.append(t[off[s]:off[e]])
        lens.append(l[s:e])
    if not toks:
        return np.zeros(0, np.int32), np.zeros(0, np.int32)
    return np.concatenate(toks), np.concatenate(lens)


def queries_np(n_queries: int, vocab: int, df: np.ndarray | None = None, seed: int = QUERY_SEED,
               kind: str = "round0"):
    """CSR query batch (q_indptr i64[B+1], q_terms i32[nnz]).  `df` (global document
    frequencies) drops terms unknown to the corpus, as bm25s does on the query side."""
    cdf = zipf_mandelbrot_cdf(vocab)
    rng = np.random.default_rng([seed, 0 if kind == "round0" else 1])
    if kind == "round0":
        lens = np.clip(1 + rng.poisson(5.0, size=n_queries), 1, 32)
    elif kind == "later":
        lens = np.clip(np.rint(rng.normal(350.0, 100.0, size=n_queries)), 64, 1024)
    else:
        raise ValueError(kind)
    lens = lens.astype(np.int64)
    u = rng.random(int(lens.sum()))
    terms = np.minimum(np.searchsorted(cdf, u, side="right"), vocab - 1).astype(np.int32)
    qid = np.repeat(np.arange(n_queries), lens)
    if df is not None:
        keep = np.asarray(df)[terms] > 0
        terms, qid = terms[keep], qid[keep]
    q_indptr = np.zeros(n_queries + 1, dtype=np.int64)
    np.cumsum(np.bincount(qid, minlength=n_queries), out=q_indptr[1:])
    return q_indptr, terms


# ----------------------------------------------------------------------------- torch (GPU)
def _block_generator(device, seed: int, block: int) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed((seed << 24) ^ (block * 2654435761 % (1 << 24)) ^ (block << 1))
    return g


def corpus_block_torch(block: int, n_docs_total: int, cdf_t: torch.Tensor, seed: int = CORPUS_SEED):
    """Same shape as `corpus_block_np` but generated on `cdf_t.device` with torch's RNG
    (a different, equally seeded stream: the 21M corpus never exists on the host)."""
    dev = cdf_t.device
    lo = block * DOC_BLOCK
    n = max(0, min(DOC_BLOCK, n_docs_total - lo))
    g = _block_generator(dev, seed, block)
    lens = torch.randn(n, generator=g, device=dev, dtype=torch.float32) * DOC_LEN_STD + DOC_LEN_MEAN
    lens = torch.clamp(torch.round(lens), DOC_LEN_MIN, DOC_LEN_MAX).to(torch.int32)
    total = int(lens.sum().item())
    u = torch.rand(total, generator=g, device=dev, dtype=torch.float64)
    tokens = torch.searchsorted(cdf_t, u, right=True).clamp_(max=cdf_t.numel() - 1).to(torch.int32)
    return tokens, lens


# ----------------------------------------------------------------------------- prober workload (BASELINE config 4)
D_MODEL = 2048                          # gemma-2b d_model (Config_Maker, /root/reference/utils.py:288)
HIDDEN = 512                            # ImprovedProbe default hidden_size (utils.py:30)
N_CLASSES = 2                           # Config_Maker.num_classes (utils.py:290)
PROBE_LAYERS = tuple(range(6, 17, 2))   # exp_rag.py:311


def make_prober_state(seed: int, d_model: int = D_MODEL, hidden: int = HIDDEN,
                      trained_like: bool = True) -> dict:
    """Deterministic synthetic checkpoint (no trained checkpoints are shipped, SURVEY 8d).
    numpy PCG64 streams, so the same tensors regenerate on any box; LayerNorm affine
    parameters are perturbed away from (1, 0) so they are exercised."""
    rng = np.random.default_rng(1000 + seed)

    def u(shape, bound):
        return torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))

    sd = {
        "layer_norm_input.weight": 1.0 + u((d_model,), 0.2 if trained_like else 0.0),
        "layer_norm_input.bias": u((d_model,), 0.1 if trained_like else 0.0),
        "fc1.weight": u((hidden, d_model), d_model ** -0.5),
        "fc1.bias": u((hidden,), d_model ** -0.5),
        "layer_norm1.weight": 1.0 + u((hidden,), 0.2 if trained_like else 0.0),
        "layer_norm1.bias": u((hidden,), 0.1 if trained_like else 0.0),
        "fc2.weight": u((hidden, hidden), hidden ** -0.5),
        "fc2.bias": u((hidden,), hidden ** -0.5),
        "layer_norm2.weight": 1.0 + u((hidden,), 0.2 if trained_like else 0.0),
        "layer_norm2.bias": u((hidden,), 0.1 if trained_like else 0.0),
        "fc3.weight": u((N_CLASSES, hidden), 4.0 * hidden ** -0.5),
        "fc3.bias": u((N_CLASSES,), 0.1),
    }
    return sd


def make_hidden_states(n: int, seed: int, n_probers: int = 6, d_model: int = D_MODEL) -> torch.Tensor:
    """X[n, 6, d] = s * Normal(0,1), per-row s ~ LogUniform(10, 300): a sum of up to 149
    residual-stream vectors (SURVEY 8d, exp_rag.py:386)."""
    rng = np.random.default_rng(7000 + seed)
    x = rng.standard_normal((n, n_probers, d_model), dtype=np.float32)
    s = np.exp(rng.uniform(np.log(10.0), np.log(300.0), size=(n, 1, 1))).astype(np.float32)
    return torch.from_numpy(x * s)


# ----------------------------------------------------------------------------- dense embeddings (faiss IndexFlatL2 path)
EMB_SEED = 2468
EMB_BLOCK = 1 << 20
EMB_CLUSTERS = 4096
EMB_CENTROID_NORM = 1.5      # contriever-like: unnormalised mean-pooled embeddings of norm ~1.5
EMB_NOISE_NORM = 0.6
EMB_QUERY_NOISE_NORM = 0.3


def dense_rows(n: int, d: int, device="cuda", kind: str = "clustered", seed: int = EMB_SEED, row_lo: int = 0,
               row_hi: int | None = None) -> torch.Tensor:
    """f32 [n, d] embeddings generated on `device` in blocks of EMB_BLOCK rows, each block from its own seeded
    generator (the 21M x 768 corpus never exists on the host).  "clustered": one of EMB_CLUSTERS random centroids
    plus isotropic noise; "isotropic": N(0, 1/d) per dimension, the worst case of any filter (distances concentrate).
    row_lo / row_hi: exactly dense_rows(n, d)[row_lo:row_hi], generating only the blocks that overlap the range
    (whole blocks: a block's generator cannot be sought into) -- a row-range shard builds just its own rows."""
    if kind not in ("clustered", "isotropic"):
        raise ValueError(kind)
    row_hi = n if row_hi is None else row_hi
    if not 0 <= row_lo <= row_hi <= n:
        raise ValueError(f"row range [{row_lo}, {row_hi}) outside [0, {n})")
    out = torch.empty((row_hi - row_lo, d), dtype=torch.float32, device=device)
    g = _block_generator(device, seed, 1 << 20)
    cent = torch.randn((EMB_CLUSTERS, d), generator=g, device=device) * (EMB_CENTROID_NORM / d ** 0.5)
    for blk in range(row_lo // EMB_BLOCK, (row_hi + EMB_BLOCK - 1) // EMB_BLOCK):
        a, b = blk * EMB_BLOCK, min(n, (blk + 1) * EMB_BLOCK)
        g = _block_generator(device, seed, blk)
        noise = torch.randn((b - a, d), generator=g, device=device)
        if kind == "isotropic":
            block = noise * d ** -0.5
        else:
            c = torch.randint(0, EMB_CLUSTERS, (b - a,), generator=g, device=device)
            block = cent[c] + noise * (EMB_NOISE_NORM / d ** 0.5)
        s, e = max(a, row_lo), min(b, row_hi)
        out[s - row_lo:e - row_lo] = block[s - a:e - a]
    return out


def dense_queries(rows: torch.Tensor, n_queries: int, seed: int = EMB_SEED + 1) -> torch.Tensor:
    """f32 [n_queries, d]: perturbed copies of random rows (a question near its passage)."""
    g = _block_generator(rows.device, seed, 0)
    d = rows.shape[1]
    idx = torch.randint(0, rows.shape[0], (n_queries,), generator=g, device=rows.device)
    return rows[idx] + torch.randn((n_queries, d), generator=g, device=rows.device) * (EMB_QUERY_NOISE_NORM / d ** 0.5)


def dense_queries_of(n: int, d: int, n_queries: int, device="cuda", kind: str = "clustered", row_seed: int = EMB_SEED,
                     seed: int = EMB_SEED + 1) -> torch.Tensor:
    """Exactly dense_queries(dense_rows(n, d, device, kind, row_seed), n_queries, seed) without the rows: the same
    randint and randn draws, and only the blocks that hold the sampled rows are regenerated (every rank of a sharded
    index builds the same query batch from the shape alone)."""
    g = _block_generator(device, seed, 0)
    idx = torch.randint(0, n, (n_queries,), generator=g, device=device)
    noise = torch.randn((n_queries, d), generator=g, device=device)
    picked = torch.empty((n_queries, d), dtype=torch.float32, device=device)
    blocks = idx // EMB_BLOCK
    for blk in torch.unique(blocks).tolist():
        a = blk * EMB_BLOCK
        rows = dense_rows(n, d, device, kind, row_seed, row_lo=a, row_hi=min(n, a + EMB_BLOCK))
        sel = torch.nonzero(blocks == blk).flatten()
        picked[sel] = rows[idx[sel] - a]
    return picked + noise * (EMB_QUERY_NOISE_NORM / d ** 0.5)
