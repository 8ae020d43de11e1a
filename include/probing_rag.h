/* probing_rag.h -- C ABI of libprobingrag.so, the B200 (sm_100a) retrieval hot path of
 * Probing-RAG: batched BM25 scoring + top-k over a CSR inverted index in HBM, the k-way
 * merge of per-shard candidate lists, and the prober gate.
 *
 * The reference (baekingeol/Probing-RAG) is pure Python and has no FFI; each entry point
 * below names the reference call it replaces.  Host code stays Python/PyTorch and binds
 * these symbols with ctypes (see INTEGRATION.md); no torch types cross this boundary.
 *
 * Conventions
 *   - every function returns PR_OK (0) or a negative PR_E* code; pr_last_error() gives the
 *     thread-local message of the last failure on the calling thread.
 *   - all *_dev pointers are device pointers on the handle's device, owned by the caller
 *     (PyTorch tensors); the library allocates no device memory.
 *   - work is enqueued on the caller's stream; results are valid once that stream is
 *     synchronised.  No entry point synchronises the host except where stated.
 *   - ranked lists use the canonical total order: score descending, doc id ascending.
 *     Missing entries (fewer candidates than k) are (-INFINITY, -1).
 */
#ifndef PROBING_RAG_H
#define PROBING_RAG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PR_VERSION 201 /* 0.2.0 */

#define PR_OK 0
#define PR_EINVAL (-1)     /* bad argument (null pointer, k out of range, misaligned buffer) */
#define PR_ECUDA (-2)      /* a CUDA runtime call failed; message in pr_last_error()         */
#define PR_ERANGE (-3)     /* k > number of documents, or a term id outside [0, n_terms)     */
#define PR_EWORKSPACE (-4) /* workspace_bytes smaller than pr_bm25_workspace_bytes()         */
#define PR_EUNSUPPORTED (-5)

#define PR_MAX_K 128

typedef struct pr_index pr_index_t;
typedef void *pr_stream_t; /* cudaStream_t */

/* Tunables of the BM25 launch plan; zero fields keep the default. */
typedef struct pr_bm25_tuning {
    int32_t subs_per_item;   /* consecutive 2048-document sub-tiles one warp scores for one query (default 24; halved
                                automatically for batches too small to give every resident warp items_per_warp items) */
    int32_t warps_per_cta;   /* 4, 8 (default) or 12 */
    int32_t docs_per_launch; /* document range one launch covers for large batches (default 393216); bounds the
                                per-item list storage in the workspace ([n_queries][chunks per launch][k] pairs) */
    int32_t min_items;       /* a launch covers at least this many (query, chunk) work items (default 32768), so a
                                small batch is ONE scoring launch + one merge */
    int32_t items_per_warp;  /* small batches: work items per resident warp the plan aims for (default 1:
                                per-item set-up dominates a single query, measured in profiles/r02) */
    int32_t tile_epochs;     /* large batches: 4 (default) = the score tile is re-zeroed every 4th sub-tile (needs every
                                weight in [2^-30, 2^8], else 2 is used), 2 = every 2nd (A/B and tests) */
    int32_t batch_variant;   /* which variant of the scoring kernel runs: 3 (default) = by batch size (batches smaller
                                than twice the resident warps take the small-batch variant, whose warps re-read a query's
                                bound in front of tile scans), 1 = always the small-batch, 2 = always the large-batch variant */
} pr_bm25_tuning_t;

int pr_version(void);
const char *pr_last_error(void);

/* Inverted index handle over caller-owned device arrays -- the {data, indices, indptr,
 * num_docs} that bm25s.BM25.index() builds inside BM25Retriever.from_defaults
 * (/root/reference/exp_rag.py:242; SURVEY App. A.4), term-major with ascending doc ids:
 *   indptr_dev  int64[n_terms+1], doc_ids_dev int32[nnz] (LOCAL ids, 0-based, ascending per
 *   term), weights_dev float[nnz] (>= 0; precomputed idf*tfc).  doc_ids_dev and weights_dev
 *   must be 16-byte aligned and readable up to nnz rounded up to a multiple of 4 elements
 *   (the kernels use 128-bit loads; what lies past nnz is ignored).  n_docs is this shard's document count, doc_id_base the global
 *   id of local doc 0, n_docs_global the whole corpus size (k is checked against it).
 * Validates the arrays on the device and synchronises once. */
int pr_index_create(pr_index_t **out, int device, int64_t n_docs_global, int32_t doc_id_base,
                    int32_t n_docs, int32_t n_terms, int64_t nnz, const int64_t *indptr_dev,
                    const int32_t *doc_ids_dev, const float *weights_dev);
int pr_index_destroy(pr_index_t *index);

/* Per-index structures of the scoring kernel, built once per index into caller-owned device memory of
 * pr_index_aux_bytes(index, budget) bytes:
 *   - the COLD posting stream: every posting as an interleaved (tile byte offset, weight) pair, 8 bytes per posting
 *     (pr_index_aux_bytes adds it on top of the budget);
 *   - heavy_row[n_terms] and, for every term whose df exceeds a threshold chosen so the table fits a fifth of
 *     `table_budget_bytes`, the posting offset of each 2048-document boundary;
 *   - the HOT posting stream: for the terms with >= 8 postings per 2048 documents, as many as fit the rest of the
 *     budget and the 32-bit granule space, a padded, bank-aware, mask-free copy of their postings (about 10 bytes
 *     per hot posting).
 * pr_index_build_aux synchronises `stream`. */
typedef struct pr_index_aux_info {
    int32_t table_rows;        /* terms with a boundary table row */
    int32_t hot_rows;          /* terms in the hot stream */
    int32_t n_sub_tiles;       /* 2048-document sub-tiles of this shard */
    int64_t table_min_df;      /* df above which a term is tabulated */
    int64_t hot_min_df;        /* df from which a term is hot */
    int64_t hot_stream_bytes;
    int64_t cold_stream_bytes;
} pr_index_aux_info_t;
size_t pr_index_aux_bytes(const pr_index_t *index, size_t table_budget_bytes);
int pr_index_build_aux(pr_index_t *index, void *aux_dev, size_t aux_bytes, pr_stream_t stream);
int pr_index_aux_info(const pr_index_t *index, pr_index_aux_info_t *info);
int pr_index_set_tuning(pr_index_t *index, const pr_bm25_tuning_t *tuning);
int pr_index_get_tuning(const pr_index_t *index, pr_bm25_tuning_t *tuning);

/* Bytes of scratch pr_bm25_topk needs for a batch of n_queries at depth k. */
size_t pr_bm25_workspace_bytes(const pr_index_t *index, int32_t n_queries, int32_t k);

/* Batched BM25Retriever.retrieve (/root/reference/exp_rag.py:426, 428, 492; utils.py:640;
 * bm25s.BM25.retrieve + selection.topk, SURVEY App. A.5-A.6) at token-id level.
 *   q_indptr_dev int64[n_queries+1], q_terms_dev int32[n_q_terms]: CSR batch of query term ids in
 *   query-token order, duplicates kept.  Scores are accumulated in fp32 in that order, one
 *   rounded add per posting, exactly as the reference's dense accumulator does.
 *   out_scores_dev float[n_queries*k], out_doc_ids_dev int32[n_queries*k] (GLOBAL doc ids).
 * Fewer than k positive scores: the tail is filled with this shard's lowest doc ids at
 * score 0.0.  Both arrays are validated ON THE DEVICE, nothing is read out of bounds: a query whose
 * q_indptr slice is negative, decreasing or not inside [0, n_q_terms) (or a batch whose offsets do not
 * start at 0) scores nothing and makes pr_bm25_status() report PR_EINVAL; a term id outside
 * [0, n_terms) is skipped and reported as PR_ERANGE (bm25s raises ValueError there, App. A.5). */
int pr_bm25_topk(pr_index_t *index, int32_t n_queries, const int64_t *q_indptr_dev,
                 const int32_t *q_terms_dev, int64_t n_q_terms, int32_t k, float *out_scores_dev,
                 int32_t *out_doc_ids_dev, void *workspace_dev, size_t workspace_bytes,
                 pr_stream_t stream);

/* The same call cut at launch boundaries, for doc-range shards on several GPUs (SURVEY 8e).  A call
 * walks its shard in pr_bm25_num_launches() launches.  The workspace holds, at byte offset
 * pr_bm25_theta_offset(), float theta[n_queries]: the best known LOWER BOUND of every query's final
 * k-th score (-1 = none).  The scoring warps read and raise it while they run; between two ranges the
 * caller may raise it further with what the other shards found -- e.g. an all-reduce(MAX) of that
 * array over the ranks: the global k-th score is >= every shard's local k-th score, so each shard then
 * filters with the strongest bound any shard knows and the merged result stays bit-identical.
 * Ranges must be issued in order, [0, a), [a, b), ... up to the launch count, with the same arguments.
 * pr_bm25_num_launches: n_docs < 0 = this index; otherwise the count a shard of n_docs documents would have
 * under this index's tuning (ranks agree on the number of exchange rounds through the longest shard). */
int32_t pr_bm25_num_launches(const pr_index_t *index, int32_t n_queries, int32_t k, int64_t n_docs);
size_t pr_bm25_theta_offset(const pr_index_t *index, int32_t n_queries, int32_t k);
int pr_bm25_topk_range(pr_index_t *index, int32_t n_queries, const int64_t *q_indptr_dev,
                       const int32_t *q_terms_dev, int64_t n_q_terms, int32_t k, float *out_scores_dev,
                       int32_t *out_doc_ids_dev, void *workspace_dev, size_t workspace_bytes,
                       int32_t launch_begin, int32_t launch_end, pr_stream_t stream);

/* A stronger exchange for the first launches of a large batch, while bounds are still weak: the K-th largest score of
 * the UNION of all shards' running lists (the shards hold disjoint documents, so K documents scoring at least that
 * exist) instead of the best of the shards' own K-th scores.  Between two ranges the workspace holds, at byte offset
 * pr_bm25_running_scores_offset(), float run_scores[n_queries][k]: this shard's best k scores so far, descending,
 * -1 = empty slot.  The caller all-gathers those arrays ([n_lists][n_queries][k]) and hands them to
 * pr_bm25_raise_union_bound, which raises every query's bound to the k-th largest of its n_lists * k scores --
 * in the workspace or, with peers set, in this rank's peer-shared array (all ranks compute the same value). */
size_t pr_bm25_running_scores_offset(const pr_index_t *index, int32_t n_queries, int32_t k);
int pr_bm25_raise_union_bound(pr_index_t *index, int32_t n_queries, int32_t k, const float *gathered_scores_dev,
                              int32_t n_lists, void *workspace_dev, size_t workspace_bytes, pr_stream_t stream);

/* Thresholds shared LIVE between the GPUs of a doc-sharded corpus (one process per GPU, NVLink / NVSwitch peer
 * memory) -- the fused form of the exchange above: every rank keeps float theta[2][capacity] in memory its peers can
 * address (pr_peer_alloc / pr_peer_open: CUDA IPC), and a scoring warp that raises a query's bound raises it in all
 * copies with system-scope atomic maxima, so the other shards filter with it while they are still scoring -- no
 * collective, no launch boundary.  The two halves alternate from call to call (all ranks must issue the same
 * sequence of pr_bm25_topk calls, which the all-gather that ends each sharded call enforces anyway).
 *   local_dev             this rank's array (2 * capacity floats, from pr_peer_alloc); NULL = private thresholds again
 *   peer_bases_host       host array of n_peers (<= PR_MAX_PEERS) device pointers: the peers' arrays as opened here
 *   peer_table_dev        2 * PR_MAX_PEERS * sizeof(void *) bytes of device memory on this GPU, owned by the caller,
 *                         which the library fills (the kernels index it)
 * With peers set, pr_bm25_theta_offset() no longer describes where the bounds live. */
#define PR_MAX_PEERS 15
typedef struct pr_ipc_handle { unsigned char bytes[64]; } pr_ipc_handle_t;
int pr_peer_alloc(int device, size_t bytes, void **out_dev, pr_ipc_handle_t *out_handle);
int pr_peer_open(int device, const pr_ipc_handle_t *handle, void **out_dev);
int pr_peer_close(void *dev);
int pr_peer_free(void *dev);
int pr_index_set_peer_thetas(pr_index_t *index, float *local_dev, int64_t capacity, int32_t n_peers,
                             float *const *peer_bases_host, void *peer_table_dev);

/* Reads the status word pr_bm25_topk left in the workspace (synchronises `stream`). */
int pr_bm25_status(const void *workspace_dev, pr_stream_t stream);

/* Per-kernel timing for bench.py's roofline line: when enabled, pr_bm25_topk brackets every
 * launch of the scoring kernel with CUDA events on the caller's stream; pr_bm25_profile waits
 * for them and returns the summed device time and the launch count of the last call. */
int pr_index_set_profiling(pr_index_t *index, int enable);
int pr_bm25_profile(pr_index_t *index, float *score_ms, int32_t *score_launches);

/* Kernel launches the last pr_bm25_topk call on this handle enqueued (for bench accounting). */
int64_t pr_bm25_last_launches(const pr_index_t *index);

/* k-way merge of per-shard ranked lists (the step after the NCCL all-gather, SURVEY 8e):
 *   scores_dev float[n_lists, n_queries, k], ids_dev int32[n_lists, n_queries, k]
 *   -> out_scores_dev float[n_queries, k], out_ids_dev int32[n_queries, k].
 * Each input list is in the canonical order (score descending, id ascending), scores >= +0, and may end in padding
 * (score < 0, id -1), which is ignored.  The inputs must hold at least k valid entries per query over all lists,
 * which doc-range shards guarantee (each fills its zero-score tail, and together they hold >= k documents): the
 * merge fills no zero-score tail of its own, so a query with fewer valid entries ends in (-inf, -1). */
int pr_topk_merge(int32_t n_queries, int32_t k, int32_t n_lists, const float *scores_dev,
                  const int32_t *ids_dev, float *out_scores_dev, int32_t *out_ids_dev,
                  pr_stream_t stream);

/* ---- prober gate ------------------------------------------------------------------------
 * Six ImprovedProbe MLPs (/root/reference/utils.py:29-57) + softmax-sum gate
 * (/root/reference/exp_rag.py:407-415) + stream compaction of the "retrieve" rows. */
#define PR_PROBER_MAX 8

/* A set of n_probers ImprovedProbe MLPs, packed per prober and kept in caller-owned device memory
 * (probing_rag_b200/prober.py packs a list of state_dicts; utils.py:29-57 names in the comments).  The input LayerNorm
 * is folded around fc1 -- fc1(LN(x)) = rstd * (W' (x - s) - (mean - s) * rowsum(W')) + (W beta + b1) with
 * W' = W diag(gamma) and s a per-row shift (the mean of the row's first 64 features, so that the bf16 split error does
 * not grow with a common offset) -- so the tensor cores multiply the shifted hidden states and the kernel's epilogue
 * applies the row statistics:
 *   w1_hi / w1_lo   fc1.weight * layer_norm_input.weight[None, :], split for bf16x3 accumulation
 *                   (hi = bf16(w), lo = bf16(w - hi), row-major [out, in] like nn.Linear.weight)
 *   w1_rowsum       its row sums
 *   b1              fc1.bias + fc1.weight @ layer_norm_input.bias
 * The other vectors are the state_dict tensors as they are; fc2.weight is split the same way. */
typedef struct pr_prober_set {
    int32_t n_probers;               /* <= PR_PROBER_MAX; 6 in the reference (exp_rag.py:311) */
    int32_t d_model;                 /* 2048 (gemma-2b); multiple of 128, <= 2048             */
    int32_t hidden;                  /* 512                                                   */
    const float *w1_rowsum;          /* [P][hidden]    see above                              */
    const float *b1;                 /* [P][hidden]    see above                              */
    const float *ln1_w, *ln1_b;      /* [P][hidden]    layer_norm1.{weight,bias}              */
    const float *b2;                 /* [P][hidden]    fc2.bias                               */
    const float *ln2_w, *ln2_b;      /* [P][hidden]    layer_norm2.{weight,bias}              */
    const float *w3, *b3;            /* [P][2][hidden], [P][2]   fc3 (kept fp32)              */
    const void *w1_hi, *w1_lo;       /* bf16 [P][hidden][d_model]  see above, 128-byte aligned */
    const void *w2_hi, *w2_lo;       /* bf16 [P][hidden][hidden]   fc2.weight split, 128-byte aligned */
} pr_prober_set_t;

size_t pr_prober_workspace_bytes(int32_t n_probers, int32_t n_rows, int32_t d_model, int32_t hidden);

/* X_dev [n_rows, n_probers, d_model]: pooled hidden states, one per probed layer (exp_rag.py:385-386), of
 * x_dtype 0 = f32, 1 = bf16, 2 = f16 (whatever the LM produced; 16-byte aligned).  Outputs:
 * out_logits_dev float[n_rows, n_probers, 2] (may be NULL), out_probsum_dev float[n_rows, 2] = sum over
 * probers >= ablation of softmax(logits) (exp_rag.py:407-410), out_retrieve_mask_dev uint8[n_rows] (1 =
 * retrieve, i.e. NOT probsum[0] + theta < probsum[1], evaluated in double like the reference's Python floats,
 * exp_rag.py:414), out_compact_idx_dev int32[n_rows] (indices of the rows that retrieve, ascending; the first
 * *out_n_retrieve_dev are valid, the rest read -1).  workspace_dev must be 1024-byte aligned. */
int pr_prober_forward(const pr_prober_set_t *probers, int32_t n_rows, const void *X_dev, int32_t x_dtype, double theta,
                      int32_t ablation, float *out_logits_dev, float *out_probsum_dev,
                      uint8_t *out_retrieve_mask_dev, int32_t *out_compact_idx_dev,
                      int32_t *out_n_retrieve_dev, void *workspace_dev, size_t workspace_bytes,
                      pr_stream_t stream);

/* ---- hidden-state pooling (SURVEY 8f-3) ---------------------------------------------------
 * On-device replacement of the forward hooks at /root/reference/exp_rag.py:317-321 (which copy every
 * probed layer's activations to the host on every forward call) and of the concat + sum over tokens at
 * exp_rag.py:385-386.  Adds the token-sum of one forward call's activations of one probed layer into
 * the prober input matrix:
 *   acc_dev float[n_acc_rows, n_probers, d_model]  +=  sum_t act[r, t, :]   into [row, slot, :]
 *   act_dev [n_rows, n_tokens, d_model] of act_dtype (0 = f32, 1 = bf16, 2 = f16), element strides
 *   row_stride / tok_stride (feature stride 1, tok_stride 0 allowed); row_map_dev int32[n_rows] maps
 *   activation row r to an accumulator row, NULL = identity.  Negative entries and entries >= n_acc_rows
 *   skip the row.  The other entries must be distinct: each row is added with a plain (non-atomic)
 *   read-modify-write, so two rows into one accumulator row race and the result is undefined.  The
 *   function cannot check a device array; HiddenStatePooler.add (pooling.py) checks it and raises.
 * The caller skips the prefill call of a generation (the reference drops cache[name][0]).  Exact
 * arithmetic: per activation row the tokens are summed in fp32 in token order starting from 0, and that
 * sum is added to the accumulator once.  Pointers and strides must allow 4-element vector access. */
int pr_pool_accumulate(float *acc_dev, int32_t n_acc_rows, int32_t n_probers, int32_t slot, int32_t d_model,
                       const void *act_dev, int32_t act_dtype, int32_t n_rows, int32_t n_tokens,
                       int64_t row_stride, int64_t tok_stride, const int32_t *row_map_dev, pr_stream_t stream);

/* ---- dense flat L2 and inner-product search ------------------------------------------------
 * Exact replacement of faiss.IndexFlatL2(d): the index built at /root/reference/make_indexer.py:446-457, loaded at
 * exp_rag.py:243-248 and searched with k = 5 at exp_rag.py:431-438 and :496 (helpers utils.py:365-380).
 *   rows     caller-owned f32 [n][d], d a multiple of 64 in [64, PR_FLAT_MAX_D], n <= 2^31 - 1, 16-byte aligned
 *   result   squared L2 distances f32 [B][k], ascending, ties by row id ascending; row ids i64 [B][k];
 *            rows short of k (k > n) are padded with (FLT_MAX, -1), the neutral entry of faiss's max-heap
 * The distance is ||q - x||^2 evaluated in float64 in a fixed order and rounded once to f32 (DESIGN §3), so results
 * do not depend on the launch plan.  Rows of the index are filtered with a bf16 tensor-core product and a proven
 * lower bound of the exact distance; only rows that can enter the top-k are evaluated exactly (DESIGN §4.6). */
#define PR_FLAT_MAX_D 1024
typedef struct pr_flat pr_flat_t;

/* faiss's metric numbering.  PR_METRIC_INNER_PRODUCT replaces faiss.IndexFlatIP(d), the index Contriever's and DPR's
 * own indexing code builds:
 *   result   scores q.x f32 [B][k], descending, ties by row id ascending; NaN scores rank after -inf, among
 *            themselves by id (and come back as the NaN with bit pattern 0xFFFFFFFF); row ids i64 [B][k]; rows short of
 *            k are padded with (-FLT_MAX, -1), the neutral entry of faiss's min-heap.  A real row whose score is
 *            -FLT_MAX or -inf still ranks before the padding.
 * The score is q.x evaluated in float64 in a fixed order and rounded once to f32, never -0 (DESIGN §3); rows are
 * filtered with the same bf16 tensor-core product and a proven upper bound of the exact score (DESIGN §4.6). */
#define PR_METRIC_INNER_PRODUCT 0
#define PR_METRIC_L2 1

/* Launch plan of pr_flat_search; zero fields keep the default. */
typedef struct pr_flat_tuning {
    int64_t first_chunk_rows; /* rows of the first filter + refine round (default 2048, rounded up to 128): every one of
                                 them is a candidate, as no bound is known yet */
    int32_t growth;           /* each later chunk is this many times the one before (default 4) */
    int32_t cand_capacity;    /* candidates kept per query and chunk (default 8192); a query that finds more in a chunk
                                 has that chunk scanned exactly instead (same result, slower) */
} pr_flat_tuning_t;

/* What the last pr_flat_search on a handle did, for benchmarks. */
typedef struct pr_flat_stats {
    int64_t launches;         /* kernel launches enqueued */
    int64_t chunks;           /* filter + refine rounds */
    int64_t candidates;       /* (query, row) pairs the filter passed, summed over queries and chunks */
    int64_t max_candidates;   /* largest count of one query in one chunk */
    int64_t fallback_queries; /* (query, chunk) pairs whose candidates overflowed and were scanned exactly */
} pr_flat_stats_t;

/* Handle over caller-owned rows (no copy; the rows must outlive the handle).  Reads the device's SM count; enqueues
 * nothing.  pr_flat_create is pr_flat_create_metric(..., PR_METRIC_L2); any other metric than the two above returns
 * PR_EUNSUPPORTED.  Every other pr_flat_* function serves the handle's metric. */
int pr_flat_create(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d);
int pr_flat_create_metric(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d, int metric);
int pr_flat_destroy(pr_flat_t *index);
/* faiss.IndexScalarQuantizer(d, QT_fp16, metric): a handle over caller-owned IEEE binary16 codes [n][d] (the rows as
 * stored, e.g. torch's .to(float16) of the f32 rows: round to nearest even, overflow to +-inf), with the checks of
 * pr_flat_create_metric (codes_dev 16-byte aligned).  Every other pr_flat_* function serves it, with the results an
 * f32 handle returns over the decoded rows, bit for bit; its aux holds no copy of the rows (12 bytes a row: ||x||^2,
 * ||x|| and the norm of the row's fp16-subnormal elements), and the filter runs on the codes (DESIGN §4.6). */
int pr_flat_create_fp16(pr_flat_t **out, int device, const uint16_t *codes_dev, int64_t n, int32_t d, int metric);
/* The bf16 copy of the rows and their norms (fp16 handle: the norms only), built once into caller memory (1024-byte
 * aligned) of pr_flat_aux_bytes() bytes; the handle keeps the pointer.  pr_flat_build_aux synchronises `stream`. */
size_t pr_flat_aux_bytes(const pr_flat_t *index);
int pr_flat_build_aux(pr_flat_t *index, void *aux_dev, size_t aux_bytes, pr_stream_t stream);
int pr_flat_set_tuning(pr_flat_t *index, const pr_flat_tuning_t *tuning);
int pr_flat_get_tuning(const pr_flat_t *index, pr_flat_tuning_t *tuning);
/* Scratch for a batch of n_queries at depth k (1 <= k <= PR_MAX_K) under the current tuning; 0 on bad arguments. */
size_t pr_flat_workspace_bytes(const pr_flat_t *index, int32_t n_queries, int32_t k);
/* IndexFlatL2.search / IndexFlatIP.search(queries, k): queries_dev f32 [n_queries][d] (16-byte aligned), workspace 1024-byte aligned. */
int pr_flat_search(pr_flat_t *index, int32_t n_queries, const float *queries_dev, int32_t k, float *out_dist_dev,
                   int64_t *out_ids_dev, void *workspace_dev, size_t workspace_bytes, pr_stream_t stream);
/* Counters of the last pr_flat_search with this workspace and shape (synchronises `stream`). */
int pr_flat_last_stats(const pr_flat_t *index, const void *workspace_dev, int32_t n_queries, int32_t k,
                       pr_flat_stats_t *out, pr_stream_t stream);

/* IndexFlatL2.range_search / IndexFlatIP.range_search(queries, radius) for the handle's metric (DESIGN §3):
 *   L2  row r is a result of query q iff its exact distance D(q, r) < radius;  IP  iff its exact score S(q, r) > radius.
 *   The values are those pr_flat_search returns; NaN values are never results, and a NaN radius gives none.
 * Results are placed by the caller: query q's hits, in ascending row id, are written to dist_dev / ids_dev at
 * [lims_in_dev[q], lims_in_dev[q + 1]) (i64 [n_queries + 1], on the device), and count_dev i64 [n_queries] receives
 * each query's full number of hits, including those past the segment's end, which are not written.  Call it once with
 * segments of a fixed staging size; if some count exceeds it, call it again with lims_in_dev = the exclusive prefix sum
 * of the counts: the second call evaluates the same rows and writes every hit.  Results do not depend on the launch plan.
 * A (query, chunk) with more candidates than min(cand_capacity, 8192) is scanned exactly, in row order.
 * queries_dev 16-byte aligned, workspace_dev 1024-byte aligned, lims_in_dev, count_dev, ids_dev 8-byte aligned.
 * Enqueues on `stream`, no sync.  pr_flat_last_stats(index, workspace, n_queries, 1, ...) reads its counters. */
size_t pr_flat_range_workspace_bytes(const pr_flat_t *index, int32_t n_queries);
int pr_flat_range_search(pr_flat_t *index, int32_t n_queries, const float *queries_dev, float radius,
                         const int64_t *lims_in_dev, int64_t *count_dev, float *dist_dev, int64_t *ids_dev,
                         void *workspace_dev, size_t workspace_bytes, pr_stream_t stream);

/* Merge n_lists ranked dense lists per query into one, in the order pr_flat_search produces (the step after the
 * all-gather of a row-range sharded search, dense.ShardedIndexFlatL2).
 *   dist_dev f32 [n_lists][n_queries][k], ids_dev i64 [n_lists][n_queries][k]: each list sorted as pr_flat_search
 *   outputs it; entries with id < 0 are padding and are ignored whatever their distance.
 *   id_base  host array of n_lists non-negative offsets added to every real id of list l (local row -> global row).
 *   -> out_dist_dev f32 [n_queries][k], out_ids_dev i64 [n_queries][k], short rows padded (FLT_MAX, -1).
 * Order: (uint32 bit pattern of the distance, global id) ascending. That is the key order of pr_flat_search's
 * ranked lists, so a sharded search equals the single index bit for bit.  Enqueues one kernel on `stream` on the
 * current device; no sync, no allocation. */
#define PR_FLAT_MAX_LISTS 32
int pr_flat_merge(int32_t n_queries, int32_t k, int32_t n_lists, const float *dist_dev, const int64_t *ids_dev,
                  const int64_t *id_base, float *out_dist_dev, int64_t *out_ids_dev, pr_stream_t stream);
/* pr_flat_merge for lists of either metric (pr_flat_merge is its PR_METRIC_L2 case).  PR_METRIC_INNER_PRODUCT: the same
 * rules, in the inner-product order above: (key of the score, global id) ascending, where the key ascends as the score
 * descends and puts NaN after -inf -- the key of pr_flat_search's inner-product lists; padding ranks after every real
 * entry (-FLT_MAX, -inf and NaN included) and short rows are padded (-FLT_MAX, -1).  Another metric: PR_EUNSUPPORTED. */
int pr_flat_merge_metric(int32_t n_queries, int32_t k, int32_t n_lists, const float *dist_dev, const int64_t *ids_dev,
                         const int64_t *id_base, float *out_dist_dev, int64_t *out_ids_dev, pr_stream_t stream,
                         int metric);

#ifdef __cplusplus
}
#endif
#endif /* PROBING_RAG_H */
