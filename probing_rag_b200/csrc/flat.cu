// Exact flat L2 and inner-product search (faiss IndexFlatL2 / IndexFlatIP drop-ins) on B200 tensor cores (sm_100a).
//
// Replaces faiss.IndexFlatL2(768).search(q, k), the brute-force CPU scan the reference's dense path runs
// (/root/reference/exp_rag.py:243-248, 431-438, 496; utils.py:365-380; index built at make_indexer.py:446-457).
//
// The result is EXACT: distances (scores) are evaluated in float64 in a fixed order (DESIGN §3) and the ranked list is
// the canonical (distance asc, id asc) order, or (score desc, id asc) for inner products.  The tensor cores only decide
// which rows need that evaluation:
//
//   prep     flat_prep_kernel        bf16 copy (RNE) of every row, ||x||^2 and ||x|| in f32 (aux buffer, once per index;
//                                    the same kernel prepares the query batch per call)
//   filter   flat_filter_kernel      persistent tcgen05 GEMM, M = 128 rows of the index x N = 32..256 queries, K = d:
//                                      warp 0  TMA producer (doc tile 128 x 64 + query tile N x 64 per stage)
//                                      warp 1  MMA issuer (kind::f16, fp32 accumulators, two TMEM buffers)
//                                      warp 2  TMEM allocator
//                                      warps 4-7 epilogue: lower bound ||q||^2 + ||x||^2 - 2 q.x - margin(q, x) of the
//                                              exact distance; (query, row) pairs whose bound does not exceed the
//                                              query's running bound theta[q] go to a per-query candidate list
//            flat_ip_filter_kernel   the same GEMM; epilogue: upper bound q.x + margin(q, x) of the exact score, pairs
//                                    whose bound is not below theta[q] are candidates
//   refine   flat_refine_kernel      one CTA per query: exact distances of the candidates (or of the whole chunk
//                                    when the list overflowed), merged into the running top-k; theta[q] = its k-th
//                                    distance, a valid upper bound of the final k-th distance
//            flat_ip_refine_kernel   the same with exact inner products; theta[q] = the k-th score, a lower bound of
//                                    the final k-th score
//   output   flat_output_kernel      running lists -> (distance, id) with (FLT_MAX, -1) padding, (-FLT_MAX, -1) for IP
//   range    pr_flat_range_search: the same filter with theta[q] = radius throughout, then the range refine of
//            flat_range.cu per chunk (each query's candidates in row order, hits appended to the query's segment)
//   merge    flat_merge_kernel       pr_flat_merge: the lists of row-range shards -> one list in the same order
//   fp16     pr_flat_create_fp16: rows stored as IEEE binary16 codes; the same host plan launches the fp16 kernels of
//            flat_fp16.cu (the same GEMM and refines on the codes themselves, no bf16 copy)
//
// One host plan (flat_plan) serves both searches and both storage types: init (theta[q] = +-inf for top-k search, the
// radius for range search), query prep, the two tensor maps and the filter's arguments, then the rows cut into chunks
// of growing size, filter and refine alternating per chunk on the caller's stream, so that every chunk filters with
// the bound the earlier ones established ("bounds raised between launches", as BM25 does).  The caller chooses the
// refine: the top-k refine, then the output kernel (pr_flat_search), or the range refine (pr_flat_range_search).  Each
// stage's kernel is picked by the storage type at one call site and by the metric in the launcher of its translation
// unit.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "flat_exact.cuh"
#include "flat_filter.cuh"
#include "tcgen05.cuh"

struct pr_flat {
    int device;
    int n_sm;
    int64_t n;
    int32_t d;
    const float *rows;
    const __nv_bfloat16 *rows_bf;   // aux: bf16 copy [n][d]
    const float *norm2, *norm;      // aux: ||x||^2, ||x|| (f32)
    int metric;                     // PR_METRIC_L2 or PR_METRIC_INNER_PRODUCT
    int32_t fp16;                   // pr_flat_create_fp16; in the padding before `tun`, so that the fields up to
                                    // last_chunks keep the offsets tests/test_flat_range_oracle.py mirrors (_FakeFlat)
    pr_flat_tuning_t tun;
    int64_t last_launches, last_chunks;
    const __half *codes;            // fp16 only (read only when fp16 != 0): the rows [n][d] and the aux ||x_sub||
    const float *nsub;
};

namespace {

constexpr int64_t kDefaultFirstChunk = 2048;
constexpr int32_t kDefaultGrowth = 4;
constexpr int32_t kDefaultCapacity = 8192;

inline size_t up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------------------------ prep
// One warp per row: bf16 copy (RNE) and ||x||^2, ||x|| (summed in f64, rounded once to f32).  Rows in [n, n_out)
// are written as zeros (the padded query rows of a batch).
__global__ void flat_prep_kernel(const float *__restrict__ x, int64_t n, int64_t n_out, int d,
                                 __nv_bfloat16 *__restrict__ xb, float *__restrict__ norm2, float *__restrict__ norm)
{
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_out) return;
    double s = 0.0;
    for (int j = 2 * lane; j < d; j += 64) {
        float2 v = make_float2(0.f, 0.f);
        if (row < n) v = *reinterpret_cast<const float2 *>(x + row * d + j);
        s = fma((double)v.x, (double)v.x, s);
        s = fma((double)v.y, (double)v.y, s);
        *reinterpret_cast<__nv_bfloat162 *>(xb + row * d + j) = __floats2bfloat162_rn(v.x, v.y);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(PR_FULL_MASK, s, o);
    if (lane == 0) {
        norm2[row] = (float)s;
        norm[row] = (float)sqrt(s);
    }
}

__global__ void flat_init_kernel(int n_queries, int k, float theta0, float *__restrict__ theta,
                                 int32_t *__restrict__ count, uint64_t *__restrict__ topk,
                                 unsigned long long *__restrict__ stats)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (int64_t)n_queries * k) topk[i] = kEmptyKey;
    if (i < n_queries) {
        theta[i] = theta0;
        count[i] = 0;
    }
    if (i < 4) stats[i] = 0;
}

__global__ void __launch_bounds__(kFilterThreads, 1)
flat_filter_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                   const FilterArgs g)
{
    flat_filter<PR_METRIC_L2>(map_x, map_q, g);
}

__global__ void __launch_bounds__(kFilterThreads, 1)
flat_ip_filter_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                      const FilterArgs g)
{
    flat_filter<PR_METRIC_INNER_PRODUCT>(map_x, map_q, g);
}

__global__ void __launch_bounds__(kRefineThreads) flat_refine_kernel(const RefineArgs g) { flat_refine<PR_METRIC_L2>(g); }

__global__ void __launch_bounds__(kRefineThreads) flat_ip_refine_kernel(const RefineArgs g)
{
    flat_refine<PR_METRIC_INNER_PRODUCT>(g);
}

__global__ void flat_output_kernel(int64_t total, const uint64_t *__restrict__ topk, float *__restrict__ dist,
                                   int64_t *__restrict__ ids, int metric)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint64_t key = topk[i];
    const bool ip = metric == PR_METRIC_INNER_PRODUCT;
    if (key == kEmptyKey) {
        dist[i] = ip ? -FLT_MAX : FLT_MAX;
        ids[i] = -1;
    } else {
        const uint32_t hi = (uint32_t)(key >> 32);
        dist[i] = __uint_as_float(ip ? ip_bits(hi) : hi);
        ids[i] = (int64_t)(uint32_t)key;
    }
}

// ------------------------------------------------------------------------------------ merge of shard lists
// One warp per query.  The query's n_lists lists are first staged in shared memory; lane l then holds the head of
// list l (entries with id < 0 skipped) and each of the k rounds takes the warp-wide minimum of (key, global id, lane)
// and advances the winner's list.  The key is the refine's: l2_key of the distance or ip_key of the score.  A head
// past the end of its list carries hi = 2^32, above every real key, so padding ranks after FLT_MAX and +inf (L2) or
// -FLT_MAX, -inf and NaN (IP); once the minimum is padding, so is the rest.
struct MergeArgs {
    int n_queries, k, n_lists, warps, metric;
    const float *dist;
    const int64_t *ids;
    float *out_dist;
    int64_t *out_ids;
    int64_t base[PR_FLAT_MAX_LISTS];
};

constexpr int kMergeSmemBudget = 48 * 1024;    // the default limit: 32 lists x k = 128 fit one warp
constexpr int kMergeMaxWarps = 8;

__global__ void __launch_bounds__(kMergeMaxWarps * 32) flat_merge_kernel(const MergeArgs g)
{
    extern __shared__ __align__(16) unsigned char merge_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * g.warps + warp;
    if (q >= g.n_queries) return;
    const int k = g.k, L = g.n_lists;
    int64_t *s_id = reinterpret_cast<int64_t *>(merge_smem) + (size_t)warp * L * k;
    float *s_d = reinterpret_cast<float *>(reinterpret_cast<int64_t *>(merge_smem) + (size_t)g.warps * L * k) +
                 (size_t)warp * L * k;
    for (int l = 0; l < L; ++l) {
        const size_t src = ((size_t)l * g.n_queries + q) * k;
        for (int i = lane; i < k; i += 32) {
            s_d[l * k + i] = __ldg(g.dist + src + i);
            s_id[l * k + i] = __ldg(g.ids + src + i);
        }
    }
    __syncwarp();
    const bool ip = g.metric == PR_METRIC_INNER_PRODUCT;
    const bool mine = lane < L;
    const int64_t base = mine ? g.base[lane] : 0;
    int pos = 0;
    if (mine)
        while (pos < k && s_id[lane * k + pos] < 0) ++pos;
    float *od = g.out_dist + (size_t)q * k;
    int64_t *oi = g.out_ids + (size_t)q * k;
    for (int r = 0; r < k; ++r) {
        const bool live = mine && pos < k;
        const uint32_t bits = live ? __float_as_uint(s_d[lane * k + pos]) : 0u;
        uint64_t hi = live ? (uint64_t)(ip ? ip_key(bits) : l2_key(bits)) : (1ull << 32);
        int64_t gid = live ? s_id[lane * k + pos] + base : INT64_MAX;
        int who = lane;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const uint64_t h2 = __shfl_xor_sync(PR_FULL_MASK, hi, o);
            const int64_t g2 = __shfl_xor_sync(PR_FULL_MASK, gid, o);
            const int w2 = __shfl_xor_sync(PR_FULL_MASK, who, o);
            if (h2 < hi || (h2 == hi && (g2 < gid || (g2 == gid && w2 < who)))) {
                hi = h2;
                gid = g2;
                who = w2;
            }
        }
        if (hi >> 32) {                       // every list is exhausted: pad the rest of the row
            for (int i = r + lane; i < k; i += 32) {
                od[i] = ip ? -FLT_MAX : FLT_MAX;
                oi[i] = -1;
            }
            break;
        }
        if (lane == who) {
            od[r] = __uint_as_float(ip ? ip_bits((uint32_t)hi) : (uint32_t)hi);
            oi[r] = gid;
            ++pos;
            while (pos < k && s_id[lane * k + pos] < 0) ++pos;
        }
    }
}

// ------------------------------------------------------------------------------------ host
struct FlatLayout {
    int nq, n_qb, b_pad;
    size_t q_bf, qn2, qn, theta, count, cand, topk, stats, qscale, total;
};

// queries per tile: as few 32-column groups as cover the batch in equal blocks of at most 256.  fp16 storage: q_bf holds
// the fp16 query copy and the per-query scales follow the counters.
FlatLayout flat_layout(int d, int n_queries, int k, int cap, bool fp16)
{
    FlatLayout l;
    l.n_qb = (n_queries + kMaxNQ - 1) / kMaxNQ;
    const int per = (n_queries + l.n_qb - 1) / l.n_qb;
    l.nq = (per + 31) / 32 * 32;
    l.b_pad = l.n_qb * l.nq;
    size_t o = 0;
    l.q_bf = o;  o = up(o + (size_t)l.b_pad * d * 2, 256);
    l.qn2 = o;   o = up(o + (size_t)l.b_pad * 4, 256);
    l.qn = o;    o = up(o + (size_t)l.b_pad * 4, 256);
    l.theta = o; o = up(o + (size_t)n_queries * 4, 256);
    l.count = o; o = up(o + (size_t)n_queries * 4, 256);
    l.cand = o;  o = up(o + (size_t)n_queries * cap * 4, 256);
    l.topk = o;  o = up(o + (size_t)n_queries * k * 8, 256);
    l.stats = o; o = up(o + 4 * 8, 256);
    l.qscale = o;
    if (fp16) o = up(o + (size_t)l.b_pad * 4, 256);
    l.total = o;
    return l;
}

// The workspace of one call, carved by its layout.  q_ops: the queries' bf16 copy, or their scaled fp16 copy.
struct FlatWs {
    void *q_ops;
    float *qn2, *qn, *theta;
    int32_t *count, *cand;
    uint64_t *topk;
    unsigned long long *stats;
    float *qscale;                  // fp16 storage only
};

FlatWs flat_ws(const FlatLayout &l, void *base)
{
    unsigned char *ws = (unsigned char *)base;
    return {ws + l.q_bf, (float *)(ws + l.qn2), (float *)(ws + l.qn), (float *)(ws + l.theta),
            (int32_t *)(ws + l.count), (int32_t *)(ws + l.cand), (uint64_t *)(ws + l.topk),
            (unsigned long long *)(ws + l.stats), (float *)(ws + l.qscale)};
}

size_t aux_norm2_offset(const pr_flat *h) { return h->fp16 ? 0 : up((size_t)h->n * h->d * 2, 256); }
size_t aux_norm_offset(const pr_flat *h) { return up(aux_norm2_offset(h) + (size_t)h->n * 4, 256); }
size_t aux_nsub_offset(const pr_flat *h) { return up(aux_norm_offset(h) + (size_t)h->n * 4, 256); }

pr_flat_tuning_t effective_tuning(const pr_flat *h)
{
    pr_flat_tuning_t t = h->tun;
    if (t.first_chunk_rows <= 0) t.first_chunk_rows = kDefaultFirstChunk;
    if (t.growth <= 0) t.growth = kDefaultGrowth;
    if (t.cand_capacity <= 0) t.cand_capacity = kDefaultCapacity;
    return t;
}

// Upper bound, rounded up to f32, of the coefficient of |q||x| in the margin (derivation: DESIGN §4.6):
// bf16 rounding of both operands, 2 (2u + u^2), u = 2^-8, plus the tensor core's fp32 accumulation, assumed no worse
// than K 2^-22 relative to sum |q^_i x^_i| <= (1 + u)^2 |q||x|, times the 2 of -2 q.x; 2^-10 of head room covers the
// f32 evaluation of the margin itself.
float margin_c1(int K)
{
    const double u = std::ldexp(1.0, -8);
    const double c = 2.0 * ((2.0 * u + u * u) + K * std::ldexp(1.0, -22) * (1.0 + u) * (1.0 + u)) * (1.0 + std::ldexp(1.0, -10));
    return std::nextafter((float)c, INFINITY);
}

// The same for the inner-product bound q.x + margin (derivation: DESIGN §4.6): the bf16 rounding, 2u + u^2, and the
// assumed fp32 accumulation, K 2^-22 (1 + u)^2, without the factor 2; (K + 5) 2^-53 for the f64 sum of the exact score
// and 2^-22 for its f32 rounding and that of the bound's last add; 2^-10 of head room covers the f32 rounding of |q|,
// |x| and of the margin's own evaluation.
float margin_c1ip(int K)
{
    const double u = std::ldexp(1.0, -8);
    const double c = ((2.0 * u + u * u) + K * std::ldexp(1.0, -22) * (1.0 + u) * (1.0 + u) +
                      (K + 5) * std::ldexp(1.0, -53) + std::ldexp(1.0, -22)) * (1.0 + std::ldexp(1.0, -10));
    return std::nextafter((float)c, INFINITY);
}

// fp16 storage (derivation: DESIGN §4.6, "The fp16 margin").  The rows are exact, only the scaled query is rounded:
// u = 2^-11 relative where the scaled element is normal, and at most 2^-14 absolute (a subnormal flushed) where it is
// not, which is sqrt(K) 2^-28 relative to |q||x| since max |q_j| 2^e_q >= 2^14; the assumed fp32 accumulation,
// K 2^-22 relative to sum |q^_j x_j| <= (1 + 2^-10) |q||x|; then the same factor 2, f64 and f32 terms and head room as
// the bf16 coefficients above.
float margin_c1_f16(int K)
{
    const double u = std::ldexp(1.0, -11), a = u + std::sqrt((double)K) * std::ldexp(1.0, -28);
    const double c = 2.0 * (a + K * std::ldexp(1.0, -22) * (1.0 + std::ldexp(1.0, -10))) * (1.0 + std::ldexp(1.0, -10));
    return std::nextafter((float)c, INFINITY);
}

float margin_c1ip_f16(int K)
{
    const double u = std::ldexp(1.0, -11), a = u + std::sqrt((double)K) * std::ldexp(1.0, -28);
    const double c = (a + K * std::ldexp(1.0, -22) * (1.0 + std::ldexp(1.0, -10)) + (K + 5) * std::ldexp(1.0, -53) +
                      std::ldexp(1.0, -22)) * (1.0 + std::ldexp(1.0, -10));
    return std::nextafter((float)c, INFINITY);
}

// The coefficient of |q| ||x_sub||: a tensor core that flushes the row's fp16-subnormal elements loses at most
// |q^| ||x_sub|| <= (1 + 2^-10) |q| ||x_sub|| of the dot product (Cauchy-Schwarz), twice that in the L2 bound; the
// second 1 + 2^-10 covers the f32 evaluation of the term.
float margin_csub_f16(int metric)
{
    const double c = (metric == PR_METRIC_L2 ? 2.0 : 1.0) * (1.0 + std::ldexp(1.0, -10)) * (1.0 + std::ldexp(1.0, -10));
    return std::nextafter((float)c, INFINITY);
}

// The checks and the construction of every pr_flat_create*: fn is the name the messages start with, arg the name of
// the rows argument; fp16 handles hold `rows` as codes.
int flat_create(pr_flat_t **out, const char *fn, const char *arg, int device, const void *rows, int64_t n, int32_t d,
                int metric, bool fp16)
{
    if (!out || (n > 0 && !rows) || n < 0) {
        pr_set_error("%s: bad argument (null pointer or negative row count)", fn);
        return PR_EINVAL;
    }
    *out = nullptr;
    if (metric != PR_METRIC_L2 && metric != PR_METRIC_INNER_PRODUCT) {
        pr_set_error("%s: metric %d unsupported (PR_METRIC_INNER_PRODUCT = 0 or PR_METRIC_L2 = 1)", fn, metric);
        return PR_EUNSUPPORTED;
    }
    if (d < 64 || d > PR_FLAT_MAX_D || d % 64 != 0) {
        pr_set_error("%s: d = %d unsupported (a multiple of 64 in [64, %d])", fn, d, PR_FLAT_MAX_D);
        return PR_EUNSUPPORTED;
    }
    if (n > INT32_MAX) {
        pr_set_error("%s: %lld rows, at most 2^31 - 1 per index", fn, (long long)n);
        return PR_EUNSUPPORTED;
    }
    if ((uintptr_t)rows & 15) {
        pr_set_error("%s: %s must be 16-byte aligned", fn, arg);
        return PR_EINVAL;
    }
    PR_CUDA_CHECK(cudaSetDevice(device));
    int n_sm = 0;
    PR_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    pr_flat *h = new pr_flat();
    h->device = device;
    h->n_sm = n_sm;
    h->n = n;
    h->d = d;
    h->metric = metric;
    h->fp16 = fp16;
    if (fp16)
        h->codes = (const __half *)rows;
    else
        h->rows = (const float *)rows;
    *out = h;
    return PR_OK;
}

// The launches of flat.cu's f32 kernels, in the argument order of flat_fp16.cu's: the metric picks the kernel.  A function
// attribute holds for the current device only: it is set on every launch (host-only and cheap), so that an index on a
// second GPU of the process launches as the first one did.
int flat_filter_launch(int metric, unsigned grid, size_t smem, const CUtensorMap &map_x, const CUtensorMap &map_q,
                       const FilterArgs &fa, cudaStream_t st)
{
    const bool ip = metric == PR_METRIC_INNER_PRODUCT;
    const void *filter = ip ? (const void *)flat_ip_filter_kernel : (const void *)flat_filter_kernel;
    PR_CUDA_CHECK(cudaFuncSetAttribute(filter, cudaFuncAttributeMaxDynamicSharedMemorySize, kFilterSmemMax));
    if (ip)
        flat_ip_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa);
    else
        flat_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

int flat_refine_launch(int metric, int n_queries, const RefineArgs &ra, cudaStream_t st)
{
    if (metric == PR_METRIC_INNER_PRODUCT)
        flat_ip_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
    else
        flat_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

// The launch plan of both searches (stated at the top of this file) on the workspace `w` of layout `l`: theta0 is
// every query's starting bound, cap the candidates per (query, chunk) the filter stores, and refine(begin, end)
// launches the caller's refine of the chunk [begin, end) (PR_OK or an error code).  Records the launches and chunks
// in the handle.
template <typename Refine>
int flat_plan(pr_flat *h, int n_queries, const float *queries, int k, const FlatLayout &l, const FlatWs &w,
              float theta0, int cap, cudaStream_t st, Refine refine)
{
    flat_init_kernel<<<(unsigned)(((int64_t)n_queries * k + 255) / 256), 256, 0, st>>>(n_queries, k, theta0, w.theta,
                                                                                     w.count, w.topk, w.stats);
    PR_CUDA_CHECK(cudaGetLastError());
    int64_t launches = 1;
    if (h->n == 0) {
        h->last_launches = launches;
        return PR_OK;
    }
    int rc;
    if (h->fp16) {
        if ((rc = flat_fp16_prep_queries(queries, n_queries, l.b_pad, h->d, (__half *)w.q_ops, w.qn2, w.qn,
                                         w.qscale, st)) != PR_OK)
            return rc;
    } else {
        flat_prep_kernel<<<(unsigned)((l.b_pad + 7) / 8), 256, 0, st>>>(queries, n_queries, l.b_pad, h->d,
                                                                        (__nv_bfloat16 *)w.q_ops, w.qn2, w.qn);
        PR_CUDA_CHECK(cudaGetLastError());
    }
    ++launches;
    CUtensorMap map_x, map_q;
    const CUtensorMapDataType dtype = h->fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const void *x_ops = h->fp16 ? (const void *)h->codes : (const void *)h->rows_bf;
    if ((rc = make_map(&map_x, x_ops, (uint64_t)h->n, (uint64_t)h->d, kRowsPerTile, dtype)) != PR_OK) return rc;
    if ((rc = make_map(&map_q, w.q_ops, (uint64_t)l.b_pad, (uint64_t)h->d, (uint32_t)l.nq, dtype)) != PR_OK) return rc;
    const bool ip = h->metric == PR_METRIC_INNER_PRODUCT;
    const int stage_bytes = kDocTileBytes + l.nq * kBK * 2;
    FilterArgs fa;
    fa.n_queries = n_queries;
    fa.nq = l.nq;
    fa.n_qb = l.n_qb;
    fa.K = h->d;
    fa.n_stages = std::min(kMaxStages, kStageBudget / stage_bytes);
    // D f32; A and B BF16 (format 1) or, for fp16 storage, F16 (format 0); N = nq; M = 128
    fa.idesc = (1u << 4) | (h->fp16 ? 0u : (1u << 7) | (1u << 10)) | ((uint32_t)(l.nq >> 3) << 17) |
               ((uint32_t)(kRowsPerTile >> 4) << 24);
    fa.tmem_cols = 32;
    while (fa.tmem_cols < (uint32_t)(2 * l.nq)) fa.tmem_cols <<= 1;
    fa.c1 = h->fp16 ? (ip ? margin_c1ip_f16(h->d) : margin_c1_f16(h->d)) : (ip ? margin_c1ip(h->d) : margin_c1(h->d));
    fa.c2 = ip ? 0.f : std::ldexp(1.f, -17);
    fa.c3 = std::ldexp(1.f, -100);
    fa.norm2 = h->norm2;
    fa.norm = h->norm;
    fa.qn2 = w.qn2;
    fa.qn = w.qn;
    fa.theta = w.theta;
    fa.count = w.count;
    fa.cand = w.cand;
    fa.cap = cap;
    const FilterF16Args fh = {w.qscale, h->nsub, margin_csub_f16(h->metric)};   // (read by the fp16 filters only)
    const size_t smem = kFilterSmemFixed + (size_t)fa.n_stages * stage_bytes;
    const pr_flat_tuning_t tun = effective_tuning(h);
    int64_t chunk = (tun.first_chunk_rows + kRowsPerTile - 1) / kRowsPerTile * kRowsPerTile;
    for (int64_t begin = 0; begin < h->n;) {
        const int64_t end = std::min(h->n, begin + chunk);
        fa.row_begin = begin;
        fa.row_end = end;
        const int64_t tiles = (end - begin + kRowsPerTile - 1) / kRowsPerTile * l.n_qb;
        const unsigned grid = (unsigned)std::min<int64_t>(tiles, h->n_sm);
        rc = h->fp16 ? flat_fp16_filter_launch(h->metric, grid, smem, map_x, map_q, fa, fh, st)
                     : flat_filter_launch(h->metric, grid, smem, map_x, map_q, fa, st);
        if (rc != PR_OK) return rc;
        if ((rc = refine(begin, end)) != PR_OK) return rc;
        launches += 2;
        ++h->last_chunks;
        begin = end;
        chunk = std::min<int64_t>(chunk * tun.growth, (int64_t)1 << 40);
    }
    h->last_launches = launches;
    return PR_OK;
}

}  // namespace

extern "C" int pr_flat_create_metric(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d,
                                     int metric)
{
    return flat_create(out, metric == PR_METRIC_L2 ? "pr_flat_create" : "pr_flat_create_metric", "rows_dev", device,
                       rows_dev, n, d, metric, false);
}

extern "C" int pr_flat_create(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d)
{
    return flat_create(out, "pr_flat_create", "rows_dev", device, rows_dev, n, d, PR_METRIC_L2, false);
}

extern "C" int pr_flat_create_fp16(pr_flat_t **out, int device, const uint16_t *codes_dev, int64_t n, int32_t d,
                                   int metric)
{
    return flat_create(out, "pr_flat_create_fp16", "codes_dev", device, codes_dev, n, d, metric, true);
}

extern "C" int pr_flat_destroy(pr_flat_t *h)
{
    delete h;
    return PR_OK;
}

extern "C" size_t pr_flat_aux_bytes(const pr_flat_t *h)
{
    if (!h) return 0;
    return up((h->fp16 ? aux_nsub_offset(h) : aux_norm_offset(h)) + (size_t)h->n * 4, 256);
}

extern "C" int pr_flat_build_aux(pr_flat_t *h, void *aux_dev, size_t aux_bytes, pr_stream_t stream)
{
    if (!h || (!aux_dev && h->n > 0)) {
        pr_set_error("pr_flat_build_aux: null argument");
        return PR_EINVAL;
    }
    if (aux_bytes < pr_flat_aux_bytes(h)) {
        pr_set_error("pr_flat_build_aux: aux buffer of %zu bytes, need %zu", aux_bytes, pr_flat_aux_bytes(h));
        return PR_EWORKSPACE;
    }
    if ((uintptr_t)aux_dev & 1023) {
        pr_set_error("pr_flat_build_aux: aux_dev must be 1024-byte aligned");
        return PR_EINVAL;
    }
    unsigned char *a = (unsigned char *)aux_dev;
    h->rows_bf = h->fp16 ? nullptr : (const __nv_bfloat16 *)a;
    h->norm2 = (const float *)(a + aux_norm2_offset(h));
    h->norm = (const float *)(a + aux_norm_offset(h));
    if (h->fp16) h->nsub = (const float *)(a + aux_nsub_offset(h));
    if (h->n == 0) return PR_OK;
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (h->fp16) {
        int rc;
        if ((rc = flat_fp16_prep_rows(h->codes, h->n, h->d, (float *)h->norm2, (float *)h->norm, (float *)h->nsub,
                                      st)) != PR_OK)
            return rc;
    } else {
        flat_prep_kernel<<<(unsigned)((h->n + 7) / 8), 256, 0, st>>>(h->rows, h->n, h->n, h->d,
                                                                     (__nv_bfloat16 *)h->rows_bf, (float *)h->norm2,
                                                                     (float *)h->norm);
        PR_CUDA_CHECK(cudaGetLastError());
    }
    PR_CUDA_CHECK(cudaStreamSynchronize(st));
    return PR_OK;
}

extern "C" int pr_flat_set_tuning(pr_flat_t *h, const pr_flat_tuning_t *t)
{
    if (!h || !t || t->first_chunk_rows < 0 || t->growth < 0 || t->cand_capacity < 0) {
        pr_set_error("pr_flat_set_tuning: bad argument (null pointer or negative field)");
        return PR_EINVAL;
    }
    h->tun = *t;
    return PR_OK;
}

extern "C" int pr_flat_get_tuning(const pr_flat_t *h, pr_flat_tuning_t *t)
{
    if (!h || !t) {
        pr_set_error("pr_flat_get_tuning: null argument");
        return PR_EINVAL;
    }
    *t = effective_tuning(h);
    return PR_OK;
}

extern "C" size_t pr_flat_workspace_bytes(const pr_flat_t *h, int32_t n_queries, int32_t k)
{
    if (!h || n_queries < 1 || k < 1 || k > PR_MAX_K) return 0;
    return flat_layout(h->d, n_queries, k, effective_tuning(h).cand_capacity, h->fp16).total;
}

extern "C" int pr_flat_search(pr_flat_t *h, int32_t n_queries, const float *queries_dev, int32_t k, float *out_dist_dev,
                              int64_t *out_ids_dev, void *workspace_dev, size_t workspace_bytes, pr_stream_t stream)
{
    if (!h || n_queries < 0 || (n_queries > 0 && (!queries_dev || !out_dist_dev || !out_ids_dev || !workspace_dev))) {
        pr_set_error("pr_flat_search: bad argument (null pointer or negative batch)");
        return PR_EINVAL;
    }
    if (k < 1 || k > PR_MAX_K) {
        pr_set_error("pr_flat_search: k must be in [1, %d], got %d", PR_MAX_K, k);
        return PR_EINVAL;
    }
    if (h->n > 0 && !h->norm2) {
        pr_set_error("pr_flat_search: pr_flat_build_aux has not been called on this handle");
        return PR_EINVAL;
    }
    if (((uintptr_t)queries_dev & 15) || ((uintptr_t)workspace_dev & 1023)) {
        pr_set_error("pr_flat_search: queries_dev must be 16-byte aligned, workspace_dev 1024-byte aligned");
        return PR_EINVAL;
    }
    h->last_launches = 0;
    h->last_chunks = 0;
    if (n_queries == 0) return PR_OK;
    const int cap = effective_tuning(h).cand_capacity;
    const FlatLayout l = flat_layout(h->d, n_queries, k, cap, h->fp16);
    if (workspace_bytes < l.total) {
        pr_set_error("pr_flat_search: workspace of %zu bytes, need %zu", workspace_bytes, l.total);
        return PR_EWORKSPACE;
    }
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const FlatWs w = flat_ws(l, workspace_dev);
    RefineArgs ra;
    ra.rows = h->rows;
    ra.rows_h = h->codes;
    ra.queries = queries_dev;
    ra.d = h->d;
    ra.k = k;
    ra.cap = cap;
    ra.count = w.count;
    ra.cand = w.cand;
    ra.topk = w.topk;
    ra.theta = w.theta;
    ra.stats = w.stats;
    const float theta0 = h->metric == PR_METRIC_INNER_PRODUCT ? -INFINITY : INFINITY;
    const int rc = flat_plan(h, n_queries, queries_dev, k, l, w, theta0, cap, st, [&](int64_t begin, int64_t end) {
        ra.row_begin = begin;
        ra.row_end = end;
        return h->fp16 ? flat_fp16_refine_launch(h->metric, n_queries, ra, st)
                       : flat_refine_launch(h->metric, n_queries, ra, st);
    });
    if (rc != PR_OK) return rc;
    const int64_t total = (int64_t)n_queries * k;
    flat_output_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, w.topk, out_dist_dev, out_ids_dev,
                                                                       h->metric);
    PR_CUDA_CHECK(cudaGetLastError());
    ++h->last_launches;
    return PR_OK;
}

extern "C" int pr_flat_last_stats(const pr_flat_t *h, const void *workspace_dev, int32_t n_queries, int32_t k,
                                  pr_flat_stats_t *out, pr_stream_t stream)
{
    if (!h || !workspace_dev || !out || n_queries < 1 || k < 1 || k > PR_MAX_K) {
        pr_set_error("pr_flat_last_stats: bad argument");
        return PR_EINVAL;
    }
    const FlatLayout l = flat_layout(h->d, n_queries, k, effective_tuning(h).cand_capacity, h->fp16);
    unsigned long long s[4];
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    PR_CUDA_CHECK(cudaMemcpyAsync(s, flat_ws(l, const_cast<void *>(workspace_dev)).stats, sizeof(s),
                                  cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    PR_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    out->launches = h->last_launches;
    out->chunks = h->last_chunks;
    out->candidates = (int64_t)s[0];
    out->max_candidates = (int64_t)s[1];
    out->fallback_queries = (int64_t)s[2];
    return PR_OK;
}

// The workspace of a search at k = 1, so that pr_flat_last_stats(..., k = 1) reads the range search's counters.
extern "C" size_t pr_flat_range_workspace_bytes(const pr_flat_t *h, int32_t n_queries)
{
    if (!h || n_queries < 1) return 0;
    return flat_layout(h->d, n_queries, 1, effective_tuning(h).cand_capacity, h->fp16).total;
}

extern "C" int pr_flat_range_search(pr_flat_t *h, int32_t n_queries, const float *queries_dev, float radius,
                                    const int64_t *lims_in_dev, int64_t *count_dev, float *dist_dev, int64_t *ids_dev,
                                    void *workspace_dev, size_t workspace_bytes, pr_stream_t stream)
{
    if (!h || n_queries < 0 || (n_queries > 0 && (!queries_dev || !lims_in_dev || !count_dev || !dist_dev || !ids_dev ||
                                                  !workspace_dev))) {
        pr_set_error("pr_flat_range_search: bad argument (null pointer or negative batch)");
        return PR_EINVAL;
    }
    if (h->n > 0 && !h->norm2) {
        pr_set_error("pr_flat_range_search: pr_flat_build_aux has not been called on this handle");
        return PR_EINVAL;
    }
    if (((uintptr_t)queries_dev & 15) || ((uintptr_t)workspace_dev & 1023) || ((uintptr_t)lims_in_dev & 7) ||
        ((uintptr_t)count_dev & 7) || ((uintptr_t)dist_dev & 3) || ((uintptr_t)ids_dev & 7)) {
        pr_set_error("pr_flat_range_search: queries_dev must be 16-byte aligned, workspace_dev 1024-byte aligned, "
                     "lims_in_dev, count_dev and ids_dev 8-byte aligned, dist_dev 4-byte aligned");
        return PR_EINVAL;
    }
    h->last_launches = 0;
    h->last_chunks = 0;
    if (n_queries == 0) return PR_OK;
    const pr_flat_tuning_t tun = effective_tuning(h);
    const FlatLayout l = flat_layout(h->d, n_queries, 1, tun.cand_capacity, h->fp16);
    if (workspace_bytes < l.total) {
        pr_set_error("pr_flat_range_search: workspace of %zu bytes, need %zu", workspace_bytes, l.total);
        return PR_EWORKSPACE;
    }
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const FlatWs w = flat_ws(l, workspace_dev);
    PR_CUDA_CHECK(cudaMemsetAsync(count_dev, 0, (size_t)n_queries * sizeof(int64_t), st));
    if (std::isnan(radius)) {                  // no results; the counters read zero
        PR_CUDA_CHECK(cudaMemsetAsync(w.stats, 0, 4 * 8, st));
        return PR_OK;
    }
    FlatRangeArgs ra;
    ra.rows = h->rows;
    ra.rows_h = h->codes;
    ra.queries = queries_dev;
    ra.d = h->d;
    ra.cap = std::min<int>(tun.cand_capacity, kFlatRangeMaxCap);
    ra.radius = radius;
    ra.count = w.count;
    ra.cand = w.cand;
    ra.lims = lims_in_dev;
    ra.hits = count_dev;
    ra.dist = dist_dev;
    ra.ids = ids_dev;
    ra.stats = w.stats;
    return flat_plan(h, n_queries, queries_dev, 1, l, w, radius, ra.cap, st, [&](int64_t begin, int64_t end) {
        ra.row_begin = begin;
        ra.row_end = end;
        return h->fp16 ? flat_fp16_range_refine_launch(h->metric, n_queries, ra, st)
                       : flat_range_refine_launch(h->metric, n_queries, ra, st);
    });
}

extern "C" int pr_flat_merge_metric(int32_t n_queries, int32_t k, int32_t n_lists, const float *dist_dev,
                                    const int64_t *ids_dev, const int64_t *id_base, float *out_dist_dev,
                                    int64_t *out_ids_dev, pr_stream_t stream, int metric)
{
    const char *fn = metric == PR_METRIC_L2 ? "pr_flat_merge" : "pr_flat_merge_metric";
    if (n_queries < 0 || !id_base ||
        (n_queries > 0 && (!dist_dev || !ids_dev || !out_dist_dev || !out_ids_dev))) {
        pr_set_error("%s: bad argument (null pointer or negative batch)", fn);
        return PR_EINVAL;
    }
    if (metric != PR_METRIC_L2 && metric != PR_METRIC_INNER_PRODUCT) {
        pr_set_error("%s: metric %d unsupported (PR_METRIC_INNER_PRODUCT = 0 or PR_METRIC_L2 = 1)", fn, metric);
        return PR_EUNSUPPORTED;
    }
    if (n_lists < 1 || n_lists > PR_FLAT_MAX_LISTS) {
        pr_set_error("%s: n_lists must be in [1, %d], got %d", fn, PR_FLAT_MAX_LISTS, n_lists);
        return PR_EINVAL;
    }
    if (k < 1 || k > PR_MAX_K) {
        pr_set_error("%s: k must be in [1, %d], got %d", fn, PR_MAX_K, k);
        return PR_EINVAL;
    }
    MergeArgs a;
    for (int l = 0; l < n_lists; ++l) {
        if (id_base[l] < 0) {
            pr_set_error("%s: id_base[%d] = %lld is negative", fn, l, (long long)id_base[l]);
            return PR_EINVAL;
        }
        a.base[l] = id_base[l];
    }
    if (n_queries == 0) return PR_OK;
    const size_t per_warp = (size_t)n_lists * k * (sizeof(float) + sizeof(int64_t));
    a.n_queries = n_queries;
    a.k = k;
    a.n_lists = n_lists;
    a.metric = metric;
    a.warps = (int)std::max<size_t>(1, std::min<size_t>(kMergeMaxWarps, kMergeSmemBudget / per_warp));
    a.dist = dist_dev;
    a.ids = ids_dev;
    a.out_dist = out_dist_dev;
    a.out_ids = out_ids_dev;
    const unsigned grid = (unsigned)((n_queries + a.warps - 1) / a.warps);
    flat_merge_kernel<<<grid, a.warps * 32, a.warps * per_warp, (cudaStream_t)stream>>>(a);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

extern "C" int pr_flat_merge(int32_t n_queries, int32_t k, int32_t n_lists, const float *dist_dev, const int64_t *ids_dev,
                             const int64_t *id_base, float *out_dist_dev, int64_t *out_ids_dev, pr_stream_t stream)
{
    return pr_flat_merge_metric(n_queries, k, n_lists, dist_dev, ids_dev, id_base, out_dist_dev, out_ids_dev, stream,
                                PR_METRIC_L2);
}
