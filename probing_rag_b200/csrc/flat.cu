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
//   merge    flat_merge_kernel       pr_flat_merge: the lists of row-range shards -> one list in the same order
//
// The rows are cut into chunks of growing size; filter and refine alternate per chunk on the caller's stream, so
// every chunk filters with the bound the earlier ones established ("bounds raised between launches", as BM25 does).
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
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
    pr_flat_tuning_t tun;
    int64_t last_launches, last_chunks;
};

namespace {

constexpr int kRowsPerTile = 128;
constexpr int kMaxNQ = 256;
constexpr int kMaxStages = 8;
constexpr int kDocTileBytes = kRowsPerTile * kBK * 2;   // 16 KB
constexpr int kStageBudget = 192 * 1024;
constexpr int kFilterThreads = 256;
constexpr int kRefineThreads = 256;
constexpr int kRefineKeys = 2048;                       // running list + new exact candidates of one round
constexpr uint64_t kEmptyKey = ~0ull;
constexpr int64_t kDefaultFirstChunk = 2048;
constexpr int32_t kDefaultGrowth = 4;
constexpr int32_t kDefaultCapacity = 8192;

inline size_t up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Key of an inner-product score's bits: ascends as the score descends (+inf first, -inf last), with every NaN mapped
// to 0xFFFFFFFF, above -inf.  ip_bits inverts it (a NaN comes back as the NaN 0xFFFFFFFF).
__device__ __forceinline__ uint32_t ip_key(uint32_t bits)
{
    if ((bits & 0x7FFFFFFFu) > 0x7F800000u) return 0xFFFFFFFFu;
    return (bits & 0x80000000u) ? bits : bits ^ 0x7FFFFFFFu;
}

__device__ __forceinline__ uint32_t ip_bits(uint32_t key) { return (key & 0x80000000u) ? key : key ^ 0x7FFFFFFFu; }

// Key of a squared L2 distance's bits: the bits themselves (a distance is +0, positive or +inf), with every NaN, of
// either sign and any payload, mapped to 0x7FFFFFFF, above +inf.  The key is also the distance returned, so a NaN
// distance comes back as the NaN 0x7FFFFFFF.
__device__ __forceinline__ uint32_t l2_key(uint32_t bits)
{
    return (bits & 0x7FFFFFFFu) > 0x7F800000u ? 0x7FFFFFFFu : bits;
}

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

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

// ------------------------------------------------------------------------------------ filter
struct FilterArgs {
    int64_t row_begin, row_end;     // the chunk
    int n_queries, nq, n_qb;        // batch, queries per tile (multiple of 32), query blocks
    int K;                          // d
    int n_stages;
    uint32_t idesc;
    uint32_t tmem_cols;
    float c1, c2, c3;               // margin(q, x) = c1 |q| |x| + c2 (|q|^2 + |x|^2) + c3 (1 + |q| + |x|) (IP: c2 = 0)
    const float *norm2, *norm;      // rows
    const float *qn2, *qn;          // queries
    const float *theta;
    int32_t *count;
    int32_t *cand;
    int cap;
};

// The GEMM and its pipeline are shared; M (PR_METRIC_*) selects only the epilogue's bound and comparison.
template <int M>
__device__ __forceinline__ void flat_filter(const CUtensorMap &map_x, const CUtensorMap &map_q, const FilterArgs &g)
{
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    const int stage_bytes = kDocTileBytes + g.nq * kBK * 2;
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + (size_t)g.n_stages * stage_bytes);
    uint64_t *empty_bar = full_bar + kMaxStages;
    uint64_t *tfull_bar = empty_bar + kMaxStages;   // [2] accumulator complete
    uint64_t *tempty_bar = tfull_bar + 2;           // [2] accumulator drained by the epilogue
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_row_tiles = (g.row_end - g.row_begin + kRowsPerTile - 1) / kRowsPerTile;
    const int64_t n_tiles = n_row_tiles * g.n_qb;
    const int n_kb = g.K / kBK;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < g.n_stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4);   // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) tmem_alloc_1cta(tmem_slot, g.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer
        uint32_t kb_total = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const int row0 = (int)(g.row_begin + (t / g.n_qb) * kRowsPerTile);
            const int q0 = (int)(t % g.n_qb) * g.nq;
            for (int kb = 0; kb < n_kb; ++kb, ++kb_total) {
                const int s = (int)(kb_total % (uint32_t)g.n_stages);
                const uint32_t ph = (kb_total / (uint32_t)g.n_stages) & 1u;
                mbar_wait(&empty_bar[s], ph ^ 1u);
                unsigned char *st = smem + (size_t)s * stage_bytes;
                mbar_expect_tx(&full_bar[s], (uint32_t)stage_bytes);
                tma_load_2d(st, &map_x, &full_bar[s], kb * kBK, row0);
                tma_load_2d(st + kDocTileBytes, &map_q, &full_bar[s], kb * kBK, q0);
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer: acc[a][128 rows][nq queries] = X_tile . Q_tile^T
        uint32_t kb_total = 0, it = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t a = it & 1u;
            mbar_wait(&tempty_bar[a], ((it >> 1) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + a * (uint32_t)g.nq;
            for (int kb = 0; kb < n_kb; ++kb, ++kb_total) {
                const int s = (int)(kb_total % (uint32_t)g.n_stages);
                const uint32_t ph = (kb_total / (uint32_t)g.n_stages) & 1u;
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + (size_t)s * stage_bytes);
                const uint64_t da = umma_desc_sw128(st), db = umma_desc_sw128(st + kDocTileBytes);
#pragma unroll
                for (int k = 0; k < kBK / 16; ++k) {
                    const uint64_t adv = (uint64_t)((k * 16 * 2) >> 4);
                    umma_bf16_1cta(d_tmem, da + adv, db + adv, g.idesc, (kb | k) ? 1u : 0u);
                }
                umma_commit_1cta(&empty_bar[s]);
            }
            umma_commit_1cta(&tfull_bar[a]);
        }
    } else if (warp >= 4) {
        // ===== epilogue: thread = one row of the tile (TMEM lane), 32 query columns per tcgen05.ld
        const int quad = warp & 3;
        uint32_t it = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t a = it & 1u;
            const int64_t row = g.row_begin + (t / g.n_qb) * kRowsPerTile + quad * 32 + lane;
            const int q0 = (int)(t % g.n_qb) * g.nq;
            const bool live = row < g.row_end;
            const float nx2 = (M == PR_METRIC_L2 && live) ? __ldg(g.norm2 + row) : 0.f;
            const float nx = live ? __ldg(g.norm + row) : 0.f;
            mbar_wait(&tfull_bar[a], (it >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr = tmem_base + a * (uint32_t)g.nq + ((uint32_t)(quad * 32) << 16);
            for (int c0 = 0; c0 < g.nq && q0 + c0 < g.n_queries; c0 += 32) {
                uint32_t r[32];
                tmem_ld32_nowait(taddr + (uint32_t)c0, r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int q = q0 + c0 + j;
                    if (q >= g.n_queries) continue;   // (warp-uniform)
                    bool take;
                    if constexpr (M == PR_METRIC_L2) {
                        const float qn2 = __ldg(g.qn2 + q), qn = __ldg(g.qn + q), th = __ldg(g.theta + q);
                        const float s2 = qn2 + nx2;
                        const float margin = fmaf(g.c1 * qn, nx, fmaf(g.c2, s2, g.c3 * (1.f + qn + nx)));
                        const float bound = fmaf(-2.f, __uint_as_float(r[j]), s2) - margin;
                        take = live && !(bound > th);          // (a NaN bound is a candidate)
                    } else {
                        const float qn = __ldg(g.qn + q), th = __ldg(g.theta + q);
                        const float bound = __uint_as_float(r[j]) + fmaf(g.c1 * qn, nx, g.c3 * (1.f + qn + nx));
                        take = live && !(bound < th);          // (a NaN bound is a candidate)
                    }
                    const unsigned m = __ballot_sync(PR_FULL_MASK, take);
                    if (m) {
                        int base = 0;
                        const int leader = __ffs(m) - 1;
                        if (lane == leader) base = atomicAdd(g.count + q, __popc(m));
                        base = __shfl_sync(PR_FULL_MASK, base, leader);
                        const int slot = base + __popc(m & ((1u << lane) - 1u));
                        if (take && slot < g.cap) g.cand[(size_t)q * g.cap + slot] = (int32_t)row;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[a]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_1cta(tmem_base, g.tmem_cols);
    }
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

// ------------------------------------------------------------------------------------ refine
// The exact distance (DESIGN §3): lane l sums (q_j - x_j)^2 over j = l, l+32, ... in increasing j, every difference,
// square and add a separately rounded f64 operation (no contraction), then an xor butterfly over the 32 lanes
// (offsets 16, 8, 4, 2, 1), rounded once to f32.  Every lane ends with the same value.
__device__ __forceinline__ float exact_dist(const float *__restrict__ sq, const float *__restrict__ x, int d, int lane)
{
    double s = 0.0;
    for (int j = lane; j < d; j += 32) {
        const double df = __dsub_rn((double)sq[j], (double)__ldg(x + j));
        s = __dadd_rn(s, __dmul_rn(df, df));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(PR_FULL_MASK, s, o));
    return __double2float_rn(s);
}

// The exact inner product (DESIGN §3): lane l starts at +0.0 and adds q_j x_j over j = l, l+32, ... in increasing j
// (the product of two floats is exact in f64; __dmul_rn keeps it from contracting into an FMA), then the same butterfly
// and one rounding to f32.  A negative sum that underflows f32 would round to -0; adding +0 makes it +0, so a score is
// never -0.
__device__ __forceinline__ float exact_ip(const float *__restrict__ sq, const float *__restrict__ x, int d, int lane)
{
    double s = 0.0;
    for (int j = lane; j < d; j += 32) s = __dadd_rn(s, __dmul_rn((double)sq[j], (double)__ldg(x + j)));
#pragma unroll
    for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(PR_FULL_MASK, s, o));
    return __fadd_rn(__double2float_rn(s), 0.f);
}

// ascending bitonic sort of keys[0, n), n a power of two, by the whole block
__device__ void block_bitonic_sort(uint64_t *keys, int n)
{
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const uint64_t a = keys[lo], b = keys[hi];
                if ((a > b) == asc) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
        }
    }
    __syncthreads();
}

struct RefineArgs {
    const float *rows, *queries;
    int d, k, cap;
    int64_t row_begin, row_end;
    int32_t *count;
    const int32_t *cand;
    uint64_t *topk;                 // [B][k] keys (l2_key of the distance or ip_key of the score, << 32 | row), ascending
    float *theta;
    unsigned long long *stats;      // candidates, max candidates, fallback queries
};

template <int M>
__device__ __forceinline__ void flat_refine(const RefineArgs &g)
{
    __shared__ uint64_t s_keys[kRefineKeys];
    __shared__ float s_q[PR_FLAT_MAX_D];
    __shared__ int s_new;
    const int q = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_warps = blockDim.x >> 5;
    const int cnt = g.count[q];
    const bool overflow = cnt > g.cap;
    const int64_t n_items = overflow ? g.row_end - g.row_begin : cnt;
    for (int j = threadIdx.x; j < g.d; j += blockDim.x) s_q[j] = g.queries[(size_t)q * g.d + j];
    for (int i = threadIdx.x; i < g.k; i += blockDim.x) s_keys[i] = g.topk[(size_t)q * g.k + i];
    if (threadIdx.x == 0) {
        s_new = 0;
        if (cnt) {
            atomicAdd(g.stats + 0, (unsigned long long)cnt);
            atomicMax(g.stats + 1, (unsigned long long)cnt);
        }
        if (overflow) atomicAdd(g.stats + 2, 1ull);
    }
    __syncthreads();
    uint64_t kth = s_keys[g.k - 1];
    const int round = kRefineKeys - g.k;
    for (int64_t base = 0; base < n_items; base += round) {
        const int64_t end = min(n_items, base + round);
        for (int64_t i = base + warp; i < end; i += n_warps) {
            const int64_t row = overflow ? g.row_begin + i : (int64_t)g.cand[(size_t)q * g.cap + i];
            uint32_t hi;
            if constexpr (M == PR_METRIC_L2)
                hi = l2_key(__float_as_uint(exact_dist(s_q, g.rows + row * g.d, g.d, lane)));
            else
                hi = ip_key(__float_as_uint(exact_ip(s_q, g.rows + row * g.d, g.d, lane)));
            const uint64_t key = ((uint64_t)hi << 32) | (uint64_t)row;
            if (lane == 0 && key < kth) s_keys[g.k + atomicAdd(&s_new, 1)] = key;
        }
        __syncthreads();
        const int m = g.k + s_new;
        if (m > g.k) {
            int p = 1;
            while (p < m) p <<= 1;
            for (int i = m + threadIdx.x; i < p; i += blockDim.x) s_keys[i] = kEmptyKey;
            block_bitonic_sort(s_keys, p);
            kth = s_keys[g.k - 1];
        }
        __syncthreads();
        if (threadIdx.x == 0) s_new = 0;
        __syncthreads();
    }
    for (int i = threadIdx.x; i < g.k; i += blockDim.x) g.topk[(size_t)q * g.k + i] = s_keys[i];
    if (threadIdx.x == 0) {
        if constexpr (M == PR_METRIC_L2)
            g.theta[q] = kth == kEmptyKey ? INFINITY : __uint_as_float((uint32_t)(kth >> 32));
        else
            g.theta[q] = kth == kEmptyKey ? -INFINITY : __uint_as_float(ip_bits((uint32_t)(kth >> 32)));
        g.count[q] = 0;
    }
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
    size_t q_bf, qn2, qn, theta, count, cand, topk, stats, total;
};

// queries per tile: as few 32-column groups as cover the batch in equal blocks of at most 256
FlatLayout flat_layout(int d, int n_queries, int k, int cap)
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
    l.total = o;
    return l;
}

size_t aux_norm2_offset(const pr_flat *h) { return up((size_t)h->n * h->d * 2, 256); }
size_t aux_norm_offset(const pr_flat *h) { return up(aux_norm2_offset(h) + (size_t)h->n * 4, 256); }

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

}  // namespace

extern "C" int pr_flat_create_metric(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d,
                                     int metric)
{
    const char *fn = metric == PR_METRIC_L2 ? "pr_flat_create" : "pr_flat_create_metric";
    if (!out || (n > 0 && !rows_dev) || n < 0) {
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
    if ((uintptr_t)rows_dev & 15) {
        pr_set_error("%s: rows_dev must be 16-byte aligned", fn);
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
    h->rows = rows_dev;
    h->metric = metric;
    *out = h;
    return PR_OK;
}

extern "C" int pr_flat_create(pr_flat_t **out, int device, const float *rows_dev, int64_t n, int32_t d)
{
    return pr_flat_create_metric(out, device, rows_dev, n, d, PR_METRIC_L2);
}

extern "C" int pr_flat_destroy(pr_flat_t *h)
{
    delete h;
    return PR_OK;
}

extern "C" size_t pr_flat_aux_bytes(const pr_flat_t *h)
{
    if (!h) return 0;
    return up(aux_norm_offset(h) + (size_t)h->n * 4, 256);
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
    h->rows_bf = (const __nv_bfloat16 *)a;
    h->norm2 = (const float *)(a + aux_norm2_offset(h));
    h->norm = (const float *)(a + aux_norm_offset(h));
    if (h->n == 0) return PR_OK;
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t blocks = (h->n + 7) / 8;
    flat_prep_kernel<<<(unsigned)blocks, 256, 0, st>>>(h->rows, h->n, h->n, h->d, (__nv_bfloat16 *)h->rows_bf,
                                                       (float *)h->norm2, (float *)h->norm);
    PR_CUDA_CHECK(cudaGetLastError());
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
    return flat_layout(h->d, n_queries, k, effective_tuning(h).cand_capacity).total;
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
    if (h->n > 0 && !h->rows_bf) {
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
    const pr_flat_tuning_t tun = effective_tuning(h);
    const FlatLayout l = flat_layout(h->d, n_queries, k, tun.cand_capacity);
    if (workspace_bytes < l.total) {
        pr_set_error("pr_flat_search: workspace of %zu bytes, need %zu", workspace_bytes, l.total);
        return PR_EWORKSPACE;
    }
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace_dev;
    __nv_bfloat16 *q_bf = (__nv_bfloat16 *)(ws + l.q_bf);
    float *qn2 = (float *)(ws + l.qn2), *qn = (float *)(ws + l.qn), *theta = (float *)(ws + l.theta);
    int32_t *count = (int32_t *)(ws + l.count), *cand = (int32_t *)(ws + l.cand);
    uint64_t *topk = (uint64_t *)(ws + l.topk);
    unsigned long long *stats = (unsigned long long *)(ws + l.stats);
    const int64_t total = (int64_t)n_queries * k;

    const bool ip = h->metric == PR_METRIC_INNER_PRODUCT;
    flat_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(n_queries, k, ip ? -INFINITY : INFINITY, theta,
                                                                     count, topk, stats);
    int64_t launches = 1;
    if (h->n > 0) {
        flat_prep_kernel<<<(unsigned)((l.b_pad + 7) / 8), 256, 0, st>>>(queries_dev, n_queries, l.b_pad, h->d, q_bf, qn2, qn);
        ++launches;
        CUtensorMap map_x, map_q;
        int rc;
        if ((rc = make_map(&map_x, h->rows_bf, (uint64_t)h->n, (uint64_t)h->d, kRowsPerTile)) != PR_OK) return rc;
        if ((rc = make_map(&map_q, q_bf, (uint64_t)l.b_pad, (uint64_t)h->d, (uint32_t)l.nq)) != PR_OK) return rc;
        const int stage_bytes = kDocTileBytes + l.nq * kBK * 2;
        FilterArgs fa;
        fa.n_queries = n_queries;
        fa.nq = l.nq;
        fa.n_qb = l.n_qb;
        fa.K = h->d;
        fa.n_stages = std::min(kMaxStages, kStageBudget / stage_bytes);
        fa.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(l.nq >> 3) << 17) | ((uint32_t)(kRowsPerTile >> 4) << 24);
        fa.tmem_cols = 32;
        while (fa.tmem_cols < (uint32_t)(2 * l.nq)) fa.tmem_cols <<= 1;
        fa.c1 = ip ? margin_c1ip(h->d) : margin_c1(h->d);
        fa.c2 = ip ? 0.f : std::ldexp(1.f, -17);
        fa.c3 = std::ldexp(1.f, -100);
        fa.norm2 = h->norm2;
        fa.norm = h->norm;
        fa.qn2 = qn2;
        fa.qn = qn;
        fa.theta = theta;
        fa.count = count;
        fa.cand = cand;
        fa.cap = tun.cand_capacity;
        const size_t smem = 1024 + (size_t)fa.n_stages * stage_bytes + (2 * kMaxStages + 4) * 8 + 16;
        const void *filter = ip ? (const void *)flat_ip_filter_kernel : (const void *)flat_filter_kernel;
        // A function attribute holds for the current device only: set it on every call (host-only and cheap), so that
        // an index on a second GPU of the process launches as the first one did.
        PR_CUDA_CHECK(cudaFuncSetAttribute(filter, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           1024 + kStageBudget + (2 * kMaxStages + 4) * 8 + 16));
        RefineArgs ra;
        ra.rows = h->rows;
        ra.queries = queries_dev;
        ra.d = h->d;
        ra.k = k;
        ra.cap = tun.cand_capacity;
        ra.count = count;
        ra.cand = cand;
        ra.topk = topk;
        ra.theta = theta;
        ra.stats = stats;
        int64_t chunk = (tun.first_chunk_rows + kRowsPerTile - 1) / kRowsPerTile * kRowsPerTile;
        for (int64_t begin = 0; begin < h->n;) {
            const int64_t end = std::min(h->n, begin + chunk);
            fa.row_begin = ra.row_begin = begin;
            fa.row_end = ra.row_end = end;
            const int64_t tiles = (end - begin + kRowsPerTile - 1) / kRowsPerTile * l.n_qb;
            const unsigned grid = (unsigned)std::min<int64_t>(tiles, h->n_sm);
            if (ip) {
                flat_ip_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa);
                flat_ip_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
            } else {
                flat_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa);
                flat_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
            }
            PR_CUDA_CHECK(cudaGetLastError());
            launches += 2;
            ++h->last_chunks;
            begin = end;
            chunk = std::min<int64_t>(chunk * tun.growth, (int64_t)1 << 40);
        }
    }
    flat_output_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, topk, out_dist_dev, out_ids_dev,
                                                                       h->metric);
    PR_CUDA_CHECK(cudaGetLastError());
    h->last_launches = launches + 1;
    return PR_OK;
}

extern "C" int pr_flat_last_stats(const pr_flat_t *h, const void *workspace_dev, int32_t n_queries, int32_t k,
                                  pr_flat_stats_t *out, pr_stream_t stream)
{
    if (!h || !workspace_dev || !out || n_queries < 1 || k < 1 || k > PR_MAX_K) {
        pr_set_error("pr_flat_last_stats: bad argument");
        return PR_EINVAL;
    }
    const FlatLayout l = flat_layout(h->d, n_queries, k, effective_tuning(h).cand_capacity);
    unsigned long long s[4];
    PR_CUDA_CHECK(cudaSetDevice(h->device));
    PR_CUDA_CHECK(cudaMemcpyAsync(s, (const unsigned char *)workspace_dev + l.stats, sizeof(s), cudaMemcpyDeviceToHost,
                                  (cudaStream_t)stream));
    PR_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    out->launches = h->last_launches;
    out->chunks = h->last_chunks;
    out->candidates = (int64_t)s[0];
    out->max_candidates = (int64_t)s[1];
    out->fallback_queries = (int64_t)s[2];
    return PR_OK;
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
