// The filter GEMM and the top-k refine of the exact flat search, shared by the f32-row kernels of flat.cu (bf16 filter)
// and the fp16-row kernels of flat_fp16.cu; each translation unit instantiates the templates it launches.  The
// algorithm is described at the top of flat.cu and in DESIGN §4.6.
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "flat_exact.cuh"
#include "tcgen05.cuh"

namespace {

constexpr int kRowsPerTile = 128;
constexpr int kMaxNQ = 256;
constexpr int kMaxStages = 8;
constexpr int kDocTileBytes = kRowsPerTile * kBK * 2;   // 16 KB
constexpr int kStageBudget = 192 * 1024;
constexpr int kFilterSmemFixed = 1024 + (2 * kMaxStages + 4) * 8 + 16;   // alignment slack, barriers, TMEM slot
constexpr int kFilterSmemMax = kFilterSmemFixed + kStageBudget;          // the filters' dynamic shared memory limit
constexpr int kFilterThreads = 256;
constexpr int kRefineThreads = 256;
constexpr int kRefineKeys = 2048;                       // running list + new exact candidates of one round
constexpr uint64_t kEmptyKey = ~0ull;
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

}  // namespace

// The kernels' argument structs (outside the anonymous namespace: flat.cu fills them for the launches of flat_fp16.cu).
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

// What the fp16 filter reads besides FilterArgs: a parameter of its own, since a larger FilterArgs changed the bf16
// kernels' SASS.
struct FilterF16Args {
    const float *qscale;            // per query: 2^-e_q, the inverse of the scale of its fp16 copy
    const float *nsub;              // per row: ||x_sub||, rounded up (the row's fp16-subnormal elements)
    float csub;                     // margin(q, x) += csub |q| ||x_sub||
};

struct RefineArgs {
    const float *rows, *queries;
    int d, k, cap;
    int64_t row_begin, row_end;
    int32_t *count;
    const int32_t *cand;
    uint64_t *topk;                 // [B][k] keys (l2_key of the distance or ip_key of the score, << 32 | row), ascending
    float *theta;
    unsigned long long *stats;      // candidates, max candidates, fallback queries
    const __half *rows_h;           // fp16 storage: the rows (then `rows` is unused; appended, as in FilterArgs)
};

namespace {

// ------------------------------------------------------------------------------------ filter
// The GEMM and its pipeline are shared; M (PR_METRIC_*) selects only the epilogue's bound and comparison.  F16: the
// operands are fp16 (the rows as stored, the queries scaled by 2^e_q), so the epilogue unscales the accumulator by
// qscale[q] and adds the margin's csub |q| ||x_sub|| term (DESIGN §4.6).
template <int M, bool F16 = false>
__device__ __forceinline__ void flat_filter(const CUtensorMap &map_x, const CUtensorMap &map_q, const FilterArgs &g,
                                            const FilterF16Args &h = FilterF16Args{})
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
            float nsub = 0.f;
            if constexpr (F16) nsub = live ? __ldg(h.nsub + row) : 0.f;
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
                    if constexpr (F16 && M == PR_METRIC_L2) {
                        const float qn2 = __ldg(g.qn2 + q), qn = __ldg(g.qn + q), th = __ldg(g.theta + q);
                        const float s2 = qn2 + nx2;
                        const float margin = fmaf(g.c1 * qn, nx, fmaf(h.csub * qn, nsub,
                                                                      fmaf(g.c2, s2, g.c3 * (1.f + qn + nx))));
                        const float dot = __uint_as_float(r[j]) * __ldg(h.qscale + q);
                        const float bound = fmaf(-2.f, dot, s2) - margin;
                        take = live && !(bound > th);          // (a NaN bound is a candidate)
                    } else if constexpr (F16) {
                        const float qn = __ldg(g.qn + q), th = __ldg(g.theta + q);
                        const float dot = __uint_as_float(r[j]) * __ldg(h.qscale + q);
                        const float bound = dot + fmaf(g.c1 * qn, nx, fmaf(h.csub * qn, nsub, g.c3 * (1.f + qn + nx)));
                        take = live && !(bound < th);          // (a NaN bound is a candidate)
                    } else if constexpr (M == PR_METRIC_L2) {
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

// ------------------------------------------------------------------------------------ refine
// T is the rows' storage type (float, or __half for fp16 storage).
template <int M, typename T = float>
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
                hi = l2_key(__float_as_uint(exact_dist(s_q, rows_of<T>(g) + row * g.d, g.d, lane)));
            else
                hi = ip_key(__float_as_uint(exact_ip(s_q, rows_of<T>(g) + row * g.d, g.d, lane)));
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

}  // namespace

// ------------------------------------------------------------------------------------ fp16 storage (flat_fp16.cu)
// The launches of the fp16-row kernels, for the host code of flat.cu; each returns PR_OK or PR_ECUDA.  The launchers
// take (metric, grid, ..., arguments, stream) as those of flat.cu and flat_range.cu do, and the metric picks the kernel.
// Aux of one index: ||x||^2, ||x|| (f64 sums of the decoded row, rounded once to f32) and ||x_sub|| rounded up.
int flat_fp16_prep_rows(const __half *codes, int64_t n, int d, float *norm2, float *norm, float *nsub, cudaStream_t st);
// Per call: rows [n, n_out) of q_h, qn2, qn, qscale of the zero-padded batch; q_h = fp16(q 2^e_q), qscale = 2^-e_q.
int flat_fp16_prep_queries(const float *queries, int64_t n, int64_t n_out, int d, __half *q_h, float *qn2, float *qn,
                           float *qscale, cudaStream_t st);
int flat_fp16_filter_launch(int metric, unsigned grid, size_t smem, const CUtensorMap &map_x, const CUtensorMap &map_q,
                            const FilterArgs &fa, const FilterF16Args &fh, cudaStream_t st);
int flat_fp16_refine_launch(int metric, int n_queries, const RefineArgs &ra, cudaStream_t st);
int flat_fp16_range_refine_launch(int metric, int n_queries, const FlatRangeArgs &ra, cudaStream_t st);
