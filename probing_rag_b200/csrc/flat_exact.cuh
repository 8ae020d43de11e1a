// The exact evaluation shared by the flat search's refine (flat.cu, flat_fp16.cu) and the flat range search
// (flat_range.cu, flat_fp16.cu), the range refine itself and its launch interface.  The range refine's f32 kernels live
// in a translation unit of their own, and the fp16 kernels in another, so that the filter kernels of flat.cu are
// compiled in the same module as before, to the same SASS.
#pragma once

#include <cuda_fp16.h>
#include <stdint.h>
#include <type_traits>

#include "common.cuh"

namespace {

// A row element widened exactly: f32 as it is, IEEE binary16 (fp16 storage) through f32, which holds every fp16 value.
__device__ __forceinline__ float row_value(float v) { return v; }
__device__ __forceinline__ float row_value(__half v) { return __half2float(v); }

// The exact distance (DESIGN §3): lane l sums (q_j - x_j)^2 over j = l, l+32, ... in increasing j, every difference,
// square and add a separately rounded f64 operation (no contraction), then an xor butterfly over the 32 lanes
// (offsets 16, 8, 4, 2, 1), rounded once to f32.  Every lane ends with the same value.
template <typename T>
__device__ __forceinline__ float exact_dist(const float *__restrict__ sq, const T *__restrict__ x, int d, int lane)
{
    double s = 0.0;
    for (int j = lane; j < d; j += 32) {
        const double df = __dsub_rn((double)sq[j], (double)row_value(__ldg(x + j)));
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
template <typename T>
__device__ __forceinline__ float exact_ip(const float *__restrict__ sq, const T *__restrict__ x, int d, int lane)
{
    double s = 0.0;
    for (int j = lane; j < d; j += 32) s = __dadd_rn(s, __dmul_rn((double)sq[j], (double)row_value(__ldg(x + j))));
#pragma unroll
    for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(PR_FULL_MASK, s, o));
    return __fadd_rn(__double2float_rn(s), 0.f);
}

// ascending bitonic sort of keys[0, n), n a power of two, by the whole block
template <typename T>
__device__ void block_bitonic_sort(T *keys, int n)
{
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const T a = keys[lo], b = keys[hi];
                if ((a > b) == asc) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
        }
    }
    __syncthreads();
}

// The rows of a refine's argument struct: f32 `rows`, or fp16 `rows_h` (appended to the struct, so that the f32 kernels'
// parameter offsets stay as they were).
template <typename T, typename A>
__device__ __forceinline__ const T *rows_of(const A &g)
{
    if constexpr (std::is_same<T, __half>::value)
        return g.rows_h;
    else
        return g.rows;
}

}  // namespace

constexpr int kFlatRangeMaxCap = 8192;   // candidates of one (query, chunk) the range refine sorts in shared memory

// One chunk of pr_flat_range_search after its filter launch (flat_range.cu).
struct FlatRangeArgs {
    const float *rows, *queries;
    int d, cap;
    float radius;
    int64_t row_begin, row_end;
    int32_t *count;                 // the filter's candidates per query in this chunk (reset to 0 here)
    const int32_t *cand;
    const int64_t *lims;            // [B + 1] segment bounds
    int64_t *hits;                  // [B] hits in the chunks so far
    float *dist;
    int64_t *ids;
    unsigned long long *stats;      // candidates, max candidates, fallback queries
    const __half *rows_h;           // fp16 storage: the rows (then `rows` is unused)
};

// Enqueues the range refine of one chunk for n_queries queries on `stream`; PR_OK or PR_ECUDA.
int flat_range_refine_launch(int metric, int n_queries, const FlatRangeArgs &g, cudaStream_t stream);

namespace {

constexpr int kRangeThreads = 256;

// The range refine of one chunk (flat_range.cu states the algorithm); T is the rows' storage type.
template <int M, typename T>
__device__ __forceinline__ void flat_range_refine(const FlatRangeArgs &g)
{
    __shared__ uint32_t s_rows[kFlatRangeMaxCap];
    __shared__ float s_q[PR_FLAT_MAX_D];
    __shared__ uint32_t s_mask[kRangeThreads / 32];
    const int q = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_warps = blockDim.x >> 5;
    const int cnt = g.count[q];
    const bool overflow = cnt > g.cap;
    const int64_t n_items = overflow ? g.row_end - g.row_begin : cnt;
    for (int j = threadIdx.x; j < g.d; j += blockDim.x) s_q[j] = g.queries[(size_t)q * g.d + j];
    if (threadIdx.x == 0) {
        if (cnt) {
            atomicAdd(g.stats + 0, (unsigned long long)cnt);
            atomicMax(g.stats + 1, (unsigned long long)cnt);
        }
        if (overflow) atomicAdd(g.stats + 2, 1ull);
    }
    if (!overflow) {
        int p = 1;
        while (p < cnt) p <<= 1;
        for (int i = threadIdx.x; i < p; i += blockDim.x)
            s_rows[i] = i < cnt ? (uint32_t)g.cand[(size_t)q * g.cap + i] : 0xFFFFFFFFu;
        block_bitonic_sort(s_rows, p);
    }
    __syncthreads();
    const int64_t seg = g.lims[q], room = g.lims[q + 1] - seg;
    int64_t hits = g.hits[q];
    // rounds of 32 items per warp; warp w takes items [base + 32 w, base + 32 w + 32) and lane j keeps item j's value,
    // so the hit masks of the warps, in warp order, give every hit its place in row order
    for (int64_t base = 0; base < n_items; base += 32 * n_warps) {
        const int64_t first = base + 32 * warp;
        uint32_t mask = 0;
        float mine = 0.f;
        int64_t my_row = 0;
        for (int j = 0; j < 32 && first + j < n_items; ++j) {      // (warp-uniform)
            const int64_t row = overflow ? g.row_begin + first + j : (int64_t)s_rows[first + j];
            float v;
            bool hit;
            if constexpr (M == PR_METRIC_L2) {
                v = exact_dist(s_q, rows_of<T>(g) + row * g.d, g.d, lane);
                hit = v < g.radius;                                 // (NaN is never a hit)
            } else {
                v = exact_ip(s_q, rows_of<T>(g) + row * g.d, g.d, lane);
                hit = v > g.radius;
            }
            mask |= (uint32_t)hit << j;
            if (lane == j) {
                mine = v;
                my_row = row;
            }
        }
        if (lane == 0) s_mask[warp] = mask;
        __syncthreads();
        int64_t pos = hits;
        int total = 0;
        for (int w = 0; w < n_warps; ++w) {
            const int c = __popc(s_mask[w]);
            if (w < warp) pos += c;
            total += c;
        }
        if ((mask >> lane) & 1u) {
            pos += __popc(mask & ((1u << lane) - 1u));
            if (pos < room) {
                g.dist[seg + pos] = mine;
                g.ids[seg + pos] = my_row;
            }
        }
        hits += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        g.hits[q] = hits;
        g.count[q] = 0;
    }
}

}  // namespace
