// The exact evaluation shared by the flat search's refine (flat.cu) and the flat range search (flat_range.cu), and the
// range refine's launch interface.  The range refine lives in a translation unit of its own so that the filter kernels
// of flat.cu are compiled in the same module as before, to the same SASS.
#pragma once

#include <stdint.h>

#include "common.cuh"

namespace {

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
};

// Enqueues the range refine of one chunk for n_queries queries on `stream`; PR_OK or PR_ECUDA.
int flat_range_refine_launch(const FlatRangeArgs &g, int metric, int n_queries, cudaStream_t stream);
