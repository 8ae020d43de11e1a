// The range refine of pr_flat_range_search (flat.cu runs the filter and the chunk loop).
//
// The filter runs unchanged with theta[q] = radius for the whole call: a result has D < radius (IP: S > radius) and the
// filter's bound L <= D (U >= S), so it passes !(L > theta) (!(U < theta)).  Then, per chunk in ascending row order,
// one CTA per query sorts the chunk's candidates by row id, evaluates them exactly and appends the hits in row order to
// the query's segment [lims[q], lims[q + 1]); hits[q] counts every hit, including those past the segment's end, which
// are not written.  A (query, chunk) with more candidates than `cap` scans the whole chunk in row order instead.
// Only this CTA writes query q's segment in this chunk, and the chunks run in sequence, so no global sort is needed.
#include "flat_exact.cuh"

namespace {

constexpr int kRangeThreads = 256;

template <int M>
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
                v = exact_dist(s_q, g.rows + row * g.d, g.d, lane);
                hit = v < g.radius;                                 // (NaN is never a hit)
            } else {
                v = exact_ip(s_q, g.rows + row * g.d, g.d, lane);
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

__global__ void __launch_bounds__(kRangeThreads) flat_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_L2>(g);
}

__global__ void __launch_bounds__(kRangeThreads) flat_ip_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_INNER_PRODUCT>(g);
}

}  // namespace

int flat_range_refine_launch(const FlatRangeArgs &g, int metric, int n_queries, cudaStream_t stream)
{
    if (metric == PR_METRIC_INNER_PRODUCT)
        flat_ip_range_refine_kernel<<<n_queries, kRangeThreads, 0, stream>>>(g);
    else
        flat_range_refine_kernel<<<n_queries, kRangeThreads, 0, stream>>>(g);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}
