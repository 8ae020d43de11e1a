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

__global__ void __launch_bounds__(kRangeThreads) flat_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_L2, float>(g);
}

__global__ void __launch_bounds__(kRangeThreads) flat_ip_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_INNER_PRODUCT, float>(g);
}

}  // namespace

int flat_range_refine_launch(int metric, int n_queries, const FlatRangeArgs &g, cudaStream_t stream)
{
    if (metric == PR_METRIC_INNER_PRODUCT)
        flat_ip_range_refine_kernel<<<n_queries, kRangeThreads, 0, stream>>>(g);
    else
        flat_range_refine_kernel<<<n_queries, kRangeThreads, 0, stream>>>(g);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}
