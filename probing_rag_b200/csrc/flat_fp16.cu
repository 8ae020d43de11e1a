// Exact flat search over fp16 rows (faiss IndexScalarQuantizer(d, QT_fp16) drop-in, pr_flat_create_fp16): the kernels
// of an fp16 handle.  flat.cu's host code runs the same launch plan and calls the launches below.
//
//   prep     flat_fp16_prep_kernel         once per index: ||x||^2, ||x|| of the decoded row (f64 sum, one f32
//                                          rounding) and ||x_sub||, the norm of its fp16-subnormal elements, rounded up
//            flat_fp16_query_prep_kernel   per call: fp16 copy of q 2^e_q (max |q_j| 2^e_q in [2^14, 2^15), so that the
//                                          rounding is relative 2^-11 almost everywhere), 2^-e_q, ||q||^2 and ||q||
//   filter   flat_fp16_filter_kernel / flat_fp16_ip_filter_kernel: the GEMM of flat_filter.cuh on the fp16 codes
//            themselves (no bf16 or f32 copy); the epilogue unscales the accumulator and adds the fp16 margin
//   refine   flat_fp16_refine_kernel / flat_fp16_ip_refine_kernel and the range refines: the refines of flat.cu and
//            flat_range.cu reading __half rows, widened exactly, so every value equals the f32 index's over the
//            decoded rows bit for bit
//
// The kernels live in this translation unit, apart from flat.cu and flat_range.cu, so that the f32 kernels there are
// compiled in the same modules as before, to the same SASS.
#include <cuda_fp16.h>

#include "common.cuh"
#include "flat_exact.cuh"
#include "flat_filter.cuh"
#include "tcgen05.cuh"

namespace {

constexpr float kF16MinNormal = 6.103515625e-05f;   // 2^-14: below it an fp16 value is subnormal

// One warp per row, the order of flat_prep_kernel: lane l sums x_j^2 for j = 2l, 2l + 1, 2l + 64, ... in f64.
__global__ void flat_fp16_prep_kernel(const __half *__restrict__ x, int64_t n, int d, float *__restrict__ norm2,
                                      float *__restrict__ norm, float *__restrict__ nsub)
{
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    double s = 0.0, sub = 0.0;
    for (int j = 2 * lane; j < d; j += 64) {
        const float2 v = __half22float2(*reinterpret_cast<const __half2 *>(x + row * d + j));
        s = fma((double)v.x, (double)v.x, s);
        s = fma((double)v.y, (double)v.y, s);
        if (fabsf(v.x) < kF16MinNormal) sub = fma((double)v.x, (double)v.x, sub);
        if (fabsf(v.y) < kF16MinNormal) sub = fma((double)v.y, (double)v.y, sub);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        s += __shfl_xor_sync(PR_FULL_MASK, s, o);
        sub += __shfl_xor_sync(PR_FULL_MASK, sub, o);
    }
    if (lane == 0) {
        norm2[row] = (float)s;
        norm[row] = (float)sqrt(s);
        // the squares of fp16 subnormals (>= 2^-48) and their sum are exact in f64 up to (d - 1) 2^-53 relative; one
        // ulp of the f64 sum before the upward rounding keeps the stored value above the true norm
        nsub[row] = __double2float_ru(sqrt(sub * (1.0 + 0x1p-40)));
    }
}

// One warp per query row of the padded batch.  Rows in [n, n_out) are zeros with scale 1.
__global__ void flat_fp16_query_prep_kernel(const float *__restrict__ q, int64_t n, int64_t n_out, int d,
                                            __half *__restrict__ qh, float *__restrict__ norm2, float *__restrict__ norm,
                                            float *__restrict__ qscale)
{
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_out) return;
    double s = 0.0;
    float amax = 0.f;
    bool finite = true;
    for (int j = 2 * lane; j < d; j += 64) {
        float2 v = make_float2(0.f, 0.f);
        if (row < n) v = *reinterpret_cast<const float2 *>(q + row * d + j);
        s = fma((double)v.x, (double)v.x, s);
        s = fma((double)v.y, (double)v.y, s);
        finite = finite && isfinite(v.x) && isfinite(v.y);
        amax = fmaxf(amax, fmaxf(fabsf(v.x), fabsf(v.y)));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        s += __shfl_xor_sync(PR_FULL_MASK, s, o);
        amax = fmaxf(amax, __shfl_xor_sync(PR_FULL_MASK, amax, o));
    }
    finite = __all_sync(PR_FULL_MASK, finite);
    // max |q_j| in [2^(ex-1), 2^ex) -> e = 15 - ex puts it in [2^14, 2^15).  e <= 126 keeps 2^-e a normal f32 (a query
    // whose largest element is below 2^-112 keeps a smaller scale; the margin's c3 term covers its absolute error);
    // e >= -113 holds for every finite query.  All-zero and non-finite queries keep e = 0.
    int e = 0;
    if (finite && amax > 0.f) {
        int ex;
        frexpf(amax, &ex);
        e = min(15 - ex, 126);
    }
    for (int j = 2 * lane; j < d; j += 64) {
        float2 v = make_float2(0.f, 0.f);
        if (row < n) v = *reinterpret_cast<const float2 *>(q + row * d + j);
        *reinterpret_cast<__half2 *>(qh + row * d + j) = __floats2half2_rn(ldexpf(v.x, e), ldexpf(v.y, e));
    }
    if (lane == 0) {
        norm2[row] = (float)s;
        norm[row] = (float)sqrt(s);
        qscale[row] = ldexpf(1.f, -e);
    }
}

__global__ void __launch_bounds__(kFilterThreads, 1)
flat_fp16_filter_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                        const FilterArgs g, const FilterF16Args h)
{
    flat_filter<PR_METRIC_L2, true>(map_x, map_q, g, h);
}

__global__ void __launch_bounds__(kFilterThreads, 1)
flat_fp16_ip_filter_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_q,
                           const FilterArgs g, const FilterF16Args h)
{
    flat_filter<PR_METRIC_INNER_PRODUCT, true>(map_x, map_q, g, h);
}

__global__ void __launch_bounds__(kRefineThreads) flat_fp16_refine_kernel(const RefineArgs g)
{
    flat_refine<PR_METRIC_L2, __half>(g);
}

__global__ void __launch_bounds__(kRefineThreads) flat_fp16_ip_refine_kernel(const RefineArgs g)
{
    flat_refine<PR_METRIC_INNER_PRODUCT, __half>(g);
}

__global__ void __launch_bounds__(kRangeThreads) flat_fp16_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_L2, __half>(g);
}

__global__ void __launch_bounds__(kRangeThreads) flat_fp16_ip_range_refine_kernel(const FlatRangeArgs g)
{
    flat_range_refine<PR_METRIC_INNER_PRODUCT, __half>(g);
}

}  // namespace

int flat_fp16_prep_rows(const __half *codes, int64_t n, int d, float *norm2, float *norm, float *nsub, cudaStream_t st)
{
    flat_fp16_prep_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(codes, n, d, norm2, norm, nsub);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

int flat_fp16_prep_queries(const float *queries, int64_t n, int64_t n_out, int d, __half *q_h, float *qn2, float *qn,
                           float *qscale, cudaStream_t st)
{
    flat_fp16_query_prep_kernel<<<(unsigned)((n_out + 7) / 8), 256, 0, st>>>(queries, n, n_out, d, q_h, qn2, qn, qscale);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

int flat_fp16_filter_launch(int metric, unsigned grid, size_t smem, const CUtensorMap &map_x, const CUtensorMap &map_q,
                            const FilterArgs &fa, const FilterF16Args &fh, cudaStream_t st)
{
    const bool ip = metric == PR_METRIC_INNER_PRODUCT;
    const void *filter = ip ? (const void *)flat_fp16_ip_filter_kernel : (const void *)flat_fp16_filter_kernel;
    // per device, as in flat.cu: set on every launch
    PR_CUDA_CHECK(cudaFuncSetAttribute(filter, cudaFuncAttributeMaxDynamicSharedMemorySize, kFilterSmemMax));
    if (ip)
        flat_fp16_ip_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa, fh);
    else
        flat_fp16_filter_kernel<<<grid, kFilterThreads, smem, st>>>(map_x, map_q, fa, fh);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

int flat_fp16_refine_launch(int metric, int n_queries, const RefineArgs &ra, cudaStream_t st)
{
    if (metric == PR_METRIC_INNER_PRODUCT)
        flat_fp16_ip_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
    else
        flat_fp16_refine_kernel<<<n_queries, kRefineThreads, 0, st>>>(ra);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}

int flat_fp16_range_refine_launch(int metric, int n_queries, const FlatRangeArgs &ra, cudaStream_t st)
{
    if (metric == PR_METRIC_INNER_PRODUCT)
        flat_fp16_ip_range_refine_kernel<<<n_queries, kRangeThreads, 0, st>>>(ra);
    else
        flat_fp16_range_refine_kernel<<<n_queries, kRangeThreads, 0, st>>>(ra);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}
