// Prober gate on B200 tensor cores (sm_100a): tcgen05.mma + TMEM accumulators + TMA operands.
//
// Replaces, for a batch of queries, what /root/reference/exp_rag.py:381-415 does one query at
// a time with six torch-eager ImprovedProbe modules (/root/reference/utils.py:29-57):
//
//   x[B,P,2048] -> LN -> fc1(2048->512) -> SiLU -> LN -> fc2(512->512) -> SiLU -> LN -> fc3(512->2)
//   -> softmax -> sum over probers >= ablation -> retrieve unless P0 + theta < P1 -> compaction
//
// Numerics.  BASELINE asks for probabilities within 1e-3 of the fp32 reference.  One bf16
// GEMM misses that by 10x on generic weights (measured: 1e-2), so both GEMMs run as bf16x3:
// every fp32 operand is split into hi + lo bf16 halves and hi*hi + lo*hi + hi*lo is
// accumulated in fp32 in TMEM (three tcgen05.mma per k-step; error ~2e-5 on probabilities).
// LayerNorm statistics, SiLU, softmax and fc3 (512->2) stay in fp32 on the CUDA cores.
//
// Kernels
//   prober_gemm_kernel<EPI>  a CTA PAIR (cluster of 2, the two SMs of a TPC) = 256 rows x 512 columns of one prober;
//                            each CTA owns 128 rows and the whole 128x512 fp32 accumulator of them in its TMEM.
//        warp 0  TMA producer   per k-block of 64: this CTA's A(hi,lo)[128x64] and HALF of B: for each 256-column
//                               half of the output its 128 of the 256 weight rows (hi,lo) -- 96 KB per stage, 128B
//                               swizzle, loaded with the cta_group::2 form that signals the leader CTA's barrier
//        warp 1  MMA issuer     leader CTA only: tcgen05.mma.cta_group::2.kind::f16, M=256 N=256 K=16 -- every operand
//                               byte is read from shared memory once per PAIR.  (With one CTA per tile the kernel
//                               was bound by L2 -> SM operand traffic: bf16x3 doubles the operand bytes, and every
//                               128-row tile re-read all of B: 192 KB per k-block, tensor pipe 41% busy.)
//        warp 2  TMEM allocator (cta_group::2, 512 columns)
//        warps 4-11 epilogue    tcgen05.ld -> bias -> SiLU -> LN (3 passes over TMEM) ->
//                               EPI 1: (hi,lo) bf16 A2 to global; EPI 2: fc3 + softmax
//   prober_gate_kernel + compaction kernels
#include <cuda.h>
#include <cuda_bf16.h>


#include <cuda_fp16.h>

#include "common.cuh"
#include "tcgen05.cuh"   // PTX wrappers, umma_desc_sw128, make_map; kBK (64 K elements per stage)

namespace {

constexpr int kBM = 128;       // rows per CTA (a CTA pair covers 256)
constexpr int kBNH = 256;      // columns per MMA (half of the hidden size)
constexpr int kBNC = kBNH / 2; // weight rows of one MMA that each CTA of the pair holds
constexpr int kHidden = 512;
constexpr int kStages = 2;
constexpr int kTileBytes = kBM * kBK * 2;      // every operand tile is 128 rows x 64 k of bf16 = 16 KB
// stage: A_hi A_lo | B_hi(half 0) B_hi(half 1) | B_lo(half 0) B_lo(half 1)
constexpr int kStageBytes = 6 * kTileBytes;    // 96 KB
static_assert(kBNC == kBM, "operand tiles share one box shape");
#ifndef PR_EPI_SPLIT
#define PR_EPI_SPLIT 4
#endif
// Epilogue threads per row, each owning kHidden / kEpiSplit columns.  The epilogue (tcgen05.ld -> SFU -> tcgen05.st
// chains) and the A-operand producer of fc1 are latency-bound: 4 (16 warps, 96 registers) measured 0.77 ms per
// 16,384 x 6 against 0.80 ms with 2 (8 warps).
constexpr int kEpiSplit = PR_EPI_SPLIT;
constexpr int kEpiThreads = 128 * kEpiSplit;
constexpr int kGemmThreads = 128 + kEpiThreads;    // warps 0-2: TMA / MMA / TMEM alloc, warp 3 idle, then the epilogue
constexpr int kEpiCols = kHidden / kEpiSplit;
constexpr float kLnEps = 1e-5f;

// cute::UMMA::InstrDescriptor: fp32 accumulate, bf16 x bf16, both K-major, M=256 (the pair), N=256
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBNH >> 3) << 17) | ((uint32_t)((2 * kBM) >> 4) << 24);

// SiLU with the SFU exponential and reciprocal (2 ulp each: ~1e-7 on the activations, against a 1e-3 bar on the
// probabilities); the accurate expf + IEEE division were a quarter of the epilogue's instructions
__device__ __forceinline__ float silu(float v) { return __fdividef(v, 1.f + __expf(-v)); }

__device__ __forceinline__ void split_bf16(float y, __nv_bfloat16 &hi, __nv_bfloat16 &lo)
{
    hi = __float2bfloat16_rn(y);
    lo = __float2bfloat16_rn(y - __bfloat162float(hi));
}

// ------------------------------------------------------------------- LN_in + split (kernel 0)
// one warp per (row, prober): 2048 floats = 16 float4 per lane, statistics in fp32 exactly as
// torch.nn.LayerNorm (biased variance, eps inside the sqrt)
// four consecutive features of the pooled hidden states, whatever dtype the LM produced them in
// (/root/reference/exp_rag.py:385-387 feeds the prober the LM's own dtype), widened to fp32
template <typename T>
__device__ __forceinline__ float4 load_x4(const T *x, int i);
template <>
__device__ __forceinline__ float4 load_x4<float>(const float *x, int i) { return reinterpret_cast<const float4 *>(x)[i]; }
template <>
__device__ __forceinline__ float4 load_x4<__nv_bfloat16>(const __nv_bfloat16 *x, int i)
{
    const uint2 u = reinterpret_cast<const uint2 *>(x)[i];
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
}
template <>
__device__ __forceinline__ float4 load_x4<__half>(const __half *x, int i)
{
    const uint2 u = reinterpret_cast<const uint2 *>(x)[i];
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

// ------------------------------------------------------------------ GEMM + fused epilogue
struct GemmArgs {
    int n_rows, rows_pad, K;
    // epilogue parameters, indexed [prober][...]
    const float *bias, *ln_w, *ln_b;  // [P][512]
    const float *w3, *b3;             // [P][2][512], [P][2]          (EPI 2)
    __nv_bfloat16 *out_hi, *out_lo;   // [P][rows_pad][512]           (EPI 1)
    float *logits;                    // [rows][P][2] or null         (EPI 2)
    float *probs;                     // [rows][P][2]                 (EPI 2)
    int n_probers;
    int p0;                           // first prober of this launch (blockIdx.y counts from it)
    // EPI 1: the A operand is produced in the kernel from the pooled hidden states (input LayerNorm fused)
    const void *X;                    // [rows][P][d_model] of the kernel's XT
    const float *w1_rowsum;           // [P][512] row sums of fc1.weight * layer_norm_input.weight
};

constexpr size_t kGemmSmemBytes =
    1024 /*align slack*/ + (size_t)kStages * kStageBytes + 5 * kHidden * 4 + 256 + 4 * kEpiThreads * 4 + 2 * kBM * 4;

// EPI 1 (fc1): the input LayerNorm is folded AROUND the GEMM and the A operand never exists in global memory.
//     fc1(LN(x)) = rstd * (W' x - mean * rowsum(W')) + (W beta + b1),   W' = W diag(gamma)
// so the tensor cores multiply the hidden states (raw but for a per-row shift) by W' (packed once per checkpoint, prober.py) and the epilogue
// applies rstd, the mean term and the shifted bias per row.  The 8 epilogue warps -- idle while the MMAs run -- stream
// X[128 rows, 64 features] k-block by k-block (each element of X is read from HBM exactly once, one k-block ahead of
// the MMAs), subtract a per-row shift s (the mean of the row's first k-block), split x - s into (hi, lo) bf16 straight
// into the stage in the 128-byte-swizzled K-major layout the tensor core reads, and accumulate every row's sum and sum
// of squares of x - s on the way: by
// the time the accumulator is complete so are mean and rstd.  This replaces a separate LayerNorm kernel that read X
// and wrote + re-read 2 x 403 MB of split operand (0.32 of 1.05 ms at 16,384 rows) and needs no statistics pre-pass.
// XT = dtype of X (f32 / bf16 / f16).   EPI 2 (fc2) loads A with TMA.
template <int EPI, typename XT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
prober_gemm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                   const GemmArgs g)
{
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char *stage_base = smem;                                       // kStages x 96 KB, 1024-aligned
    float *s_bias = reinterpret_cast<float *>(smem + (size_t)kStages * kStageBytes);
    float *s_lnw = s_bias + kHidden;
    float *s_lnb = s_lnw + kHidden;
    float *s_w3 = s_lnb + kHidden;                                          // [2][512]
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(s_w3 + 2 * kHidden);  // [kStages]
    uint64_t *empty_bar = full_bar + kStages;                               // [kStages]
    uint64_t *acc_bar = empty_bar + kStages;                                // accumulator complete
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_bar + 1);
    float *s_red = reinterpret_cast<float *>(reinterpret_cast<unsigned char *>(full_bar) + 256);  // [4][kEpiThreads] row partials
    float *s_mean = s_red + 4 * kEpiThreads;                                // [kBM] input LayerNorm mean - s, rstd (EPI 1)
    float *s_rstd = s_mean + kBM;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = g.p0 + blockIdx.y;          // prober
    const int row0 = blockIdx.x * kBM;        // first row of this CTA's tile (the pair: blockIdx.x even and odd)
    const uint32_t cta_rank = cluster_ctarank();
    const int n_iter = g.K / kBK;             // k-blocks

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) {
            // (used in the leader CTA only) its producer's arrive + both CTAs' TMA bytes; EPI 1: + one arrival per
            // CTA once its epilogue warps have written their A tiles
            mbar_init(&full_bar[s], EPI == 1 ? 3 : 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(acc_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    if (warp >= 4) {  // epilogue parameters of this prober
        const int t = threadIdx.x - 128;
        for (int i = t; i < kHidden; i += kEpiThreads) {
            s_bias[i] = g.bias[(size_t)p * kHidden + i];
            s_lnw[i] = g.ln_w[(size_t)p * kHidden + i];
            s_lnb[i] = g.ln_b[(size_t)p * kHidden + i];
            if (EPI == 2) {
                s_w3[i] = g.w3[((size_t)p * 2 + 0) * kHidden + i];
                s_w3[kHidden + i] = g.w3[((size_t)p * 2 + 1) * kHidden + i];
            } else {
                s_w3[i] = g.w1_rowsum[(size_t)p * kHidden + i];   // (EPI 1 has no fc3: the array holds rowsum(W'))
            }
        }
    }
    tc_fence_before();
    cluster_sync();   // both CTAs: barriers initialised, TMEM allocated (the peer's TMA completions and the leader's
    tc_fence_after(); // MMAs touch the other CTA's barriers / TMEM)
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer (both CTAs): this CTA's A rows and its half of the weight rows of either column half.
        // Completion bytes of BOTH CTAs are counted by the leader's full barrier, which only the leader arms.
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % kStages;
            const uint32_t ph = (uint32_t)(it / kStages) & 1u;
            mbar_wait(&empty_bar[s], ph ^ 1u);
            unsigned char *st = stage_base + (size_t)s * kStageBytes;
            if (cta_rank == 0) mbar_expect_tx(&full_bar[s], 2 * (EPI == 1 ? 4 : 6) * kTileBytes);
            const int a_row = p * g.rows_pad + row0, b_row = p * kHidden + (int)cta_rank * kBNC;
            if (EPI == 2) {
                tma_load_2d_pair(st, &map_a_hi, &full_bar[s], it * kBK, a_row);
                tma_load_2d_pair(st + kTileBytes, &map_a_lo, &full_bar[s], it * kBK, a_row);
            }
            tma_load_2d_pair(st + 2 * kTileBytes, &map_b_hi, &full_bar[s], it * kBK, b_row);
            tma_load_2d_pair(st + 3 * kTileBytes, &map_b_hi, &full_bar[s], it * kBK, b_row + kBNH);
            tma_load_2d_pair(st + 4 * kTileBytes, &map_b_lo, &full_bar[s], it * kBK, b_row);
            tma_load_2d_pair(st + 5 * kTileBytes, &map_b_lo, &full_bar[s], it * kBK, b_row + kBNH);
        }
    } else if (warp == 1 && lane == 0 && cta_rank == 0) {
        // ===== MMA issuer (leader CTA): acc[256 rows, nh*256 .. +256) += A_hi*B_hi + A_lo*B_hi + A_hi*B_lo
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % kStages;
            const uint32_t ph = (uint32_t)(it / kStages) & 1u;
            mbar_wait_cluster(&full_bar[s], ph);
            tc_fence_after();
            const uint32_t st = smem_u32(stage_base + (size_t)s * kStageBytes);
            const uint64_t a_hi = umma_desc_sw128(st), a_lo = umma_desc_sw128(st + kTileBytes);
#pragma unroll
            for (int nh = 0; nh < 2; ++nh) {
                const uint32_t d_tmem = tmem_base + (uint32_t)(nh * kBNH);
                const uint64_t b_hi = umma_desc_sw128(st + (2 + nh) * kTileBytes), b_lo = umma_desc_sw128(st + (4 + nh) * kTileBytes);
#pragma unroll
                for (int k = 0; k < kBK / 16; ++k) {
                    const uint64_t adv = (uint64_t)((k * 16 * 2) >> 4);  // 32 bytes per K=16 step, 16-byte units
                    umma_bf16(d_tmem, a_hi + adv, b_hi + adv, kIdesc, (it | k) ? 1u : 0u);
                    umma_bf16(d_tmem, a_lo + adv, b_hi + adv, kIdesc, 1u);
                    umma_bf16(d_tmem, a_hi + adv, b_lo + adv, kIdesc, 1u);
                }
            }
            umma_commit_pair(&empty_bar[s]);  // frees the stage in both CTAs once these MMAs have read it
        }
        umma_commit_pair(acc_bar);            // accumulators complete (both CTAs' epilogues wait on their own copy)
    } else if (warp >= 4) {
        // ===== epilogue: TMEM lane t = row row0+t is shared by kEpiSplit threads (warps w, w+4, w+8, .. see the same
        // lane quadrant): thread (part, t) owns columns [part * kEpiCols, +kEpiCols) and the row statistics are combined
        // through shared memory (every thread of a row sums the parts in the same order: identical values)
        const int et = threadIdx.x - 128;
        auto epi_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); };
        if (EPI == 1) {
            // ===== A-operand producer.  Lane l of warp w owns the 4 features [4 (l % 16), +4) of the k-block in the 8
            // rows w * 16 + 2 i + l / 16 (i = 0..7): every load instruction of a warp covers two whole 256-byte row
            // segments of X (coalesced), and the k-block after the current one is already in registers while the
            // barrier of the current stage is awaited.  (A first version -- one thread per half row, no look-ahead,
            // the row normalised here after a statistics pre-pass -- made fc1 1.8x slower than the unfused kernel.)  Tile layout (what TMA's SWIZZLE_128B writes): row r at byte
            // r * 128, its 16-byte chunk j stored at chunk position j ^ (r % 8).
            const int c4 = lane & 15, rsub = lane >> 4, rbase = (warp - 4) * (kBM / (kEpiThreads / 32));
            constexpr int kRowsPerThread = kBM / (kEpiThreads / 32) / 2;   // 8
            const XT *xrow[kRowsPerThread];
            uint32_t dst[kRowsPerThread];   // byte offset of this thread's 8 bytes inside an A tile
            float shift[kRowsPerThread], sum[kRowsPerThread], sq[kRowsPerThread];
            float4 cur[kRowsPerThread], nxt[kRowsPerThread];
#pragma unroll
            for (int i = 0; i < kRowsPerThread; ++i) {
                const int r = rbase + 2 * i + rsub;
                const bool live = row0 + r < g.n_rows;   // (padding rows read row 0: their results are never stored)
                xrow[i] = reinterpret_cast<const XT *>(g.X) + ((size_t)(live ? row0 + r : 0) * g.n_probers + p) * g.K;
                dst[i] = (uint32_t)(r * 128 + (((c4 >> 1) ^ (r & 7)) << 4) + ((c4 & 1) << 3));
                cur[i] = load_x4<XT>(xrow[i], c4);
                // Per-row shift s = mean of the row's first 64 features (the 16 lanes of the row hold them; the xor
                // butterfly leaves the same value in all 16).  The tensor cores multiply the split of x - s, not of x:
                //     W'x - mean * rowsum(W') = W'(x - s) - (mean - s) * rowsum(W')   for any s,
                // and the bf16 split error of x - s is relative to |x - s|, about sigma, where that of x is relative
                // to |x|: with a common offset c the error after scaling by rstd grew like |c| / sigma.  The row
                // statistics are accumulated around the same s (no E[x^2] - mean^2 cancellation either).
                float s4 = (cur[i].x + cur[i].y) + (cur[i].z + cur[i].w);
#pragma unroll
                for (int o = 8; o; o >>= 1) s4 += __shfl_xor_sync(PR_FULL_MASK, s4, o);
                shift[i] = s4 * (1.f / kBK);
                sum[i] = 0.f;
                sq[i] = 0.f;
            }
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % kStages;
                const uint32_t ph = (uint32_t)(it / kStages) & 1u;
                if (it + 1 < n_iter) {
                    const int qn = (it + 1) * (kBK / 4) + c4;   // this thread's 4-feature group in the next k-block
#pragma unroll
                    for (int i = 0; i < kRowsPerThread; ++i) nxt[i] = load_x4<XT>(xrow[i], qn);
                }
                mbar_wait(&empty_bar[s], ph ^ 1u);
                unsigned char *a_hi_t = stage_base + (size_t)s * kStageBytes, *a_lo_t = a_hi_t + kTileBytes;
#pragma unroll
                for (int i = 0; i < kRowsPerThread; ++i) {
                    const float x[4] = {cur[i].x, cur[i].y, cur[i].z, cur[i].w};
                    __nv_bfloat16 hh[4], ll[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float d = x[k] - shift[i];
                        split_bf16(d, hh[k], ll[k]);
                        sum[i] += d;
                        sq[i] = fmaf(d, d, sq[i]);
                    }
                    *reinterpret_cast<uint2 *>(a_hi_t + dst[i]) =
                        make_uint2((uint32_t)__bfloat16_as_ushort(hh[0]) | ((uint32_t)__bfloat16_as_ushort(hh[1]) << 16),
                                   (uint32_t)__bfloat16_as_ushort(hh[2]) | ((uint32_t)__bfloat16_as_ushort(hh[3]) << 16));
                    *reinterpret_cast<uint2 *>(a_lo_t + dst[i]) =
                        make_uint2((uint32_t)__bfloat16_as_ushort(ll[0]) | ((uint32_t)__bfloat16_as_ushort(ll[1]) << 16),
                                   (uint32_t)__bfloat16_as_ushort(ll[2]) | ((uint32_t)__bfloat16_as_ushort(ll[3]) << 16));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
                epi_sync();
                if (et == 0) mbar_arrive_leader(&full_bar[s]);
#pragma unroll
                for (int i = 0; i < kRowsPerThread; ++i) cur[i] = nxt[i];
            }
            // row statistics: the 16 lanes that share a row add up their parts
#pragma unroll
            for (int i = 0; i < kRowsPerThread; ++i) {
                float a = sum[i], b = sq[i];
#pragma unroll
                for (int o = 8; o; o >>= 1) {
                    a += __shfl_xor_sync(PR_FULL_MASK, a, o);
                    b += __shfl_xor_sync(PR_FULL_MASK, b, o);
                }
                if (c4 == 0) {
                    const float inv_k = 1.f / (float)g.K, m = a * inv_k;   // m = mean - s
                    s_mean[rbase + 2 * i + rsub] = m;
                    s_rstd[rbase + 2 * i + rsub] = rsqrtf(fmaxf(b * inv_k - m * m, 0.f) + kLnEps);   // biased variance
                }
            }
            epi_sync();
        }
        mbar_wait(acc_bar, 0);
        tc_fence_after();
        const int part = et >> 7, t = et & 127;
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        const int row = row0 + t;
        const int cb = part * kEpiCols, ce = cb + kEpiCols;
        uint32_t r[32];
        // pass 1: bias + SiLU, keep the activations in TMEM; row mean and centred second moment in the same pass:
        // exact two-pass statistics of every 32-column chunk while it sits in registers, chunks (and then the parts
        // of the row) merged with Chan's formula -- no second sweep over TMEM, no E[x^2] - mean^2 cancellation
        float run_mean = 0.f, run_m2 = 0.f;
        const float in_rstd = EPI == 1 ? s_rstd[t] : 1.f, in_mean_rstd = EPI == 1 ? s_mean[t] * s_rstd[t] : 0.f;
        for (int c0 = cb; c0 < ce; c0 += 32) {
            tmem_ld32(taddr + c0, r);
            float csum = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                // EPI 1: fc1(LN(x))_j = rstd * acc_j - ((mean - s) * rstd) * rowsum(W')_j + (W beta + b1)_j, acc = W'(x - s)
                const float pre = EPI == 1 ? fmaf(__uint_as_float(r[j]), in_rstd, fmaf(-in_mean_rstd, s_w3[c0 + j], s_bias[c0 + j]))
                                           : __uint_as_float(r[j]) + s_bias[c0 + j];
                const float a = silu(pre);
                csum += a;
                r[j] = __float_as_uint(a);
            }
            tmem_st32(taddr + c0, r);
            const float cmean = csum * (1.f / 32.f);
            float cm2 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float d = __uint_as_float(r[j]) - cmean;
                cm2 = fmaf(d, d, cm2);
            }
            const float n_a = (float)(c0 - cb), n_ab = n_a + 32.f, delta = cmean - run_mean;
            run_mean += delta * (32.f / n_ab);
            run_m2 += cm2 + delta * delta * (n_a * 32.f / n_ab);
        }
        s_red[et] = run_mean;
        s_red[kEpiThreads + et] = run_m2;
        epi_sync();
        // equal-sized parts: mean = average of the part means, M2 = sum M2_i + kEpiCols * sum (mean_i - mean)^2
        float mean = 0.f, m2 = 0.f;
#pragma unroll
        for (int i = 0; i < kEpiSplit; ++i) mean += s_red[i * 128 + t];
        mean *= 1.f / kEpiSplit;
#pragma unroll
        for (int i = 0; i < kEpiSplit; ++i) {
            const float d = s_red[i * 128 + t] - mean;
            m2 += s_red[kEpiThreads + i * 128 + t] + d * d * (float)kEpiCols;
        }
        const float rstd = rsqrtf(m2 * (1.f / kHidden) + kLnEps);   // torch.nn.LayerNorm: biased variance
        // pass 2: normalise; EPI 1 writes the split bf16 operand of fc2, EPI 2 applies fc3 + softmax
        float z0 = 0.f, z1 = 0.f;
        for (int c0 = cb; c0 < ce; c0 += 32) {
            tmem_ld32(taddr + c0, r);
            if (EPI == 1) {
                uint32_t hp[16], lp[16];  // bf16 pairs
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float y0 = (__uint_as_float(r[j]) - mean) * rstd * s_lnw[c0 + j] + s_lnb[c0 + j];
                    const float y1 = (__uint_as_float(r[j + 1]) - mean) * rstd * s_lnw[c0 + j + 1] + s_lnb[c0 + j + 1];
                    __nv_bfloat16 h0, l0, h1, l1;
                    split_bf16(y0, h0, l0);
                    split_bf16(y1, h1, l1);
                    hp[j >> 1] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                    lp[j >> 1] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
                }
                if (row < g.n_rows) {
                    const size_t o = ((size_t)p * g.rows_pad + row) * kHidden + c0;
                    uint4 *dh = reinterpret_cast<uint4 *>(g.out_hi + o), *dl = reinterpret_cast<uint4 *>(g.out_lo + o);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        dh[q] = make_uint4(hp[4 * q], hp[4 * q + 1], hp[4 * q + 2], hp[4 * q + 3]);
                        dl[q] = make_uint4(lp[4 * q], lp[4 * q + 1], lp[4 * q + 2], lp[4 * q + 3]);
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float y = (__uint_as_float(r[j]) - mean) * rstd * s_lnw[c0 + j] + s_lnb[c0 + j];
                    z0 = fmaf(y, s_w3[c0 + j], z0);
                    z1 = fmaf(y, s_w3[kHidden + c0 + j], z1);
                }
            }
        }
        if (EPI == 2) {
            s_red[2 * kEpiThreads + et] = z0;
            s_red[3 * kEpiThreads + et] = z1;
            epi_sync();
            if (part == 0 && row < g.n_rows) {
                z0 = z1 = 0.f;
#pragma unroll
                for (int i = 0; i < kEpiSplit; ++i) {
                    z0 += s_red[2 * kEpiThreads + i * 128 + t];
                    z1 += s_red[3 * kEpiThreads + i * 128 + t];
                }
                z0 += g.b3[p * 2 + 0];
                z1 += g.b3[p * 2 + 1];
                const size_t o = ((size_t)row * g.n_probers + p) * 2;
                if (g.logits) {
                    g.logits[o] = z0;
                    g.logits[o + 1] = z1;
                }
                const float m = fmaxf(z0, z1);
                const float e0 = expf(z0 - m), e1 = expf(z1 - m);
                const float inv = 1.f / (e0 + e1);
                g.probs[o] = e0 * inv;
                g.probs[o + 1] = e1 * inv;
            }
        }
        tc_fence_before();
    }
    cluster_sync();   // neither CTA may free TMEM (or exit) while the pair's MMAs or loads can still touch it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------ gate + compaction
// P = sum_{l >= ablation} softmax(logits_l), in prober order; retrieve unless P0 + theta < P1
// (/root/reference/exp_rag.py:407-415)
__global__ void prober_gate_kernel(const float *__restrict__ probs, int n_rows, int n_probers, double theta, int ablation,
                                   float *__restrict__ probsum, uint8_t *__restrict__ mask, int32_t *__restrict__ block_cnt)
{
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    int ret = 0;
    if (row < n_rows) {
        float p0 = 0.f, p1 = 0.f;
        for (int l = ablation; l < n_probers; ++l) {
            p0 += probs[((size_t)row * n_probers + l) * 2];
            p1 += probs[((size_t)row * n_probers + l) * 2 + 1];
        }
        probsum[(size_t)row * 2] = p0;
        probsum[(size_t)row * 2 + 1] = p1;
        // the reference compares Python floats: `P0.item() + threshold < P1.item()` (exp_rag.py:414) -- the f32 sums
        // widened to double, the threshold a double (0.1 is not an f32)
        ret = !((double)p0 + theta < (double)p1);
        mask[row] = (uint8_t)ret;
    }
    const int c = __syncthreads_count(ret);
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = c;
}

// Ordered compaction of the rows that retrieve.  Every block adds up the counts of the blocks before it itself (a few
// dozen values: no scan kernel), block 0 publishes the total, and the thread of row i also writes the -1 that fills
// slot i when i lies past the total (no memset in front).
__global__ void prober_compact_kernel(const uint8_t *__restrict__ mask, int n_rows, const int32_t *__restrict__ block_cnt,
                                      int32_t *__restrict__ compact, int32_t *__restrict__ n_retrieve)
{
    __shared__ int warp_cnt[32];
    __shared__ int s_before, s_total;
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int flag = row < n_rows && mask[row];
    const unsigned m = __ballot_sync(PR_FULL_MASK, flag);
    if (lane == 0) warp_cnt[w] = __popc(m);
    if (w == 0) {
        int before = 0, total = 0;
        for (int i = lane; i < (int)gridDim.x; i += 32) {
            const int c = block_cnt[i];
            total += c;
            if (i < (int)blockIdx.x) before += c;
        }
        for (int o = 16; o; o >>= 1) {
            before += __shfl_xor_sync(PR_FULL_MASK, before, o);
            total += __shfl_xor_sync(PR_FULL_MASK, total, o);
        }
        if (lane == 0) {
            s_before = before;
            s_total = total;
            if (blockIdx.x == 0) *n_retrieve = total;
        }
    }
    __syncthreads();
    int before = s_before;
    for (int i = 0; i < w; ++i) before += warp_cnt[i];
    if (flag) compact[before + __popc(m & ((1u << lane) - 1u))] = row;
    if (row < n_rows && row >= s_total) compact[row] = -1;
}

// ------------------------------------------------------------------------------------ host

inline size_t up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct ProberLayout {
    int rows_pad;
    size_t a2_hi, a2_lo, probs, block_cnt, total;
};

ProberLayout prober_layout(int P, int n_rows, int d_model, int hidden)
{
    ProberLayout l;
    l.rows_pad = (n_rows + 2 * kBM - 1) / (2 * kBM) * (2 * kBM);   // whole CTA pairs
    size_t o = 0;
    l.a2_hi = o; o = up(o + (size_t)P * l.rows_pad * hidden * 2, 1024);
    l.a2_lo = o; o = up(o + (size_t)P * l.rows_pad * hidden * 2, 1024);
    l.probs = o; o = up(o + (size_t)n_rows * P * 2 * 4, 256);
    l.block_cnt = o; o = up(o + ((size_t)n_rows / 256 + 2) * 4, 256);
    l.total = o;
    return l;
}

}  // namespace

extern "C" size_t pr_prober_workspace_bytes(int32_t n_probers, int32_t n_rows, int32_t d_model, int32_t hidden)
{
    if (n_probers < 1 || n_rows < 0 || d_model < 1 || hidden < 1) return 0;
    return prober_layout(n_probers, n_rows, d_model, hidden).total;
}

extern "C" int pr_prober_forward(const pr_prober_set_t *ps, int32_t n_rows, const void *X_dev, int32_t x_dtype, double theta,
                                 int32_t ablation, float *out_logits_dev, float *out_probsum_dev,
                                 uint8_t *out_retrieve_mask_dev, int32_t *out_compact_idx_dev,
                                 int32_t *out_n_retrieve_dev, void *workspace_dev, size_t workspace_bytes,
                                 pr_stream_t stream)
{
    if (!ps || n_rows < 0 || !X_dev || !out_probsum_dev || !out_retrieve_mask_dev || !out_compact_idx_dev ||
        !out_n_retrieve_dev || !workspace_dev) {
        pr_set_error("pr_prober_forward: null argument");
        return PR_EINVAL;
    }
    const int P = ps->n_probers;
    if (P < 1 || P > PR_PROBER_MAX || ps->hidden != kHidden || ps->d_model < 128 || ps->d_model > 2048 ||
        ps->d_model % 128 != 0) {
        pr_set_error("pr_prober_forward: unsupported shape (n_probers=%d d_model=%d hidden=%d; hidden must be 512, "
                     "d_model a multiple of 128 up to 2048)", P, ps->d_model, ps->hidden);
        return PR_EUNSUPPORTED;
    }
    if (x_dtype < 0 || x_dtype > 2) {
        pr_set_error("pr_prober_forward: x_dtype must be 0 (f32), 1 (bf16) or 2 (f16), got %d", x_dtype);
        return PR_EINVAL;
    }
    if ((uintptr_t)X_dev & 15) {
        pr_set_error("pr_prober_forward: X_dev must be 16-byte aligned");
        return PR_EINVAL;
    }
    if (ablation < 0 || ablation > P) {
        pr_set_error("pr_prober_forward: ablation %d outside [0, %d]", ablation, P);
        return PR_EINVAL;
    }
    const ProberLayout l = prober_layout(P, n_rows, ps->d_model, ps->hidden);
    if (workspace_bytes < l.total) {
        pr_set_error("pr_prober_forward: workspace of %zu bytes, need %zu", workspace_bytes, l.total);
        return PR_EWORKSPACE;
    }
    if (((uintptr_t)workspace_dev & 1023) || ((uintptr_t)ps->w1_hi & 127) || ((uintptr_t)ps->w1_lo & 127) ||
        ((uintptr_t)ps->w2_hi & 127) || ((uintptr_t)ps->w2_lo & 127)) {
        pr_set_error("pr_prober_forward: workspace must be 1024-byte aligned, weight matrices 128-byte aligned");
        return PR_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows == 0) {
        PR_CUDA_CHECK(cudaMemsetAsync(out_n_retrieve_dev, 0, 4, st));
        return PR_OK;
    }
    unsigned char *ws = (unsigned char *)workspace_dev;
    __nv_bfloat16 *a2_hi = (__nv_bfloat16 *)(ws + l.a2_hi), *a2_lo = (__nv_bfloat16 *)(ws + l.a2_lo);
    float *probs = (float *)(ws + l.probs);
    int32_t *block_cnt = (int32_t *)(ws + l.block_cnt);

    CUtensorMap m_w1h, m_w1l, m_a2h, m_a2l, m_w2h, m_w2l;
    int rc;
    if ((rc = make_map(&m_w1h, ps->w1_hi, (uint64_t)P * kHidden, ps->d_model, kBNC)) != PR_OK) return rc;
    if ((rc = make_map(&m_w1l, ps->w1_lo, (uint64_t)P * kHidden, ps->d_model, kBNC)) != PR_OK) return rc;
    if ((rc = make_map(&m_a2h, a2_hi, (uint64_t)P * l.rows_pad, kHidden, kBM)) != PR_OK) return rc;
    if ((rc = make_map(&m_a2l, a2_lo, (uint64_t)P * l.rows_pad, kHidden, kBM)) != PR_OK) return rc;
    if ((rc = make_map(&m_w2h, ps->w2_hi, (uint64_t)P * kHidden, kHidden, kBNC)) != PR_OK) return rc;
    if ((rc = make_map(&m_w2l, ps->w2_lo, (uint64_t)P * kHidden, kHidden, kBNC)) != PR_OK) return rc;

    typedef void (*gemm_fn_t)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const GemmArgs);
    const gemm_fn_t fc1 = x_dtype == 0 ? prober_gemm_kernel<1, float>
                          : x_dtype == 1 ? prober_gemm_kernel<1, __nv_bfloat16> : prober_gemm_kernel<1, __half>;
    const gemm_fn_t fc2 = prober_gemm_kernel<2, float>;
    // A function attribute holds for the current device only: set it on every call (host-only and cheap), so that a
    // gate on a second GPU of the process launches as the first one did.
    PR_CUDA_CHECK(cudaFuncSetAttribute((const void *)fc1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmemBytes));
    PR_CUDA_CHECK(cudaFuncSetAttribute((const void *)fc2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmemBytes));
    GemmArgs g;
    g.n_rows = n_rows;
    g.rows_pad = l.rows_pad;
    g.n_probers = P;
    g.p0 = 0;
    g.w3 = ps->w3;
    g.b3 = ps->b3;
    g.out_hi = a2_hi;
    g.out_lo = a2_lo;
    g.logits = out_logits_dev;
    g.probs = probs;
    g.X = X_dev;
    g.w1_rowsum = ps->w1_rowsum;
    const dim3 grid((unsigned)(l.rows_pad / kBM), (unsigned)P);
    // kernel 1: input LayerNorm (folded around the GEMM) + fc1 + SiLU + LN1 -> split operand of fc2
    g.K = ps->d_model;
    g.bias = ps->b1;
    g.ln_w = ps->ln1_w;
    g.ln_b = ps->ln1_b;
    fc1<<<grid, kGemmThreads, kGemmSmemBytes, st>>>(m_w1h, m_w1l, m_w1h, m_w1l, g);   // (the A maps are unused by EPI 1)
    PR_CUDA_CHECK(cudaGetLastError());
    // kernel 2: fc2 + SiLU + LN2 + fc3 + softmax
    g.K = kHidden;
    g.bias = ps->b2;
    g.ln_w = ps->ln2_w;
    g.ln_b = ps->ln2_b;
    fc2<<<grid, kGemmThreads, kGemmSmemBytes, st>>>(m_a2h, m_a2l, m_w2h, m_w2l, g);
    PR_CUDA_CHECK(cudaGetLastError());
    // gate + ordered compaction of the rows that retrieve
    const int nb = (n_rows + 255) / 256;
    prober_gate_kernel<<<nb, 256, 0, st>>>(probs, n_rows, P, theta, ablation, out_probsum_dev, out_retrieve_mask_dev, block_cnt);
    prober_compact_kernel<<<nb, 256, 0, st>>>(out_retrieve_mask_dev, n_rows, block_cnt, out_compact_idx_dev, out_n_retrieve_dev);
    PR_CUDA_CHECK(cudaGetLastError());
    return PR_OK;
}
