// Device helpers of the tensor-core screened K-means assignment kernel (kmeans_tc.cu): TF32
// rounding, the TMA bulk copy of a row tile, the screening bound and the float32 / float64
// refinement of the candidates (stages B and C, see kmeans_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kmeans_common.cuh"

namespace gsl {

constexpr int kTcPairs = 32;             // (row, candidate) pairs a warp refines cooperatively per tile;
                                         // 32 * (4 + 2) B fit in the warp's 32 candidate-mask slots, which they reuse

__device__ __forceinline__ uint32_t to_tf32(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

// ---- TMA 1-D bulk copy of a whole tile (global -> shared), completion on an mbarrier ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// One thread: order prior generic-proxy accesses to the buffer before the async-proxy write,
// arm the barrier with the byte count and launch the copy.
__device__ __forceinline__ void bulk_load_tile(void *dst, const void *src, unsigned bytes, void *bar)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_wait(void *bar, unsigned parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// E_k = 1.5 * 2^-9 |x'| |c'_k| + 2^-22 (|x'| + |c'_k|)^2, evaluated as an upper bound with
// (a + b)^2 <= 2 a^2 + 2 b^2:   E_k <= |x'| * ea_k + eb_k + 2^-21 |x'|^2,
// ea_k = 1.5 * 2^-9 |c'_k| and eb_k = 2^-21 |c'_k|^2 tabulated per centroid.
__device__ __forceinline__ float screen_bound(float nx, float nx_term, float ea, float eb)
{
    return fmaf(nx, ea, eb) + nx_term;
}

// The row-wide bound B = screen_bound(nx, ., ea_max, eb_max) holds only where stage A's float32
// arithmetic neither overflows nor underflows.  B >= 2^-21 (|x'|^2 + max|c'_k|^2) and
// B >= 1.5 * 2^-9 |x'| max|c'_k|, so:
//   B < 2^104   ->  |x'|^2, |c'_k|^2 < 2^125 and |x'| |c'_k| < 2^113: no product, dot product,
//                   |c'_k|^2 or g_k comes near FLT_MAX (~2^128), whatever the TF32 rounding;
//   B >= 2^-80  ->  max(|x'|, |c'_k|) >= 2^-29.5: subnormal products, operands flushed to zero by
//                   the tensor cores and the absolute rounding of subnormal partial sums add up to
//                   less than 2^-120 + 2^-123 max(|x'|, |c'_k|) < 2^-40 B.
// Rows outside that range (and NaN/Inf rows, whose B is not finite) take every centroid.
__device__ __forceinline__ bool screen_in_range(float bnd)
{
    return bnd >= 0x1p-80f && bnd < 0x1p104f;
}

// Stages B and C for one row: candidates given as a bit mask over k.  A float32 distance that
// overflowed (s = +inf) needs no special case: s1 (1 + eps) is finite only for s1 < FLT_MAX / (1 + eps),
// and eps exceeds the sum's real error, so such a candidate is really farther than the band; when
// s1 (1 + eps) overflows, the row is not decided in float32 and the band (bound = +inf) keeps every
// candidate.  Rows with s1 <= 1e-30 (subnormal partial sums) go to float64 with every candidate.
__device__ __forceinline__ int refine_row(unsigned long long mask, const float *__restrict__ x,
                                          const float *__restrict__ centroids, int D, float eps)
{
    if (__popcll(mask) == 1) return __ffsll((long long)mask) - 1;
    float s1 = INFINITY, s2 = INFINITY;
    int k1 = 0;
    for (unsigned long long m = mask; m; m &= m - 1) {
        const int k = __ffsll((long long)m) - 1;
        const float *c = centroids + (size_t)k * D;
        float s = 0.f;
        for (int d = 0; d < D; ++d) {
            const float df = x[d] - __ldg(c + d);
            s = fmaf(df, df, s);
        }
        if (s < s1) { s2 = s1; s1 = s; k1 = k; }
        else if (s < s2) s2 = s;
    }
    if ((s2 * (1.f - eps) > s1 * (1.f + eps)) && (s1 > 1e-30f)) return k1;
    const float bound = s1 * (1.f + 2.f * eps);
    double best = INFINITY;
    int mine = 0;                                    // the float64 scan starts from (inf, 0) and needs d2 < best
    for (unsigned long long m = mask; m; m &= m - 1) {
        const int k = __ffsll((long long)m) - 1;
        const float *c = centroids + (size_t)k * D;
        float s = 0.f;
        for (int d = 0; d < D; ++d) {
            const float df = x[d] - __ldg(c + d);
            s = fmaf(df, df, s);
        }
        if (!(s * (1.f - 2.f * eps) <= bound) && (s1 > 1e-30f)) continue;
        const double d2 = sqdist_scipy(c, x, D);
        if (d2 < best) { best = d2; mine = k; }
    }
    return mine;
}

__device__ __forceinline__ float sqdist_f32(const float *__restrict__ x, const float *__restrict__ c, int D)
{
    float s = 0.f;
    for (int d = 0; d < D; ++d) {
        const float df = x[d] - __ldg(c + d);
        s = fmaf(df, df, s);
    }
    return s;
}

// Stages B and C for the 32 rows of a warp (lane = row).  Rows with one candidate are done.  The
// (row, candidate) pairs of the others are pooled and dealt out one per lane, so the float32
// distances cost one pass over D for the whole warp instead of one pass per candidate of the
// unluckiest lane.  Falls back to refine_row when the pool would overflow.
__device__ __forceinline__ int refine_warp(unsigned long long mask, const float *__restrict__ xt, int pitch,
                                           const float *__restrict__ centroids, int D, float eps,
                                           unsigned short *__restrict__ pair, float *__restrict__ dist, int lane)
{
    const int n = __popcll(mask);
    const int want = n > 1 ? n : 0;
    int incl = want;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return __ffsll((long long)mask) - 1;                 // whole warp decided by stage A
    if (total > kTcPairs) return refine_row(mask, xt + lane * pitch, centroids, D, eps);
    const int off = incl - want;
    if (want) {
        int i = off;
        for (unsigned long long m = mask; m; m &= m - 1) pair[i++] = (unsigned short)((lane << 8) | (__ffsll((long long)m) - 1));
    }
    __syncwarp();
    for (int p = lane; p < total; p += 32) {
        const unsigned pr = pair[p];
        dist[p] = sqdist_f32(xt + (pr >> 8) * pitch, centroids + (size_t)(pr & 0xffu) * D, D);
    }
    __syncwarp();
    int mine = __ffsll((long long)mask) - 1;
    if (want) {
        float s1 = INFINITY, s2 = INFINITY;
        int k1 = 0;
        for (int i = off; i < off + want; ++i) {
            const float s = dist[i];
            const int k = pair[i] & 0xffu;
            if (s < s1) { s2 = s1; s1 = s; k1 = k; }
            else if (s < s2) s2 = s;
        }
        if ((s2 * (1.f - eps) > s1 * (1.f + eps)) && (s1 > 1e-30f)) {
            mine = k1;
        } else {                                                          // float64, near ties only
            const float bound = s1 * (1.f + 2.f * eps);
            double best = INFINITY;
            mine = 0;                                                     // the float64 scan starts from (inf, 0)
            for (int i = off; i < off + want; ++i) {
                if (!(dist[i] * (1.f - 2.f * eps) <= bound) && (s1 > 1e-30f)) continue;
                const int k = pair[i] & 0xffu;
                const double d2 = sqdist_scipy(centroids + (size_t)k * D, xt + lane * pitch, D);
                if (d2 < best) { best = d2; mine = k; }
            }
        }
    }
    __syncwarp();
    return mine;
}

}  // namespace gsl
