// Device helpers shared by the K-means kernels (kmeans.cu, kmeans_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gsl {

// scipy ckdtree sqeuclidean_distance_double on float64 copies of float32 values.
__device__ __forceinline__ double sqdist_scipy(const float *__restrict__ c, const float *__restrict__ x, int D)
{
    double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
    int i = 0;
    for (; i + 4 <= D; i += 4) {
        const double d0 = (double)c[i] - (double)x[i];
        const double d1 = (double)c[i + 1] - (double)x[i + 1];
        const double d2 = (double)c[i + 2] - (double)x[i + 2];
        const double d3 = (double)c[i + 3] - (double)x[i + 3];
        a0 += d0 * d0; a1 += d1 * d1; a2 += d2 * d2; a3 += d3 * d3;
    }
    double s = a0 + a1 + a2 + a3;
    for (; i < D; ++i) {
        const double d = (double)c[i] - (double)x[i];
        s += d * d;
    }
    return s;
}

// Stage the contiguous [rows x D] float32 block at `src` into shared memory with `pitch` floats
// per row.  `vec` = the block is 16-byte aligned and a whole number of float4.  Loads are issued
// five at a time before any of them is consumed (one round trip per batch, not per load).
__device__ __forceinline__ void stage_tile(float *__restrict__ tile, int pitch, const float *__restrict__ src,
                                           int rows, int D, bool vec, int t, int n_threads)
{
    const int n_el = rows * D;
    if (vec) {
        constexpr int B = 5;
        const float4 *src4 = reinterpret_cast<const float4 *>(src);
        const int n4 = n_el >> 2;
        for (int i0 = t; i0 < n4; i0 += B * n_threads) {
            float4 v[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = i0 + b * n_threads;
                if (i < n4) v[b] = __ldcs(src4 + i);
            }
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = i0 + b * n_threads;
                if (i < n4) {
                    const int e = i << 2;
                    int r = e / D, d = e - r * D;
                    const float vv[4] = {v[b].x, v[b].y, v[b].z, v[b].w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        tile[r * pitch + d] = vv[j];
                        if (++d == D) { d = 0; ++r; }
                    }
                }
            }
        }
    } else {
        for (int i = t; i < n_el; i += n_threads) {
            const int r = i / D, d = i - r * D;
            tile[r * pitch + d] = __ldcs(src + i);
        }
    }
}

// Segmented reduction of one staged tile into the CTA's [K][D+1] float64 accumulator, as a
// counting sort of the tile's rows by label followed by one sequential walk per cluster:
//   zero_member_bits   clear bits[K][n_warps]
//   tile_member_bits   every warp groups its 32 rows by label with one match_any; the lowest lane
//                      of each group publishes the group's lane mask: bits[k][w] = rows of warp w
//                      with label k
//   tile_cluster_starts  (warp 0) member count per cluster and its exclusive scan -> cstart[K+1]
//   tile_row_order     every row computes its slot: cstart[k] + members in lower warps + members in
//                      lower lanes of its own warp -> order[slot] = row.  Ascending row order inside
//                      every cluster, no atomics.
//   accumulate_tile    warp w owns the clusters k = w (mod n_warps): walks order[cstart[k] ..
//                      cstart[k+1]) and adds the rows lane-per-dimension in float64.
// Fixed order everywhere: results are bit-reproducible.  A __syncthreads separates the steps.
__device__ __forceinline__ void zero_member_bits(unsigned *__restrict__ bits, int K, int n_warps, int t, int n_threads)
{
    for (int i = t; i < K * n_warps; i += n_threads) bits[i] = 0u;
}

// Returns the mask of lanes of this warp that share this thread's label.
__device__ __forceinline__ unsigned tile_member_bits(unsigned *__restrict__ bits, int lab, int n_warps, int lane, int warp)
{
    const unsigned same = __match_any_sync(0xffffffffu, lab);
    if (lab >= 0 && lane == __ffs(same) - 1) bits[lab * n_warps + warp] = same;
    return same;
}

__device__ __forceinline__ void tile_cluster_starts(const unsigned *__restrict__ bits, unsigned short *__restrict__ cstart,
                                                    int K, int n_warps, int lane)
{
    // clusters are dealt to the lanes in contiguous runs so that one warp scan finishes the job
    const int per = (K + 31) / 32;
    const int k0 = min(lane * per, K), k1 = min(k0 + per, K);
    int mine = 0;
    for (int k = k0; k < k1; ++k)
        for (int w = 0; w < n_warps; ++w) mine += __popc(bits[k * n_warps + w]);
    int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    int run = incl - mine;
    for (int k = k0; k < k1; ++k) {
        cstart[k] = (unsigned short)run;
        for (int w = 0; w < n_warps; ++w) run += __popc(bits[k * n_warps + w]);
    }
    if (lane == 31) cstart[K] = (unsigned short)incl;
}

__device__ __forceinline__ void tile_row_order(const unsigned *__restrict__ bits, const unsigned short *__restrict__ cstart,
                                               unsigned short *__restrict__ order, int lab, unsigned same,
                                               int n_warps, int t, int lane, int warp)
{
    if (lab < 0) return;
    int slot = cstart[lab] + __popc(same & ((1u << lane) - 1u));
    for (int w = 0; w < warp; ++w) slot += __popc(bits[lab * n_warps + w]);
    order[slot] = (unsigned short)t;
}

__device__ __forceinline__ void accumulate_tile(double *__restrict__ acc, const float *__restrict__ tile, int pitch,
                                                const unsigned short *__restrict__ cstart,
                                                const unsigned short *__restrict__ order, int K, int D,
                                                int lane, int warp, int n_warps)
{
    for (int k = warp; k < K; k += n_warps) {
        const int i0 = cstart[k], i1 = cstart[k + 1];
        if (i0 == i1) continue;
        for (int d0 = 0; d0 < D; d0 += 64) {
            const int da = d0 + lane, db = da + 32;
            const bool ina = da < D, inb = db < D;
            double sa = 0.0, sb = 0.0;
            for (int i = i0; i < i1; ++i) {
                const float *row = tile + (int)order[i] * pitch;
                if (ina) sa += (double)row[da];
                if (inb) sb += (double)row[db];
            }
            if (ina) acc[k * (D + 1) + da] += sa;
            if (inb) acc[k * (D + 1) + db] += sb;
        }
        if (lane == 0) acc[k * (D + 1) + D] += (double)(i1 - i0);
    }
}

}  // namespace gsl
