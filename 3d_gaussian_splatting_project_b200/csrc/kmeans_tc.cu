// K-means assignment with tensor-core screening (K <= 64, 8 <= D <= 64), sm_100a.
//
// The labels must be exactly those of scipy's float64 scan (3D_clustering/k_means.py:116-122);
// what can be approximate is the WORK that proves most centroids cannot win.  Three stages per
// 256-row tile, every stage with a rigorous error bound so that the set it forwards always
// contains the true nearest centroid (and every exact tie):
//
//   A  tensor cores: with m = mean of the centroids, x' = x - m, c' = c - m (distances are
//      translation invariant), rank k by  g_k = |c'_k|^2 - 2 x'.c'_k  where the dot products of
//      a 32-row x 64-centroid block are TF32 mma.sync.m16n8k8 (operands rounded with
//      cvt.rna.tf32, FP32 accumulate).  |g_k - exact| <= E_k = 1.5 * 2^-9 |x'| |c'_k| +
//      2^-22 (|x'| + |c'_k|)^2 (operand rounding 2^-11 each, doubled by the factor 2, 1.5x margin
//      for the accumulation; second term: rounding of the centring itself).  The kernel uses the
//      row-wide bound E = max_k E_k (one value per row instead of one per pair):  candidates =
//      { k : g_k <= min_j g_j + 2 E }, a superset of { k : g_k - E_k <= min_j (g_j + E_j) }.
//      Typically one or two per row.  The bound is proven only where stage A's float32 arithmetic
//      neither overflows nor underflows; rows outside that range take every centroid
//      (screen_in_range, kmeans_screen.cuh).
//   B  CUDA cores, candidates only: float32 sum of (x-c)^2 on the original values, relative
//      error (D + 3) 2^-24; decided when the two smallest differ by more than that.
//   C  float64, near ties only: scipy-order distance, lowest index first.
//
// gsl_kmeans_screen_selftest measures stage A's bound on real data: for every (row, k) it
// compares (g_k - g_0) with the float64 (d2_k - d2_0) and counts violations of E_k + E_0; rows
// outside screen_in_range are counted apart, not checked.
//
// The per-cluster float64 sums that follow are the shared segmented reduction
// (kmeans_common.cuh).  Compiled with -fmad=false.
#include "common.cuh"
#include "kmeans_common.cuh"
#include "kmeans_screen.cuh"

namespace gsl {

constexpr int kTcThreads = 256;          // 8 warps x 32 rows
constexpr int kTcRows = 256;
constexpr int kTcKP = 64;                // centroids padded to 64 (8 n-tiles)
constexpr int kTcCPitch = 68;            // c' row pitch: 68 % 32 == 4 -> conflict-free B fragments

struct TcSmem {
    size_t acc, cprime, cn2, nc, mean, tile, lab, mask, bar, total;
    int pitch;     // tile row pitch in floats (= D: the global block is copied verbatim)
    int ksteps;    // ceil(D / 8)
};

static inline TcSmem tc_layout(int D, int K, bool accumulate)
{
    TcSmem s;
    s.ksteps = (D + 7) / 8;
    s.pitch = D;        // rows stay packed: the tile is one contiguous bulk copy of the [256][D] block
    size_t o = 0;
    s.acc = o;    o += accumulate ? align_up((size_t)K * (D + 1) * sizeof(double), 16) : 0;
    s.cprime = o; o += (size_t)kTcKP * kTcCPitch * sizeof(float);
    s.cn2 = o;    o += kTcKP * sizeof(float);
    s.nc = o;     o += 2 * kTcKP * sizeof(float);
    s.mean = o;   o += 64 * sizeof(float);
    s.tile = o;   o += align_up((size_t)kTcRows * s.pitch * sizeof(float), 16);
    s.lab = o;    o += accumulate ? align_up((size_t)K * (kTcThreads / 32) * sizeof(unsigned) + (size_t)(K + 2) * 2 + (size_t)kTcRows * 2, 16) : 0;   // member bits [K][warps], cstart[K+1], order[rows]
    s.mask = o;   o += kTcRows * sizeof(unsigned long long);
    s.bar = o;    o += 16;                                   // mbarrier of the bulk copy
    s.total = o;
    return s;
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Stage A for the 32 rows of one warp.  On return, for mt in {0,1}, h in {0,1}: row
// mt*16 + (lane>>2) + 8h has, in this thread, g[mt][j][2h+c] and E[...] for centroid
// 8j + 2(lane&3) + c, and nx[mt][h] = |x'| (upper bound).
struct ScreenOut {
    float g[2][8][4];
    float nx[2][2];
};

__device__ __forceinline__ void screen_warp(ScreenOut &o, const float *__restrict__ xt, int pitch, int D, int ksteps,
                                            const float *__restrict__ cprime, const float *__restrict__ cn2,
                                            const float *__restrict__ mean, int lane)
{
    const int g = lane >> 2, t = lane & 3;
    float nx2[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) o.g[mt][j][c] = 0.f;

    for (int ks = 0; ks < ksteps; ++ks) {
        const int d0 = 8 * ks + t, d1 = d0 + 4;
        const bool in0 = d0 < D, in1 = d1 < D;
        const float m0 = mean[d0], m1 = mean[d1];
        uint32_t a[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const float *r0 = xt + (mt * 16 + g) * pitch, *r1 = r0 + 8 * pitch;
            const float x00 = in0 ? r0[d0] - m0 : 0.f, x10 = in0 ? r1[d0] - m0 : 0.f;
            const float x01 = in1 ? r0[d1] - m1 : 0.f, x11 = in1 ? r1[d1] - m1 : 0.f;
            nx2[mt][0] = fmaf(x00, x00, fmaf(x01, x01, nx2[mt][0]));
            nx2[mt][1] = fmaf(x10, x10, fmaf(x11, x11, nx2[mt][1]));
            a[mt][0] = to_tf32(x00); a[mt][1] = to_tf32(x10); a[mt][2] = to_tf32(x01); a[mt][3] = to_tf32(x11);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float *cp = cprime + (8 * j + g) * kTcCPitch + 8 * ks + t;
            const uint32_t b0 = __float_as_uint(cp[0]), b1 = __float_as_uint(cp[4]);
            mma_tf32(o.g[0][j], a[0], b0, b1);
            mma_tf32(o.g[1][j], a[1], b0, b1);
        }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float v = nx2[mt][h];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            o.nx[mt][h] = sqrtf(v) * 1.0001f;
        }
    // dot -> g = |c'|^2 - 2 x'.c'
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) o.g[mt][j][c] = cn2[8 * j + 2 * t + (c & 1)] - 2.f * o.g[mt][j][c];
}

template <bool kAccumulate, bool kCheck>
__global__ void __launch_bounds__(kTcThreads, 2)
kmeans_step_tc_kernel(const float *__restrict__ data, int64_t N, int D, const float *__restrict__ centroids,
                      int K, int32_t *__restrict__ labels, double *__restrict__ partials,
                      TcSmem L, int vec_ok, float eps, unsigned long long *__restrict__ check_out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *acc = reinterpret_cast<double *>(smem + L.acc);
    float *cprime = reinterpret_cast<float *>(smem + L.cprime);
    float *cn2 = reinterpret_cast<float *>(smem + L.cn2);
    float *eab = reinterpret_cast<float *>(smem + L.nc);       // interleaved {ea_k, eb_k}, see screen_bound
    float *mean = reinterpret_cast<float *>(smem + L.mean);
    float *tile = reinterpret_cast<float *>(smem + L.tile);
    unsigned *bits = reinterpret_cast<unsigned *>(smem + L.lab);
    unsigned short *cstart = reinterpret_cast<unsigned short *>(bits + K * (kTcThreads / 32));
    unsigned short *order = cstart + ((K + 2) & ~1);
    unsigned long long *maskbuf = reinterpret_cast<unsigned long long *>(smem + L.mask);
    void *bar = smem + L.bar;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int pitch = L.pitch;

    // ---- per-CTA prologue: centre the centroids, round to TF32, norms
    if (t < 64) {
        float s = 0.f;
        if (t < D)
            for (int k = 0; k < K; ++k) s += centroids[k * D + t];
        mean[t] = t < D ? s / (float)K : 0.f;
    }
    __syncthreads();
    for (int i = t; i < kTcKP * kTcCPitch; i += kTcThreads) {
        const int k = i / kTcCPitch, d = i - k * kTcCPitch;
        const float v = (k < K && d < D) ? centroids[k * D + d] - mean[d] : 0.f;
        cprime[i] = v;                                  // float32 for now; rounded to TF32 below
    }
    __syncthreads();
    if (t < kTcKP) {
        float s = 0.f;
        for (int d = 0; d < D; ++d) s = fmaf(cprime[t * kTcCPitch + d], cprime[t * kTcCPitch + d], s);
        cn2[t] = t < K ? s : INFINITY;                  // padded centroids can never be candidates
        const float ncu = t < K ? sqrtf(s) * 1.0001f : 0.f;
        eab[2 * t] = 2.9296875e-3f * ncu;               // 1.5 * 2^-9 |c'_k|
        eab[2 * t + 1] = 4.76837158203125e-7f * ncu * ncu * 1.0001f;   // 2^-21 |c'_k|^2
    }
    __syncthreads();
    // row-wide bound: the largest ea_k, eb_k over the real centroids (both grow with |c'_k|)
    float ea_max = 0.f, eb_max = 0.f;
    for (int k = 0; k < K; ++k) { ea_max = fmaxf(ea_max, eab[2 * k]); eb_max = fmaxf(eb_max, eab[2 * k + 1]); }
    for (int i = t; i < kTcKP * kTcCPitch; i += kTcThreads) cprime[i] = __uint_as_float(to_tf32(cprime[i]));
    if (kAccumulate)
        for (int i = t; i < K * (D + 1); i += kTcThreads) acc[i] = 0.0;
    const unsigned long long kmask = K >= 64 ? ~0ull : ((1ull << K) - 1ull);
    unsigned long long n_viol = 0, n_cand = 0, n_skip = 0;

    // Tiles arrive by TMA bulk copy: full 256-row tiles of a 16-byte aligned matrix are one
    // cp.async.bulk each (no staging instructions, no registers); the copy of the NEXT tile is
    // launched as soon as the buffer is free, i.e. right after this tile's accumulation.
    const int64_t n_tiles = (N + kTcRows - 1) / kTcRows;
    const unsigned tile_bytes = (unsigned)(kTcRows * D * sizeof(float));
    unsigned phase = 0;
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    auto bulk_ok = [&](int64_t tl) { return vec_ok && (tl + 1) * kTcRows <= N; };
    if (t == 0 && (int64_t)blockIdx.x < n_tiles && bulk_ok(blockIdx.x))
        bulk_load_tile(tile, data + (int64_t)blockIdx.x * kTcRows * D, tile_bytes, bar);
    for (int64_t tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
        const int64_t row0 = tl * kTcRows;
        const int rows = (int)min((int64_t)kTcRows, N - row0);
        if (bulk_ok(tl)) {
            mbar_wait(bar, phase);
            phase ^= 1u;
        } else {                                         // ragged last tile or unaligned matrix
            stage_tile(tile, pitch, data + row0 * D, rows, D, false, t, kTcThreads);
            for (int i = rows * pitch + t; i < kTcRows * pitch; i += kTcThreads) tile[i] = 0.f;
        }
        if (kAccumulate) zero_member_bits(bits, K, kTcThreads / 32, t, kTcThreads);
        __syncthreads();

        // ---- stage A: this warp's 32 rows against all centroids
        ScreenOut so;
        screen_warp(so, tile + warp * 32 * pitch, pitch, D, L.ksteps, cprime, cn2, mean, lane);
        const int g = lane >> 2, tq = lane & 3;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float nx = so.nx[mt][h];
                const float nx_term = 4.76837158203125e-7f * nx * nx * 1.0001f;        // 2^-21 |x'|^2
                // smallest ranking value of the row, then every k within 2 E of it (padded centroids
                // carry g = +inf and never qualify)
                float gmin = INFINITY;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    gmin = fminf(gmin, fminf(so.g[mt][j][2 * h], so.g[mt][j][2 * h + 1]));
                gmin = fminf(gmin, __shfl_xor_sync(0xffffffffu, gmin, 1));
                gmin = fminf(gmin, __shfl_xor_sync(0xffffffffu, gmin, 2));
                const float bnd = screen_bound(nx, nx_term, ea_max, eb_max);
                const float thr = gmin + 2.f * (bnd * 1.000001f);
                unsigned m_lo = 0, m_hi = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int n = 8 * j + 2 * tq + c;
                        const unsigned bit = (so.g[mt][j][2 * h + c] <= thr) ? 1u : 0u;
                        if (n < 32) m_lo |= bit << n; else m_hi |= bit << (n - 32);
                    }
                m_lo |= __shfl_xor_sync(0xffffffffu, m_lo, 1); m_hi |= __shfl_xor_sync(0xffffffffu, m_hi, 1);
                m_lo |= __shfl_xor_sync(0xffffffffu, m_lo, 2); m_hi |= __shfl_xor_sync(0xffffffffu, m_hi, 2);
                unsigned long long mask = (((unsigned long long)m_hi << 32) | m_lo) & kmask;
                // rows outside the range where the bound is proven (screen_in_range), and NaN/Inf rows:
                // everything is a candidate
                const bool in_range = screen_in_range(bnd);
                if (mask == 0 || !in_range) mask = kmask;
                if (tq == 0) maskbuf[warp * 32 + mt * 16 + g + 8 * h] = mask;

                if (kCheck) {
                    // bound check: (g_k - g_0) vs float64 (d2_k - d2_0), tolerance E_k + E_0
                    const int r = warp * 32 + mt * 16 + g + 8 * h;
                    const float g0 = __shfl_sync(0xffffffffu, so.g[mt][0][2 * h], lane & ~3);
                    const float e0 = screen_bound(nx, nx_term, eab[0], eab[1]);
                    if (r < rows && !in_range && tq == 0) ++n_skip;
                    if (r < rows && in_range) {
                        const float *x = tile + r * pitch;
                        const double d0 = sqdist_scipy(centroids, x, D);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                const int n = 8 * j + 2 * tq + c;
                                if (n >= K) continue;
                                const double dk = sqdist_scipy(centroids + (size_t)n * D, x, D);
                                const double err = fabs(((double)so.g[mt][j][2 * h + c] - (double)g0) - (dk - d0));
                                const double tol = (double)screen_bound(nx, nx_term, eab[2 * n], eab[2 * n + 1]) + (double)e0;
                                if (!(err <= tol)) ++n_viol;
                            }
                    }
                }
            }
        __syncwarp();

        // ---- stages B, C: lane = row
        int mine = -1;
        {
            const unsigned long long mask = t < rows ? maskbuf[t] : 1ull;  // rows past the end: decided, ignored
            __syncwarp();                                 // masks are in registers: their slots become the work list
            if (kCheck && t < rows) n_cand += __popcll(mask);
            float *distbuf = reinterpret_cast<float *>(maskbuf + warp * 32);
            unsigned short *pairbuf = reinterpret_cast<unsigned short *>(distbuf + kTcPairs);
            const int k = refine_warp(mask, tile + warp * 32 * pitch, pitch, centroids, D, eps, pairbuf, distbuf, lane);
            if (t < rows) {
                mine = k;
                labels[row0 + t] = mine;
            }
        }
        if (kAccumulate) {
            const unsigned same = tile_member_bits(bits, mine, kTcThreads / 32, lane, warp);
            __syncthreads();
            if (warp == 0) tile_cluster_starts(bits, cstart, K, kTcThreads / 32, lane);
            __syncthreads();
            tile_row_order(bits, cstart, order, mine, same, kTcThreads / 32, t, lane, warp);
            __syncthreads();
            accumulate_tile(acc, tile, pitch, cstart, order, K, D, lane, warp, kTcThreads / 32);
        }
        __syncthreads();                                 // every reader of the tile is done
        const int64_t nxt = tl + gridDim.x;
        if (t == 0 && nxt < n_tiles && bulk_ok(nxt))
            bulk_load_tile(tile, data + nxt * kTcRows * D, tile_bytes, bar);
    }
    if (kAccumulate) {
        __syncthreads();
        double *out = partials + (size_t)blockIdx.x * K * (D + 1);
        for (int i = t; i < K * (D + 1); i += kTcThreads) out[i] = acc[i];
    }
    if (kCheck) {
        atomicAdd(check_out, n_viol);
        atomicAdd(check_out + 1, n_cand);
        atomicAdd(check_out + 2, n_skip);
    }
}

bool tc_supported(int D, int K)
{
    return K >= 1 && K <= 64 && D >= 8 && D <= 64;
}

template <bool kAcc, bool kCheck>
static int launch_tc_t(const float *data, int64_t N, int D, const float *centroids, int K, int32_t *labels,
                       double *partials, int grid, unsigned long long *check_out, cudaStream_t st)
{
    const TcSmem L = tc_layout(D, K, kAcc);
    if (L.total > 227 * 1024) return fail(GSL_EINVAL, "kmeans (tensor-core screening): %zu B of shared memory", L.total);
    GSL_CUDA_TRY(cudaFuncSetAttribute(kmeans_step_tc_kernel<kAcc, kCheck>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    const int vec_ok = (((uintptr_t)data & 15) == 0);        // 256 rows x D floats is always a multiple of 16 bytes
    const float eps = (float)((D + 12) * 5.9604644775390625e-08);
    kmeans_step_tc_kernel<kAcc, kCheck><<<grid, kTcThreads, L.total, st>>>(data, N, D, centroids, K, labels, partials, L, vec_ok, eps, check_out);
    GSL_LAUNCH_CHECK("kmeans_step_tc_kernel");
    return GSL_OK;
}

int launch_step_tc(bool accumulate, const float *data, int64_t N, int D, const float *centroids, int K,
                   int32_t *labels, double *partials, int grid, cudaStream_t st)
{
    return accumulate ? launch_tc_t<true, false>(data, N, D, centroids, K, labels, partials, grid, nullptr, st)
                      : launch_tc_t<false, false>(data, N, D, centroids, K, labels, partials, grid, nullptr, st);
}

}  // namespace gsl

using namespace gsl;

extern "C" int gsl_kmeans_screen_selftest(const float *data, int64_t N, int D, const float *centroids, int K,
                                          int32_t *labels, unsigned long long *out3, void *stream)
{
    if (!data || !centroids || !labels || !out3 || N < 0) return fail(GSL_EINVAL, "gsl_kmeans_screen_selftest: bad argument");
    if (!tc_supported(D, K)) return fail(GSL_EINVAL, "gsl_kmeans_screen_selftest: needs K <= 64 and 8 <= D <= 64");
    if (N == 0) return GSL_OK;
    const int64_t tiles = (N + kTcRows - 1) / kTcRows;
    const int64_t cap = (int64_t)sm_count() * 2;
    return launch_tc_t<false, true>(data, N, D, centroids, K, labels, nullptr, (int)(tiles < cap ? tiles : cap), out3, (cudaStream_t)stream);
}
