// K-means labelling for sm_100a: assignment, fused per-cluster sums, finalize.
//
// Replaces the per-point KDTree.query loop and the K boolean-mask means of
// k_means_with_color / k_means_kd_tree (3D_clustering/k_means.py:113-144, "km" below).
//
//   kmeans_step_kernel<kAccumulate>
//        persistent CTAs, one tile of TR rows at a time staged in shared memory
//        (coalesced float4 loads of the contiguous [TR x D] block).  One thread per row
//        evaluates scipy's float64 squared distance to every centroid in scipy's own
//        summation order (four running lanes, no FMA; see oracle/gsl_oracle.c) and keeps
//        the first minimum.  With kAccumulate the tile is then reduced per cluster:
//        each warp owns the clusters k = warp (mod warps), finds their rows with ballots in
//        ascending row order, and adds them lane-per-dimension in float64 into the CTA's
//        [K][D+1] accumulator in shared memory -- a segmented reduction with no atomics
//        and a fixed order, so results are bit-reproducible.
//   kmeans_reduce_kernel      fixed-order sum of the per-CTA partials -> sums[K][D+1]
//   kmeans_finalize_kernel    new = float32(sum / count) or old; shift = ||new - old||_F
//   kmeans_exchange_kernel    reduce + push to every rank over peer memory + rank-ordered total + finalize
//
// Compiled with -fmad=false (the distance must not be contracted).
#include <stdlib.h>

#include "common.cuh"
#include "kmeans_common.cuh"

namespace gsl {

constexpr int kStepThreads = 256;   // rows per tile == threads per CTA
constexpr int kStepWarps = kStepThreads / 32;

struct StepSmem {
    // byte offsets into dynamic shared memory
    size_t tile, cent, acc, lab, total;
    int pitch;    // row pitch of the tile in floats (odd -> conflict-free row-per-lane reads)
    int cpitch;   // row pitch of the centroid block in floats (D, or DREG zero-padded)
};

static inline StepSmem step_layout(int D, int K, bool accumulate, int dreg)
{
    StepSmem s;
    s.pitch = D | 1;
    s.cpitch = dreg ? dreg : D;
    size_t o = 0;
    s.acc = o;  o += accumulate ? align_up((size_t)K * (D + 1) * sizeof(double), 16) : 0;
    s.cent = o; o += align_up((size_t)K * s.cpitch * sizeof(float), 16);
    s.tile = o; o += align_up((size_t)kStepThreads * s.pitch * sizeof(float), 16);
    s.lab = o;  o += accumulate ? align_up((size_t)K * kStepWarps * sizeof(unsigned) + (size_t)(K + 2) * 2 + (size_t)kStepThreads * 2, 16) : 0;   // member bits [K][warps], cstart[K+1], order[rows]
    s.total = o;
    return s;
}

// Float32 screening distance: sum of fmaf((x-c), (x-c), s) over DREG zero-padded dims, the row
// in registers, the centroid read as broadcast 16-byte shared loads.  Every partial sum is
// non-negative, so the result is within (DREG + 3) ulp-relative of the real distance.
template <int DREG>
__device__ __forceinline__ float sqdist_screen(const float (&x)[DREG], const float *__restrict__ c)
{
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int i = 0; i < DREG; i += 4) {
        const float4 cv = *reinterpret_cast<const float4 *>(c + i);
        const float d0 = x[i] - cv.x, d1 = x[i + 1] - cv.y, d2 = x[i + 2] - cv.z, d3 = x[i + 3] - cv.w;
        s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s0 = fmaf(d2, d2, s0); s1 = fmaf(d3, d3, s1);
    }
    return s0 + s1;
}

// Nearest centroid of one row, exactly as the float64 scan would find it (first minimum of the
// scipy-order distance), at float32 cost: screen all K in float32, and only when the two
// smallest screened distances are closer than the screening error can explain, evaluate the
// float64 distance of the candidates inside the error band.
template <int DREG>
__device__ __forceinline__ int nearest_screened(const float *__restrict__ xrow, const float *__restrict__ cent,
                                                int K, int D, float eps)
{
    float x[DREG];
#pragma unroll
    for (int i = 0; i < DREG; ++i) x[i] = i < D ? xrow[i] : 0.f;
    float s1 = INFINITY, s2 = INFINITY;
    int k1 = 0;
    for (int k = 0; k < K; ++k) {
        const float s = sqdist_screen<DREG>(x, cent + k * DREG);
        if (s < s1) { s2 = s1; s1 = s; k1 = k; }
        else if (s < s2) s2 = s;
    }
    // unique  <=>  every other real distance exceeds the smallest one even after both move by eps
    const bool unique = (s2 * (1.f - eps) > s1 * (1.f + eps)) && (s1 > 1e-30f);
    if (unique) return k1;
    const float bound = s1 * (1.f + 2.f * eps);
    double best = INFINITY;
    int mine = 0;
    for (int k = 0; k < K; ++k) {
        const float s = sqdist_screen<DREG>(x, cent + k * DREG);
        if (!(s * (1.f - 2.f * eps) <= bound) && (s1 > 1e-30f)) continue;     // outside the band
        const double d2 = sqdist_scipy(cent + k * DREG, xrow, D);
        if (d2 < best) { best = d2; mine = k; }
    }
    return mine;
}

// DREG = 0: float64 scan of every centroid (any D).  DREG > 0: float32 screening with the row
// in DREG registers (D <= DREG), float64 only for near ties.  Both give identical labels.
template <int DREG, bool kAccumulate>
__global__ void __launch_bounds__(kStepThreads)
kmeans_step_kernel(const float *__restrict__ data, int64_t N, int D, const float *__restrict__ centroids,
                   int K, int32_t *__restrict__ labels, double *__restrict__ partials,
                   StepSmem L, int vec_ok, float eps)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *acc = reinterpret_cast<double *>(smem + L.acc);
    float *tile = reinterpret_cast<float *>(smem + L.tile);
    float *cent = reinterpret_cast<float *>(smem + L.cent);
    unsigned *bits = reinterpret_cast<unsigned *>(smem + L.lab);
    unsigned short *cstart = reinterpret_cast<unsigned short *>(bits + K * kStepWarps);
    unsigned short *order = cstart + ((K + 2) & ~1);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int pitch = L.pitch, cpitch = L.cpitch;

    for (int i = t; i < K * cpitch; i += kStepThreads) {
        const int k = i / cpitch, d = i - k * cpitch;
        cent[i] = d < D ? centroids[k * D + d] : 0.f;
    }
    if (kAccumulate)
        for (int i = t; i < K * (D + 1); i += kStepThreads) acc[i] = 0.0;

    const int64_t n_tiles = (N + kStepThreads - 1) / kStepThreads;
    for (int64_t tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
        const int64_t row0 = tl * kStepThreads;
        const int rows = (int)min((int64_t)kStepThreads, N - row0);
        __syncthreads();   // previous tile fully consumed (and cent/acc initialised)
        stage_tile(tile, pitch, data + row0 * D, rows, D, vec_ok && rows == kStepThreads, t, kStepThreads);
        if (kAccumulate) zero_member_bits(bits, K, kStepWarps, t, kStepThreads);
        __syncthreads();
        // ---- assignment: thread = row
        int mine = -1;
        if (t < rows) {
            const float *x = tile + t * pitch;
            if (DREG > 0) {
                mine = nearest_screened<(DREG > 0 ? DREG : 4)>(x, cent, K, D, eps);
            } else {
                double best = sqdist_scipy(cent, x, D);
                mine = 0;
                for (int k = 1; k < K; ++k) {
                    const double d2 = sqdist_scipy(cent + k * cpitch, x, D);
                    if (d2 < best) { best = d2; mine = k; }
                }
            }
            labels[row0 + t] = mine;
        }
        if (!kAccumulate) continue;
        const unsigned same = tile_member_bits(bits, mine, kStepWarps, lane, warp);
        __syncthreads();
        if (warp == 0) tile_cluster_starts(bits, cstart, K, kStepWarps, lane);
        __syncthreads();
        tile_row_order(bits, cstart, order, mine, same, kStepWarps, t, lane, warp);
        __syncthreads();
        accumulate_tile(acc, tile, pitch, cstart, order, K, D, lane, warp, kStepWarps);
    }
    if (kAccumulate) {
        __syncthreads();
        double *out = partials + (size_t)blockIdx.x * K * (D + 1);
        for (int i = t; i < K * (D + 1); i += kStepThreads) out[i] = acc[i];
    }
}

// Fixed-order sum of the per-CTA partials.  A block of 32 warps owns 32 consecutive elements; warp
// w adds the partials p = w, w + 32, ... (coalesced 256-byte rows, a handful of independent loads
// per thread), then warp 0 adds the 32 warp sums in warp order -- the same grouping on every run
// and in both kernels that use it, so the result is reproducible.
constexpr int kReduceThreads = 1024;

__device__ __forceinline__ void reduce_partials(const double *__restrict__ partials, int n_parts, int n_el,
                                                double (&part)[32][33], int i, int lane, int w)
{
    double s = 0.0;
    if (i < n_el) {
#pragma unroll 4
        for (int p = w; p < n_parts; p += 32) s += __ldcs(partials + (size_t)p * n_el + i);
    }
    part[w][lane] = s;
    __syncthreads();
}

__global__ void __launch_bounds__(kReduceThreads)
kmeans_reduce_kernel(const double *__restrict__ partials, int n_parts, int n_el, double *__restrict__ sums)
{
    __shared__ double part[32][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    reduce_partials(partials, n_parts, n_el, part, i, lane, w);
    if (w == 0 && i < n_el) {
        double t = part[0][lane];
        for (int ww = 1; ww < 32; ++ww) t += part[ww][lane];
        sums[i] = t;
    }
}

// One CTA.  new = (float)(sum / count) (float64 quotient, as np.mean's true_divide with an
// intp count does, km:126) or old when empty; shift = Frobenius norm of the float32 difference.
__global__ void __launch_bounds__(1024)
kmeans_finalize_kernel(const double *__restrict__ sums, const float *__restrict__ old_c, int K, int D,
                       float *__restrict__ new_c, float *__restrict__ shift)
{
    __shared__ double red[32];
    double sq = 0.0;
    for (int i = threadIdx.x; i < K * D; i += blockDim.x) {
        const int k = i / D, d = i - k * D;
        const double n = sums[k * (D + 1) + D];
        const float o = old_c[i];
        const float v = n > 0.0 ? (float)(sums[k * (D + 1) + d] / n) : o;
        new_c[i] = v;
        const float df = v - o;
        sq += (double)df * (double)df;
    }
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        *shift = (float)sqrt(s);
    }
}

// ---------------------------------------------------------------------------------------
// Reduction fused with the cross-rank exchange and the update (one kernel per iteration instead of
// reduce + NCCL all-reduce + finalize).  Every rank owns an exchange buffer that all ranks can
// address (peer mapping over NVLink: torch symmetric memory on the Python side):
//     [0]    done counter of the local grid          [128] flags[rank], one u64 per source rank
//     [256]  slots[parity][source rank][n_el] float64
//   1. every CTA sums its 32 elements over the per-CTA partials of the step kernel (same fixed
//      grouping as kmeans_reduce_kernel) and PUSHES the result into slot[parity][my rank] of every
//      rank's buffer -- 256-byte coalesced stores straight into peer memory;
//   2. the last CTA to finish (device-scope ticket after a system-scope fence) publishes
//      flag[my rank] = seq on every rank with a system-scope release store, then waits until its
//      own flags from all ranks have reached seq (acquire loads);
//   3. it adds the `world` slots in RANK ORDER -- the same order on every rank, so all ranks get
//      bit-identical totals and centroids -- and forms the new centroids and the shift.
// seq grows by one per call; slots alternate by its parity.  That is enough: a rank can only be
// one exchange ahead of a peer (to start exchange s + 1 it needs that peer's flag for s), so
// the data of exchange s is never overwritten before exchange s + 2, by which time every rank has
// finished reading s.  The wait is bounded (GSLIFT_EXCHANGE_TIMEOUT_MS, default 30 s -- ranks of a
// job are lined up by a barrier before their first exchange, k_means.lloyd): on a time-out the
// shift comes back NaN.
// ---------------------------------------------------------------------------------------
constexpr int kMaxRanks = 16;
constexpr size_t kXchgFlags = 128, kXchgSlots = 256;

struct PeerTable {
    unsigned char *base[kMaxRanks];
};

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __launch_bounds__(kReduceThreads)
kmeans_exchange_kernel(const double *__restrict__ partials, int n_parts, int n_el, PeerTable peers, int rank, int world,
                       unsigned long long seq, unsigned long long timeout_ns, const float *__restrict__ old_c, int K, int D,
                       float *__restrict__ new_c, float *__restrict__ shift, double *__restrict__ sums)
{
    __shared__ double part[32][33];
    __shared__ int s_last, s_timeout;
    __shared__ double red[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const size_t slot_off = kXchgSlots + ((size_t)(seq & 1ull) * world + rank) * (size_t)n_el * sizeof(double);
    {
        const int i = blockIdx.x * 32 + lane;
        reduce_partials(partials, n_parts, n_el, part, i, lane, w);
        if (w == 0 && i < n_el) {
            double t = part[0][lane];
            for (int ww = 1; ww < 32; ++ww) t += part[ww][lane];
            for (int p = 0; p < world; ++p)                                  // push: own sums into everyone's slot[rank]
                reinterpret_cast<double *>(peers.base[p] + slot_off)[i] = t;
        }
    }
    __threadfence_system();
    __syncthreads();
    unsigned *counter = reinterpret_cast<unsigned *>(peers.base[rank]);
    if (threadIdx.x == 0) {
        s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
        s_timeout = 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence_system();
    if (threadIdx.x == 0) *counter = 0u;                                     // next call on this stream starts from zero
    if (threadIdx.x < world) {
        st_release_sys(reinterpret_cast<unsigned long long *>(peers.base[threadIdx.x] + kXchgFlags) + rank, seq);
        const unsigned long long *mine = reinterpret_cast<const unsigned long long *>(peers.base[rank] + kXchgFlags) + threadIdx.x;
        const unsigned long long t0 = global_ns();
        while (ld_acquire_sys(mine) < seq)
            if (global_ns() - t0 > timeout_ns) { s_timeout = 1; break; }
    }
    __syncthreads();
    const double *slots = reinterpret_cast<const double *>(peers.base[rank] + kXchgSlots + (size_t)(seq & 1ull) * world * (size_t)n_el * sizeof(double));
    for (int i = threadIdx.x; i < n_el; i += blockDim.x) {
        double t = 0.0;
        for (int p = 0; p < world; ++p) t += __ldcg(slots + (size_t)p * n_el + i);   // rank order; L2 is the coherence point
        sums[i] = t;
    }
    __syncthreads();                                                         // this CTA's writes to `sums` are visible to it
    double sq = 0.0;
    for (int i = threadIdx.x; i < K * D; i += blockDim.x) {
        const int k = i / D, d = i - k * D;
        const double n = sums[k * (D + 1) + D];
        const float o = old_c[i];
        const float v = n > 0.0 ? (float)(sums[k * (D + 1) + d] / n) : o;    // km:126; empty cluster keeps its centroid
        new_c[i] = v;
        const float df = v - o;
        sq += (double)df * (double)df;
    }
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if (lane == 0) red[w] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int ww = 0; ww < 32; ++ww) s += red[ww];
        *shift = s_timeout ? __int_as_float(0x7fc00000) : (float)sqrt(s);
    }
}

__global__ void __launch_bounds__(256)
recolor_kernel(const int32_t *__restrict__ labels, int64_t N, const float *__restrict__ palette,
               float *__restrict__ colors)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int c = labels[i] & 7;    // labels >= 0, so & 7 == % len(COLORS) (km:100, :148)
    colors[3 * i + 0] = palette[3 * c + 0];
    colors[3 * i + 1] = palette[3 * c + 1];
    colors[3 * i + 2] = palette[3 * c + 2];
}

static int step_grid(int64_t N)
{
    const int64_t tiles = (N + kStepThreads - 1) / kStepThreads;
    const int64_t cap = (int64_t)sm_count() * 2;
    return (int)(tiles < cap ? (tiles < 1 ? 1 : tiles) : cap);
}

}  // namespace gsl

using namespace gsl;

static int check_kd(const char *who, int64_t N, int D, int K)
{
    if (N < 0) return fail(GSL_EINVAL, "%s: negative N", who);
    if (D < 1 || D > GSL_KMEANS_MAX_D) return fail(GSL_EINVAL, "%s: D=%d not in [1, %d]", who, D, GSL_KMEANS_MAX_D);
    if (K < 1 || K > GSL_KMEANS_MAX_K) return fail(GSL_EINVAL, "%s: K=%d not in [1, %d]", who, K, GSL_KMEANS_MAX_K);
    return GSL_OK;
}

extern "C" size_t gsl_kmeans_workspace_bytes(int64_t N, int D, int K)
{
    if (N < 0 || D < 1 || K < 1) return 0;
    const size_t parts = (size_t)sm_count() * 2;
    const size_t step = parts * (size_t)K * (D + 1) * sizeof(double) + 256;
    const size_t ord = ordered_workspace_bytes(N, D, K);
    return step > ord ? step : ord;
}

// GSLIFT_KMEANS_EXACT=1 forces the float64 scan (the screening path must give the same labels).
static bool force_exact()
{
    const char *e = getenv("GSLIFT_KMEANS_EXACT");
    return e && e[0] == '1';
}

template <int DREG, bool kAcc>
static int launch_step_t(const float *data, int64_t N, int D, const float *centroids, int K,
                         int32_t *labels, double *partials, int grid, cudaStream_t st)
{
    const StepSmem L = step_layout(D, K, kAcc, DREG);
    if (L.total > 227 * 1024) return fail(GSL_EINVAL, "kmeans: K=%d, D=%d needs %zu B of shared memory (> 227 KB)", K, D, L.total);
    GSL_CUDA_TRY(cudaFuncSetAttribute(kmeans_step_kernel<DREG, kAcc>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    const int vec_ok = (((uintptr_t)data & 15) == 0) && (((size_t)kStepThreads * D) % 4 == 0);
    // screening error: (DREG + 3) roundings on non-negative partial sums, plus the float32
    // products of the comparison itself; 2^-24 per rounding, generous margin.
    const float eps = (float)((DREG + 12) * 5.9604644775390625e-08);
    kmeans_step_kernel<DREG, kAcc><<<grid, kStepThreads, L.total, st>>>(data, N, D, centroids, K, labels, partials, L, vec_ok, eps);
    GSL_LAUNCH_CHECK("kmeans_step_kernel");
    return GSL_OK;
}

// GSLIFT_KMEANS_TC=0 keeps the float32 CUDA-core screening even where tensor cores apply.
static bool allow_tc()
{
    const char *e = getenv("GSLIFT_KMEANS_TC");
    return !(e && e[0] == '0');
}

// One assignment pass (+ one block of partial sums per CTA when kAcc).
template <bool kAcc>
static int launch_step(const float *data, int64_t N, int D, const float *centroids, int K,
                       int32_t *labels, double *partials, int grid, cudaStream_t st)
{
    if (!force_exact() && allow_tc() && K >= 16 && tc_supported(D, K))
        return launch_step_tc(kAcc, data, N, D, centroids, K, labels, partials, grid, st);
    // the screened kernel pads the centroid block to DREG floats per row: fall back to the
    // float64 scan when that does not fit or the row does not fit the register block
    if (!force_exact() && D <= 64) {
        const int dreg = D <= 8 ? 8 : D <= 16 ? 16 : D <= 32 ? 32 : 64;
        if (step_layout(D, K, kAcc, dreg).total <= 227 * 1024) {
            switch (dreg) {
                case 8:  return launch_step_t<8, kAcc>(data, N, D, centroids, K, labels, partials, grid, st);
                case 16: return launch_step_t<16, kAcc>(data, N, D, centroids, K, labels, partials, grid, st);
                case 32: return launch_step_t<32, kAcc>(data, N, D, centroids, K, labels, partials, grid, st);
                default: return launch_step_t<64, kAcc>(data, N, D, centroids, K, labels, partials, grid, st);
            }
        }
    }
    return launch_step_t<0, kAcc>(data, N, D, centroids, K, labels, partials, grid, st);
}

extern "C" int gsl_kmeans_assign(const float *data, int64_t N, int D, const float *centroids, int K,
                                 int32_t *labels, void *ws, size_t ws_bytes, void *stream)
{
    (void)ws; (void)ws_bytes;
    if (int rc = check_kd("gsl_kmeans_assign", N, D, K)) return rc;
    if (N == 0) return GSL_OK;
    if (!data || !centroids || !labels) return fail(GSL_EINVAL, "gsl_kmeans_assign: null pointer");
    return launch_step<false>(data, N, D, centroids, K, labels, nullptr, step_grid(N), (cudaStream_t)stream);
}

extern "C" int gsl_kmeans_step(const float *data, int64_t N, int D, const float *centroids, int K,
                               int32_t *labels, double *sums, void *ws, size_t ws_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = check_kd("gsl_kmeans_step", N, D, K)) return rc;
    if (!centroids || !sums) return fail(GSL_EINVAL, "gsl_kmeans_step: null pointer");
    const int n_el = K * (D + 1);
    if (N == 0) {
        GSL_CUDA_TRY(cudaMemsetAsync(sums, 0, sizeof(double) * (size_t)n_el, st));
        return GSL_OK;
    }
    if (!data || !labels || !ws) return fail(GSL_EINVAL, "gsl_kmeans_step: null pointer");
    if (ws_bytes < gsl_kmeans_workspace_bytes(N, D, K)) return fail(GSL_EWORKSPACE, "gsl_kmeans_step: workspace %zu < %zu", ws_bytes, gsl_kmeans_workspace_bytes(N, D, K));
    double *partials = reinterpret_cast<double *>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    const int grid = step_grid(N);
    if (int rc = launch_step<true>(data, N, D, centroids, K, labels, partials, grid, st)) return rc;
    kmeans_reduce_kernel<<<(n_el + 31) / 32, kReduceThreads, 0, st>>>(partials, grid, n_el, sums);
    GSL_LAUNCH_CHECK("kmeans_reduce_kernel");
    return GSL_OK;
}

extern "C" size_t gsl_kmeans_exchange_bytes(int world, int D, int K)
{
    if (world < 1 || world > kMaxRanks || D < 1 || K < 1) return 0;
    return kXchgSlots + 2 * (size_t)world * (size_t)K * (D + 1) * sizeof(double);
}

extern "C" int gsl_kmeans_step_exchange(const float *data, int64_t N, int D, const float *centroids, int K,
                                        int32_t *labels, int rank, int world, void *const *xbufs, uint64_t seq,
                                        float *new_centroids, float *shift, double *sums,
                                        void *ws, size_t ws_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = check_kd("gsl_kmeans_step_exchange", N, D, K)) return rc;
    if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(GSL_EINVAL, "gsl_kmeans_step_exchange: rank %d / world %d (at most %d ranks)", rank, world, kMaxRanks);
    if (!centroids || !sums || !xbufs || !new_centroids || !shift || seq == 0) return fail(GSL_EINVAL, "gsl_kmeans_step_exchange: null pointer or seq == 0");
    PeerTable peers;
    for (int p = 0; p < kMaxRanks; ++p) {
        peers.base[p] = p < world ? reinterpret_cast<unsigned char *>(xbufs[p]) : nullptr;
        if (p < world && (!xbufs[p] || ((uintptr_t)xbufs[p] & 255))) return fail(GSL_EINVAL, "gsl_kmeans_step_exchange: exchange buffer %d is null or not 256-byte aligned", p);
    }
    const int n_el = K * (D + 1);
    double *partials = nullptr;
    int grid = 0;
    if (N > 0) {
        if (!data || !labels || !ws) return fail(GSL_EINVAL, "gsl_kmeans_step_exchange: null pointer");
        if (ws_bytes < gsl_kmeans_workspace_bytes(N, D, K)) return fail(GSL_EWORKSPACE, "gsl_kmeans_step_exchange: workspace %zu < %zu", ws_bytes, gsl_kmeans_workspace_bytes(N, D, K));
        partials = reinterpret_cast<double *>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
        grid = step_grid(N);
        if (int rc = launch_step<true>(data, N, D, centroids, K, labels, partials, grid, st)) return rc;
    }
    // how long a rank waits inside the kernel for its peers (milliseconds)
    const char *tmo = getenv("GSLIFT_EXCHANGE_TIMEOUT_MS");
    const unsigned long long timeout_ns = (unsigned long long)((tmo && atof(tmo) > 0 ? atof(tmo) : 30000.0) * 1e6);
    kmeans_exchange_kernel<<<(n_el + 31) / 32, kReduceThreads, 0, st>>>(partials, grid, n_el, peers, rank, world, (unsigned long long)seq,
                                                              timeout_ns, centroids, K, D, new_centroids, shift, sums);
    GSL_LAUNCH_CHECK("kmeans_exchange_kernel");
    return GSL_OK;
}

extern "C" int gsl_kmeans_finalize(const double *sums, const float *old_centroids, int K, int D,
                                   float *new_centroids, float *shift, void *stream)
{
    if (int rc = check_kd("gsl_kmeans_finalize", 0, D, K)) return rc;
    if (!sums || !old_centroids || !new_centroids || !shift) return fail(GSL_EINVAL, "gsl_kmeans_finalize: null pointer");
    kmeans_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(sums, old_centroids, K, D, new_centroids, shift);
    GSL_LAUNCH_CHECK("kmeans_finalize_kernel");
    return GSL_OK;
}

extern "C" int gsl_recolor(const int32_t *labels, int64_t N, const float *palette, float *colors, void *stream)
{
    if (N < 0) return fail(GSL_EINVAL, "gsl_recolor: negative N");
    if (N == 0) return GSL_OK;
    if (!labels || !colors || !palette) return fail(GSL_EINVAL, "gsl_recolor: null pointer");
    recolor_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(labels, N, palette, colors);
    GSL_LAUNCH_CHECK("recolor_kernel");
    return GSL_OK;
}
