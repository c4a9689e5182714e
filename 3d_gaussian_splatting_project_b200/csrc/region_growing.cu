// Normals and residuals of the reference's other clustering script (SURVEY.md section 8f, N4;
// 3D_clustering/region_growing.py, `rg` below):
//
//   compute_normals    rg:78-127   per point: k nearest neighbours (scipy KDTree, k = 2000 in
//                                  __main__), centroid, 3x3 covariance of the centred neighbours,
//                                  eigenvector of the smallest eigenvalue, oriented so that
//                                  dot(normal, point - centroid) <= 0, normalised
//   compute_residuals  rg:130-163  |dot(normal_i, point_i - centroid_i)|
//   segmentation_3D    rg:166-221  serial region growing over k = 10 neighbour lists (host side,
//                                  gsl_region_grow below; the neighbour lists come from the GPU)
//
// The neighbour SET is exact: float64 squared distances in scipy's summation order
// (((dx*dx) + dy*dy) + dz*dz, no FMA), the k smallest by (distance, index).  scipy breaks exact
// distance ties at the k-th neighbour by tree layout; here the lower index wins (documented
// exemption, as for the K-means ties).  Centroid and covariance are accumulated in float64 around
// the query point (the reference: float32 sequential mean, float32 sgemm, LAPACK ssyevr -- not
// reproducible bit for bit; tests state the tolerance), the eigenvector comes from cyclic Jacobi
// rotations in float64.
//
// Search structure: points sorted by a 21-bit Morton code on a 128^3 grid of cubic cells over the
// bounding box; every coarser level's cells are prefixes of that code, so ONE sorted array serves
// grids of 2^L cells per axis, L = 1..7, each with a dense cell-start table.  A warp owns a query:
// it looks for the finest (level, ring) whose cube of (2*ring+1)^3 cells provably contains the k
// nearest neighbours (at least k points within ring * cell_size of the query), then selects the
// k-th smallest squared distance by a 10-bit-per-walk radix select over the float64 bit
// patterns, rebased so that the leading digit resolves [R^2 / 1024, R^2] (per-warp histogram in
// shared memory; the first digit is counted by the walk that validates the cube), and accumulates
// the moments of the selected points.  Each step is a walk over the cube's non-empty cell ranges, kept in shared memory.
#include <float.h>
#include <math.h>
#include <math_constants.h>

#include <algorithm>
#include <deque>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "radix_sort.cuh"

namespace gsl {
namespace rg {

constexpr int kLevels = 7;                 // finest grid: 128 cells per axis
constexpr int kFinest = 1 << kLevels;
constexpr int kDigitBits = 10;
constexpr int kDigits = 1 << kDigitBits;
constexpr int kWarps = 8;
constexpr int kMaxRanges = 343;            // (2 * 3 + 1)^3 cells
constexpr int kMaxList = 64;               // lists of k <= 64 are ordered inside knn_pca_kernel, longer ones by knn_order_kernel
constexpr int kBucketCap = 256;            // candidates of the k-th value's histogram bucket resolved in shared memory

struct BucketEntry {                       // 16 bytes: kBucketCap of them reuse the 4 KB of the histogram
    double d2;
    uint32_t pos;                          // position in the sorted array
    uint32_t idx;                          // original index
};
static_assert(sizeof(BucketEntry) * kBucketCap <= sizeof(uint32_t) * kDigits, "bucket list aliases the histogram");

struct GridInfo {            // device-resident, written by bbox_final_kernel, refined by grid_box_kernel
    double lo[3];            // low corner of the grid
    double h7;               // side of a finest cell
    double inv_h7;
    double full_lo[3], full_hi[3];     // bounding box of the points
};

constexpr int kBoxBins = 1024;          // coordinate histogram bins per axis

struct Tables {
    const uint32_t *start[kLevels + 1];    // [L] : 8^L + 1 entries, L = 1..7
};

__host__ __device__ inline size_t table_entries(int L) { return ((size_t)1 << (3 * L)) + 1; }

__device__ __forceinline__ uint32_t spread3(uint32_t v)
{
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__device__ __forceinline__ uint32_t morton3(uint32_t x, uint32_t y, uint32_t z)
{
    return spread3(x) | (spread3(y) << 1) | (spread3(z) << 2);
}
__device__ __forceinline__ int cell_coord(double p, double lo, double inv_h)
{
    const double c = floor(__dmul_rn(__dsub_rn(p, lo), inv_h));
    return (int)fmin(fmax(c, 0.0), (double)(kFinest - 1));
}

// ---- bounding box -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bbox_kernel(const float *__restrict__ pos, int64_t N, float *__restrict__ part)
{
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = pos[3 * i + a];
            lo[a] = fminf(lo[a], v);
            hi[a] = fmaxf(hi[a], v);
        }
    __shared__ float s[8][6];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if ((threadIdx.x & 31) == 0) {
            s[threadIdx.x >> 5][a] = lo[a];
            s[threadIdx.x >> 5][3 + a] = hi[a];
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float v = s[0][threadIdx.x];
        for (int w = 1; w < 8; ++w) v = threadIdx.x < 3 ? fminf(v, s[w][threadIdx.x]) : fmaxf(v, s[w][threadIdx.x]);
        part[blockIdx.x * 6 + threadIdx.x] = v;
    }
}

__global__ void __launch_bounds__(256) bbox_final_kernel(const float *__restrict__ part, int n, GridInfo *__restrict__ g)
{
    __shared__ float s[8][6];
    float v[6];
#pragma unroll
    for (int a = 0; a < 6; ++a) v[a] = a < 3 ? FLT_MAX : -FLT_MAX;
    for (int b = threadIdx.x; b < n; b += 256)
#pragma unroll
        for (int a = 0; a < 6; ++a) v[a] = a < 3 ? fminf(v[a], part[b * 6 + a]) : fmaxf(v[a], part[b * 6 + a]);
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const float t = __shfl_xor_sync(0xffffffffu, v[a], o);
            v[a] = a < 3 ? fminf(v[a], t) : fmaxf(v[a], t);
        }
        if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5][a] = v[a];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    float lo[3], hi[3];
    for (int a = 0; a < 3; ++a) {
        lo[a] = s[0][a];
        hi[a] = s[0][3 + a];
        for (int w = 1; w < 8; ++w) {
            lo[a] = fminf(lo[a], s[w][a]);
            hi[a] = fmaxf(hi[a], s[w][3 + a]);
        }
    }
    double side = 0;
    for (int a = 0; a < 3; ++a) side = fmax(side, (double)hi[a] - (double)lo[a]);
    if (!(side > 0)) side = 1.0;                       // all points coincide
    side *= 1.0 + 1e-6;
    for (int a = 0; a < 3; ++a) {
        g->lo[a] = (double)lo[a];
        g->full_lo[a] = (double)lo[a];
        g->full_hi[a] = (double)hi[a];
    }
    g->h7 = side / kFinest;
    g->inv_h7 = kFinest / side;
}

// The grid should resolve where the points ARE: a few far outliers (floaters are common in splat
// clouds) would otherwise stretch the 128^3 cells until the whole scene sits in a handful of them and
// every query walks nearly everything.  So the grid covers, per axis, the 0.5 % .. 99.5 % quantile
// range (from a 1024-bin histogram over the bounding box) and points outside it are assigned to the
// border cells.  That keeps the search exact: clamping a coordinate into the grid's box is
// order preserving and non-expansive, so two points whose cells differ by more than `ring` along an
// axis are at least ring * cell_size apart along that axis, clamped or not.
__global__ void __launch_bounds__(256) coord_hist_kernel(const float *__restrict__ pos, int64_t N, const GridInfo *__restrict__ g,
                                                         unsigned *__restrict__ hist)
{
    __shared__ unsigned sh[3][kBoxBins];
    for (int i = threadIdx.x; i < 3 * kBoxBins; i += 256) (&sh[0][0])[i] = 0u;
    __syncthreads();
    double lo[3], scale[3];
    for (int a = 0; a < 3; ++a) {
        lo[a] = g->full_lo[a];
        const double ext = g->full_hi[a] - lo[a];
        scale[a] = ext > 0 ? kBoxBins / ext : 0.0;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int b = min(kBoxBins - 1, max(0, (int)(((double)pos[3 * i + a] - lo[a]) * scale[a])));
            atomicAdd(&sh[a][b], 1u);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * kBoxBins; i += 256) {
        const unsigned c = (&sh[0][0])[i];
        if (c) atomicAdd(&hist[i], c);
    }
}

__global__ void grid_box_kernel(const unsigned *__restrict__ hist, int64_t N, GridInfo *__restrict__ g)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long cut = (unsigned long long)(N / 200);           // 0.5 % of the points on either side
    double lo[3], hi[3], side = 0;
    for (int a = 0; a < 3; ++a) {
        const double ext = g->full_hi[a] - g->full_lo[a], w = ext / kBoxBins;
        unsigned long long run = 0;
        int b0 = 0, b1 = kBoxBins - 1;
        for (int b = 0; b < kBoxBins; ++b) {
            run += hist[a * kBoxBins + b];
            if (run > cut) { b0 = b; break; }
        }
        run = 0;
        for (int b = kBoxBins - 1; b >= 0; --b) {
            run += hist[a * kBoxBins + b];
            if (run > cut) { b1 = b; break; }
        }
        if (b1 < b0) b1 = b0;
        lo[a] = g->full_lo[a] + b0 * w;                                       // left edge of the first kept bin
        hi[a] = g->full_lo[a] + (b1 + 1) * w;                                 // right edge of the last one
        side = fmax(side, hi[a] - lo[a]);
    }
    if (!(side > 0)) side = 1.0;
    side *= 1.0 + 1e-6;
    for (int a = 0; a < 3; ++a) g->lo[a] = lo[a];
    g->h7 = side / kFinest;
    g->inv_h7 = kFinest / side;
}

__global__ void __launch_bounds__(256) cell_key_kernel(const float *__restrict__ pos, int64_t N, const GridInfo *__restrict__ g,
                                                       uint32_t *__restrict__ keys)
{
    const GridInfo G = *g;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const int cx = cell_coord((double)pos[3 * i], G.lo[0], G.inv_h7), cy = cell_coord((double)pos[3 * i + 1], G.lo[1], G.inv_h7),
                  cz = cell_coord((double)pos[3 * i + 2], G.lo[2], G.inv_h7);
        keys[i] = morton3(cx, cy, cz);
    }
}

__global__ void __launch_bounds__(256) gather_sorted_kernel(const float *__restrict__ pos, const uint32_t *__restrict__ order,
                                                            int64_t N, float4 *__restrict__ sorted)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t j = order[i];
        sorted[i] = make_float4(pos[3 * (size_t)j], pos[3 * (size_t)j + 1], pos[3 * (size_t)j + 2], __uint_as_float(j));
    }
}

// start_L[c] = number of sorted keys whose level-L prefix is below c (lower bound).
__global__ void __launch_bounds__(256) cell_start_kernel(const uint32_t *__restrict__ keys, int64_t N, int L,
                                                         uint32_t *__restrict__ start)
{
    const size_t n = table_entries(L);
    const int sh = 3 * (kLevels - L);
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (size_t)gridDim.x * blockDim.x) {
        int64_t a = 0, b = N;
        while (a < b) {
            const int64_t m = (a + b) >> 1;
            if ((size_t)(keys[m] >> sh) < c) a = m + 1;
            else b = m;
        }
        start[c] = (uint32_t)a;
    }
}

// ---- per-query search ---------------------------------------------------------------------------
struct QueryOut {
    double *normals;           // [N][3] out, may be NULL
    const double *normals_in;  // [N][3] normals for the residual, may be NULL (then the computed one)
    double *residuals;         // [N] out, may be NULL
    double *centroids;         // [N][3] out, may be NULL
    int32_t *knn;              // [N][k] out, k <= GSL_REGION_MAX_LIST, may be NULL
};

struct WarpScratch {
    uint32_t hist[kDigits];
    uint32_t end[kMaxRanges + 1];      // end[r] = points in ranges 0..r (inclusive prefix of the range lengths)
    uint32_t off[kMaxRanges + 1];      // off[r] = start of range r in the sorted array - points before range r
    double list_d[kMaxList];
    uint32_t list_i[kMaxList];
};

__device__ __forceinline__ double sqdist(const float4 p, double qx, double qy, double qz)
{
    const double dx = __dsub_rn((double)p.x, qx), dy = __dsub_rn((double)p.y, qy), dz = __dsub_rn((double)p.z, qz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// Non-empty cell ranges of the cube of `ring` cells around (cx, cy, cz) at level L, as a flat index
// space: candidate v (0 <= v < total) is sorted[off[r] + v] for the r with end[r - 1] <= v < end[r].
// Returns the number of ranges; *total = points in the cube.  L == 0: the whole array.
__device__ int build_ranges(const Tables &T, int64_t N, int L, int ring, int cx, int cy, int cz, WarpScratch &sc,
                            unsigned lane, int64_t *total)
{
    if (L == 0) {
        if (lane == 0) {
            sc.end[0] = (uint32_t)N;
            sc.off[0] = 0u;
        }
        __syncwarp();
        *total = N;
        return 1;
    }
    const int n = 1 << L;
    const int x0 = max(cx - ring, 0), x1 = min(cx + ring, n - 1), y0 = max(cy - ring, 0), y1 = min(cy + ring, n - 1),
              z0 = max(cz - ring, 0), z1 = min(cz + ring, n - 1);
    const int nx = x1 - x0 + 1, ny = y1 - y0 + 1, ncell = nx * ny * (z1 - z0 + 1);
    const uint32_t *start = T.start[L];
    int cnt = 0;
    uint32_t tot = 0;
    for (int base = 0; base < ncell; base += 32) {
        const int id = base + (int)lane;
        uint32_t s = 0, e = 0;
        if (id < ncell) {
            const int ix = id % nx, iy = (id / nx) % ny, iz = id / (nx * ny);
            const uint32_t c = morton3(x0 + ix, y0 + iy, z0 + iz);
            s = start[c];
            e = start[c + 1];
        }
        const uint32_t len = e - s;
        uint32_t inc = len;                       // inclusive prefix of the lengths over the lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (unsigned)o) inc += t;
        }
        const unsigned full = __ballot_sync(0xffffffffu, len != 0);
        if (len != 0) {
            const int at = cnt + __popc(full & radix::lanemask_lt());
            sc.end[at] = tot + inc;
            sc.off[at] = s - (tot + inc - len);
        }
        cnt += __popc(full);
        tot += __shfl_sync(0xffffffffu, inc, 31);
    }
    __syncwarp();
    *total = tot;
    return cnt;
}

// Calls f(valid, point, position in the sorted array) for every point of the ranges, all 32 lanes in lockstep and all lanes busy: lane l
// takes candidates l, l + 32, ... of the flat index space and advances its own range cursor.
template <class F>
__device__ __forceinline__ void walk(const float4 *__restrict__ sorted, const WarpScratch &sc, uint32_t total, unsigned lane, F f)
{
    if (total == 0) return;
    constexpr int U = 4;                    // independent loads in flight per lane
    int r = 0;
    uint32_t r_end = sc.end[0], off = sc.off[0];
    for (uint32_t v0 = 0; v0 < total; v0 += 32 * U) {
        float4 p[U];
        uint32_t at[U];
        bool valid[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t v = v0 + 32 * u + lane;
            valid[u] = v < total;
            const uint32_t vv = valid[u] ? v : total - 1;
            while (vv >= r_end) {
                ++r;
                r_end = sc.end[r];
                off = sc.off[r];
            }
            at[u] = off + vv;
            p[u] = __ldg(sorted + at[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (v0 + 32 * u < total) f(valid[u], p[u], at[u]);      // warp-uniform condition
    }
}

// Smallest-eigenvalue eigenvector of the symmetric 3x3 matrix (a00 a01 a02 / a11 a12 / a22), cyclic Jacobi.
__device__ void smallest_eigenvector(double a00, double a01, double a02, double a11, double a12, double a22, double v[3])
{
    double A[3][3] = {{a00, a01, a02}, {a01, a11, a12}, {a02, a12, a22}};
    double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
        const double diag = fabs(A[0][0]) + fabs(A[1][1]) + fabs(A[2][2]);
        if (off <= 1e-300 || off <= 1e-17 * diag) break;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            const double apq = A[p][q];
            if (apq == 0.0) continue;
            const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
            const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
            for (int k = 0; k < 3; ++k) {          // A <- A J
                const double akp = A[k][p], akq = A[k][q];
                A[k][p] = c * akp - s * akq;
                A[k][q] = s * akp + c * akq;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {          // A <- J^T A
                const double apk = A[p][k], aqk = A[q][k];
                A[p][k] = c * apk - s * aqk;
                A[q][k] = s * apk + c * aqk;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double vkp = V[k][p], vkq = V[k][q];
                V[k][p] = c * vkp - s * vkq;
                V[k][q] = s * vkp + c * vkq;
            }
        }
    }
    int m = 0;
    if (A[1][1] < A[m][m]) m = 1;
    if (A[2][2] < A[m][m]) m = 2;
    v[0] = V[0][m];
    v[1] = V[1][m];
    v[2] = V[2][m];
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// kLongList: the caller asked for lists of k > 64, written straight out in walk order (a separate
// instantiation, so that the other calls run the code they always ran)
template <bool kLongList>
__global__ void __launch_bounds__(kWarps * 32, 3) knn_pca_kernel(const float4 *__restrict__ sorted, int64_t N, int k,
                                                              const GridInfo *__restrict__ ginfo, Tables T, QueryOut out,
                                                              unsigned long long *__restrict__ stats)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpScratch &sc = reinterpret_cast<WarpScratch *>(smem_raw)[threadIdx.x >> 5];
    const unsigned lane = threadIdx.x & 31u;
    const GridInfo G = *ginfo;
    const int64_t n_warps = (int64_t)gridDim.x * kWarps;
    for (int64_t qi = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); qi < N; qi += n_warps) {
        const float4 q4 = sorted[qi];
        const double qx = q4.x, qy = q4.y, qz = q4.z;
        const uint32_t q_index = __float_as_uint(q4.w);
        const int c7x = cell_coord(qx, G.lo[0], G.inv_h7), c7y = cell_coord(qy, G.lo[1], G.inv_h7),
                  c7z = cell_coord(qz, G.lo[2], G.inv_h7);

        // Key of a squared distance: its float64 bit pattern (monotone for d2 >= 0), clamped from below at
        // `floor_bits` and rebased there.  With floor = R2 / 1024 the leading 10-bit digit resolves the range
        // [R2 / 1024, R2], where the k-th distance almost always lies, into ~640 bins (64 per binade) instead of
        // spending a walk on the exponent field; the histogram's atomics then rarely collide.
        unsigned long long floor_bits = 0;
        int top_shift = 54;                 // raw keys (floor_bits == 0) are below 2^63: leading digit = bits 63..54
        auto key_of = [&](double d2) -> unsigned long long {
            const unsigned long long b = (unsigned long long)__double_as_longlong(d2);
            return (b > floor_bits ? b : floor_bits) - floor_bits;
        };
        unsigned long long n_walks = 0, n_walked = 0, n_failed = 0, n_select = 0;

        // 1. the finest cube that provably holds the k nearest neighbours; the counting walk also fills the
        //    histogram of the leading digit
        int64_t in_cube = 0;
        double R2 = CUDART_INF;
        bool have_hist = false;
        for (int L = kLevels; L >= 0; --L) {
            bool found = false;
            for (int ring = (L == kLevels ? 1 : 2); ring <= 3; ++ring) {
                build_ranges(T, N, L, ring, c7x >> (kLevels - L), c7y >> (kLevels - L), c7z >> (kLevels - L), sc, lane,
                                        &in_cube);
                if (L == 0) {
                    R2 = CUDART_INF;
                    floor_bits = 0;
                    top_shift = 54;
                    found = true;
                    break;
                }
                // a ball of `ring` cells fills 0.155 / 0.27 / 0.33 of its cube: do not walk a cube whose points would
                // have to be 25 % denser inside the ball than outside to reach k (a walk that fails is wasted)
                const double fill = ring == 1 ? 0.155 : (ring == 2 ? 0.268 : 0.329);
                if ((double)in_cube * fill * 1.25 < (double)k) continue;
                // every point outside the cube is farther than ring cells of this level
                const double rad = (double)ring * G.h7 * (double)(1 << (kLevels - L)) * (1.0 - 1e-9);
                R2 = rad * rad;
                const unsigned long long r2_bits = (unsigned long long)__double_as_longlong(R2);
                const bool clamp = r2_bits > (11ull << 52);
                floor_bits = clamp ? r2_bits - (10ull << 52) : 0ull;          // bits of R2 / 1024
                top_shift = clamp ? 46 : 54;                                   // clamped keys are <= 10 * 2^52 < 2^56
                for (int d = lane; d < kDigits; d += 32) sc.hist[d] = 0;
                __syncwarp();
                int inside = 0;
                walk(sorted, sc, (uint32_t)in_cube, lane, [&](bool valid, const float4 p, uint32_t) {
                    const double d2 = sqdist(p, qx, qy, qz);
                    if (valid && d2 <= R2) {
                        ++inside;
                        atomicAdd(&sc.hist[(unsigned)(key_of(d2) >> top_shift)], 1u);
                    }
                });
                ++n_walks;
                n_walked += (unsigned long long)in_cube;
#pragma unroll
                for (int o = 16; o; o >>= 1) inside += __shfl_xor_sync(0xffffffffu, inside, o);
                __syncwarp();
                if (inside >= k) {
                    have_hist = true;
                    found = true;
                    break;
                }
                ++n_failed;
            }
            if (found) break;
        }

        // 2. radix select of the k-th smallest key among the points within R2, 10 bits per walk
        unsigned long long prefix = 0;      // the digits chosen so far = key >> shift
        int shift = top_shift + kDigitBits, need = k;
        bool exact = false;                 // every key with (key >> shift) <= prefix is selected
        bool use_list = false;              // the bucket of the k-th value is small: resolved from a list in shared memory
        bool first = true;
        while (shift > 0 && !exact) {
            const int bits = shift >= kDigitBits ? kDigitBits : shift;
            const int new_shift = shift - bits;
            if (!(first && have_hist)) {
                for (int d = lane; d < kDigits; d += 32) sc.hist[d] = 0;
                __syncwarp();
                walk(sorted, sc, (uint32_t)in_cube, lane, [&](bool valid, const float4 p, uint32_t) {
                    const double d2 = sqdist(p, qx, qy, qz);
                    const unsigned long long key = key_of(d2);
                    if (valid && d2 <= R2 && (first || (key >> shift) == prefix))
                        atomicAdd(&sc.hist[(unsigned)(key >> new_shift) & ((1u << bits) - 1u)], 1u);
                });
                ++n_walks;
                ++n_select;
                n_walked += (unsigned long long)in_cube;
                __syncwarp();
            }
            // locate the digit holding the need-th smallest: lane l owns bins [32 l, 32 l + 32)
            constexpr int kPerLane = kDigits / 32;
            uint32_t mine = 0;
            for (int d = 0; d < kPerLane; ++d) mine += sc.hist[lane * kPerLane + d];
            uint32_t inc = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= (unsigned)o) inc += t;
            }
            const unsigned has = __ballot_sync(0xffffffffu, inc >= (uint32_t)need);
            const int owner = __ffs(has) - 1;            // has != 0: at least `need` points are within R2
            int digit = 0, below = 0, bucket = 0;
            if ((int)lane == owner) {
                uint32_t run = inc - mine;
                for (int d = 0; d < kPerLane; ++d) {
                    const uint32_t h = sc.hist[lane * kPerLane + d];
                    if (run + h >= (uint32_t)need) {
                        digit = lane * kPerLane + d;
                        below = run;
                        bucket = h;
                        break;
                    }
                    run += h;
                }
            }
            digit = __shfl_sync(0xffffffffu, digit, owner);
            below = __shfl_sync(0xffffffffu, below, owner);
            bucket = __shfl_sync(0xffffffffu, bucket, owner);
            __syncwarp();
            if (first && floor_bits != 0 && digit == 0) {
                // the k-th distance is below the clamp (tiny k): select again on the raw bit patterns
                floor_bits = 0;
                top_shift = 54;
                shift = top_shift + kDigitBits;
                have_hist = false;
                continue;
            }
            need -= below;
            prefix = (prefix << bits) | (unsigned long long)digit;
            shift = new_shift;
            exact = need == bucket;
            first = false;
            if (!exact && bucket <= kBucketCap) {
                use_list = true;            // the next walk collects the bucket and sums everything below it
                break;
            }
        }
        // here: keys with (key >> shift) < prefix are all selected; of those equal to prefix, `need` are
        // (all of them when `exact`; otherwise shift == 0 and they are exact ties: lowest indices win)

        // 3. moments of the selected neighbours around the query
        double s1[3] = {0, 0, 0}, s2[6] = {0, 0, 0, 0, 0, 0};
        int n_list = 0;
        const bool want_list = out.knn != nullptr;
        constexpr bool emit = kLongList;                  // k > 64: the list goes out in walk order, knn_order_kernel sorts it
        auto take = [&](bool sel, const float4 p, double d2) {
            if (sel) {
                const double dx = __dsub_rn((double)p.x, qx), dy = __dsub_rn((double)p.y, qy), dz = __dsub_rn((double)p.z, qz);
                s1[0] += dx; s1[1] += dy; s1[2] += dz;
                s2[0] += dx * dx; s2[1] += dx * dy; s2[2] += dx * dz;
                s2[3] += dy * dy; s2[4] += dy * dz; s2[5] += dz * dz;
            }
            if (want_list) {
                const unsigned m = __ballot_sync(0xffffffffu, sel);
                if (sel) {
                    const int at = n_list + __popc(m & radix::lanemask_lt());
                    if (emit) {
                        if (at < k) out.knn[(size_t)q_index * k + at] = (int32_t)__float_as_uint(p.w);
                    } else if (at < kMaxList) {
                        sc.list_d[at] = d2;
                        sc.list_i[at] = __float_as_uint(p.w);
                    }
                }
                n_list += __popc(m);
            }
        };
        BucketEntry *blist = reinterpret_cast<BucketEntry *>(sc.hist);        // the histogram is not needed any more
        int n_bucket = 0;
        __syncwarp();
        walk(sorted, sc, (uint32_t)in_cube, lane, [&](bool valid, const float4 p, uint32_t at) {
            const double d2 = sqdist(p, qx, qy, qz);
            const unsigned long long key = key_of(d2) >> shift;
            const bool in_ball = valid && d2 <= R2;
            const bool sel = in_ball && (exact ? key <= prefix : key < prefix);
            take(sel, p, d2);
            if (use_list) {
                const bool mine = in_ball && key == prefix;
                const unsigned m = __ballot_sync(0xffffffffu, mine);
                if (mine) {
                    const int slot = n_bucket + __popc(m & radix::lanemask_lt());
                    if (slot < kBucketCap) blist[slot] = BucketEntry{d2, at, __float_as_uint(p.w)};
                }
                n_bucket += __popc(m);
            }
        });
        ++n_walks;
        n_walked += (unsigned long long)in_cube;
        if (use_list) {
            // the `need` smallest of the bucket by (distance, index): rank by counting, 32 entries at a time
            __syncwarp();
            const int nb = min(n_bucket, kBucketCap);
            for (int a0 = 0; a0 < nb; a0 += 32) {
                const int a = a0 + (int)lane;
                bool sel = false;
                float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
                double d2 = 0.0;
                if (a < nb) {
                    const BucketEntry e = blist[a];
                    int rank = 0;
                    for (int b = 0; b < nb; ++b) {
                        const BucketEntry o = blist[b];
                        rank += (o.d2 < e.d2 || (o.d2 == e.d2 && o.idx < e.idx)) ? 1 : 0;
                    }
                    sel = rank < need;
                    d2 = e.d2;
                    if (sel) p = __ldg(sorted + e.pos);
                }
                take(sel, p, d2);
            }
        }
        if (!exact && !use_list) {
            // exact ties at the k-th distance (a bucket too large for the list that stayed tied through every digit): take the `need` lowest original indices among them
            long long last = -1;
            for (int t = 0; t < need; ++t) {
                unsigned long long best = ~0ull;      // (index << 32) | sorted position is not needed: index is unique
                float4 bp = make_float4(0.f, 0.f, 0.f, 0.f);
                walk(sorted, sc, (uint32_t)in_cube, lane, [&](bool valid, const float4 p, uint32_t) {
                    const double d2 = sqdist(p, qx, qy, qz);
                    const unsigned long long key = key_of(d2);
                    const long long idx = (long long)__float_as_uint(p.w);
                    if (valid && d2 <= R2 && key == prefix && idx > last && (unsigned long long)idx < best) {
                        best = (unsigned long long)idx;
                        bp = p;
                    }
                });
                unsigned long long wbest = best;
#pragma unroll
                for (int o = 16; o; o >>= 1) wbest = min(wbest, __shfl_xor_sync(0xffffffffu, wbest, o));
                take(best == wbest && best != ~0ull, bp, __longlong_as_double((long long)(prefix + floor_bits)));
                ++n_walks;
                n_walked += (unsigned long long)in_cube;
                last = (long long)wbest;
            }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) s1[a] = warp_sum(s1[a]);
#pragma unroll
        for (int a = 0; a < 6; ++a) s2[a] = warp_sum(s2[a]);

        // 4. centroid, covariance, normal, residual (every lane holds the same sums)
        const double inv_k = 1.0 / (double)k;
        const double mx = s1[0] * inv_k, my = s1[1] * inv_k, mz = s1[2] * inv_k;      // centroid - query
        double nrm[3] = {0, 0, 0};
        if (out.normals) {
            smallest_eigenvector(s2[0] - s1[0] * mx, s2[1] - s1[0] * my, s2[2] - s1[0] * mz, s2[3] - s1[1] * my,
                                 s2[4] - s1[1] * mz, s2[5] - s1[2] * mz, nrm);
            // rg:118-119: flip when dot(normal, pos - centroid) > 0; pos - centroid = -(mx, my, mz)
            const double dot = -(nrm[0] * mx + nrm[1] * my + nrm[2] * mz);
            if (dot > 0) {
                nrm[0] = -nrm[0]; nrm[1] = -nrm[1]; nrm[2] = -nrm[2];
            }
            const double len = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1] + nrm[2] * nrm[2]);     // rg:124
            nrm[0] /= len; nrm[1] /= len; nrm[2] /= len;
            if (lane < 3) out.normals[3 * (size_t)q_index + lane] = nrm[lane];
        }
        if (out.centroids && lane < 3) out.centroids[3 * (size_t)q_index + lane] = (lane == 0 ? qx + mx : lane == 1 ? qy + my : qz + mz);
        if (out.residuals) {
            if (out.normals_in) {
                nrm[0] = out.normals_in[3 * (size_t)q_index];
                nrm[1] = out.normals_in[3 * (size_t)q_index + 1];
                nrm[2] = out.normals_in[3 * (size_t)q_index + 2];
            }
            if (lane == 0) out.residuals[q_index] = fabs(-(nrm[0] * mx + nrm[1] * my + nrm[2] * mz));    // rg:161
        }
        if (want_list && !emit) {
            // order the k <= 64 selected neighbours by (distance, index): rank sort in shared memory
            __syncwarp();
            const int n = min(n_list, kMaxList);
            for (int a = lane; a < n; a += 32) {
                const double da = sc.list_d[a];
                const uint32_t ia = sc.list_i[a];
                int rank = 0;
                for (int b = 0; b < n; ++b) {
                    const double db = sc.list_d[b];
                    rank += (db < da || (db == da && sc.list_i[b] < ia)) ? 1 : 0;
                }
                out.knn[(size_t)q_index * k + rank] = (int32_t)ia;
            }
            __syncwarp();
        }
        if (stats && lane == 0) {
            atomicAdd(&stats[0], n_walks);
            atomicAdd(&stats[1], n_walked);
            atomicAdd(&stats[2], n_failed);
            atomicAdd(&stats[3], n_select);
        }
    }
}

// Lists of k > 64 leave knn_pca_kernel in walk order.  This kernel puts every row into increasing
// (distance, index) order, KDTree.query's: the key of a neighbour is the float64 bit pattern of its
// squared distance (recomputed from pos with the selector's own sqdist, monotone for d2 >= 0) and its
// index, so keys are unique and the order is a total one.  A row's keys, padded to a power of two P
// with +inf sentinels, are bitonic-sorted in shared memory; rows of small k share a CTA.
constexpr int kOrderThreads = 256;
constexpr int kOrderMinKeys = 2048;        // keys per CTA: rows of P < 2048 share one
constexpr int kOrderKeyBytes = 12;         // 8-byte distance bits + 4-byte index
static_assert((size_t)GSL_REGION_MAX_LIST * kOrderKeyBytes <= 227 * 1024, "a row of keys fits one CTA's shared memory");

__global__ void __launch_bounds__(kOrderThreads) knn_order_kernel(const float *__restrict__ pos, int64_t N, int k, int log_p,
                                                                  int rows_per_cta, int32_t *__restrict__ knn)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int P = 1 << log_p, keys = P * rows_per_cta;
    unsigned long long *kd = reinterpret_cast<unsigned long long *>(smem_raw);
    uint32_t *ki = reinterpret_cast<uint32_t *>(kd + keys);
    const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
    for (int t = threadIdx.x; t < keys; t += kOrderThreads) {
        const int64_t row = row0 + (t >> log_p);
        const int i = t & (P - 1);
        unsigned long long d = 0x7ff0000000000000ull;          // +inf: every real d2 of finite float32 points is finite
        uint32_t j = 0xffffffffu;
        if (row < N && i < k) {
            j = (uint32_t)knn[(size_t)row * k + i];
            const float4 p = make_float4(pos[3 * (size_t)j], pos[3 * (size_t)j + 1], pos[3 * (size_t)j + 2], 0.f);
            d = (unsigned long long)__double_as_longlong(
                sqdist(p, (double)pos[3 * (size_t)row], (double)pos[3 * (size_t)row + 1], (double)pos[3 * (size_t)row + 2]));
        }
        kd[t] = d;
        ki[t] = j;
    }
    const int half = keys >> 1;
    for (int size = 2; size <= P; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < half; t += kOrderThreads) {
                // pair t: rows hold P / 2 pairs each; within a row, a = the lower element of the pair
                const int r = t >> (log_p - 1), i = t & ((P >> 1) - 1);
                const int a = ((i & ~(stride - 1)) << 1) | (i & (stride - 1));
                const int ga = (r << log_p) + a, gb = ga + stride;
                const unsigned long long da = kd[ga], db = kd[gb];
                const uint32_t ia = ki[ga], ib = ki[gb];
                const bool a_after_b = da > db || (da == db && ia > ib);
                if (a_after_b == ((a & size) == 0)) {          // ascending runs where bit `size` of a is clear
                    kd[ga] = db; kd[gb] = da;
                    ki[ga] = ib; ki[gb] = ia;
                }
            }
        }
    __syncthreads();
    for (int t = threadIdx.x; t < keys; t += kOrderThreads) {
        const int64_t row = row0 + (t >> log_p);
        const int i = t & (P - 1);
        if (row < N && i < k) knn[(size_t)row * k + i] = (int32_t)ki[t];
    }
}

struct Plan {
    size_t keys_a, keys_b, idx_a, idx_b, hist, sorted, tables[kLevels + 1], ginfo, bbox, chist, total;
};
static Plan plan(int64_t N)
{
    Plan p;
    size_t o = 0;
    const size_t n = (size_t)(N > 0 ? N : 0);
    p.keys_a = o; o = align_up(o + n * 4, 256);
    p.keys_b = o; o = align_up(o + n * 4, 256);
    p.idx_a = o;  o = align_up(o + n * 4, 256);
    p.idx_b = o;  o = align_up(o + n * 4, 256);
    p.hist = o;   o = align_up(o + radix::hist_words(N, 7) * 4, 256);
    p.sorted = o; o = align_up(o + n * 16, 256);
    p.tables[0] = 0;
    for (int L = 1; L <= kLevels; ++L) {
        p.tables[L] = o;
        o = align_up(o + table_entries(L) * 4, 256);
    }
    p.ginfo = o; o = align_up(o + sizeof(GridInfo), 256);
    p.bbox = o;  o = align_up(o + 1024 * 6 * sizeof(float), 256);
    p.chist = o; o = align_up(o + 3 * kBoxBins * sizeof(unsigned), 256);
    p.total = o;
    return p;
}

}  // namespace rg
}  // namespace gsl

using namespace gsl;

extern "C" size_t gsl_region_workspace_bytes(int64_t N) { return rg::plan(N).total; }

extern "C" int gsl_region_knn_pca(const float *pos, int64_t N, int k, const double *normals_in, double *normals,
                                  double *residuals, double *centroids, int32_t *knn, unsigned long long *stats,
                                  void *ws, size_t ws_bytes, void *stream)
{
    if (N < 0 || k < 1 || (N > 0 && (!pos || !ws))) return fail(GSL_EINVAL, "gsl_region_knn_pca: bad argument");
    if (N > 0x7fffffffLL) return fail(GSL_EINVAL, "gsl_region_knn_pca: more than 2^31 - 1 points");
    if (k > N && N > 0) return fail(GSL_EINVAL, "gsl_region_knn_pca: k = %d exceeds the number of points %lld", k, (long long)N);
    if (knn && k > GSL_REGION_MAX_LIST)
        return fail(GSL_EINVAL, "gsl_region_knn_pca: neighbour lists are returned for k <= %d (GSL_REGION_MAX_LIST), k = %d",
                    GSL_REGION_MAX_LIST, k);
    if (N == 0) return GSL_OK;
    const rg::Plan p = rg::plan(N);
    if (ws_bytes < p.total) return fail(GSL_EWORKSPACE, "gsl_region_knn_pca: workspace %zu < %zu", ws_bytes, p.total);
    cudaStream_t st = (cudaStream_t)stream;
    char *w = (char *)ws;
    uint32_t *keys_a = (uint32_t *)(w + p.keys_a), *keys_b = (uint32_t *)(w + p.keys_b), *idx_a = (uint32_t *)(w + p.idx_a),
             *idx_b = (uint32_t *)(w + p.idx_b), *hist = (uint32_t *)(w + p.hist);
    float4 *sorted = (float4 *)(w + p.sorted);
    rg::GridInfo *ginfo = (rg::GridInfo *)(w + p.ginfo);
    float *bbox = (float *)(w + p.bbox);

    const int grid = (int)std::min<int64_t>((N + 255) / 256, 1024);
    rg::bbox_kernel<<<grid, 256, 0, st>>>(pos, N, bbox);
    GSL_LAUNCH_CHECK("rg::bbox_kernel");
    rg::bbox_final_kernel<<<1, 256, 0, st>>>(bbox, grid, ginfo);
    GSL_LAUNCH_CHECK("rg::bbox_final_kernel");
    unsigned *chist = (unsigned *)(w + p.chist);
    GSL_CUDA_TRY(cudaMemsetAsync(chist, 0, 3 * rg::kBoxBins * sizeof(unsigned), st));
    rg::coord_hist_kernel<<<std::min(grid, sm_count() * 4), 256, 0, st>>>(pos, N, ginfo, chist);
    GSL_LAUNCH_CHECK("rg::coord_hist_kernel");
    rg::grid_box_kernel<<<1, 32, 0, st>>>(chist, N, ginfo);
    GSL_LAUNCH_CHECK("rg::grid_box_kernel");
    const int wide = (int)std::min<int64_t>((N + 255) / 256, (int64_t)sm_count() * 8);
    rg::cell_key_kernel<<<wide, 256, 0, st>>>(pos, N, ginfo, keys_a);
    GSL_LAUNCH_CHECK("rg::cell_key_kernel");
    // 21-bit Morton keys: three stable 7-bit passes (a -> b -> a -> b)
    int rc = radix::pass<7>(keys_a, nullptr, keys_b, idx_b, N, 0, hist, 0xffffffffu, 0, st);
    if (rc) return rc;
    rc = radix::pass<7>(keys_b, idx_b, keys_a, idx_a, N, 7, hist, 0xffffffffu, 0, st);
    if (rc) return rc;
    rc = radix::pass<7>(keys_a, idx_a, keys_b, idx_b, N, 14, hist, 0xffffffffu, 0, st);
    if (rc) return rc;
    rg::gather_sorted_kernel<<<wide, 256, 0, st>>>(pos, idx_b, N, sorted);
    GSL_LAUNCH_CHECK("rg::gather_sorted_kernel");
    rg::Tables T;
    T.start[0] = nullptr;
    for (int L = 1; L <= rg::kLevels; ++L) {
        uint32_t *start = (uint32_t *)(w + p.tables[L]);
        T.start[L] = start;
        const int g = (int)std::min<size_t>((rg::table_entries(L) + 255) / 256, (size_t)sm_count() * 8);
        rg::cell_start_kernel<<<g, 256, 0, st>>>(keys_b, N, L, start);
        GSL_LAUNCH_CHECK("rg::cell_start_kernel");
    }
    rg::QueryOut out{normals, normals_in, residuals, centroids, knn};
    const size_t smem = sizeof(rg::WarpScratch) * rg::kWarps;
    const bool long_list = knn && k > rg::kMaxList;
    const auto kernel = long_list ? rg::knn_pca_kernel<true> : rg::knn_pca_kernel<false>;
    GSL_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int qgrid = (int)std::min<int64_t>((N + rg::kWarps - 1) / rg::kWarps, (int64_t)sm_count() * 16);
    kernel<<<qgrid, rg::kWarps * 32, smem, st>>>(sorted, N, k, ginfo, T, out, stats);
    GSL_LAUNCH_CHECK("rg::knn_pca_kernel");
    if (long_list) {
        int log_p = 0;
        while ((1 << log_p) < k) ++log_p;
        const int rows = std::max(1, rg::kOrderMinKeys >> log_p);
        const size_t osmem = (size_t)rows * ((size_t)1 << log_p) * rg::kOrderKeyBytes;
        GSL_CUDA_TRY(cudaFuncSetAttribute(rg::knn_order_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)osmem));
        const int64_t ogrid = (N + rows - 1) / rows;
        rg::knn_order_kernel<<<(unsigned)ogrid, rg::kOrderThreads, osmem, st>>>(pos, N, k, log_p, rows, knn);
        GSL_LAUNCH_CHECK("rg::knn_order_kernel");
    }
    return GSL_OK;
}

/*
 * segmentation_3D (rg:166-221), host side: the growth loop is serial by construction (every
 * accepted neighbour changes the availability set the next test reads).  Inputs are HOST arrays;
 * the neighbour lists come from gsl_region_knn_pca.  Python's `min(A, key=...)` over a set of
 * small ints visits them in increasing order, so the lowest index wins a residual tie.
 */
extern "C" int64_t gsl_region_grow(const int32_t *knn, int k, const double *normals, const double *residuals, int64_t N,
                                   double residual_threshold, double angle_threshold, int32_t *region_of,
                                   int64_t *region_sizes)
{
    if (N < 0 || k < 1 || (N > 0 && (!knn || !normals || !residuals || !region_of)))
        return fail(GSL_EINVAL, "gsl_region_grow: bad argument");
    std::vector<int32_t> by_residual((size_t)N);
    std::iota(by_residual.begin(), by_residual.end(), 0);
    std::stable_sort(by_residual.begin(), by_residual.end(), [&](int32_t a, int32_t b) { return residuals[a] < residuals[b]; });
    std::vector<char> available((size_t)N, 1);
    const double cos_thr = cos(angle_threshold);                                   // rg:207
    std::vector<int64_t> sizes;
    std::deque<int32_t> queue;
    size_t cursor = 0;
    for (;;) {
        while (cursor < (size_t)N && !available[by_residual[cursor]]) ++cursor;    // rg:193: min residual among A
        if (cursor == (size_t)N) break;
        const int32_t seed0 = by_residual[cursor];
        const int32_t region = (int32_t)sizes.size();
        int64_t size = 1;
        available[seed0] = 0;
        region_of[seed0] = region;
        queue.clear();
        queue.push_back(seed0);
        while (!queue.empty()) {                                                   // rg:201-215
            const int32_t seed = queue.front();
            queue.pop_front();
            const double *ns = normals + 3 * (size_t)seed;
            for (int j = 0; j < k; ++j) {
                const int32_t nb = knn[(size_t)seed * k + j];
                if (nb < 0 || nb >= N || !available[nb]) continue;
                const double *nn = normals + 3 * (size_t)nb;
                const double cos_angle = fabs(ns[0] * nn[0] + ns[1] * nn[1] + ns[2] * nn[2]);   // rg:205
                if (cos_angle > cos_thr) {
                    region_of[nb] = region;
                    available[nb] = 0;
                    ++size;
                    if (residuals[nb] < residual_threshold) queue.push_back(nb);   // rg:212-214
                }
            }
        }
        sizes.push_back(size);
    }
    if (region_sizes)
        for (size_t r = 0; r < sizes.size(); ++r) region_sizes[r] = sizes[r];
    return (int64_t)sizes.size();
}
