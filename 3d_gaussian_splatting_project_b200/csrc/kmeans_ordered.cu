// Reference-order centroid update for sm_100a.
//
// NumPy evaluates `data[labels == c].mean(axis=0)` (3D_clustering/k_means.py:125-128) as a
// float32 sum started from the identity +0.0, then one float64 division rounded to float32 (see
// oracle/gsl_oracle.c: orc_kmeans_update).  For D >= 2 the sum is SEQUENTIAL over the members in
// index order; for D = 1 the reduced axis is contiguous and NumPy uses its pairwise summation
// (ordered_pairwise_kernel below).  Float32 addition is not associative, so reproducing the
// reference bit for bit means keeping that order: one serial chain per (cluster, dimension).
// The K*D chains are independent, so the work is:
//
//   ordered_count_kernel     per 1024-row tile, member count per cluster
//   ordered_scan_kernel      per cluster, exclusive scan of the tile counts (+ totals)
//   ordered_start_kernel     exclusive scan of the totals -> segment starts
//   ordered_scatter_kernel   stable scatter of row indices into per-cluster member lists
//                            (warp match_any ranks keep ascending row order)
//   ordered_gather_kernel    member rows in list order into a contiguous, padded array per 32-dim chunk
//   ordered_stream_kernel    one warp per (cluster, 32 dims): TMA bulk copies of its contiguous rows into
//                            a shared-memory ring, added in order, lane = dimension
//   (D = 1: ordered_column_kernel gathers the members into one dense column and
//    ordered_pairwise_kernel sums each cluster's slice of it with NumPy's pairwise tree)
//   shift_kernel             ||new - old||_F
//
// This is the parity mode (single device).  The throughput mode is gsl_kmeans_step's float64
// segmented reduction, which is sharded and all-reduced.
#include <algorithm>
#include <mutex>

#include "common.cuh"
#include "kmeans_screen.cuh"

namespace gsl {

constexpr int kOrdTile = 1024;
constexpr int kOrdThreads = 256;

__global__ void __launch_bounds__(kOrdThreads)
ordered_count_kernel(const int32_t *__restrict__ labels, int64_t N, int K, int32_t *__restrict__ tile_counts,
                     int *__restrict__ bad_label)
{
    extern __shared__ int hist[];
    for (int i = threadIdx.x; i < K; i += kOrdThreads) hist[i] = 0;
    __syncthreads();
    const int64_t row0 = (int64_t)blockIdx.x * kOrdTile;
    for (int r = threadIdx.x; r < kOrdTile; r += kOrdThreads) {
        const int64_t row = row0 + r;
        if (row < N) {
            const int lab = labels[row];
            if ((unsigned)lab < (unsigned)K) atomicAdd(&hist[lab], 1);
            else *bad_label = 1;                         // skipped here and in the scatter; the shift comes back NaN
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K; i += kOrdThreads) tile_counts[(size_t)i * gridDim.x + blockIdx.x] = hist[i];      // [K][n_tiles]: the scan reads a cluster's row contiguously
}

// Block k: tile_counts[k][:] -> exclusive offsets in place, total[k].
__global__ void __launch_bounds__(kOrdThreads)
ordered_scan_kernel(int32_t *__restrict__ tile_counts, int n_tiles, int K, int64_t *__restrict__ total)
{
    __shared__ int64_t part[kOrdThreads];
    const int k = blockIdx.x, t = threadIdx.x;
    const int seg = (n_tiles + kOrdThreads - 1) / kOrdThreads;
    const int lo = min(t * seg, n_tiles), hi = min(lo + seg, n_tiles);
    int64_t s = 0;
    for (int i = lo; i < hi; ++i) s += tile_counts[(size_t)k * n_tiles + i];
    part[t] = s;
    __syncthreads();
    if (t == 0) {
        int64_t run = 0;
        for (int i = 0; i < kOrdThreads; ++i) { const int64_t v = part[i]; part[i] = run; run += v; }
        total[k] = run;
    }
    __syncthreads();
    int64_t run = part[t];
    for (int i = lo; i < hi; ++i) {
        const int c = tile_counts[(size_t)k * n_tiles + i];
        tile_counts[(size_t)k * n_tiles + i] = (int32_t)run;   // within-cluster offset (< N < 2^31)
        run += c;
    }
}

// The chain of the largest cluster is the critical path (2.2 ms at C5, where one cluster holds 12 % of the
// rows), the gather in front of it is not: clusters with at least 1/16 of the (valid) members are gathered
// first and their chains start on a helper stream while the caller's stream gathers and sums the rest.
//   phase 0: every cluster   1: the big ones   2: the others
__device__ __forceinline__ bool in_phase(int phase, int64_t n, int64_t n_members)
{
    const bool big = n * 16 >= n_members && n > 0;
    return phase == 0 || (phase == 1) == big;
}

// start[k] = members before cluster k; pstart[k] = the same with every cluster padded to a multiple of four
// rows (pstart[K] = padded total): the streamed chain reads its rows in groups of four.  *n_big = the number
// of clusters that phase 1 takes (second word of the workspace header, read by the tests).
__global__ void ordered_start_kernel(const int64_t *__restrict__ total, int K, int64_t *__restrict__ start,
                                     int64_t *__restrict__ pstart, int *__restrict__ n_big)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int64_t run = 0, prun = 0;
        for (int k = 0; k < K; ++k) {
            start[k] = run;
            pstart[k] = prun;
            run += total[k];
            prun += (total[k] + 3) & ~(int64_t)3;
        }
        pstart[K] = prun;
        int big = 0;
        for (int k = 0; k < K; ++k) big += in_phase(1, total[k], run);
        *n_big = big;
    }
}

__global__ void __launch_bounds__(kOrdThreads)
ordered_scatter_kernel(const int32_t *__restrict__ labels, int64_t N, int K,
                       const int32_t *__restrict__ tile_offsets, const int64_t *__restrict__ start,
                       int32_t *__restrict__ members)
{
    extern __shared__ int wc[];                 // [8][K] counts, then absolute bases (as int64 would
    int64_t *base = reinterpret_cast<int64_t *>(wc + 8 * K + ((8 * K) & 1));  // overflow int): [8][K] int64
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    for (int i = t; i < 8 * K; i += kOrdThreads) wc[i] = 0;
    __syncthreads();
    const int64_t row0 = (int64_t)blockIdx.x * kOrdTile + w * 128;
    int lab[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int64_t row = row0 + c * 32 + lane;
        lab[c] = row < N ? labels[row] : -1;
        if ((unsigned)lab[c] >= (unsigned)K) lab[c] = -1;        // out-of-range labels belong to no cluster
        if (lab[c] >= 0) atomicAdd(&wc[w * K + lab[c]], 1);
    }
    __syncthreads();
    for (int k = t; k < K; k += kOrdThreads) {
        int64_t run = start[k] + tile_offsets[(size_t)k * gridDim.x + blockIdx.x];
        for (int ww = 0; ww < 8; ++ww) { base[ww * K + k] = run; run += wc[ww * K + k]; }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int key = lab[c] >= 0 ? lab[c] : -1 - lane;     // invalid rows never match
        const unsigned m = __match_any_sync(0xffffffffu, key);
        if (lab[c] >= 0) {
            const int rank = __popc(m & ((1u << lane) - 1u));
            const int64_t b = base[w * K + lab[c]];
            members[b + rank] = (int32_t)(row0 + c * 32 + lane);
        }
        __syncwarp();
        if (lab[c] >= 0 && lane == __ffs(m) - 1) base[w * K + lab[c]] += __popc(m);
        __syncwarp();
    }
}

// ---- the chains: gather, then stream ---------------------------------------------------------------
// A chain that collects its own member rows needs one 4-byte copy per lane and row (rows of D = 59
// floats are only 4-byte aligned), and that, not the dependent adds, is what paces it: measured
// ~2750 cycles per 224-row batch against ~900 for the 224 adds.  Splitting the work removes the
// gather from the serial part:
//   ordered_gather_kernel   fully parallel and bandwidth bound: member rows in list order into a
//                           contiguous array per 32-dimension chunk (128 bytes per row and chunk,
//                           zero padded; layout below)
//   ordered_stream_kernel   one WARP per (cluster, chunk): its rows are one contiguous, 16-byte
//                           aligned stream, fetched by TMA bulk copies of up to 512 rows (one
//                           instruction per 64 KB stage, completion on an mbarrier) two stages ahead,
//                           and added in order, lane = dimension.  No other warp, no block barrier.
constexpr int kStreamRows = 512;       // rows per stage (64 KB)
constexpr int kStreamStages = 3;

// rows32[chunk][group][lane][4]: the rows of a cluster start at a multiple of four slots (pstart), four
// consecutive rows form a group, and a lane's four values of a group are contiguous -- the stream kernel
// fetches them with one 16-byte shared load.  One warp per group: four member rows read lane = dimension,
// one coalesced 512-byte store per chunk.
__global__ void __launch_bounds__(256)
ordered_gather_kernel(const float *__restrict__ data, int D, int n_chunks, const int32_t *__restrict__ members,
                      const int64_t *__restrict__ start, const int64_t *__restrict__ pstart, const int64_t *__restrict__ total,
                      int K, int64_t slots_pad, float *__restrict__ rows32, int phase)
{
    const int64_t n_members = start[K - 1] + total[K - 1];
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_groups = pstart[K] >> 2;
    for (int64_t g = warp; g < n_groups; g += n_warps) {
        const int64_t slot = g << 2;
        int lo = 0, hi = K - 1;                              // the cluster whose padded range holds the group
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (pstart[mid] <= slot) lo = mid;
            else hi = mid - 1;
        }
        const int64_t m = slot - pstart[lo], n = total[lo], s = start[lo] + m;
        if (!in_phase(phase, n, n_members)) continue;
        int row[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) row[j] = m + j < n ? __ldg(members + s + j) : -1;
        for (int c = 0; c < n_chunks; ++c) {
            const int d = c * 32 + lane;
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = (row[j] >= 0 && d < D) ? __ldg(data + (size_t)row[j] * D + d) : 0.f;
            __stcs(reinterpret_cast<float4 *>(rows32 + ((size_t)c * slots_pad + (size_t)slot) * 32) + lane,
                   make_float4(v[0], v[1], v[2], v[3]));
        }
    }
}

__global__ void __launch_bounds__(32)
ordered_stream_kernel(const float *__restrict__ rows32, int64_t slots_pad, int D, int K, const int64_t *__restrict__ start,
                      const int64_t *__restrict__ pstart, const int64_t *__restrict__ total, const float *__restrict__ old_c,
                      float *__restrict__ new_c, int phase)
{
    extern __shared__ __align__(128) float sbuf[];           // [kStreamStages][kStreamRows / 4][32][4]
    __shared__ __align__(8) unsigned long long bars[kStreamStages];
    const int k = blockIdx.x, lane = threadIdx.x, d = blockIdx.y * 32 + lane;
    const bool live = d < D;
    const int64_t n = total[k];
    if (!in_phase(phase, n, start[K - 1] + total[K - 1])) return;
    if (n == 0) {
        if (live) new_c[(size_t)k * D + d] = old_c[(size_t)k * D + d];   // km:126 else-branch
        return;
    }
    const float *src = rows32 + ((size_t)blockIdx.y * slots_pad + (size_t)pstart[k]) * 32;
    const int64_t n_batches = (n + kStreamRows - 1) / kStreamRows;
    if (lane == 0)
        for (int s = 0; s < kStreamStages; ++s) mbar_init(&bars[s], 1);
    __syncwarp();
    auto issue = [&](int64_t b) {                            // lane 0: the copy of batch b into its stage
        if (lane == 0 && b < n_batches) {
            const int64_t rows = (min((int64_t)kStreamRows, n - b * kStreamRows) + 3) & ~(int64_t)3;   // whole groups
            bulk_load_tile(sbuf + (size_t)(b % kStreamStages) * kStreamRows * 32, src + (size_t)b * kStreamRows * 32,
                           (unsigned)(rows * 128), &bars[b % kStreamStages]);
        }
    };
    for (int b = 0; b < kStreamStages - 1; ++b) issue(b);
    float acc = 0.0f;               // NumPy's add.reduce starts from its identity: a column of -0.0 sums to +0.0
    for (int64_t b = 0; b < n_batches; ++b) {
        __syncwarp();               // every lane is done reading batch b - 1, whose stage is refilled now
        issue(b + kStreamStages - 1);
        mbar_wait(&bars[b % kStreamStages], (unsigned)((b / kStreamStages) & 1));
        const int cnt = (int)min((int64_t)kStreamRows, n - b * kStreamRows);
        const float4 *grp = reinterpret_cast<const float4 *>(sbuf + (size_t)(b % kStreamStages) * kStreamRows * 32) + lane;
        // One dependent chain of adds, 32 rows = 8 groups = 8 shared loads of 16 bytes at a time; two
        // register sets alternate so that one is being loaded while the other is added.  Measured: 6.1
        // cycles per add (2.2 ms for the 719 k members of the largest C5 cluster); FFMA x * 1 + acc in place
        // of FADD, 256-row instead of 512-row stages and 6 instead of 3 stages all measured the same.
        int i = 0;                                           // rows done
        const int nb = cnt >> 5;                             // whole blocks of 32 rows
        if (nb > 0) {
            float4 x[8], y[8];
            auto add8 = [&](const float4 (&v)[8]) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc = __fadd_rn(acc, v[j].x); acc = __fadd_rn(acc, v[j].y); acc = __fadd_rn(acc, v[j].z); acc = __fadd_rn(acc, v[j].w);
                }
            };
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = grp[j * 32];
            int blk = 0;                                     // invariant: x holds block blk, not yet added
            for (; blk + 2 <= nb; blk += 2) {
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = grp[((blk + 1) * 8 + j) * 32];
                add8(x);
                if (blk + 2 < nb) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = grp[((blk + 2) * 8 + j) * 32];
                }
                add8(y);
            }
            if (blk < nb) add8(x);
            i = nb << 5;
        }
        for (; i < cnt; i += 4) {                            // remaining groups; the last one may be partial
            const float4 v = grp[(i >> 2) * 32];
            acc = __fadd_rn(acc, v.x);
            if (i + 1 < cnt) acc = __fadd_rn(acc, v.y);
            if (i + 2 < cnt) acc = __fadd_rn(acc, v.z);
            if (i + 3 < cnt) acc = __fadd_rn(acc, v.w);
        }
    }
    if (live) new_c[(size_t)k * D + d] = (float)((double)acc / (double)n);
}

// ---- D = 1: NumPy's pairwise sum ---------------------------------------------------------------------
// With one feature, data[mask] is an (n, 1) array whose reduced axis is contiguous, and NumPy's add loop
// sums it with pairwise_sum (numpy/_core/src/umath/loops_utils.h.src), float32 throughout:
//   n < 8          plain adds
//   n <= 128       eight strided accumulators, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail in order
//   n > 128        split at n2 = n/2 - (n/2 mod 8): pairwise(first n2) + pairwise(the rest)
// One tree over the whole member list.  Its shape depends on n only, so subtrees can be summed apart and
// combined in the tree's order.
constexpr int kPwBlock = 128;          // NumPy's PW_BLOCKSIZE
constexpr int kPwLevels = 10;          // top levels of the tree spread over the threads of one block
constexpr int kPwThreads = 1 << kPwLevels;

__device__ __forceinline__ int64_t pairwise_split(int64_t n)
{
    const int64_t h = n / 2;
    return h - h % 8;
}

__device__ float pairwise_leaf(const float *a, int n)      // n <= kPwBlock
{
    if (n < 8) {
        float r = 0.0f;
        for (int i = 0; i < n; ++i) r = __fadd_rn(r, a[i]);
        return r;
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - n % 8; i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], a[i + j]);
    }
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                          __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __fadd_rn(res, a[i]);
    return res;
}

// pairwise_sum(a, n) without recursion: a stack of pending right halves; bit s of `done` says that the
// left half of frame s is summed (in left[s]) and the value in hand is its right half.
__device__ float pairwise_sum(const float *a, int64_t n)
{
    int64_t r_off[32], r_n[32];        // n < 2^31 splits fewer than 25 times
    float left[32];
    unsigned done = 0;
    int sp = 0;
    int64_t off = 0, m = n;
    for (;;) {
        while (m > kPwBlock) {
            const int64_t h = pairwise_split(m);
            r_off[sp] = off + h; r_n[sp] = m - h; done &= ~(1u << sp); ++sp;
            m = h;
        }
        float v = pairwise_leaf(a + off, (int)m);
        while (sp > 0 && (done >> (sp - 1) & 1u)) { --sp; v = __fadd_rn(left[sp], v); }
        if (sp == 0) return v;
        left[sp - 1] = v; done |= 1u << (sp - 1);
        off = r_off[sp - 1]; m = r_n[sp - 1];
    }
}

// col[i] = the value of member i (members in list order, so cluster k is col[start[k], start[k] + total[k])).
__global__ void __launch_bounds__(256)
ordered_column_kernel(const float *__restrict__ data, const int32_t *__restrict__ members, const int64_t *__restrict__ start,
                      const int64_t *__restrict__ total, int K, float *__restrict__ col, int phase)
{
    const int64_t n_members = start[K - 1] + total[K - 1];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_members; i += (int64_t)gridDim.x * blockDim.x) {
        int lo = 0, hi = K - 1;                              // the last cluster starting at or before i holds it
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (start[mid] <= i) lo = mid;
            else hi = mid - 1;
        }
        if (in_phase(phase, total[lo], n_members)) col[i] = __ldg(data + members[i]);
    }
}

// One block per cluster.  Thread j walks the top kPwLevels levels of the cluster's tree along the bits of j
// (most significant first, 1 = right half) and sums the node it reaches; a path that meets a leaf early
// stops there, and only the thread whose remaining bits are zero owns that leaf.  The owners' sums are
// then combined bottom up, left + right, in shared memory.
__global__ void __launch_bounds__(kPwThreads)
ordered_pairwise_kernel(const float *__restrict__ col, const int64_t *__restrict__ start, const int64_t *__restrict__ total,
                        int K, const float *__restrict__ old_c, float *__restrict__ new_c, int phase)
{
    __shared__ float part[kPwThreads];
    const int k = blockIdx.x, j = threadIdx.x;
    const int64_t n = total[k];
    if (!in_phase(phase, n, start[K - 1] + total[K - 1])) return;
    if (n == 0) {
        if (j == 0) new_c[k] = old_c[k];                     // km:126 else-branch
        return;
    }
    int64_t off = start[k], m = n;
    int depth = 0;                                           // the nodes above `depth` on j's path are split
    for (; depth < kPwLevels && m > kPwBlock; ++depth) {
        const int64_t h = pairwise_split(m);
        if ((j >> (kPwLevels - 1 - depth)) & 1) { off += h; m -= h; }
        else m = h;
    }
    const bool owner = (j & ((1 << (kPwLevels - depth)) - 1)) == 0;
    if (owner) part[j] = pairwise_sum(col + off, m);
    for (int l = kPwLevels - 1; l >= 0; --l) {               // the node at depth l on j's path: children at j, j + step
        __syncthreads();
        const int step = 1 << (kPwLevels - 1 - l);
        if (owner && (j & (2 * step - 1)) == 0 && l < depth) part[j] = __fadd_rn(part[j], part[j + step]);
    }
    if (j == 0) new_c[k] = (float)((double)__fadd_rn(0.0f, part[0]) / (double)n);   // the reduction's identity, then the mean
}

__global__ void __launch_bounds__(256)
shift_kernel(const float *__restrict__ a, const float *__restrict__ b, int n, float *__restrict__ shift,
             const int *__restrict__ bad_label)
{
    __shared__ double red[8];
    double sq = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float df = a[i] - b[i];
        sq += (double)df * (double)df;
    }
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red[w];
        *shift = (bad_label && *bad_label) ? __int_as_float(0x7fc00000) : (float)sqrt(s);
    }
}

struct OrdWs { size_t tile_counts, total, start, pstart, members, rows32, slots_pad, bytes; };

static OrdWs ordered_layout(int64_t N, int D, int K)
{
    OrdWs o;
    const size_t n_tiles = (size_t)((N + kOrdTile - 1) / kOrdTile);
    size_t off = 256;                // [0, 256) of the aligned base: the header (out-of-range flag, big-cluster count)
    o.tile_counts = off; off += align_up(n_tiles * K * sizeof(int32_t), 256);
    o.total = off;       off += align_up((size_t)K * sizeof(int64_t), 256);
    o.start = off;       off += align_up((size_t)K * sizeof(int64_t), 256);
    o.pstart = off;      off += align_up((size_t)(K + 1) * sizeof(int64_t), 256);
    o.members = off;     off += align_up((size_t)N * sizeof(int32_t), 256);
    // the member rows per 32-dimension chunk, 128 bytes each (the TMA copies want 16-byte
    // aligned sources; the slot count is padded so that every chunk starts on a 256-byte boundary)
    o.slots_pad = align_up((size_t)(N > 0 ? N : 1) + 4 * (size_t)K, 4);      // every cluster padded to whole groups of four
    o.rows32 = off;      off += align_up((size_t)((D + 31) / 32) * o.slots_pad * 32 * sizeof(float), 256);
    o.bytes = off + 256;             // + slack for aligning the caller's pointer to 256 bytes
    return o;
}

size_t ordered_workspace_bytes(int64_t N, int D, int K) { return ordered_layout(N, D, K).bytes; }

// The stream on which gsl_kmeans_update_ordered runs the chains of the big clusters while the
// caller's stream gathers and sums the others (see in_phase).  High priority and non-blocking; one
// per device, created on first use (NULL if that fails).
static cudaStream_t helper_stream()
{
    static std::mutex mu;
    static cudaStream_t streams[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!streams[dev]) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&streams[dev], cudaStreamNonBlocking, hi) != cudaSuccess) {
            cudaGetLastError();
            streams[dev] = nullptr;
        }
    }
    return streams[dev];
}

}  // namespace gsl

using namespace gsl;

extern "C" int gsl_kmeans_update_ordered(const float *data, const int32_t *labels, int64_t N, int D, int K,
                                         const float *old_centroids, float *new_centroids, float *shift,
                                         void *ws, size_t ws_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (N < 0 || N >= ((int64_t)1 << 31)) return fail(GSL_EINVAL, "gsl_kmeans_update_ordered: N out of range");
    if (D < 1 || D > GSL_KMEANS_MAX_D || K < 1 || K > GSL_KMEANS_MAX_K) return fail(GSL_EINVAL, "gsl_kmeans_update_ordered: bad K/D");
    if (!old_centroids || !new_centroids || !shift) return fail(GSL_EINVAL, "gsl_kmeans_update_ordered: null pointer");
    if (N > 0 && (!data || !labels || !ws)) return fail(GSL_EINVAL, "gsl_kmeans_update_ordered: null pointer");
    const OrdWs L = ordered_layout(N, D, K);
    if (ws_bytes < L.bytes) return fail(GSL_EWORKSPACE, "gsl_kmeans_update_ordered: workspace %zu < %zu", ws_bytes, L.bytes);
    unsigned char *base = reinterpret_cast<unsigned char *>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    int32_t *tile_counts = reinterpret_cast<int32_t *>(base + L.tile_counts);
    int64_t *total = reinterpret_cast<int64_t *>(base + L.total);
    int64_t *start = reinterpret_cast<int64_t *>(base + L.start);
    int64_t *pstart = reinterpret_cast<int64_t *>(base + L.pstart);
    int32_t *members = reinterpret_cast<int32_t *>(base + L.members);
    const int n_tiles = (int)((N + kOrdTile - 1) / kOrdTile);
    int *bad_label = reinterpret_cast<int *>(base);          // first word of the workspace header
    int *n_big = bad_label + 1;                              // second word: clusters chained on the helper stream
    GSL_CUDA_TRY(cudaMemsetAsync(bad_label, 0, 2 * sizeof(int), st));

    if (N == 0) {
        GSL_CUDA_TRY(cudaMemsetAsync(total, 0, sizeof(int64_t) * (size_t)K, st));
        GSL_CUDA_TRY(cudaMemsetAsync(start, 0, sizeof(int64_t) * (size_t)K, st));
        GSL_CUDA_TRY(cudaMemsetAsync(pstart, 0, sizeof(int64_t) * (size_t)(K + 1), st));
    } else {
        ordered_count_kernel<<<n_tiles, kOrdThreads, K * sizeof(int), st>>>(labels, N, K, tile_counts, bad_label);
        GSL_LAUNCH_CHECK("ordered_count_kernel");
        ordered_scan_kernel<<<K, kOrdThreads, 0, st>>>(tile_counts, n_tiles, K, total);
        GSL_LAUNCH_CHECK("ordered_scan_kernel");
        ordered_start_kernel<<<1, 32, 0, st>>>(total, K, start, pstart, n_big);
        GSL_LAUNCH_CHECK("ordered_start_kernel");
        const size_t sc_smem = (size_t)(8 * K + ((8 * K) & 1)) * sizeof(int) + (size_t)8 * K * sizeof(int64_t);
        GSL_CUDA_TRY(cudaFuncSetAttribute(ordered_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc_smem));
        ordered_scatter_kernel<<<n_tiles, kOrdThreads, sc_smem, st>>>(labels, N, K, tile_counts, start, members);
        GSL_LAUNCH_CHECK("ordered_scatter_kernel");
    }
    const dim3 grid((unsigned)K, (unsigned)((D + 31) / 32));
    float *rows32 = reinterpret_cast<float *>(base + L.rows32);
    const size_t st_smem = (size_t)kStreamStages * kStreamRows * 32 * sizeof(float);
    GSL_CUDA_TRY(cudaFuncSetAttribute(ordered_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_smem));
    const int64_t warps = (N + 3) / 4 + K;
    const unsigned g = (unsigned)std::min<int64_t>((warps * 32 + 255) / 256, (int64_t)sm_count() * 16);
    auto gather = [&](int phase, cudaStream_t s) -> int {
        if (N == 0) return GSL_OK;
        if (D == 1) {                                        // one dense column (N floats) in the rows32 area
            ordered_column_kernel<<<g, 256, 0, s>>>(data, members, start, total, K, rows32, phase);
            GSL_LAUNCH_CHECK("ordered_column_kernel");
            return GSL_OK;
        }
        ordered_gather_kernel<<<g, 256, 0, s>>>(data, D, (int)grid.y, members, start, pstart, total, K, (int64_t)L.slots_pad, rows32, phase);
        GSL_LAUNCH_CHECK("ordered_gather_kernel");
        return GSL_OK;
    };
    auto chains = [&](int phase, cudaStream_t s) -> int {
        if (D == 1) {
            ordered_pairwise_kernel<<<K, kPwThreads, 0, s>>>(rows32, start, total, K, old_centroids, new_centroids, phase);
            GSL_LAUNCH_CHECK("ordered_pairwise_kernel");
            return GSL_OK;
        }
        ordered_stream_kernel<<<grid, 32, st_smem, s>>>(rows32, (int64_t)L.slots_pad, D, K, start, pstart, total, old_centroids, new_centroids, phase);
        GSL_LAUNCH_CHECK("ordered_stream_kernel");
        return GSL_OK;
    };
    cudaStream_t side = N >= (1 << 18) ? helper_stream() : nullptr;
    cudaEvent_t ev = nullptr;
    if (side && cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); side = nullptr; }
    if (!side) {
        if (int rc = gather(0, st)) return rc;
        if (int rc = chains(0, st)) return rc;
    } else {
        int rc = gather(1, st);
        if (rc == GSL_OK && (cudaEventRecord(ev, st) != cudaSuccess || cudaStreamWaitEvent(side, ev, 0) != cudaSuccess)) rc = fail(GSL_ECUDA, "gsl_kmeans_update_ordered: fork failed");
        if (rc == GSL_OK) rc = chains(1, side);
        if (rc == GSL_OK) rc = gather(2, st);
        if (rc == GSL_OK) rc = chains(2, st);
        // the caller's stream continues only after the big clusters' chains (also when something above failed)
        if (cudaEventRecord(ev, side) != cudaSuccess || cudaStreamWaitEvent(st, ev, 0) != cudaSuccess) { if (rc == GSL_OK) rc = fail(GSL_ECUDA, "gsl_kmeans_update_ordered: join failed"); }
        cudaEventDestroy(ev);
        if (rc != GSL_OK) return rc;
    }
    shift_kernel<<<1, 256, 0, st>>>(new_centroids, old_centroids, K * D, shift, bad_label);
    GSL_LAUNCH_CHECK("shift_kernel");
    return GSL_OK;
}
