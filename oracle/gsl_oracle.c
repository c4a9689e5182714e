/*
 * gsl_oracle.c -- CPU restatement of the reference hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this library.  The product (3d_gaussian_splatting_project_b200/) never does.
 *
 * Every function cites the lines of /root/reference it restates.  The reference is pure
 * Python; its arithmetic is IEEE float64 (lifting) and float64 distance / float32 mean
 * (K-means).  Two pieces of arithmetic live in un-vendored third-party code and are
 * restated from probes (see oracle/make_golden.py, which re-runs the probes against the
 * verbatim reference and pins this file to them):
 *   - NumPy's 3x3 `R @ v` (OpenBLAS 0.3.30 dgemv, Haswell kernel) rounds each row as
 *       fma(R[r][2], z, fma(R[r][0], x, R[r][1] * y))
 *   - scipy 1.18.1 cKDTree's squared distance (ckdtree/src/distance_base.h,
 *     sqeuclidean_distance_double): four running lanes over blocks of four dims,
 *     ((a0 + a1) + a2) + a3, then a sequential tail, no FMA.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -fopenmp).  -ffp-contract=off is
 * load-bearing: the compiler must not fuse the products of the distance loop.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* One camera view as the oracle consumes it.  Layout is private to oracle/ (the product
 * has its own struct in include/gslift.h); oracle/oracle.py builds it with a NumPy dtype. */
typedef struct {
    double R[9];          /* camera["rotation"], row-major, NOT transposed (dls.py:60)      */
    double t[3];          /* -R @ p                                        (dls.py:66)      */
    double fx, fy;        /*                                               (dls.py:54-55)   */
    double half_w, half_h;/* width / 2, height / 2                         (dls.py:76-77)   */
    double width, height; /* bounds                                        (dls.py:80)      */
    double scale_x, scale_y; /* seg_w / orig_w, seg_h / orig_h             (dls.py:270-271) */
    int32_t seg_w, seg_h; /* seg_map.shape[1], shape[0]                    (dls.py:267)     */
    int64_t map_offset;   /* element offset of this view's map in `maps`                    */
} OrcView;

int orc_version(void) { return 1; }

/* Thread count of the parallel loops below.  `torchrun` exports OMP_NUM_THREADS=1 to its workers;
 * bench.py's reference arm sets the count from the process' CPU affinity instead, so that the CPU
 * baseline uses the box's cores at every rank count. */
void orc_set_threads(int n)
{
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
#else
    (void)n;
#endif
}

int orc_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* R @ v with the probed dgemv rounding (deep_learning_segmentation.py:66,69). */
static inline double row_dot(const double *Rr, double x, double y, double z)
{
    return fma(Rr[2], z, fma(Rr[0], x, Rr[1] * y));
}

/* t = -R @ p (deep_learning_segmentation.py:66): negate R elementwise, then dgemv. */
void orc_translation(const double *R, const double *p, double *t)
{
    for (int r = 0; r < 3; ++r) {
        double nr[3] = { -R[3 * r], -R[3 * r + 1], -R[3 * r + 2] };
        t[r] = row_dot(nr, p[0], p[1], p[2]);
    }
}

/* project_gaussian (deep_learning_segmentation.py:43-82) followed by the rescale + clamp
 * of assign_labels (:281-286).  Returns 1 and the seg-map pixel when visible, else 0.
 * `near` (optional) is set when the f64 image coordinate lies within `eps` px of an
 * integer (pixel edge or image border) or the camera depth within `eps` of 0. */
static inline int project_one(const OrcView *vw, double X, double Y, double Z,
                              int *px, int *py, double eps, int *near)
{
    double cx = row_dot(vw->R + 0, X, Y, Z) + vw->t[0];   /* :69 */
    double cy = row_dot(vw->R + 3, X, Y, Z) + vw->t[1];
    double cz = row_dot(vw->R + 6, X, Y, Z) + vw->t[2];
    if (near && fabs(cz) < eps) *near = 1;
    if (cz <= 0) return 0;                                 /* :72 */
    double x = (vw->fx * cx / cz) + vw->half_w;            /* :76 */
    double y = (vw->fy * cy / cz) + vw->half_h;            /* :77 */
    if (near) {
        if (fabs(x - nearbyint(x)) < eps || fabs(y - nearbyint(y)) < eps) *near = 1;
    }
    if (!(0 <= x && x < vw->width && 0 <= y && y < vw->height)) return 0;  /* :80 */
    int xi = (int)x, yi = (int)y;                          /* :81 */
    int xs = (int)((double)xi * vw->scale_x);              /* :281 */
    int ys = (int)((double)yi * vw->scale_y);              /* :282 */
    if (xs < 0) xs = 0;                                    /* :285-286 */
    if (xs > vw->seg_w - 1) xs = vw->seg_w - 1;
    if (ys < 0) ys = 0;
    if (ys > vw->seg_h - 1) ys = vw->seg_h - 1;
    *px = xs; *py = ys;
    return 1;
}

/* Scalar entry used by the probe tests: one Gaussian, one view. */
int orc_project(const OrcView *vw, const float *pos, int *px, int *py)
{
    return project_one(vw, (double)pos[0], (double)pos[1], (double)pos[2], px, py, 0.0, NULL);
}

/*
 * assign_labels (deep_learning_segmentation.py:241-308) with the segmentation maps given.
 *   pos      f32[N][3]            gaussians['position']
 *   views    V entries, already filtered for missing images (:257-259), in camera order
 *   maps     int32, view v's map at maps + views[v].map_offset, row-major [seg_h][seg_w]
 *   label_min, n_classes: every map value must lie in [label_min, label_min + n_classes)
 *   labels   int32[N] out; -1 when never visible (:306)
 *   near     uint8[N] out or NULL: 1 when some (Gaussian, view) is within eps of a boundary
 *   visible_pairs  out or NULL: number of (Gaussian, view) pairs that passed the test
 * Majority (:297-303): Python max() over an insertion-ordered dict returns the FIRST key
 * with the maximal count, i.e. the label first seen earliest in camera order.
 * Returns 0, or -1 when a map value is outside the class range.
 */
int orc_lift_votes(const float *pos, int64_t N, const OrcView *views, int V,
                   const int32_t *maps, int label_min, int n_classes,
                   int32_t *labels, uint8_t *near, double eps, int64_t *visible_pairs)
{
    int bad = 0;
    int64_t vis_total = 0;
#pragma omp parallel reduction(+ : vis_total) reduction(| : bad)
    {
        int32_t *count = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_classes);
        int32_t *first = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_classes);
#pragma omp for schedule(static)
        for (int64_t i = 0; i < N; ++i) {
            double X = (double)pos[3 * i], Y = (double)pos[3 * i + 1], Z = (double)pos[3 * i + 2];
            memset(count, 0, sizeof(int32_t) * (size_t)n_classes);
            int seen = 0, nr = 0;
            for (int v = 0; v < V; ++v) {
                int px, py;
                if (!project_one(&views[v], X, Y, Z, &px, &py, eps, near ? &nr : NULL)) continue;
                ++vis_total;
                int32_t lab = maps[views[v].map_offset + (int64_t)py * views[v].seg_w + px]; /* :288 */
                int c = lab - label_min;
                if (c < 0 || c >= n_classes) { bad = 1; continue; }
                if (count[c] == 0) first[c] = v;           /* :293-294 dict insertion */
                ++count[c];                                /* :295 */
                seen = 1;
            }
            int32_t out = -1;                              /* :306 */
            if (seen) {
                int best = -1;
                for (int c = 0; c < n_classes; ++c) {
                    if (count[c] == 0) continue;
                    if (best < 0 || count[c] > count[best] ||
                        (count[c] == count[best] && first[c] < first[best]))
                        best = c;
                }
                out = best + label_min;                    /* :303 */
            }
            labels[i] = out;
            if (near) near[i] = (uint8_t)nr;
        }
        free(count);
        free(first);
    }
    if (visible_pairs) *visible_pairs = vis_total;
    return bad ? -1 : 0;
}

/* scipy cKDTree sqeuclidean_distance_double on float64 copies of float32 inputs
 * (k_means.py:116-122: KDTree(centroids) converts to float64; query(point) likewise). */
static inline double sqdist_scipy(const float *u, const float *v, int n)
{
    double acc0 = 0., acc1 = 0., acc2 = 0., acc3 = 0.;
    int i = 0;
    for (; i + 4 <= n; i += 4) {
        double d0 = (double)u[i] - (double)v[i];
        double d1 = (double)u[i + 1] - (double)v[i + 1];
        double d2 = (double)u[i + 2] - (double)v[i + 2];
        double d3 = (double)u[i + 3] - (double)v[i + 3];
        acc0 += d0 * d0; acc1 += d1 * d1; acc2 += d2 * d2; acc3 += d3 * d3;
    }
    double s = acc0 + acc1 + acc2 + acc3;
    for (; i < n; ++i) {
        double d = (double)u[i] - (double)v[i];
        s += d * d;
    }
    return s;
}

double orc_sqdist(const float *u, const float *v, int n) { return sqdist_scipy(u, v, n); }

/*
 * Assignment step (k_means.py:116-122, 140-144): nearest centroid by the distance above.
 * Brute force; exact ties resolve to the lowest index (cKDTree's winner on an exact tie
 * depends on its leaf order -- the documented exemption).  `gap` (optional, f64[N]) gets
 * second_best - best so callers can spot ties.
 */
void orc_kmeans_assign(const float *data, int64_t N, int D, const float *centroids, int K,
                       int64_t *labels, double *gap)
{
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < N; ++i) {
        const float *x = data + i * (int64_t)D;
        double best = INFINITY, second = INFINITY;
        int bi = 0;
        for (int k = 0; k < K; ++k) {
            double d = sqdist_scipy(centroids + (int64_t)k * D, x, D);
            if (d < best) { second = best; best = d; bi = k; }
            else if (d < second) second = d;
        }
        labels[i] = bi;
        if (gap) gap[i] = second - best;
    }
}

/*
 * NumPy's pairwise_sum (numpy/_core/src/umath/loops_utils.h.src) of x[0..n), float32 throughout:
 * plain adds below 8 values, eight strided accumulators up to 128 values, and above that the sum
 * of the two halves split at n/2 rounded down to a multiple of 8.
 */
static float pairwise_sum_f32(const float *x, int64_t n)
{
    if (n < 8) {
        float res = 0.f;
        for (int64_t i = 0; i < n; ++i) res = res + x[i];
        return res;
    }
    if (n <= 128) {
        float r[8];
        int64_t i;
        for (int j = 0; j < 8; ++j) r[j] = x[j];
        for (i = 8; i < n - (n % 8); i += 8)
            for (int j = 0; j < 8; ++j) r[j] = r[j] + x[i + j];
        float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res = res + x[i];
        return res;
    }
    int64_t n2 = n / 2;
    n2 -= n2 % 8;
    return pairwise_sum_f32(x, n2) + pairwise_sum_f32(x + n2, n - n2);
}

/*
 * Update step (k_means.py:125-128): data[labels == c].mean(axis=0), else the old centroid.
 * NumPy's add.reduce starts every column from its identity +0.0 (so a column of -0.0 sums to
 * +0.0).  For D >= 2 it reduces axis 0 of the gathered float32 [n, D] block row by row: every
 * column is a float32 sequential sum in index order.  For D = 1 the reduced axis is contiguous
 * and the whole column goes through one pairwise_sum.  np.mean then calls true_divide(sum_f32,
 * np.intp(n), out=sum_f32, casting='unsafe'): the quotient is formed in float64 and cast back to
 * float32 (numpy/_core/_methods.py:_mean).
 * counts (int64[K], optional) receives the member counts.
 */
void orc_kmeans_update(const float *data, const int64_t *labels, int64_t N, int D, int K,
                       const float *old_centroids, float *new_centroids, int64_t *counts)
{
#pragma omp parallel for schedule(dynamic, 1)
    for (int c = 0; c < K; ++c) {
        float *sum = new_centroids + (int64_t)c * D;
        int64_t n = 0;
        for (int d = 0; d < D; ++d) sum[d] = 0.f;
        if (D == 1) {
            for (int64_t i = 0; i < N; ++i) n += labels[i] == c;
            float *col = n ? (float *)malloc((size_t)n * sizeof(float)) : NULL;
            int64_t m = 0;
            for (int64_t i = 0; i < N && col; ++i)
                if (labels[i] == c) col[m++] = data[i];
            if (n) sum[0] = 0.f + pairwise_sum_f32(col, n);
            free(col);
        } else {
            for (int64_t i = 0; i < N; ++i) {
                if (labels[i] != c) continue;
                const float *x = data + i * (int64_t)D;
                for (int d = 0; d < D; ++d) sum[d] = sum[d] + x[d];
                ++n;
            }
        }
        if (n == 0) {
            for (int d = 0; d < D; ++d) sum[d] = old_centroids[(int64_t)c * D + d];
        } else {
            for (int d = 0; d < D; ++d) sum[d] = (float)((double)sum[d] / (double)n);
        }
        if (counts) counts[c] = n;
    }
}

/* Same update with float64 accumulation: the "exact mean" yardstick reported beside the
 * reference's float32 one (not a restatement of reference code). */
void orc_kmeans_update_f64(const float *data, const int64_t *labels, int64_t N, int D, int K,
                           const float *old_centroids, double *new_centroids)
{
#pragma omp parallel for schedule(dynamic, 1)
    for (int c = 0; c < K; ++c) {
        double *sum = new_centroids + (int64_t)c * D;
        int64_t n = 0;
        for (int d = 0; d < D; ++d) sum[d] = 0.;
        for (int64_t i = 0; i < N; ++i) {
            if (labels[i] != c) continue;
            const float *x = data + i * (int64_t)D;
            for (int d = 0; d < D; ++d) sum[d] += (double)x[d];
            ++n;
        }
        for (int d = 0; d < D; ++d)
            sum[d] = n ? sum[d] / (double)n : (double)old_centroids[(int64_t)c * D + d];
    }
}
