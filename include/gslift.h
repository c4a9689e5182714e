/*
 * gslift.h -- C ABI of libgslift.so: B200 (sm_100a) label lifting and K-means labelling.
 *
 * The reference (GloireLINVANI/3D_Gaussian_Splatting_Project) is pure Python and has no
 * FFI; its seam for this path is function level.  Each entry point below names the
 * reference lines it replaces (paths relative to the reference root):
 *
 *   dls = deep_learning_segmentation.py      km = 3D_clustering/k_means.py
 *   gs  = Web_Viewer_Gaussians_Selection/gaussians_selection.js
 *   rg  = 3D_clustering/region_growing.py
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the caller unless the
 *     parameter is documented "host".  The library never allocates device memory: scratch
 *     comes from the caller (`*_workspace_bytes`).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All work
 *     is enqueued on it; no entry point synchronises the device.
 *   - return 0 on success, a negative GSL_E* code otherwise; gsl_last_error() then returns
 *     a thread-local message.  Nothing throws, nothing calls exit().
 *   - entry points keep no global state besides a launch counter (tables travel through the
 *     caller's workspace), so calls on distinct streams with distinct workspaces are independent.
 *   - there is no CPU fallback: without a CUDA device every compute entry fails with
 *     GSL_ECUDA.
 */
#ifndef GSLIFT_H
#define GSLIFT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSL_ABI_VERSION 4

#define GSL_OK        0
#define GSL_EINVAL   -1   /* bad argument (NULL pointer, negative size, V/K/D out of range) */
#define GSL_EWORKSPACE -2 /* workspace too small                                            */
#define GSL_ECUDA    -3   /* CUDA runtime error (message carries cudaGetErrorString)        */
#define GSL_ERANGE   -4   /* label value outside the packable range                         */

#define GSL_MAX_VIEWS   65535   /* view index is kept in 16 bits by the vote keys            */
#define GSL_MAX_CODES   254     /* distinct label values per call (uint8 code 0 = "no vote",
                                   255 = the coarse table's "mixed cell" marker)             */
#define GSL_KMEANS_MAX_K 1024
#define GSL_KMEANS_MAX_D 256
#define GSL_REGION_MAX_LIST 16384  /* longest neighbour list gsl_region_knn_pca returns: one row's
                                      12-byte sort keys fill one CTA's shared memory */

/*
 * One camera view, host side.  Everything project_gaussian (dls:43-82) and the rescale in
 * assign_labels (dls:261-286) read, already in float64 exactly as Python would hold it.
 */
typedef struct GslView {
    double R[9];       /* camera["rotation"] row-major, NOT transposed            dls:60    */
    double t[3];       /* -R @ camera["position"], computed by the caller          dls:66    */
    double fx, fy;     /*                                                          dls:54-55 */
    double half_w;     /* camera["width"] / 2                                      dls:76    */
    double half_h;     /* camera["height"] / 2                                     dls:77    */
    double width;      /* camera["width"], camera["height"]: bounds test           dls:80    */
    double height;
    double scale_x;    /* seg_width / orig_width   (orig = opened image size)      dls:271   */
    double scale_y;    /* seg_height / orig_height                                 dls:270   */
    int32_t seg_w;     /* seg_map.shape[1]                                         dls:267   */
    int32_t seg_h;     /* seg_map.shape[0]                                                   */
    int64_t map_offset;/* byte offset of this view's packed map (gsl_pack_labels) in `packed`*/
} GslView;             /* 176 bytes */

/* ABI version (GSL_ABI_VERSION of the built library). */
int gsl_version(void);

/* Message for the last non-zero return on this thread ("" if none). */
const char *gsl_last_error(void);

/* Kernels this process has launched through the library so far (statistics only: benchmarks
 * report the difference around their timed region). */
unsigned long long gsl_launch_count(void);

/* Number of CUDA devices visible to the library, or a negative error code. */
int gsl_device_count(void);

/*
 * Stage label maps: int32 values as segment_image returns them (dls:158, :124) -> uint8
 * codes  code = label - label_min + 1  (0 is reserved for "not visible").
 * Values outside [label_min, label_min + n_classes) set *d_err (device int, caller zeroes
 * it) to 1 and are written as code 0.  n_classes <= GSL_MAX_CODES.
 *
 *   maps    n_maps row-major int32 maps of seg_h x seg_w, back to back (4-byte aligned; 16-byte
 *           alignment and seg_w % 4 == 0 enable the vector path)
 *   packed  n_maps packed maps of gsl_packed_map_bytes(seg_w, seg_h) bytes each, back to back
 *           (16-byte aligned).  The packed layout is private to the library: strips 16 pixels wide
 *           (a 128-byte line = 16 x 8 pixels) inside a ring of zero codes, so that the 32 gathers
 *           of a warp of neighbouring Gaussians touch a few cache lines instead of one per row.
 * Views with different map shapes are packed by separate calls; GslView.map_offset is the byte
 * offset of a view's packed map inside the buffer handed to gsl_lift_votes.
 */
int64_t gsl_packed_map_bytes(int seg_w, int seg_h);
int gsl_pack_labels(const int32_t *maps, int n_maps, int seg_w, int seg_h, uint8_t *packed,
                    int label_min, int n_classes, int *d_err, void *stream);

/*
 * Hybrid staging from HOST int32 maps (the PCIe transfer of 4 bytes per pixel is what a call from
 * host maps waits for): gsl_host_pack_labels is a HOST-side helper (no device work) that narrows
 * maps to the same uint8 codes on n_threads host threads (0 = all), so that some views can cross
 * the bus as 1 byte per pixel while the DMA engine moves the others as int32; gsl_tile_codes turns
 * such row-major codes (device) into the packed layout gsl_pack_labels produces.
 *   maps[m]   HOST pointer to the n_px[m] int32 values of map m; its codes go to out + sum(n_px[0..m))
 *   minmax    HOST int[2], in/out: running min / max of the values seen
 *   bad       HOST int, out: 1 if a value fell outside [label_min, label_min + n_classes) (code 0)
 */
int gsl_host_pack_labels(const int32_t *const *maps, const int64_t *n_px, int n_maps, int label_min,
                         int n_classes, uint8_t *out, int n_threads, int *minmax, int *bad);
int gsl_tile_codes(const uint8_t *codes, int n_maps, int seg_w, int seg_h, uint8_t *packed, void *stream);

/* Device min/max of an int32 buffer into d_minmax[2] (caller initialises to INT_MAX,
 * INT_MIN); lets the host choose label_min / n_classes without a CPU pass. */
int gsl_label_range(const int32_t *maps, int64_t n_px, int *d_minmax, void *stream);

/* Scratch needed by the gsl_lift_* entry points for N Gaussians and V views (the vote sheet, one
 * byte per (Gaussian, view), plus about 40 bytes per Gaussian and 2 bytes per (256-Gaussian tile, view)). */
size_t gsl_lift_workspace_bytes(int64_t N, int V);

/*
 * The vote loop and the majority of assign_labels (dls:255-306) for precomputed maps:
 * for every Gaussian, every view in order: project (dls:43-82, float64 -- evaluated in float32
 * first and re-evaluated in float64 wherever the float32 error bound cannot prove the float64
 * outcome), test z > 0 and image bounds, rescale + clamp (dls:281-286), gather the code, count; then
 * labels[i] = the label with the most votes, the one seen first in view order on a tie
 * (Python max() over an insertion-ordered dict, dls:303), or -1 if never visible (dls:306).
 *
 *   pos        float32 [N][3]         gaussians['position'] (dls:36-38)
 *   views      HOST array of V views in camera order, views whose image is missing already
 *              dropped (dls:257-259).  Copied during the call.
 *   packed     uint8 codes from gsl_pack_labels, view v at packed + views[v].map_offset
 *   label_min, n_classes   the pair the maps were packed with
 *   labels     int32 [N] out
 *   near       optional uint8 [N] out (may be NULL): gsl_lift_near's diagnostic
 *
 * gsl_lift_votes == gsl_lift_prepare, gsl_lift_gather, gsl_lift_majority on the same stream and
 * workspace.
 */
int gsl_lift_votes(const float *pos, int64_t N, const GslView *views, int V,
                   const uint8_t *packed, int label_min, int n_classes, int32_t *labels,
                   uint8_t *near, double near_eps,
                   void *ws, size_t ws_bytes, void *stream);

/*
 * The two steps of gsl_lift_votes.  prepare reads camera parameters and positions only (no maps,
 * so it can run while maps are still being uploaded): it uploads the view tables, sorts the
 * Gaussians into spatial order, boxes every run of 256 and decides per (tile, view) whether the
 * view can be skipped, swept with the tile-wide error bound, or needs the per-pair / float64
 * treatment.  sweep needs all packed maps resident and the workspace prepare filled.
 *   best       optional uint32 [N] out (may be NULL): votes of the winning label << 16 |
 *              (65535 - view of its first sighting), 0 when labels[i] == -1.  Label sets wider than
 *              GSL_MAX_CODES are lifted in several passes over disjoint label ranges and merged
 *              with gsl_lift_merge: the larger key wins, exactly the reference's rule.
 */
int gsl_lift_prepare(const float *pos, int64_t N, const GslView *views, int V,
                     void *ws, size_t ws_bytes, void *stream);
int gsl_lift_sweep(const float *pos, int64_t N, const GslView *views, int V,
                   const uint8_t *packed, int label_min, int n_classes, int32_t *labels,
                   uint32_t *best, void *ws, size_t ws_bytes, void *stream);
/*
 * The two kernels of gsl_lift_sweep, separately callable (benchmarks time them one by one):
 * gather fills the vote sheet in `ws` (one uint8 code per (Gaussian, view), 4 views to a word),
 * majority reduces it to labels.  `views` must be the host array gsl_lift_prepare was given: the
 * float32 constants of the swept views travel to the kernel as launch parameters, with the map
 * addresses resolved against `packed`.
 */
int gsl_lift_gather(const float *pos, int64_t N, const GslView *views, int V,
                    const uint8_t *packed, void *ws, size_t ws_bytes, void *stream);
/* gather for views [v_begin, v_end) only (v_begin a multiple of 16; v_end a multiple of 16 or V):
 * lets a caller sweep the views whose packed maps are already resident while later maps are still
 * crossing PCIe.  gsl_lift_gather == the range [0, V). */
int gsl_lift_gather_range(const float *pos, int64_t N, const GslView *views, int V, int v_begin, int v_end,
                          const uint8_t *packed, void *ws, size_t ws_bytes, void *stream);
int gsl_lift_majority(int64_t N, int V, int label_min, int n_classes, int32_t *labels, uint32_t *best,
                      void *ws, size_t ws_bytes, void *stream);
/* labels[i], best[i] = the pair with the larger key of (labels, best) and (labels_b, best_b). */
int gsl_lift_merge(int32_t *labels, uint32_t *best, const int32_t *labels_b, const uint32_t *best_b,
                   int64_t N, void *stream);

/*
 * Diagnostic of the parity criterion: near[i] = 1 when some (Gaussian i, view) has an image
 * coordinate within near_eps px of an integer or |z_cam| < near_eps -- the set exempt from
 * bit-exactness.  Evaluates every pair with the float64 expressions (no culling).
 */
int gsl_lift_near(const float *pos, int64_t N, const GslView *views, int V, uint8_t *near,
                  double near_eps, void *ws, size_t ws_bytes, void *stream);

/* Test hook: counts (into *n_bad, device) the i for which the kernel's shared-reciprocal
 * division of a1[i]/b[i], a2[i]/b[i] differs in any bit from IEEE-754 division. */
int gsl_div_selftest(const double *a1, const double *a2, const double *b, int64_t n,
                     unsigned long long *n_bad, void *stream);

/* Scratch needed by the K-means entry points. */
size_t gsl_kmeans_workspace_bytes(int64_t N, int D, int K);

/*
 * Assignment (km:116-122, :140-144): labels[i] = argmin_k d2(centroids[k], data[i]) with
 * scipy cKDTree's float64 squared distance (four running lanes, no FMA).  Exact ties
 * resolve to the lowest k.
 *   data float32 [N][D] row-major (km:109), centroids float32 [K][D], labels int32 [N].
 */
int gsl_kmeans_assign(const float *data, int64_t N, int D, const float *centroids, int K,
                      int32_t *labels, void *ws, size_t ws_bytes, void *stream);

/*
 * One Lloyd pass over this rank's rows: assignment as above, fused with per-cluster
 * float64 sums and counts.  sums[K][D+1] (float64, out, overwritten): sums[k][0..D) = sum
 * of member rows, sums[k][D] = member count.  Deterministic (fixed reduction order).
 * Multi-GPU: all-reduce(sum) `sums` across ranks, then call gsl_kmeans_finalize.
 */
int gsl_kmeans_step(const float *data, int64_t N, int D, const float *centroids, int K,
                    int32_t *labels, double *sums, void *ws, size_t ws_bytes, void *stream);

/*
 * Update + convergence metric (km:125-131) from reduced sums: new[k] = float32(sum/count),
 * or old[k] when the cluster is empty; *shift = ||new - old||_F as float32 (device scalar).
 */
int gsl_kmeans_finalize(const double *sums, const float *old_centroids, int K, int D,
                        float *new_centroids, float *shift, void *stream);

/*
 * One Lloyd pass of a job sharded over `world` ranks (one process per GPU), with the exchange
 * step fused into the reduction kernel: assignment + per-CTA sums as in gsl_kmeans_step, then ONE
 * kernel that reduces the partials, pushes this rank's K x (D+1) float64 sums into every rank's
 * exchange buffer over peer memory (NVLink), waits for the other ranks' sums, adds them in rank
 * order (bit-identical totals on every rank) and forms the new centroids and the shift -- what
 * gsl_kmeans_step + all-reduce + gsl_kmeans_finalize compute, without the collective library.
 *   xbufs   HOST array of `world` device pointers; xbufs[r] = rank r's exchange buffer of
 *           gsl_kmeans_exchange_bytes(world, D, K) bytes, 256-byte aligned, zeroed once before
 *           first use, mapped into this process (peer access; e.g. torch symmetric memory).
 *           world == 1: any device buffer of that size.
 *   seq     exchange counter: 1 on the first call on these buffers, +1 per call, equal on all
 *           ranks.  Every rank must make the call (it is a collective); a rank with N == 0 joins
 *           with zero sums.
 *   sums    float64 [K][D+1] out: the totals over all ranks.
 *   shift   NaN if another rank did not arrive within GSLIFT_EXCHANGE_TIMEOUT_MS (default 30 s).
 */
size_t gsl_kmeans_exchange_bytes(int world, int D, int K);
int gsl_kmeans_step_exchange(const float *data, int64_t N, int D, const float *centroids, int K,
                             int32_t *labels, int rank, int world, void *const *xbufs, uint64_t seq,
                             float *new_centroids, float *shift, double *sums,
                             void *ws, size_t ws_bytes, void *stream);

/*
 * Reference-order update (km:125-128 exactly): every centroid coordinate is the float32
 * SEQUENTIAL sum of its members in index order, divided in float64 and rounded to float32
 * -- what NumPy's mean(axis=0) produces.  Single device only (the order cannot be sharded).
 *   labels int32 [N] from gsl_kmeans_assign / gsl_kmeans_step.  A label outside [0, K) is skipped
 *   and reported: *shift comes back NaN (the call is asynchronous, so there is no return code for it).
 */
int gsl_kmeans_update_ordered(const float *data, const int32_t *labels, int64_t N, int D, int K,
                              const float *old_centroids, float *new_centroids, float *shift,
                              void *ws, size_t ws_bytes, void *stream);

/*
 * Test hook for the tensor-core screening of gsl_kmeans_assign/step (K <= 64, 8 <= D <= 64):
 * runs the assignment and, for every (row, centroid), compares the screened ranking value with
 * the float64 distance.  out3[0] += number of (row, centroid) pairs whose error exceeds the
 * bound the kernel relies on (must stay 0); out3[1] += total candidates forwarded to the
 * float32/float64 stages; out3[2] += rows outside the range where the bound is proven (values
 * near float32 overflow or underflow, NaN/Inf): they take every centroid as a candidate and are
 * not checked.  out3 is a device array of three counters the caller zeroes.
 */
int gsl_kmeans_screen_selftest(const float *data, int64_t N, int D, const float *centroids, int K,
                               int32_t *labels, unsigned long long *out3, void *stream);

/* Recolouring (km:99-101, :147-149): colors[i][0..3) = palette[labels[i] % 8]; `palette` is a
 * device float32 [8][3] the host fills with COLORS (km:8), divided by 255.0 or not. */
int gsl_recolor(const int32_t *labels, int64_t N, const float *palette, float *colors, void *stream);

/*
 * Host-side helper (no device work): ASCII body of a labelled PLY as plyfile writes it with
 * text=True (km:190-193): every field through "%.18g" of its float64 value, one space between
 * fields, one vertex per line.  `records` = n_rows packed little-endian records of record_size
 * bytes; types[f] in {0:int8 1:uint8 2:int16 3:uint16 4:int32 5:uint32 6:float32 7:float64},
 * offsets[f] = byte offset of field f.  Formats on n_threads host threads (0 = all).  Returns the
 * number of bytes written to `out` (40 bytes per field always suffice) or a negative GSL_E* code.
 */
int64_t gsl_ply_format_ascii(const void *records, int64_t n_rows, int record_size, int n_fields,
                             const int *types, const int *offsets, char *out, int64_t out_cap,
                             int n_threads);

/*
 * Viewer-side consumers of the labels (SURVEY.md section 8f, N3): the per-Gaussian loops the
 * WebGL viewer's worker runs on every camera move and click.  JavaScript numbers are float64 and
 * `| 0` is ToInt32; both entry points reproduce that arithmetic in the reference's order.
 *   pos      float32, Gaussian i at pos + i * stride (stride in floats: 8 for the viewer's 32-byte
 *            rows gs:237, 3 for gaussians['position'])
 *
 * gsl_viewer_depth_sort -- runSort (gs:417-462) without its early-out (gs:421-425, the caller's
 * business): depth_i = ((vp[2]*x + vp[6]*y + vp[10]*z) * 4096) | 0, bucket_i = ((depth_i - min) *
 * (65536 / (max - min))) | 0, depth_index = Gaussian indices in a STABLE order of increasing bucket
 * (the counting sort of gs:449-457).  Gaussians whose bucket evaluates to 65536 fall off the end of
 * the reference's 65536-entry typed arrays: they are absent from depthIndex and the tail of
 * depthIndex keeps its initial zeros -- reproduced here.
 *   view_proj    HOST float64 [16], the message the worker receives (gs:626); entries 2, 6, 10 are read
 *   depth_index  uint32 [N] out (Uint32Array, gs:453)
 */
size_t gsl_viewer_sort_workspace_bytes(int64_t N);
int gsl_viewer_depth_sort(const float *pos, int64_t N, int stride, const double *view_proj,
                          uint32_t *depth_index, void *ws, size_t ws_bytes, void *stream);

/*
 * gsl_viewer_hit_test -- performHitTesting (gs:361-395): project every Gaussian with the combined
 * matrix (gs:398-405; skipped when w <= 0), screen = (ndc + 1) * 0.5 * viewport, dist =
 * Math.hypot(screen - click) (V8's algorithm), and among those with dist < 10 the one with the
 * smallest (dist, depth), the lowest index winning a full tie, exactly as the sequential scan does
 * (including its behaviour on a NaN depth).
 *   matrix        HOST float64 [16] = multiply4(projectionMatrix, viewMatrix) (gs:110-123, :364)
 *   labels        int32 [N] (labelData, gs:241)
 *   no_selection  value written when nothing is within 10 px (NO_SELECTION = -999999, gs:6)
 *   label_out     int32 device scalar out (may be NULL);  index_out  int64 device scalar out (may be
 *                 NULL): index of the selected Gaussian or -1
 */
size_t gsl_viewer_hit_workspace_bytes(void);
int gsl_viewer_hit_test(const float *pos, const int32_t *labels, int64_t N, int stride, const double *matrix,
                        double x, double y, double viewport_w, double viewport_h, int32_t no_selection,
                        int32_t *label_out, int64_t *index_out, void *ws, size_t ws_bytes, void *stream);

/*
 * Normals and residuals of 3D_clustering/region_growing.py (SURVEY.md section 8f, N4).
 *
 * gsl_region_knn_pca -- for every point the k nearest neighbours (itself included, as
 * KDTree.query of a tree point returns it, rg:100), their centroid (rg:105) and, from the
 * covariance of the centred neighbours (rg:108-111), the eigenvector of the smallest eigenvalue
 * (rg:114-117), flipped when dot(normal, point - centroid) > 0 (rg:120-121) and normalised
 * (rg:124); residual_i = |dot(normal_i, point_i - centroid_i)| (rg:161).
 * The neighbour set is exact (float64 squared distances in scipy's summation order, smallest k by
 * (distance, index); an exact distance tie at the k-th neighbour goes to the lower index where
 * scipy's answer depends on its tree layout).  Moments are accumulated in float64 (the reference:
 * float32 mean, float32 sgemm, LAPACK float32 eigh), so normals and residuals agree with the
 * reference to float32 accuracy, not bit for bit.
 *   pos         float32 [N][3], finite (scipy's KDTree rejects non-finite data as well)
 *   k           1 <= k <= N  (rg:272-274 use 2000; rg:278 uses 10)
 *   normals_in  optional float64 [N][3]: normals to form the residual with (compute_residuals takes
 *               them as an argument, rg:130); NULL = the normals computed by this call
 *   normals     optional float64 [N][3] out        residuals  optional float64 [N] out
 *   centroids   optional float64 [N][3] out
 *   knn         optional int32 [N][k] out, k <= GSL_REGION_MAX_LIST (larger k with knn != NULL:
 *               GSL_EINVAL before any device work; the other outputs take any k <= N):
 *               neighbour indices in increasing (distance, index) order (KDTree.query order)
 *   stats       optional uint64 [4], device, caller zeroes: += walks over candidate cells, += points visited by
 *               those walks, += cubes that turned out too small, += walks spent on further select digits
 *               (work counters for benchmarks)
 */
size_t gsl_region_workspace_bytes(int64_t N);
int gsl_region_knn_pca(const float *pos, int64_t N, int k, const double *normals_in, double *normals,
                       double *residuals, double *centroids, int32_t *knn, unsigned long long *stats,
                       void *ws, size_t ws_bytes, void *stream);

/*
 * segmentation_3D (rg:166-221) given the neighbour lists: HOST-side helper (no device work; the
 * growth loop is serial by construction).  All pointers are HOST pointers.  Seeds are taken in
 * increasing residual among the still available points (rg:193), a neighbour joins the region when
 * |dot(n_seed, n_neighbour)| > cos(angle_threshold) (rg:205-209) and becomes a seed itself when its
 * residual is below residual_threshold (rg:212-214).
 *   region_of     int32 [N] out: region number of every point, in order of creation
 *   region_sizes  optional int64 [N] out: size of every region created
 * Returns the number of regions, or a negative GSL_E* code.
 */
int64_t gsl_region_grow(const int32_t *knn, int k, const double *normals, const double *residuals, int64_t N,
                        double residual_threshold, double angle_threshold, int32_t *region_of,
                        int64_t *region_sizes);

#ifdef __cplusplus
}
#endif
#endif /* GSLIFT_H */
