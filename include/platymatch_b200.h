/*
 * platymatch_b200.h — C ABI of libplatymatch_b200.so (hand-written CUDA for sm_100a).
 *
 * Drop-in boundary for the estimate_transform hot path of juglab/PlatyMatch.  The reference has no
 * FFI layer: its boundary is the Python function API imported by the napari widget
 * (platymatch/_dock_widget.py:10,16-21).  Every entry point below names the reference function
 * (file:line, relative to the reference repo) whose arithmetic it replaces; INTEGRATION.md shows
 * the ctypes stub a maintainer would put behind each reference function.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / numpy types.
 *   - `pm_*` entry points take DEVICE pointers and a `cudaStream_t` passed as `void*` (0 = legacy
 *     default stream); they enqueue work and return without synchronising unless stated.
 *     The caller owns every buffer (inputs, outputs, workspace); the library never frees or
 *     retains a pointer after the call's work has completed on the stream.
 *   - `pm_host_*` entry points take HOST pointers (what a numpy caller holds), copy in, run,
 *     copy out and synchronise.
 *   - point clouds are N x 3 float64 row-major, coordinate order as given (the reference uses zyx);
 *     transforms are 4 x 4 float64 row-major acting on column vectors (apply_transform.py:14-17).
 *   - return value: 0 = ok; negative = error (PM_ERR_*), message via pm_last_error_string().
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef PLATYMATCH_B200_H
#define PLATYMATCH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PM_OK 0
#define PM_ERR_INVALID_ARGUMENT (-1)
#define PM_ERR_CUDA (-2)
#define PM_ERR_WORKSPACE (-3)
#define PM_ERR_INFEASIBLE (-4)
#define PM_ERR_UNSUPPORTED (-5)

#define PM_NBINS 360          /* 5 r x 6 theta x 12 phi  (shape_context.py:10) */
/* the widget's "Transform" choice (_dock_widget.py:627; shape_context.py:126-129, perform_icp.py:17-20) */
#define PM_TRANSFORM_AFFINE 0
#define PM_TRANSFORM_SIMILAR 1
#define PM_STATS_DOUBLES 16   /* layout of the cloud-stats block, see pm_cloud_stats */

/* ---- library ------------------------------------------------------------------------------ */
int pm_version(void);
const char *pm_last_error_string(void);  /* thread-local; valid until the next failing call */
int pm_device_count(void);               /* number of visible CUDA devices (0 if none) */
int pm_sm_count(int device);
/* number of kernels this library has launched in this process (bench.py's `gpu_launches`) */
unsigned long long pm_launch_count(void);
/* FP32 FMA issue-rate probe: `blocks` x 256 threads, each `iters` x 16 dependent-chain-free FFMAs;
 * returns the FLOP count through *flops_out (host); time it with events around the call. */
int pm_probe_fp32_fma(int blocks, int iters, float *sink, double *flops_out, void *stream);

/* ---- K0  cloud statistics -------------------------------------------------------------------
 * get_centroid (platymatch/utils/utils.py:48-56) and the PCA first axis computed inside get_unary
 * (shape_context.py:162-165: sklearn PCA.components_[0], sign: largest-|.| entry positive).
 * stats[0:3] centroid, stats[3:6] first principal axis x0, stats[6:12] covariance (xx,xy,xz,yy,yz,zz,
 * divided by n-1), stats[12] n, stats[13:16] eigenvalues descending.  All float64 on device. */
int pm_cloud_stats(const double *pts, int n, double *stats, void *stream);

/* ---- label image -> detections (SURVEY §8f row 2) --------------------------------------------
 * The per-id loops of _dock_widget.py:497-521: for every non-zero id (ascending, np.unique order)
 * centroid = mean z / y / x of its voxels, size = anisotropy * voxel count.  One streaming pass over
 * the volume (HBM-bound); exact integer sums, so the means equal np.mean bit for bit.
 *   labels      [nz][ny][nx] int32 (PM_LABEL_I32) or uint16 (PM_LABEL_U16), device; ids <= 0 = background
 *   table_size  > largest id (pm_label_max_id finds it); ids >= table_size are ignored
 *   ids [capacity] int32, centroids [capacity][3] float64 (z, y, x), sizes [capacity] float64,
 *   n_out [1] int32 = number of non-empty ids (may exceed capacity: then only the first are written)
 * workspace: pm_label_workspace_bytes(table_size). */
#define PM_LABEL_I32 0
#define PM_LABEL_U16 1
int pm_label_max_id(const void *labels, int dtype, size_t n_voxels, uint32_t *max_id, void *stream);
size_t pm_label_workspace_bytes(uint32_t table_size);
int pm_label_centroids(const void *labels, int dtype, int nz, int ny, int nx, uint32_t table_size, double anisotropy,
                       int capacity, int32_t *ids, double *centroids, double *sizes, int32_t *n_out, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ---- two label volumes -> contingency table (DESIGN §8 row 7) ------------------------------------------------
 * What a segmentation is scored with when there are no keypoints: for volumes A, B of one shape, every pair of ids
 * (a, b) != (0, 0) that meet at some voxel and its voxel count (np.unique of the pair keys a << 32 | b with the
 * (0, 0) entry removed).  Ids <= 0 count as background (0).  Instance sizes are the table's row and column sums,
 * IoU(a, b) = n / (|A_a| + |B_b| - n).  One streaming pass over both volumes (HBM-bound) into an open-addressing hash
 * table of `capacity` slots in the workspace, then a compaction.  Offsets and counts are 64-bit.
 *   labels_a, labels_b  [nz][ny][nx] int32 (PM_LABEL_I32) or uint16 (PM_LABEL_U16) each, device
 *   capacity   table slots, a power of two; a pair that finds no slot within 128 probes is not stored (keep the
 *              table at most half full: pm_label_max_id of both volumes bounds the number of pairs in practice)
 *   keys [capacity] uint64 out: a << 32 | b of the first n_out[0] entries, any order;  counts [capacity] uint64 out
 *   n_out [2] uint64 out: pairs written, voxels whose pair was NOT stored (non-zero = overflow: rerun with a larger
 *              capacity; the pairs written are then incomplete)
 * Every pointer must be 16-byte aligned.  workspace: pm_label_overlap_workspace_bytes(capacity). */
size_t pm_label_overlap_workspace_bytes(uint64_t capacity);
int pm_label_overlap(const void *labels_a, int dtype_a, const void *labels_b, int dtype_b, int nz, int ny, int nx,
                     uint64_t capacity, uint64_t *keys, uint64_t *counts, uint64_t *n_out, void *workspace,
                     size_t workspace_bytes, void *stream);

/* ---- resample a volume through an affine map (SURVEY §8f row 5) --------------------------------------
 * The transformed-image export of EvaluateMetrics._export_transformed_image (_dock_widget.py:1095-1130): the
 * moving image resampled into the fixed image's grid, so the two can be overlaid voxel by voxel.  Contract:
 * scipy.ndimage.affine_transform(src, M[:3,:3], offset=M[:3,3], output_shape, order, mode='constant', cval)
 * in voxel index space (the reference goes through SimpleITK; agreement with that is not verified).
 *   src    [sz][sy][sx] int32 (PM_LABEL_I32), uint16 (PM_LABEL_U16) or float32 (PM_RESAMPLE_F32), device
 *   M      16 float64, device: maps an output index (z, y, x, 1) to a source index; for a registration transform
 *          T (moving zyx -> fixed zyx) this is inv(T).  c_h = ((z M[h][0] + y M[h][1]) + x M[h][2]) + M[h][3] in
 *          float64 without FMA; an output voxel with any c_h NaN, < 0 or > n_h - 1 gets cval
 *   order  0: src[floor(c + 0.5)];  1: trilinear in float64, neighbours past the last voxel clamped
 *   dst    [dz][dy][dx], same dtype; float32 rounds to nearest, integers round half away from zero and saturate
 * No workspace; src and dst must not overlap.  Offsets are 64-bit (volumes above 2^31 voxels are fine). */
#define PM_RESAMPLE_F32 2
int pm_resample_affine(const void *src, int dtype, int sz, int sy, int sx, const double *M, int order, double cval,
                       void *dst, int dz, int dy, int dx, void *stream);

/* ---- thin-plate spline deformation (DESIGN §8 row 8) -------------------------------------------------------------
 * The smooth local deformation left after an affine registration: a smoothing thin-plate spline fitted to matched
 * nuclei, and volumes warped through it.  A spline with centres y [k][3] (zyx, float64, device), coefficients
 * c [k + 4][3] and shift_scale [6] = (shift[3], scale[3]) maps a point x to
 *   f(x) = sum_{i<k} c_i * (-||x - y_i||) + c_k + sum_h c_{k+1+h} * (x_h - shift_h) / scale_h      (c_i = row i of c)
 * = scipy.interpolate.RBFInterpolator(y, d, kernel='linear', degree=1, smoothing) with scipy's shift = (min + max) / 2
 * and scale = (max - min) / 2 (0 -> 1) per axis, computed by the caller.  -||d|| is -sqrt((dz*dz + dy*dy) + dx*dx) in
 * float64 without FMA, correctly rounded; the sum runs over the centres in ascending order, one FMA per term, so
 * pm_spline_eval and pm_resample_spline give the same coordinate bits.  No workspace; outputs must not overlap inputs.
 *
 * pm_spline_system: the whole (k + 4) x (k + 4) float64 matrix [-R + smoothing I, P; P^T, 0] of the fit into lhs (row
 *   stride ld >= k + 4): R_ij = ||y_i - y_j||, P = [1, (y - shift) / scale]; smoothing finite and >= 0.
 * pm_spline_eval: out [n][3] = f(pts [n][3]).
 * pm_resample_spline: the volume warp.  For output voxel x (index zyx in dst) the source coordinate is f(x); src is
 *   sampled there exactly as pm_resample_affine does (cval outside or NaN, order 0 src[floor(c + 0.5)], order 1 clamped
 *   trilinear, the same casts and dtypes, 64-bit offsets). */
int pm_spline_system(const double *centres, int k, const double *shift_scale, double smoothing, double *lhs, long long ld,
                     void *stream);
int pm_spline_eval(const double *centres, const double *coeffs, int k, const double *shift_scale, const double *pts,
                   long long n, double *out, void *stream);
int pm_resample_spline(const void *src, int dtype, int sz, int sy, int sx, const double *centres, const double *coeffs,
                       int k, const double *shift_scale, int order, double cval, void *dst, int dz, int dy, int dx,
                       void *stream);

/* ---- nuclei detection: scale-space LoG (SURVEY §2 row 10) --------------------------------------------------
 * DetectNuclei / find_spheres (platymatch/detect_nuclei/ss_log.py:25-87).  The contract is this project's own
 * (DESIGN §8 row 6; the reference's parameters are not available and agreement with it is unverified):
 * L_k = float32(sigma_k^2) * gaussian_laplace(img, (sigma_k / a, sigma_k, sigma_k)) as 8 separable passes, (value,
 * index) minima over 3x3x3x3 above 0.2 x Otsu, greedy sphere-overlap suppression.  Offsets are 64-bit.
 *
 * pm_detect_pass: one 1-D correlation of src [nz][ny][nx] float32 along `axis` (0 z, 1 y, 2 x) with the symmetric
 *   float64 weights w[0..lw] (centre, then offsets 1..lw; device), mode 'reflect', float64 accumulation in scipy's
 *   order (centre, then tap pairs outermost first), float32 result.  t0, t1 non-NULL: dst = scale * ((t0 + t1) + v)
 *   in float32 (the Laplacian's sum and scale-normalisation).  lw <= 384; src, t0, t1 must not overlap dst. */
int pm_detect_pass(const float *src, int nz, int ny, int nx, int axis, const double *weights, int lw, const float *t0,
                   const float *t1, float scale, float *dst, void *stream);
/* pm_detect_otsu: out[0] = skimage's threshold_otsu(img, nbins=256) (np.histogram binning of float32 data with float32
 *   edges, float64 statistics, first maximum; a constant image gives its value), out[1] = factor * out[0]; device. */
size_t pm_detect_otsu_workspace_bytes(void);
int pm_detect_otsu(const float *img, size_t n, double factor, double *out, void *workspace, size_t workspace_bytes,
                   void *stream);
/* pm_detect_minima: scale k's candidates.  l_prev / l_next are L_{k-1} / L_{k+1} (NULL = absent).  A voxel whose
 *   (L, linear index in (k, z, y, x) order) is strictly smaller than that of every present neighbour of its 3x3x3x3
 *   neighbourhood, and with -(double)L > threshold[1], is appended: keys[pos] = linear index, values[pos] = L, pos from
 *   *count (uint64, device, accumulated across calls; the caller zeroes it).  *count > capacity: the candidates past
 *   capacity were not stored; retry with more.  At most one candidate lies in any 2x2x2x2 block. */
int pm_detect_minima(const float *l_prev, const float *l_cur, const float *l_next, int nz, int ny, int nx, int k,
                     const double *threshold, long long capacity, long long *keys, float *values,
                     unsigned long long *count, void *stream);
/* pm_detect_suppress: keys [capacity] sorted by priority, the first min(*count, capacity) are the candidates.  Each is a
 *   sphere at (z * anisotropy, y, x) of radius radii[k] (device, every radius <= max_radius).  In priority order a
 *   candidate is kept unless its lens volume with an already kept sphere is greater than overlap x the smaller
 *   sphere's volume (float64, no FMA; same formula as ss_log.sphere_intersection).  state[i] = 1 kept, 2 dropped.
 *   workspace: pm_detect_suppress_workspace_bytes(capacity, nz, ny, nx, max_radius, anisotropy). */
size_t pm_detect_suppress_workspace_bytes(long long capacity, int nz, int ny, int nx, double max_radius,
                                          double anisotropy);
int pm_detect_suppress(const long long *keys, const unsigned long long *count, long long capacity, int nz, int ny,
                       int nx, const double *radii, double max_radius, double anisotropy, double overlap,
                       unsigned char *state, void *workspace, size_t workspace_bytes, void *stream);

/* ---- Euclidean distance matrix (SURVEY §8f row 3) ----------------------------------------------
 * scipy.spatial.distance.cdist as called by EvaluateMetrics._calculate_metrics (_dock_widget.py:1032,
 * 1038,1050): out[i * ldo + j] = ||a_i - b_j|| (float64 arithmetic, stored as the float32 costs the
 * assignment kernel consumes).  a [n1][3], b [n2][3] float64. */
int pm_cdist(const double *a, int n1, const double *b, int n2, float *out, int ldo, void *stream);

/* ---- K1  mean pairwise distance -------------------------------------------------------------
 * get_mean_distance (utils.py:58-75): mean of ||p_i - p_j|| over unordered pairs.  Deterministic
 * (fixed-order two-level reduction).  out_mean: 1 float64 on device.
 * workspace: pm_mean_distance_workspace_bytes(n) bytes on device. */
size_t pm_mean_distance_workspace_bytes(int n);
int pm_mean_distance(const double *pts, int n, double *out_mean, void *workspace, size_t workspace_bytes,
                     void *stream);

/* ---- K2  3D log-polar shape-context histograms ------------------------------------------------
 * get_unary / transform / get_shape_context / get_bin_index (shape_context.py:144-188, :61-84,
 * :10-42, :46-58).  For every nucleus builds the local frame (z radial from `centroid`, x = x0
 * Gram-Schmidt'ed against z, y = z x x) and bins all other nuclei: r/mean_dist against r_edges
 * (ring n_redges-1 open-ended), theta = acos(c/r) // (pi/6), phi = atan2 wrapped // (pi/6), linear
 * index un-clamped, indices outside 0..359 and NaN dropped — float64 throughout, numpy `//` semantics.
 * n_variants = 2 ('moving': sc, sc2) or 4 ('fixed': sc, sc2, sc3, sc4) or 1 (sc only).
 *   centroid   3 float64 (device)     x0  3 float64 (device)    mean_dist 1 float64 (device)
 *   r_edges    n_redges float64 (device) — numpy's logspace(log10(1/8), log10(2), 5) doubles
 *   counts     [n_variants][rows][360] uint32  integer histograms (reference row = counts / row sum)
 *   dropped    [n_variants][rows] uint32       neighbours not counted (overflow bins / NaN)
 *   edge_ties  [1] uint64, accumulated: neighbours whose r, theta or phi lies within 64 ulp of a
 *              bin edge (where another libm could decide differently); may be NULL.
 * Only the query nuclei [row_begin, row_end) are described, rows = row_end - row_begin (0, n for the whole
 * cloud; descriptor rows shard across GPUs, SURVEY §8e). */
int pm_shape_context_hist_rows(const double *pts, int n, const double *centroid, const double *x0,
                               const double *mean_dist, const double *r_edges, int n_redges, int n_variants,
                               int row_begin, int row_end, uint32_t *counts, uint32_t *dropped,
                               unsigned long long *edge_ties, void *stream);

/* ---- K3  chi^2 histogram-distance cost matrix ---------------------------------------------------
 * get_unary_distance (shape_context.py:88-99) over all pairs (_dock_widget.py:547-602):
 * cost[i][j] = 0.5 * sum_k (a_ik - b_jk)^2 / (a_ik + b_jk), equal bins skipped.  Packed FP32,
 * register tiled, two bins per reciprocal, structurally empty bins skipped per warp (16 rows x 128
 * columns).
 *
 * pm_chi2_operand prepares one cloud's histograms for either side of the matrix:
 *   out   [361][ld] float32 bin-major, ld = n rounded up to 128: count / row total (one rounding);
 *         empty bins, pad columns and the extra "null bin" row 360 hold PM_CHI2_EPS (2^-60), which
 *         makes equal-and-empty bins contribute exactly 0 without a branch
 *   mask  [ld/128][12] uint32: bit k of block q = some histogram in rows [128q, 128q+128) has a
 *         non-empty bin k
 *   fine  [ld/16][12] uint32: the same per block of 16 rows
 * pm_chi2_cost writes rows [row_begin,row_end) of the n1 x n2 matrix to cost + (i - row_begin) * ldc
 * (row sharding across GPUs: each rank passes its own 128-aligned range and buffer).  a_fine is the row
 * side's fine mask, b_mask the column side's 128-block mask. */
#define PM_CHI2_EPS 8.673617379884035e-19f
int pm_chi2_operand(const uint32_t *counts, int n, float *out, int ld, uint32_t *mask, uint32_t *fine, void *stream);
/* same from already-normalised float32 histograms [n][360] (values <= 0 count as empty) */
int pm_chi2_operand_f32(const float *hist, int n, float *out, int ld, uint32_t *mask, uint32_t *fine, void *stream);
int pm_chi2_cost(const float *a_t, int lda, const uint32_t *a_fine, int n1, const float *b_t, int ldb,
                 const uint32_t *b_mask, int n2, int row_begin, int row_end, float *cost, int ldc, void *stream);

/* ---- K4  linear sum assignment ------------------------------------------------------------------
 * Replaces scipy.optimize.linear_sum_assignment at _dock_widget.py:604-611 for nr <= nc
 * (the host mirror transposes otherwise, as scipy does).  Exact, two phases: an epsilon = 0 auction
 * (keeps complementary slackness exactly) followed by shortest augmenting paths with float64 duals
 * for the rows the auction parks — optimal for the float32 matrix given.
 * Problems with few or no slack columns (nc - nr <= 2 % of nc: specimens of equal size) are solved as
 * a square problem with nc - nr zero-cost dummy rows: truncated eps-scaling phases of the same auction
 * prepare the prices, then an exact finish (tight filter, epsilon = 0 auction, augmenting paths)
 * restores exact complementary slackness: same optimum, same call.  The statistics then count the
 * dummy rows as well (rows_after_bidding, augmentations).
 *   algorithm  PM_LAP_ALGO_AUTO picks the sparse asynchronous auction (certified candidate lists,
 *              prices in shared memory) whenever the column prices fit in shared memory, else the
 *              dense grid-wide auction; max_bid_rounds = 0 skips the auction (pure augmenting paths);
 *              for the sparse auction a "round" is a budget of one bid per row
 *   cost     [batch][nr][ldc] float32, ldc >= nc
 *   col4row  [batch][nr] int32 out (column assigned to each row; rows are implicitly 0..nr-1)
 *   total    [batch] float64 out: sum of assigned costs
 *   stats    [batch][PM_LAP_STATS] int64 out, may be NULL (see PM_LAP_STAT_*)
 * workspace: pm_lap_workspace_bytes(batch, nr, nc). */
#define PM_LAP_STATS 16
#define PM_LAP_STAT_BID_ROUNDS 0 /* dense: rounds run; sparse: largest number of bids made by one warp */
#define PM_LAP_STAT_ROWS_AFTER_BIDDING 1
#define PM_LAP_STAT_AUGMENTATIONS 2
#define PM_LAP_STAT_DIJKSTRA_STEPS 3
#define PM_LAP_STAT_STATUS 4 /* 0 ok, -4 infeasible */
#define PM_LAP_STAT_BIDS 5      /* sparse auction: bids committed or parked */
#define PM_LAP_STAT_REFRESHES 6 /* sparse auction: candidate lists rebuilt from the dense row */
#define PM_LAP_STAT_RETRIES 7   /* sparse auction: bids recomputed because the price moved */
#define PM_LAP_STAT_PARKED 8          /* sparse auction: rows parked for phase 2 (zero-increment steals) */
#define PM_LAP_STAT_REFRESH_CYCLES 9  /* sparse auction: SM cycles spent rebuilding lists, summed over warps */
#define PM_LAP_STAT_AUCTION_CYCLES 10 /* sparse auction: SM cycles of the longest-running warp */
#define PM_LAP_STAT_BULK_BIDS 11      /* sparse auction: bids made by the multi-SM bulk kernel */
#define PM_LAP_STAT_SAP_DENSE_RELAX 12 /* sparse augmenting paths: tree rows that had to be relaxed densely */
#define PM_LAP_STAT_PATH 13           /* kernels this solve ran: PM_LAP_PATH_* bits */
#define PM_LAP_STAT_SAP_CYCLES 14     /* sparse augmenting paths: SM cycles of pm_lap_sap_sparse_kernel, entry to exit */
/* path bits: squared with dummy rows; the auction that ran (neither bit: max_bid_rounds = 0, augmenting paths only);
 * exactly one finishing kernel; the sparse auction's ring of displaced rows in shared memory (else global memory) */
#define PM_LAP_PATH_SQUARED 1
#define PM_LAP_PATH_SPARSE_AUCTION 2
#define PM_LAP_PATH_DENSE_AUCTION 4
#define PM_LAP_PATH_SAP_SPARSE 8   /* augmenting paths over the candidate lists (pm_lap_sap_sparse_kernel) */
#define PM_LAP_PATH_SAP_DENSE8 16  /* dense augmenting paths, 8 columns per thread, prices in registers */
#define PM_LAP_PATH_SAP_DENSE16 32 /* dense augmenting paths, 16 columns per thread */
#define PM_LAP_PATH_SAP_DENSE24 64 /* dense augmenting paths, 24 columns per thread */
#define PM_LAP_PATH_RING_SMEM 128
#define PM_LAP_ALGO_AUTO 0
#define PM_LAP_ALGO_SPARSE_AUCTION 1
#define PM_LAP_ALGO_DENSE_AUCTION 2
size_t pm_lap_workspace_bytes(int batch, int nr, int nc);
int pm_lap_solve(const float *cost, int batch, int nr, int nc, int ldc, int max_bid_rounds, int algorithm,
                 int32_t *col4row, double *total, int64_t *stats, void *workspace, size_t workspace_bytes,
                 void *stream);

/* ---- K5  affine RANSAC ---------------------------------------------------------------------------
 * do_ransac (shape_context.py:103-139) with get_affine_transform (find_transform.py:4-17) on the
 * sampled pairs and apply_affine_transform (apply_transform.py:3-17) + inlier count on all pairs.
 *   moving, fixed   [k][3] float64, already in correspondence order (_dock_widget.py:622-623)
 *   sample_idx      [trials][min_samples] int32 (device) or NULL -> drawn on device from `seed`
 *                   (Philox counter RNG, distinct indices per trial)
 *   best_A [16] float64, best_inliers [1] int32, best_trial [1] int32  (first strictly-better trial;
 *   A = all ones and inliers = 0 if no trial has an inlier, as the reference)
 *   inliers_per_trial  [trials] int32 out, may be NULL.
 * workspace: pm_ransac_workspace_bytes(trials). */
size_t pm_ransac_workspace_bytes(int trials);
/* do_ransac with its `transform` argument: PM_TRANSFORM_AFFINE fits get_affine_transform on the sampled pairs
 * (degenerate samples: pinv's minimum-norm answer), PM_TRANSFORM_SIMILAR fits get_similar_transform
 * (find_transform.py:21-99, Horn's closed form with the eigenvector of the largest eigenvalue). */
int pm_ransac(const double *moving, const double *fixed, int k, const int32_t *sample_idx, int trials, int min_samples,
              double error, unsigned long long seed, int transform, double *best_A, int32_t *best_inliers,
              int32_t *best_trial, int32_t *inliers_per_trial, void *workspace, size_t workspace_bytes, void *stream);

/* ---- K6  ICP with affine re-fit -------------------------------------------------------------------
 * perform_icp (perform_icp.py:7-26): `iterations` x { nearest fixed point per moving point (first
 * minimum wins), least-squares affine over all pairs (find_transform.py:4-17 = F M^T (M M^T)^-1),
 * apply, compose }.  Always exactly `iterations` iterations.
 *   moving [n1][3] float64 — NOT modified;  fixed [n2][3] float64
 *   A_icp [16] float64 out; residuals [iterations] float64 out (mean ||moving' - fixed[nn]||,
 *   get_error utils.py:77-88), may be NULL;  nn_out [n1] int32 last nearest-neighbour map, may be NULL.
 * Nearest neighbours come from a uniform grid over the fixed cloud (exact, ~50x fewer candidates); fewer than 256
 * fixed points are searched by brute force.
 * workspace: pm_icp_workspace_bytes2(n1, n2), else PM_ERR_WORKSPACE. */
size_t pm_icp_workspace_bytes2(int n1, int n2);
/* perform_icp with its `transform` argument (re-fit = get_affine_transform or get_similar_transform, :17-20) */
int pm_icp(const double *moving, int n1, const double *fixed, int n2, int iterations, int transform, double *A_icp,
           double *residuals, int32_t *nn_out, void *workspace, size_t workspace_bytes, void *stream);

/* ---- small ops -------------------------------------------------------------------------------------
 * get_affine_transform (find_transform.py:4-17) = fixed_h @ pinv(moving_h) for K >= 1 pairs: float64 normal
 * equations; rank-deficient point sets (coplanar keypoints, K < 4) get pinv's minimum-norm solution. */
int pm_fit_affine(const double *moving, const double *fixed, int k, double *A, void *stream);
/* get_similar_transform (find_transform.py:21-99): scale * rotation + translation by Horn's closed form. */
int pm_fit_similar(const double *moving, const double *fixed, int k, double *A, void *stream);
/* np.argmax(inliers) of the pipeline (_dock_widget.py:683-703), on the device: best[0] = first maximum of
 * inliers[n_hyp], A_best[16] = A_all[best] ([n_hyp][16]). */
int pm_select_best(const int32_t *inliers, const double *A_all, int n_hyp, int32_t *best, double *A_best, void *stream);
/* apply_affine_transform (apply_transform.py:3-17): out[i] = (A [p_i;1])[:3];  in-place allowed. */
int pm_apply_affine(const double *pts, int n, const double *A, double *out, void *stream);
/* out[i] = pts[index[i]] (the reordering moving[:, row_ind] / fixed[:, col_ind], _dock_widget.py:622-623) */
int pm_gather_points(const double *pts, const int32_t *index, int k, double *out, void *stream);
/* C = A @ B for 4x4 float64 (icp @ sc, _dock_widget.py:428) */
int pm_compose(const double *A, const double *B, double *C, void *stream);

/* ---- peer-memory windows (multi-GPU, SURVEY §8e; the reference is single-process) ---------------------
 * A window is a cudaMalloc allocation exported with CUDA IPC so that the chi^2 kernels of the OTHER ranks of the
 * box store their cost-matrix rows straight into the owner's matrix over NVLink (pm_chi2_cost with the mapped
 * address as its output pointer).  handle64: PM_PEER_HANDLE_BYTES opaque bytes to pass between processes. */
#define PM_PEER_HANDLE_BYTES 64
int pm_peer_alloc(size_t bytes, void **ptr);
int pm_peer_free(void *ptr);
int pm_peer_export(void *ptr, unsigned char *handle64);
int pm_peer_open(const unsigned char *handle64, void **ptr);
int pm_peer_close(void *ptr);

/* ---- host-buffer entry points (numpy callers; copy in, run, copy out, synchronise) ----------------- */
/* get_mean_distance (utils.py:58-75) */
int pm_host_mean_distance(const double *pts, int n, int device, double *out_mean);
/* get_unary (shape_context.py:144-188): counts [n_variants][n][360] uint32, dropped [n_variants][n],
 * x0_out[3] (PCA axis used), edge_ties_out (may be NULL). */
int pm_host_shape_context(const double *pts, int n, const double *centroid, double mean_dist,
                          const double *r_edges, int n_redges, int n_variants, int device, uint32_t *counts,
                          uint32_t *dropped, double *x0_out, unsigned long long *edge_ties_out);

#ifdef __cplusplus
}
#endif
#endif /* PLATYMATCH_B200_H */
