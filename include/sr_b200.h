/*
 * sr_b200.h — C ABI of the B200-native dense-matching hot path.
 *
 * This is the drop-in boundary a maintainer of thegedge/StereoReconstruction binds
 * to.  The reference has no FFI: its boundary is the C++ class API of stereo/ and
 * project/ (SURVEY.md §8b).  The C++ classes shipped in include/stereo, include/project
 * and include/util keep the reference's signatures and are implemented *only* by
 * packing their inputs into the POD structs below and calling these entry points.
 *
 * Every entry point cites the reference code it replaces (paths relative to the
 * reference tree).  Conventions:
 *   - plain pointers and sizes, no C++/torch types; every function returns an
 *     int status (SR_OK == 0) except the trivial getters;
 *   - no exceptions cross the ABI; sr_last_error() gives the message;
 *   - a context is bound to one CUDA device and is single-threaded;
 *   - "host" pointers are ordinary (pageable or pinned) host memory, borrowed for
 *     the duration of the call;
 *   - there is NO CPU fallback: without a usable CUDA device sr_ctx_create fails.
 */
#ifndef SR_B200_H
#define SR_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SR_OK 0
#define SR_ERR_INVALID 1   /* bad argument                                  */
#define SR_ERR_CUDA 2      /* CUDA runtime error (see sr_last_error)        */
#define SR_ERR_STATE 3     /* call made before its prerequisites            */
#define SR_ERR_CANCELLED 4 /* sr_request_cancel() observed between launches */
#define SR_ERR_NCCL 5      /* NCCL error                                    */
#define SR_ERR_NOMEM 6

/* Weight functor selected by typedef in the reference
 * (stereo/twoviewstereo.cpp:84, stereo/multiviewstereo.cpp:109). */
#define SR_WEIGHT_ADAPTIVE 0 /* stereo/adaptiveweight.cpp:33-79   */
#define SR_WEIGHT_GEODESIC 1 /* stereo/geodesicweight.cpp:49-131  */

/* Matching cost. */
#define SR_COST_NCC_TWOVIEW 0 /* stereo/twoviewstereo.cpp:909-977  (lower is better)  */
#define SR_COST_NCC_MVS 1     /* stereo/multiviewstereo.cpp:113-189 (higher is better) */
#define SR_COST_SAD_TWOVIEW 2 /* stereo/twoviewstereo.cpp:864-905  (lower is better)  */

/* depthFromLabel variants. */
#define SR_DEPTH_LINEAR 0 /* stereo/multiviewstereo.cpp:733-736 */
#define SR_DEPTH_INV5 1   /* stereo/twoviewstereo.cpp:981-985   */

/* Selection rule applied by the fused aggregate+WTA kernel. */
#define SR_SELECT_TWOVIEW 0 /* first strict minimum with 1e-10 margin + second-best
                               ratio test, stereo/twoviewstereo.cpp:293-305,320-325 */
#define SR_SELECT_MVS 1     /* max (ncc, depth) among ncc > threshold, else -1,
                               stereo/multiviewstereo.cpp:589-602,654-660          */

/* Integer sentinels of the depth-index map (extension; the reference keeps only
 * double depths: NaN / +INF / -1, stereo/twoviewstereo.hpp:41). */
#define SR_INDEX_NONE (-1)     /* no label selected (depth NaN two-view, -1 MVS)    */
#define SR_INDEX_MASKED (-2)   /* reference pixel outside its mask                  */
#define SR_INDEX_REJECTED (-3) /* second-best ratio test failed (depth +INF)        */

/* Camera POD == the state of project/camera.hpp:168-185 that the hot path reads.
 * All matrices row-major.  Derived members (Kinv, Rinv, C, prin_dir, flags) are
 * filled by the host Camera class exactly as project/camera.cpp:205-298,326-342
 * does, so the device never re-derives them. */
typedef struct sr_camera {
    double K[9];
    double Kinv[9];
    double R[9];
    double Rinv[9];
    double t[3];
    double C[3];
    double dist[5];     /* k1 k2 p1 p2 k3, project/project.cpp:143-147           */
    double plane_n[3];  /* unit interface normal, camera-local (util/plane.hpp:33) */
    double plane_d;     /* interface distance                                     */
    double n;           /* refractive index ratio far/camera-side                 */
    double prin_dir[3]; /* principleRay().direction(), global (camera.cpp:292-298) */
    int32_t is_refractive; /* n != 1 && plane_d != 0 (camera.cpp:329,339)         */
    int32_t is_distorted;  /* any |dist[i]| > 1e-10 (camera.cpp:305-309)          */
} sr_camera;

/* Runtime parameters.  Defaults (sr_params_default) are the reference's file-scope
 * constants: stereo/twoviewstereo.cpp:64-80, stereo/multiviewstereo.cpp:90-102. */
typedef struct sr_params {
    double min_depth;
    double max_depth;
    int32_t num_levels;   /* numDepthLevels                                       */
    double image_scale;   /* imageScale; images passed in are already scaled      */
    int32_t radius;       /* WINDOW_RADIUS: 5 two-view, 2 MVS                     */
    int32_t weight_kind;  /* SR_WEIGHT_*                                          */
    int32_t cost_kind;    /* SR_COST_*                                            */
    int32_t depth_kind;   /* SR_DEPTH_*                                           */
    int32_t select_kind;  /* SR_SELECT_*                                          */
    double second_best_factor; /* SECOND_BEST_FACTOR 0.95; <= 0 disables the test */
    double ncc_threshold;      /* 0.95, stereo/multiviewstereo.cpp:589            */
    int32_t keep_cost_volume;  /* bit 0: keep the FP32 cost volume for sr_get_cost_volume;
                                * bit 1: keep the K = 9 peak lists for sr_get_peaks (MVS selection) */
    int32_t row_begin;    /* rows [row_begin,row_end) of the reference view are     */
    int32_t row_end;      /* processed (row sharding); row_end <= 0 means height  */
} sr_params;

typedef struct sr_ctx sr_ctx;

/* ---- context ----------------------------------------------------------------*/
int sr_ctx_create(int device, sr_ctx **out);
void sr_ctx_destroy(sr_ctx *ctx);
const char *sr_last_error(const sr_ctx *ctx); /* ctx may be NULL: last create error */
/* Replaces Task::cancel()/isCancelled() polling (gui/task.hpp:71-80). */
void sr_request_cancel(sr_ctx *ctx);
void sr_clear_cancel(sr_ctx *ctx);
/* All work is enqueued on this stream (cudaStream_t passed as void*); NULL = the
 * context's own stream.  Lets a caller time with its own CUDA events. */
int sr_set_stream(sr_ctx *ctx, void *cuda_stream);
void sr_params_default(sr_params *p, int multi_view);
/* Number of kernels this context has launched since creation. */
int64_t sr_launch_count(const sr_ctx *ctx);
/* Per-stage device timing with CUDA events on the context stream (replaces the QTime
 * prints of stereo/twoviewstereo.cpp:260,333).  sr_get_stage_ms synchronises and returns
 * {build ms, match ms, build bands, match launches} accumulated since its last call. */
int sr_set_profiling(sr_ctx *ctx, int on);
int sr_get_stage_ms(sr_ctx *ctx, double *out4);
/* Debug counters of the screened MVS match kernel (FP32 screen + FP64 verify), accumulated since
 * sr_ctx_create when the environment has SR_MATCH_STATS=1: out8[0] pixels, [1] labels screened in
 * FP32, [2] labels forced to FP64, [3] FP64 verifications, [4] pixels evaluated in FP64 only,
 * [5] bit pattern (low 32 bits, IEEE float) of the largest |ncc32 - ncc64| seen on a verified label,
 * [6] verified labels whose FP32 value lay outside its error bar (must be 0),
 * [7] reserved, always 0. */
int sr_get_match_stats(sr_ctx *ctx, uint64_t *out8);
/* Self-check counters of the refractive tap-volume build (same switch, SR_MATCH_STATS=1): with
 * the switch on, every interpolated label is ALSO projected exactly.  out4[0] labels taken from
 * the anchor interpolation, [1] labels that fell back to the exact projection because the
 * interpolated coordinate was within the guard of a pixel boundary, [2] interpolated labels
 * whose integer tap differs from the exact projection's (must be 0). */
int sr_get_build_stats(sr_ctx *ctx, uint64_t *out4);

/* ---- inputs -----------------------------------------------------------------*/
/* Replaces the image/mask ingestion of TwoViewStereo::TwoViewStereo
 * (stereo/twoviewstereo.cpp:89-124) and MultiViewStereo::initialize
 * (stereo/multiviewstereo.cpp:193-247): V views of w*h RGBA8 (byte order R,G,B,A,
 * the channels VectorImage::fromQImage extracts, util/vectorimage.cpp:57-64) and
 * one mask byte per pixel (255 == WHITE, anything else is not).  mask8[i] may be
 * NULL (all WHITE).  rgba8[i] may be NULL for a view this context only needs the
 * camera of (multi-GPU: a view another rank computes and that is no neighbour of this
 * rank's views); using such a view as reference or neighbour is an error.  Copies straight from the caller's
 * buffers to the device on the context stream (cudaMemcpyAsync: truly asynchronous when the caller's memory is
 * pinned, staged by the driver when it is pageable; the buffers may be reused when the call returns only in the
 * pageable case — keep pinned buffers alive until sr_synchronize) and runs the per-view preparation kernels. */
int sr_set_views(sr_ctx *ctx, int num_views, const sr_camera *cams,
                 const uint8_t *const *rgba8, const uint8_t *const *mask8, int w, int h);
int sr_set_params(sr_ctx *ctx, const sr_params *p);

/* ---- the hot path -----------------------------------------------------------*/
/* Cost-volume build + support-weight aggregation + WTA for reference view `ref`
 * against `num_nbrs` neighbour views.  Replaces the label sweep of
 * TwoViewStereo::computeCostVolumes (stereo/twoviewstereo.cpp:265-332, 436-500)
 * and, with SR_SELECT_MVS, the per-pixel search of
 * MultiViewStereo::computeInitialEstimate (stereo/multiviewstereo.cpp:543-604,654-660)
 * restated over depth labels.  Asynchronous; results stay on the device. */
int sr_run_view(sr_ctx *ctx, int ref, const int32_t *nbrs, int num_nbrs);
/* Curve-mode search: rasterised refractive epipolar curve, exactly the live path
 * of the reference (stereo/multiviewstereo.cpp:574-602,754-810 and
 * stereo/twoviewstereo.cpp:285-305,999-1054).  The candidates of a pixel are the WHITE-mask
 * pixels of the Bresenham segments joining consecutive label projections; a candidate's depth is
 * the z of the midpoint of the two viewing rays' closest approach.  Results: sr_get_depth (the
 * winner's depth hypothesis; -1 / NaN / +INF sentinels as in label mode), sr_get_best_cost, and
 * sr_get_depth_index = ordinal of the winning candidate along the concatenated curves (>= 0), or
 * the sentinels.  keep_cost_volume is not available in this mode. */
int sr_run_view_curve(sr_ctx *ctx, int ref, const int32_t *nbrs, int num_nbrs);
/* Neighbour selection of MultiViewStereo::runTask (stereo/multiviewstereo.cpp:335-360).
 * out_nbrs has room for max_nbrs entries per view; out_counts[v] receives the count. */
int sr_select_neighbours(sr_ctx *ctx, int max_nbrs, int32_t *out_nbrs, int32_t *out_counts);
/* crossCheck: stereo/twoviewstereo.cpp:596-672 (two_view != 0: both directions,
 * failing pixels -> +INF) or stereo/multiviewstereo.cpp:666-729 (any other view may
 * confirm; failing pixels -> NaN).  Operates on the device-resident depth maps. */
int sr_cross_check(sr_ctx *ctx, int two_view, double threshold);
/* Consecutive sr_run_view calls alternate between two internal streams (so that one view's last,
 * partially filled wave of blocks overlaps the next view's launches; SR_LANES=1 turns this off).
 * Every other entry point first orders that work before the context stream; a caller that times
 * or synchronises with ITS OWN events on the stream of sr_set_stream calls sr_flush() first: it makes
 * the context stream wait for all views enqueued so far, without blocking the host.  sr_synchronize
 * blocks the host until everything is done.  (Replaces the tbb::parallel_for join of
 * stereo/multiviewstereo.cpp:548-556.) */
int sr_flush(sr_ctx *ctx);
int sr_synchronize(sr_ctx *ctx);

/* ---- results (device -> host) ----------------------------------------------*/
/* Depth-label index map, int32 w*h (extension, see SR_INDEX_*); after sr_mrf_select, the chosen
 * peak-list slot 0..8. */
int sr_get_depth_index(sr_ctx *ctx, int view, int32_t *out);
/* computedDepth* / computedDepths[view] (stereo/twoviewstereo.hpp:41,
 * stereo/multiviewstereo.hpp:106-107): doubles with NaN / +INF / -1 sentinels. */
int sr_get_depth(sr_ctx *ctx, int view, double *out);
/* Best cost per pixel (min cost two-view, max ncc MVS), double w*h. */
int sr_get_best_cost(sr_ctx *ctx, int view, double *out);
/* The cost volume of the last sr_run_view with keep_cost_volume, float
 * [nbr][d][row - row_begin][x] (label-major planes, the layout the kernels stream);
 * NaN where the label could not be evaluated. */
int sr_get_cost_volume(sr_ctx *ctx, float *out, size_t out_elems);
/* The K = 9 largest (ncc, depth) pairs of every pixel of the last sr_run_view or
 * sr_run_view_curve with keep_cost_volume & 2, ascending, padded with (0, -1):
 * CostFunction::peakPairs, the input of the reference's MRF stage
 * (stereo/multiviewstereo.cpp:479-482,562,583-602).  out = h*w*9*2 doubles,
 * [pixel][k][ncc, depth]; in curve mode depth is the z of the rays' closest approach (:583-588).
 * Evaluates every candidate in FP64. */
int sr_get_peaks(sr_ctx *ctx, int view, double *out);
/* Replaces depth upload for cross-check under view sharding (each rank receives
 * the other ranks' depth maps before sr_cross_check). */
int sr_set_depth(sr_ctx *ctx, int view, const double *depth);
/* colorFromDepth + depthMap(view) of stereo/multiviewstereo.cpp:257-286: gray ramp,
 * masked -> WHITE.  RGBA8 w*h*4 out.  mvs must be nonzero: mvs == 0 returns SR_ERR_INVALID,
 * because the two-view HSV ramp (stereo/twoviewstereo.cpp:128-146, QColor semantics) is
 * coloured on the host by the two-view class. */
int sr_get_depth_image(sr_ctx *ctx, int view, int mvs, uint8_t *rgba8_out);
/* The coloured point cloud of `view`'s current depth map (the input of outputPLYFile,
 * stereo/multiviewstereo.cpp:291-315).  For every pixel (x, y) whose depth d is finite and
 * d + 1e-5 >= min_depth of the last sr_set_params: the intersection of
 * Camera::unproject((x + .5) / image_scale, (y + .5) / image_scale) with the plane through C + d n,
 * n = principleRay().direction() (pointFromDepth, :740-750; pixels whose intersection fails are
 * skipped), and the pixel's R, G, B.  Points come in row-major pixel order, whatever wrote the map
 * (a run, sr_cross_check, sr_set_depth, a gather) and whichever sentinels it holds.
 * out_xyz = 3 * capacity doubles, out_rgb = 3 * capacity bytes, out_pixel = capacity pixel indices
 * y * w + x (may be NULL).  *out_count receives the number of points; capacity 0 (pointers NULL)
 * only counts.  SR_ERR_INVALID when capacity < count (*out_count is set, nothing else written);
 * SR_ERR_STATE for a view without an image or before sr_set_params. */
int sr_get_points(sr_ctx *ctx, int view, int64_t capacity, double *out_xyz, uint8_t *out_rgb,
                  int32_t *out_pixel, int64_t *out_count);
/* One fused point cloud from the current depth maps of all V views, read as a snapshot (no map is
 * modified, no view sees another's result; whatever wrote them does not matter), with the views'
 * images and cameras and min_depth and image_scale s of the last sr_set_params.
 *   1. Points.  The point of pixel (v, x, y) is the one sr_get_points gives it (finite d with
 *      d + 1e-5 >= min_depth, the ray of Camera::unproject((x + .5) / s, (y + .5) / s) meeting the
 *      plane through C + d n, n = prin_dir); a pixel whose intersection fails has none.
 *   2. Agreement.  Let X be the point of source pixel p of view v.  Another view u agrees with p when
 *      cam_project(u, X) succeeds, the projection times s is (x2, y2) with 0 <= x2 < w and
 *      0 <= y2 < h, the pixel q = ((int)x2, (int)y2) of u has a point X_u (taken at q's centre), and
 *      |X - X_u| is finite and < max_dist.  A(p) is the set of agreeing views, support(p) = |A(p)|.
 *   3. Kept: support(p) >= min_views.
 *   4. Emitted once: a kept p is emitted unless a view u in A(p) with u < v has its pixel q kept, so a
 *      surface sample belongs to the lowest view that keeps it.  Agreement is not symmetric, so this is
 *      not an exact one-to-one matching: two points of one surface sample can both be emitted.
 *   5. Fused point: the FP64 sum of X and then the X_u of u in A(p) ascending, divided by
 *      n = 1 + support(p); colour per channel (sum + n / 2) / n in integers over the same pixels.
 *   6. Order: view-major, row-major pixel order within a view.
 * With max_dist = 0 and min_views = 0 the result is the concatenation of sr_get_points over the views.
 * The buffers follow sr_get_points: out_xyz = 3 * capacity doubles, out_rgb = 3 * capacity bytes,
 * out_source = 2 * capacity int32 (view, y * w + x) (may be NULL); capacity 0 (pointers NULL) only
 * counts.  SR_ERR_INVALID when capacity < count (*out_count is set, nothing else written), for a
 * NULL out_count, a capacity > 0 without xyz or rgb, max_dist negative or not finite, or
 * min_views < 0 (min_views > V - 1 is legal and gives no points).  SR_ERR_STATE without views or
 * params, or when a view was given no image.  Scratch: 32 bytes per pixel of each view. */
int sr_fuse_points(sr_ctx *ctx, double max_dist, int min_views, int64_t capacity, double *out_xyz,
                   uint8_t *out_rgb, int32_t *out_source, int64_t *out_count);

/* ---- MRF stage on the peak lists --------------------------------------------*/
/* The second stage of the multiple-hypothesis multi-view stereo the reference implements only in part
 * (stereo/multiviewstereo.cpp:22-27): a Markov random field over the in-mask pixels (mask byte 255) of
 * one view, 4-connected, whose labels are the 9 slots of a pixel's peak list plus U ("unknown").  A slot
 * is a hypothesis when its ncc and depth are finite and it is not the padding (0, -1); other slots cannot
 * be chosen.  With thr = ncc_threshold and step = (max_depth - min_depth) / (num_levels - 1) of the last
 * sr_set_params:
 *   D(k)    = max(0, (1 - ncc_k) / (1 - thr))            (FP64, rounded to FP32 once)
 *   D(U)    = unknown_cost
 *   V(k, l) = smooth_weight * min(|z_k - z_l|, smooth_trunc), z = depth / step (FP64, rounded to FP32
 *             once and clamped to the finite FP32 range), so the truncation is in label steps
 *   V(k, U) = V(U, k) = unknown_pair,  V(U, U) = 0.
 * Solver: min-sum loopy belief propagation with FP32 messages on a checkerboard schedule; one iteration
 * updates the messages sent by the pixels with (x + y) even, then by those with (x + y) odd.  The final
 * label is argmin D + the four incoming messages; the highest hypothesis slot wins a tie, U loses every
 * tie.  iterations = 0 gives the argmin of the unary term. */
typedef struct sr_mrf_params {
    int32_t iterations;    /* checkerboard iterations (both colours); 0 = argmin of the unary term */
    double unknown_cost;   /* D(U)                                                    */
    double smooth_weight;  /* V(k,l) = smooth_weight * min(|dz| / step, smooth_trunc) */
    double smooth_trunc;   /* label steps                                             */
    double unknown_pair;   /* V(k,U) = V(U,k); V(U,U) = 0                             */
} sr_mrf_params;
void sr_mrf_params_default(sr_mrf_params *p);
/* Uploads peak lists for `view` (peaks = h*w*9*2 doubles, [pixel][k][ncc, depth], the layout of
 * sr_get_peaks), replacing the lists the context keeps; sr_get_peaks and sr_mrf_select then read them.
 * Any values are accepted: lists need not be sorted, and slots that are no hypothesis are skipped. */
int sr_set_peaks(sr_ctx *ctx, int view, const double *peaks);
/* Runs the MRF on the device-resident peak lists of `view` (a run with keep_cost_volume & 2, or
 * sr_set_peaks) and writes that view's maps in place, on in-mask pixels only: depth = the chosen
 * hypothesis's depth from the list (or -1 for U), best cost = its ncc (or 0), and the index map = the
 * chosen SLOT 0..8 of the peak list (or SR_INDEX_NONE) -- after the MRF the index is a slot, not a depth
 * label.  The peak lists are not modified.  out_energy (may be NULL) receives the energy of the final
 * labelling: its FP32 unary and pairwise terms summed in FP64 in a fixed order.
 * SR_ERR_STATE: no views, no params, or no peak lists for `view`.  SR_ERR_INVALID: a parameter negative
 * or not finite, unknown_cost, unknown_pair or smooth_weight * smooth_trunc above 1e30 (which keeps every
 * FP32 sum finite), iterations < 0, ncc_threshold >= 1 or not finite, max_depth <= min_depth, or a row
 * band in the params (the MRF needs the whole view).  SR_ERR_CANCELLED: sr_request_cancel observed
 * between iterations; the maps are then left as they were. */
int sr_mrf_select(sr_ctx *ctx, int view, const sr_mrf_params *p, double *out_energy);

/* ---- building blocks exposed for the C++ class API and the parity tests -----*/
/* Camera::unproject on every pixel centre ((x+.5)/scale,(y+.5)/scale)
 * (project/camera.cpp:423-459): out = w*h*6 doubles (source xyz, direction xyz). */
int sr_unproject_grid(sr_ctx *ctx, int view, double *out_rays);
/* Camera::project (project/camera.cpp:380-419) for n global points: out_xy = 2n
 * doubles, out_ok = n flags. */
int sr_project_points(sr_ctx *ctx, int view, int n, const double *xyz, double *out_xy,
                      int32_t *out_ok);
/* The residual of the refractive-interface calibration, RefractiveCalibrationFunction::diff
 * (stereo/refractioncalibration.cpp:175-201), for n correspondences: view_pairs = 2n camera
 * indices into cams[num_cams], pixels = n * (x1, y1, x2, y2); out[i] = distance of the two
 * unprojected rays scaled by 0.5*fx/z in both views.  Independent of sr_set_views; the
 * Levenberg-Marquardt loop around it (util/lm.cpp) stays on the host. */
int sr_calibration_residuals(sr_ctx *ctx, int num_cams, const sr_camera *cams, int n,
                             const int32_t *view_pairs, const double *pixels, double *out);
/* The same for num_models camera sets in one launch: cams = num_models * num_cams PODs
 * (set m at cams + m*num_cams), out = num_models * n residuals.  One Levenberg-Marquardt
 * step of the interface calibration evaluates the current model and the two finite-difference
 * perturbations of every free parameter (RefractiveCalibrationFunction::gradient,
 * stereo/refractioncalibration.cpp:203-236) this way; include/stereo/refractioncalibration.hpp
 * is the caller. */
int sr_calibration_residuals_batch(sr_ctx *ctx, int num_models, int num_cams, const sr_camera *cams,
                                   int n, const int32_t *view_pairs, const double *pixels, double *out);
/* AdaptiveWeight/GeodesicWeight::init_weights for n window centres
 * (stereo/adaptiveweight.cpp:47-58, stereo/geodesicweight.cpp:59-131):
 * out = n * (2r+1)^2 doubles, [row+r][col+r] as operator()(row,col) indexes. */
int sr_compute_weights(sr_ctx *ctx, int view, int weight_kind, int radius, int n,
                       const int32_t *cx, const int32_t *cy, double *out);

/* ---- multi-GPU (one process per GPU) ---------------------------------------*/
/* NCCL communicator for depth-map all-gather (view sharding) and row gathers
 * (row sharding).  unique_id is the 128-byte ncclUniqueId from rank 0. */
int sr_comm_unique_id(void *out_128_bytes);
int sr_comm_init(sr_ctx *ctx, const void *unique_id_128_bytes, int rank, int nranks);
/* In-place all-gather of depth/index maps: view v is owned by rank owner[v]. */
int sr_comm_allgather_views(sr_ctx *ctx, const int32_t *owner);
/* Row-sharded variant: rank r owns rows [row_begin[r], row_end[r]) of `view`. */
int sr_comm_allgather_rows(sr_ctx *ctx, int view, const int32_t *row_begin,
                           const int32_t *row_end);

#ifdef __cplusplus
}
#endif
#endif /* SR_B200_H */
