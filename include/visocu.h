/* visocu.h -- the drop-in boundary: a thin extern "C" layer over the sm_100a CUDA kernels.
 *
 * It takes the place of the reference's device runtime (viso/opencl_wrapper.hh:19-166: Container / Buffer<T> /
 * Kernel) and of the host loops that the reference runs on the CPU for this path.  POD arguments only, no
 * C++/torch types, every function returns 0 on success or a negative VISOCU_E* code and never throws.
 *
 * One context = one GPU + one CUDA stream + a pool of device-resident "frames".  A frame holds everything the
 * reference keeps per image in Matcher's ring buffer (matcher.h:232-241): the Sobel planes, the two feature
 * record lists (sparse pass / dense pass) and their bin index.  Every entry point is batched: it takes arrays
 * of frames / pairs and processes them with one launch per kernel, because a single 1241x376 frame is far too
 * small to fill a B200 (SURVEY.md 7, hard part 3).
 *
 * Which reference interface each entry point replaces is cited next to it (paths relative to the reference).
 */
#ifndef VISOCU_H
#define VISOCU_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the libraries are built with -fvisibility=hidden */
#endif

#define VISOCU_OK            0
#define VISOCU_EINVAL       -1   /* bad argument (also: dims <= 0, bpl < width -- matcher.cpp:103-106) */
#define VISOCU_ECUDA        -2   /* CUDA runtime error, text in visocu_last_error */
#define VISOCU_ENODEVICE    -3   /* no sm_100 device: there is no CPU fallback */
#define VISOCU_ECAPACITY    -4   /* an output list overflowed its buffer */
#define VISOCU_ESTATE       -5   /* frame not computed yet / context not configured */

typedef struct visocu_ctx visocu_ctx;

/* Matcher::parameters, viso/matcher.h:42-69 -- same field order, same defaults (set by the C++ wrapper). */
typedef struct {
  int32_t nms_n, nms_tau, match_binsize, match_radius, match_disp_tolerance;
  int32_t outlier_disp_tolerance, outlier_flow_tolerance, multi_stage, half_resolution, refinement;
  double f, cu, cv, base;
} visocu_params;

/* Matcher::p_match, viso/matcher.h:86-100 (48 bytes). */
typedef struct {
  float u1p, v1p; int32_t i1p;
  float u2p, v2p; int32_t i2p;
  float u1c, v1c; int32_t i1c;
  float u2c, v2c; int32_t i2c;
} visocu_pmatch;

/* Matcher::range, viso/matcher.h:152-157: search window per circle stage for one statistics bin. */
typedef struct { float u_min[4], u_max[4], v_min[4], v_max[4]; } visocu_range;

/* One matching job = the four ring-buffer entries of Matcher::matching (matcher.cpp:965); -1 = unused. */
typedef struct { int32_t f1p, f2p, f1c, f2c; } visocu_quad;

/* ---- runtime (replaces OpenCL::Container::init / getDevice, opencl_wrapper.cpp:66-128) ----
 * A process that drives several contexts from several threads should export CUDA_DEVICE_MAX_CONNECTIONS=32 before its
 * first CUDA call (one hardware queue per stream); the library never changes its host's environment. */
int  visocu_create(int device, visocu_ctx** out);
void visocu_destroy(visocu_ctx* ctx);
const char* visocu_last_error(const visocu_ctx* ctx);          /* ctx may be NULL: last create() error */
int  visocu_device_info(const visocu_ctx* ctx, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, char* name64);
/* Allocates n_frames frame slots for width x height images.  `param.match_radius` is used as given (the C++
 * Matcher halves it for half_resolution exactly like matcher.cpp:59-60 before calling).  Re-configurable. */
int  visocu_configure(visocu_ctx* ctx, const visocu_params* param, int32_t width, int32_t height, int32_t n_frames);
/* Matcher::setIntrinsics (matcher.h:78-83): calibration used by the motion-predicted quad search */
int  visocu_set_intrinsics(visocu_ctx* ctx, double f, double cu, double cv, double base);
int  visocu_sync(visocu_ctx* ctx);
/* CUDA-event timing on the context's stream (replaces Container::durationOfEvent, opencl_wrapper.cpp:157-164). */
int  visocu_timer_start(visocu_ctx* ctx);
int  visocu_timer_stop(visocu_ctx* ctx, float* ms);
/* pinned host staging memory (optional, for callers that want truly asynchronous H2D) */
int  visocu_host_alloc(visocu_ctx* ctx, size_t bytes, void** out);
int  visocu_host_free(visocu_ctx* ctx, void* p);
int  visocu_device_alloc(visocu_ctx* ctx, size_t bytes, void** out);
int  visocu_device_free(visocu_ctx* ctx, void* p);
int  visocu_memcpy_h2d(visocu_ctx* ctx, void* dst, const void* src, size_t bytes);

/* ---- feature front end: Matcher::pushBack -> computeFeatures (matcher.cpp:95-181, 649-732) ----
 * imgs[k] is image k, `bpl_in` bytes per line.  on_device = 0: host memory, read only during the call (the reference's
 * pushBack copies the image before it returns, matcher.cpp:158-175); 1: device pointers (inputs already resident in HBM);
 * 2: host memory that stays valid and unchanged until the results of the step have been collected (copies from pinned
 * memory then run asynchronously; with on_device = 0 the call waits for them).  For every frame: copy into the 16-byte-stride layout
 * (matcher.cpp:158-175), [half image (630-647)], fused sobel5x5 / blob5x5 / checkerboard5x5 + both
 * nonMaximumSuppression passes (filter.cpp:316-365, matcher.cpp:330-431, 684-694), computeDescriptors
 * (433-477) and the bin index of createIndexVector (870-890).  n_sparse / n_dense (may be NULL) receive the
 * record counts n?1 / n?2; the call reads them back and waits only if they are requested (otherwise it returns as soon as
 * the work is enqueued, and visocu_frame_counts or the next matching call learns the counts). */
int  visocu_push_frames(visocu_ctx* ctx, int32_t n, const int32_t* frames, const uint8_t* const* imgs,
                        int32_t bpl_in, int32_t on_device, int32_t* n_sparse, int32_t* n_dense);
int  visocu_frame_counts(visocu_ctx* ctx, int32_t n, const int32_t* frames, int32_t* n_sparse, int32_t* n_dense);
/* the exported 12 x int32 records {u*s, v*s, 0, class, d1..d8} of matcher.cpp:707-731; pass 0 = sparse, 1 = dense */
int  visocu_get_features(visocu_ctx* ctx, int32_t frame, int32_t pass, int32_t* out12, int32_t cap, int32_t* n_out);
/* planes for parity checks / getGain: which = 0 du, 1 dv (matching resolution), 2 du_full, 3 dv_full,
 * 4 padded input image, 5 half-resolution image.  dims3 = {w, h, bpl} of that plane. */
int  visocu_get_plane(visocu_ctx* ctx, int32_t frame, int32_t which, uint8_t* out, size_t cap, int32_t* dims3);
/* The tile configurations of the fused filter + NMS kernel that visocu_configure built, largest first (at most 3):
 * out5[5 k .. 5 k + 4] = {kx, ky, ntx, nty, threads} of level k (kx x ky cells of the aligning NMS pass per tile, ntx x nty
 * tiles per frame, threads per CTA).  *pick = the level a launch of n_launch frames (1..128) runs on.  For tests and
 * tuning: which tiles run depends on how many frames one push launch carries. */
int  visocu_tile_levels(const visocu_ctx* ctx, int32_t n_launch, int32_t* n_levels, int32_t* out5, int32_t* pick);

/* ---- rectification of raw camera images (not in the reference, which expects undistorted, rectified images) ----
 * A camera: raw pinhole K = (fx, fy, cx, cy), radial-tangential distortion k1, k2, p1, p2, k3 (OpenCV's and KITTI's model),
 * the rectifying rotation R (raw camera -> rectified coordinates, row-major) and the rectified projection f, cu, cv.
 * visocu_set_rectification builds one map per camera for raw images of src_w x src_h and the configured (output) size: the
 * output pixel (u, v) samples the raw image at the distorted projection of the ray R^T ((u - cu) / f, (v - cv) / f, 1),
 * in 1/32 pixel and clamped to the raw image (the border is replicated); host/rectify.h states it exactly.  At most 2
 * cameras; n_cams = 0 removes the maps; visocu_configure removes them as well.  VISOCU_EINVAL, before anything changes, for
 * a non-finite parameter, fx, fy or f <= 0, src_w or src_h outside [16, 8191] or an output pixel whose rotated ray has
 * z <= 0; VISOCU_ESTATE on a context that is not configured.
 * visocu_push_frames_rectified is visocu_push_frames for raw images (bpl_in >= src_w): image k is resampled with map cam[k]
 * into its frame (bilinear in 1/32 pixel, integer arithmetic: ((32-fx)(32-fy) p00 + fx(32-fy) p01 + (32-fx) fy p10 +
 * fx fy p11 + 512) >> 10), then the features are computed as for a plain push.  VISOCU_ESTATE without maps, VISOCU_EINVAL
 * for a camera index out of range or bpl_in < src_w, both before anything is enqueued.
 * visocu_get_rectify_map copies map `cam` (2 int32 per output pixel, x then y in 1/32 pixel, row-major) to out; cap in
 * int32 entries. */
typedef struct { double fx, fy, cx, cy, k1, k2, p1, p2, k3, R[9], f, cu, cv; } visocu_camera;
int  visocu_set_rectification(visocu_ctx* ctx, int32_t n_cams, const visocu_camera* cams, int32_t src_w, int32_t src_h);
int  visocu_push_frames_rectified(visocu_ctx* ctx, int32_t n, const int32_t* frames, const uint8_t* const* imgs, const int32_t* cam,
                                  int32_t bpl_in, int32_t on_device, int32_t* n_sparse, int32_t* n_dense);
int  visocu_get_rectify_map(visocu_ctx* ctx, int32_t cam, int32_t* out, size_t cap);

/* ---- dense stereo disparity (not in the reference): semi-global matching on the images of pushed frames ----
 * visocu_disparity computes, for pair k, the disparity map of frame left[k] against frame right[k] from their
 * full-resolution images as pushed (the rectified bytes after a rectifying push, whatever half_resolution says):
 * census 9x7 (62 bits, neighbour < centre, coordinates clamped), cost = Hamming distance of cenL(x, y) and cenR(x - d, y)
 * (62 where x - d < 0), 4 paths (+-x, +-y) or 8 (and the diagonals) of L_r(p, d) = C(p, d) + min(L_r(p-r, d),
 * L_r(p-r, d+-1) + p1, min_k L_r(p-r, k) + p2) - min_k L_r(p-r, k) (L_r = C at the border), S = the sum of the paths;
 * d* = the smallest d of min S.  Invalid (-1): uniqueness (some |d - d*| > 1 with 100 S(d*) > uniqueness S(d)) and, when
 * lr_max_diff >= 0, x - d* < 0 or |dR(x - d*) - d*| > lr_max_diff, dR(x') = the smallest d < min(D, w - x') of
 * min S(x' + d, y, d).  out[k] receives w x h int16 (row stride w) in 1/16 pixel: 16 d* plus, with subpixel = 1 and
 * 0 < d* < D - 1, floor((16 (a - c) + den) / (2 den)) for den = a + c - 2 b > 0 (a, b, c = S at d* - 1, d*, d* + 1).
 * Valid: max_disp D in {64, 128, 256}, paths in {4, 8}, 1 <= p1 < p2 <= 150, 0 <= uniqueness <= 100,
 * -1 <= lr_max_diff <= D, subpixel in {0, 1}; oracle/sgm_oracle.c states the algorithm in plain C.
 * out_on_device = 0: out[k] are host memory; 1: device memory of the context's GPU.  The call runs on the current lane,
 * behind the last push of every lane, and waits for its work.  VISOCU_EINVAL for bad parameters, a frame index out of
 * range, a null pointer or n_pairs < 0; VISOCU_ESTATE for a frame never pushed or an unconfigured context; both before
 * anything is enqueued or written.  Per group of at most 128 pairs: 4 launches with 4 paths, 6 with 8, and scratch of
 * w h (16 + 2 D) bytes per pair (+ 2 w h for host outputs). */
typedef struct { int32_t max_disp, paths, p1, p2, uniqueness, lr_max_diff, subpixel; } visocu_sgm_params;
int  visocu_disparity(visocu_ctx* ctx, int32_t n_pairs, const int32_t* left, const int32_t* right,
                      const visocu_sgm_params* p, int16_t* const* out, int32_t out_on_device);
/* VISOCU_OK if p is non-null and inside the valid ranges above, else VISOCU_EINVAL (for callers that store parameters) */
int  visocu_sgm_check(const visocu_sgm_params* p);

/* ---- filter:: functions (viso/filter.h:78-94), host buffers in and out, same argument order ---- */
int  visocu_sobel5x5(visocu_ctx* ctx, const uint8_t* in, uint8_t* out_v, uint8_t* out_h, int32_t w, int32_t h);
int  visocu_sobel3x3(visocu_ctx* ctx, const uint8_t* in, uint8_t* out_v, uint8_t* out_h, int32_t w, int32_t h);
int  visocu_blob5x5(visocu_ctx* ctx, const uint8_t* in, int16_t* out, int32_t w, int32_t h);
int  visocu_checkerboard5x5(visocu_ctx* ctx, const uint8_t* in, int16_t* out, int32_t w, int32_t h);
/* Matcher::nonMaximumSuppression on caller-supplied response maps (matcher.cpp:330-431): out4 = (u,v,val,c) */
int  visocu_nms(visocu_ctx* ctx, const int16_t* f1, const int16_t* f2, int32_t w, int32_t h, int32_t bpl,
                int32_t nms_n, int32_t tau, int32_t* out4, int32_t cap, int32_t* n_out);

/* ---- SAD circle matching: Matcher::matching + findMatch (+ pixel refinement) ----
 * (matcher.cpp:965-1205, 892-963, 1379-1585).  method 0 = flow, 1 = stereo, 2 = quad.  pass 0 = sparse sets,
 * 1 = dense.  ranges[j] (host, u_bins*v_bins entries, matcher.cpp:734-868) is read only if use_prior.  refine = 1
 * applies relocateMinimum (pixel), refine = 2 parabolicFitting (sub-pixel; drops the matches the reference drops)
 * before the matches are returned.  out[j] receives at most cap[j] matches in the reference's order (ascending
 * i1c for flow and stereo, ascending i1p for quad).  tr_delta (optional, quad only): per job the first three rows
 * (12 doubles) of the previous motion estimate; enables the motion-predicted search of matcher.cpp:1112-1138 with the
 * calibration f, cu, cv, base of the configured parameters (VisualOdometryStereo::process, viso_stereo.cpp:35).
 * outliers (optional, n_jobs entries): if non-null, Matcher::removeOutliers (matcher.cpp:1207-1377) runs on the device
 * right after the matching / refinement and only the survivors are copied back; outliers[j] is set to 1.  A list the
 * device path cannot take (too long for shared memory, or two matches on the same pixel) comes back complete with
 * outliers[j] = 0, and the caller has to run the vote itself. */
int  visocu_match(visocu_ctx* ctx, int32_t n_jobs, const visocu_quad* jobs, int32_t method, int32_t pass,
                  int32_t use_prior, const visocu_range* const* ranges, const double* const* tr_delta, int32_t refine,
                  visocu_pmatch* const* out, const int32_t* cap, int32_t* n_out, int32_t* outliers);
/* Both passes of multi-stage FLOW matching in one submission (matcher.cpp:219-233 without a host round trip): first pass on
 * the sparse features, its outlier removal, Matcher::computePriorStatistics (matcher.cpp:734-868) on the survivors - on the
 * device -, second pass on the dense features with those ranges, refinement (0 or 1), outlier removal.  The kernels take
 * the record counts of the frames from device memory and everything is sized by the capacity of the record lists, so the
 * frames may have been pushed without reading their counts back (visocu_push_frames with null count pointers): pushing
 * and matching a frame is then ONE submission, and the wait at the end of this call the only one.  The results are
 * written by the last kernel into pinned memory owned by the context: list1[j] / list2[j] point into it and stay valid
 * until the next matching call on this context.  done1 / done2 say whether the outlier removal of the list ran on the
 * device (if done1[j] is 0 the second list of job j is meaningless: the caller votes on list 1 itself and repeats the second
 * pass with visocu_match); ranges_out[j] (optional, u_bins * v_bins entries) receives the prior ranges; counts (optional,
 * 4 per job) the sparse and dense record counts of f1p and of f1c.  *list2_compact says how the records of list2 crossed
 * PCIe: 0 = complete 48-byte records; 1 = the 24 bytes of a flow match that say something, (u1p, v1p, i1p, u1c, v1c, i1c),
 * six words per match - the other six fields of p_match are -1 (matcher.cpp:1037); 2 = the same in 12 bytes, three words
 * (u1p | v1p << 16), (u1c | v1c << 16), (i1p | i1c << 16): without sub-pixel refinement (refine != 2) the coordinates are
 * whole pixels, and they and the indices fit 16 bits (the kernel checks every value).  At most 128 jobs. */
int  visocu_match_fused(visocu_ctx* ctx, int32_t n_jobs, const visocu_quad* jobs, int32_t refine,
                        const visocu_pmatch** list1, int32_t* n1, int32_t* done1,
                        const visocu_pmatch** list2, int32_t* n2, int32_t* done2,
                        visocu_range* const* ranges_out, int32_t* counts, int32_t* list2_compact);
/* The same call in two halves, for callers that keep several steps in flight: _submit enqueues everything on the current
 * lane and returns, _collect waits for that lane and delivers what visocu_match_fused delivers.  after_lane (or -1): the
 * lane on which the previous frames of the jobs were pushed, if it is not the current one - the matching then starts
 * behind that lane's feature kernels.  flags: 1 = deliver the prior ranges, 2 = deliver the first list as well (else
 * list1[j] is null unless the device declined that list and the caller has to vote on it).  A step that repeats with the same frames, jobs and sizes (a runner walking
 * sequences through the lanes in turn) is captured as a CUDA graph and replayed: one graph launch per half step.
 * Lanes: a context holds several complete sets of per-step resources (stream, scratch and staging memory, result area);
 * visocu_set_lane(ctx, k), 0 <= k < 6, makes set k the one every following call works with.  Lane 0 is the default. */
int  visocu_set_lane(visocu_ctx* ctx, int32_t lane);
int  visocu_match_fused_submit(visocu_ctx* ctx, int32_t n_jobs, const visocu_quad* jobs, int32_t refine, int32_t flags,
                               int32_t after_lane);
int  visocu_match_fused_collect(visocu_ctx* ctx, const visocu_pmatch** list1, int32_t* n1, int32_t* done1,
                                const visocu_pmatch** list2, int32_t* n2, int32_t* done2,
                                visocu_range* const* ranges_out, int32_t* counts, int32_t* list2_compact);
/* Matcher::removeOutliers alone on caller-supplied match lists (host memory, compacted in place).  status[j] = 0: done,
 * 1: list unchanged, not handled by the device path (see visocu_match). */
int  visocu_remove_outliers(visocu_ctx* ctx, int32_t n_jobs, int32_t method, visocu_pmatch* const* inout, const int32_t* n,
                            int32_t* n_out, int32_t* status);
/* Lists too long for the device path of removeOutliers (more than about 5 700 vertices: 3840x2160 frames): the
 * triangulation is a divide-and-conquer tree (triangle.cpp divconqdelaunay with alternating cuts, matcher.cpp:1255), and
 * its lower part - all the work but the seams of the top few merges - consists of independent nodes that fit the device
 * kernel.  visocu_delaunay_subtrees triangulates such nodes: pts = the vertices of the whole problem (x | y << 16, both
 * below 8192, all distinct), node j = pts[first[j] .. first[j] + count[j]) with 4 <= count[j] <= 5000, axis[j] = direction
 * of the node's own cut (0 = vertical).  The result is ONE mesh in the numbering of the whole problem, ready to be merged
 * further: *mesh = *n_halfedges records of four words (onext, oprev, origin vertex, x | y << 16 of the origin; sym(e) =
 * e ^ 1; origin -1 = deleted or unused) followed by room for extra_halfedges more; node j owns the half-edges from
 * mesh_first[j] (2 * visocu_delaunay_edge_capacity(count[j]) of them) and numbers its vertices first[j] + v, v in the order
 * of its partition tree, (*vert)[first[j] + v] = index within the node of vertex v.  (*result)[16 j + 1] = status (0 =
 * done), [16 j + 2] = edges allocated, [16 j + 4], [16 j + 5] = hull handles (counter-clockwise hull edge out of the
 * leftmost vertex, clockwise hull edge out of the rightmost).  The memory belongs to the context and stays valid (and
 * writable) until the next call on this lane.  The caller (host/delaunay.cpp) runs the merges above the nodes and votes. */
int32_t visocu_delaunay_edge_capacity(int32_t n_vertices);
int  visocu_delaunay_subtrees(visocu_ctx* ctx, const uint32_t* pts, int32_t n_pts, int32_t n_jobs, const int32_t* first,
                              const int32_t* count, const int32_t* axis, int32_t extra_halfedges, int32_t** mesh,
                              int32_t* mesh_first, int32_t* n_halfedges, const int32_t** vert, const int32_t** result);
/* Matcher::refinement alone on caller-supplied matches: mode 1 = pixel, 2 = sub-pixel (n_out <= n survive) */
int  visocu_refine(visocu_ctx* ctx, const visocu_quad* job, int32_t method, int32_t mode, visocu_pmatch* inout, int32_t n,
                   int32_t* n_out);
/* work counters since the previous visocu_match_stats call: candidates that passed the window test (matcher.cpp:943) and
 * bin entries scanned, summed over all jobs and hops -- the SAD roofline unit of SURVEY.md 8(d) */
int  visocu_match_stats(visocu_ctx* ctx, uint64_t* sad_candidates, uint64_t* entries_scanned);

/* ---- RANSAC: VisualOdometryMono::ransacEstimateF (viso_mono.cpp:41-72; virtual hook viso_mono.h:74) ----
 * uv[j]: N[j] x 4 floats (u1p,v1p,u1c,v1c) already Hartley-normalised (viso_mono.cpp:217-263).
 * samples[j]: iters x 8 indices drawn by the host with the reference's generator (viso.cpp:86-102).
 * Per job: one warp per hypothesis does the 8-point fit (viso_mono.cpp:265-296), a batched pass scores all
 * hypotheses (getInlier, 298-345, FP64 Sampson, |d| < thresh), the earliest hypothesis with the strictly
 * largest count wins (56-57) and F is refitted on its inliers (61-69).  n_inliers < 10 => F9 = 0 (59-60).
 * counts (iters, optional) and F_all (iters x 9, optional) expose per-hypothesis results for parity tests. */
int  visocu_ransac_F(visocu_ctx* ctx, int32_t n_jobs, const float* const* uv, const int32_t* N,
                     const int32_t* const* samples, int32_t iters, double thresh,
                     double* F9, uint8_t* const* inlier_mask, int32_t* n_inliers, int32_t* best_iter,
                     int32_t* const* counts, double* const* F_all);

/* ---- stereo odometry: VisualOdometryStereo::estimateMotion (viso_stereo.cpp:42-145) for n_jobs match lists at once ----
 * matches[j]: N[j] >= 6 p_match records (u1p, v1p, u2p: previous stereo pair; u1c, v1c, u2c, v2c: current).  samples[j]:
 * p->ransac_iters x 3 indices drawn by the host with the reference's generator (one getRandomSample(N, 3) per iteration).
 * Per job: one thread per hypothesis runs Gauss-Newton from tr = 0 on the 12 rows of its sample (step 1, eps 1e-6, at most
 * 22 updates; the 6x6 normal equations solved as Matrix::solve does, a failed solve drops the hypothesis); one thread per
 * match scores every hypothesis (unweighted squared reprojection error of u1c, v1c, u2c, v2c < inlier_threshold^2); the
 * earliest hypothesis with the strictly largest count (> 0) wins; one CTA refines on all its inliers (eps 1e-8, at most 102
 * updates, a fixed reduction tree: a call is bit-identical from run to run).  Out per job: ok[j] (>= 6 inliers and the
 * refinement converged), tr6 (rx, ry, rz, tx, ty, tz; valid if ok, else 0), inlier_mask (optional, N[j] bytes: the winning
 * hypothesis' inliers), n_inliers (optional), best_iter (optional, -1 if no hypothesis had an inlier).  Optional, for
 * parity tests: counts[j] (iters; -1 = that hypothesis' Gauss-Newton failed) and tr_all[j] (iters x 6).  N[j] < 6, a
 * sample index outside [0, N[j]) or a null input gives VISOCU_EINVAL before anything is written.  One upload, three
 * launches and one read-back per 128 jobs, on the context's current lane. */
typedef struct { double f, cu, cv, base, inlier_threshold; int32_t ransac_iters, reweighting; } visocu_stereo_params;
int  visocu_stereo_motion(visocu_ctx* ctx, int32_t n_jobs, const visocu_pmatch* const* matches, const int32_t* N,
                          const int32_t* const* samples, const visocu_stereo_params* p, double* tr6, int32_t* ok,
                          uint8_t* const* inlier_mask, int32_t* n_inliers, int32_t* best_iter,
                          int32_t* const* counts, double* const* tr_all);

/* ---- reconstruction: the finished tracks of Reconstruction::update (reconstruction.cpp:50-146), many updates at once ----
 * One job = the tracks that ended with one update of one Reconstruction (host/reconstruction.h: batchPrepare fills it).
 * frames: the update's window, oldest first, frames[n_frames - 1] = the newest camera; per frame proj = K * inv[0:3, 0:4],
 * inv = rows 0..2 of the inverse of fwd (frame -> newest camera), center = fwd[0:3, 3], all row-major.  tracks: obs k was
 * seen from frame first + k.  cam_road: rows 0..2 of the camera -> road transform of the point types.
 * Per track, in the host's order and with its semantics: initPoint (null vector of the 4x4 system of the first observation
 * in frame `first` and the last one in the NEWEST frame, point in float), pointType on that point, refinePoint (Gauss-Newton
 * over all observations, the point kept in float between updates, the 3x3 normal equations solved as Matrix::solve does,
 * converged when all three updates are below 1e-5, at most 22 updates), pointDistance to the centre of frame
 * n_frames - 1 - (n_frames - first) / 2, rayAngle between the first and the newest centre (1000 for a degenerate ray).
 * status[j][i]: 0 kept, 1 initPoint failed (|w| < 1e-10), 2 point type below point_type, 3 refinePoint failed (c^2 < 1e-10,
 * singular solve or no convergence), 4 distance >= max_dist, 5 ray angle <= min_angle.  xyz[j][3 i ..]: the point as last
 * computed - the initial point for status 2, the refined one for 0, 4 and 5, zeros for 1 and 3.  One thread per track in
 * FP64; the null vector comes from a Jacobi rotation, not the host's SVD, so points agree with the host to rounding.
 * A null pointer (status[j], xyz[j] and tracks may be null only for a job without tracks), n_frames outside [1, 8],
 * n_tracks < 0, n_obs outside [2, 6] or first < 0 or first + n_obs > n_frames gives VISOCU_EINVAL before anything is
 * written.  One upload, one launch and one read-back per call, on the context's current lane; a call whose jobs hold no
 * tracks launches nothing. */
typedef struct { double proj[12], inv[12], center[3]; } visocu_recon_frame;
typedef struct { int32_t first, n_obs; float u[6], v[6]; } visocu_recon_track;
typedef struct {
  const visocu_recon_frame* frames; int32_t n_frames;
  const visocu_recon_track* tracks; int32_t n_tracks;
  double cam_road[12]; double max_dist, min_angle; int32_t point_type;
} visocu_recon_job;
int  visocu_recon_points(visocu_ctx* ctx, int32_t n_jobs, const visocu_recon_job* jobs, int32_t* const* status,
                         float* const* xyz);

/* ---- device point store: Reconstruction's point list (reconstruction.cpp:41, 146) kept in HBM ----
 * A store holds one sequence's reconstructed points as float x, y, z (n x 3, packed) in device memory of the context that
 * created it.  The context owns its stores: visocu_destroy frees those still alive.  A store is not tied to a lane; every
 * call runs on the context's current lane and waits for its work before it returns.  Growth doubles the capacity.
 * _append copies n host points behind the stored ones; _read copies points first .. first + count - 1 to the host; both
 * give VISOCU_EINVAL for a range outside the store or a null pointer.  _points gives the device address and the count;
 * the address stays valid until the next call that changes the store. */
typedef struct visocu_recon_store visocu_recon_store;
int  visocu_recon_store_create(visocu_ctx* ctx, int64_t initial_capacity, visocu_recon_store** out);
int  visocu_recon_store_destroy(visocu_ctx* ctx, visocu_recon_store* store);
int  visocu_recon_store_append(visocu_ctx* ctx, visocu_recon_store* store, const float* xyz, int64_t n);
int  visocu_recon_store_read(visocu_ctx* ctx, const visocu_recon_store* store, int64_t first, int64_t count, float* xyz);
int  visocu_recon_store_points(const visocu_recon_store* store, const float** d_xyz, int64_t* n);
/* Reconstruction::update's device half for n_jobs stores (one per sequence): per job j, in this order,
 *   (a) every point of stores[j] becomes rows 0..2 of tr12[j] (12 doubles, row-major) applied to (p, 1), with the bytes of
 *       the host's affineTransform (host/reconstruction.cpp);
 *   (b) jobs[j] is evaluated exactly as visocu_recon_points evaluates it;
 *   (c) the points with status 0 are appended to stores[j] in track order.
 * n_kept[j] (optional) = points appended.  status / xyz (optional, each null or n_jobs entries) receive what
 * visocu_recon_points returns.  Every check of visocu_recon_points, a null store or tr12, a store of another context and a
 * store named twice give VISOCU_EINVAL before anything is enqueued or written.  If a store cannot grow, the move still runs,
 * nothing is appended to any store and the call returns VISOCU_ECAPACITY.  One upload, at most three launches (move,
 * evaluation, append; a stage without work launches nothing) and one read-back; the call waits at the end. */
int  visocu_recon_update(visocu_ctx* ctx, int32_t n_jobs, visocu_recon_store* const* stores, const double* const* tr12,
                         const visocu_recon_job* jobs, int32_t* n_kept, int32_t* const* status, float* const* xyz);

/* ---- pose recovery helpers after RANSAC (SURVEY.md 8f rank 2) ----
 * visocu_triangulate: VisualOdometryMono::triangulateChieral (viso_mono.cpp:394-431) for up to four (R|t) candidates
 * at once.  uv: N x 4 floats (u1p,v1p,u1c,v1c) in pixels; P1: 3x4 projection of the previous camera, P2: n_sol 3x4
 * projections of the current camera (row-major).  X receives n_sol blocks of 4 x N homogeneous points (row-major, not
 * normalised: the null vector of each 4x4 system, sign arbitrary); n_front[s] = points in front of both cameras.
 * visocu_best_plane: VisualOdometryMono::findBestPlane (viso_mono.cpp:74-98; the reference's OpenCL hook
 * viso_mono_cl.cpp:255-280): index of the candidate d_i > threshold with the largest sum_j exp(-(d_j-d_i)^2 weight),
 * first maximum wins, 0 if there is no candidate. */
int  visocu_triangulate(visocu_ctx* ctx, const float* uv, int32_t N, const double* P1, const double* P2, int32_t n_sol,
                        double* X, int32_t* n_front);
int  visocu_best_plane(visocu_ctx* ctx, const double* d, int32_t n, double threshold, double weight, int32_t* best_idx);
/* batched forms: one upload, one launch, one read-back for n_jobs problems (at most 128) */
int  visocu_triangulate_batch(visocu_ctx* ctx, int32_t n_jobs, const float* const* uv, const int32_t* N, const double* const* P1,
                              const double* const* P2, const int32_t* n_sol, double* const* X, int32_t* const* n_front);
int  visocu_best_plane_batch(visocu_ctx* ctx, int32_t n_jobs, const double* const* d, const int32_t* n, const double* threshold,
                             const double* weight, int32_t* best_idx);

/* host<->device bytes copied by this context since creation (bench.py's h2d / d2h bytes per step) */
int  visocu_transfer_bytes(const visocu_ctx* ctx, uint64_t* h2d, uint64_t* d2h);
/* event timing of the fused filter+NMS launches on the context's stream (replaces the per-call
 * Container::durationOfEvent prints of viso_mono_cl.cpp:245-248).  While enabled every fused launch is
 * followed by an event synchronise; read = accumulated milliseconds, launches and frames since enable. */
int  visocu_profile(visocu_ctx* ctx, int32_t enable);
int  visocu_profile_read(const visocu_ctx* ctx, double* filter_ms, uint64_t* launches, uint64_t* frames);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
int  visocu_launch_count(const visocu_ctx* ctx, uint64_t* n);
/* device outlier removal so far: out8 = lists handled, lists declined (too long, duplicates, guard: [2..4]), and the
 * summed kernel time of the handled lists in nanoseconds ([5] sort + partition, [6] build, [7] vote + compaction) */
int  visocu_outlier_stats(const visocu_ctx* ctx, uint64_t* out8);
/* visocu_delaunay_subtrees: out2[0] = calls (lists too long for the device path as a whole), out2[1] = nodes built */
int  visocu_node_stats(const visocu_ctx* ctx, uint64_t* out2);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif
