/*
 * svob200.h — C ABI of the B200-native SVO tracking front end (libsvob200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, int status
 * returns (0 = ok, <0 = error; svob200_last_error() gives the text).  Each entry point names
 * the reference interface it replaces (paths relative to
 * /root/reference/app/src/main/cpp/svo).  INTEGRATION.md shows the reference-side bindings.
 *
 * Conventions
 *   pose      double[7] = {tx,ty,tz, qx,qy,qz,qw}   (SE3 ctor order, include/svo/SE3.h:17-19)
 *   camera    distortion-free pinhole (pinhole_camera.cpp:48-53, :83-87)
 *   frames    device-resident image pyramids keyed by a caller-chosen 64-bit id (Frame::id_);
 *             a frame may hold a BATCH of independent images of equal size (one per sequence)
 *   mem       every array argument of a compute call lives either in host memory
 *             (SVOB200_MEM_HOST: the call stages, copies H2D/D2H and synchronises) or in device
 *             memory (SVOB200_MEM_DEVICE: no copies, asynchronous on the context's stream)
 *   batching  per-item arrays carry the image (= sequence) index inside the frame batch
 *
 * There is no CPU fallback: every compute entry point launches CUDA kernels and fails with
 * SVOB200_ERR_CUDA if no device is usable.
 *
 * Threading: a context (and every tracker created on it) is used by ONE host thread at a time — it owns one stream, one staging
 * arena, one error string.  Callers that share it across threads serialise their calls (the C++ drop-in does, behind its runtime
 * lock); independent threads create independent contexts.
 */
#ifndef SVOB200_H_
#define SVOB200_H_
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVOB200_MAX_LEVELS 8          /* array extent; the fused pyramid kernel supports <= 7 */

enum { SVOB200_OK = 0, SVOB200_ERR_ARG = -1, SVOB200_ERR_CUDA = -2, SVOB200_ERR_NOFRAME = -3,
       SVOB200_ERR_UNSUPPORTED = -4, SVOB200_ERR_NOMEM = -5 };
enum { SVOB200_MEM_HOST = 0, SVOB200_MEM_DEVICE = 1 };
/* vk::halfSample rounding (vision.cpp): TRUNC = scalar/NEON (a+b+c+d)/4; SSE2 = x86 double avg */
enum { SVOB200_ROUND_TRUNC = 0, SVOB200_ROUND_SSE2 = 1 };

typedef struct svob200_ctx svob200_ctx;
typedef struct { int width, height; double fx, fy, cx, cy; } svob200_camera;

/* ---------------------------------------------------------------- context */
int         svob200_ctx_create(int device, svob200_ctx** out);
void        svob200_ctx_destroy(svob200_ctx* ctx);
const char* svob200_last_error(const svob200_ctx* ctx);
int         svob200_ctx_sync(svob200_ctx* ctx);
void*       svob200_ctx_stream(svob200_ctx* ctx);             /* cudaStream_t */
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
long long   svob200_ctx_launch_count(const svob200_ctx* ctx);
/* CUDA-event timing on the context's stream (events are created lazily) */
int         svob200_ctx_timer_start(svob200_ctx* ctx);
int         svob200_ctx_timer_stop_ms(svob200_ctx* ctx, float* ms);

/* sizeof() of the ABI structs in declaration order (camera, corner, align_opts, align_result,
 * matcher_opts, feature_ref, match_result, epi_result, seed, seed_obs, step_stats, map_point, reproj_result,
 * reproj_stats, pose_opt_result, pose_opt_opts); returns how many there are */
int         svob200_abi_sizes(int* sizes, int cap);

/* ---------------------------------------------------------------- frames / pyramid
 * replaces: Frame::initFrame -> frame_utils::createImgPyramid -> vk::halfSample
 *           (frame.cpp:51-64, :186-195; vision.cpp:71-110) */
/* x86 host dispatch rule of vk::halfSample (vision.cpp:78): SSE2 iff in_cols % 16 == 0 */
int svob200_round_mode_x86(int in_cols);
/* allocate a device pyramid for `batch` images of w x h with n_levels levels */
int svob200_frame_create(svob200_ctx* ctx, int64_t frame_id, int batch, int w, int h, int n_levels);
/* copy level 0 (gray: batch images, row stride `stride` bytes, image stride stride*h) and build
 * levels 1..n-1.  round_modes: n_levels-1 entries (mode used to produce level l+1 from l) or
 * NULL for the x86 host rule.  mem says where `gray` lives. */
int svob200_frame_upload(svob200_ctx* ctx, int64_t frame_id, const uint8_t* gray, int stride,
                         const int* round_modes, int mem);
/* level 0 ALIASES the caller's device buffer (like the reference, where level 0 aliases the caller's
 * cv::Mat, frame.cpp:189): no copy, the pyramid kernel reads the frame where it already lies in HBM.
 * dev_gray and stride must be 16-byte aligned; the buffer must outlive the frame's use. */
int svob200_frame_bind(svob200_ctx* ctx, int64_t frame_id, const uint8_t* dev_gray, int stride,
                       const int* round_modes);
/* frame-table slot of a resident frame (>= 0).  In SVOB200_MEM_DEVICE mode the ref_frame_id field
 * of svob200_feature_ref records must already hold this slot instead of the id. */
int svob200_frame_slot(svob200_ctx* ctx, int64_t frame_id);
/* download one level of one image into a dense (or strided) host buffer */
int svob200_frame_download(svob200_ctx* ctx, int64_t frame_id, int image, int level,
                           uint8_t* out, int out_stride);
/* copy ONE level of one image verbatim from host memory: mirrors a host pyramid (Frame::img_pyr_,
 * frame.h) on the device exactly as the host holds it; used by the C++ drop-in's frame cache */
int svob200_frame_upload_level(svob200_ctx* ctx, int64_t frame_id, int image, int level, const uint8_t* data, int stride);
int svob200_frame_release(svob200_ctx* ctx, int64_t frame_id);
int svob200_frame_info(svob200_ctx* ctx, int64_t frame_id, int* batch, int* w, int* h, int* n_levels);
/* stand-alone vk::halfSample(in,out) on host buffers (vision.h:38): upload, one level, download */
int svob200_half_sample(svob200_ctx* ctx, const uint8_t* in, int w, int h, int in_stride,
                        uint8_t* out, int out_stride, int round_mode);

/* ---------------------------------------------------------------- FAST + Shi-Tomasi + grid
 * replaces: FastDetector::detect (feature_detection.cpp:77-122), cv::FAST(img,kps,10,true)
 *           (OpenCV 4.5.4 features2d, FAST-9/16), vk::shiTomasiScore (vision.cpp:113-154) */
typedef struct { int x, y, level; float score; } svob200_corner;
/* cells_out: batch * n_cells entries (n_cells = ceil(W/cell)*ceil(H/cell)), each initialised to
 * (0,0,0,thr) like the reference; a cell holds a feature iff score > thr.  occupancy: batch*n_cells
 * bytes or NULL.  n_features_out: batch ints (may be NULL). */
int svob200_fast_detect(svob200_ctx* ctx, int64_t frame_id, int n_detect_levels, int cell_size,
                        double detection_threshold, const uint8_t* occupancy,
                        svob200_corner* cells_out, int* n_features_out, int mem);
/* raw cv::FAST keypoints of one level of one image (row-major order), for parity tests.
 * Returns the keypoint count (<0 on error); writes at most cap entries. */
int svob200_fast_corners(svob200_ctx* ctx, int64_t frame_id, int image, int level, int threshold,
                         int nonmax, int cap, int* xs, int* ys, int* scores);

/* vk::shiTomasiScore(img,u,v) (vision.cpp:113-154, vision.h:40) for n pixels (uv: 2 ints each) of a host image */
int svob200_shi_tomasi(svob200_ctx* ctx, const uint8_t* img, int w, int h, int stride, int n, const int* uv, float* scores);

/* ---------------------------------------------------------------- sparse image alignment
 * replaces: SparseImgAlign::run (sparse_img_align.cpp:51-92) incl. precomputeReferencePatches,
 *           computeResiduals, solve, update and vk::NLLSSolver::optimizeGaussNewton
 *           (nlls_solver_impl.hpp:25-100) */
typedef struct { int max_level, min_level, n_iter; double eps; } svob200_align_opts;
typedef struct {
  double T_cur_ref[7];
  double H[36];          /* row-major; H_ of the last linearisation (getFisherInformation = H/(5e-4*255^2)) */
  double Jres[6];
  double x[6];
  double chi2;
  int    n_meas;         /* run() returns n_meas/16 */
  int    iters[SVOB200_MAX_LEVELS];
  int    stop;
  int    n_exact_chi2;   /* iterations whose rollback decision needed the sequential float chi2 */
  int    n_factorisations; /* iterations that summed H_ again and factorised it (the others re-used both: the set of features inside
                              the current image was unchanged, and a feature's share of J J^T is constant over a level) */
} svob200_align_result;
/* One alignment problem per image of the batch.  ftr_offsets: batch+1 prefix offsets into the
 * per-feature arrays; px: 2 doubles (level-0 pixels); xyz_ref: 3 doubles (= f*depth,
 * sparse_img_align.cpp:132-134); has_point: 1 byte; T_cur_ref: 7 doubles per image (in);
 * results: one svob200_align_result per image (out). */
int svob200_sparse_align(svob200_ctx* ctx, int64_t ref_frame_id, int64_t cur_frame_id,
                         const svob200_camera* cam, int batch, const int* ftr_offsets,
                         const double* px, const double* xyz_ref, const uint8_t* has_point,
                         const double* T_cur_ref, const svob200_align_opts* opts,
                         svob200_align_result* results, int mem);

/* ---------------------------------------------------------------- feature alignment
 * replaces: feature_alignment::align2D / align1D float paths (feature_alignment.cpp:35-282) */
/* n independent problems on one level of a frame.  image: n ints; patch_with_border: n*100,
 * patch: n*64 bytes; dir: n*2 floats (align1D only, NULL => align2D); px: n*2 doubles in/out at
 * that level's scale; converged: n ints; h_inv: n doubles (align1D only, may be NULL) */
int svob200_align_patches(svob200_ctx* ctx, int64_t frame_id, int level, int n, const int* image,
                          const uint8_t* patch_with_border, const uint8_t* patch, const float* dir,
                          int n_iter, double* px, int* converged, double* h_inv, int mem);

/* ---------------------------------------------------------------- matcher
 * replaces: Matcher::findMatchDirect (matcher.cpp:156-202) after Point::getCloseViewObs picked
 *           the reference observation; warp::getWarpMatrixAffine / getBestSearchLevel / warpAffine
 *           (matcher.cpp:36-116); Matcher::findEpipolarMatchDirect (matcher.cpp:207-355);
 *           vk::patch_score::ZMSSD<4> (patch_score.h) */
typedef struct {
  int align_1d, align_max_iter, max_epi_search_steps, subpix_refinement, epi_search_edgelet_filtering;
  double epi_search_edgelet_max_angle;
  int max_search_level;            /* Config::nPyrLevels()-1 */
} svob200_matcher_opts;
/* max_epi_search_steps: 0 .. INT_MAX (the reference's size_t, clamped); a walk of up to that many steps is searched,
 * whatever its length.  Every entry point that takes these options returns SVOB200_ERR_ARG for a negative value. */
void svob200_matcher_opts_default(svob200_matcher_opts* o, int n_pyr_levels);

/* reference-side description of one feature (Feature{px,f,level,type,grad}, feature.h:24-76) */
typedef struct {
  int64_t ref_frame_id; int ref_image;     /* keyframe holding the reference patch */
  int     cur_image;                       /* image inside the current frame batch */
  int     level; int type;                 /* type: 0 CORNER, 1 EDGELET */
  double  px[2]; double f[3]; double grad[2];
  double  T_cur_ref[7];                    /* cur.T_f_w_ * ref.T_f_w_.inverse() */
} svob200_feature_ref;

typedef struct {
  int success; int search_level; double px_cur[2]; double A_cur_ref[4]; double h_inv;
  uint8_t patch_with_border[100]; uint8_t patch[64];
} svob200_match_result;
/* depth_ref: n doubles = |ref_frame.pos - point.pos|; px_cur_in: n*2 doubles (initial estimate) */
int svob200_match_direct(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n,
                         const svob200_feature_ref* ftrs, const double* depth_ref,
                         const double* px_cur_in, const svob200_matcher_opts* opts,
                         svob200_match_result* results, int mem);

/* warp::getWarpMatrixAffine (matcher.cpp:36-60, matcher.h:40-48) for n items: px_ref 2, f_ref 3, depth_ref 1,
 * T_cur_ref 7, level_ref 1 per item -> A_cur_ref row-major 2x2 per item */
int svob200_warp_matrix_affine(svob200_ctx* ctx, const svob200_camera* cam, int n, const double* px_ref, const double* f_ref,
                               const double* depth_ref, const double* T_cur_ref, const int* level_ref, double* A_out, int mem);
/* warp::warpAffine (matcher.cpp:83-116, matcher.h:54-61) on a host image level; patch = (2*halfpatch_size)^2 bytes,
 * in/out: left untouched when A_cur_ref inverts to NaN, like the reference */
int svob200_warp_affine(svob200_ctx* ctx, const uint8_t* img, int w, int h, int stride, const double* A_cur_ref, const double* px_ref,
                        int level_ref, int search_level, int halfpatch_size, uint8_t* patch);

/* depthFromTriangulation (matcher.cpp:123-136) for n items: T_search_ref 7, f_ref 3, f_cur 3 per item;
 * depth is in/out (untouched where ok[i] = 0, like the reference's reference parameter) */
int svob200_depth_from_triangulation(svob200_ctx* ctx, int n, const double* T_search_ref, const double* f_ref, const double* f_cur,
                                     double* depth, int* ok);

typedef struct {
  int success; int search_level; int reject; int zmssd_best; int n_evals; int n_steps;
  double depth; double px_cur[2]; double epi_length; double A_cur_ref[4]; double h_inv;
  double epi_dir[2];         /* Matcher::epi_dir_ = A - B on the unit plane (matcher.cpp:224) */
  int px_cur_valid;          /* the reference wrote Matcher::px_cur_ on this call (matcher.cpp:259, :327, :345) */
  uint8_t patch_with_border[100]; uint8_t patch[64];
} svob200_epi_result;
/* d: n*3 doubles (d_estimate, d_min, d_max) */
int svob200_epipolar_match(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n,
                           const svob200_feature_ref* ftrs, const double* d,
                           const svob200_matcher_opts* opts, svob200_epi_result* results, int mem);

/* ---------------------------------------------------------------- depth filter
 * replaces: DepthFilter::updateSeeds loop body (depth_filter.cpp:250-340), DepthFilter::updateSeed
 *           (:368-391), DepthFilter::computeTau (:396-416), Seed ctor (:36-45) */
typedef struct { float a, b, mu, z_range, sigma2; } svob200_seed;
/* status 0: empty slot of a tracker's seed pool; TOO_OLD: erased by the ageing rule (depth_filter.cpp:258-261) */
enum { SVOB200_SEED_BEHIND = 1, SVOB200_SEED_NOT_IN_FRAME = 2, SVOB200_SEED_NO_MATCH = 3,
       SVOB200_SEED_UPDATED = 4, SVOB200_SEED_CONVERGED = 5, SVOB200_SEED_NAN_ERASED = 6, SVOB200_SEED_TOO_OLD = 7 };
typedef struct {
  int status; int search_level; int zmssd_best; int n_evals;
  double z; double px_cur[2]; double epi_length;
} svob200_seed_obs;
/* ftrs[i].T_cur_ref is ignored here: poses come as T_ref_w (7 doubles per seed) and T_cur_w
 * (7 doubles per image of the current batch) because updateSeeds derives both T_ref_cur and
 * T_cur_ref from them (depth_filter.cpp:263, matcher.cpp:216).  seeds: in/out.  obs: out. */
int svob200_seeds_update(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n,
                         const svob200_feature_ref* ftrs, const double* T_ref_w, const double* T_cur_w,
                         const svob200_matcher_opts* opts, double seed_convergence_sigma2_thresh,
                         svob200_seed* seeds, svob200_seed_obs* obs, int mem);
/* scalar helpers with the reference's static signatures (depth_filter.h:126-136); run on device */
int svob200_update_seed(svob200_ctx* ctx, int n, const float* x, const float* tau2, svob200_seed* seeds);
/* diagnostics: sparse alignment decides NLLSSolver's rollback test `new_chi2 > chi2_` (nlls_solver_impl.hpp:56) on the reference's
 * sequentially accumulated `float chi2` (sparse_img_align.cpp:259-263) when the double sums are too close to call.  This entry
 * runs the device replays of that chain over caller-supplied residuals (16 per feature, host memory) with a CTA of `block`
 * threads (128, 256 or 512): sums[0]/counts[0] = one thread adding in order, [1] = the parallel exact replay as the
 * latency-mode (cluster) alignment kernels run it, [2] = as the 128-thread batch kernel runs it (one staging buffer),
 * [3] = as the 256- and 512-thread batch kernels run it (double-buffered).  sums and counts hold 4 entries; all four must
 * be bit-identical for any input. */
int svob200_debug_chi2_chain(svob200_ctx* ctx, int block, int n_features, const float* res, const uint8_t* visible,
                             const uint8_t* contrib, float* sums, int* counts);
int svob200_compute_tau(svob200_ctx* ctx, int n, const double* T_ref_cur, const double* f, const double* z,
                        double px_error_angle, double* tau_out);

/* ---------------------------------------------------------------- glue between the operators
 * The few lines of host code that sit between the operators in the reference, as device kernels, so
 * a whole front-end step can stay on one stream (bit-identical arithmetic):
 *   features_prepare   f = cam2world(px) (feature.h:43-51); depth = |pos - ref_pos|; xyz_ref = f*depth
 *                      (sparse_img_align.cpp:132-134).  image[i] selects the T_ref_w of feature i.
 *   compose_poses      cur.T_f_w = T_cur_from_ref * ref.T_f_w (sparse_img_align.cpp:89)
 *   reproject_prepare  px = cur.w2c(point.pos) (reprojector.cpp:131-145); depth_ref = |ref.pos()-pt.pos|
 *                      and T_cur_ref = cur.T_f_w * ref.T_f_w^-1 (matcher.cpp:169-173); writes
 *                      ftrs[i].T_cur_ref.  T_kf_w: 7 doubles per feature (pose of its keyframe). */
int svob200_features_prepare(svob200_ctx* ctx, const svob200_camera* cam, int n, const double* px,
                             const double* pt_world, const int* image, int batch, const double* T_ref_w,
                             double* f_out /*may be NULL*/, double* xyz_ref_out, int mem);
int svob200_compose_poses(svob200_ctx* ctx, int batch, const svob200_align_result* results,
                          const double* T_ref_w, double* T_cur_w, int mem);
int svob200_reproject_prepare(svob200_ctx* ctx, const svob200_camera* cam, int n, svob200_feature_ref* ftrs,
                              const double* pt_world, const double* T_kf_w, int batch, const double* T_cur_w,
                              double* depth_ref_out, double* px_cur_out, int mem);

/* ---------------------------------------------------------------- tracker: one front-end step per call
 * The chain FrameHandlerMono::processFrame + DepthFilter::updateSeeds run per frame
 * (frame_handler_mono.cpp:171-262, depth_filter.cpp:237-341), restricted to the hot-path operators:
 *   pyramid(cur) -> SparseImgAlign::run(last, cur) -> Matcher::findMatchDirect for every map point of
 *   the keyframe -> DepthFilter::updateSeeds(cur) for the keyframe's seeds,
 * for a batch of independent sequences, 14 kernel launches (15 with the asynchronous depth filter), no host round trip.
 * Finished seeds (converged / NaN) are re-initialised when `reseed` is 1, which keeps the
 * per-frame workload stationary for benchmarking (0 = leave them, the caller mutates its list); with reseed = 2 EVERY seed is
 * re-initialised after every step: the "young seed" regime, where each update walks a long epipolar segment. */
typedef struct svob200_tracker svob200_tracker;
typedef struct {
  double T_cur_w[7];       /* pose after sparse alignment */
  double chi2;
  int n_tracked;           /* SparseImgAlign::run return value */
  int n_matched;           /* successful findMatchDirect */
  int n_seeds_updated, n_seeds_converged, n_seeds_failed, n_seeds_skipped;
  int align_iters, n_exact_chi2;
  int n_reproj_trials;     /* chain mode: Reprojector::n_trials_ */
  int n_pose_obs;          /* chain mode: features left after the pose optimiser (sfba_n_edges_final) */
} svob200_step_stats;
int  svob200_tracker_create(svob200_ctx* ctx, const svob200_camera* cam, int batch, int n_levels,
                            const svob200_align_opts* aopts, const svob200_matcher_opts* mopts,
                            double seed_convergence_sigma2_thresh, float depth_mean, float depth_min, int reseed,
                            svob200_tracker** out);
void svob200_tracker_destroy(svob200_tracker* t);
/* all arguments in host memory; offsets are batch+1 prefix sums.
 * Sizing calls (set_keyframe, set_detector, set_chain, add_keyframes): SVOB200_ERR_NOMEM leaves the tracker as it was. */
int  svob200_tracker_set_keyframe(svob200_tracker* t, const uint8_t* imgs, int stride, const double* T_kf_w,
                                  const int* ftr_offsets, const double* kf_px, const int* kf_level,
                                  const double* pt_world, const int* seed_offsets, const double* seed_px,
                                  const int* seed_level);
int  svob200_tracker_set_last(svob200_tracker* t, const uint8_t* imgs, int stride, int mem);
/* ---- keyframe insertion inside the tracker: DepthFilter::addKeyframe -> initializeSeeds (depth_filter.cpp:109-151), the ageing
 * rule of updateSeeds (:258-261), DepthFilter::removeKeyframe (:153-170) and the erase-on-convergence list semantics (:314-338),
 * device-resident: detect -> seed init -> update never leaves the GPU.
 * svob200_tracker_set_seed_pool (before set_keyframe): every sequence owns `capacity_per_sequence` seed slots (at least the
 *   seeds set_keyframe gives it); up to `max_keyframes` keyframes stay resident (the oldest leaves, its seeds with it); seeds
 *   older than `max_n_kfs` keyframe insertions are erased (DepthFilter::Options::max_n_kfs, default 3); reseed as in
 *   svob200_tracker_create, plus 3 = finished seeds (converged / NaN) leave the pool like they leave the reference's list.
 * svob200_tracker_set_detector: FastDetector(cell size = Config::gridSize, levels = Config::nPyrLevels) and the threshold
 *   DepthFilter::initializeSeeds passes (Config::triangMinCornerScore).  A grid of another cell count releases the detector
 *   scratch, after synchronising with the context's stream.
 * Every sequence has its own keyframe ring, as if it were its own FrameHandlerMono + DepthFilter: its own ring indices
 *   (a free one, else its oldest keyframe leaves), its own Seed::batch_counter and its own evictions.  The keyframe images live
 *   in a store of max_keyframes frame batches (ring index k of sequence b = image b of store frame k); an insertion copies the
 *   selected sequences' images, every pyramid level, into it.
 * svob200_tracker_add_keyframes: the frame of the most recent step becomes a keyframe of the sequences with which[b] != 0
 *   (which: one byte per sequence, NULL = every sequence), with the pose the step gave it: occupancy grid from the frame's
 *   features (= the map points matched in it, AbstractDetector::setExistingFeatures), FAST + Shi-Tomasi + grid selection on
 *   its pyramid, one Seed(ftr, depth_mean, depth_min) per new corner in cell order (batch_id = ++Seed::batch_counter of the
 *   sequence) into the empty slots of the sequence's pool; every map point matched in the frame gains an observation in it
 *   (Feature(frame, px_refined, search_level) + Point::addFrameRef, reprojector.cpp:219-231, frame_handler_mono.cpp:277-279),
 *   and from then on each step matches a point against its closest-view observation (Point::getCloseViewObs,
 *   point.cpp:101-125); when the sequence's oldest keyframe leaves its ring, its seeds are erased (DepthFilter::removeKeyframe)
 *   and its points forget it (Map::safeDeleteFrame).  For a selected sequence the result is what a tracker holding only that
 *   sequence computes; an unselected sequence is left untouched, its counter included.
 *   depth_mean / depth_min: one float per sequence (what FrameHandlerMono passes to DepthFilter::addKeyframe: the mean and
 *   0.5 * min of frame_utils::getSceneDepth, see svob200_tracker_scene_depth).  n_new_seeds / n_dropped (one int per
 *   sequence, may be NULL): seeds created / corners that found no empty slot (0 for an unselected sequence; without a seed
 *   pool, the corners found for both, and n_dropped 0 when n_new_seeds is NULL).  Seed::batch_id is 16 bits wide: a sequence
 *   takes at most 65,534 keyframes; a selected sequence past that is left untouched and reports -1 in both counts (the limit
 *   counts the sequence's own keyframes, not calls).  mem: where ALL
 *   the arrays live.  In SVOB200_MEM_DEVICE mode the call is ordered on the context's stream and does not synchronise with
 *   the host, except that the first insertion after set_keyframe or after set_detector changed the grid allocates the
 *   detector scratch (and the keyframe store when svob200_tracker_set_seed_pool did not).  Not available in
 *   chain mode (SVOB200_ERR_UNSUPPORTED); SVOB200_ERR_ARG before set_keyframe, before the first step, or for a bad mem.
 * svob200_tracker_add_keyframe(t, dm, dn, nn, nd) = svob200_tracker_add_keyframes(t, NULL, dm, dn, nn, nd, SVOB200_MEM_HOST).
 * svob200_tracker_scene_depth: frame_utils::getSceneDepth of the most recent step's frame, per sequence, over the point slots
 *   matched in it (candidates included, like the occupancy grid), z = (T_cur_w * pos).z: depth_mean = (float) the element of
 *   rank n/2 of the ascending depths (vk::getMedian's nth_element), depth_min = (float)(0.5 * min) (the value processFrame
 *   passes), n_points = n (may be NULL).  n == 0 leaves that sequence's depth_mean / depth_min untouched.  mem as above; in
 *   SVOB200_MEM_DEVICE mode the call does not synchronise with the host.
 * svob200_tracker_get_seed_refs: the pool slot by slot (host arrays of svob200_tracker_num_seed_slots entries, any may be NULL);
 *   kf is the ring index of the seed's keyframe in its own sequence's ring, batch_id its sequence's Seed::batch_id. */
int  svob200_tracker_set_seed_pool(svob200_tracker* t, int capacity_per_sequence, int max_keyframes, int max_n_kfs, int reseed);
int  svob200_tracker_set_detector(svob200_tracker* t, int cell_size, int n_detect_levels, double detection_threshold);
int  svob200_tracker_add_keyframes(svob200_tracker* t, const uint8_t* which, const float* depth_mean, const float* depth_min,
                                   int* n_new_seeds, int* n_dropped, int mem);
int  svob200_tracker_add_keyframe(svob200_tracker* t, const float* depth_mean, const float* depth_min, int* n_new_seeds, int* n_dropped);
int  svob200_tracker_scene_depth(svob200_tracker* t, float* depth_mean, float* depth_min, int* n_points, int mem);
int  svob200_tracker_get_seed_refs(svob200_tracker* t, double* px, int* level, int* kf, int* batch_id, int* state);
int  svob200_tracker_num_seed_slots(svob200_tracker* t);
/* ---- point pool: converged seeds become map points on the device (DepthFilter::updateSeeds -> seed_converged_cb_ ->
 * MapPointCandidates::newCandidatePoint, addCandidatePointToFrame, removeFrameCandidates).  Opt-in: without the call nothing changes.
 * svob200_tracker_set_point_pool (before set_keyframe; SVOB200_ERR_ARG after it or for a negative capacity): sequence b owns
 *   max(its set_keyframe points, capacity_per_sequence) point slots, its set_keyframe points first, then empty slots.  From then
 *   on every per-map-feature array of svob200_tracker_step (last_px, px_refined, match_ok) has one entry per SLOT
 *   (svob200_tracker_num_point_slots).  svob200_tracker_set_chain returns SVOB200_ERR_UNSUPPORTED on such a tracker.
 * Creation: a seed whose status in step k is SVOB200_SEED_CONVERGED becomes a candidate, whatever reseed then does to the seed:
 *   position kf.T_f_w.inverse() * (f * (1.0 / mu)), one observation (the seed's feature in its keyframe), type
 *   SVOB200_POINT_CANDIDATE.  A step records at most as many candidates per sequence as the sequence has point slots.
 * Insertion at the head of step k + 2: the reference's depth filter runs one frame behind tracking (its own thread), and so does
 *   the tracker's asynchronous depth filter, whose step k has finished only when step k + 2 starts; every shape (graph, in
 *   place, asynchronous, host or device memory) inserts then, so all give the same results.  Candidates take the sequence's
 *   empty slots in slot order, in the reference's list order (ascending Seed::batch_id, then seed slot).  A candidate that
 *   finds no empty slot, or whose keyframe left the ring in between, is dropped.  From its insertion a candidate is selected,
 *   matched and used in sparse alignment (with the caller's last_px) like every map point; empty slots report match_ok 0.
 * Promotion (svob200_tracker_add_keyframe): a candidate matched in the new keyframe gains the observation and becomes
 *   SVOB200_POINT_UNKNOWN; it marks the detector's occupancy grid like every matched point.  Removal: when a keyframe leaves
 *   the ring, its candidates that were not matched in the new keyframe are deleted and their slots become empty.
 * svob200_tracker_get_points (host arrays, any may be NULL; joins the asynchronous depth filter): per slot 3 doubles pos, the
 *   SVOB200_POINT_* type (DELETED: empty slot) and the observation count; per sequence the candidates created and dropped so far.
 * svob200_tracker_num_point_slots: the slot count (without a pool: the set_keyframe point count). */
int  svob200_tracker_set_point_pool(svob200_tracker* t, int capacity_per_sequence);
int  svob200_tracker_num_point_slots(svob200_tracker* t);
int  svob200_tracker_get_points(svob200_tracker* t, double* pos, int* type, int* n_obs, int* created, int* dropped);
/* Chain mode (call after set_keyframe): between sparse alignment and the depth filter the step runs
 * Reprojector::reprojectMap over the keyframe's map points (grid of cell_size, first success per cell, max_fts) and, with
 * pose_opt != 0, pose_optimizer::optimizeGaussNewton on the matched features — FrameHandlerMono::processFrame's Step 2 and
 * Step 3 (frame_handler_mono.cpp:191-222) — instead of refining every map point; the depth filter then sees the optimised
 * pose.  Every point enters as TYPE_UNKNOWN each frame (the per-point reprojection counters are host-side map management).
 * cell_size <= 0 switches back (the chain arrays stay for the next switch). */
int  svob200_tracker_set_chain(svob200_tracker* t, int cell_size, int max_fts, int pose_opt);
/* cur_imgs: batch images; T_last_w: 7 doubles per sequence (pose of the last frame); last_px: 2 doubles
 * per map feature (its pixel in the last frame).  stats (batch), px_refined (2 per feature), match_ok
 * (1 per feature) may be NULL.  mem tells where ALL pointer arguments live; in device mode level 0 of
 * the current frame aliases cur_imgs and nothing syncs.  For batches above 64 sequences the device-mode step runs the depth
 * filter ASYNCHRONOUSLY on its own stream, like the reference's depth-filter thread (depth_filter.cpp:63-103): the seed update
 * of frame k overlaps the tracking chain of frame k+1, so cur_imgs must stay valid through the next TWO steps, and the seed
 * half of `stats` (n_seeds_*), svob200_tracker_get_seeds and _get_seed_obs are complete only after a joining call
 * (svob200_ctx_sync, svob200_ctx_timer_stop_ms, svob200_dev_download, the getters themselves, any host-memory step);
 * px_refined, match_ok and the tracking half of `stats` are ordered on the context's stream as before. */
int  svob200_tracker_step(svob200_tracker* t, const uint8_t* cur_imgs, int stride, const double* T_last_w,
                          const double* last_px, svob200_step_stats* stats, double* px_refined, int* match_ok, int mem);
int  svob200_tracker_get_seeds(svob200_tracker* t, svob200_seed* out /*host*/);
int  svob200_tracker_launches_per_step(void);   /* kernels of a default-mode step on one stream: 14 (one more when the depth filter runs
                                                   on its own stream and the step records are written in two halves) */
/* diagnostics: the raw svob200_align_result records (one per sequence) of the most recent step, to host memory */
int  svob200_tracker_debug_align(svob200_tracker* t, svob200_align_result* out);
/* optional CUDA-event timing of the most recent step, one duration per stage (events recorded on the
 * launching stream between the kernels): stage names from svob200_tracker_stage_name(i), i < num_stages */
int  svob200_tracker_enable_profiling(svob200_tracker* t, int on);
int  svob200_tracker_num_stages(void);
const char* svob200_tracker_stage_name(int i);
int  svob200_tracker_stage_ms(svob200_tracker* t, float* ms, int cap);
int  svob200_tracker_get_seed_obs(svob200_tracker* t, svob200_seed_obs* out /*host*/);
/* bytes of device memory the tracker's own arrays hold now (its frames, held by the context's frame store, not included) */
long long svob200_tracker_device_bytes(const svob200_tracker* t);

/* ================================================================ callers either side of the hot path
 * (SURVEY.md §8f "next" rows; same conventions: POD, mem = HOST | DEVICE, int status) */

/* ---------------------------------------------------------------- camera input stage
 * replaces: ImageProcess::GetCVImage + YUV2RGB (../image_process.cpp:97-186: YUV_420_888 -> RGBA, integer) followed by
 *           cv::cvtColor(img, COLOR_RGBA2GRAY) (../svo_system.cpp:49-51; OpenCV 4.5.4 imgproc, 15-bit fixed point) and
 *           Frame::initFrame -> createImgPyramid (frame.cpp:51-64, :186-195).
 * One fused kernel reads the planes once, writes level 0 (gray) once and every coarser level once.
 * y/u/v, strides and pixel stride are what AImage_getPlaneData / getPlaneRowStride / getPlanePixelStride return
 * (u, v may be views into one interleaved buffer, pixel stride 2).  Image b of a batch starts y_image_stride /
 * uv_image_stride bytes after image b-1 (ignored for batch 1).  Crop rect = whole image. */
int svob200_frame_upload_yuv420(svob200_ctx* ctx, int64_t frame_id, const uint8_t* y, int y_stride, const uint8_t* u,
                                const uint8_t* v, int uv_stride, int uv_pixel_stride, size_t y_image_stride,
                                size_t uv_image_stride, const int* round_modes, int mem);

/* ---------------------------------------------------------------- reprojector
 * replaces: Reprojector::reprojectMap / reprojectCell / reprojectPoint (reprojector.cpp:72-259) incl. Point::getCloseViewObs
 *           (point.cpp:101-125) and Matcher::findMatchDirect per candidate.
 * The caller flattens its map the way reprojectMap walks it (features of the close keyframes in closeness order, each
 * point once, then the point candidates): points of image b are points[point_offsets[b] .. point_offsets[b+1]) in that
 * insertion order; observation k of a point is obs[k] (ref_frame_id / ref_image / level / type / px / f / grad are read;
 * cur_image and T_cur_ref are ignored) seen from the keyframe pose T_obs_w[7k..], in Point::obs_ list order.
 * The per-point status tells the caller which side effects the reference would have applied:
 *   FAILED  -> ++n_failed_reproj_ (and the deletion rules, :204-208)    MATCHED -> ++n_succeeded_reproj_, new Feature
 *   DELETED -> the candidate was met and erased (:190-194)              UNTRIED -> in a cell, never reached
 * cell_winner: batch * n_cells point indices (-1 = none), n_cells = ceil(W/cell)*ceil(H/cell); the new features of the
 * frame are the winners in cell order.  stats: one record per image (n_matches_ / n_trials_). */
enum { SVOB200_POINT_DELETED = 0, SVOB200_POINT_CANDIDATE = 1, SVOB200_POINT_UNKNOWN = 2, SVOB200_POINT_GOOD = 3 };   /* point.h */
enum { SVOB200_REPROJ_NOT_IN_FRAME = 0, SVOB200_REPROJ_UNTRIED = 1, SVOB200_REPROJ_DELETED = 2, SVOB200_REPROJ_FAILED = 3,
       SVOB200_REPROJ_MATCHED = 4 };
typedef struct { double pos[3]; int type; int obs_begin, obs_end; int reserved; } svob200_map_point;
typedef struct { int status, cell, obs, search_level; double px[2]; double A_cur_ref[4]; } svob200_reproj_result;
typedef struct { int n_matches, n_trials, n_in_frame, n_cells; } svob200_reproj_stats;
int svob200_reproject_map(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int batch, const double* T_cur_w,
                          const int* point_offsets, int n_points, const svob200_map_point* points, int n_obs,
                          const svob200_feature_ref* obs, const double* T_obs_w, int cell_size, int max_fts,
                          const svob200_matcher_opts* opts, svob200_reproj_result* results, int* cell_winner,
                          svob200_reproj_stats* stats, int mem);

/* ---------------------------------------------------------------- pose / structure optimisation
 * replaces: pose_optimizer::optimizeGaussNewton (pose_optimizer.cpp:31-181) with vk::robust_cost::MADScaleEstimator and
 *           TukeyWeightFunction (robust_cost.cpp), one problem per image of the batch: features of image b are
 *           [ftr_offsets[b], ftr_offsets[b+1]) with bearing f (3), pyramid level and world point pos (3).
 *           T_f_w: 7 doubles per image, in/out.  outlier[i] = 1 where the reference resets ftr->point (:149-153).
 *           Frame::Cov_ = (A * errorMultiplier2^2)^-1 is left to the caller (A is returned). */
typedef struct {
  double A[36];            /* normal matrix of the last linearisation, row-major */
  double chi2, estimated_scale, error_init, error_final;
  int iters, num_obs, rolled_back, reserved;
} svob200_pose_opt_result;
typedef struct { double reproj_thresh; int n_iter; double eps; float tukey_b; } svob200_pose_opt_opts;
void svob200_pose_opt_opts_default(svob200_pose_opt_opts* o);   /* Config::poseOptimThresh 2.0, poseOptimNumIter 10, EPS, DEFAULT_B */
int svob200_pose_optimize(svob200_ctx* ctx, const svob200_camera* cam, int batch, const int* ftr_offsets, const double* f,
                          const int* level, const double* pos, const svob200_pose_opt_opts* opts, double* T_f_w,
                          svob200_pose_opt_result* results, uint8_t* outlier, int mem);
/* replaces: Point::optimize (point.cpp:130-192) for n points (FrameHandlerBase::optimizeStructure picks them,
 *           frame_handler_base.cpp:190-210): observations of point i are [obs_offsets[i], obs_offsets[i+1]) with the
 *           observing frame's pose T_f_w (7) and bearing f (3), in Point::obs_ list order.  pos: 3 per point, in/out. */
int svob200_points_optimize(svob200_ctx* ctx, int n, const int* obs_offsets, const double* T_f_w, const double* f,
                            int n_iter, double eps, double* pos, int* iters_out /* may be NULL */, int mem);

/* ---------------------------------------------------------------- seed initialisation
 * replaces: DepthFilter::initializeSeeds (depth_filter.cpp:129-151): AbstractDetector::setExistingFeatures
 *           (feature_detection.cpp:40-58), FastDetector::detect, one Seed (depth_filter.cpp:36-45) per new corner.
 * existing_px: level-0 pixels of the frame's features, image b owns [existing_offsets[b], existing_offsets[b+1]).
 * depth_mean / depth_min: one per image.  Outputs are compacted in cell order: image b writes counts[b] entries at
 * [b * n_cells, ...). */
int svob200_seeds_initialize(svob200_ctx* ctx, int64_t frame_id, int n_detect_levels, int cell_size, double detection_threshold,
                             const int* existing_offsets, const double* existing_px, const float* depth_mean,
                             const float* depth_min, svob200_corner* corners_out, svob200_seed* seeds_out, int* counts, int mem);

/* ---------------------------------------------------------------- device-side helpers for the
 * resident ("value") path and the synthetic bench: raw device allocations and a plane renderer.
 * Not part of the reference surface. */
int svob200_dev_alloc(svob200_ctx* ctx, size_t bytes, void** dptr);
int svob200_dev_free(svob200_ctx* ctx, void* dptr);
int svob200_dev_upload(svob200_ctx* ctx, void* dptr, const void* host, size_t bytes);
int svob200_dev_download(svob200_ctx* ctx, void* host, const void* dptr, size_t bytes);
int svob200_host_alloc_pinned(svob200_ctx* ctx, size_t bytes, void** hptr);
int svob200_host_free_pinned(svob200_ctx* ctx, void* hptr);
/* render `batch` views of the textured plane z = plane_z into device memory (dense, w*h each) */
int svob200_synth_render(svob200_ctx* ctx, const uint8_t* dev_texture, int tex_size, double ppm, double plane_z,
                         const svob200_camera* cam, int batch, const double* T_f_w /*host, 7 per image*/,
                         uint8_t* dev_out);

#ifdef __cplusplus
}
#endif
#endif
