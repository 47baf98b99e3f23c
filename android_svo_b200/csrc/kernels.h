// kernels.h — host-side launchers of the CUDA kernels (internal to libsvob200).  A launcher returns the first error of its
// own launches (cudaSuccess when it launched nothing).
#pragma once
#include "common.cuh"

// Cell grids (the reprojector's, the keyframe detector's) of at most this many cells: reproj_cells_kernel and
// kf_append_seeds_kernel keep one shared-memory entry per cell.  Entry points refuse larger grids before staging anything.
constexpr int kMaxGridCells = 8192;
// cells of a grid of cell x cell pixels over a w x h image (partial cells at the right and bottom edges count)
inline long long grid_cells(int w, int h, int cell) { return (long long)((w + cell - 1) / cell) * ((h + cell - 1) / cell); }

struct AlignProblemDev;   // sparse_align.cu

// pyramid.cu
cudaError_t launch_pyramid(const DevFrame& f, const int* modes, cudaStream_t s, long long* launches);
// camera planes as AImage hands them out (../image_process.cpp:151-186): strides in bytes, image strides for batches
struct YuvPlanes {
  const uint8_t *y = nullptr, *u = nullptr, *v = nullptr;
  int y_stride = 0, uv_stride = 0, uv_pixel_stride = 1;
  unsigned long long y_img_stride = 0, uv_img_stride = 0;
};
cudaError_t launch_pyramid_yuv(const DevFrame& f, const YuvPlanes& yuv, const int* modes, cudaStream_t s, long long* launches);
cudaError_t launch_half_sample_single(const uint8_t* in, int in_pitch, int w, int h, uint8_t* out, int out_pitch, int mode,
                                      cudaStream_t s, long long* launches);

// fast.cu
// keys: batch*n_cells 64-bit cell records (device scratch); raw_scores: optional w*h score map of
// (raw_image, raw_level) for svob200_fast_corners.  d_image_sel (optional, one int per image): images with a negative entry
// are not scored (their cells are not written, their count is 0).
cudaError_t launch_fast_detect(const DevFrame& f, int n_detect_levels, int cell, int grid_cols, int grid_rows, double thr,
                               const uint8_t* d_occupancy, unsigned long long* d_keys, svob200_corner* d_cells, int* d_counts,
                               cudaStream_t s, long long* launches, const int* d_image_sel = nullptr);
cudaError_t launch_fast_raw(const DevFrame& f, int image, int level, int threshold, int nonmax, uint8_t* d_scores,
                            cudaStream_t s, long long* launches);

// sparse_align.cu
size_t sparse_align_scratch_bytes(int total_features);
cudaError_t launch_sparse_align(const DevFrame& ref, const DevFrame& cur, const DevCam& cam, int batch, int total_features, int max_per_problem,
                                const int* d_offsets, const double* d_px, const double* d_xyz, const uint8_t* d_has_point,
                                const double* d_T_init, svob200_align_opts opts, svob200_align_result* d_results,
                                void* d_scratch, cudaStream_t s, long long* launches,
                                const double* d_T_ref_w = nullptr, double* d_T_cur_w = nullptr);   // optional: T_cur_w = T_cur_ref * T_ref_w per problem

cudaError_t launch_chi2_chain_test(int block, const float* d_res, const uint8_t* d_visible, const uint8_t* d_contrib, int n, float* d_sums, int* d_cnts,
                                   cudaStream_t s, long long* launches);

// matcher.cu
size_t lk_jobs_bytes(int n);                 // scratch of launch_align_patches / launch_match_direct
cudaError_t launch_align_patches(const DevFrame* d_frames, int slot, int level, int n, const int* d_image, const uint8_t* d_pwb, const uint8_t* d_patch,
                                 const float* d_dir, int n_iter, double* d_px, int* d_converged, double* d_h_inv, void* d_scratch,
                                 cudaStream_t s, long long* launches);
// results: full records (API) or nullptr; px_out / ok_out: compact outputs (tracker) or nullptr; the scratch
// (match_scratch_bytes(scratch_total)) is indexed from `first`; marks: optional 2 events between the three kernels
size_t match_scratch_bytes(int n);
cudaError_t launch_match_direct(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs,
                                const double* d_depth_ref, const double* d_px_in, svob200_matcher_opts opts, svob200_match_result* d_results,
                                double* d_px_out, int* d_ok_out, void* d_scratch, int scratch_total, int first, cudaStream_t s, long long* launches,
                                cudaEvent_t* marks = nullptr, const uint8_t* d_active = nullptr /* per-candidate mask */,
                                int* d_level_out = nullptr, double* d_A_out = nullptr /* search level and A_cur_ref (4) per candidate */);
size_t epipolar_scratch_bytes(int n);
cudaError_t launch_epipolar(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs, const double* d_d,
                            svob200_matcher_opts opts, svob200_epi_result* d_results, void* d_scratch, cudaStream_t s, long long* launches);
size_t seeds_scratch_bytes(int n);
cudaError_t launch_seeds_update(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs,
                                const double* d_T_ref_w, const double* d_T_cur_w, svob200_matcher_opts opts, double conv_thresh,
                                svob200_seed* d_seeds, svob200_seed_obs* d_obs, void* d_scratch, int scratch_total, int first,
                                cudaStream_t s, long long* launches, cudaEvent_t* marks = nullptr /* 3 events between the four kernels */);
// The tracker's compact seed record (64 B, two sectors): the reference feature of a seed is (px, f, level) in keyframe `kf` of
// image `image`; the keyframe's frame slot comes from a table indexed by kf, and everything that depends only on the pair
// (keyframe, image) — the relative poses of depth_filter.cpp:263 / matcher.cpp:216 and the pixel error angle — from a table the
// step refreshes with one tiny kernel instead of ~600 FP64 instructions per seed.  (f = cam2world(px) stays in the record:
// recomputing it costs two divisions, a square root and three more divisions per seed and kernel, more than 24 bytes of HBM.)
// state: 0 alive, 1 free slot.  batch_id: Seed::batch_id (depth_filter.h:38) for the ageing rule.
struct __align__(16) SeedRef {
  double px[2];
  double f[3];
  int image;
  uint8_t level, kf; uint16_t batch_id;
  uint8_t state, pad0; uint16_t pad1;
  int pad2[3];
};
static_assert(sizeof(SeedRef) == 64, "SeedRef must be two 32-byte sectors");
// per (keyframe, image): T_ref_cur = ref.T_f_w * cur.T_f_w^-1 (depth_filter.cpp:263), its inverse (:264), the matcher's
// T_cur_ref = cur.T_f_w * ref.T_f_w^-1 (matcher.cpp:216) and px_error_angle (depth_filter.cpp:245-247)
struct __align__(16) SeedPoseRec { double T_ref_cur[7], T_cur_ref[7], T_cur_ref_m[7]; double px_error_angle; };
static_assert(sizeof(SeedPoseRec) == 176, "SeedPoseRec layout");
// rows (keyframe k, image b), b in [image0, image0 + n_images), of the pose table: run after the step's final T_cur_w is known
cudaError_t launch_seed_pose_table(const DevCam& cam, int batch, int n_kfs, int image0, int n_images, const double* d_T_kf_w, const double* d_T_cur_w,
                                   SeedPoseRec* d_pose_table, cudaStream_t s, long long* launches);
// d_batch_counter / max_n_kfs: Seed::batch_counter of every sequence (indexed by SeedRef::image) and DepthFilter::Options::max_n_kfs
// (seeds older than that are erased, :258-261)
cudaError_t launch_seeds_update_compact(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, SeedRef* d_refs,
                                        const int* d_kf_slot, int batch, const SeedPoseRec* d_pose_table, const int* d_batch_counter, int max_n_kfs,
                                        svob200_matcher_opts opts, double conv_thresh,
                                        svob200_seed* d_seeds, svob200_seed_obs* d_obs, void* d_scratch, int scratch_total, int first,
                                        cudaStream_t s, long long* launches, cudaEvent_t* marks = nullptr);
cudaError_t launch_update_seed(int n, const float* d_x, const float* d_tau2, svob200_seed* d_seeds, cudaStream_t s, long long* launches);
cudaError_t launch_compute_tau(int n, const double* d_T, const double* d_f, const double* d_z, double angle, double* d_out,
                               cudaStream_t s, long long* launches);

// map_ops.cu — reprojector, pose optimizer, point optimizer (SURVEY §8f)
size_t reproject_scratch_bytes(int n_points);
// the caller checks that the grid has at most kMaxGridCells cells (grid_cells(cam.width, cam.height, cell_size))
cudaError_t launch_reproject_map(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int batch, const double* d_T_cur_w, const int* d_pt_off,
                                 int n_points, const svob200_map_point* d_points, const svob200_feature_ref* d_obs, const double* d_T_obs_w,
                                 int cell_size, int max_fts, svob200_matcher_opts opts, svob200_reproj_result* d_results, int* d_cell_winner,
                                 svob200_reproj_stats* d_stats, void* d_scratch, void* d_match_scratch,
                                 double* d_m_f, int* d_m_level, double* d_m_pos, int* d_m_point, int* d_m_count,   // optional compacted matches
                                 cudaStream_t s, long long* launches,
                                 int image_base = 0, int point_base = 0, int n_range = -1 /* sub-range of a larger batch (tracker chunks) */);
cudaError_t launch_pose_optimize(const DevCam& cam, int batch, const int* d_seg_begin, const int* d_seg_end, const double* d_f, const int* d_level,
                                 const double* d_pos, double reproj_thresh, int n_iter, double eps, float tukey_b, double* d_T_io,
                                 svob200_pose_opt_result* d_results, uint8_t* d_outlier, double* d_work, cudaStream_t s, long long* launches);
cudaError_t launch_points_optimize(int n, const int* d_obs_off, const double* d_T_f_w, const double* d_f, int n_iter, double eps, double* d_pos_io,
                                   int* d_iters, cudaStream_t s, long long* launches);
cudaError_t launch_occupancy(int batch, int max_per_image, const int* d_off, const double* d_px, int cell_size, int grid_cols, int n_cells, uint8_t* d_occ,
                             cudaStream_t s, long long* launches);
cudaError_t launch_seeds_compact(int batch, const svob200_corner* d_cells, int n_cells, double thr, const float* d_depth_mean, const float* d_depth_min,
                                 svob200_corner* d_corners_out, svob200_seed* d_seeds_out, int* d_counts, cudaStream_t s, long long* launches);

// synth.cu
cudaError_t launch_synth_render(const uint8_t* d_tex, int tex_size, double ppm, double plane_z, const DevCam& cam, int batch,
                                const double* d_T_w_f_R_c /*12 doubles per image: R row-major + c*/, uint8_t* d_out,
                                cudaStream_t s, long long* launches);

// glue.cu
cudaError_t launch_features_prepare(const DevCam& cam, int n, const double* d_px, const double* d_pt, const int* d_image,
                                    const double* d_T_ref_w, double* d_f, double* d_xyz, cudaStream_t s, long long* launches);
cudaError_t launch_compose_poses(int batch, const svob200_align_result* d_res, const double* d_T_ref_w, double* d_T_cur_w,
                                 cudaStream_t s, long long* launches);
cudaError_t launch_reproject_prepare(const DevCam& cam, int n, svob200_feature_ref* d_ftrs, const double* d_pt, const double* d_T_kf_w,
                                     const double* d_T_cur_w, double* d_depth_ref, double* d_px_cur, cudaStream_t s, long long* launches);



// stand-alone helpers behind the C++ drop-in (vk::shiTomasiScore, warp::getWarpMatrixAffine, warp::warpAffine)
cudaError_t launch_shi_tomasi_points(const uint8_t* d_img, int pitch, int cols, int rows, int n, const int* d_uv, float* d_out,
                                     cudaStream_t s, long long* launches);
cudaError_t launch_warp_matrix(const DevCam& cam, int n, const double* d_px_ref, const double* d_f_ref, const double* d_depth_ref,
                               const double* d_T_cur_ref, const int* d_level_ref, double* d_A_out, cudaStream_t s, long long* launches);
cudaError_t launch_warp_affine(const uint8_t* d_img, int pitch, int cols, int rows, const double* A, const double* px_ref, int level_ref,
                               int search_level, int halfpatch, uint8_t* d_patch, cudaStream_t s, long long* launches);
cudaError_t launch_triangulate(int n, const double* d_T, const double* d_f_ref, const double* d_f_cur, double* d_depth, int* d_ok,
                               cudaStream_t s, long long* launches);
