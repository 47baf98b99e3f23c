// map_ops.cu — the callers either side of the tracking hot path (SURVEY.md §8f), as device kernels:
//   Reprojector::reprojectMap / reprojectCell / reprojectPoint     reprojector.cpp:72-259  (+ Point::getCloseViewObs point.cpp:101-125)
//   pose_optimizer::optimizeGaussNewton                            pose_optimizer.cpp:31-181
//   Point::optimize                                                point.cpp:130-192
//
// Reprojector.  The reference walks the grid cell by cell and, inside a cell, tries the candidates one after the other
// (sorted by point quality) until the first findMatchDirect succeeds; it stops after maxFts matches.  Here every
// in-frame candidate is matched in parallel (the batched findMatchDirect pipeline of matcher.cu) and the sequential
// rules are evaluated afterwards on the outcomes, which gives the same observable result:
//   * winner of a cell   = the successful candidate with the smallest key (3 - type, insertion index)  [stable sort + first success]
//   * tried candidates   = those with a key below the winner's (all of them if the cell has no winner)   [n_trials, n_failed_reproj]
//   * visited cells      = those whose exclusive prefix count of matched cells is <= maxFts              [the break at :164]
// Pose optimizer: one CTA per frame; per-feature terms in parallel, 28 double accumulators reduced by a fixed tree
// (deterministic), thread 0 solves with Eigen's exact LDLT association (ldlt.cuh) and takes the decisions.  The medians
// (vk::getMedian = nth_element at n/2) are order statistics found by rank counting.
#include "ctx_internal.h"
#include "ldlt.cuh"

namespace {

__device__ __forceinline__ v3d frame_pos(const double* T)           // Frame::pos() frame.h:105
{
  double inv[7];
  se3_inverse(T, inv);
  return {inv[0], inv[1], inv[2]};
}

// ---------------------------------------------------------------- reprojector, phase 1: per point
// reprojectPoint (:246-259) + the head of findMatchDirect (getCloseViewObs, matcher.cpp:161-173)
__global__ void __launch_bounds__(128) reproj_select_kernel(DevCam cam, const double* T_cur_w, const int* pt_off, const svob200_map_point* pts,
                                                            const svob200_feature_ref* obs, const double* T_obs_w, int cell_size, int grid_cols,
                                                            int image_base, svob200_feature_ref* ftr_out, double* depth_ref, double* px_in, uint8_t* active,
                                                            svob200_reproj_result* results)
{
  const int b = blockIdx.x;     // image inside the current frame batch
  const double* T = T_cur_w + 7 * (size_t)b;
  const v3d cur_pos = frame_pos(T);
  for (int i = pt_off[b] + threadIdx.x; i < pt_off[b + 1]; i += blockDim.x) {
    const svob200_map_point p = pts[i];
    const v3d pos = {p.pos[0], p.pos[1], p.pos[2]};
    const v3d pf = se3_transform(T, pos);
    double px, py;
    world2cam(cam, pf, px, py);
    svob200_reproj_result r;
    r.status = SVOB200_REPROJ_NOT_IN_FRAME; r.cell = -1; r.obs = -1; r.search_level = 0; r.px[0] = px; r.px[1] = py;
    r.A_cur_ref[0] = r.A_cur_ref[1] = r.A_cur_ref[2] = r.A_cur_ref[3] = 0.0;
    uint8_t act = 0;
    double dref = 0.0;
    if (in_frame(cam, x86_d2i(px), x86_d2i(py), 8)) {
      r.cell = x86_d2i(py / cell_size) * grid_cols + x86_d2i(px / cell_size);
      r.status = SVOB200_REPROJ_UNTRIED;
      if (p.type != SVOB200_POINT_DELETED && p.obs_end > p.obs_begin) {
        // Point::getCloseViewObs: arg-max of the cosine over obs_ in list order, strict >, starting from 0
        v3d od = normalized3({cur_pos.x - pos.x, cur_pos.y - pos.y, cur_pos.z - pos.z});
        int best = p.obs_begin;
        double min_cos = 0.0;
        v3d best_pos = {0, 0, 0};
        for (int k = p.obs_begin; k < p.obs_end; ++k) {
          const v3d op = frame_pos(T_obs_w + 7 * (size_t)k);
          const v3d d = normalized3({op.x - pos.x, op.y - pos.y, op.z - pos.z});
          const double c = dot3(od, d);
          if (k == p.obs_begin) best_pos = op;
          if (c > min_cos) { min_cos = c; best = k; best_pos = op; }
        }
        r.obs = best;
        if (!(min_cos < 0.5)) {
          act = 1;
          svob200_feature_ref f = obs[best];
          f.cur_image = image_base + b;
          double inv[7];
          se3_inverse(T_obs_w + 7 * (size_t)best, inv);
          se3_mul(T, inv, f.T_cur_ref);
          ftr_out[i] = f;
          dref = norm3({best_pos.x - pos.x, best_pos.y - pos.y, best_pos.z - pos.z});
        }
      }
    }
    active[i] = act;
    depth_ref[i] = dref;
    px_in[2 * (size_t)i] = px; px_in[2 * (size_t)i + 1] = py;
    results[i] = r;
  }
}

// ---------------------------------------------------------------- reprojector, phase 2: per image, the sequential rules
constexpr int REPROJ_T = 256;
constexpr int REPROJ_MAX_CELLS = 8192;       // 32 KB of keys in shared memory (1080p at cell 20 has 5,184)

__global__ void __launch_bounds__(REPROJ_T) reproj_cells_kernel(DevCam cam, const int* pt_off, const svob200_map_point* pts, const uint8_t* active,
                                                                const int* ok, const double* px_refined, const int* level, const double* A,
                                                                int n_cells, int max_fts, svob200_reproj_result* results, int* cell_winner,
                                                                svob200_reproj_stats* stats,
                                                                // optional compacted matches of image b at [b * n_cells, ...) in cell order
                                                                double* m_f, int* m_level, double* m_pos, int* m_point, int* m_count)
{
  __shared__ uint32_t s_best[REPROJ_MAX_CELLS];
  __shared__ int s_cnt[4];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int p0 = pt_off[b], p1 = pt_off[b + 1];
  for (int c = tid; c < n_cells; c += REPROJ_T) s_best[c] = 0xffffffffu;
  if (tid < 4) s_cnt[tid] = 0;
  __syncthreads();
  // winner of every cell: smallest (3 - type, insertion index) among the successful, non-deleted candidates
  for (int i = p0 + tid; i < p1; i += REPROJ_T) {
    const int cell = results[i].cell;
    if (cell >= 0 && active[i] && ok[i]) atomicMin(&s_best[cell], ((uint32_t)(3 - pts[i].type) << 28) | (uint32_t)(i - p0));
  }
  __syncthreads();
  // visited cells: exclusive prefix count of matched cells <= max_fts (reprojector.cpp:152-166)
  const int chunk = (n_cells + REPROJ_T - 1) / REPROJ_T;
  const int c0 = min(tid * chunk, n_cells), c1 = min(c0 + chunk, n_cells);
  int local = 0;
  for (int c = c0; c < c1; ++c) local += s_best[c] != 0xffffffffu;
  int total;
  int run = block_exclusive_scan<REPROJ_T>(local, &total);   // matched cells before c0
  int my_matches = 0;
  for (int c = c0; c < c1; ++c) {
    const bool has = s_best[c] != 0xffffffffu;
    const bool visited = run <= max_fts;
    int w = -1;
    if (has && visited) {
      w = p0 + (int)(s_best[c] & 0x0fffffffu);
      ++my_matches;
      if (m_point) {
        const size_t o = (size_t)b * n_cells + run;
        m_point[o] = w;
        const double u = px_refined[2 * (size_t)w], v = px_refined[2 * (size_t)w + 1];
        const v3d f = cam2world(cam, u, v);             // Feature ctor (feature.h:43-51)
        m_f[3 * o] = f.x; m_f[3 * o + 1] = f.y; m_f[3 * o + 2] = f.z;
        m_level[o] = level[w];
        m_pos[3 * o] = pts[w].pos[0]; m_pos[3 * o + 1] = pts[w].pos[1]; m_pos[3 * o + 2] = pts[w].pos[2];
      }
    }
    if (!visited) s_best[c] = 0xfffffffeu;             // marks "not visited" for the per-point pass (never a valid key)
    cell_winner[(size_t)b * n_cells + c] = w;
    run += has;
  }
  atomicAdd(&s_cnt[0], my_matches);
  __syncthreads();
  // per point: status and the trial count
  int trials = 0, in_frame_cnt = 0;
  for (int i = p0 + tid; i < p1; i += REPROJ_T) {
    svob200_reproj_result r = results[i];
    if (r.cell < 0) continue;
    ++in_frame_cnt;
    const uint32_t best = s_best[r.cell];
    const int type = pts[i].type;
    const uint32_t key = ((uint32_t)(3 - type) << 28) | (uint32_t)(i - p0);
    int status = SVOB200_REPROJ_UNTRIED;
    if (best != 0xfffffffeu) {
      if (key < best) status = type == SVOB200_POINT_DELETED ? SVOB200_REPROJ_DELETED : SVOB200_REPROJ_FAILED;
      else if (key == best) status = SVOB200_REPROJ_MATCHED;
    }
    if (status != SVOB200_REPROJ_UNTRIED) ++trials;
    r.status = status;
    if ((status == SVOB200_REPROJ_MATCHED || status == SVOB200_REPROJ_FAILED) && active[i]) {
      r.px[0] = px_refined[2 * (size_t)i]; r.px[1] = px_refined[2 * (size_t)i + 1];
      r.search_level = level[i];
      for (int k = 0; k < 4; ++k) r.A_cur_ref[k] = A[4 * (size_t)i + k];
    }
    results[i] = r;
  }
  trials = warp_sum_i(trials); in_frame_cnt = warp_sum_i(in_frame_cnt);
  if ((tid & 31) == 0) { atomicAdd(&s_cnt[1], trials); atomicAdd(&s_cnt[2], in_frame_cnt); }
  __syncthreads();
  if (tid == 0) {
    if (stats) { stats[b].n_matches = s_cnt[0]; stats[b].n_trials = s_cnt[1]; stats[b].n_in_frame = s_cnt[2]; stats[b].n_cells = n_cells; }
    if (m_count) m_count[b] = s_cnt[0];
  }
}

// ---------------------------------------------------------------- pose optimizer
constexpr int POSE_T = 128;         // a frame has ~100-1,000 matched features; 3 CTAs per SM (launch bounds) for batches
constexpr int POSE_ACC = 28;        // 21 (upper triangle of A) + 6 (b) + 1 (chi2)

// element n/2 of the sorted data (vk::getMedian, math_utils.h:125-131), by rank counting; all threads get the value
__device__ double block_median(const double* v, int n, double* s_out)
{
  const int k = n / 2;
  if (threadIdx.x == 0) *s_out = 0.0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double x = v[i];
    int lt = 0, le = 0;
    for (int j = 0; j < n; ++j) { const double y = v[j]; lt += y < x; le += y <= x; }
    if (lt <= k && k < le) *s_out = x;          // every thread that qualifies writes the same value
  }
  __syncthreads();
  const double m = *s_out;
  __syncthreads();
  return m;
}

// the reprojection error of one feature at pose T, scaled by 1/(1 << level) (pose_optimizer.cpp:49-53, :80-84)
__device__ __forceinline__ void pose_residual(const double* T, const double* f, const double* pos, int level, v3d& p, double& e0, double& e1, double& sic)
{
  p = se3_transform(T, {pos[0], pos[1], pos[2]});
  e0 = f[0] / f[2] - p.x / p.z;
  e1 = f[1] / f[2] - p.y / p.z;
  sic = 1.0 / (1 << level);
  e0 *= sic; e1 *= sic;
}

__global__ void __launch_bounds__(POSE_T, 3) pose_optimize_kernel(DevCam cam, const int* seg_begin, const int* seg_end, const double* f_all,
                                                               const int* level_all, const double* pos_all, double reproj_thresh, int n_iter,
                                                               double eps, float tukey_b, double* T_io, svob200_pose_opt_result* results,
                                                               uint8_t* outlier_all, double* work_all)
{
  __shared__ double s_red[POSE_T / 32][POSE_ACC];
  __shared__ double s_T[7], s_med;
  __shared__ int s_flag;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = seg_begin[b], n = seg_end[b] - i0;
  const double* F = f_all + 3 * (size_t)i0;
  const double* P = pos_all + 3 * (size_t)i0;
  const int* LV = level_all + i0;
  double* work = work_all + i0;
  svob200_pose_opt_result* R = &results[b];
  if (n <= 0) {                                   // errors.empty(): return untouched (:56-57)
    if (tid == 0) {
      for (int k = 0; k < 36; ++k) R->A[k] = 0.0;
      R->chi2 = R->estimated_scale = R->error_init = R->error_final = 0.0; R->iters = 0; R->num_obs = 0; R->rolled_back = 0;
    }
    return;
  }
  if (tid < 7) s_T[tid] = T_io[7 * (size_t)b + tid];
  __syncthreads();
  const double em2 = fabs(cam.fx);               // errorMultiplier2 (pinhole_camera.h:64-67)
  double T[7];
  for (int k = 0; k < 7; ++k) T[k] = s_T[k];
  // scale estimate: 1.48 * median of the (float) error norms == 1.48f * (float)sqrt(median of the squared norms)
  for (int i = tid; i < n; i += POSE_T) {
    v3d p; double e0, e1, sic;
    pose_residual(T, F + 3 * i, P + 3 * i, LV[i], p, e0, e1, sic);
    work[i] = e0 * e0 + e1 * e1;
  }
  __syncthreads();
  const double med_init = block_median(work, n, &s_med);
  const float est_f = 1.48f * (float)sqrt(med_init);
  const double estimated_scale = (double)est_f;
  double scale = estimated_scale;
  const float b_square = tukey_b * tukey_b;
  double chi2 = 0.0, T_old[7];
  for (int k = 0; k < 7; ++k) T_old[k] = T[k];
  int iters = 0, rolled_back = 0;
  double A[36];
  for (int k = 0; k < 36; ++k) A[k] = 0.0;
  for (int iter = 0; iter < n_iter; ++iter) {
    if (iter == 5) scale = 0.85 / em2;
    double acc[POSE_ACC];
#pragma unroll
    for (int k = 0; k < POSE_ACC; ++k) acc[k] = 0.0;
    for (int i = tid; i < n; i += POSE_T) {
      v3d p; double e0, e1, sic;
      pose_residual(T, F + 3 * i, P + 3 * i, LV[i], p, e0, e1, sic);
      // Frame::jacobian_xyz2uv frame.h:110-132, then J *= sqrt_inv_cov
      const double x = p.x, y = p.y, z_inv = 1. / p.z, z_inv_2 = z_inv * z_inv;
      double J0[6], J1[6];
      J0[0] = -z_inv; J0[1] = 0.0; J0[2] = x * z_inv_2; J0[3] = y * J0[2]; J0[4] = -(1.0 + x * J0[2]); J0[5] = y * z_inv;
      J1[0] = 0.0; J1[1] = -z_inv; J1[2] = y * z_inv_2; J1[3] = 1.0 + y * J1[2]; J1[4] = -J0[3]; J1[5] = -x * z_inv;
#pragma unroll
      for (int k = 0; k < 6; ++k) { J0[k] *= sic; J1[k] *= sic; }
      // TukeyWeightFunction::value(float) robust_cost.cpp
      const float xw = (float)(sqrt(e0 * e0 + e1 * e1) / scale);
      const float x_square = xw * xw;
      float wf = 0.0f;
      if (x_square <= b_square) { const float tmp = 1.0f - x_square / b_square; wf = tmp * tmp; }
      const double w = (double)wf;
      int q = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) acc[q++] += (J0[r] * J0[c] + J1[r] * J1[c]) * w;
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[21 + r] -= (J0[r] * e0 + J1[r] * e1) * w;
      acc[27] += (e0 * e0 + e1 * e1) * w;
    }
    // fixed-tree reduction: lanes by xor shuffles, then the warps in order
#pragma unroll
    for (int k = 0; k < POSE_ACC; ++k) {
      double v = acc[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) s_red[warp][k] = v;
    }
    __syncthreads();
    if (tid == 0) {
      double sum[POSE_ACC];
      for (int k = 0; k < POSE_ACC; ++k) { double v = s_red[0][k]; for (int w = 1; w < POSE_T / 32; ++w) v += s_red[w][k]; sum[k] = v; }
      int q = 0;
      for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { A[r * 6 + c] = sum[q]; A[c * 6 + r] = sum[q]; ++q; }
      double bv[6], dT[6];
      for (int r = 0; r < 6; ++r) bv[r] = sum[21 + r];
      const double new_chi2 = sum[27];
      ldlt_solve_fixed<6, true>(A, bv, dT);     // sums are tree-reduced (tolerance-matched): shared-reciprocal quotients
      ++iters;
      int flag = 0;
      if ((iter > 0 && new_chi2 > chi2 * 1.2) || isnan(dT[0])) {
        for (int k = 0; k < 7; ++k) T[k] = T_old[k];      // roll-back
        rolled_back = 1; flag = 1;
      } else {
        double E[7], T_new[7];
        se3_exp(dT, E);
        se3_mul(E, T, T_new);
        for (int k = 0; k < 7; ++k) { T_old[k] = T[k]; T[k] = T_new[k]; }
        chi2 = new_chi2;
        double nm = -1;
        for (int k = 0; k < 6; ++k) { const double a = fabs(dT[k]); if (a > nm) nm = a; }
        if (nm <= eps) flag = 1;
      }
      for (int k = 0; k < 7; ++k) s_T[k] = T[k];
      s_flag = flag;
    }
    __syncthreads();
    for (int k = 0; k < 7; ++k) T[k] = s_T[k];
    const int stop = s_flag;
    __syncthreads();
    if (stop) break;
  }
  // outliers and the final error (:142-165)
  const double thr = reproj_thresh / em2;
  int deleted = 0;
  for (int i = tid; i < n; i += POSE_T) {
    v3d p; double e0, e1, sic;
    pose_residual(T, F + 3 * i, P + 3 * i, LV[i], p, e0, e1, sic);
    const double c = e0 * e0 + e1 * e1;
    work[i] = c;
    const bool out = sqrt(c) > thr;
    outlier_all[i0 + i] = out ? 1 : 0;
    deleted += out;
  }
  deleted = warp_sum_i(deleted);
  if (tid == 0) s_flag = 0;
  __syncthreads();
  if (lane == 0) atomicAdd(&s_flag, deleted);
  __syncthreads();
  const double med_final = block_median(work, n, &s_med);
  if (tid == 0) {
    for (int k = 0; k < 7; ++k) T_io[7 * (size_t)b + k] = T[k];
    for (int k = 0; k < 36; ++k) R->A[k] = A[k];
    R->chi2 = chi2; R->estimated_scale = estimated_scale * em2;
    R->error_init = sqrt(med_init) * em2; R->error_final = sqrt(med_final) * em2;
    R->iters = iters; R->num_obs = n - s_flag; R->rolled_back = rolled_back;
  }
}

// ---------------------------------------------------------------- Point::optimize (point.cpp:130-192): thread per point
__global__ void __launch_bounds__(128) points_optimize_kernel(int n, const int* obs_off, const double* T_f_w, const double* f_all, int n_iter,
                                                              double eps, double* pos_io, int* iters_out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int o0 = obs_off[i], o1 = obs_off[i + 1];
  double pos[3] = {pos_io[3 * (size_t)i], pos_io[3 * (size_t)i + 1], pos_io[3 * (size_t)i + 2]};
  double old_point[3] = {pos[0], pos[1], pos[2]};
  double chi2 = 0.0;
  int it = 0;
  for (int iter = 0; iter < n_iter; ++iter) {
    double A[9], bv[3] = {0, 0, 0}, new_chi2 = 0.0;
#pragma unroll
    for (int k = 0; k < 9; ++k) A[k] = 0.0;
    for (int k = o0; k < o1; ++k) {
      const double* T = T_f_w + 7 * (size_t)k;
      const double* f = f_all + 3 * (size_t)k;
      const v3d p = se3_transform(T, {pos[0], pos[1], pos[2]});
      double Rm[9];
      q_matrix(T + 3, Rm);
      // Point::jacobian_xyz2uv (point.h): point_jac = -point_jac * R_f_w, sequential three-term sums
      const double z_inv = 1.0 / p.z, z_inv_sq = z_inv * z_inv;
      const double a0[3] = {z_inv, 0.0, -p.x * z_inv_sq}, a1[3] = {0.0, z_inv, -p.y * z_inv_sq};
      double J0[3], J1[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        J0[c] = ((-a0[0]) * Rm[c] + (-a0[1]) * Rm[3 + c]) + (-a0[2]) * Rm[6 + c];
        J1[c] = ((-a1[0]) * Rm[c] + (-a1[1]) * Rm[3 + c]) + (-a1[2]) * Rm[6 + c];
      }
      const double e0 = f[0] / f[2] - p.x / p.z, e1 = f[1] / f[2] - p.y / p.z;
      new_chi2 += e0 * e0 + e1 * e1;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) A[r * 3 + c] += J0[r] * J0[c] + J1[r] * J1[c];
        bv[r] -= J0[r] * e0 + J1[r] * e1;
      }
    }
    double dp[3];
    ldlt_solve_fixed<3>(A, bv, dp);
    ++it;
    if ((iter > 0 && new_chi2 > chi2) || isnan(dp[0])) { pos[0] = old_point[0]; pos[1] = old_point[1]; pos[2] = old_point[2]; break; }
#pragma unroll
    for (int k = 0; k < 3; ++k) { old_point[k] = pos[k]; pos[k] = pos[k] + dp[k]; }
    chi2 = new_chi2;
    double nm = -1;
#pragma unroll
    for (int k = 0; k < 3; ++k) { const double a = fabs(dp[k]); if (a > nm) nm = a; }
    if (nm <= eps) break;
  }
  pos_io[3 * (size_t)i] = pos[0]; pos_io[3 * (size_t)i + 1] = pos[1]; pos_io[3 * (size_t)i + 2] = pos[2];
  if (iters_out) iters_out[i] = it;
}

// ---------------------------------------------------------------- DepthFilter::initializeSeeds (depth_filter.cpp:129-151)
// AbstractDetector::setExistingFeatures (feature_detection.cpp:40-48): cell of every existing feature -> occupied
__global__ void __launch_bounds__(128) occupancy_kernel(int batch, const int* off, const double* px, int cell_size, int grid_cols, int n_cells,
                                                        uint8_t* occ)
{
  const int b = blockIdx.y;
  if (b >= batch) return;
  for (int i = off[b] + blockIdx.x * blockDim.x + threadIdx.x; i < off[b + 1]; i += gridDim.x * blockDim.x) {
    const int k = x86_d2i(px[2 * (size_t)i + 1] / cell_size) * grid_cols + x86_d2i(px[2 * (size_t)i] / cell_size);
    if (k >= 0 && k < n_cells) occ[(size_t)b * n_cells + k] = 1;     // grid_occupancy_.at(k) would throw outside
  }
}

// new corners in cell order (feature_detection.cpp:116-119) + one Seed each (depth_filter.cpp:36-45): one CTA per image
__global__ void __launch_bounds__(256) seeds_compact_kernel(const svob200_corner* cells, int n_cells, double thr, const float* depth_mean,
                                                            const float* depth_min, svob200_corner* corners_out, svob200_seed* seeds_out,
                                                            int* counts)
{
  const int b = blockIdx.x, tid = threadIdx.x;
  const svob200_corner* C = cells + (size_t)b * n_cells;
  const int chunk = (n_cells + 255) / 256;
  const int c0 = min(tid * chunk, n_cells), c1 = min(c0 + chunk, n_cells);
  int local = 0;
  for (int c = c0; c < c1; ++c) local += (double)C[c].score > thr;
  int total;
  int run = block_exclusive_scan<256>(local, &total);
  const svob200_seed sd = seed_prior(depth_mean[b], depth_min[b]);
  for (int c = c0; c < c1; ++c) {
    if (!((double)C[c].score > thr)) continue;
    corners_out[(size_t)b * n_cells + run] = C[c];
    seeds_out[(size_t)b * n_cells + run] = sd;
    ++run;
  }
  if (tid == 0) counts[b] = total;
}

inline size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

int launch_occupancy(int batch, int max_per_image, const int* d_off, const double* d_px, int cell_size, int grid_cols, int n_cells, uint8_t* d_occ,
                     cudaStream_t s, long long* launches)
{
  if (batch <= 0) return 0;
  int bx = (max_per_image + 127) / 128;
  if (bx < 1) bx = 1;
  if (bx > 64) bx = 64;
  occupancy_kernel<<<dim3(bx, batch), 128, 0, s>>>(batch, d_off, d_px, cell_size, grid_cols, n_cells, d_occ);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_seeds_compact(int batch, const svob200_corner* d_cells, int n_cells, double thr, const float* d_depth_mean, const float* d_depth_min,
                         svob200_corner* d_corners_out, svob200_seed* d_seeds_out, int* d_counts, cudaStream_t s, long long* launches)
{
  if (batch <= 0) return 0;
  seeds_compact_kernel<<<batch, 256, 0, s>>>(d_cells, n_cells, thr, d_depth_mean, d_depth_min, d_corners_out, d_seeds_out, d_counts);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------- launchers
size_t reproject_scratch_bytes(int n_points)
{
  const size_t m = (size_t)(n_points > 0 ? n_points : 1);
  return up256(m * sizeof(svob200_feature_ref)) + up256(m * sizeof(double)) + 2 * up256(m * 2 * sizeof(double)) + up256(m) + 2 * up256(m * sizeof(int))
         + up256(m * 4 * sizeof(double)) + 256;
}

int launch_reproject_map(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int batch, const double* d_T_cur_w, const int* d_pt_off,
                         int n_points, const svob200_map_point* d_points, const svob200_feature_ref* d_obs, const double* d_T_obs_w,
                         int cell_size, int max_fts, svob200_matcher_opts opts, svob200_reproj_result* d_results, int* d_cell_winner,
                         svob200_reproj_stats* d_stats, void* d_scratch, void* d_match_scratch,
                         double* d_m_f, int* d_m_level, double* d_m_pos, int* d_m_point, int* d_m_count,
                         cudaStream_t s, long long* launches, int image_base, int point_base, int n_range)
{
  // d_T_cur_w, d_pt_off, d_cell_winner, d_stats, d_m_* already point at image `image_base` (offsets in d_pt_off stay
  // ABSOLUTE indices into d_points / d_results); this call covers the points [point_base, point_base + n_range)
  if (n_range < 0) n_range = n_points - point_base;
  if (batch <= 0) return 0;
  const int cols = (cam.width + cell_size - 1) / cell_size, rows = (cam.height + cell_size - 1) / cell_size;
  const int n_cells = cols * rows;
  if (n_cells > REPROJ_MAX_CELLS) return -2;
  const size_t m = (size_t)(n_points > 0 ? n_points : 1);
  char* p = static_cast<char*>(d_scratch);
  svob200_feature_ref* ftr = reinterpret_cast<svob200_feature_ref*>(p); p += up256(m * sizeof(svob200_feature_ref));
  double* depth = reinterpret_cast<double*>(p); p += up256(m * sizeof(double));
  double* px_in = reinterpret_cast<double*>(p); p += up256(m * 2 * sizeof(double));
  double* px_out = reinterpret_cast<double*>(p); p += up256(m * 2 * sizeof(double));
  uint8_t* active = reinterpret_cast<uint8_t*>(p); p += up256(m);
  int* ok = reinterpret_cast<int*>(p); p += up256(m * sizeof(int));
  int* level = reinterpret_cast<int*>(p); p += up256(m * sizeof(int));
  double* A = reinterpret_cast<double*>(p);
  reproj_select_kernel<<<batch, 128, 0, s>>>(cam, d_T_cur_w, d_pt_off, d_points, d_obs, d_T_obs_w, cell_size, cols, image_base, ftr, depth, px_in, active, d_results);
  ++*launches;
  if (n_range > 0) {
    const size_t o = (size_t)point_base;
    if (launch_match_direct(d_frames, cur_slot, cam, n_range, ftr + o, depth + o, px_in + 2 * o, opts, nullptr, px_out + 2 * o, ok + o, d_match_scratch,
                            n_points, point_base, s, launches, nullptr, active + o, level + o, A + 4 * o))
      return -1;
  }
  reproj_cells_kernel<<<batch, REPROJ_T, 0, s>>>(cam, d_pt_off, d_points, active, ok, px_out, level, A, n_cells, max_fts, d_results, d_cell_winner, d_stats,
                                                 d_m_f, d_m_level, d_m_pos, d_m_point, d_m_count);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_pose_optimize(const DevCam& cam, int batch, const int* d_seg_begin, const int* d_seg_end, const double* d_f, const int* d_level,
                         const double* d_pos, double reproj_thresh, int n_iter, double eps, float tukey_b, double* d_T_io,
                         svob200_pose_opt_result* d_results, uint8_t* d_outlier, double* d_work, cudaStream_t s, long long* launches)
{
  if (batch <= 0) return 0;
  pose_optimize_kernel<<<batch, POSE_T, 0, s>>>(cam, d_seg_begin, d_seg_end, d_f, d_level, d_pos, reproj_thresh, n_iter, eps, tukey_b, d_T_io,
                                               d_results, d_outlier, d_work);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_points_optimize(int n, const int* d_obs_off, const double* d_T_f_w, const double* d_f, int n_iter, double eps, double* d_pos_io,
                           int* d_iters, cudaStream_t s, long long* launches)
{
  if (n <= 0) return 0;
  points_optimize_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, d_obs_off, d_T_f_w, d_f, n_iter, eps, d_pos_io, d_iters);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
