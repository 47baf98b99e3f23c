// tracker.cu — the per-frame front-end step as ONE C-ABI call over a batch of independent
// sequences: pyramid -> sparse image alignment (last -> cur) -> reprojection refinement of the map
// points against their keyframe patches -> depth-filter update of the keyframe's seeds.
//
// It chains the operators exactly the way FrameHandlerMono::processFrame + DepthFilter do
// (frame_handler_mono.cpp:171-262, depth_filter.cpp:237-341), minus the host-only stages that are
// out of scope (pose_optimizer, map management): everything between the operators that the
// reference does in host code is done by the glue kernels, so a step is 14 launches with no host round trip.  It runs in one
// of three shapes (RangeShape): graph + fork (up to GRAPH_MAX_BATCH sequences, no profiling: a CUDA graph replay whose
// independent stages run on forked branches); asynchronous depth filter (device memory, more sequences, not chain mode: the
// depth filter on df_stream, the step records in two halves, 15 launches); in place (everything else: host-memory chunks of
// CHUNK sequences, profiling, chain mode).  In SVOB200_MEM_HOST mode the step is bracketed by one H2D of the frame(s), one
// H2D of the small per-step inputs and one D2H of the per-sequence results.  With a point pool (svob200_tracker_set_point_pool)
// the step-record kernel also turns converged seeds into candidate points, and one more launch at the head of the step inserts
// the candidates of two steps ago (cand_insert_kernel): the same in every shape.
#include <atomic>
#include "ctx_internal.h"

namespace {

__global__ void init_pose_kernel(int batch, const double* T_last, double* T_init)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  // SparseImgAlign::run: SE3 T_cur_from_ref(cur->T_f_w_ * ref->T_f_w_.inverse()) with cur->T_f_w_ = last->T_f_w_
  double inv[7], out[7];
  se3_inverse(T_last + 7 * (size_t)b, inv);
  se3_mul(T_last + 7 * (size_t)b, inv, out);
  for (int k = 0; k < 7; ++k) T_init[7 * (size_t)b + k] = out[k];
}

// ---- point pool (svob200_tracker_set_point_pool): a converged seed becomes a candidate point (DepthFilter::updateSeeds ->
// seed_converged_cb_ -> MapPointCandidates::newCandidatePoint), which enters an empty point slot two steps later
struct CandRec { double pos[3], px[2], f[3]; int level, kf, batch_id, pad; };   // one candidate, with its one observation
struct CandStage {                       // where step_stats_kernel records the candidates of the step (rec == nullptr: no pool)
  CandRec* rec; int* count; int* created;  // rec: the sequence's point-slot block of this parity's staging; count / created: per sequence
  const int* pt_off; const double* T_kf; int batch, b0;   // point-slot offsets, keyframe poses [kf][batch][7], first sequence of the range
};
struct KfBatches { int v[16]; };         // Seed::batch_id of every keyframe index of the ring (svob200_tracker::kf_batch)

// Order-preserving fill of one sequence's empty slots by one CTA of NT threads: the r-th selected item (is_item, in index
// order) goes to the r-th free slot (is_free, in slot order), put(item, slot) for r < min(#items, #free).  Every thread owns
// a contiguous chunk of the items and one of the slots, so placement never depends on scheduling.  slot_of_rank holds
// min(#items, #free) entries.  Returns that count; *n_sel = #items.
template <int NT, class IsItem, class IsFree, class Put>
__device__ int fill_free_slots(int n_items, IsItem is_item, int n_slots, IsFree is_free, int* slot_of_rank, int* n_sel, Put put)
{
  const int tid = threadIdx.x;
  const int ic = (n_items + NT - 1) / NT, i0 = min(tid * ic, n_items), i1 = min(i0 + ic, n_items);
  const int sc = (n_slots + NT - 1) / NT, q0 = min(tid * sc, n_slots), q1 = min(q0 + sc, n_slots);
  int ni = 0, nf = 0;
  for (int i = i0; i < i1; ++i) ni += is_item(i);
  for (int q = q0; q < q1; ++q) nf += is_free(q);
  int f_total;
  const int i_rank = block_exclusive_scan<NT>(ni, n_sel), f_rank = block_exclusive_scan<NT>(nf, &f_total);
  const int n_fill = min(*n_sel, f_total);
  { int r = f_rank; for (int q = q0; q < q1 && r < n_fill; ++q) if (is_free(q)) slot_of_rank[r++] = q; }
  __syncthreads();
  int r = i_rank;
  for (int i = i0; i < i1 && r < n_fill; ++i) if (is_item(i)) put(i, slot_of_rank[r++]);
  return n_fill;
}

// The candidates of sequence b in the reference's list order (seeds_ is ordered by ascending Seed::batch_id, and inside one
// batch by slot, since kf_append_seeds_kernel fills slots in cell order): one pass per batch id, each a block scan over
// contiguous slot chunks, so placement never depends on scheduling.  xyz_world = kf.T_f_w.inverse() * (f * (1.0 / mu))
// (depth_filter.cpp:318-325 -> MapPointCandidates::newCandidatePoint); runs before the seed is re-initialised.
__device__ void create_candidates(const CandStage& cs, int b, int p0, int np, const svob200_seed_obs* obs, const svob200_seed* seeds,
                                  const SeedRef* refs)
{
  __shared__ int s_min;
  const int tid = threadIdx.x, ab = cs.b0 + b;
  const int chunk = (np + 127) / 128, q0 = min(tid * chunk, np), q1 = min(q0 + chunk, np);
  const int cap = cs.pt_off[ab + 1] - cs.pt_off[ab];
  CandRec* out = cs.rec + cs.pt_off[ab];
  int n_out = 0, prev = -1;
  for (;;) {
    if (tid == 0) s_min = 0x7fffffff;
    __syncthreads();
    int m = 0x7fffffff;
    for (int q = q0; q < q1; ++q)
      if (obs[p0 + q].status == SVOB200_SEED_CONVERGED && (int)refs[p0 + q].batch_id > prev) m = min(m, (int)refs[p0 + q].batch_id);
    if (m != 0x7fffffff) atomicMin(&s_min, m);
    __syncthreads();
    const int bid = s_min;
    if (bid == 0x7fffffff) break;
    int local = 0;
    for (int q = q0; q < q1; ++q) local += obs[p0 + q].status == SVOB200_SEED_CONVERGED && refs[p0 + q].batch_id == bid;
    int total;
    int r = n_out + block_exclusive_scan<128>(local, &total);
    for (int q = q0; q < q1; ++q) {
      if (obs[p0 + q].status != SVOB200_SEED_CONVERGED || refs[p0 + q].batch_id != bid) continue;
      if (r < cap) {
        const SeedRef sr = refs[p0 + q];
        double inv[7];
        se3_inverse(cs.T_kf + 7 * ((size_t)sr.kf * cs.batch + ab), inv);
        const double s = 1.0 / (double)seeds[p0 + q].mu;
        const v3d p = se3_transform(inv, {sr.f[0] * s, sr.f[1] * s, sr.f[2] * s});
        CandRec c;
        c.pos[0] = p.x; c.pos[1] = p.y; c.pos[2] = p.z; c.px[0] = sr.px[0]; c.px[1] = sr.px[1];
        c.f[0] = sr.f[0]; c.f[1] = sr.f[1]; c.f[2] = sr.f[2]; c.level = sr.level; c.kf = sr.kf; c.batch_id = sr.batch_id; c.pad = 0;
        out[r] = c;
      }
      ++r;
    }
    n_out += total; prev = bid;
  }
  if (tid == 0) { cs.count[ab] = n_out; cs.created[ab] += n_out; }
}

// one CTA per sequence: per-sequence statistics + steady-state re-seeding of finished seeds
// parts: 1 = the tracking fields (pose, alignment, matches), 2 = the depth-filter fields (+ re-seeding); 3 = both.  The
// asynchronous depth filter runs part 2 on its own stream, after the tracking chain of the same step ran part 1.  kPool: the
// tracker has a point pool, and part 2 first records the step's candidates (the instance without it keeps the lean kernel).
template <bool kPool>
__global__ void __launch_bounds__(128) step_stats_kernel(const int* ftr_off, const int* seed_off, const svob200_align_result* align,
                                                         const double* T_cur_w, const int* match_ok, const svob200_seed_obs* obs,
                                                         svob200_seed* seeds, svob200_seed init, int reseed, svob200_step_stats* stats, int parts,
                                                         SeedRef* refs, CandStage cand)
{
  const int b = blockIdx.x, tid = threadIdx.x;
  if (kPool && (parts & 2)) create_candidates(cand, b, seed_off[b], seed_off[b + 1] - seed_off[b], obs, seeds, refs);
  int matched = 0, upd = 0, conv = 0, fail = 0, skipped = 0;
  if (parts & 1) for (int i = ftr_off[b] + tid; i < ftr_off[b + 1]; i += 128) matched += match_ok[i] ? 1 : 0;
  if (parts & 2) for (int i = seed_off[b] + tid; i < seed_off[b + 1]; i += 128) {
    const int st = obs[i].status;
    if (st == 0 || st == SVOB200_SEED_TOO_OLD) continue;            // empty slot / erased by the ageing rule
    if (st == SVOB200_SEED_UPDATED) ++upd;
    else if (st == SVOB200_SEED_CONVERGED) ++conv;
    else if (st == SVOB200_SEED_NO_MATCH) ++fail;
    else ++skipped;
    // reseed 1: finished seeds start afresh (stationary workload); 2: EVERY seed starts afresh every frame (young-seed regime)
    // 3: the reference's list semantics — a converged seed (callback, depth_filter.cpp:314-331) or a NaN one (:334-338) is erased
    if (reseed == 3) { if (st == SVOB200_SEED_CONVERGED || st == SVOB200_SEED_NAN_ERASED) refs[i].state = 1; }
    else if (reseed == 2 || (reseed && (st == SVOB200_SEED_CONVERGED || st == SVOB200_SEED_NAN_ERASED))) seeds[i] = init;
  }
  __shared__ int s[5];
  if (tid < 5) s[tid] = 0;
  __syncthreads();
  matched = warp_sum_i(matched); upd = warp_sum_i(upd); conv = warp_sum_i(conv); fail = warp_sum_i(fail); skipped = warp_sum_i(skipped);
  if ((tid & 31) == 0) { atomicAdd(&s[0], matched); atomicAdd(&s[1], upd); atomicAdd(&s[2], conv); atomicAdd(&s[3], fail); atomicAdd(&s[4], skipped); }
  __syncthreads();
  if (tid == 0) {
    svob200_step_stats* o = &stats[b];
    if (parts & 1) {
      for (int k = 0; k < 7; ++k) o->T_cur_w[k] = T_cur_w[7 * (size_t)b + k];
      o->chi2 = align[b].chi2;
      o->n_tracked = align[b].n_meas / 16;
      o->n_matched = s[0];
      int it = 0;
      for (int l = 0; l < SVOB200_MAX_LEVELS; ++l) it += align[b].iters[l];
      o->align_iters = it;
      o->n_exact_chi2 = align[b].n_exact_chi2;
      o->n_reproj_trials = 0; o->n_pose_obs = 0;
    }
    if (parts & 2) { o->n_seeds_updated = s[1]; o->n_seeds_converged = s[2]; o->n_seeds_failed = s[3]; o->n_seeds_skipped = s[4]; }
  }
}

// chain mode: segment of image b in the compacted match arrays = [b * n_cells, b * n_cells + count[b])
__global__ void chain_segments_kernel(int batch, int n_cells, const int* count, int* seg_begin, int* seg_end)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  seg_begin[b] = b * n_cells;
  seg_end[b] = b * n_cells + count[b];
}

// chain mode: per-point outputs of the step in the tracker's plain arrays
__global__ void chain_export_kernel(int n, const svob200_reproj_result* res, double* px_out, int* match_ok)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const svob200_reproj_result r = res[i];
  match_ok[i] = r.status == SVOB200_REPROJ_MATCHED ? 1 : 0;
  px_out[2 * (size_t)i] = r.px[0]; px_out[2 * (size_t)i + 1] = r.px[1];
}

__global__ void chain_stats_kernel(int batch, const svob200_reproj_stats* rs, const svob200_pose_opt_result* pr, int pose_opt, svob200_step_stats* stats)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  stats[b].n_reproj_trials = rs[b].n_trials;
  stats[b].n_pose_obs = pose_opt ? pr[b].num_obs : rs[b].n_matches;
}

// ---- keyframe insertion (svob200_tracker_add_keyframe)
// occupancy of the frame's existing features = the map points matched in it (AbstractDetector::setExistingFeatures,
// feature_detection.cpp:40-58: cell of (px.y / cell, px.x / cell) with the x86 double -> int conversion)
__global__ void kf_occupancy_kernel(int n, const int* ftr_image, const double* px, const int* match_ok, int cell, int grid_cols, int n_cells, uint8_t* occ)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !match_ok[i]) return;
  const long long k = (long long)x86_d2i(px[2 * (size_t)i + 1] / cell) * grid_cols + x86_d2i(px[2 * (size_t)i] / cell);
  if (k >= 0 && k < n_cells) occ[(size_t)ftr_image[i] * n_cells + k] = 1;
}

// ---- map points with one observation per keyframe they were matched in (Point::obs_, point.h; Point::addFrameRef pushes to the front)
// point i owns the K slots [i*K, (i+1)*K) of obs / T_obs; its list, newest first, is [obs_begin, obs_end) = the top end of that block.
__device__ __forceinline__ v3d kf_frame_pos(const double* T)
{
  double inv[7];
  se3_inverse(T, inv);
  return {inv[0], inv[1], inv[2]};
}

// svob200_tracker_set_keyframe, one CTA per sequence: every point slot and seed slot of sequence b.  Point slot j holds map
// point i = ftr_off[b] + (j - pt_off[b]) while i < ftr_off[b + 1], with ONE observation, in keyframe 0 (kf_slot, pose T_kf[b]):
// the last slot of its block of K.  The slots after it are the empty slots of the point pool (has_point 0: TYPE_DELETED with
// no observation).  Seed slots likewise (an empty one has state 1).  Every record, empty or not, gets the Feature ctor's
// f = cam2world(px) (feature.h:43-51).
__global__ void __launch_bounds__(128) kf_init_slots_kernel(DevCam cam, int K, int kf_slot, const double* T_kf, const int* pt_off, const int* ftr_off,
                                                            const double* kf_px, const int* kf_level, const double* pt_world_in, const int* pool_off,
                                                            const int* seed_off, const double* seed_px, const int* seed_level, svob200_seed init,
                                                            int* image, uint8_t* has_point, int* sel, double* pt_world, svob200_feature_ref* ftrs,
                                                            svob200_map_point* pts, svob200_feature_ref* obs, double* T_obs, SeedRef* refs,
                                                            svob200_seed* seeds)
{
  const int b = blockIdx.x;
  for (int j = pt_off[b] + threadIdx.x; j < pt_off[b + 1]; j += blockDim.x) {
    const int i = ftr_off[b] + (j - pt_off[b]), o = j * K + K - 1;
    const bool real = i < ftr_off[b + 1];
    svob200_feature_ref f;
    f.ref_frame_id = real ? kf_slot : 0; f.ref_image = b; f.cur_image = b; f.level = real ? kf_level[i] : 0; f.type = 0;
    f.px[0] = real ? kf_px[2 * (size_t)i] : 0.0; f.px[1] = real ? kf_px[2 * (size_t)i + 1] : 0.0;
    const v3d fv = cam2world(cam, f.px[0], f.px[1]);
    f.f[0] = fv.x; f.f[1] = fv.y; f.f[2] = fv.z; f.grad[0] = real ? 1.0 : 0.0; f.grad[1] = 0.0;
    for (int k = 0; k < 7; ++k) { f.T_cur_ref[k] = 0.0; T_obs[7 * (size_t)o + k] = real ? T_kf[7 * (size_t)b + k] : 0.0; }
    ftrs[j] = f; obs[o] = f;
    svob200_map_point p;
    for (int k = 0; k < 3; ++k) { p.pos[k] = real ? pt_world_in[3 * (size_t)i + k] : 0.0; pt_world[3 * (size_t)j + k] = p.pos[k]; }
    p.type = real ? SVOB200_POINT_UNKNOWN : SVOB200_POINT_DELETED; p.obs_end = (j + 1) * K; p.obs_begin = real ? o : p.obs_end; p.reserved = 0;
    pts[j] = p;
    image[j] = b; has_point[j] = real; sel[j] = -1;
  }
  for (int q = pool_off[b] + threadIdx.x; q < pool_off[b + 1]; q += blockDim.x) {
    const int i = seed_off[b] + (q - pool_off[b]);
    const bool real = i < seed_off[b + 1];
    SeedRef r;
    r.px[0] = real ? seed_px[2 * (size_t)i] : 0.0; r.px[1] = real ? seed_px[2 * (size_t)i + 1] : 0.0;
    const v3d fv = cam2world(cam, r.px[0], r.px[1]);
    r.f[0] = fv.x; r.f[1] = fv.y; r.f[2] = fv.z;
    r.image = b; r.level = real ? (uint8_t)seed_level[i] : 0; r.kf = 0; r.batch_id = 0; r.state = real ? 0 : 1;
    r.pad0 = 0; r.pad1 = 0; r.pad2[0] = r.pad2[1] = r.pad2[2] = 0;
    refs[q] = r;
    seeds[q] = init;
  }
}

// The candidates of step k enter at the head of step k + 2 (the reference's depth filter runs one frame behind tracking):
// into the sequence's empty slots in slot order, in their list order.  A candidate whose keyframe left the ring since (its
// batch id is no longer that keyframe index's) or that finds no empty slot is dropped.  One CTA per sequence.
__global__ void __launch_bounds__(128) cand_insert_kernel(int K, int batch, const int* pt_off, const CandRec* cand, const int* cand_n, KfBatches kfb,
                                                          const int* kf_slot, const double* T_kf, svob200_map_point* pts, double* pt_world,
                                                          svob200_feature_ref* obs, double* T_obs, int* sel, uint8_t* has_point,
                                                          int* slot_of_rank, int* dropped)
{
  const int b = blockIdx.x, tid = threadIdx.x;
  const int P0 = pt_off[b], P = pt_off[b + 1] - P0, n = cand_n[b];
  const CandRec* C = cand + P0;
  auto valid = [&](int c) { return C[c].batch_id == kfb.v[C[c].kf]; };
  auto empty = [&](int q) { return pts[P0 + q].type == SVOB200_POINT_DELETED; };
  auto put = [&](int c, int q) {
    const CandRec cr = C[c];
    const int j = P0 + q, o = j * K + K - 1;
    svob200_feature_ref f;
    f.ref_frame_id = kf_slot[cr.kf]; f.ref_image = b; f.cur_image = b; f.level = cr.level; f.type = 0;
    f.px[0] = cr.px[0]; f.px[1] = cr.px[1]; f.f[0] = cr.f[0]; f.f[1] = cr.f[1]; f.f[2] = cr.f[2]; f.grad[0] = 1.0; f.grad[1] = 0.0;
    for (int k = 0; k < 7; ++k) { f.T_cur_ref[k] = 0.0; T_obs[7 * (size_t)o + k] = T_kf[7 * ((size_t)cr.kf * batch + b) + k]; }
    obs[o] = f;
    svob200_map_point p;
    for (int k = 0; k < 3; ++k) { p.pos[k] = cr.pos[k]; pt_world[3 * (size_t)j + k] = cr.pos[k]; }
    p.type = SVOB200_POINT_CANDIDATE; p.obs_begin = o; p.obs_end = (j + 1) * K; p.reserved = 0;
    pts[j] = p;
    sel[j] = -1; has_point[j] = 1;
  };
  int n_valid;
  const int n_fill = fill_free_slots<128>(min(n, P), valid, P, empty, slot_of_rank + P0, &n_valid, put);
  if (tid == 0) dropped[b] += n - n_fill;
}

// MapPointCandidates::removeFrameCandidates: the candidates of the keyframe that leaves the ring are deleted, except those
// matched in the new keyframe (the reference promotes them first: addCandidatePointToFrame runs before the ring drops a keyframe)
__global__ void kf_drop_candidates_kernel(int n, svob200_map_point* pts, const svob200_feature_ref* obs, const int* match_ok, uint8_t* has_point, int kf_slot)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const svob200_map_point p = pts[i];
  if (p.type != SVOB200_POINT_CANDIDATE || match_ok[i] || (int)obs[p.obs_begin].ref_frame_id != kf_slot) return;
  pts[i].type = SVOB200_POINT_DELETED; pts[i].obs_begin = p.obs_end;
  has_point[i] = 0;
}

// The head of Matcher::findMatchDirect for every map point (matcher.cpp:156-173): Point::getCloseViewObs (point.cpp:101-125: arg-max of
// the cosine over obs_ in list order, strict >, starting from 0; fails below 0.5), then px = cur.w2c(pos) (reprojector.cpp:131-145),
// depth_ref = |ref.pos() - pos| and T_cur_ref = cur.T_f_w * ref.T_f_w^-1.  The chosen observation becomes this step's ftrs[i].
__global__ void __launch_bounds__(128) points_select_kernel(DevCam cam, int n, const svob200_map_point* pts, const svob200_feature_ref* obs,
                                                            const double* T_obs, const int* image, const double* T_cur_w, svob200_feature_ref* ftrs,
                                                            double* depth_ref, double* px_in, uint8_t* active, int* sel)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const svob200_map_point p = pts[i];
  const int b = image[i];
  const double* T = T_cur_w + 7 * (size_t)b;
  const v3d pos = {p.pos[0], p.pos[1], p.pos[2]};
  double u, v;
  world2cam(cam, se3_transform(T, pos), u, v);
  px_in[2 * (size_t)i] = u; px_in[2 * (size_t)i + 1] = v;
  uint8_t act = 0;
  double dref = 0.0;
  if (p.obs_end > p.obs_begin) {
    const v3d cur_pos = kf_frame_pos(T);
    const v3d od = normalized3({cur_pos.x - pos.x, cur_pos.y - pos.y, cur_pos.z - pos.z});
    int best = p.obs_begin;
    double min_cos = 0.0;
    v3d best_pos = kf_frame_pos(T_obs + 7 * (size_t)p.obs_begin);
    for (int k = p.obs_begin; k < p.obs_end; ++k) {
      const v3d op = kf_frame_pos(T_obs + 7 * (size_t)k);
      const v3d d = normalized3({op.x - pos.x, op.y - pos.y, op.z - pos.z});
      const double c = dot3(od, d);
      if (c > min_cos) { min_cos = c; best = k; best_pos = op; }
    }
    if (!(min_cos < 0.5)) {
      act = 1;
      // the 144-byte record is copied only when the choice changes (after a keyframe insertion); every step writes the 56 bytes
      // that depend on the current pose
      if (sel[i] != best) { svob200_feature_ref f = obs[best]; f.cur_image = b; ftrs[i] = f; sel[i] = best; }
      double inv[7], Tcr[7];
      se3_inverse(T_obs + 7 * (size_t)best, inv);
      se3_mul(T, inv, Tcr);
      for (int k = 0; k < 7; ++k) ftrs[i].T_cur_ref[k] = Tcr[k];
      dref = norm3({best_pos.x - pos.x, best_pos.y - pos.y, best_pos.z - pos.z});
    }
  }
  active[i] = act;
  depth_ref[i] = dref;
}

// frame_handler_mono.cpp:277-279: every feature of the new keyframe with a point adds a frame reference to it (push_front).
// The keyframe's features are the map points matched in it: Feature(frame, px_refined, search_level) (reprojector.cpp:219-231).
__global__ void kf_add_obs_kernel(DevCam cam, int n, int K, svob200_map_point* pts, svob200_feature_ref* obs, double* T_obs, const int* image,
                                  const int* match_ok, const double* px, const int* level, int kf_slot, const double* T_cur_w)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !match_ok[i]) return;
  svob200_map_point p = pts[i];
  if (p.obs_end - p.obs_begin >= K) return;                      // (cannot happen: at most one observation per resident keyframe)
  const int slot = p.obs_begin - 1;
  svob200_feature_ref f;
  f.ref_frame_id = kf_slot; f.ref_image = image[i]; f.cur_image = image[i]; f.level = level[i]; f.type = 0;
  f.px[0] = px[2 * (size_t)i]; f.px[1] = px[2 * (size_t)i + 1];
  const v3d fv = cam2world(cam, f.px[0], f.px[1]);
  f.f[0] = fv.x; f.f[1] = fv.y; f.f[2] = fv.z; f.grad[0] = 1.0; f.grad[1] = 0.0;
  for (int k = 0; k < 7; ++k) { f.T_cur_ref[k] = 0.0; T_obs[7 * (size_t)slot + k] = T_cur_w[7 * (size_t)image[i] + k]; }
  obs[slot] = f;
  pts[i].obs_begin = slot;
  if (p.type == SVOB200_POINT_CANDIDATE) pts[i].type = SVOB200_POINT_UNKNOWN;   // MapPointCandidates::addCandidatePointToFrame
}

// Map::safeDeleteFrame -> Point::deleteFrameRef for every point seen in the keyframe that leaves the ring
__global__ void kf_drop_obs_kernel(int n, int K, svob200_map_point* pts, svob200_feature_ref* obs, double* T_obs, int kf_slot, int* sel)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  sel[i] = -1;                                                   // slots move: the next step copies its choice afresh
  const svob200_map_point p = pts[i];
  int w = p.obs_end;                                             // compact towards the top end, keeping the list order
  for (int k = p.obs_end - 1; k >= p.obs_begin; --k) {
    if ((int)obs[k].ref_frame_id == kf_slot) continue;
    --w;
    if (w != k) { obs[w] = obs[k]; for (int j = 0; j < 7; ++j) T_obs[7 * (size_t)w + j] = T_obs[7 * (size_t)k + j]; }
  }
  pts[i].obs_begin = w;
}

// seeds of a dropped keyframe leave the pool (DepthFilter::removeKeyframe, depth_filter.cpp:153-170)
__global__ void kf_erase_seeds_kernel(int n, SeedRef* refs, int kf)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && refs[i].state == 0 && refs[i].kf == kf) refs[i].state = 1;
}

// DepthFilter::initializeSeeds (depth_filter.cpp:129-151): one Seed (ctor :36-45) per new corner, in cell order, into the empty
// slots of the sequence's pool in slot order.  One CTA per sequence; corners that find no slot are counted as dropped.
__global__ void __launch_bounds__(256) kf_append_seeds_kernel(DevCam cam, const svob200_corner* cells, int n_cells, double thr, const float* depth_mean,
                                                              const float* depth_min, const int* seed_off, SeedRef* refs, svob200_seed* seeds, int kf,
                                                              int batch_id, int* appended, int* dropped)
{
  __shared__ int s_slot_of_rank[8192];                // grids up to 8,192 cells (svob200_tracker_set_detector / _add_keyframe)
  const int b = blockIdx.x, tid = threadIdx.x;
  const svob200_corner* C = cells + (size_t)b * n_cells;
  const int p0 = seed_off[b], np = seed_off[b + 1] - p0;
  const svob200_seed sd = seed_prior(depth_mean[b], depth_min[b]);
  auto is_new = [&](int i) { return (double)C[i].score > thr; };
  auto empty = [&](int q) { return refs[p0 + q].state != 0; };
  auto put = [&](int i, int q) {
    const svob200_corner c = C[i];
    SeedRef ref;
    ref.px[0] = (double)c.x; ref.px[1] = (double)c.y;                 // Feature(frame, Vector2d(x * scale, y * scale), level)
    const v3d f = cam2world(cam, ref.px[0], ref.px[1]);               // Feature ctor, feature.h:43-51
    ref.f[0] = f.x; ref.f[1] = f.y; ref.f[2] = f.z;
    ref.image = b; ref.level = (uint8_t)c.level; ref.kf = (uint8_t)kf; ref.batch_id = (uint16_t)batch_id;
    ref.state = 0; ref.pad0 = 0; ref.pad1 = 0; ref.pad2[0] = ref.pad2[1] = ref.pad2[2] = 0;
    refs[p0 + q] = ref;
    seeds[p0 + q] = sd;
  };
  int n_new;
  const int n_fill = fill_free_slots<256>(n_cells, is_new, np, empty, s_slot_of_rank, &n_new, put);
  if (tid == 0) { appended[b] = n_fill; dropped[b] = n_new - n_fill; }
}

}  // namespace

// CUDA-event stage marks of one step (svob200_tracker_stage_ms / _stage_name): one entry per kernel of the
// step, except that the first also covers the frame copy/bind and the small per-step input copy
constexpr int kNumStages = 12;
static const char* const kStageNames[kNumStages] = {"frame+pyramid", "features_prepare", "sparse_align", "reproject_prepare",
                                                    "match_geom", "match_prepare", "match_refine", "seeds_geom", "seeds_search",
                                                    "seeds_refine", "seeds_finish", "stats"};

struct svob200_tracker {
  svob200_ctx* ctx = nullptr;
  svob200_camera cam{};
  int batch = 0, n_levels = 0;
  svob200_align_opts aopts{};
  svob200_matcher_opts mopts{};
  double conv_thresh = 100.0;
  svob200_seed seed_init{};
  int reseed = 1;
  int64_t uid = 0;                     // frame ids of this tracker: -(uid << 8 | n), n = 1, 2, ... (new_frame)
  int64_t fid_last = 0, fid_cur = 0;
  // keyframes: up to max_kfs frames of the pool are keyframes (index k = position in the tables d_kf_slot / d_T_kf); the frame
  // of a keyframe may at the same time be the `last` frame of the tracking chain
  static constexpr int MAX_KFS = 16;
  int64_t fid_kfs[MAX_KFS] = {};
  int kf_batch[MAX_KFS] = {};          // Seed::batch_id of the seeds initialised in keyframe k (0 = unused slot of the ring)
  std::vector<int64_t> frame_pool;     // every frame this tracker created
  int64_t next_fid = 0;
  int batch_counter = 0;               // Seed::batch_counter (depth_filter.cpp:139)
  int max_n_kfs = 3;                   // DepthFilter::Options::max_n_kfs (depth_filter.h:75)
  int seed_capacity = 0;               // slots per sequence of the seed pool (0: exactly the seeds of set_keyframe)
  int det_cell = 30, det_levels = 3;   // Config::gridSize / nPyrLevels, Config::triangMinCornerScore
  double det_thr = 20.0;
  uint8_t* d_occ = nullptr; unsigned long long* d_det_keys = nullptr; svob200_corner* d_det_cells = nullptr;
  int *d_det_counts = nullptr, *d_kf_appended = nullptr, *d_kf_dropped = nullptr;
  float *d_depth_mean = nullptr, *d_depth_min = nullptr;
  int det_cells_alloc = 0;
  long long steps_done = 0;
  int N = 0, S = 0, max_per = 0;
  int *d_ftr_off = nullptr, *d_seed_off = nullptr, *d_ftr_image = nullptr, *d_match_ok = nullptr;
  uint8_t* d_has_point = nullptr;
  svob200_feature_ref* d_ftrs = nullptr;            // the observation chosen for each map point in the current step
  double* d_pt_world = nullptr;
  // map points: K = max_kfs observation slots each (points / observations as svob200_reproject_map takes them)
  svob200_feature_ref* d_pobs = nullptr; double* d_T_pobs = nullptr; uint8_t* d_active = nullptr;
  int* d_match_level = nullptr; double* d_match_A = nullptr;
  int* d_sel = nullptr;                    // observation slot currently copied into d_ftrs[i] (-1: none)
  // point pool (svob200_tracker_set_point_pool): every sequence owns max(its set_keyframe points, pt_capacity) point slots;
  // the candidates of the steps of each parity wait in d_cand[parity] (one entry per point slot) until two steps later
  int pt_capacity = -1;                    // -1: no pool
  CandRec* d_cand[2] = {};
  int* d_cand_n[2] = {};                   // candidates of the sequence in that step (the entries beyond its slots are dropped)
  int *d_pt_created = nullptr, *d_pt_dropped = nullptr, *d_pt_rank = nullptr;
  // depth-filter seeds: 32-byte compact records + keyframe tables (pose per (keyframe, image), frame slot per keyframe)
  SeedRef* d_seed_refs = nullptr;
  double* d_T_kf = nullptr;            // [max_kfs][batch][7]
  int* d_kf_slot = nullptr;            // [max_kfs]
  SeedPoseRec* d_seed_poses = nullptr; // [max_kfs][batch], refreshed every step
  int n_kfs = 1;                       // rows of the tables in use (highest keyframe index + 1)
  int max_kfs = 4;                     // keyframe ring (svob200_tracker_set_keyframe_ring)
  svob200_seed* d_seeds = nullptr;
  double *d_step_in = nullptr;      // [T_last_w 7B | last_px 2N]
  double *d_xyz = nullptr, *d_T_init = nullptr, *d_T_cur = nullptr, *d_depth_ref = nullptr, *d_px_in = nullptr, *d_px_out = nullptr;
  svob200_align_result* d_align = nullptr;
  svob200_seed_obs* d_obs = nullptr;
  svob200_step_stats* d_stats = nullptr;
  uint8_t* d_align_scratch = nullptr;
  uint8_t* d_seed_scratch = nullptr;
  uint8_t* d_match_scratch = nullptr;
  uint8_t* h_pinned = nullptr; size_t h_cap = 0;
  std::vector<void*> owned;
  std::vector<int> h_ftr_off, h_seed_off;
  static constexpr int CHUNK = 256;    // sequences per H2D/compute pipeline chunk (host mode)
  // Asynchronous depth filter (device-memory steps of big batches): like the reference, whose DepthFilter runs in its own
  // thread behind a frame queue (depth_filter.cpp:63-103, :191-229), the seed update of frame k runs on its own stream while
  // the tracking chain (pyramid -> alignment -> matching) of frame k+1 is already in flight: the latency-bound alignment wave
  // overlaps the issue-bound epipolar search.  Everything a chain reads that the next steps overwrite is double-buffered by
  // step parity (pose table, step records) or guarded by an event (the frame slot it searches in is reused two steps later).
  // Every synchronising entry point joins the stream (ctx_join_aux; df_join where frame roles change).
  cudaStream_t df_stream = nullptr;
  cudaEvent_t df_done[2] = {}, ev_pose = nullptr, ev_track = nullptr;
  bool df_pending[2] = {false, false};
  long long step_no = 0;
  SeedPoseRec* d_seed_poses2 = nullptr;      // second pose table (odd steps)
  svob200_step_stats* d_stats2 = nullptr;    // second step-record array (odd steps)
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_ev;
  // chain mode (svob200_tracker_set_chain): reprojector grid rules + pose optimiser instead of refining every map point
  int chain_cell = 0, chain_max_fts = 0, chain_pose_opt = 0, chain_cells = 0;
  svob200_map_point* d_points = nullptr;
  svob200_reproj_result* d_reproj = nullptr;
  svob200_reproj_stats* d_rstats = nullptr;
  svob200_pose_opt_result* d_pose = nullptr;
  int *d_winner = nullptr, *d_m_level = nullptr, *d_m_point = nullptr, *d_m_count = nullptr, *d_seg_begin = nullptr, *d_seg_end = nullptr;
  double *d_m_f = nullptr, *d_m_pos = nullptr, *d_pose_work = nullptr;
  uint8_t* d_outlier = nullptr;
  uint8_t* d_reproj_scratch = nullptr;
  // single-stream latency: in device mode with small batches the 14 launches of a step are replayed as ONE CUDA graph
  // (captured once per distinct set of buffer addresses: a camera ring buffer has only a few), which removes the
  // per-launch driver cost and most of the inter-kernel gaps
  struct StepGraph { std::vector<uintptr_t> key; cudaGraphExec_t exec; long long launches; };
  std::vector<StepGraph> graphs;
  static constexpr int GRAPH_MAX_BATCH = 64;
  // inside a captured step the independent stages fork onto a second stream (see run_range): the graph then has parallel
  // branches and its critical path is 7 kernels instead of 13
  cudaStream_t fork_stream = nullptr;
  cudaEvent_t fork_ev[4] = {};
  // optional per-stage CUDA-event timing (bench.py's stage breakdown / roofline)
  bool profiling = false;
  cudaEvent_t ev[kNumStages + 1] = {};
};

// a device buffer of n elements that the tracker owns (freed by svob200_tracker_destroy)
template <class T> static int alloc_owned(svob200_tracker* t, T*& p, size_t n)
{
  p = nullptr;
  if (cudaMalloc((void**)&p, sizeof(T) * (n ? n : 1)) != cudaSuccess) { cudaGetLastError(); return fail(t->ctx, SVOB200_ERR_NOMEM, "tracker: device alloc of %zu bytes failed", sizeof(T) * n); }
  t->owned.push_back(p);
  return 0;
}

// a new frame of the tracker's pool
static int new_frame(svob200_tracker* t, int64_t* out_id)
{
  const int64_t id = -((t->uid << 8) | t->next_fid++);
  if (int e = svob200_frame_create(t->ctx, id, t->batch, t->cam.width, t->cam.height, t->n_levels)) return e;
  t->frame_pool.push_back(id); *out_id = id;
  return 0;
}

// the context's stream waits for every depth-filter chain in flight, so none is pending any more (before frame roles change)
static int df_join(svob200_tracker* t)
{
  if (int e = ctx_join_aux(t->ctx)) return e;
  t->df_pending[0] = t->df_pending[1] = false;
  return 0;
}

// captured steps hold the addresses and values they were captured with: drop them when those change
static void drop_graphs(svob200_tracker* t)
{
  for (auto& g : t->graphs) cudaGraphExecDestroy(g.exec);
  t->graphs.clear();
}

// the second stream of captured steps and its events, created with the first graph
static int ensure_fork_stream(svob200_tracker* t)
{
  svob200_ctx* ctx = t->ctx;
  if (t->fork_stream) return 0;
  CU(cudaStreamCreateWithFlags(&t->fork_stream, cudaStreamNonBlocking));
  for (auto& e : t->fork_ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}

// Enqueue `body` on the context's stream, either directly or — single-stream latency — as a replay of a CUDA graph captured
// from it the first time this `key` (every address the kernels receive by value) is seen.
template <class Body>
static int graph_or_direct(svob200_tracker* t, bool use_graph, const std::vector<uintptr_t>& key, Body body)
{
  svob200_ctx* ctx = t->ctx;
  cudaStream_t s = ctx->stream;
  if (!use_graph) return body();
  for (auto& g : t->graphs)
    if (g.key == key) {
      CU(cudaGraphLaunch(g.exec, s));
      ctx->launches += g.launches;
      return 0;
    }
  const long long launches0 = ctx->launches;
  CU(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  const int rc = body();
  cudaGraph_t graph = nullptr;
  const cudaError_t ee = cudaStreamEndCapture(s, &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ee != cudaSuccess || !graph) { if (graph) cudaGraphDestroy(graph); return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: graph capture failed: %s", cudaGetErrorString(ee)); }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: graph instantiate failed: %s", cudaGetErrorString(ie));
  if (t->graphs.size() >= 64) drop_graphs(t);
  t->graphs.push_back({key, exec, ctx->launches - launches0});
  CU(cudaGraphLaunch(exec, s));
  return 0;
}

extern "C" {

int svob200_tracker_create(svob200_ctx* ctx, const svob200_camera* cam, int batch, int n_levels, const svob200_align_opts* aopts,
                           const svob200_matcher_opts* mopts, double conv_thresh, float depth_mean, float depth_min, int reseed,
                           svob200_tracker** out)
{
  if (!ctx || !cam || !aopts || !mopts || !out || batch <= 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_create: bad arguments");
  // a level outside the pyramid would make the kernels dereference DevFrame.lvl[l] == nullptr (a sticky device fault):
  // the same range checks as svob200_sparse_align / svob200_match_direct, before anything is launched
  if (n_levels < 1 || n_levels > 7) return fail(ctx, SVOB200_ERR_ARG, "tracker_create: n_levels %d outside [1, 7]", n_levels);
  if (aopts->min_level < 0 || aopts->min_level > aopts->max_level || aopts->max_level >= n_levels)
    return fail(ctx, SVOB200_ERR_ARG, "tracker_create: alignment level range [%d,%d] outside the %d-level pyramid", aopts->min_level, aopts->max_level, n_levels);
  if (mopts->max_search_level < 0 || mopts->max_search_level >= n_levels)
    return fail(ctx, SVOB200_ERR_ARG, "tracker_create: max_search_level %d outside the %d-level pyramid", mopts->max_search_level, n_levels);
  if (mopts->max_epi_search_steps < 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_create: negative max_epi_search_steps %d", mopts->max_epi_search_steps);
  if (cam->width <= 0 || cam->height <= 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_create: bad camera size");
  static std::atomic<int64_t> uid_counter{0};
  svob200_tracker* t = new svob200_tracker();
  t->uid = ++uid_counter;
  t->ctx = ctx; t->cam = *cam; t->batch = batch; t->n_levels = n_levels; t->aopts = *aopts; t->mopts = *mopts;
  t->conv_thresh = conv_thresh; t->reseed = reseed; t->seed_init = seed_prior(depth_mean, depth_min);
  // three frames to start with (keyframe 0, last, cur), more as keyframes are inserted
  t->next_fid = 1;
  for (int64_t* pid : {&t->fid_kfs[0], &t->fid_last, &t->fid_cur})
    if (int e = new_frame(t, pid)) { for (int64_t id : t->frame_pool) svob200_frame_release(ctx, id); delete t; return e; }
  *out = t;
  return SVOB200_OK;
}

void svob200_tracker_destroy(svob200_tracker* t)
{
  if (!t) return;
  svob200_ctx* ctx = t->ctx;
  ctx_join_aux(ctx);
  cudaStreamSynchronize(ctx->stream);
  for (int64_t id : t->frame_pool) svob200_frame_release(ctx, id);
  for (void* p : t->owned) cudaFree(p);
  if (t->h_pinned) cudaFreeHost(t->h_pinned);
  for (auto e : t->chunk_ev) cudaEventDestroy(e);
  drop_graphs(t);
  if (t->copy_stream) cudaStreamDestroy(t->copy_stream);
  if (t->df_stream) { cudaStreamSynchronize(t->df_stream); ctx_remove_aux(ctx, t->df_stream); cudaStreamDestroy(t->df_stream); }
  for (auto e : t->df_done) if (e) cudaEventDestroy(e);
  if (t->ev_pose) cudaEventDestroy(t->ev_pose);
  if (t->ev_track) cudaEventDestroy(t->ev_track);
  if (t->fork_stream) cudaStreamDestroy(t->fork_stream);
  for (auto e : t->fork_ev) if (e) cudaEventDestroy(e);
  for (int k = 0; k <= kNumStages; ++k) if (t->ev[k]) cudaEventDestroy(t->ev[k]);
  delete t;
}

// Keyframe of every sequence: image, pose, map features (kf_px at level kf_level observing pt_world)
// and depth-filter seeds (seed_px at seed_level), all in HOST memory.
int svob200_tracker_set_keyframe(svob200_tracker* t, const uint8_t* imgs, int stride, const double* T_kf_w, const int* ftr_offsets,
                                 const double* kf_px, const int* kf_level, const double* pt_world, const int* seed_offsets,
                                 const double* seed_px, const int* seed_level)
{
  if (!t || !imgs || !T_kf_w || !ftr_offsets || !seed_offsets) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (t->d_stats) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_keyframe: keyframe already set (svob200_tracker_add_keyframe inserts further ones)");
  const int B = t->batch;
  const int N_in = ftr_offsets[B];
  const int S_in = seed_offsets[B];
  // validate everything BEFORE the first launch / allocation
  if (N_in < 0 || S_in < 0 || ftr_offsets[0] != 0 || seed_offsets[0] != 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: bad offsets");
  for (int b = 0; b < B; ++b)
    if (ftr_offsets[b + 1] < ftr_offsets[b] || seed_offsets[b + 1] < seed_offsets[b]) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: offsets must be non-decreasing");
  if (N_in > 0 && (!kf_px || !kf_level || !pt_world)) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: null feature arrays with %d features", N_in);
  if (S_in > 0 && (!seed_px || !seed_level)) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: null seed arrays with %d seeds", S_in);
  for (int i = 0; i < N_in; ++i) if (kf_level[i] < 0 || kf_level[i] >= t->n_levels) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: kf_level[%d] = %d outside the pyramid", i, kf_level[i]);
  for (int i = 0; i < S_in; ++i) if (seed_level[i] < 0 || seed_level[i] >= t->n_levels) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_keyframe: seed_level[%d] = %d outside the pyramid", i, seed_level[i]);
  if (int e = svob200_frame_upload(ctx, t->fid_kfs[0], imgs, stride, nullptr, SVOB200_MEM_HOST)) return e;
  // slots: sequence b owns [off[b], off[b+1]) = its items followed by empty slots up to the capacity (seeds: the seed pool;
  // map points: the point pool, capacity -1 without one)
  auto slot_offsets = [B](const int* item_off, int capacity) {
    std::vector<int> off(B + 1, 0);
    for (int b = 0; b < B; ++b) off[b + 1] = off[b] + std::max(item_off[b + 1] - item_off[b], capacity);
    return off;
  };
  const std::vector<int> pt_off = slot_offsets(ftr_offsets, t->pt_capacity), pool_off = slot_offsets(seed_offsets, t->seed_capacity);
  const int N = pt_off[B], S = pool_off[B];
  t->N = N; t->S = S;
  t->h_ftr_off = pt_off;
  t->h_seed_off = pool_off;
  for (int b = 0; b < B; ++b) t->max_per = std::max(t->max_per, pt_off[b + 1] - pt_off[b]);
  const int slot = svob200_frame_slot(ctx, t->fid_kfs[0]);
  t->kf_batch[0] = 0; t->n_kfs = 1;
  int err = 0;
  auto own = [&](auto*& p, size_t n) { if (!err) err = alloc_owned(t, p, n); };
  own(t->d_ftr_off, B + 1); own(t->d_seed_off, B + 1); own(t->d_ftr_image, N); own(t->d_match_ok, N); own(t->d_has_point, N);
  own(t->d_ftrs, N); own(t->d_seed_refs, S); own(t->d_pt_world, 3 * (size_t)N);
  own(t->d_pobs, (size_t)N * t->max_kfs); own(t->d_T_pobs, 7 * (size_t)N * t->max_kfs); own(t->d_active, N); own(t->d_match_level, N); own(t->d_match_A, 4 * (size_t)N); own(t->d_sel, N);
  own(t->d_points, N);
  own(t->d_T_kf, 7 * (size_t)B * t->max_kfs); own(t->d_kf_slot, t->max_kfs); own(t->d_seed_poses, (size_t)B * t->max_kfs); own(t->d_seed_poses2, (size_t)B * t->max_kfs);
  own(t->d_seeds, S); own(t->d_step_in, 7 * (size_t)B + 2 * (size_t)N); own(t->d_xyz, 3 * (size_t)N); own(t->d_T_init, 7 * (size_t)B);
  own(t->d_T_cur, 7 * (size_t)B); own(t->d_depth_ref, N); own(t->d_px_in, 2 * (size_t)N); own(t->d_px_out, 2 * (size_t)N);
  own(t->d_align, B); own(t->d_obs, S); own(t->d_stats, B); own(t->d_stats2, B);
  own(t->d_align_scratch, sparse_align_scratch_bytes(N)); own(t->d_seed_scratch, seeds_scratch_bytes(S)); own(t->d_match_scratch, match_scratch_bytes(N));
  if (t->pt_capacity >= 0) {
    for (int p = 0; p < 2; ++p) { own(t->d_cand[p], N); own(t->d_cand_n[p], B); }
    own(t->d_pt_created, B); own(t->d_pt_dropped, B); own(t->d_pt_rank, N);
  }
  if (err) {                 // an allocation that failed leaves the tracker as it was before the call (it can be retried or destroyed)
    for (void* q : t->owned) cudaFree(q);
    t->owned.clear();
    t->N = t->S = 0; t->max_per = 0; t->d_stats = nullptr; t->d_reproj = nullptr; t->det_cells_alloc = 0; t->d_det_counts = nullptr;
    return err;
  }
  cudaStream_t s = ctx->stream;
  CU(cudaMemcpyAsync(t->d_ftr_off, pt_off.data(), sizeof(int) * (B + 1), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_seed_off, pool_off.data(), sizeof(int) * (B + 1), cudaMemcpyHostToDevice, s));
  if (t->pt_capacity >= 0) {
    for (int p = 0; p < 2; ++p) CU(cudaMemsetAsync(t->d_cand_n[p], 0, sizeof(int) * B, s));
    CU(cudaMemsetAsync(t->d_pt_created, 0, sizeof(int) * B, s));
    CU(cudaMemsetAsync(t->d_pt_dropped, 0, sizeof(int) * B, s));
  }
  CU(cudaMemcpyAsync(t->d_T_kf, T_kf_w, sizeof(double) * 7 * B, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_kf_slot, &slot, sizeof(int), cudaMemcpyHostToDevice, s));
  // the caller's arrays in one copy; every point slot and seed slot is written on the device
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_fo = st.add(ftr_offsets, nullptr, sizeof(int) * (B + 1), 0), i_px = st.add(kf_px, nullptr, sizeof(double) * 2 * N_in, 0);
  const int i_lv = st.add(kf_level, nullptr, sizeof(int) * N_in, 0), i_pt = st.add(pt_world, nullptr, sizeof(double) * 3 * N_in, 0);
  const int i_so = st.add(seed_offsets, nullptr, sizeof(int) * (B + 1), 0), i_spx = st.add(seed_px, nullptr, sizeof(double) * 2 * S_in, 0);
  const int i_slv = st.add(seed_level, nullptr, sizeof(int) * S_in, 0);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (N || S) {
    kf_init_slots_kernel<<<B, 128, 0, s>>>(to_cam(&t->cam), t->max_kfs, slot, t->d_T_kf, t->d_ftr_off, st.dev<int>(i_fo), st.dev<double>(i_px),
                                           st.dev<int>(i_lv), st.dev<double>(i_pt), t->d_seed_off, st.dev<int>(i_so), st.dev<double>(i_spx),
                                           st.dev<int>(i_slv), t->seed_init, t->d_ftr_image, t->d_has_point, t->d_sel, t->d_pt_world, t->d_ftrs,
                                           t->d_points, t->d_pobs, t->d_T_pobs, t->d_seed_refs, t->d_seeds);
    ++ctx->launches;
    if (cudaGetLastError() != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "tracker_set_keyframe: launch error");
  }
  return st.download();                                  // the caller's arrays are host memory
}

int svob200_tracker_set_seed_pool(svob200_tracker* t, int capacity_per_sequence, int max_keyframes, int max_n_kfs, int reseed)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (t->d_stats) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_seed_pool: call before set_keyframe");
  if (capacity_per_sequence < 0 || max_keyframes < 1 || max_keyframes > svob200_tracker::MAX_KFS || max_n_kfs < 0 || reseed < 0 || reseed > 3)
    return fail(ctx, SVOB200_ERR_ARG, "tracker_set_seed_pool: bad arguments");
  t->seed_capacity = capacity_per_sequence; t->max_kfs = max_keyframes; t->max_n_kfs = max_n_kfs; t->reseed = reseed;
  // the whole frame pool now (keyframe ring + last + cur), so that no keyframe insertion allocates
  int64_t id;
  while ((int)t->frame_pool.size() < t->max_kfs + 2)
    if (int e = new_frame(t, &id)) return e;
  return SVOB200_OK;
}

int svob200_tracker_set_point_pool(svob200_tracker* t, int capacity_per_sequence)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (t->d_stats) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_point_pool: call before set_keyframe");
  if (capacity_per_sequence < 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_point_pool: negative capacity %d", capacity_per_sequence);
  t->pt_capacity = capacity_per_sequence;
  return SVOB200_OK;
}

int svob200_tracker_set_detector(svob200_tracker* t, int cell_size, int n_detect_levels, double detection_threshold)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (cell_size <= 0 || n_detect_levels < 1 || n_detect_levels > t->n_levels) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_detector: bad arguments");
  const int n_cells = ((t->cam.width + cell_size - 1) / cell_size) * ((t->cam.height + cell_size - 1) / cell_size);
  if (n_cells > 8192) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_detector: grid of %d cells exceeds the kernel's table (8192)", n_cells);
  t->det_cell = cell_size; t->det_levels = n_detect_levels; t->det_thr = detection_threshold;
  return SVOB200_OK;
}

// The frame of the most recent step becomes a keyframe of every sequence.
int svob200_tracker_add_keyframe(svob200_tracker* t, const float* depth_mean, const float* depth_min, int* n_new_seeds, int* n_dropped)
{
  if (!t || !depth_mean || !depth_min) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (!t->d_stats || t->steps_done == 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_add_keyframe: needs a keyframe and at least one step");
  if (t->chain_cell > 0) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_add_keyframe: not available in chain mode");
  const int B = t->batch, N = t->N, S = t->S;
  cudaStream_t s = ctx->stream;
  if (int e = df_join(t)) return e;                        // the depth filter of the last step may still be running
  drop_graphs(t);                                          // captured steps hold the old keyframe tables' values / frame roles
  // 1. the keyframe's index in the ring: a free one, else the oldest keyframe leaves (its seeds with it: removeKeyframe)
  int k = -1;
  for (int i = 0; i < t->max_kfs; ++i) if (t->fid_kfs[i] == 0) { k = i; break; }
  if (k < 0) {
    k = 0;
    for (int i = 1; i < t->max_kfs; ++i) if (t->kf_batch[i] < t->kf_batch[k]) k = i;
    if (S) { kf_erase_seeds_kernel<<<(S + 255) / 256, 256, 0, s>>>(S, t->d_seed_refs, k); ++ctx->launches; }
    if (N) {                                                 // Map::safeDeleteFrame: the points forget the keyframe
      FrameRec* old = find_frame(ctx, t->fid_kfs[k]);
      if (t->pt_capacity >= 0) {
        kf_drop_candidates_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->d_points, t->d_pobs, t->d_match_ok, t->d_has_point, old->slot); ++ctx->launches;
      }
      kf_drop_obs_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->max_kfs, t->d_points, t->d_pobs, t->d_T_pobs, old->slot, t->d_sel); ++ctx->launches;
    }
    t->fid_kfs[k] = 0;
  }
  // 2. the frame: the last step's current frame (now `last`).  Its level 0 may alias the caller's buffer: the keyframe owns a copy.
  FrameRec* r = find_frame(ctx, t->fid_last);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "tracker_add_keyframe: last frame missing");
  if (int e = frame_own_level0(ctx, r, true)) return e;
  t->fid_kfs[k] = t->fid_last;
  t->kf_batch[k] = ++t->batch_counter;                      // ++Seed::batch_counter (depth_filter.cpp:139)
  if (t->batch_counter >= 65535) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_add_keyframe: batch counter exhausted");
  t->n_kfs = std::max(t->n_kfs, k + 1);
  const int slot = r->slot;
  CU(cudaMemcpyAsync(t->d_kf_slot + k, &slot, sizeof(int), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_T_kf + 7 * (size_t)B * k, t->d_T_cur, sizeof(double) * 7 * B, cudaMemcpyDeviceToDevice, s));   // the frame's pose
  // 3. detector scratch
  const int gc = (t->cam.width + t->det_cell - 1) / t->det_cell, gr = (t->cam.height + t->det_cell - 1) / t->det_cell;
  const int n_cells = gc * gr;
  if (n_cells > 8192) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_add_keyframe: grid of %d cells exceeds the kernel's table (8192)", n_cells);
  if (t->det_cells_alloc < n_cells) {
    const size_t M = (size_t)B * n_cells;
    int err = 0;
    auto own = [&](auto*& p, size_t n) { if (!err) err = alloc_owned(t, p, n); };
    own(t->d_occ, M); own(t->d_det_keys, M); own(t->d_det_cells, M);
    if (!t->d_det_counts) { own(t->d_det_counts, B); own(t->d_kf_appended, B); own(t->d_kf_dropped, B); own(t->d_depth_mean, B); own(t->d_depth_min, B); }
    if (err) return err;
    t->det_cells_alloc = n_cells;
  }
  CU(cudaMemcpyAsync(t->d_depth_mean, depth_mean, sizeof(float) * B, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_depth_min, depth_min, sizeof(float) * B, cudaMemcpyHostToDevice, s));
  // 4. occupancy from the frame's features (the map points matched in it), FAST + Shi-Tomasi + grid, one seed per new corner
  CU(cudaMemsetAsync(t->d_occ, 0, (size_t)B * n_cells, s));
  if (N) { kf_occupancy_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->d_ftr_image, t->d_px_out, t->d_match_ok, t->det_cell, gc, n_cells, t->d_occ); ++ctx->launches; }
  if (launch_fast_detect(r->f, t->det_levels, t->det_cell, gc, gr, t->det_thr, t->d_occ, t->d_det_keys, t->d_det_cells, t->d_det_counts, s, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "tracker_add_keyframe: detector launch failed");
  if (S) {
    kf_append_seeds_kernel<<<B, 256, 0, s>>>(to_cam(&t->cam), t->d_det_cells, n_cells, t->det_thr, t->d_depth_mean, t->d_depth_min, t->d_seed_off, t->d_seed_refs,
                                             t->d_seeds, k, t->batch_counter, t->d_kf_appended, t->d_kf_dropped);
    ++ctx->launches;
  }
  // 5. the matched map points gain an observation in the new keyframe (frame_handler_mono.cpp:277-279)
  if (N) {
    kf_add_obs_kernel<<<(N + 255) / 256, 256, 0, s>>>(to_cam(&t->cam), N, t->max_kfs, t->d_points, t->d_pobs, t->d_T_pobs, t->d_ftr_image, t->d_match_ok, t->d_px_out,
                                                      t->d_match_level, slot, t->d_T_cur);
    ++ctx->launches;
  }
  if (cudaGetLastError() != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "tracker_add_keyframe: launch error");
  if (n_new_seeds) CU(cudaMemcpyAsync(n_new_seeds, S ? t->d_kf_appended : t->d_det_counts, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
  if (n_dropped && S) CU(cudaMemcpyAsync(n_dropped, t->d_kf_dropped, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));                             // depth_mean / depth_min are the caller's; the counts go back
  if (n_dropped && !S) for (int b = 0; b < B; ++b) n_dropped[b] = n_new_seeds ? n_new_seeds[b] : 0;
  return SVOB200_OK;
}

// the seed pool as it stands: 2 doubles px, level, keyframe index, batch id, state (0 alive, 1 empty) per slot (host arrays of S slots)
int svob200_tracker_get_seed_refs(svob200_tracker* t, double* px, int* level, int* kf, int* batch_id, int* state)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (int e = ctx_join_aux(ctx)) return e;
  std::vector<SeedRef> refs((size_t)std::max(t->S, 1));
  CU(cudaMemcpyAsync(refs.data(), t->d_seed_refs, sizeof(SeedRef) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < t->S; ++i) {
    if (px) { px[2 * i] = refs[i].px[0]; px[2 * i + 1] = refs[i].px[1]; }
    if (level) level[i] = refs[i].level;
    if (kf) kf[i] = refs[i].kf;
    if (batch_id) batch_id[i] = refs[i].batch_id;
    if (state) state[i] = refs[i].state;
  }
  return SVOB200_OK;
}
int svob200_tracker_num_seed_slots(svob200_tracker* t) { return t ? t->S : 0; }

// the point slots as they stand (host arrays of N slots: 3 doubles pos, SVOB200_POINT_* type, observation count) and the
// candidates created / dropped so far (one int per sequence); any pointer may be NULL
int svob200_tracker_get_points(svob200_tracker* t, double* pos, int* type, int* n_obs, int* created, int* dropped)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (int e = ctx_join_aux(ctx)) return e;
  const int B = t->batch;
  std::vector<svob200_map_point> pts((size_t)std::max(t->N, 1));
  std::vector<int> cr(B, 0), dr(B, 0);
  if (t->N) CU(cudaMemcpyAsync(pts.data(), t->d_points, sizeof(svob200_map_point) * (size_t)t->N, cudaMemcpyDeviceToHost, ctx->stream));
  if (t->d_pt_created) {
    CU(cudaMemcpyAsync(cr.data(), t->d_pt_created, sizeof(int) * B, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(dr.data(), t->d_pt_dropped, sizeof(int) * B, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < t->N; ++i) {
    if (pos) for (int k = 0; k < 3; ++k) pos[3 * (size_t)i + k] = pts[i].pos[k];
    if (type) type[i] = pts[i].type;
    if (n_obs) n_obs[i] = pts[i].obs_end - pts[i].obs_begin;
  }
  if (created) memcpy(created, cr.data(), sizeof(int) * B);
  if (dropped) memcpy(dropped, dr.data(), sizeof(int) * B);
  return SVOB200_OK;
}
int svob200_tracker_num_point_slots(svob200_tracker* t) { return t ? t->N : 0; }

int svob200_tracker_set_chain(svob200_tracker* t, int cell_size, int max_fts, int pose_opt)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (!t->d_stats) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_chain: set_keyframe first");
  if (t->pt_capacity >= 0) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_chain: not available with a point pool");
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaStreamSynchronize(ctx->stream));
  drop_graphs(t);                                                  // captured steps belong to the other mode
  if (cell_size <= 0) { t->chain_cell = 0; return SVOB200_OK; }
  const int B = t->batch, N = t->N;
  const int n_cells = ((t->cam.width + cell_size - 1) / cell_size) * ((t->cam.height + cell_size - 1) / cell_size);
  if (n_cells > 8192) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_chain: grid of %d cells exceeds the kernel's table (8192)", n_cells);
  if (!t->d_reproj || n_cells != t->chain_cells) {
    const size_t M = (size_t)B * n_cells;
    int err = 0;
    auto own = [&](auto*& p, size_t n) { if (!err) err = alloc_owned(t, p, n); };
    if (!t->d_reproj) { own(t->d_reproj, N); own(t->d_rstats, B); own(t->d_pose, B); own(t->d_m_count, B); own(t->d_seg_begin, B); own(t->d_seg_end, B);
                        own(t->d_reproj_scratch, reproject_scratch_bytes(N)); }
    own(t->d_winner, M); own(t->d_m_level, M); own(t->d_m_point, M); own(t->d_m_f, 3 * M); own(t->d_m_pos, 3 * M); own(t->d_pose_work, M); own(t->d_outlier, M);
    if (err) return err;
  }
  // the map points as reprojector candidates: insertion order = the keyframe's fts_ order, every point TYPE_UNKNOWN (d_points /
  // d_obs / d_T_obs already hold them with their observation lists)
  CU(cudaMemsetAsync(t->d_pose, 0, sizeof(svob200_pose_opt_result) * (size_t)B, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  t->chain_cell = cell_size; t->chain_max_fts = max_fts; t->chain_pose_opt = pose_opt ? 1 : 0; t->chain_cells = n_cells;
  return SVOB200_OK;
}

int svob200_tracker_set_last(svob200_tracker* t, const uint8_t* imgs, int stride, int mem)
{
  if (!t || !imgs) return SVOB200_ERR_ARG;
  if (int e = df_join(t)) return e;                    // a depth-filter chain may still be reading the frame slots
  return svob200_frame_upload(t->ctx, t->fid_last, imgs, stride, nullptr, mem);
}

// sub-batch view of a frame batch: images [c0, c0+cnt)
static DevFrame frame_view(const DevFrame& f, int c0, int cnt)
{
  DevFrame v = f;
  for (int l = 0; l < f.n_levels; ++l) v.lvl[l] = f.lvl[l] + (size_t)c0 * f.img_stride[l];
  v.batch = cnt;
  return v;
}

// the shape of one run_range call (see the head of the file)
struct RangeShape {
  cudaStream_t side;               // the fork branch of a captured step, else the context's stream
  bool defer_df;                   // the range stops after the tracking half of the step records: the depth filter goes to df_stream
  SeedPoseRec* pose_table;         // the pose table and the step records of this step (of its parity when deferred)
  svob200_step_stats* stats;
};

// DepthFilter::updateSeeds(cur) for the seeds of the sequences [c0, c1), on stream st
static int enqueue_seeds_update(svob200_tracker* t, int c0, int c1, const SeedPoseRec* table, cudaStream_t st, cudaEvent_t* marks)
{
  svob200_ctx* ctx = t->ctx;
  const int s0 = t->h_seed_off[c0], ns = t->h_seed_off[c1] - s0;
  if (launch_seeds_update_compact(ctx->d_table, find_frame(ctx, t->fid_cur)->slot, to_cam(&t->cam), ns, t->d_seed_refs + s0, t->d_kf_slot, t->batch, table,
                                  t->batch_counter, t->max_n_kfs, t->mopts, t->conv_thresh, t->d_seeds + s0, t->d_obs + s0, t->d_seed_scratch, t->S, s0,
                                  st, &ctx->launches, marks))
    return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: seeds_update failed");
  return 0;
}

// the step records of the sequences [c0, c1), on stream st: `parts` of step_stats_kernel, then the chain-mode fields
static int enqueue_step_stats(svob200_tracker* t, int c0, int c1, int parts, svob200_step_stats* d_stats, cudaStream_t st)
{
  svob200_ctx* ctx = t->ctx;
  const int cnt = c1 - c0, par = (int)(t->step_no & 1);
  const CandStage cand = {t->d_cand[par], t->d_cand_n[par], t->d_pt_created, t->d_ftr_off, t->d_T_kf, t->batch, c0};
  auto kernel = cand.rec ? step_stats_kernel<true> : step_stats_kernel<false>;
  kernel<<<cnt, 128, 0, st>>>(t->d_ftr_off + c0, t->d_seed_off + c0, t->d_align + c0, t->d_T_cur + 7 * (size_t)c0, t->d_match_ok, t->d_obs,
                              t->d_seeds, t->seed_init, t->reseed, d_stats + c0, parts, t->d_seed_refs, cand);
  ++ctx->launches;
  if (t->chain_cell > 0) {
    chain_stats_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(cnt, t->d_rstats + c0, t->d_pose + c0, t->chain_pose_opt, d_stats + c0); ++ctx->launches;
  }
  if (cudaGetLastError() != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: launch error");
  return 0;
}

// point pool: the candidates of two steps ago take their slots, at the head of the step on the context's stream (outside any
// captured graph).  Every shape waits for that step's depth filter first, so every shape inserts the same candidates.
static int enqueue_insert_candidates(svob200_tracker* t)
{
  if (t->pt_capacity < 0) return 0;
  svob200_ctx* ctx = t->ctx;
  const int par = (int)(t->step_no & 1);
  KfBatches kfb;
  for (int k = 0; k < svob200_tracker::MAX_KFS; ++k) kfb.v[k] = t->kf_batch[k];
  cand_insert_kernel<<<t->batch, 128, 0, ctx->stream>>>(t->max_kfs, t->batch, t->d_ftr_off, t->d_cand[par], t->d_cand_n[par], kfb, t->d_kf_slot, t->d_T_kf,
                                                        t->d_points, t->d_pt_world, t->d_pobs, t->d_T_pobs, t->d_sel, t->d_has_point, t->d_pt_rank,
                                                        t->d_pt_dropped);
  ++ctx->launches;
  if (cudaGetLastError() != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: candidate insertion launch error");
  return 0;
}

// all stages of one step for the sequences [c0, c1) on the context's stream, in the shape sh (level 0 of cur is in place)
// out_px / out_ok: optional device destinations of the refined pixels / match flags (device-mode callers): copied as soon as
// the matching stage is done, beside the depth filter in a forked step
static int run_range(svob200_tracker* t, int c0, int c1, const double* d_T_last, const double* d_last_px, bool marks, const RangeShape& sh,
                     double* out_px = nullptr, int* out_ok = nullptr)
{
  svob200_ctx* ctx = t->ctx;
  cudaStream_t s = ctx->stream;
  const DevCam cam = to_cam(&t->cam);
  FrameRec* last = find_frame(ctx, t->fid_last);
  FrameRec* cur = find_frame(ctx, t->fid_cur);
  const int cnt = c1 - c0;
  const int f0 = t->h_ftr_off[c0], nf = t->h_ftr_off[c1] - f0;
  const DevFrame vlast = frame_view(last->f, c0, cnt), vcur = frame_view(cur->f, c0, cnt);
#define MARK(k) do { if (marks && t->profiling) cudaEventRecord(t->ev[k], s); } while (0)
  // Captured steps (single-stream latency) fork: the per-feature preparation does not read the new pyramid, and the depth
  // filter and the map-point matching both depend on the aligned pose only (default mode), so each pair runs as parallel
  // branches of the graph; s2 == s everywhere else.
  cudaStream_t s2 = sh.side;
  const bool fork = s2 != s;
  if (fork) { CU(cudaEventRecord(t->fork_ev[0], s)); CU(cudaStreamWaitEvent(s2, t->fork_ev[0], 0)); }
  // 1. fused pyramid of the current frames
  {
    int modes[SVOB200_MAX_LEVELS];
    pyramid_round_modes(vcur, nullptr, modes);
    if (launch_pyramid(vcur, modes, s, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: pyramid launch failed");
  }
  MARK(1);
  // 2. Feature ctor / xyz_ref of the last frame's features, initial relative pose
  if (launch_features_prepare(cam, nf, d_last_px + 2 * (size_t)f0, t->d_pt_world + 3 * (size_t)f0, t->d_ftr_image + f0, d_T_last, nullptr,
                              t->d_xyz + 3 * (size_t)f0, s2, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: features_prepare failed");
  init_pose_kernel<<<(cnt + 127) / 128, 128, 0, s2>>>(cnt, d_T_last + 7 * (size_t)c0, t->d_T_init + 7 * (size_t)c0); ++ctx->launches;
  if (fork) { CU(cudaEventRecord(t->fork_ev[1], s2)); CU(cudaStreamWaitEvent(s, t->fork_ev[1], 0)); }
  MARK(2);
  // 3. SparseImgAlign::run(last, cur)
  if (launch_sparse_align(vlast, vcur, cam, cnt, t->N, t->max_per, t->d_ftr_off + c0, d_last_px, t->d_xyz, t->d_has_point,
                          t->d_T_init + 7 * (size_t)c0, t->aopts, t->d_align + c0, t->d_align_scratch, s, &ctx->launches,
                          d_T_last + 7 * (size_t)c0, t->d_T_cur + 7 * (size_t)c0))
    return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: sparse_align failed");
  MARK(3);
  // 4. cur.T_f_w = T_cur_from_ref * last.T_f_w (written by the alignment kernel's epilogue) ; reprojection of the map points
  // chain mode: the depth filter waits for the pose optimiser's T_cur, so its branch cannot start here
  cudaStream_t s_seeds = (fork && t->chain_cell <= 0) ? s2 : s;
  if (s_seeds != s) { CU(cudaEventRecord(t->fork_ev[2], s)); CU(cudaStreamWaitEvent(s_seeds, t->fork_ev[2], 0)); }
  if (t->chain_cell <= 0 && nf > 0) {
    // Point::getCloseViewObs per map point + px = cur.w2c(pos), depth_ref, T_cur_ref (the head of findMatchDirect)
    points_select_kernel<<<(nf + 127) / 128, 128, 0, s>>>(cam, nf, t->d_points + f0, t->d_pobs, t->d_T_pobs, t->d_ftr_image + f0, t->d_T_cur, t->d_ftrs + f0,
                                                          t->d_depth_ref + f0, t->d_px_in + 2 * (size_t)f0, t->d_active + f0, t->d_sel + f0);
    ++ctx->launches;
  }
  MARK(4);
  if (t->chain_cell > 0) {
    // 4b-5. chain mode: Reprojector::reprojectMap (grid, every in-frame candidate matched in parallel, per-cell first success,
    // maxFts) over the keyframe's map points, then pose_optimizer::optimizeGaussNewton on the frame's new features (in place
    // on T_cur, so the depth filter sees the optimised pose).
    const size_t cb = (size_t)c0 * t->chain_cells;
    const int rc = launch_reproject_map(ctx->d_table, cur->slot, cam, cnt, t->d_T_cur + 7 * (size_t)c0, t->d_ftr_off + c0, t->N, t->d_points, t->d_pobs,
                                        t->d_T_pobs, t->chain_cell, t->chain_max_fts, t->mopts, t->d_reproj, t->d_winner + cb, t->d_rstats + c0,
                                        t->d_reproj_scratch, t->d_match_scratch, t->d_m_f + 3 * cb, t->d_m_level + cb, t->d_m_pos + 3 * cb,
                                        t->d_m_point + cb, t->d_m_count + c0, s, &ctx->launches, c0, f0, nf);
    if (rc) return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: reproject_map failed (%d)", rc);
    MARK(5); MARK(6);
    chain_export_kernel<<<(nf + 127) / 128, 128, 0, s>>>(nf, t->d_reproj + f0, t->d_px_out + 2 * (size_t)f0, t->d_match_ok + f0); ++ctx->launches;
    if (t->chain_pose_opt) {
      chain_segments_kernel<<<(cnt + 127) / 128, 128, 0, s>>>(cnt, t->chain_cells, t->d_m_count + c0, t->d_seg_begin + c0, t->d_seg_end + c0); ++ctx->launches;
      // segments are relative to this range's slice of the compacted arrays
      if (launch_pose_optimize(cam, cnt, t->d_seg_begin + c0, t->d_seg_end + c0, t->d_m_f + 3 * cb, t->d_m_level + cb, t->d_m_pos + 3 * cb, 2.0, 10,
                               0.0000000001, 8.6851f, t->d_T_cur + 7 * (size_t)c0, t->d_pose + c0, t->d_outlier + cb, t->d_pose_work + cb, s, &ctx->launches))
        return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: pose_optimize failed");
    }
    MARK(7);
  } else {
  // 5. Matcher::findMatchDirect per map point (keyframe patch -> current frame)
  // (item indices inside the call are relative to f0, so the output arrays are passed at f0 as well)
  if (launch_match_direct(ctx->d_table, cur->slot, cam, nf, t->d_ftrs + f0, t->d_depth_ref + f0, t->d_px_in + 2 * (size_t)f0, t->mopts, nullptr,
                          t->d_px_out + 2 * (size_t)f0, t->d_match_ok + f0, t->d_match_scratch, t->N, f0, s, &ctx->launches,
                          (marks && t->profiling) ? &t->ev[5] : nullptr, t->d_active + f0, t->d_match_level + f0, t->d_match_A + 4 * (size_t)f0))
    return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: match_direct failed");
  MARK(7);
  }
  if (out_px) CU(cudaMemcpyAsync(out_px + 2 * (size_t)f0, t->d_px_out + 2 * (size_t)f0, sizeof(double) * 2 * (size_t)nf, cudaMemcpyDeviceToDevice, s));
  if (out_ok) CU(cudaMemcpyAsync(out_ok + f0, t->d_match_ok + f0, sizeof(int) * (size_t)nf, cudaMemcpyDeviceToDevice, s));
  // 6. DepthFilter::updateSeeds(cur): this range's rows of the pose table (from the step's final T_cur), then the seeds
  if (launch_seed_pose_table(cam, t->batch, t->n_kfs, c0, cnt, t->d_T_kf, t->d_T_cur, sh.pose_table, s_seeds, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "tracker_step: seed pose table failed");
  if (sh.defer_df) {
    // asynchronous depth filter (never forked: s_seeds == s): the df stream starts from the pose rows and writes its half of
    // the step records after the tracking half; the events tell it when
    CU(cudaEventRecord(t->ev_pose, s));
    if (int e = enqueue_step_stats(t, c0, c1, 1, sh.stats, s)) return e;
    CU(cudaEventRecord(t->ev_track, s));
    return 0;
  }
  if (int e = enqueue_seeds_update(t, c0, c1, sh.pose_table, s_seeds, (marks && t->profiling) ? &t->ev[8] : nullptr)) return e;
  if (s_seeds != s) { CU(cudaEventRecord(t->fork_ev[3], s_seeds)); CU(cudaStreamWaitEvent(s, t->fork_ev[3], 0)); }
  MARK(11);
  // 7. per-sequence statistics (+ steady-state re-seeding)
  if (int e = enqueue_step_stats(t, c0, c1, 3, sh.stats, s)) return e;
  MARK(12);
#undef MARK
  return 0;
}

int svob200_tracker_step(svob200_tracker* t, const uint8_t* cur_imgs, int stride, const double* T_last_w, const double* last_px,
                         svob200_step_stats* stats, double* px_refined, int* match_ok, int mem)
{
  if (!t || !cur_imgs || !T_last_w || !last_px) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (!t->d_stats) return fail(ctx, SVOB200_ERR_ARG, "tracker_step: set_keyframe first");
  const int B = t->batch, N = t->N;
  cudaStream_t s = ctx->stream;
  const size_t in_bytes = sizeof(double) * (7 * (size_t)B + 2 * (size_t)N);
  // the frame that receives the new images must not be a keyframe's (the frame of the step before a keyframe insertion is one):
  // take a free frame of the pool, or create one (the pool holds at most max_kfs + 2 frames)
  {
    auto is_kf = [&](int64_t id) { for (int i = 0; i < svob200_tracker::MAX_KFS; ++i) if (t->fid_kfs[i] == id) return true; return false; };
    if (is_kf(t->fid_cur)) {
      if (int e = df_join(t)) return e;                   // frame roles change: no depth-filter chain may be in flight
      int64_t pick = 0;
      for (int64_t id : t->frame_pool) if (id != t->fid_last && !is_kf(id)) { pick = id; break; }
      if (!pick) if (int e = new_frame(t, &pick)) return e;
      t->fid_cur = pick;
    }
  }
  if (t->profiling) cudaEventRecord(t->ev[0], s);
  if (mem == SVOB200_MEM_DEVICE) {
    // the frame slot that becomes `cur` now, the pose table and the step records of this parity were last used by the depth
    // filter chain of two steps ago: wait for it (the chain of the previous step keeps running beside this step's tracking)
    const int par = (int)(t->step_no & 1);
    if (t->df_pending[par]) { CU(cudaStreamWaitEvent(s, t->df_done[par], 0)); t->df_pending[par] = false; }
    // level 0 of the current frames aliases the caller's device buffer: no copy at all
    if (int e = frame_bind_level0(ctx, find_frame(ctx, t->fid_cur), cur_imgs, stride)) return e;
    const bool use_graph = !t->profiling && B <= svob200_tracker::GRAPH_MAX_BATCH;
    // everything the kernels of a step receive BY VALUE: the buffers of this call and the two frame views
    FrameRec* last = find_frame(ctx, t->fid_last);
    const std::vector<uintptr_t> key = {1, (uintptr_t)cur_imgs, (uintptr_t)stride, (uintptr_t)T_last_w, (uintptr_t)last_px, (uintptr_t)stats,
                                        (uintptr_t)px_refined, (uintptr_t)match_ok, (uintptr_t)t->fid_cur, (uintptr_t)t->fid_last,
                                        (uintptr_t)last->f.lvl[0], (uintptr_t)last->f.pitch[0], (uintptr_t)(t->pt_capacity >= 0 ? par : 0)};
    if (use_graph) if (int e = ensure_fork_stream(t)) return e;
    // direct launches of a big batch: the depth filter follows on its own stream (graphs, profiling and chain mode run it in place)
    const bool df_on_stream = !use_graph && !t->profiling && t->chain_cell <= 0 && t->S > 0;
    if (df_on_stream && !t->df_stream) {
      CU(cudaStreamCreateWithFlags(&t->df_stream, cudaStreamNonBlocking));
      if (int e = ctx_add_aux(ctx, t->df_stream)) return e;
      for (auto& e : t->df_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&t->ev_pose, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&t->ev_track, cudaEventDisableTiming));
    }
    if (!df_on_stream && (t->df_pending[0] || t->df_pending[1]))       // a step that runs the depth filter in place after asynchronous ones
      if (int e = df_join(t)) return e;
    if (int e = enqueue_insert_candidates(t)) return e;
    // graph + fork (only a capture runs the body then), asynchronous depth filter on this parity's pose table and step
    // records, or in place; with a point pool the captured step records its candidates into this parity's staging
    const RangeShape shape = {use_graph ? t->fork_stream : s, df_on_stream, (df_on_stream && par) ? t->d_seed_poses2 : t->d_seed_poses,
                              (df_on_stream && par) ? t->d_stats2 : t->d_stats};
    const int rc = graph_or_direct(t, use_graph, key, [&]() -> int {
      if (int e = run_range(t, 0, B, T_last_w, last_px, true, shape, px_refined, match_ok)) return e;
      if (!df_on_stream) {
        if (stats) CU(cudaMemcpyAsync(stats, shape.stats, sizeof(svob200_step_stats) * B, cudaMemcpyDeviceToDevice, s));
        return 0;
      }
      // the depth filter of the whole batch on its own stream: it starts as soon as the pose rows are written, and its
      // half of the step records (and their copy to the caller) follows the tracking half
      cudaStream_t df = t->df_stream;
      CU(cudaStreamWaitEvent(df, t->ev_pose, 0));
      if (int e = enqueue_seeds_update(t, 0, B, shape.pose_table, df, nullptr)) return e;
      CU(cudaStreamWaitEvent(df, t->ev_track, 0));
      if (int e = enqueue_step_stats(t, 0, B, 2, shape.stats, df)) return e;
      if (stats) CU(cudaMemcpyAsync(stats, shape.stats, sizeof(svob200_step_stats) * B, cudaMemcpyDeviceToDevice, df));
      CU(cudaEventRecord(t->df_done[par], df));
      t->df_pending[par] = true;
      return 0;
    });
    if (rc) return rc;
  } else {
    // host buffers: the frame copy is split into chunks on a copy stream so that chunk c+1 crosses
    // PCIe while chunk c is being processed; one small H2D for the per-step inputs, one D2H for results
    if (int e = df_join(t)) return e;                  // a depth-filter chain of earlier device-memory steps
    FrameRec* r = find_frame(ctx, t->fid_cur);
    if (int e = frame_own_level0(ctx, r, false)) return e;    // drop an earlier device binding
    const size_t out_bytes = sizeof(svob200_step_stats) * B + sizeof(double) * 2 * (size_t)N + sizeof(int) * (size_t)N;
    if (t->h_cap < in_bytes + out_bytes + 512) {
      if (t->h_pinned) cudaFreeHost(t->h_pinned);
      t->h_pinned = nullptr; t->h_cap = 0;
      CU(cudaMallocHost((void**)&t->h_pinned, in_bytes + out_bytes + 512));
      t->h_cap = in_bytes + out_bytes + 512;
    }
    const double* d_T_last = t->d_step_in;
    const double* d_last_px = t->d_step_in + 7 * (size_t)B;
    // the per-step inputs (poses, last pixel positions: 16 B per feature) are queued BEFORE the frame chunks: H2D copies are
    // served in submission order whatever their stream, and the first chunk's kernels wait for these (queued after the
    // chunks they cost 24.1 -> 30.7 ms per step).  Page-locked caller buffers are read by the copy engine directly, pageable
    // ones go through the staging buffer.
    {
      auto is_pinned = [](const void* p) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return at.type == cudaMemoryTypeHost;
      };
      if (B >= 64 && is_pinned(T_last_w) && is_pinned(last_px)) {
        CU(cudaMemcpyAsync(t->d_step_in, T_last_w, sizeof(double) * 7 * B, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(t->d_step_in + 7 * (size_t)B, last_px, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, s));
      } else {
        memcpy(t->h_pinned, T_last_w, sizeof(double) * 7 * B);
        memcpy(t->h_pinned + sizeof(double) * 7 * B, last_px, sizeof(double) * 2 * (size_t)N);
        CU(cudaMemcpyAsync(t->d_step_in, t->h_pinned, in_bytes, cudaMemcpyHostToDevice, s));
      }
    }
    if (int e = enqueue_insert_candidates(t)) return e;
    const int chunk = (t->profiling || B <= svob200_tracker::CHUNK) ? B : svob200_tracker::CHUNK;
    const int n_chunks = (B + chunk - 1) / chunk;
    if (!t->copy_stream) CU(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    while ((int)t->chunk_ev.size() < n_chunks + 1) { cudaEvent_t e; CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); t->chunk_ev.push_back(e); }
    // the copy stream must not overwrite level 0 before earlier work on the compute stream is done
    CU(cudaEventRecord(t->chunk_ev[n_chunks], s));
    CU(cudaStreamWaitEvent(t->copy_stream, t->chunk_ev[n_chunks], 0));
    const int h = r->f.h[0];
    for (int c = 0; c < n_chunks; ++c) {
      const int c0 = c * chunk, c1 = std::min(B, c0 + chunk);
      // contiguous on both sides (pitch == stride == width): one linear copy, which the copy engine moves a few percent
      // faster than the same bytes as a 2D copy of h * count rows
      if (r->f.pitch[0] == stride && stride == r->f.w[0])
        CU(cudaMemcpyAsync(r->f.lvl[0] + (size_t)c0 * r->f.img_stride[0], cur_imgs + (size_t)c0 * h * stride, (size_t)stride * h * (c1 - c0),
                           cudaMemcpyHostToDevice, t->copy_stream));
      else
        CU(cudaMemcpy2DAsync(r->f.lvl[0] + (size_t)c0 * r->f.img_stride[0], r->f.pitch[0], cur_imgs + (size_t)c0 * h * stride, stride,
                             r->f.w[0], (size_t)h * (c1 - c0), cudaMemcpyHostToDevice, t->copy_stream));
      CU(cudaEventRecord(t->chunk_ev[c], t->copy_stream));
    }
    // small batches: the kernels of the step (not the copies: the caller's host pointers change from call to call) are
    // replayed as the same forked graph as in device mode; the kernels only see the tracker's own buffers here, so two
    // graphs (the frame pair swaps every step) serve every call.  (A graph WITHOUT the parallel branches gained nothing in
    // host mode: 0.202 -> 0.199 ms for C2.)
    const bool use_graph = !t->profiling && n_chunks == 1 && B <= svob200_tracker::GRAPH_MAX_BATCH;
    if (use_graph) if (int e = ensure_fork_stream(t)) return e;
    const RangeShape shape = {use_graph ? t->fork_stream : s, false, t->d_seed_poses, t->d_stats};
    // each chunk's kernels wait for its own frame copy
    for (int c = 0; c < n_chunks; ++c) {
      const int c0 = c * chunk, c1 = std::min(B, c0 + chunk);
      CU(cudaStreamWaitEvent(s, t->chunk_ev[c], 0));
      if (use_graph) {
        FrameRec* last = find_frame(ctx, t->fid_last);
        const std::vector<uintptr_t> key = {2, (uintptr_t)t->fid_cur, (uintptr_t)t->fid_last, (uintptr_t)r->f.lvl[0], (uintptr_t)r->f.pitch[0],
                                            (uintptr_t)last->f.lvl[0], (uintptr_t)last->f.pitch[0], (uintptr_t)d_T_last,
                                            (uintptr_t)(t->pt_capacity >= 0 ? (t->step_no & 1) : 0)};
        if (int e = graph_or_direct(t, true, key, [&]() { return run_range(t, 0, B, d_T_last, d_last_px, true, shape); })) return e;
      } else if (int e = run_range(t, c0, c1, d_T_last, d_last_px, n_chunks == 1, shape)) return e;
    }
    uint8_t* ho = t->h_pinned + ((in_bytes + 255) & ~(size_t)255);
    uint8_t* h_stats = ho; uint8_t* h_px = h_stats + sizeof(svob200_step_stats) * B; uint8_t* h_ok = h_px + sizeof(double) * 2 * (size_t)N;
    if (stats) CU(cudaMemcpyAsync(h_stats, t->d_stats, sizeof(svob200_step_stats) * B, cudaMemcpyDeviceToHost, s));
    if (px_refined) CU(cudaMemcpyAsync(h_px, t->d_px_out, sizeof(double) * 2 * (size_t)N, cudaMemcpyDeviceToHost, s));
    if (match_ok) CU(cudaMemcpyAsync(h_ok, t->d_match_ok, sizeof(int) * (size_t)N, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (stats) memcpy(stats, h_stats, sizeof(svob200_step_stats) * B);
    if (px_refined) memcpy(px_refined, h_px, sizeof(double) * 2 * (size_t)N);
    if (match_ok) memcpy(match_ok, h_ok, sizeof(int) * (size_t)N);
  }
  std::swap(t->fid_last, t->fid_cur);       // the current frame becomes the last frame
  ++t->step_no; ++t->steps_done;
  return SVOB200_OK;
}

int svob200_tracker_get_seeds(svob200_tracker* t, svob200_seed* out)
{
  if (!t || !out) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaMemcpyAsync(out, t->d_seeds, sizeof(svob200_seed) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

int svob200_tracker_launches_per_step(void) { return 14; }

// raw svob200_align_result records of the most recent step (diagnostics: tools/align_timing.py)
int svob200_tracker_debug_align(svob200_tracker* t, svob200_align_result* out)
{
  if (!t || !out || !t->d_align) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  CU(cudaMemcpyAsync(out, t->d_align, sizeof(svob200_align_result) * (size_t)t->batch, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// stage timing: CUDA events recorded on the launching stream between the kernels of a step
int svob200_tracker_enable_profiling(svob200_tracker* t, int on)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (on && !t->ev[0]) for (int k = 0; k <= kNumStages; ++k) CU(cudaEventCreate(&t->ev[k]));
  t->profiling = on != 0;
  return SVOB200_OK;
}

int svob200_tracker_num_stages(void) { return kNumStages; }
const char* svob200_tracker_stage_name(int i) { return (i >= 0 && i < kNumStages) ? kStageNames[i] : ""; }

int svob200_tracker_stage_ms(svob200_tracker* t, float* ms, int cap)
{
  if (!t || !ms || !t->ev[0] || cap < kNumStages) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  CU(cudaEventSynchronize(t->ev[kNumStages]));
  for (int k = 0; k < kNumStages; ++k) CU(cudaEventElapsedTime(&ms[k], t->ev[k], t->ev[k + 1]));
  return SVOB200_OK;
}

// per-seed observation records of the last step (status, n_evals, ...) for workload accounting
int svob200_tracker_get_seed_obs(svob200_tracker* t, svob200_seed_obs* out)
{
  if (!t || !out) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaMemcpyAsync(out, t->d_obs, sizeof(svob200_seed_obs) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

}  // extern "C"
