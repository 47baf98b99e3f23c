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

// ---- keyframe insertion (svob200_tracker_add_keyframes): a kernel of a sequence that is not selected (kf_new < 0) or loses no
// keyframe (kf_old < 0) leaves it untouched
// occupancy of the frame's existing features = the map points matched in it (AbstractDetector::setExistingFeatures,
// feature_detection.cpp:40-58: cell of (px.y / cell, px.x / cell) with the x86 double -> int conversion)
__global__ void kf_occupancy_kernel(int n, const int* ftr_image, const double* px, const int* match_ok, const int* kf_new, int cell, int grid_cols,
                                    int n_cells, uint8_t* occ)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !match_ok[i] || kf_new[ftr_image[i]] < 0) return;
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
__global__ void __launch_bounds__(128) cand_insert_kernel(int K, int batch, const int* pt_off, const CandRec* cand, const int* cand_n, const int* kf_batch,
                                                          const int* kf_slot, const double* T_kf, svob200_map_point* pts, double* pt_world,
                                                          svob200_feature_ref* obs, double* T_obs, int* sel, uint8_t* has_point,
                                                          int* slot_of_rank, int* dropped)
{
  const int b = blockIdx.x, tid = threadIdx.x;
  const int P0 = pt_off[b], P = pt_off[b + 1] - P0, n = cand_n[b];
  const CandRec* C = cand + P0;
  auto valid = [&](int c) { return C[c].batch_id == kf_batch[C[c].kf * batch + b]; };
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
__global__ void kf_drop_candidates_kernel(int n, svob200_map_point* pts, const svob200_feature_ref* obs, const int* match_ok, uint8_t* has_point,
                                          const int* image, const int* kf_old, const int* kf_slot)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int k = kf_old[image[i]];
  if (k < 0) return;
  const svob200_map_point p = pts[i];
  if (p.type != SVOB200_POINT_CANDIDATE || match_ok[i] || (int)obs[p.obs_begin].ref_frame_id != kf_slot[k]) return;
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
                                  const int* match_ok, const double* px, const int* level, const int* kf_new, const int* kf_slot_of, const double* T_cur_w)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !match_ok[i] || kf_new[image[i]] < 0) return;
  const int kf_slot = kf_slot_of[kf_new[image[i]]];
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
__global__ void kf_drop_obs_kernel(int n, int K, svob200_map_point* pts, svob200_feature_ref* obs, double* T_obs, const int* image, const int* kf_old,
                                   const int* kf_slot_of, int* sel)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || kf_old[image[i]] < 0) return;
  const int kf_slot = kf_slot_of[kf_old[image[i]]];
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
__global__ void kf_erase_seeds_kernel(int n, SeedRef* refs, const int* kf_old)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && refs[i].state == 0 && refs[i].kf == kf_old[refs[i].image]) refs[i].state = 1;
}

// DepthFilter::initializeSeeds (depth_filter.cpp:129-151): one Seed (ctor :36-45) per new corner, in cell order, into the empty
// slots of the sequence's pool in slot order.  One CTA per sequence; corners that find no slot are counted as dropped.
__global__ void __launch_bounds__(256) kf_append_seeds_kernel(DevCam cam, const svob200_corner* cells, int n_cells, double thr, const float* depth_mean,
                                                              const float* depth_min, const int* seed_off, SeedRef* refs, svob200_seed* seeds,
                                                              const int* kf_new, const int* batch_counter, int* appended, int* dropped)
{
  __shared__ int s_slot_of_rank[kMaxGridCells];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int kf = kf_new[b], batch_id = batch_counter[b];
  if (kf < 0) { if (tid == 0) appended[b] = dropped[b] = kf == -2 ? -1 : 0; return; }   // refused (batch counter exhausted) / not selected
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
  // without a seed pool (no slot anywhere) the counts are the corners found, every one of them dropped
  if (tid == 0) { appended[b] = seed_off[gridDim.x] ? n_fill : n_new; dropped[b] = n_new - n_fill; }
}

// ---- per-sequence keyframe rings (svob200_tracker_add_keyframes): ring index k of sequence b is image b of store frame k;
// kf_batch[k * batch + b] is the Seed::batch_id of that keyframe (-1: free), batch_counter[b] the sequence's Seed::batch_counter.
// One thread per sequence: a selected sequence takes its first free index, else its oldest keyframe leaves (kf_old = that index);
// the new keyframe is the frame of the most recent step, with its pose.  kf_new / kf_old = -1: not selected / nothing leaves.
// Seed::batch_id is 16 bits wide (SeedRef): a sequence whose counter reached kMaxBatchId takes no further keyframe (kf_new = -2).
constexpr int kMaxBatchId = 65534;
__global__ void kf_select_kernel(int batch, int max_kfs, const uint8_t* which, int* kf_batch, int* batch_counter, int* kf_new, int* kf_old,
                                 const double* T_cur_w, double* T_kf)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  kf_old[b] = -1;
  if (which && !which[b]) { kf_new[b] = -1; return; }
  if (batch_counter[b] >= kMaxBatchId) { kf_new[b] = -2; return; }
  int k = -1, old = -1;
  for (int i = 0; i < max_kfs; ++i) if (kf_batch[i * batch + b] < 0) { k = i; break; }
  if (k < 0) {
    old = 0;
    for (int i = 1; i < max_kfs; ++i) if (kf_batch[i * batch + b] < kf_batch[old * batch + b]) old = i;
    k = old;
  }
  const int id = ++batch_counter[b];                        // ++Seed::batch_counter (depth_filter.cpp:139)
  kf_batch[k * batch + b] = id;
  kf_new[b] = k; kf_old[b] = old;
  for (int j = 0; j < 7; ++j) T_kf[7 * ((size_t)k * batch + b) + j] = T_cur_w[7 * (size_t)b + j];
}

// The images of the selected sequences, every pyramid level, into their keyframe's store frame (frames[kf_slot[kf_new[b]]]).
// Rows are copied in 16-byte words up to the width rounded up to 16: both pitches are multiples of 16 and at least that.
__global__ void __launch_bounds__(256) kf_store_copy_kernel(DevFrame src, const DevFrame* frames, const int* kf_slot, const int* kf_new)
{
  const int b = blockIdx.y;
  const int k = kf_new[b];
  if (k < 0) return;
  const DevFrame& dst = frames[kf_slot[k]];
  for (int l = 0; l < src.n_levels; ++l) {
    const int words = (src.w[l] + 15) / 16, n = words * src.h[l];
    const uint8_t* in = src.lvl[l] + (size_t)b * src.img_stride[l];
    uint8_t* out = dst.lvl[l] + (size_t)b * dst.img_stride[l];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
      const int y = i / words, x = 16 * (i - y * words);
      *reinterpret_cast<uint4*>(out + (size_t)y * dst.pitch[l] + x) = __ldg(reinterpret_cast<const uint4*>(in + (size_t)y * src.pitch[l] + x));
    }
  }
}

// frame_utils::getSceneDepth of the most recent step's frame, one CTA per sequence: the depths z = (T_cur_w * pos).z of the
// point slots matched in it, compacted in slot order into z_buf; depth_mean = (float) the element of rank n/2 of the ascending
// depths (vk::getMedian: nth_element), depth_min = (float)(0.5 * min).  n == 0 leaves depth_mean / depth_min as they are.
__global__ void __launch_bounds__(128) scene_depth_kernel(const int* pt_off, const svob200_map_point* pts, const int* match_ok, const double* T_cur_w,
                                                          double* z_buf, float* depth_mean, float* depth_min, int* n_points)
{
  const int b = blockIdx.x, tid = threadIdx.x;
  const int p0 = pt_off[b], np = pt_off[b + 1] - p0;
  const int chunk = (np + 127) / 128, q0 = min(tid * chunk, np), q1 = min(q0 + chunk, np);
  const double* T = T_cur_w + 7 * (size_t)b;
  int local = 0;
  for (int q = q0; q < q1; ++q) local += match_ok[p0 + q] != 0;
  int n;
  int r = block_exclusive_scan<128>(local, &n);
  double zmin = INFINITY;
  for (int q = q0; q < q1; ++q) {
    if (!match_ok[p0 + q]) continue;
    const svob200_map_point p = pts[p0 + q];
    const double z = se3_transform(T, {p.pos[0], p.pos[1], p.pos[2]}).z;
    z_buf[p0 + r++] = z;
    zmin = fmin(zmin, z);
  }
  __shared__ double s_min[4];
  for (int o = 16; o > 0; o >>= 1) zmin = fmin(zmin, __shfl_xor_sync(0xffffffffu, zmin, o));
  if ((tid & 31) == 0) s_min[tid >> 5] = zmin;
  __syncthreads();                                         // (also publishes z_buf to the CTA)
  if (tid == 0 && n_points) n_points[b] = n;
  if (n == 0) return;
  if (tid == 0) depth_min[b] = (float)(0.5 * fmin(fmin(s_min[0], s_min[1]), fmin(s_min[2], s_min[3])));
  const double* Z = z_buf + p0;
  const int want = n / 2;
  for (int i = tid; i < n; i += 128) {                     // the element whose rank (ties by position) is n/2
    const double zi = Z[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += (Z[j] < zi) || (Z[j] == zi && j < i);
    if (rank == want) depth_mean[b] = (float)zi;
  }
}

}  // namespace

// CUDA-event stage marks of one step (svob200_tracker_stage_ms / _stage_name): one entry per kernel of the
// step, except that the first also covers the frame copy/bind and the small per-step input copy
constexpr int kNumStages = 12;
static const char* const kStageNames[kNumStages] = {"frame+pyramid", "features_prepare", "sparse_align", "reproject_prepare",
                                                    "match_geom", "match_prepare", "match_refine", "seeds_geom", "seeds_search",
                                                    "seeds_refine", "seeds_finish", "stats"};

// The device arrays of one group, one cudaMalloc each, and their byte total; all are freed with the owner.  Move-only: a
// move-assignment swaps, so the arrays it replaces are freed when the moved-from temporary goes.
class DevArrays {
 public:
  DevArrays() = default;
  DevArrays(const DevArrays&) = delete;
  DevArrays& operator=(const DevArrays&) = delete;
  DevArrays(DevArrays&& o) noexcept { swap(o); }
  DevArrays& operator=(DevArrays&& o) noexcept { swap(o); return *this; }
  ~DevArrays() { for (void* p : ptrs_) cudaFree(p); }
  // p = an array of n elements (of one element when n == 0: an array that is present is never null); false if it failed
  template <class T> bool alloc(T*& p, size_t n)
  {
    const size_t bytes = sizeof(T) * (n ? n : 1);
    if (cudaMalloc((void**)&p, bytes) != cudaSuccess) { cudaGetLastError(); return false; }
    ptrs_.push_back(p);
    bytes_ += (long long)bytes;
    return true;
  }
  bool empty() const { return ptrs_.empty(); }
  long long bytes() const { return bytes_; }

 private:
  void swap(DevArrays& o) { std::swap(ptrs_, o.ptrs_); std::swap(bytes_, o.bytes_); }
  std::vector<void*> ptrs_;
  long long bytes_ = 0;
};

// The tracker's device arrays, grouped by the call that sizes them.  A sizing call builds a whole new group before it changes
// the tracker and then moves it in, so a failed allocation leaves the tracker as it was.  A group exists once its call made it.
// Slots (set_keyframe): the point and seed slots of every sequence, the keyframe tables, the step buffers and their scratch.
struct Slots {
  DevArrays mem;
  int *ftr_off = nullptr, *seed_off = nullptr, *ftr_image = nullptr, *match_ok = nullptr;
  uint8_t* has_point = nullptr;
  svob200_feature_ref* ftrs = nullptr;            // the observation chosen for each map point in the current step
  double* pt_world = nullptr;
  svob200_map_point* points = nullptr;
  // map points: K = max_kfs observation slots each (points / observations as svob200_reproject_map takes them)
  svob200_feature_ref* pobs = nullptr; double* T_pobs = nullptr; uint8_t* active = nullptr;
  int* match_level = nullptr; double* match_A = nullptr;
  int* sel = nullptr;                    // observation slot currently copied into ftrs[i] (-1: none)
  // point pool (present only with one): the candidates of the steps of each parity wait in cand[parity] (one entry per point
  // slot) until two steps later
  CandRec* cand[2] = {};
  int* cand_n[2] = {};                   // candidates of the sequence in that step (the entries beyond its slots are dropped)
  int *pt_created = nullptr, *pt_dropped = nullptr, *pt_rank = nullptr;
  // keyframe rings: kf_batch[k][b] = Seed::batch_id of ring index k of sequence b (-1: free), batch_counter[b] =
  // Seed::batch_counter (depth_filter.cpp:139)
  int *kf_batch = nullptr, *batch_counter = nullptr;
  int *kf_new = nullptr, *kf_old = nullptr;     // of the latest insertion: the ring index taken / left, per sequence (-1: none)
  uint8_t* kf_which = nullptr;                  // host-memory insertion masks, staged
  float *depth_mean = nullptr, *depth_min = nullptr;
  double* sd_z = nullptr;                // svob200_tracker_scene_depth: the depths of the matched point slots
  int* sd_n = nullptr;
  // depth-filter seeds: 32-byte compact records + keyframe tables (pose per (keyframe, image), frame slot per keyframe)
  SeedRef* seed_refs = nullptr;
  double* T_kf = nullptr;                // [max_kfs][batch][7]
  int* kf_slot = nullptr;                // [max_kfs]
  SeedPoseRec *seed_poses = nullptr, *seed_poses2 = nullptr;   // [max_kfs][batch], refreshed every step (2: odd steps)
  svob200_seed* seeds = nullptr;
  double* step_in = nullptr;             // [T_last_w 7B | last_px 2N]
  double *xyz = nullptr, *T_init = nullptr, *T_cur = nullptr, *depth_ref = nullptr, *px_in = nullptr, *px_out = nullptr;
  svob200_align_result* align = nullptr;
  svob200_seed_obs* obs = nullptr;
  svob200_step_stats *stats = nullptr, *stats2 = nullptr;     // step records (2: odd steps)
  uint8_t *align_scratch = nullptr, *seed_scratch = nullptr, *match_scratch = nullptr;
};

// Detector (the first add_keyframes after set_keyframe or after set_detector changed the grid): scratch of n_cells per image
struct Detector {
  DevArrays mem;
  int n_cells = 0;
  uint8_t* occ = nullptr; unsigned long long* keys = nullptr; svob200_corner* cells = nullptr;
  int *counts = nullptr, *kf_appended = nullptr, *kf_dropped = nullptr;
};

// Chain (set_chain on a tracker without one, or with another grid): the reprojector's and the pose optimiser's arrays
struct Chain {
  DevArrays mem;
  int n_cells = 0;
  svob200_reproj_result* reproj = nullptr;
  svob200_reproj_stats* rstats = nullptr;
  svob200_pose_opt_result* pose = nullptr;
  int *winner = nullptr, *m_level = nullptr, *m_point = nullptr, *m_count = nullptr, *seg_begin = nullptr, *seg_end = nullptr;
  double *m_f = nullptr, *m_pos = nullptr, *pose_work = nullptr;
  uint8_t* outlier = nullptr;
  uint8_t* reproj_scratch = nullptr;
};

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
  // keyframes: every sequence has its own ring of max_kfs keyframes.  Ring index k of sequence b is image b of the keyframe
  // store's frame fid_kfs[k] (frame slot slots.kf_slot[k], pose slots.T_kf[k][b]); the ring state lives on the device
  static constexpr int MAX_KFS = 16;
  int64_t fid_kfs[MAX_KFS] = {};
  std::vector<int64_t> frame_pool;     // every frame this tracker created
  int64_t next_fid = 0;
  int max_n_kfs = 3;                   // DepthFilter::Options::max_n_kfs (depth_filter.h:75)
  int seed_capacity = 0;               // slots per sequence of the seed pool (0: exactly the seeds of set_keyframe)
  int det_cell = 30, det_levels = 3;   // Config::gridSize / nPyrLevels, Config::triangMinCornerScore
  double det_thr = 20.0;
  long long steps_done = 0;
  int N = 0, S = 0, max_per = 0;
  // point pool (svob200_tracker_set_point_pool): every sequence owns max(its set_keyframe points, pt_capacity) point slots
  int pt_capacity = -1;                // -1: no pool
  int n_kfs = 1;                       // rows of the tables in use (no sequence has more keyframes: min(max_kfs, 1 + insertions))
  int max_kfs = 4;                     // keyframe ring (svob200_tracker_set_keyframe_ring)
  Slots slots;
  Detector det;
  Chain chain;
  uint8_t* h_pinned = nullptr; size_t h_cap = 0;
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
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_ev;
  // chain mode (svob200_tracker_set_chain): reprojector grid rules + pose optimiser instead of refining every map point
  int chain_cell = 0, chain_max_fts = 0, chain_pose_opt = 0;
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

// the frame slot of every store frame that exists (slots.kf_slot, constant once the store is complete)
static int upload_kf_slots(svob200_tracker* t)
{
  svob200_ctx* ctx = t->ctx;
  int slots[svob200_tracker::MAX_KFS] = {};
  for (int k = 0; k < t->max_kfs; ++k) if (t->fid_kfs[k]) slots[k] = svob200_frame_slot(ctx, t->fid_kfs[k]);
  CU(cudaMemcpyAsync(t->slots.kf_slot, slots, sizeof(int) * t->max_kfs, cudaMemcpyHostToDevice, ctx->stream));
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
  // three frames to start with (store frame 0, last, cur); the other store frames come with set_seed_pool or the first insertion
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
  if (!t->slots.mem.empty()) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_keyframe: keyframe already set (svob200_tracker_add_keyframe inserts further ones)");
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
  int max_per = 0;
  for (int b = 0; b < B; ++b) max_per = std::max(max_per, pt_off[b + 1] - pt_off[b]);
  const int slot = svob200_frame_slot(ctx, t->fid_kfs[0]);
  const size_t K = t->max_kfs;
  Slots g;
  DevArrays& m = g.mem;
  bool ok = m.alloc(g.ftr_off, B + 1) && m.alloc(g.seed_off, B + 1) && m.alloc(g.ftr_image, N) && m.alloc(g.match_ok, N) && m.alloc(g.has_point, N) &&
            m.alloc(g.ftrs, N) && m.alloc(g.seed_refs, S) && m.alloc(g.pt_world, 3 * (size_t)N) &&
            m.alloc(g.pobs, N * K) && m.alloc(g.T_pobs, 7 * (size_t)N * K) && m.alloc(g.active, N) && m.alloc(g.match_level, N) && m.alloc(g.match_A, 4 * (size_t)N) &&
            m.alloc(g.sel, N) && m.alloc(g.points, N) &&
            m.alloc(g.T_kf, 7 * (size_t)B * K) && m.alloc(g.kf_slot, K) && m.alloc(g.seed_poses, B * K) && m.alloc(g.seed_poses2, B * K) &&
            m.alloc(g.seeds, S) && m.alloc(g.step_in, 7 * (size_t)B + 2 * (size_t)N) && m.alloc(g.xyz, 3 * (size_t)N) && m.alloc(g.T_init, 7 * (size_t)B) &&
            m.alloc(g.T_cur, 7 * (size_t)B) && m.alloc(g.depth_ref, N) && m.alloc(g.px_in, 2 * (size_t)N) && m.alloc(g.px_out, 2 * (size_t)N) &&
            m.alloc(g.align, B) && m.alloc(g.obs, S) && m.alloc(g.stats, B) && m.alloc(g.stats2, B) &&
            m.alloc(g.kf_batch, B * K) && m.alloc(g.batch_counter, B) && m.alloc(g.kf_new, B) && m.alloc(g.kf_old, B) && m.alloc(g.kf_which, B) &&
            m.alloc(g.depth_mean, B) && m.alloc(g.depth_min, B) && m.alloc(g.sd_n, B) && m.alloc(g.sd_z, N) &&
            m.alloc(g.align_scratch, sparse_align_scratch_bytes(N)) && m.alloc(g.seed_scratch, seeds_scratch_bytes(S)) &&
            m.alloc(g.match_scratch, match_scratch_bytes(N));
  if (ok && t->pt_capacity >= 0)
    ok = m.alloc(g.cand[0], N) && m.alloc(g.cand_n[0], B) && m.alloc(g.cand[1], N) && m.alloc(g.cand_n[1], B) && m.alloc(g.pt_created, B) &&
         m.alloc(g.pt_dropped, B) && m.alloc(g.pt_rank, N);
  if (!ok) return fail(ctx, SVOB200_ERR_NOMEM, "tracker_set_keyframe: out of device memory for the slot arrays");
  t->slots = std::move(g);
  t->N = N; t->S = S; t->max_per = max_per;
  t->h_ftr_off = pt_off;
  t->h_seed_off = pool_off;
  t->n_kfs = 1;
  cudaStream_t s = ctx->stream;
  CU(cudaMemcpyAsync(t->slots.ftr_off, pt_off.data(), sizeof(int) * (B + 1), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->slots.seed_off, pool_off.data(), sizeof(int) * (B + 1), cudaMemcpyHostToDevice, s));
  if (t->pt_capacity >= 0) {
    for (int p = 0; p < 2; ++p) CU(cudaMemsetAsync(t->slots.cand_n[p], 0, sizeof(int) * B, s));
    CU(cudaMemsetAsync(t->slots.pt_created, 0, sizeof(int) * B, s));
    CU(cudaMemsetAsync(t->slots.pt_dropped, 0, sizeof(int) * B, s));
  }
  // every ring index starts with keyframe 0's pose: the pose table of a step covers rows whose index a sequence has not used yet
  for (int k = 0; k < t->max_kfs; ++k) CU(cudaMemcpyAsync(t->slots.T_kf + 7 * (size_t)B * k, T_kf_w, sizeof(double) * 7 * B, cudaMemcpyHostToDevice, s));
  {                                                      // every sequence's ring holds keyframe 0 (batch id 0), nothing else
    std::vector<int> kb((size_t)B * t->max_kfs, -1);
    std::fill(kb.begin(), kb.begin() + B, 0);
    CU(cudaMemcpyAsync(t->slots.kf_batch, kb.data(), sizeof(int) * kb.size(), cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(t->slots.batch_counter, 0, sizeof(int) * B, s));
  }
  if (int e = upload_kf_slots(t)) return e;
  // the caller's arrays in one copy; every point slot and seed slot is written on the device
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_fo = st.add(ftr_offsets, nullptr, sizeof(int) * (B + 1), 0), i_px = st.add(kf_px, nullptr, sizeof(double) * 2 * N_in, 0);
  const int i_lv = st.add(kf_level, nullptr, sizeof(int) * N_in, 0), i_pt = st.add(pt_world, nullptr, sizeof(double) * 3 * N_in, 0);
  const int i_so = st.add(seed_offsets, nullptr, sizeof(int) * (B + 1), 0), i_spx = st.add(seed_px, nullptr, sizeof(double) * 2 * S_in, 0);
  const int i_slv = st.add(seed_level, nullptr, sizeof(int) * S_in, 0);
  if (int e = st.layout()) return e;
  if (int e = st.push()) return e;
  if (N || S) {
    kf_init_slots_kernel<<<B, 128, 0, s>>>(to_cam(&t->cam), t->max_kfs, slot, t->slots.T_kf, t->slots.ftr_off, st.dev<int>(i_fo), st.dev<double>(i_px),
                                           st.dev<int>(i_lv), st.dev<double>(i_pt), t->slots.seed_off, st.dev<int>(i_so), st.dev<double>(i_spx),
                                           st.dev<int>(i_slv), t->seed_init, t->slots.ftr_image, t->slots.has_point, t->slots.sel, t->slots.pt_world, t->slots.ftrs,
                                           t->slots.points, t->slots.pobs, t->slots.T_pobs, t->slots.seed_refs, t->slots.seeds);
    ++ctx->launches;
    CU_AT("tracker_set_keyframe: kf_init_slots_kernel", cudaGetLastError());
  }
  return st.download();                                  // the caller's arrays are host memory
}

int svob200_tracker_set_seed_pool(svob200_tracker* t, int capacity_per_sequence, int max_keyframes, int max_n_kfs, int reseed)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (!t->slots.mem.empty()) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_seed_pool: call before set_keyframe");
  if (capacity_per_sequence < 0 || max_keyframes < 1 || max_keyframes > svob200_tracker::MAX_KFS || max_n_kfs < 0 || reseed < 0 || reseed > 3)
    return fail(ctx, SVOB200_ERR_ARG, "tracker_set_seed_pool: bad arguments");
  t->seed_capacity = capacity_per_sequence; t->max_kfs = max_keyframes; t->max_n_kfs = max_n_kfs; t->reseed = reseed;
  // the whole frame pool now (keyframe store + last + cur), so that no keyframe insertion allocates
  for (int k = 1; k < t->max_kfs; ++k)
    if (!t->fid_kfs[k]) if (int e = new_frame(t, &t->fid_kfs[k])) return e;
  return SVOB200_OK;
}

int svob200_tracker_set_point_pool(svob200_tracker* t, int capacity_per_sequence)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (!t->slots.mem.empty()) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_point_pool: call before set_keyframe");
  if (capacity_per_sequence < 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_point_pool: negative capacity %d", capacity_per_sequence);
  t->pt_capacity = capacity_per_sequence;
  return SVOB200_OK;
}

int svob200_tracker_set_detector(svob200_tracker* t, int cell_size, int n_detect_levels, double detection_threshold)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (cell_size <= 0 || n_detect_levels < 1 || n_detect_levels > t->n_levels) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_detector: bad arguments");
  const long long n_cells = grid_cells(t->cam.width, t->cam.height, cell_size);
  if (n_cells > kMaxGridCells) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_detector: grid of %lld cells exceeds the limit of %d", n_cells, kMaxGridCells);
  // a grid of another size releases the detector scratch (the next insertion makes it anew) once no insertion reads it
  if (!t->det.mem.empty() && t->det.n_cells != n_cells) {
    if (int e = ctx_join_aux(ctx)) return e;
    CU(cudaStreamSynchronize(ctx->stream));
    t->det = Detector();
  }
  t->det_cell = cell_size; t->det_levels = n_detect_levels; t->det_thr = detection_threshold;
  return SVOB200_OK;
}

// The frame of the most recent step becomes a keyframe of the sequences `which` selects (NULL: every sequence), each in its
// own ring: what svob200_tracker_add_keyframe did for a tracker of that sequence alone.  Every per-sequence choice is made on
// the device, so in SVOB200_MEM_DEVICE mode nothing here waits for the device.
int svob200_tracker_add_keyframes(svob200_tracker* t, const uint8_t* which, const float* depth_mean, const float* depth_min, int* n_new_seeds,
                                  int* n_dropped, int mem)
{
  if (!t || !depth_mean || !depth_min) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (mem != SVOB200_MEM_HOST && mem != SVOB200_MEM_DEVICE) return fail(ctx, SVOB200_ERR_ARG, "tracker_add_keyframes: bad mem %d", mem);
  if (t->slots.mem.empty() || t->steps_done == 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_add_keyframes: needs a keyframe and at least one step");
  if (t->chain_cell > 0) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_add_keyframes: not available in chain mode");
  const int B = t->batch, N = t->N, S = t->S;
  const long long grid = grid_cells(t->cam.width, t->cam.height, t->det_cell);
  if (grid > kMaxGridCells) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_add_keyframes: grid of %lld cells exceeds the limit of %d", grid, kMaxGridCells);
  const int gc = (t->cam.width + t->det_cell - 1) / t->det_cell, gr = (t->cam.height + t->det_cell - 1) / t->det_cell, n_cells = (int)grid;
  cudaStream_t s = ctx->stream;
  // the detector scratch when the tracker has none (after set_keyframe, or after set_detector released it once no work in
  // flight used it), then the keyframe store when set_seed_pool did not make it; the scratch goes in once both exist
  Detector det;
  if (t->det.mem.empty()) {
    const size_t M = (size_t)B * n_cells;
    DevArrays& m = det.mem;
    if (!(m.alloc(det.occ, M) && m.alloc(det.keys, M) && m.alloc(det.cells, M) && m.alloc(det.counts, B) && m.alloc(det.kf_appended, B) &&
          m.alloc(det.kf_dropped, B)))
      return fail(ctx, SVOB200_ERR_NOMEM, "tracker_add_keyframes: out of device memory for the detector scratch");
    det.n_cells = n_cells;
  }
  bool new_store = false;
  for (int k = 1; k < t->max_kfs; ++k)
    if (!t->fid_kfs[k]) { if (int e = new_frame(t, &t->fid_kfs[k])) return e; new_store = true; }
  if (new_store) if (int e = upload_kf_slots(t)) return e;
  if (t->det.mem.empty()) t->det = std::move(det);
  if (int e = df_join(t)) return e;                        // the depth filter of the last step may still be running
  const float *d_dm = depth_mean, *d_dn = depth_min;
  const uint8_t* d_which = which;
  if (mem == SVOB200_MEM_HOST) {
    CU(cudaMemcpyAsync(t->slots.depth_mean, depth_mean, sizeof(float) * B, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(t->slots.depth_min, depth_min, sizeof(float) * B, cudaMemcpyHostToDevice, s));
    if (which) CU(cudaMemcpyAsync(t->slots.kf_which, which, (size_t)B, cudaMemcpyHostToDevice, s));
    d_dm = t->slots.depth_mean; d_dn = t->slots.depth_min; d_which = which ? t->slots.kf_which : nullptr;
  }
  // 1. every selected sequence's ring index: a free one, else its oldest keyframe leaves (its seeds with it: removeKeyframe)
  const bool may_evict = t->n_kfs == t->max_kfs;           // (no sequence holds more keyframes than n_kfs)
  kf_select_kernel<<<(B + 127) / 128, 128, 0, s>>>(B, t->max_kfs, d_which, t->slots.kf_batch, t->slots.batch_counter, t->slots.kf_new, t->slots.kf_old,
                                                   t->slots.T_cur, t->slots.T_kf);
  ++ctx->launches;
  CU_AT("tracker_add_keyframes: kf_select_kernel", cudaGetLastError());
  if (!may_evict) { t->n_kfs = std::min(t->max_kfs, t->n_kfs + 1); drop_graphs(t); }   // captured steps hold n_kfs
  if (may_evict) {
    if (S) {
      kf_erase_seeds_kernel<<<(S + 255) / 256, 256, 0, s>>>(S, t->slots.seed_refs, t->slots.kf_old); ++ctx->launches;
      CU_AT("tracker_add_keyframes: kf_erase_seeds_kernel", cudaGetLastError());
    }
    if (N) {                                                 // Map::safeDeleteFrame: the points forget the keyframe
      if (t->pt_capacity >= 0) {
        kf_drop_candidates_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->slots.points, t->slots.pobs, t->slots.match_ok, t->slots.has_point, t->slots.ftr_image, t->slots.kf_old,
                                                                  t->slots.kf_slot);
        ++ctx->launches;
        CU_AT("tracker_add_keyframes: kf_drop_candidates_kernel", cudaGetLastError());
      }
      kf_drop_obs_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->max_kfs, t->slots.points, t->slots.pobs, t->slots.T_pobs, t->slots.ftr_image, t->slots.kf_old, t->slots.kf_slot,
                                                         t->slots.sel);
      ++ctx->launches;
      CU_AT("tracker_add_keyframes: kf_drop_obs_kernel", cudaGetLastError());
    }
  }
  // 2. the frame: the last step's current frame (now `last`), every level, into the store
  FrameRec* r = resident_frame(ctx, t->fid_last, "tracker_add_keyframes"); if (!r) return SVOB200_ERR_NOFRAME;
  kf_store_copy_kernel<<<dim3(16, B), 256, 0, s>>>(r->f, ctx->d_table, t->slots.kf_slot, t->slots.kf_new);
  ++ctx->launches;
  CU_AT("tracker_add_keyframes: kf_store_copy_kernel", cudaGetLastError());
  // 3. occupancy from the frame's features (the map points matched in it), FAST + Shi-Tomasi + grid on the selected images,
  // one seed per new corner
  CU(cudaMemsetAsync(t->det.occ, 0, (size_t)B * n_cells, s));
  if (N) {
    kf_occupancy_kernel<<<(N + 255) / 256, 256, 0, s>>>(N, t->slots.ftr_image, t->slots.px_out, t->slots.match_ok, t->slots.kf_new, t->det_cell, gc, n_cells, t->det.occ);
    ++ctx->launches;
    CU_AT("tracker_add_keyframes: kf_occupancy_kernel", cudaGetLastError());
  }
  CU_AT("tracker_add_keyframes: launch_fast_detect",
        launch_fast_detect(r->f, t->det_levels, t->det_cell, gc, gr, t->det_thr, t->det.occ, t->det.keys, t->det.cells, t->det.counts, s, &ctx->launches,
                           t->slots.kf_new));
  kf_append_seeds_kernel<<<B, 256, 0, s>>>(to_cam(&t->cam), t->det.cells, n_cells, t->det_thr, d_dm, d_dn, t->slots.seed_off, t->slots.seed_refs,
                                           t->slots.seeds, t->slots.kf_new, t->slots.batch_counter, t->det.kf_appended, t->det.kf_dropped);
  ++ctx->launches;
  CU_AT("tracker_add_keyframes: kf_append_seeds_kernel", cudaGetLastError());
  // 4. the matched map points gain an observation in the new keyframe (frame_handler_mono.cpp:277-279)
  if (N) {
    kf_add_obs_kernel<<<(N + 255) / 256, 256, 0, s>>>(to_cam(&t->cam), N, t->max_kfs, t->slots.points, t->slots.pobs, t->slots.T_pobs, t->slots.ftr_image,
                                                      t->slots.match_ok, t->slots.px_out, t->slots.match_level, t->slots.kf_new, t->slots.kf_slot, t->slots.T_cur);
    ++ctx->launches;
    CU_AT("tracker_add_keyframes: kf_add_obs_kernel", cudaGetLastError());
  }
  // the counts (unselected sequences: 0, refused ones: -1).  Without a seed pool n_dropped repeats n_new_seeds, and is 0 when
  // n_new_seeds is not asked for (as svob200_tracker_add_keyframe always reported it)
  const cudaMemcpyKind kind = mem == SVOB200_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  if (n_new_seeds) CU(cudaMemcpyAsync(n_new_seeds, t->det.kf_appended, sizeof(int) * B, kind, s));
  const bool zero_dropped = n_dropped && !S && !n_new_seeds;
  if (n_dropped && !zero_dropped) CU(cudaMemcpyAsync(n_dropped, t->det.kf_dropped, sizeof(int) * B, kind, s));
  if (zero_dropped && mem == SVOB200_MEM_DEVICE) CU(cudaMemsetAsync(n_dropped, 0, sizeof(int) * B, s));
  if (mem == SVOB200_MEM_HOST) CU(cudaStreamSynchronize(s));   // depth_mean / depth_min / which are the caller's; the counts go back
  if (zero_dropped && mem == SVOB200_MEM_HOST) memset(n_dropped, 0, sizeof(int) * B);
  return SVOB200_OK;
}

int svob200_tracker_add_keyframe(svob200_tracker* t, const float* depth_mean, const float* depth_min, int* n_new_seeds, int* n_dropped)
{
  return svob200_tracker_add_keyframes(t, nullptr, depth_mean, depth_min, n_new_seeds, n_dropped, SVOB200_MEM_HOST);
}

int svob200_tracker_scene_depth(svob200_tracker* t, float* depth_mean, float* depth_min, int* n_points, int mem)
{
  if (!t || !depth_mean || !depth_min) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (mem != SVOB200_MEM_HOST && mem != SVOB200_MEM_DEVICE) return fail(ctx, SVOB200_ERR_ARG, "tracker_scene_depth: bad mem %d", mem);
  if (t->slots.mem.empty() || t->steps_done == 0) return fail(ctx, SVOB200_ERR_ARG, "tracker_scene_depth: needs a keyframe and at least one step");
  const int B = t->batch;
  cudaStream_t s = ctx->stream;
  const bool dev = mem == SVOB200_MEM_DEVICE;
  scene_depth_kernel<<<B, 128, 0, s>>>(t->slots.ftr_off, t->slots.points, t->slots.match_ok, t->slots.T_cur, t->slots.sd_z, dev ? depth_mean : t->slots.depth_mean,
                                       dev ? depth_min : t->slots.depth_min, dev ? n_points : t->slots.sd_n);
  ++ctx->launches;
  CU_AT("tracker_scene_depth: scene_depth_kernel", cudaGetLastError());
  if (dev) return SVOB200_OK;
  std::vector<float> dm(B), dn(B);
  std::vector<int> n(B);
  CU(cudaMemcpyAsync(dm.data(), t->slots.depth_mean, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(dn.data(), t->slots.depth_min, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(n.data(), t->slots.sd_n, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (int b = 0; b < B; ++b) {
    if (n[b] > 0) { depth_mean[b] = dm[b]; depth_min[b] = dn[b]; }
    if (n_points) n_points[b] = n[b];
  }
  return SVOB200_OK;
}

// the seed pool as it stands: 2 doubles px, level, keyframe index, batch id, state (0 alive, 1 empty) per slot (host arrays of S slots)
int svob200_tracker_get_seed_refs(svob200_tracker* t, double* px, int* level, int* kf, int* batch_id, int* state)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (int e = ctx_join_aux(ctx)) return e;
  std::vector<SeedRef> refs((size_t)std::max(t->S, 1));
  CU(cudaMemcpyAsync(refs.data(), t->slots.seed_refs, sizeof(SeedRef) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
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
  if (t->N) CU(cudaMemcpyAsync(pts.data(), t->slots.points, sizeof(svob200_map_point) * (size_t)t->N, cudaMemcpyDeviceToHost, ctx->stream));
  if (t->pt_capacity >= 0 && !t->slots.mem.empty()) {          // a point pool
    CU(cudaMemcpyAsync(cr.data(), t->slots.pt_created, sizeof(int) * B, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(dr.data(), t->slots.pt_dropped, sizeof(int) * B, cudaMemcpyDeviceToHost, ctx->stream));
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
long long svob200_tracker_device_bytes(const svob200_tracker* t) { return t ? t->slots.mem.bytes() + t->det.mem.bytes() + t->chain.mem.bytes() : 0; }

int svob200_tracker_set_chain(svob200_tracker* t, int cell_size, int max_fts, int pose_opt)
{
  if (!t) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  if (t->slots.mem.empty()) return fail(ctx, SVOB200_ERR_ARG, "tracker_set_chain: set_keyframe first");
  if (t->pt_capacity >= 0) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_chain: not available with a point pool");
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaStreamSynchronize(ctx->stream));
  drop_graphs(t);                                                  // captured steps belong to the other mode
  if (cell_size <= 0) { t->chain_cell = 0; return SVOB200_OK; }
  const int B = t->batch, N = t->N;
  const long long n_cells = grid_cells(t->cam.width, t->cam.height, cell_size);
  if (n_cells > kMaxGridCells) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "tracker_set_chain: grid of %lld cells exceeds the limit of %d", n_cells, kMaxGridCells);
  if (t->chain.mem.empty() || n_cells != t->chain.n_cells) {
    const size_t M = (size_t)B * n_cells;
    Chain g;
    DevArrays& m = g.mem;
    if (!(m.alloc(g.reproj, N) && m.alloc(g.rstats, B) && m.alloc(g.pose, B) && m.alloc(g.m_count, B) && m.alloc(g.seg_begin, B) &&
          m.alloc(g.seg_end, B) && m.alloc(g.reproj_scratch, reproject_scratch_bytes(N)) && m.alloc(g.winner, M) && m.alloc(g.m_level, M) &&
          m.alloc(g.m_point, M) && m.alloc(g.m_f, 3 * M) && m.alloc(g.m_pos, 3 * M) && m.alloc(g.pose_work, M) && m.alloc(g.outlier, M)))
      return fail(ctx, SVOB200_ERR_NOMEM, "tracker_set_chain: out of device memory for the chain arrays");
    g.n_cells = (int)n_cells;
    t->chain = std::move(g);
  }
  t->chain_cell = cell_size; t->chain_max_fts = max_fts; t->chain_pose_opt = pose_opt ? 1 : 0;
  // the map points as reprojector candidates: insertion order = the keyframe's fts_ order, every point TYPE_UNKNOWN (slots.points
  // / pobs / T_pobs already hold them with their observation lists)
  CU(cudaMemsetAsync(t->chain.pose, 0, sizeof(svob200_pose_opt_result) * (size_t)B, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
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
  CU_AT("tracker_step: launch_seeds_update_compact",
        launch_seeds_update_compact(ctx->d_table, find_frame(ctx, t->fid_cur)->slot, to_cam(&t->cam), ns, t->slots.seed_refs + s0, t->slots.kf_slot, t->batch, table,
                                    t->slots.batch_counter, t->max_n_kfs, t->mopts, t->conv_thresh, t->slots.seeds + s0, t->slots.obs + s0, t->slots.seed_scratch, t->S, s0,
                                    st, &ctx->launches, marks));
  return 0;
}

// the step records of the sequences [c0, c1), on stream st: `parts` of step_stats_kernel, then the chain-mode fields
static int enqueue_step_stats(svob200_tracker* t, int c0, int c1, int parts, svob200_step_stats* d_stats, cudaStream_t st)
{
  svob200_ctx* ctx = t->ctx;
  const int cnt = c1 - c0, par = (int)(t->step_no & 1);
  const CandStage cand = {t->slots.cand[par], t->slots.cand_n[par], t->slots.pt_created, t->slots.ftr_off, t->slots.T_kf, t->batch, c0};
  auto kernel = cand.rec ? step_stats_kernel<true> : step_stats_kernel<false>;
  kernel<<<cnt, 128, 0, st>>>(t->slots.ftr_off + c0, t->slots.seed_off + c0, t->slots.align + c0, t->slots.T_cur + 7 * (size_t)c0, t->slots.match_ok, t->slots.obs,
                              t->slots.seeds, t->seed_init, t->reseed, d_stats + c0, parts, t->slots.seed_refs, cand);
  ++ctx->launches;
  CU_AT("tracker_step: step_stats_kernel", cudaGetLastError());
  if (t->chain_cell > 0) {
    chain_stats_kernel<<<(cnt + 127) / 128, 128, 0, st>>>(cnt, t->chain.rstats + c0, t->chain.pose + c0, t->chain_pose_opt, d_stats + c0); ++ctx->launches;
    CU_AT("tracker_step: chain_stats_kernel", cudaGetLastError());
  }
  return 0;
}

// point pool: the candidates of two steps ago take their slots, at the head of the step on the context's stream (outside any
// captured graph).  Every shape waits for that step's depth filter first, so every shape inserts the same candidates.
static int enqueue_insert_candidates(svob200_tracker* t)
{
  if (t->pt_capacity < 0) return 0;
  svob200_ctx* ctx = t->ctx;
  const int par = (int)(t->step_no & 1);
  cand_insert_kernel<<<t->batch, 128, 0, ctx->stream>>>(t->max_kfs, t->batch, t->slots.ftr_off, t->slots.cand[par], t->slots.cand_n[par], t->slots.kf_batch,
                                                        t->slots.kf_slot, t->slots.T_kf, t->slots.points, t->slots.pt_world, t->slots.pobs, t->slots.T_pobs, t->slots.sel,
                                                        t->slots.has_point, t->slots.pt_rank, t->slots.pt_dropped);
  ++ctx->launches;
  CU_AT("tracker_step: cand_insert_kernel", cudaGetLastError());
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
    CU_AT("tracker_step: launch_pyramid", launch_pyramid(vcur, modes, s, &ctx->launches));
  }
  MARK(1);
  // 2. Feature ctor / xyz_ref of the last frame's features, initial relative pose
  CU_AT("tracker_step: launch_features_prepare",
        launch_features_prepare(cam, nf, d_last_px + 2 * (size_t)f0, t->slots.pt_world + 3 * (size_t)f0, t->slots.ftr_image + f0, d_T_last, nullptr,
                                t->slots.xyz + 3 * (size_t)f0, s2, &ctx->launches));
  init_pose_kernel<<<(cnt + 127) / 128, 128, 0, s2>>>(cnt, d_T_last + 7 * (size_t)c0, t->slots.T_init + 7 * (size_t)c0); ++ctx->launches;
  CU_AT("tracker_step: init_pose_kernel", cudaGetLastError());
  if (fork) { CU(cudaEventRecord(t->fork_ev[1], s2)); CU(cudaStreamWaitEvent(s, t->fork_ev[1], 0)); }
  MARK(2);
  // 3. SparseImgAlign::run(last, cur)
  CU_AT("tracker_step: launch_sparse_align",
        launch_sparse_align(vlast, vcur, cam, cnt, t->N, t->max_per, t->slots.ftr_off + c0, d_last_px, t->slots.xyz, t->slots.has_point,
                            t->slots.T_init + 7 * (size_t)c0, t->aopts, t->slots.align + c0, t->slots.align_scratch, s, &ctx->launches,
                            d_T_last + 7 * (size_t)c0, t->slots.T_cur + 7 * (size_t)c0));
  MARK(3);
  // 4. cur.T_f_w = T_cur_from_ref * last.T_f_w (written by the alignment kernel's epilogue) ; reprojection of the map points
  // chain mode: the depth filter waits for the pose optimiser's T_cur, so its branch cannot start here
  cudaStream_t s_seeds = (fork && t->chain_cell <= 0) ? s2 : s;
  if (s_seeds != s) { CU(cudaEventRecord(t->fork_ev[2], s)); CU(cudaStreamWaitEvent(s_seeds, t->fork_ev[2], 0)); }
  if (t->chain_cell <= 0 && nf > 0) {
    // Point::getCloseViewObs per map point + px = cur.w2c(pos), depth_ref, T_cur_ref (the head of findMatchDirect)
    points_select_kernel<<<(nf + 127) / 128, 128, 0, s>>>(cam, nf, t->slots.points + f0, t->slots.pobs, t->slots.T_pobs, t->slots.ftr_image + f0, t->slots.T_cur,
                                                          t->slots.ftrs + f0, t->slots.depth_ref + f0, t->slots.px_in + 2 * (size_t)f0, t->slots.active + f0, t->slots.sel + f0);
    ++ctx->launches;
    CU_AT("tracker_step: points_select_kernel", cudaGetLastError());
  }
  MARK(4);
  if (t->chain_cell > 0) {
    // 4b-5. chain mode: Reprojector::reprojectMap (grid, every in-frame candidate matched in parallel, per-cell first success,
    // maxFts) over the keyframe's map points, then pose_optimizer::optimizeGaussNewton on the frame's new features (in place
    // on T_cur, so the depth filter sees the optimised pose).
    const size_t cb = (size_t)c0 * t->chain.n_cells;
    CU_AT("tracker_step: launch_reproject_map",
          launch_reproject_map(ctx->d_table, cur->slot, cam, cnt, t->slots.T_cur + 7 * (size_t)c0, t->slots.ftr_off + c0, t->N, t->slots.points, t->slots.pobs,
                               t->slots.T_pobs, t->chain_cell, t->chain_max_fts, t->mopts, t->chain.reproj, t->chain.winner + cb, t->chain.rstats + c0,
                               t->chain.reproj_scratch, t->slots.match_scratch, t->chain.m_f + 3 * cb, t->chain.m_level + cb, t->chain.m_pos + 3 * cb,
                               t->chain.m_point + cb, t->chain.m_count + c0, s, &ctx->launches, c0, f0, nf));
    MARK(5); MARK(6);
    chain_export_kernel<<<(nf + 127) / 128, 128, 0, s>>>(nf, t->chain.reproj + f0, t->slots.px_out + 2 * (size_t)f0, t->slots.match_ok + f0); ++ctx->launches;
    CU_AT("tracker_step: chain_export_kernel", cudaGetLastError());
    if (t->chain_pose_opt) {
      chain_segments_kernel<<<(cnt + 127) / 128, 128, 0, s>>>(cnt, t->chain.n_cells, t->chain.m_count + c0, t->chain.seg_begin + c0, t->chain.seg_end + c0); ++ctx->launches;
      CU_AT("tracker_step: chain_segments_kernel", cudaGetLastError());
      // segments are relative to this range's slice of the compacted arrays
      CU_AT("tracker_step: launch_pose_optimize",
            launch_pose_optimize(cam, cnt, t->chain.seg_begin + c0, t->chain.seg_end + c0, t->chain.m_f + 3 * cb, t->chain.m_level + cb, t->chain.m_pos + 3 * cb, 2.0, 10,
                                 0.0000000001, 8.6851f, t->slots.T_cur + 7 * (size_t)c0, t->chain.pose + c0, t->chain.outlier + cb, t->chain.pose_work + cb, s, &ctx->launches));
    }
    MARK(7);
  } else {
  // 5. Matcher::findMatchDirect per map point (keyframe patch -> current frame)
  // (item indices inside the call are relative to f0, so the output arrays are passed at f0 as well)
  CU_AT("tracker_step: launch_match_direct",
        launch_match_direct(ctx->d_table, cur->slot, cam, nf, t->slots.ftrs + f0, t->slots.depth_ref + f0, t->slots.px_in + 2 * (size_t)f0, t->mopts, nullptr,
                            t->slots.px_out + 2 * (size_t)f0, t->slots.match_ok + f0, t->slots.match_scratch, t->N, f0, s, &ctx->launches,
                            (marks && t->profiling) ? &t->ev[5] : nullptr, t->slots.active + f0, t->slots.match_level + f0, t->slots.match_A + 4 * (size_t)f0));
  MARK(7);
  }
  if (out_px) CU(cudaMemcpyAsync(out_px + 2 * (size_t)f0, t->slots.px_out + 2 * (size_t)f0, sizeof(double) * 2 * (size_t)nf, cudaMemcpyDeviceToDevice, s));
  if (out_ok) CU(cudaMemcpyAsync(out_ok + f0, t->slots.match_ok + f0, sizeof(int) * (size_t)nf, cudaMemcpyDeviceToDevice, s));
  // 6. DepthFilter::updateSeeds(cur): this range's rows of the pose table (from the step's final T_cur), then the seeds
  CU_AT("tracker_step: launch_seed_pose_table",
        launch_seed_pose_table(cam, t->batch, t->n_kfs, c0, cnt, t->slots.T_kf, t->slots.T_cur, sh.pose_table, s_seeds, &ctx->launches));
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
  if (t->slots.mem.empty()) return fail(ctx, SVOB200_ERR_ARG, "tracker_step: set_keyframe first");
  const int B = t->batch, N = t->N;
  cudaStream_t s = ctx->stream;
  const size_t in_bytes = sizeof(double) * (7 * (size_t)B + 2 * (size_t)N);
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
    const RangeShape shape = {use_graph ? t->fork_stream : s, df_on_stream, (df_on_stream && par) ? t->slots.seed_poses2 : t->slots.seed_poses,
                              (df_on_stream && par) ? t->slots.stats2 : t->slots.stats};
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
    if (int e = frame_own_level0(ctx, r)) return e;           // drop an earlier device binding
    const size_t out_bytes = sizeof(svob200_step_stats) * B + sizeof(double) * 2 * (size_t)N + sizeof(int) * (size_t)N;
    if (t->h_cap < in_bytes + out_bytes + 512) {
      if (t->h_pinned) cudaFreeHost(t->h_pinned);
      t->h_pinned = nullptr; t->h_cap = 0;
      CU(cudaMallocHost((void**)&t->h_pinned, in_bytes + out_bytes + 512));
      t->h_cap = in_bytes + out_bytes + 512;
    }
    const double* d_T_last = t->slots.step_in;
    const double* d_last_px = t->slots.step_in + 7 * (size_t)B;
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
        CU(cudaMemcpyAsync(t->slots.step_in, T_last_w, sizeof(double) * 7 * B, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(t->slots.step_in + 7 * (size_t)B, last_px, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, s));
      } else {
        memcpy(t->h_pinned, T_last_w, sizeof(double) * 7 * B);
        memcpy(t->h_pinned + sizeof(double) * 7 * B, last_px, sizeof(double) * 2 * (size_t)N);
        CU(cudaMemcpyAsync(t->slots.step_in, t->h_pinned, in_bytes, cudaMemcpyHostToDevice, s));
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
    const RangeShape shape = {use_graph ? t->fork_stream : s, false, t->slots.seed_poses, t->slots.stats};
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
    if (stats) CU(cudaMemcpyAsync(h_stats, t->slots.stats, sizeof(svob200_step_stats) * B, cudaMemcpyDeviceToHost, s));
    if (px_refined) CU(cudaMemcpyAsync(h_px, t->slots.px_out, sizeof(double) * 2 * (size_t)N, cudaMemcpyDeviceToHost, s));
    if (match_ok) CU(cudaMemcpyAsync(h_ok, t->slots.match_ok, sizeof(int) * (size_t)N, cudaMemcpyDeviceToHost, s));
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
  CU(cudaMemcpyAsync(out, t->slots.seeds, sizeof(svob200_seed) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

int svob200_tracker_launches_per_step(void) { return 14; }

// raw svob200_align_result records of the most recent step (diagnostics: tools/align_timing.py)
int svob200_tracker_debug_align(svob200_tracker* t, svob200_align_result* out)
{
  if (!t || !out || t->slots.mem.empty()) return SVOB200_ERR_ARG;
  svob200_ctx* ctx = t->ctx;
  CU(cudaMemcpyAsync(out, t->slots.align, sizeof(svob200_align_result) * (size_t)t->batch, cudaMemcpyDeviceToHost, ctx->stream));
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
  CU(cudaMemcpyAsync(out, t->slots.obs, sizeof(svob200_seed_obs) * (size_t)t->S, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

}  // extern "C"
