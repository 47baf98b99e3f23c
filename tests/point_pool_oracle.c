/*
 * point_pool_oracle.c — CPU restatement of the tracker's point pool (svob200_tracker_set_point_pool) around the oracle's
 * unchanged sequence step.  TEST INFRASTRUCTURE ONLY: built by tests/point_pool_oracle.py together with the oracle's sources
 * and flags; it includes oracle/svo_cpu_pipeline.c for the sequence state.
 *
 * The reference's loop, per sequence:
 *   DepthFilter::updateSeeds -> seed_converged_cb_ -> MapPointCandidates::newCandidatePoint: a converged seed becomes a
 *     candidate at kf.T_f_w.inverse() * (f * (1.0 / mu)) (depth_filter.cpp:318-325), in list order (ascending batch id, then
 *     seed slot), before any re-seeding;
 *   the candidates of step k take the empty point slots, in slot order, at the head of step k + 2 (the depth filter runs one
 *     frame behind tracking); one whose keyframe left the ring in between, or that finds no empty slot, is dropped;
 *   MapPointCandidates::addCandidatePointToFrame: a candidate matched in a new keyframe gains the observation and becomes a
 *     map point; removeFrameCandidates, after it: the unpromoted candidates of the keyframe that leaves the ring are deleted.
 * The sequence is set up with one point slot per pool entry (its map points, then empty slots); pp_attach empties the slots
 * beyond the map points.
 */
#include "../oracle/svo_cpu_pipeline.c"

typedef struct { double pos[3], px[2], f[3]; int level, kf, batch; } pp_cand;

typedef struct {
  svo_seq* s;
  int *type, *src_kf;                  /* SVO_POINT_* per slot; keyframe index of a candidate */
  pp_cand* cand[2]; int cand_n[2];     /* the candidates of the last two steps, by step parity */
  long long step_no;
  int created, dropped;
} pp_pool;

pp_pool* pp_attach(svo_seq* s, int n_points)
{
  pp_pool* p = (pp_pool*)calloc(1, sizeof(pp_pool));
  p->s = s;
  p->type = (int*)malloc(sizeof(int) * (size_t)(s->N + 1)); p->src_kf = (int*)calloc((size_t)s->N + 1, sizeof(int));
  for (int q = 0; q < 2; ++q) p->cand[q] = (pp_cand*)calloc((size_t)s->N + 1, sizeof(pp_cand));
  for (int i = 0; i < s->N; ++i) {
    p->type[i] = i < n_points ? SVO_POINT_UNKNOWN : SVO_POINT_DELETED;
    if (i >= n_points) { s->has_point[i] = 0; s->pobs_n[i] = 0; memset(s->pt_world + 3 * i, 0, sizeof(double) * 3); }
  }
  return p;
}

void pp_destroy(pp_pool* p)
{
  if (!p) return;
  free(p->type); free(p->src_kf); free(p->cand[0]); free(p->cand[1]); free(p);
}

static void pp_insert(pp_pool* p)
{
  svo_seq* s = p->s;
  const int par = (int)(p->step_no & 1), n = p->cand_n[par], stored = n < s->N ? n : s->N;
  int j = 0, filled = 0;
  for (int c = 0; c < stored; ++c) {
    const pp_cand* cd = &p->cand[par][c];
    if (cd->batch != s->kf_batch[cd->kf]) continue;
    while (j < s->N && p->type[j] != SVO_POINT_DELETED) ++j;
    if (j >= s->N) break;
    const size_t o = (size_t)j * SVO_SEQ_MAX_KFS;
    memcpy(s->pt_world + 3 * j, cd->pos, sizeof(cd->pos));
    p->type[j] = SVO_POINT_CANDIDATE; p->src_kf[j] = cd->kf; s->has_point[j] = 1;
    s->pobs_n[j] = 1; s->pobs_kf[o] = cd->kf; s->pobs_level[o] = cd->level;
    memcpy(s->pobs_px + 2 * o, cd->px, sizeof(cd->px)); memcpy(s->pobs_f + 3 * o, cd->f, sizeof(cd->f));
    ++j; ++filled;
  }
  p->dropped += n - filled;
}

/* one step: insertion, the oracle's step with re-seeding held back, the step's candidates, then the re-seeding rule of
 * svo_oracle_seq_step over the same statuses */
void pp_step(pp_pool* p, const uint8_t* cur_img, const double* T_last_w, const double* last_px, svo_step_stats* st,
             double* px_refined, int* match_ok)
{
  svo_seq* s = p->s;
  pp_insert(p);
  const int reseed = s->reseed;
  s->reseed = 0;
  svo_oracle_seq_step(s, cur_img, T_last_w, last_px, st, px_refined, match_ok);
  s->reseed = reseed;
  pp_cand* conv = (pp_cand*)malloc(sizeof(pp_cand) * (size_t)(s->S + 1));
  int n_conv = 0;
  for (int i = 0; i < s->S; ++i) {
    if (s->obs[i].status != SVO_SEED_CONVERGED) continue;
    pp_cand* cd = &conv[n_conv++];
    const int kfi = s->seed_kf[i];
    double Tinv[7], v[3];
    svo_oracle_se3_inverse(s->T_kfs[kfi], Tinv);
    const double sc = 1.0 / (double)s->seeds[i].mu;
    v[0] = s->seed_f[3 * i] * sc; v[1] = s->seed_f[3 * i + 1] * sc; v[2] = s->seed_f[3 * i + 2] * sc;
    svo_oracle_se3_transform(Tinv, v, cd->pos);
    memcpy(cd->px, s->seed_px + 2 * i, sizeof(cd->px)); memcpy(cd->f, s->seed_f + 3 * i, sizeof(cd->f));
    cd->level = s->seed_level[i]; cd->kf = kfi; cd->batch = s->seed_batch[i];
  }
  /* list order: a stable pass per batch id over the slot-ordered candidates; a step records at most one per point slot */
  const int par = (int)(p->step_no & 1);
  int m = 0, prev = -1;
  for (;;) {
    int bid = -1;
    for (int c = 0; c < n_conv; ++c) if (conv[c].batch > prev && (bid < 0 || conv[c].batch < bid)) bid = conv[c].batch;
    if (bid < 0) break;
    for (int c = 0; c < n_conv; ++c) if (conv[c].batch == bid) { if (m < s->N) p->cand[par][m] = conv[c]; ++m; }
    prev = bid;
  }
  p->cand_n[par] = n_conv; p->created += n_conv;
  free(conv);
  for (int i = 0; i < s->S; ++i) {
    const int status = s->obs[i].status;
    if (status == 0 || status == SVO_SEED_TOO_OLD) continue;          /* empty slot / erased by the ageing rule */
    if (reseed == 3) { if (status == SVO_SEED_CONVERGED || status == SVO_SEED_NAN_ERASED) s->seed_alive[i] = 0; }
    else if (reseed == 2 || (reseed && (status == SVO_SEED_CONVERGED || status == SVO_SEED_NAN_ERASED))) s->seeds[i] = s->seed_init;
  }
  p->step_no++;
}

/* svo_oracle_seq_add_keyframe with the candidates: removal of the leaving keyframe's unpromoted ones first (its observations are
 * dropped by the oracle), promotion of the matched ones after the oracle added their observation */
int pp_add_keyframe(pp_pool* p, float depth_mean, float depth_min)
{
  svo_seq* s = p->s;
  if (s->have_step) {
    int k = -1;
    for (int i = 0; i < s->max_kfs; ++i) if (!s->kf_used[i]) { k = i; break; }
    if (k < 0) {
      k = 0;
      for (int i = 1; i < s->max_kfs; ++i) if (s->kf_batch[i] < s->kf_batch[k]) k = i;
      for (int i = 0; i < s->N; ++i)
        if (p->type[i] == SVO_POINT_CANDIDATE && p->src_kf[i] == k && !s->step_ok[i]) {
          p->type[i] = SVO_POINT_DELETED; s->has_point[i] = 0; s->pobs_n[i] = 0;
        }
    }
  }
  const int n = svo_oracle_seq_add_keyframe(s, depth_mean, depth_min);
  for (int i = 0; i < s->N; ++i) if (p->type[i] == SVO_POINT_CANDIDATE && s->step_ok[i]) p->type[i] = SVO_POINT_UNKNOWN;
  return n;
}

/* per slot: position, SVO_POINT_* type (DELETED: empty slot), observation count; the candidates created / dropped so far.
 * p may be NULL (a sequence without a pool: every slot is a map point). */
void pp_get_points(const svo_seq* s, const pp_pool* p, double* pos, int* type, int* n_obs, int* created, int* dropped)
{
  for (int i = 0; i < s->N; ++i) {
    memcpy(pos + 3 * i, s->pt_world + 3 * i, sizeof(double) * 3);
    type[i] = p ? p->type[i] : SVO_POINT_UNKNOWN; n_obs[i] = s->pobs_n[i];
  }
  *created = p ? p->created : 0; *dropped = p ? p->dropped : 0;
}
