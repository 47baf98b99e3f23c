// sparse_align.cu — inverse-compositional sparse image alignment over 4x4 patches.
//
// reference: SparseImgAlign::run / precomputeReferencePatches / computeResiduals / solve / update
// (sparse_img_align.cpp:51-308) driven by vk::NLLSSolver<6,SE3>::optimizeGaussNewton
// (nlls_solver_impl.hpp:25-100), SE3::exp (SE3.h:153-182), Frame::jacobian_xyz2uv (frame.h:110-132).
//
// B200 design: the whole run() — every pyramid level, every Gauss-Newton iteration, the 6x6
// solve, the SE3 update and the solver's convergence / rollback logic — is ONE kernel launch with
// one CTA (or, for a handful of sequences, one thread-block cluster) per alignment problem.  A GN iteration is a
// dependency chain, not a bandwidth problem, so the design minimises round trips: the model lives in shared memory; each
// iteration is ONE thread-per-feature pass (projection, the 5x5 window under the patch from ten aligned word loads, 16
// bilinear residuals, J^T r from two patch sums — the 16 Jacobian rows of a patch are dx*a + dy*b with the same a, b), a
// transposing shuffle reduction per warp and one shared-memory pass, and thread 0 solves and decides.  The Hessian is a
// constant of the level as long as the same features contribute (inverse compositional): it is summed and factorised again
// only when a block-wide vote says the set changed; the other iterations reduce 8 sums and do a substitution.
//
// Parity: per-residual arithmetic (bilinear weights with their double promotions, unfused float
// sums, Jacobian rows) is bit-identical to the reference.  H/Jres are summed in double in a
// different order (tolerance-matched).  The rollback test `new_chi2 > chi2_` hangs on a float sum
// accumulated sequentially in the reference; it is decided here on the double sum unless the two
// values are closer than the worst-case rounding error of the float chain, in which case the CTA
// replays the exact sequential float chain in parallel (counted in n_exact_chi2).
#include <cooperative_groups.h>
#include "common.cuh"
#include "kernels.h"
#include "ldlt.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int JAB = 15;

struct AlignArgs {
  DevFrame ref, cur;
  DevCam cam;
  const int* offsets;
  const double* px;
  const double* xyz;
  const uint8_t* has_point;
  const double* T_init;
  const double* T_ref_w;   // optional (tracker): pose of the reference frames, 7 per problem ...
  double* T_cur_w;         // ... and where T_cur_ref * T_ref_w goes (frame_handler_mono.cpp:186-188: cur.T_f_w_ = T_cur_from_ref * last.T_f_w_)
  svob200_align_opts opts;
  svob200_align_result* results;
  // scratch, indexed by global feature / feature-pixel
  float* ref_patch;   // 16 per feature, persists across levels (sparse_img_align.cpp:66)
  float* gdx;         // 16 per feature: image gradient of the reference patch (zero when the feature is
  float* gdy;         //                 outside the level's border => zero Jacobian, :76)
  float* res[2];      // residuals of the last two evaluations (ping-pong), for the exact chi2 chain
  double* jab;        // JAB per feature: a = J0*fl, b = J1*fl (pixel Jacobian row = dx*a + dy*b), then sum dx^2, sum dx*dy, sum dy^2 of the patch
  uint8_t* visible;   // sticky across levels (:67)
  uint8_t* contrib[2];
};

// The 6x6 solve is ldlt_factor_rcp<6> + ldlt_subst_rcp<6> (ldlt.cuh): Eigen's pivoted LDL^T with the exact associations of its
// fixed-size triangular solves, fully unrolled so the matrix lives in thread 0's registers; the factor stays in shared memory
// and is re-used while the Hessian does not change (see the kernel).  (A warp-cooperative version with the
// matrix in shared memory — five swap lanes, parallel column updates, the four libm calls of SE3::exp on four lanes — was
// measured with tools/align_timing.py: 9.3 k cycles per solve against 6.2 k for this one; the shared-memory round trips and
// warp barriers of a 6x6 problem cost more than the serial FP64 chain they replace.)
// The reference's `float chi2; chi2 += res*res*weight` in feature-list / row-major pixel order.  The chain of float
// additions is inherently sequential (4 cycles per FADD); everything around it is not: the whole CTA fetches the
// residuals of a chunk of features (coalesced, L2: the other CTAs of a cluster wrote some of them), squares them
// (res*res*1.0f, the reference's float term) into shared memory, and thread 0 only adds.  Bit-identical to the
// single-thread loop it replaces, at ~64 cycles per contributing feature instead of ~150-200.
constexpr int CHAIN_F = 128;            // features per staged chunk (8 KB of squares)

__device__ void exact_chi2_chain_block(const float* res, const uint8_t* visible, const uint8_t* contrib, int N, float* s_sq, uint8_t* s_fl,
                                       float* out_sum, int* out_cnt, int tid, int nthreads)
{
  float chi2 = 0.0f;
  int cnt = 0;
  for (int c0 = 0; c0 < N; c0 += CHAIN_F) {
    const int m = min(CHAIN_F, N - c0);
    for (int k = tid; k < m; k += nthreads) s_fl[k] = (__ldcg(visible + c0 + k) && __ldcg(contrib + c0 + k)) ? 1 : 0;
    const float4* src = reinterpret_cast<const float4*>(res + 16 * (size_t)c0);
    for (int k = tid; k < m * 4; k += nthreads) {
      const float4 a = __ldcg(src + k);
      reinterpret_cast<float4*>(s_sq)[k] = make_float4(a.x * a.x * 1.0f, a.y * a.y * 1.0f, a.z * a.z * 1.0f, a.w * a.w * 1.0f);
    }
    __syncthreads();
    if (tid == 0) {
      for (int f = 0; f < m; ++f) {
        if (!s_fl[f]) continue;
        const float4* p = reinterpret_cast<const float4*>(s_sq + 16 * f);
        const float4 a = p[0], b = p[1], c = p[2], d = p[3];
        chi2 += a.x; chi2 += a.y; chi2 += a.z; chi2 += a.w;
        chi2 += b.x; chi2 += b.y; chi2 += b.z; chi2 += b.w;
        chi2 += c.x; chi2 += c.y; chi2 += c.z; chi2 += c.w;
        chi2 += d.x; chi2 += d.y; chi2 += d.z; chi2 += d.w;
        cnt += 16;
      }
    }
    __syncthreads();
  }
  if (tid == 0) { *out_sum = chi2; *out_cnt = cnt; }
}

// The same chain, EXACT and parallel.  Inside one binade [2^e, 2^(e+1)) the running sum is M*q with q = 2^(e-23) and M an
// integer in [2^23, 2^24), and a round-to-nearest addition of t >= 0 is M += round_half_even(t/q) as long as the result
// stays below 2^24: every term then contributes an integer that does not depend on M — except exact ties (fraction 1/2,
// probability 2^-d for a term d binades below the sum), which look at the parity of M, and the term that crosses into the
// next binade, which rounds with the doubled quantum.  So: stage a chunk of 2,048 squared residuals (the next chunk's loads
// are already in flight), convert each to its integer contribution in parallel (t/q is an exact float: floorf and the
// fraction are exact too; all of this is FP32 / INT32), take a block-wide prefix sum, find the first "special" term (tie or
// crossing) together with the integer sum just before it in ONE 64-bit shared-memory minimum, jump the sum there (an integer
// below 2^24 times q: exact), apply that one term with a real float addition, and repeat from the term after it in the new
// binade.  Two block barriers per round, one per chunk.  The first HEAD terms, where the sum is a few terms large and
// every other addition is a tie or a crossing, are added by one thread: 256 in the latency-mode (cluster) kernels; the whole
// first chunk in the batch kernels, where a round costs the SM ~1,000 warp instructions that its other resident CTAs could
// use and one thread adding costs 1 per term (measured: 4,096 C2 problems 0.80 ms with the sequential head, 0.85 ms with the
// short one).  NBUF = 2 double-buffers the staged squares (one barrier less per chunk).  Bit-identical to the sequential chain
// (tests/test_gpu_parity.py::test_exact_chi2_chain_parallel_property drives it with adversarial data: ties, binade
// crossings, zeros, huge and non-finite terms, sums that stay tiny).
constexpr int CHAIN_TERMS = CHAIN_F * 16;
constexpr int CHAIN_HEAD_LATENCY = 256;   // terms added sequentially at the start of the chain (latency mode)
constexpr int CHAIN_MAX_ROUNDS = 40;      // per chunk; a chunk that needs more (adversarial data) is finished sequentially
template <int NBUF>
struct ChainSmem {
  __align__(16) float sq[NBUF][CHAIN_TERMS]; // squares of the staged chunk
  uint8_t fl[CHAIN_F];                    // (the sequential replay's feature flags)
  int wsum[2][16];                        // per-warp totals (double-buffered across rounds)
  unsigned long long key[2];              // min over (first special term << 32 | integer sum before it)
  float val;
  int cnt;
};

template <int NT, int HEAD, int NBUF>
__device__ void exact_chi2_chain_parallel(const float* res, const uint8_t* visible, const uint8_t* contrib, int N, ChainSmem<NBUF>* S,
                                          float* out_sum, int* out_cnt, int tid)
{
  constexpr int TPT = CHAIN_TERMS / NT;            // consecutive terms per thread
  constexpr int F4 = CHAIN_F * 4 / NT;             // float4 loads per thread and chunk
  constexpr int SAT = 1 << 25;                     // prefix sums saturate here (anything >= 2^24 only says "crossed")
  const int lane = tid & 31, warp = tid >> 5;
  float s = 0.0f;                                  // uniform over the block
  int cnt = 0;
  int par = 0;                                     // round parity (wsum / key buffers)
  float4 pre[F4];
  bool pre_on[F4];
  auto fetch = [&](int c0) {
    const int m = min(CHAIN_F, N - c0);
    const float4* src = reinterpret_cast<const float4*>(res + 16 * (size_t)c0);
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      const int k = tid + j * NT, f = k >> 2;
      pre_on[j] = f < m && __ldcg(visible + c0 + f) && __ldcg(contrib + c0 + f);
      pre[j] = f < m ? __ldcg(src + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  fetch(0);
  int buf = 0;
  for (int c0 = 0; c0 < N; c0 += CHAIN_F, buf ^= NBUF - 1) {
    float* sq = S->sq[buf];
    if (NBUF == 1 && c0 > 0) __syncthreads();     // the previous chunk's last reads
#pragma unroll
    for (int j = 0; j < F4; ++j) {
      // a feature that does not contribute adds +0: the sum is unchanged
      const float4 a = pre[j];
      reinterpret_cast<float4*>(sq)[tid + j * NT] = pre_on[j] ? make_float4(a.x * a.x * 1.0f, a.y * a.y * 1.0f, a.z * a.z * 1.0f, a.w * a.w * 1.0f)
                                                               : make_float4(0.f, 0.f, 0.f, 0.f);
      cnt += pre_on[j] ? 4 : 0;
    }
    __syncthreads();
    if (c0 + CHAIN_F < N) fetch(c0 + CHAIN_F);     // in flight during this chunk's rounds
    const int mterms = 16 * min(CHAIN_F, N - c0);  // terms past this are zero
    int pos = 0, rounds = 0;
    bool seq = c0 == 0;                            // the head of the chain
    int seq_end = min(HEAD, mterms);
    while (pos < mterms) {
      const int E = (__float_as_int(s) >> 23) & 255;
      if (!seq && (E < 32 || E > 250 || ++rounds > CHAIN_MAX_ROUNDS)) { seq = true; seq_end = mterms; }   // tiny / non-finite sum, pathological chunk
      if (seq) {
        if (tid == 0) { float a = s; for (int k = pos; k < seq_end; ++k) a += sq[k]; S->val = a; }
        __syncthreads();
        s = S->val;
        __syncthreads();
        pos = seq_end; seq = false;
        continue;
      }
      const float inv_q = __int_as_float((277 - E) << 23);             // 2^(150 - E)
      const float q = __int_as_float((E - 23) << 23);                   // 2^(E - 150) = ulp(s)
      const int M0 = (int)(s * inv_q);                                  // integer in [2^23, 2^24)
      int c[TPT];
      unsigned tie_mask = 0;
      int mine = 0;
#pragma unroll
      for (int j4 = 0; j4 < TPT / 4; ++j4) {
        const float4 t4 = reinterpret_cast<const float4*>(sq)[tid * (TPT / 4) + j4];
        const float t[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = 4 * j4 + i, k = tid * TPT + j;
          const float r = t[i] * inv_q;                                  // exact (power of two), or inf / NaN / below 2^-126
          const float a = floorf(r), f = r - a;                          // exact
          int cj = (int)a + (f > 0.5f ? 1 : 0);
          if (!(r < 16777216.0f)) cj = 1 << 24;                          // crosses for sure (also inf / NaN)
          if (k < pos) cj = 0;
          else if (f == 0.5f) tie_mask |= 1u << j;
          c[j] = cj;
          mine += cj;
        }
      }
      mine = min(mine, SAT);
      // block-wide exclusive prefix of the per-thread sums (exact below 2^24, saturating above)
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl = min(incl + v, SAT); }
      if (lane == 31) S->wsum[par][warp] = incl;
      if (tid == 0) S->key[par] = ~0ull;
      __syncthreads();
      int base = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) base = 0;
#pragma unroll
      for (int w = 0; w < NT / 32; ++w) base += w < warp ? S->wsum[par][w] : 0;
      base = min(base, SAT);
      // first special term of this thread (a tie, or the first term whose inclusive prefix reaches 2^24) and the sum before it
      int kspec = CHAIN_TERMS, before = 0;
      int run = base;
#pragma unroll
      for (int j = 0; j < TPT; ++j) {
        const int prev = run;
        run += c[j];
        if (kspec == CHAIN_TERMS && (((tie_mask >> j) & 1u) || M0 + run >= (1 << 24))) { kspec = tid * TPT + j; before = prev; }
      }
      if (kspec < CHAIN_TERMS) atomicMin(&S->key[par], ((unsigned long long)kspec << 32) | (unsigned)(M0 + before));
      else if (tid == NT - 1) atomicMin(&S->key[par], ((unsigned long long)CHAIN_TERMS << 32) | (unsigned)(M0 + run));   // no special at all: the total
      __syncthreads();
      const unsigned long long key = S->key[par];
      const int ks = (int)(key >> 32);             // first special term of the block (CHAIN_TERMS: none)
      s = (float)(int)(unsigned)key * q;            // the sum just before it: an integer below 2^24 times q, exact
      if (ks < CHAIN_TERMS) s = s + sq[ks];         // the special term: one real float addition (every thread, same value)
      pos = ks + 1;
      par ^= 1;
    }
  }
  // the count of contributing pixels
  cnt = warp_sum_i(cnt);
  __syncthreads();
  if (tid == 0) S->cnt = 0;
  __syncthreads();
  if (lane == 0 && cnt) atomicAdd(&S->cnt, cnt);
  __syncthreads();
  if (tid == 0) { *out_sum = s; *out_cnt = S->cnt; }
  __syncthreads();
}

#ifndef ALIGN_TIMING_PROBE
#define ALIGN_TIMING_PROBE 7      // the worker thread whose sub-phase clocks the timing build reports (a feature visible at every level)
#endif
constexpr int NACC = 32;   // 21 (H upper) + 6 (J*res) + chi2 + n_meas + 3 pad
// resident CTAs per SM of the 128-thread batch kernel: 4 (128 registers); 5 / 6 (96 / 80 registers, 1.5 / 2.5 KB of spills per
// thread) measured 0.91 / 0.98 ms against 0.82 ms per 4,096 problems
#ifndef ALIGN_CTAS_128
#define ALIGN_CTAS_128 4
#endif

// After this, lane L of the warp holds the warp-wide sum of v[L]  (31 shuffles instead of 160).
__device__ __forceinline__ double warp_transpose_reduce(double (&v)[NACC], int lane)
{
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int j = 0; j < half; ++j) {
      const double send = up ? v[j] : v[j + half];
      const double keep = up ? v[j + half] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];
}

// Entries 0..7 of an 8-entry accumulator: lane L of the warp ends with the warp-wide sum of v[L & 7], added in the SAME tree
// as warp_transpose_reduce adds any one of its entries (partners 16, 8, 4, 2, 1 lanes away, in that order; IEEE addition is
// commutative, so which partner "keeps" does not matter) — bit-identical to entries 21..28 of the 32-entry reduction.
__device__ __forceinline__ double warp_transpose_reduce8(double (&v)[8], int lane)
{
#pragma unroll
  for (int half = 16; half >= 8; half >>= 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += __shfl_xor_sync(0xffffffffu, v[j], half);
  }
#pragma unroll
  for (int half = 4; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int j = 0; j < half; ++j) {
      const double send = up ? v[j] : v[j + half];
      const double keep = up ? v[j + half] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];
}

// entry h of the packed upper triangle (row-major, 21 entries) into both halves of the full 6x6 matrix
__device__ __forceinline__ void store_h_entry(double* H, int h, double t)
{
  int r = 0, base = 0;
  for (int len = 6; h >= base + len; base += len, --len) ++r;
  const int c = r + (h - base);
  H[r * 6 + c] = t;
  H[c * 6 + r] = t;
}

// One CTA per alignment problem.  Every Gauss-Newton iteration is ONE data-parallel pass with a thread per feature:
//   project xyz_ref with the current model (double), bounds test; fetch the 5x5 window of the current image under the
//   4x4 patch once (10 aligned word loads instead of 64 byte loads); 16 bilinear residuals (float, bit-identical to the
//   reference); the 16 pixel Jacobian rows of a feature are dx*a + dy*b with the SAME two 6-vectors a, b, so
//   sum J J^T = Sxx aa^T + Sxy (ab^T + ba^T) + Syy bb^T and sum J r = Sxr a + Syr b : five double sums, then 27 entries
// followed by one block reduction and the serial solve / update / decision on thread 0.
//
// CLUSTER > 1 (single-stream latency): one thread-block CLUSTER per problem.  Each CTA of the cluster owns a contiguous
// slice of the features and runs P1-P3 on it on its own SM; the 29 partial sums travel to rank 0 through distributed
// shared memory, rank 0 adds them in rank order (deterministic), solves, decides, and pushes the new model and the
// control word into every CTA's shared memory; two hardware cluster barriers per iteration.
template <int BLOCK, int CLUSTER>
__global__ void __launch_bounds__(BLOCK, CLUSTER > 1 ? 1 : (BLOCK == 128 ? ALIGN_CTAS_128 : 512 / BLOCK)) sparse_align_kernel(AlignArgs A)
{
  constexpr int NW = BLOCK / 32;
  __shared__ double s_model[7];
  __shared__ double s_old[7];
  __shared__ double s_red[NW][NACC];
  __shared__ double s_tot[NACC];
  __shared__ double s_clu[CLUSTER > 1 ? CLUSTER : 1][NACC];   // rank 0 only: the partial sums of every CTA of the cluster
  __shared__ int s_ctrl;          // 0 continue iterating, 1 leave this level
  __shared__ double s_H[36], s_Jx[12];   // H_, Jres_, x_ of the last linearisation (copied to the result record once, at the end)
  __shared__ LdltFactor<6> s_fac;        // the LDL^T factor of s_H (re-used while H_ stays the same)
  __shared__ int s_iters[SVOB200_MAX_LEVELS], s_nmeas;
  __shared__ int s_need;          // exact chi2 replay wanted: bit 0 this evaluation, bit 1 the previous one as well
  __shared__ float s_chain[2];
  __shared__ int s_chain_n[2];
  constexpr int CHAIN_HEAD = CLUSTER > 1 ? CHAIN_HEAD_LATENCY : CHAIN_TERMS;
  constexpr int CHAIN_NBUF = (CLUSTER == 1 && BLOCK == 128) ? 1 : 2;       // <= 128 features per problem there: one chunk
  __shared__ ChainSmem<CHAIN_NBUF> s_chainmem;

  const int b = CLUSTER > 1 ? blockIdx.x / CLUSTER : blockIdx.x;
  const int rank = CLUSTER > 1 ? (int)(blockIdx.x % CLUSTER) : 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int f0 = A.offsets[b], N = A.offsets[b + 1] - f0;
  // this CTA's slice of the features
  const int lo = CLUSTER > 1 ? (int)(((long long)N * rank) / CLUSTER) : 0;
  const int hi = CLUSTER > 1 ? (int)(((long long)N * (rank + 1)) / CLUSTER) : N;
  svob200_align_result* R = &A.results[b];
  const bool lead = rank == 0 && tid == 0;

  if (tid < 7) s_model[tid] = A.T_init[7 * b + tid];
  if (lead) {
    for (int k = 0; k < 7; ++k) R->T_cur_ref[k] = A.T_init[7 * b + k];
    for (int k = 0; k < 36; ++k) { R->H[k] = 0; s_H[k] = 0; }
    for (int k = 0; k < 6; ++k) { R->Jres[k] = 0; R->x[k] = 0; s_Jx[k] = 0; s_Jx[6 + k] = 0; }
    R->chi2 = 1e10; R->n_meas = 0; R->stop = 0; R->n_exact_chi2 = 0; R->n_factorisations = 0; s_nmeas = 0;
    for (int k = 0; k < SVOB200_MAX_LEVELS; ++k) { R->iters[k] = 0; s_iters[k] = 0; }
  }
  if (N <= 0) return;                                   // sparse_img_align.cpp:55-59 (uniform over the cluster)
  for (int i = lo + tid; i < hi; i += BLOCK) { A.visible[f0 + i] = 0; A.contrib[0][f0 + i] = 0; A.contrib[1][f0 + i] = 0; }
  __syncthreads();

  const double* px = A.px + 2 * (size_t)f0;
  const double* xyz = A.xyz + 3 * (size_t)f0;
  const uint8_t* has_point = A.has_point + f0;
  uint8_t* visible = A.visible + f0;
  float* ref_patch = A.ref_patch + 16 * (size_t)f0;
  float* gdx = A.gdx + 16 * (size_t)f0;
  float* gdy = A.gdy + 16 * (size_t)f0;
  double* jab = A.jab + JAB * (size_t)f0;
  const double focal_length = fabs(A.cam.fx);          // errorMultiplier2()

  // thread-0 solver state (NLLSSolver::reset nlls_solver_impl.hpp:299-309)
  double chi2_ = 1e10;
  bool chi2_exact = true;
  bool stop_ = false;
  int n_exact = 0, n_fac = 0;
  int pp = 0;                                          // ping-pong index of the *current* evaluation
#ifdef ALIGN_TIMING
  long long tA = 0, tB = 0, tC = 0, tD = 0, tP = 0, c0 = clock64(), cstart = c0;
  long long tS[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s0 = 0;          // sub-phases of the pass as ONE worker thread sees them
#define TICK(acc) do { const long long c1_ = clock64(); acc += c1_ - c0; c0 = c1_; } while (0)
#define SUBTICK0() do { s0 = clock64(); } while (0)
#define SUBTICK(k, dep) do { if ((dep) == 123456.789) s0 += 1; const long long c1_ = clock64(); tS[k] += c1_ - s0; s0 = c1_; } while (0)
#else
#define TICK(acc) do { } while (0)
#define SUBTICK0() do { } while (0)
#define SUBTICK(k, dep) do { } while (0)
#endif

  for (int level = A.opts.max_level; level >= A.opts.min_level; --level) {
    const float scale = 1.0f / (1 << level);
    // ---------------- precomputeReferencePatches (sparse_img_align.cpp:105-178)
    {
      const uint8_t* img = A.ref.lvl[level] + (size_t)b * A.ref.img_stride[level];
      const int cols = A.ref.w[level], rows = A.ref.h[level], stride = A.ref.pitch[level];
      const double fl = focal_length / (1 << level);
      // thread per feature: the 7x7 window under the 4x4 patch and its central-difference gradients is fetched once
      // (three aligned words per row, all 21 loads in flight together) and every tap reads it from registers
      for (int i = lo + tid; i < hi; i += BLOCK) {
        const float u_ref = (float)(px[2 * i] * (double)scale);
        const float v_ref = (float)(px[2 * i + 1] * (double)scale);
        const int u_i = (int)floorf(u_ref), v_i = (int)floorf(v_ref);
        const bool ok = has_point[i] && !(u_i - 3 < 0 || v_i - 3 < 0 || u_i + 3 >= cols || v_i + 3 >= rows);
        float4* gx4 = reinterpret_cast<float4*>(gdx + 16 * (size_t)i);
        float4* gy4 = reinterpret_cast<float4*>(gdy + 16 * (size_t)i);
        if (!ok) {                                                    // jacobian_cache_.setZero() (:76)
#pragma unroll
          for (int q = 0; q < 4; ++q) { gx4[q] = make_float4(0.f, 0.f, 0.f, 0.f); gy4[q] = make_float4(0.f, 0.f, 0.f, 0.f); }
          jab[JAB * (size_t)i + 12] = 0.0; jab[JAB * (size_t)i + 13] = 0.0; jab[JAB * (size_t)i + 14] = 0.0;   // the sums of a zero gradient
          continue;
        }
        visible[i] = 1;
        {
          // Frame::jacobian_xyz2uv (frame.h:110-132), scaled by focal_length / 2^level
          const double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
          const double z_inv = 1. / z, z_inv_2 = z_inv * z_inv;
          const double j02 = x * z_inv_2, j03 = y * j02, j12 = y * z_inv_2;
          double* ja = jab + JAB * (size_t)i;
          ja[0] = -z_inv * fl; ja[1] = 0.0; ja[2] = j02 * fl; ja[3] = j03 * fl; ja[4] = -(1.0 + x * j02) * fl; ja[5] = y * z_inv * fl;
          ja[6] = 0.0; ja[7] = -z_inv * fl; ja[8] = j12 * fl; ja[9] = (1.0 + y * j12) * fl; ja[10] = -j03 * fl; ja[11] = -x * z_inv * fl;
        }
        const float su = u_ref - u_i, sv = v_ref - v_i;
        const float w_tl = (float)((1.0 - su) * (1.0 - sv));
        const float w_tr = (float)(su * (1.0 - sv));
        const float w_bl = (float)((1.0 - su) * sv);
        const float w_br = su * sv;
        // window rows v_i-3 .. v_i+3, columns u_i-3 .. u_i+3 (7 bytes = at most three aligned words per row)
        uint32_t wlo[7], whi[7];
        {
          const uintptr_t a0 = reinterpret_cast<uintptr_t>(img + (size_t)(v_i - 3) * stride + (u_i - 3));
          const unsigned sh = (unsigned)(a0 & 3) * 8;
          const uint8_t* base = reinterpret_cast<const uint8_t*>(a0 & ~(uintptr_t)3);
#pragma unroll
          for (int r = 0; r < 7; ++r) {
            const uint32_t* q = reinterpret_cast<const uint32_t*>(base + (size_t)r * stride);          // stride % 4 == 0
            const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1);
            const uint32_t w2 = sh >= 16 ? __ldg(q + 2) : 0u;        // the third word holds a needed byte only then (never crosses the pitch)
            wlo[r] = __funnelshift_r(w0, w1, sh); whi[r] = __funnelshift_r(w1, w2, sh);
          }
        }
        // pixel (row r, column c) of the window, r and c compile-time after unrolling; window (3,3) is (v_i, u_i)
#define WPX(r, c) byte_to_float((c) < 4 ? wlo[r] : whi[r], (c) & 3)
        float4* rp4 = reinterpret_cast<float4*>(ref_patch + 16 * (size_t)i);
        double Sxx = 0, Sxy = 0, Syy = 0;      // the patch's share of J J^T in the (a, b) basis: constant over the level's iterations
#pragma unroll
        for (int yy = 0; yy < 4; ++yy) {
          float pv[4], xv[4], yv[4];
#pragma unroll
          for (int xx = 0; xx < 4; ++xx) {
            // q = window(yy + 1, xx + 1): q[a + b*stride] = WPX(yy + 1 + b, xx + 1 + a)
            const int r = yy + 1, c = xx + 1;
            pv[xx] = w_tl * WPX(r, c) + w_tr * WPX(r, c + 1) + w_bl * WPX(r + 1, c) + w_br * WPX(r + 1, c + 1);
            xv[xx] = 0.5f * ((w_tl * WPX(r, c + 1) + w_tr * WPX(r, c + 2) + w_bl * WPX(r + 1, c + 1) + w_br * WPX(r + 1, c + 2))
                             - (w_tl * WPX(r, c - 1) + w_tr * WPX(r, c) + w_bl * WPX(r + 1, c - 1) + w_br * WPX(r + 1, c)));
            yv[xx] = 0.5f * ((w_tl * WPX(r + 1, c) + w_tr * WPX(r + 1, c + 1) + w_bl * WPX(r + 2, c) + w_br * WPX(r + 2, c + 1))
                             - (w_tl * WPX(r - 1, c) + w_tr * WPX(r - 1, c + 1) + w_bl * WPX(r, c) + w_br * WPX(r, c + 1)));
            const double X = (double)xv[xx], Y = (double)yv[xx];
            Sxx += X * X; Sxy += X * Y; Syy += Y * Y;
          }
          rp4[yy] = make_float4(pv[0], pv[1], pv[2], pv[3]);
          gx4[yy] = make_float4(xv[0], xv[1], xv[2], xv[3]);
          gy4[yy] = make_float4(yv[0], yv[1], yv[2], yv[3]);
        }
        jab[JAB * (size_t)i + 12] = Sxx; jab[JAB * (size_t)i + 13] = Sxy; jab[JAB * (size_t)i + 14] = Syy;
#undef WPX
      }
    }
    if (tid < 7) s_old[tid] = s_model[tid];
    __syncthreads();
    TICK(tP);

    const uint8_t* cimg = A.cur.lvl[level] + (size_t)b * A.cur.img_stride[level];
    const int ccols = A.cur.w[level], crows = A.cur.h[level], cstride = A.cur.pitch[level];

    for (int iter = 0; iter < A.opts.n_iter; ++iter) {
      float* res = A.res[pp] + 16 * (size_t)f0;
      uint8_t* contrib = A.contrib[pp] + f0;
      // ---------------- one pass, thread per feature (sparse_img_align.cpp:219-266 + the normal equations):
      //   project with the current model (double) -> bounds test -> the 5x5 window of the current image that the 4x4
      //   patch's bilinear taps touch (two aligned words per row) -> 16 residuals (float, the reference's expression and
      //   order per pixel) -> J^T r.  Nothing but `res` / `contrib` (needed by the exact chi2 replay) goes back to memory.
      // The alignment is inverse compositional: the Jacobian is taken at the reference patch, so a feature's 21 entries of
      // J J^T — Sxx aa^T + Sxy (ab^T + ba^T) + Syy bb^T with the patch sums of precomputeReferencePatches — are the SAME in
      // every iteration of a level, and H_ changes only when the set of features inside the current image does (the reference
      // re-adds the same numbers every iteration, sparse_img_align.cpp:253-262).  So an iteration whose set equals the previous
      // one's (one block-wide vote) reduces 8 sums instead of 29, keeps H_, and the solve re-uses the LDL^T factor: only J^T r,
      // chi2 and the substitution are new.  Bit-identical to recomputing: the sums run over the same features in the same tree.
      double a8[8];                                    // J^T r (6), sum of res^2, pixel count
#pragma unroll
      for (int k = 0; k < 8; ++k) a8[k] = 0.0;
      bool flag = false;                               // an own feature entered or left the image since the last evaluation
      {
        double m[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) m[k] = s_model[k];
        const uint8_t* was = A.contrib[pp ^ 1] + f0;
        for (int i = lo + tid; i < hi; i += BLOCK) {
          SUBTICK0();
          if (!visible[i]) continue;
          const v3d pc = se3_transform(m, {xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]});
          double pxd, pyd;
          world2cam(A.cam, pc, pxd, pyd);
          SUBTICK(0, pxd + pyd);
          const float u_cur = (float)pxd * scale, v_cur = (float)pyd * scale;
          const int u_i = (int)floorf(u_cur), v_i = (int)floorf(v_cur);
          const bool in = !(u_i < 0 || v_i < 0 || u_i - 3 < 0 || v_i - 3 < 0 || u_i + 3 >= ccols || v_i + 3 >= crows);
          if (iter > 0 && (was[i] != 0) != in) flag = true;
          contrib[i] = in ? 1 : 0;
          if (!in) continue;
          const float su = u_cur - u_i, sv = v_cur - v_i;
          const float w_tl = (float)((1.0 - su) * (1.0 - sv));
          const float w_tr = (float)(su * (1.0 - sv));
          const float w_bl = (float)((1.0 - su) * sv);
          const float w_br = su * sv;
          // window rows v_i-2 .. v_i+2, columns u_i-2 .. u_i+2
          float W[5][5];
          {
            const uintptr_t a0 = reinterpret_cast<uintptr_t>(cimg + (size_t)(v_i - 2) * cstride + (u_i - 2));
            const unsigned sh = (unsigned)(a0 & 3) * 8;
            const uint8_t* base = reinterpret_cast<const uint8_t*>(a0 & ~(uintptr_t)3);
#pragma unroll
            for (int r = 0; r < 5; ++r) {
              const uint32_t* q = reinterpret_cast<const uint32_t*>(base + (size_t)r * cstride);      // cstride % 4 == 0
              const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1);
              const uint32_t lo4 = __funnelshift_r(w0, w1, sh), b4 = (w1 >> sh) & 0xffu;
              W[r][0] = byte_to_float(lo4, 0); W[r][1] = byte_to_float(lo4, 1); W[r][2] = byte_to_float(lo4, 2);
              W[r][3] = byte_to_float(lo4, 3); W[r][4] = byte_to_float(b4, 0);
            }
          }
          SUBTICK(1, (double)(W[0][0] + W[1][1] + W[2][2] + W[3][3] + W[4][4]));
          const float4* p4 = reinterpret_cast<const float4*>(ref_patch + 16 * (size_t)i);
          const float4* x4 = reinterpret_cast<const float4*>(gdx + 16 * (size_t)i);
          const float4* y4 = reinterpret_cast<const float4*>(gdy + 16 * (size_t)i);
          float4* r4 = reinterpret_cast<float4*>(res + 16 * (size_t)i);
          double Sxr = 0, Syr = 0, Srr = 0;
#pragma unroll
          for (int yy = 0; yy < 4; ++yy) {
            const float4 rp = p4[yy], dx = x4[yy], dy = y4[yy];
            const float pv[4] = {rp.x, rp.y, rp.z, rp.w}, xv[4] = {dx.x, dx.y, dx.z, dx.w}, yv[4] = {dy.x, dy.y, dy.z, dy.w};
            float rv[4];
#pragma unroll
            for (int xx = 0; xx < 4; ++xx) {
              const float intensity = w_tl * W[yy][xx] + w_tr * W[yy][xx + 1] + w_bl * W[yy + 1][xx] + w_br * W[yy + 1][xx + 1];
              rv[xx] = intensity - pv[xx];
              const double X = (double)xv[xx], Y = (double)yv[xx], Rr = (double)rv[xx];
              Sxr += X * Rr; Syr += Y * Rr;
              Srr += (double)(rv[xx] * rv[xx] * 1.0f);          // the reference's float term res*res*weight
            }
            r4[yy] = make_float4(rv[0], rv[1], rv[2], rv[3]);
          }
          SUBTICK(2, Sxr + Syr + Srr);
          const double* ja = jab + JAB * (size_t)i;
#pragma unroll
          for (int r = 0; r < 6; ++r) a8[r] += Sxr * ja[r] + Syr * ja[6 + r];
          a8[6] += Srr;
          a8[7] += 16.0;
          SUBTICK(3, a8[0] + a8[5]);
        }
      }
      SUBTICK0();
      // does this CTA's share of H_ have to be summed again?  (uniform over the CTA; iter is uniform over the cluster)
      const bool full = iter == 0 || __syncthreads_or(flag ? 1 : 0) != 0;
      SUBTICK(4, 0.0);
      // ---------------- block reduction: lane L of a warp ends with the warp's sum of entry L
      if (full) {
        double acc[NACC];
#pragma unroll
        for (int k = 0; k < NACC; ++k) acc[k] = 0.0;
        for (int i = lo + tid; i < hi; i += BLOCK) {
          if (!visible[i] || !contrib[i]) continue;     // contrib[i]: this thread's own store of a moment ago
          const double* ja = jab + JAB * (size_t)i;
          double a[6], bb[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) { a[k] = ja[k]; bb[k] = ja[6 + k]; }
          const double Sxx = ja[12], Sxy = ja[13], Syy = ja[14];
          int h = 0;
#pragma unroll
          for (int r = 0; r < 6; ++r) {
#pragma unroll
            for (int c = r; c < 6; ++c) acc[h++] += Sxx * (a[r] * a[c]) + Sxy * (a[r] * bb[c] + bb[r] * a[c]) + Syy * (bb[r] * bb[c]);
          }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[21 + k] = a8[k];
        const double mine = warp_transpose_reduce(acc, lane);
        s_red[warp][lane] = mine;
      } else {
        const double mine = warp_transpose_reduce8(a8, lane);     // the same addition tree as entries 21..28 of the full one
        if (lane < 8) s_red[warp][21 + lane] = mine;
      }
      SUBTICK(5, 0.0);
      __syncthreads();
      SUBTICK(6, 0.0);
      if (warp == 0 && (full || lane >= 21)) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) t += s_red[w][lane];
        if (lane == 29) t = full ? 1.0 : 0.0;          // entry 29 (a pad of the sums): "H_ was summed again"
        if (CLUSTER > 1) cg::this_cluster().map_shared_rank(&s_clu[0][0], 0)[rank * NACC + lane] = t;
        else { s_tot[lane] = t; if (lane < 21) store_h_entry(s_H, lane, t); }
      }
      if (CLUSTER > 1) {
        __threadfence();                               // residuals / flags of this slice: visible to rank 0's exact chi2 replay
        cg::this_cluster().sync();
        if (rank == 0 && warp == 0) {
          // every rank's H_ share is still in its row of s_clu when that rank did not sum it again
          double t = s_clu[0][lane];
#pragma unroll
          for (int r = 1; r < CLUSTER; ++r) t += s_clu[r][lane];
          s_tot[lane] = t;
          if (lane < 21) store_h_entry(s_H, lane, t);
        }
      }
      __syncthreads();
      SUBTICK(7, 0.0);

      TICK(tA);
      // ---------------- solve (thread 0 of rank 0), nlls_solver_impl.hpp:36-99
      double xs[6];
      int n_meas = 0;
      double new_chi2 = 0.0;
      bool new_exact = false;
      if (lead) {
        double Jres[6];
#pragma unroll
        for (int r = 0; r < 6; ++r) Jres[r] = -s_tot[21 + r];
        n_meas = (int)s_tot[28];
        new_chi2 = (double)((float)s_tot[27] / (float)n_meas);
        if (s_tot[29] != 0.0) { ldlt_factor_rcp<6>(s_H, &s_fac); ++n_fac; }     // H_ (warp 0 wrote it out) changed: factor it again
        ldlt_subst_rcp<6>(&s_fac, Jres, xs);
        if (isnan(xs[0])) stop_ = true;
#pragma unroll
        for (int k = 0; k < 6; ++k) { s_Jx[k] = Jres[k]; s_Jx[6 + k] = xs[k]; }
        s_nmeas = n_meas;
        s_iters[level] += 1;
        int need = 0;
        if (iter > 0 && !stop_) {
          // worst-case first-order rounding error of two sequential float sums of n_meas terms
          const double tol = 2.0 * (double)n_meas * 5.9604644775390625e-08;
          const double big = fmax(fabs(new_chi2), fabs(chi2_));
          if (fabs(new_chi2 - chi2_) <= tol * big) need = chi2_exact ? 1 : 3;
        }
        s_need = need;
      }
      TICK(tB);
      // ---------------- exact replay of the reference's float chi2 chain(s), when the decision hangs on it (rank 0's CTA)
      if (rank == 0) {
        __syncthreads();
        const int need = s_need;
#ifdef ALIGN_CHAIN_SERIAL   // A/B builds: one thread adds the staged squares in order
        if (need & 1) exact_chi2_chain_block(res, visible, contrib, N, s_chainmem.sq[0], s_chainmem.fl, &s_chain[0], &s_chain_n[0], tid, BLOCK);
        if (need & 2) exact_chi2_chain_block(A.res[pp ^ 1] + 16 * (size_t)f0, visible, A.contrib[pp ^ 1] + f0, N, s_chainmem.sq[0], s_chainmem.fl, &s_chain[1], &s_chain_n[1], tid, BLOCK);
#else
        if (need & 1) exact_chi2_chain_parallel<BLOCK, CHAIN_HEAD, CHAIN_NBUF>(res, visible, contrib, N, &s_chainmem, &s_chain[0], &s_chain_n[0], tid);
        // the previous evaluation lives in the other ping-pong buffer
        if (need & 2) exact_chi2_chain_parallel<BLOCK, CHAIN_HEAD, CHAIN_NBUF>(A.res[pp ^ 1] + 16 * (size_t)f0, visible, A.contrib[pp ^ 1] + f0, N, &s_chainmem, &s_chain[1], &s_chain_n[1], tid);
#endif
        if (need) __syncthreads();
      }
      TICK(tC);
      // ---------------- decide / update (thread 0 of rank 0)
      if (lead) {
        int ctrl = 0;
        const int need = s_need;
        if (need & 1) {
          ++n_exact;
          new_chi2 = (double)(s_chain[0] / (float)n_meas);
          new_exact = true;
          if (need & 2) { chi2_ = (double)(s_chain[1] / (float)s_chain_n[1]); chi2_exact = true; }
        }
        if ((iter > 0 && new_chi2 > chi2_) || stop_) {
#pragma unroll
          for (int k = 0; k < 7; ++k) s_model[k] = s_old[k];        // rollback
          ctrl = 1;
        } else {
          double nx[6], E[7], nm[7], cm[7];
#pragma unroll
          for (int k = 0; k < 6; ++k) nx[k] = -xs[k];
#pragma unroll
          for (int k = 0; k < 7; ++k) cm[k] = s_model[k];
          se3_exp(nx, E);                                            // update(): T * exp(-x)
          se3_mul(cm, E, nm);
#pragma unroll
          for (int k = 0; k < 7; ++k) { s_old[k] = cm[k]; s_model[k] = nm[k]; }
          chi2_ = new_chi2;
          chi2_exact = new_exact;
          double nmax = 0;
#pragma unroll
          for (int k = 0; k < 6; ++k) nmax = fmax(nmax, fabs(xs[k]));   // vk::norm_max
          if (nmax <= A.opts.eps) ctrl = 1;
        }
        s_ctrl = ctrl;
      }
      pp ^= 1;
      if (CLUSTER > 1) {
        // every other CTA of the cluster PULLS the new model, the rollback model and the control word from rank 0 through
        // distributed shared memory, 15 threads in parallel (rank 0 next writes them after the next iteration's barrier)
        cg::cluster_group cl = cg::this_cluster();
        cl.sync();
        if (rank != 0) {
          if (tid < 7) s_model[tid] = cl.map_shared_rank(&s_model[0], 0)[tid];
          else if (tid < 14) s_old[tid - 7] = cl.map_shared_rank(&s_old[0], 0)[tid - 7];
          else if (tid == 14) s_ctrl = *cl.map_shared_rank(&s_ctrl, 0);
        }
        __syncthreads();
      } else {
        __syncthreads();
      }
      TICK(tD);
      if (s_ctrl) break;
    }
    if (CLUSTER > 1) cg::this_cluster().sync(); else __syncthreads();
  }
  if (lead) {
    for (int k = 0; k < 36; ++k) R->H[k] = s_H[k];
    for (int k = 0; k < 6; ++k) { R->Jres[k] = s_Jx[k]; R->x[k] = s_Jx[6 + k]; }
    R->n_meas = s_nmeas;
    for (int k = 0; k < SVOB200_MAX_LEVELS; ++k) R->iters[k] = s_iters[k];
    for (int k = 0; k < 7; ++k) R->T_cur_ref[k] = s_model[k];
    R->chi2 = chi2_;
    R->stop = stop_ ? 1 : 0;
    R->n_exact_chi2 = n_exact;
    R->n_factorisations = n_fac;
    if (A.T_cur_w) {
      double Tm[7], out[7];
#pragma unroll
      for (int k = 0; k < 7; ++k) Tm[k] = s_model[k];
      se3_mul(Tm, A.T_ref_w + 7 * (size_t)b, out);
#pragma unroll
      for (int k = 0; k < 7; ++k) A.T_cur_w[7 * (size_t)b + k] = out[k];
    }
#ifdef ALIGN_TIMING
    R->H[0] = (double)tP; R->H[1] = (double)tA; R->H[2] = (double)tB; R->H[3] = (double)tC; R->H[4] = (double)tD; R->H[5] = (double)(clock64() - cstart);
#endif
  }
#ifdef ALIGN_TIMING
  __syncthreads();
  if (rank == 0 && tid == ALIGN_TIMING_PROBE) for (int k = 0; k < 8; ++k) R->H[6 + k] = (double)tS[k];
#endif
}

// diagnostics (svob200_debug_chi2_chain): the replays of the float chi2 chain over caller-supplied residuals, one CTA:
// [0] one thread adding, [1] the parallel replay as the latency-mode kernels run it, [2] as the batch kernels run it
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) chi2_chain_test_kernel(const float* res, const uint8_t* visible, const uint8_t* contrib, int N, float* sums, int* cnts)
{
  __shared__ ChainSmem<2> s_chainmem;
  const int tid = threadIdx.x;
  exact_chi2_chain_block(res, visible, contrib, N, s_chainmem.sq[0], s_chainmem.fl, sums + 0, cnts + 0, tid, BLOCK);
  __syncthreads();
  exact_chi2_chain_parallel<BLOCK, CHAIN_HEAD_LATENCY, 2>(res, visible, contrib, N, &s_chainmem, sums + 1, cnts + 1, tid);
  __syncthreads();
  exact_chi2_chain_parallel<BLOCK, CHAIN_TERMS, 1>(res, visible, contrib, N, reinterpret_cast<ChainSmem<1>*>(&s_chainmem), sums + 2, cnts + 2, tid);
}

}  // namespace

int launch_chi2_chain_test(int block, const float* d_res, const uint8_t* d_visible, const uint8_t* d_contrib, int n, float* d_sums, int* d_cnts,
                           cudaStream_t s, long long* launches)
{
  if (block == 128) chi2_chain_test_kernel<128><<<1, 128, 0, s>>>(d_res, d_visible, d_contrib, n, d_sums, d_cnts);
  else if (block == 256) chi2_chain_test_kernel<256><<<1, 256, 0, s>>>(d_res, d_visible, d_contrib, n, d_sums, d_cnts);
  else if (block == 512) chi2_chain_test_kernel<512><<<1, 512, 0, s>>>(d_res, d_visible, d_contrib, n, d_sums, d_cnts);
  else return -1;
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// per feature: 16 floats x (ref_patch, gdx, gdy, res0, res1) + 15 doubles (a, b, patch gradient sums) + 3 flag bytes
size_t sparse_align_scratch_bytes(int total_features)
{
  const size_t n = (size_t)(total_features > 0 ? total_features : 1);
  return n * (16 * sizeof(float) * 5 + JAB * sizeof(double) + 3) + 4096;
}

int launch_sparse_align(const DevFrame& ref, const DevFrame& cur, const DevCam& cam, int batch, int total_features, int max_per_problem,
                        const int* d_offsets, const double* d_px, const double* d_xyz, const uint8_t* d_has_point,
                        const double* d_T_init, svob200_align_opts opts, svob200_align_result* d_results,
                        void* d_scratch, cudaStream_t s, long long* launches, const double* d_T_ref_w, double* d_T_cur_w)
{
  AlignArgs A{};
  A.T_ref_w = d_T_ref_w; A.T_cur_w = d_T_cur_w;
  A.ref = ref; A.cur = cur; A.cam = cam; A.offsets = d_offsets; A.px = d_px; A.xyz = d_xyz; A.has_point = d_has_point;
  A.T_init = d_T_init; A.opts = opts; A.results = d_results;
  // carve the scratch in the order sparse_align_scratch_bytes() counts it (all sub-arrays stay 16-byte aligned)
  const size_t T = (size_t)(total_features > 0 ? total_features : 1);
  char* p = static_cast<char*>(d_scratch);
  auto take = [&p](size_t bytes) { char* q = p; p += (bytes + 255) & ~(size_t)255; return q; };
  const size_t fsz = T * 16 * sizeof(float);
  A.jab = reinterpret_cast<double*>(take(T * JAB * sizeof(double)));
  A.ref_patch = reinterpret_cast<float*>(take(fsz));
  A.gdx = reinterpret_cast<float*>(take(fsz));
  A.gdy = reinterpret_cast<float*>(take(fsz));
  A.res[0] = reinterpret_cast<float*>(take(fsz));
  A.res[1] = reinterpret_cast<float*>(take(fsz));
  A.visible = reinterpret_cast<uint8_t*>(take(T));
  A.contrib[0] = reinterpret_cast<uint8_t*>(take(T));
  A.contrib[1] = reinterpret_cast<uint8_t*>(take(T));
  // few problems (single-stream latency): spread each problem over a thread-block cluster, one SM per CTA, so the
  // per-iteration work of a 1,000-feature frame is shared by 8 SMs instead of serialising on one;
  // small problems / few problems: more threads per problem (latency); big batches: more CTAs per SM (throughput)
  int cluster = 1;
  if (batch <= 16 && max_per_problem >= 64) cluster = 8;
  else if (batch <= 32 && max_per_problem >= 64) cluster = 4;
  else if (batch <= 64 && max_per_problem >= 128) cluster = 2;
  if (cluster > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)batch * cluster, 1, 1); cfg.blockDim = dim3(256, 1, 1); cfg.dynamicSmemBytes = 0; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e;
    if (cluster == 8) e = cudaLaunchKernelEx(&cfg, sparse_align_kernel<256, 8>, A);
    else if (cluster == 4) e = cudaLaunchKernelEx(&cfg, sparse_align_kernel<256, 4>, A);
    else e = cudaLaunchKernelEx(&cfg, sparse_align_kernel<256, 2>, A);
    ++*launches;
    return e == cudaSuccess && cudaGetLastError() == cudaSuccess ? 0 : -1;
  }
  if (max_per_problem > 512) sparse_align_kernel<512, 1><<<batch, 512, 0, s>>>(A);
  else if (max_per_problem > 128 || batch < 296) sparse_align_kernel<256, 1><<<batch, 256, 0, s>>>(A);
  // (64-thread CTAs, two features per thread and twice the problems resident per SM: 0.629 ms per 4,096 problems against 0.619 ms,
  // 0.176 against 0.143 ms per 512 — the pass is bound by its own dependent latency, not by how many problems share the SM)
  else sparse_align_kernel<128, 1><<<batch, 128, 0, s>>>(A);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
