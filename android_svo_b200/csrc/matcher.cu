// matcher.cu — affine patch warp, 2D/1D Lucas-Kanade refinement, epipolar ZMSSD search and the
// depth-filter seed update.
//
// reference: warp::getWarpMatrixAffine / getBestSearchLevel / warpAffine (matcher.cpp:36-116),
// vk::interpolateMat_8u (vision.h:19-36), feature_alignment::align2D / align1D float paths
// (feature_alignment.cpp:35-282), vk::patch_score::ZMSSD<4> (patch_score.h:40-220),
// Matcher::findMatchDirect / findEpipolarMatchDirect (matcher.cpp:156-355),
// depthFromTriangulation (matcher.cpp:123-136), DepthFilter::updateSeeds loop body, updateSeed,
// computeTau (depth_filter.cpp:250-416).
//
// B200 design (deviates from north_star's "block per seed, warp per patch batch", DESIGN.md section 0): GROUPS OF 8 LANES — four
// seeds or four reprojection candidates per warp in lockstep — warp the 10x10 patch into shared memory (13 rounds of 8 taps) and
// walk the epipolar segment (one sample per lane, the 8x8 reference patch in 16 registers, ZMSSD by dp4a on funnel-shifted
// aligned words, the strict-minimum "first wins" rule as a 64-bit min over (score << 32 | step index)); the Lucas-Kanade
// refinement runs THREAD PER PROBLEM on 128-byte job records the groups emit; geometry before and the seed update after are
// thread per seed in double precision.  The search kernel is persistent (SEARCH_CTAS resident CTAs per SM).
//
// Parity: the warp, ZMSSD and the LK iterations are bit-identical to the reference.  The LK sums (H, Jres) are float
// accumulations whose order matters, so they are NOT tree-reduced: each thread replays the reference's sequential loop over its
// own problem.  The epipolar sample positions come from the reference's running sum `uv += step`, replayed by two lanes of the
// group (x and y are independent chains).  Only libm calls (acos/sin/atan/exp) are tolerance-matched — and fed the same pose they
// reproduce the oracle's seeds bit for bit (DESIGN.md section 3).
#include <cuda_fp16.h>
#include "common.cuh"
#include "kernels.h"

namespace {

// ---------------------------------------------------------------- warp (matcher.cpp:36-116)
__device__ inline void warp_matrix_affine(const DevCam& cam, const double* px_ref, v3d f_ref, double depth_ref,
                                          const double* T_cur_ref, int level_ref, double* A /*row-major*/)
{
  const int halfpatch_size = 5;
  const v3d xyz_ref = {f_ref.x * depth_ref, f_ref.y * depth_ref, f_ref.z * depth_ref};
  v3d du = cam2world(cam, px_ref[0] + (double)halfpatch_size * (1 << level_ref), px_ref[1] + 0.0 * (1 << level_ref));
  v3d dv = cam2world(cam, px_ref[0] + 0.0 * (1 << level_ref), px_ref[1] + (double)halfpatch_size * (1 << level_ref));
  const double su = xyz_ref.z / du.z, sv = xyz_ref.z / dv.z;
  du = {du.x * su, du.y * su, du.z * su};
  dv = {dv.x * sv, dv.y * sv, dv.z * sv};
  double pcx, pcy, pux, puy, pvx, pvy;
  world2cam(cam, se3_transform(T_cur_ref, xyz_ref), pcx, pcy);
  world2cam(cam, se3_transform(T_cur_ref, du), pux, puy);
  world2cam(cam, se3_transform(T_cur_ref, dv), pvx, pvy);
  A[0] = (pux - pcx) / halfpatch_size; A[2] = (puy - pcy) / halfpatch_size;
  A[1] = (pvx - pcx) / halfpatch_size; A[3] = (pvy - pcy) / halfpatch_size;
}

__device__ __forceinline__ int best_search_level(const double* A, int max_level)
{
  int search_level = 0;
  double D = A[0] * A[3] - A[2] * A[1];
  while (D > 3.0 && search_level < max_level) { search_level += 1; D *= 0.25; }
  return search_level;
}

// vision.h:19-36
__device__ __forceinline__ float interpolate_8u(const uint8_t* img, int stride, float u, float v)
{
  const int x = (int)floorf(u), y = (int)floorf(v);     // == floor((double)u) for a float argument
  const float sx = u - x, sy = v - y;
  const float w00 = (1.0f - sx) * (1.0f - sy);
  const float w01 = (1.0f - sx) * sy;
  const float w10 = sx * (1.0f - sy);
  const float w11 = 1.0f - w00 - w01 - w10;
  const uint8_t* p = img + (size_t)y * stride + x;
  return w00 * p[0] + w01 * p[stride] + w10 * p[1] + w11 * p[stride + 1];
}


// ---------------------------------------------------------------- feature alignment: one THREAD per problem
// feature_alignment::align2D / align1D float paths (feature_alignment.cpp:35-282).
//
// The reference accumulates H and J*res pixel by pixel in float (`acc += term`); float addition is not
// associative, so the sums cannot be tree-reduced without changing results.  With millions of
// independent problems per step the natural mapping is therefore the reference's own loop, one thread
// per problem: the 10x10 template lives in 25 registers, the per-pixel template gradient (an integer in
// [-255,255] per axis) is staged once as packed binary16 pairs in shared memory ([64][LK_T] words, conflict
// free), the 9x9 search window is streamed row by row with three aligned word loads per row, and every
// float operation happens in the reference's order.  Results are bit-identical to the CPU code.
constexpr int LK_T = 128;
// resident CTAs per SM: 4 (128 registers, no spills since the byte conversions left the XU pipe: 0.702 -> 0.664 ms per 2.4 M jobs
// against 3 CTAs at 167 registers; 5 CTAs = 96 registers spill)
#ifndef LK_CTAS
#define LK_CTAS 4
#endif

// One refinement problem, written by the warp-cooperative producers with ONE coalesced 128-byte store.
struct __align__(16) LkJob {
  uint8_t pwb[100];        // 10x10 (patch with border), row-major
  float u, v;              // start position at the scale of the search image (the reference's first statement casts to float)
  float dirx, diry;        // align1D direction
  int item;                // index of the seed / candidate / problem the result belongs to
  int image;               // image inside the frame batch
  int level_mode;          // search level | mode << 8 (0 align2D, 1 align1D); < 0: nothing to do
};
static_assert(sizeof(LkJob) == 128, "LkJob must be one 128-byte line");

// Eigen Matrix3f::inverse(), cofactor path (Eigen/src/LU/InverseImpl.h)
__device__ __forceinline__ void inv3f(const float* m, float* r)
{
#define M_(i, j) m[(i) * 3 + (j)]
#define COF_(i, j) (M_(((i) + 1) % 3, ((j) + 1) % 3) * M_(((i) + 2) % 3, ((j) + 2) % 3) - M_(((i) + 1) % 3, ((j) + 2) % 3) * M_(((i) + 2) % 3, ((j) + 1) % 3))
  const float c00 = COF_(0, 0), c10 = COF_(1, 0), c20 = COF_(2, 0);
  const float det = c00 * M_(0, 0) + (c10 * M_(1, 0) + c20 * M_(2, 0));
  const float invdet = 1.0f / det;
  r[3] = COF_(0, 1) * invdet; r[4] = COF_(1, 1) * invdet; r[6] = COF_(0, 2) * invdet;
  r[5] = COF_(2, 1) * invdet; r[7] = COF_(1, 2) * invdet; r[8] = COF_(2, 2) * invdet;
  r[0] = c00 * invdet; r[1] = c10 * invdet; r[2] = c20 * invdet;
#undef COF_
#undef M_
}

// byte k of a register-resident byte array (k is a compile-time constant after unrolling)
template <int NW> __device__ __forceinline__ int reg_byte(const uint32_t (&w)[NW], int k) { return (int)((w[k >> 2] >> ((k & 3) * 8)) & 0xffu); }

template <int NW> __device__ __forceinline__ float reg_byte_f(const uint32_t (&w)[NW], int k) { return byte_to_float(w[k >> 2], k & 3); }

// nine consecutive pixels starting at p (any alignment) as floats; reads the three aligned words that hold them
__device__ __forceinline__ void load_row9(const uint8_t* p, float (&o)[9])
{
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;
  const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
  const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh), b8 = w2 >> sh;
#pragma unroll
  for (int k = 0; k < 4; ++k) { o[k] = byte_to_float(lo, k); o[4 + k] = byte_to_float(hi, k); }
  o[8] = byte_to_float(b8, 0);
}

// align2D (feature_alignment.cpp:154-282).  w: template with border, rp: 8x8 reference patch, sd: this thread's
// column of the shared gradient array.  u, v in/out at the scale of `img`.  Returns converged.
__device__ bool lk_align2d(const uint8_t* img, int pitch, int cols, int rows, const uint32_t (&w)[25], const uint32_t (&rp)[16],
                           int n_iter, float& u_io, float& v_io, uint32_t* sd)
{
  float h00 = 0.f, h01 = 0.f, h02 = 0.f, h11 = 0.f, h12 = 0.f;
#pragma unroll
  for (int y = 0; y < 8; ++y) {
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const int k = (y + 1) * 10 + 1 + x;
      const int dxi = reg_byte(w, k + 1) - reg_byte(w, k - 1), dyi = reg_byte(w, k + 10) - reg_byte(w, k - 10);
      const float j0 = 0.5f * (float)dxi, j1 = 0.5f * (float)dyi;      // exact: 0.5 * int (the reference goes through double)
      h00 += j0 * j0; h01 += j0 * j1; h02 += j0; h11 += j1 * j1; h12 += j1;
      // staged as two halves: 0.5 * [-255, 255] is exact in binary16, and half -> float is a full-rate instruction
      const __half2 jh = __floats2half2_rn(j0, j1);
      sd[(y * 8 + x) * LK_T] = *reinterpret_cast<const uint32_t*>(&jh);
    }
  }
  const float H[9] = {h00, h01, h02, h01, h11, h12, h02, h12, 64.0f};
  float Hinv[9];
  inv3f(H, Hinv);
  float mean_diff = 0.f;
  float u = u_io, v = v_io;
  const float min_update_squared = (float)(0.5 * 0.5);
  bool converged = false;
  for (int iter = 0; iter < n_iter; ++iter) {
    const int u_r = (int)floorf(u), v_r = (int)floorf(v);
    if (u_r < 4 || v_r < 4 || u_r >= cols - 4 || v_r >= rows - 4) break;
    if (isnan(u) || isnan(v)) return false;
    const float sx = u - u_r, sy = v - v_r;
    const float wTL = (float)((1.0 - sx) * (1.0 - sy));
    const float wTR = (float)(sx * (1.0 - sy));
    const float wBL = (float)((1.0 - sx) * sy);
    const float wBR = sx * sy;
    const uint8_t* base = img + (size_t)(v_r - 4) * pitch + (u_r - 4);
    float J0 = 0.f, J1 = 0.f, J2 = 0.f;
    float top[9], bot[9];
    load_row9(base, top);
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      load_row9(base + (size_t)(y + 1) * pitch, bot);
#pragma unroll
      for (int x = 0; x < 8; ++x) {
        const float search_pixel = wTL * top[x] + wTR * top[x + 1] + wBL * bot[x] + wBR * bot[x + 1];
        const float res = search_pixel - reg_byte_f(rp, y * 8 + x) + mean_diff;
        const uint32_t d = sd[(y * 8 + x) * LK_T];
        const float2 j = __half22float2(*reinterpret_cast<const __half2*>(&d));
        J0 -= res * j.x; J1 -= res * j.y; J2 -= res;
      }
#pragma unroll
      for (int x = 0; x < 9; ++x) top[x] = bot[x];
    }
    // update = Hinv * Jres (Eigen lazy product: x0 + (x1 + x2))
    const float up0 = Hinv[0] * J0 + (Hinv[1] * J1 + Hinv[2] * J2);
    const float up1 = Hinv[3] * J0 + (Hinv[4] * J1 + Hinv[5] * J2);
    const float up2 = Hinv[6] * J0 + (Hinv[7] * J1 + Hinv[8] * J2);
    u += up0; v += up1; mean_diff += up2;
    if (up0 * up0 + up1 * up1 < min_update_squared) { converged = true; break; }
  }
  u_io = u; v_io = v;
  return converged;
}

// align1D (feature_alignment.cpp:35-152): motion restricted to `dir`; the projected template gradient is a
// general float, staged as float bits.
__device__ bool lk_align1d(const uint8_t* img, int pitch, int cols, int rows, float dir0, float dir1, const uint32_t (&w)[25],
                           const uint32_t (&rp)[16], int n_iter, float& u_io, float& v_io, double& h_inv, uint32_t* sd)
{
  float h00 = 0.f, h01 = 0.f;
#pragma unroll
  for (int y = 0; y < 8; ++y) {
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const int k = (y + 1) * 10 + 1 + x;
      const int dxi = reg_byte(w, k + 1) - reg_byte(w, k - 1), dyi = reg_byte(w, k + 10) - reg_byte(w, k - 10);
      const float j0 = (float)(0.5 * (double)(dir0 * (float)dxi + dir1 * (float)dyi));
      h00 += j0 * j0; h01 += j0;
      sd[(y * 8 + x) * LK_T] = __float_as_uint(j0);
    }
  }
  const float h11 = 64.0f;
  h_inv = 1.0 / h00 * 8 * 8;
  const float det = h00 * h11 - h01 * h01;
  const float invdet = 1.0f / det;
  const float Hinv[4] = {h11 * invdet, -h01 * invdet, -h01 * invdet, h00 * invdet};
  float mean_diff = 0.f;
  float u = u_io, v = v_io;
  const float min_update_squared = (float)(0.03 * 0.03);
  float chi2 = 0.f, up0 = 0.f, up1 = 0.f;
  bool converged = false;
  for (int iter = 0; iter < n_iter; ++iter) {
    const int u_r = (int)floorf(u), v_r = (int)floorf(v);
    if (u_r < 4 || v_r < 4 || u_r >= cols - 4 || v_r >= rows - 4) break;
    if (isnan(u) || isnan(v)) return false;
    const float sx = u - u_r, sy = v - v_r;
    const float wTL = (float)((1.0 - sx) * (1.0 - sy));
    const float wTR = (float)(sx * (1.0 - sy));
    const float wBL = (float)((1.0 - sx) * sy);
    const float wBR = sx * sy;
    const uint8_t* base = img + (size_t)(v_r - 4) * pitch + (u_r - 4);
    float J0 = 0.f, J1 = 0.f, new_chi2 = 0.f;
    float top[9], bot[9];
    load_row9(base, top);
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      load_row9(base + (size_t)(y + 1) * pitch, bot);
#pragma unroll
      for (int x = 0; x < 8; ++x) {
        const float search_pixel = wTL * top[x] + wTR * top[x + 1] + wBL * bot[x] + wBR * bot[x + 1];
        const float res = search_pixel - reg_byte_f(rp, y * 8 + x) + mean_diff;
        const float j0 = __uint_as_float(sd[(y * 8 + x) * LK_T]);
        J0 -= res * j0; J1 -= res; new_chi2 += res * res;
      }
#pragma unroll
      for (int x = 0; x < 9; ++x) top[x] = bot[x];
    }
    if (iter > 0 && new_chi2 > chi2) { u -= up0; v -= up1; break; }   // sic (:122-123)
    chi2 = new_chi2;
    up0 = Hinv[0] * J0 + Hinv[1] * J1;
    up1 = Hinv[2] * J0 + Hinv[3] * J1;
    u += up0 * dir0; v += up0 * dir1; mean_diff += up1;
    if (up0 * up0 + up1 * up1 < min_update_squared) { converged = true; break; }
  }
  u_io = u; v_io = v;
  return converged;
}

// ---------------------------------------------------------------- ZMSSD (patch_score.h)
struct RefPatchRegs { uint32_t w[16]; int sumA, sumAA; };

__device__ __forceinline__ void load_ref_patch(const uint8_t* patch /*64 B, 4-aligned*/, RefPatchRegs& r)
{
  const uint32_t* p = reinterpret_cast<const uint32_t*>(patch);
  uint32_t sa = 0, saa = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    r.w[i] = p[i];
    sa = __dp4a(r.w[i], 0x01010101u, sa);
    saa = __dp4a(r.w[i], r.w[i], saa);
  }
  r.sumA = (int)sa; r.sumAA = (int)saa;
}

// cur points at the top-left pixel of the 8x8 window (any alignment)
__device__ __forceinline__ int zmssd_8x8(const RefPatchRegs& r, const uint8_t* cur, int pitch)
{
  uint32_t sb = 0, sbb = 0, sab = 0;
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(cur);
  const unsigned sh = (unsigned)(a0 & 3) * 8;
#pragma unroll
  for (int y = 0; y < 8; ++y) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>((a0 & ~(uintptr_t)3) + (size_t)y * pitch);   // pitch % 4 == 0
    const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
    const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
    sb = __dp4a(lo, 0x01010101u, sb); sb = __dp4a(hi, 0x01010101u, sb);
    sbb = __dp4a(lo, lo, sbb); sbb = __dp4a(hi, hi, sbb);
    sab = __dp4a(lo, r.w[2 * y], sab); sab = __dp4a(hi, r.w[2 * y + 1], sab);
  }
  const int sumB = (int)sb, sumBB = (int)sbb, sumAB = (int)sab;
  return r.sumAA - 2 * sumAB + sumBB - (r.sumA * r.sumA - 2 * r.sumA * sumB + sumB * sumB) / 64;
}

// matcher.cpp:123-136 (association of the 3-term sums as generated by Eigen 3.4 / SSE2)
__device__ inline bool depth_from_triangulation(const double* T, v3d f_ref, v3d f_cur, double* depth)
{
  double R[9];
  q_matrix(T + 3, R);
  v3d a0;
  a0.x = (R[0] * f_ref.x + R[1] * f_ref.y) + R[2] * f_ref.z;
  a0.y = (R[3] * f_ref.x + R[4] * f_ref.y) + R[5] * f_ref.z;
  a0.z = R[6] * f_ref.x + (R[7] * f_ref.y + R[8] * f_ref.z);
  const v3d a1 = f_cur;
  const double m00 = dot3(a0, a0), m01 = dot3(a0, a1), m11 = dot3(a1, a1);
  const double det = m00 * m11 - m01 * m01;
  if (det < 0.000001) return false;
  const double invdet = 1.0 / det;
  const double i00 = m11 * invdet, i01 = -m01 * invdet;
  const double r0 = i00 * a0.x + i01 * a1.x, r1 = i00 * a0.y + i01 * a1.y, r2 = i00 * a0.z + i01 * a1.z;
  const double d0 = -((r0 * T[0] + r1 * T[1]) + r2 * T[2]);
  *depth = fabs(d0);
  return true;
}

// ---------------------------------------------------------------- depth filter scalars
__device__ inline double normal_pdf(double x, double mean, double std_dev)
{
  const double SQRT_2_PI = 1.41421356237309505;          // sic, depth_filter.cpp:360
  const double q = (x - mean) / std_dev;
  const double exponent = -0.5 * (q * q);                // pow(q, 2)
  return (1 / (std_dev * SQRT_2_PI)) * exp(exponent);
}

// DepthFilter::updateSeed depth_filter.cpp:368-391 (float variables, double where a `1.` literal appears)
__device__ inline void update_seed(float x, float tau2, svob200_seed* seed)
{
  const float norm_scale = sqrtf(seed->sigma2 + tau2);
  if (isnan(norm_scale)) return;
  const float s2 = (float)(1. / (1. / seed->sigma2 + 1. / tau2));
  const float m = s2 * (seed->mu / seed->sigma2 + x / tau2);
  float C1 = (float)((double)(seed->a / (seed->a + seed->b)) * normal_pdf(x, seed->mu, norm_scale));
  float C2 = (float)((double)(seed->b / (seed->a + seed->b)) * 1. / (double)seed->z_range);
  const float normalization_constant = C1 + C2;
  C1 /= normalization_constant;
  C2 /= normalization_constant;
  const float f = (float)((double)C1 * (seed->a + 1.) / (seed->a + seed->b + 1.) + (double)(C2 * seed->a) / (seed->a + seed->b + 1.));
  const float e = (float)((double)C1 * (seed->a + 1.) * (seed->a + 2.) / ((seed->a + seed->b + 1.) * (seed->a + seed->b + 2.))
                          + (double)(C2 * seed->a * (seed->a + 1.0f) / ((seed->a + seed->b + 1.0f) * (seed->a + seed->b + 2.0f))));
  const float mu_new = C1 * m + C2 * seed->mu;
  seed->sigma2 = C1 * (s2 + m * m) + C2 * (seed->sigma2 + seed->mu * seed->mu) - mu_new * mu_new;
  seed->mu = mu_new;
  seed->a = (e - f) / (f - e / f);
  seed->b = seed->a * (1.0f - f) / f;
}

// DepthFilter::computeTau depth_filter.cpp:396-416
__device__ inline double compute_tau(const double* T_ref_cur, v3d f, double z, double px_error_angle)
{
  const double PI_ = 3.14159265;                         // svo::PI global.h:92
  const v3d t = {T_ref_cur[0], T_ref_cur[1], T_ref_cur[2]};
  const v3d a = {f.x * z - t.x, f.y * z - t.y, f.z * z - t.z};
  const double t_norm = norm3(t), a_norm = norm3(a);
  const double alpha = acos(dot3(f, t) / t_norm);
  const double beta = acos(dot3(a, v3_neg(t)) / (t_norm * a_norm));
  const double beta_plus = beta + px_error_angle;
  const double gamma_plus = PI_ - alpha - beta_plus;
  const double z_plus = t_norm * sin(beta_plus) / sin(gamma_plus);
  return z_plus - z;
}

// ---------------------------------------------------------------- findEpipolarMatchDirect in phases
// Phase 1 (per-thread double geometry), phase 2 (warp-cooperative patch warp + ZMSSD walk), phase 3
// (thread-per-problem LK refinement, shared with findMatchDirect), phase 4 (per-thread triangulation /
// seed update).  Each phase is its own kernel so that every one of them runs with the mapping that suits
// it and the FP64 pipe never executes the same geometry redundantly across a warp.

enum { EPI_MODE_NONE = 0, EPI_MODE_DIRECT = 1, EPI_MODE_WALK = 2 };
enum { EPI_FOUND_NONE = 0, EPI_FOUND_REFINED = 1, EPI_FOUND_UV_ONLY = 2 };

// everything epi_geometry() derives (thread-local); split into a cold record (finish kernels) and a packed task (search kernel)
struct EpiGeom {
  double T_cur_ref[7];
  double A[4];                          // A_cur_ref, row-major
  double Bx0, By0, stepx, stepy;        // epipolar sample chain: uv_0 = B - step, uv_{i+1} = uv_i + step
  double px_mid[2];                     // (px_A + px_B) / 2
  double ex, ey;                        // epi_dir_ = A - B on the unit plane (matcher.cpp:224)
  double epi_length;
  float a00, a01, a10, a11, pr0, pr1;   // A_ref_cur (float) and px_ref at the reference level
  float dirx, diry;                     // (px_A - px_B).cast<float>().normalized()
  uint32_t n;                           // samples of the walk: n_steps + 1 <= INT_MAX + 1
  int warp_ok, L, mode, n_steps_report, reject;
};

// what the per-item finish kernels need, 128 B
struct __align__(16) EpiCold {
  double T_cur_ref[7];
  double A[4];
  double ex, ey;
  double epi_length;
  int L, mode, reject, n_steps_report;
};
static_assert(sizeof(EpiCold) == 128, "EpiCold layout");

// what the search kernel needs, packed into ONE 128-byte line: a warp fetches it with a single coalesced load (lane k
// holds word k) one item ahead of the item it is working on, and pulls fields out by shuffle.  The first 16 bytes (flags, levels,
// epi_length) are all the depth filter's finish kernel reads of it: one 32-byte sector per seed instead of a 128-byte cold record.
struct __align__(16) SearchTask { uint32_t w[32]; };
enum { ST_FLAGS = 0, ST_LEVELS = 1, ST_EPILEN = 2, ST_REF_SLOT = 4, ST_REF_IMAGE = 5, ST_CUR_IMAGE = 6, ST_NSAMP = 7, ST_A00 = 8, ST_A01 = 9, ST_A10 = 10, ST_A11 = 11,
       ST_PR0 = 12, ST_PR1 = 13, ST_DIRX = 14, ST_DIRY = 15, ST_BX0 = 16, ST_BY0 = 18, ST_STEPX = 20, ST_STEPY = 22, ST_MIDX = 24, ST_MIDY = 26 };
// flags: bit 0 search this item, bit 1 the warp matrix is finite, bits 2-3 EPI_MODE_*, bits 4-6 the depth filter's early status
// (SVOB200_SEED_BEHIND / _NOT_IN_FRAME / _TOO_OLD; 0 = the matcher runs), bit 7 z_inv_min is NaN (depth_filter.cpp:334)
// levels: search level | reference level << 8; nsamp: samples of the walk (a full word: the reference walks any length)
enum { ST_ACTIVE = 1, ST_WARP_OK = 2, ST_MODE_SHIFT = 2, ST_STATUS_SHIFT = 4, ST_ZMIN_NAN = 128, ST_FREE = 256 /* empty slot of a seed pool */ };

// the reference feature of an item, wherever its record lives (caller's svob200_feature_ref or the tracker's compact SeedRef)
struct RefFtr {
  double px[2]; v3d f; int level, type; double grad[2];
  int ref_slot, ref_image, cur_image, kf;
  int state, batch_id;                 // seed pools only (SeedRef)
};
__device__ __forceinline__ RefFtr ref_ftr_of(const svob200_feature_ref& r)
{
  RefFtr f;
  f.px[0] = r.px[0]; f.px[1] = r.px[1]; f.f = {r.f[0], r.f[1], r.f[2]}; f.level = r.level; f.type = r.type; f.grad[0] = r.grad[0]; f.grad[1] = r.grad[1];
  f.ref_slot = (int)r.ref_frame_id; f.ref_image = r.ref_image; f.cur_image = r.cur_image; f.kf = 0; f.state = 0; f.batch_id = 0;
  return f;
}

// cold: stand-alone queries only (nullptr for the depth filter, whose finish kernel recomputes the poses and reads the task's head)
__device__ inline void store_geometry(const EpiGeom& g, const RefFtr& f, bool active, uint32_t extra_flags, EpiCold* cold, SearchTask* task)
{
  if (cold) {
    EpiCold c;
    for (int k = 0; k < 7; ++k) c.T_cur_ref[k] = g.T_cur_ref[k];
    for (int k = 0; k < 4; ++k) c.A[k] = g.A[k];
    c.ex = g.ex; c.ey = g.ey; c.epi_length = g.epi_length; c.L = g.L; c.mode = g.mode; c.reject = g.reject; c.n_steps_report = g.n_steps_report;
    *cold = c;
  }
  SearchTask t;
#pragma unroll
  for (int k = 0; k < 32; ++k) t.w[k] = 0;
  t.w[ST_FLAGS] = (active ? ST_ACTIVE : 0) | (g.warp_ok ? ST_WARP_OK : 0) | ((uint32_t)g.mode << ST_MODE_SHIFT) | extra_flags;
  t.w[ST_LEVELS] = (uint32_t)g.L | ((uint32_t)f.level << 8);
  t.w[ST_NSAMP] = g.n;
  t.w[ST_EPILEN] = (uint32_t)__double2loint(g.epi_length); t.w[ST_EPILEN + 1] = (uint32_t)__double2hiint(g.epi_length);
  t.w[ST_REF_SLOT] = (uint32_t)f.ref_slot; t.w[ST_REF_IMAGE] = (uint32_t)f.ref_image; t.w[ST_CUR_IMAGE] = (uint32_t)f.cur_image;
  t.w[ST_A00] = __float_as_uint(g.a00); t.w[ST_A01] = __float_as_uint(g.a01); t.w[ST_A10] = __float_as_uint(g.a10); t.w[ST_A11] = __float_as_uint(g.a11);
  t.w[ST_PR0] = __float_as_uint(g.pr0); t.w[ST_PR1] = __float_as_uint(g.pr1); t.w[ST_DIRX] = __float_as_uint(g.dirx); t.w[ST_DIRY] = __float_as_uint(g.diry);
  const double d[6] = {g.Bx0, g.By0, g.stepx, g.stepy, g.px_mid[0], g.px_mid[1]};
#pragma unroll
  for (int k = 0; k < 6; ++k) { t.w[ST_BX0 + 2 * k] = (uint32_t)__double2loint(d[k]); t.w[ST_BX0 + 2 * k + 1] = (uint32_t)__double2hiint(d[k]); }
  uint4* dst = reinterpret_cast<uint4*>(task);
#pragma unroll
  for (int k = 0; k < 8; ++k) dst[k] = make_uint4(t.w[4 * k], t.w[4 * k + 1], t.w[4 * k + 2], t.w[4 * k + 3]);
}

struct __align__(16) EpiSearch {
  int found;                            // EPI_FOUND_*
  int zmssd_best, n_evals;
  int px_cur_valid;                     // the reference wrote Matcher::px_cur_ (matcher.cpp:259, :327, :345)
  double px_cur[2], uv_best[2], h_inv;
  double pad_;
};
static_assert(sizeof(EpiSearch) == 64, "EpiSearch layout");

// the depth filter's 32-byte variant of EpiSearch: xy = the matched pixel (REFINED, or the pre-refinement pixel while
// found == NONE) or uv_best on the unit plane (UV_ONLY: the pixel is world2cam_uv(xy), recomputed by the consumer)
struct __align__(16) SeedMatch {
  int found, zmssd_best, n_evals, xy_valid;
  double xy[2];
};
static_assert(sizeof(SeedMatch) == 32, "SeedMatch layout");

__device__ __forceinline__ EpiSearch epi_search_none()
{
  EpiSearch s;
  s.found = EPI_FOUND_NONE; s.zmssd_best = 2000 * 64; s.n_evals = 0; s.px_cur_valid = 0; s.px_cur[0] = s.px_cur[1] = 0;
  s.uv_best[0] = s.uv_best[1] = 0; s.h_inv = 0; s.pad_ = 0;
  return s;
}

// The search and patch-warp kernels work in GROUPS of 8 lanes: one item (seed / reprojection candidate) per group, four
// items per warp in lockstep.  Per item the code path is ~1,300 SASS instructions of mostly straight-line work (task decode,
// 100 bilinear taps, patch extraction, a short epipolar walk, reductions, job emission); run by a full warp it executed
// once per item at ~22 of 32 lanes busy (ncu: 936 warp instructions per seed).  Four items per warp share every one of those
// instructions, and the 8 taps a group issues per load still fall into 1-2 cache lines, so L1 wavefronts per item do not grow
// (a thread-per-item mapping would need 32 lines per load instruction and is LSU-bound).
constexpr int GL = 8;                    // lanes per group
constexpr int GPW = 32 / GL;             // groups (items) per warp
constexpr int EPI_GCHUNK = 32;           // epipolar samples a group stages per round (steady-state walks are <= 47 steps)
#ifndef SEARCH_CTAS_PER_SM
#define SEARCH_CTAS_PER_SM 5
#endif
// resident CTAs per SM of the persistent search kernel.  Measured per 3.1 M seeds with the current patch-warp code (value of the
// whole step in k frames/s): 4 CTAs (121 registers) 1.73 ms / 890 k, 5 (96 registers) 1.62 ms / 925 k, 6 (80) 1.67 ms / 907 k,
// 7 (72, spills) 1.63 ms / 911 k, 8 (64, spills) 1.79 ms / 878 k: with 96 registers ptxas keeps a pass's 16 pixel loads in flight
constexpr int SEARCH_CTAS = SEARCH_CTAS_PER_SM;

struct EpiGroupSmem {
  __align__(16) uint8_t pwb[112];       // 100 used
  __align__(16) uint8_t patch[64];
  double uv[2 * EPI_GCHUNK];            // the reference's running sums uv += step (x, y interleaved)
  short2 pxi[EPI_GCHUNK + 1];
  int pad_[3];
};
static_assert(sizeof(EpiGroupSmem) % 16 == 0, "EpiGroupSmem must keep 16-byte alignment in an array");

// word k of the 128-byte task a group holds as one uint4 per lane (lane s of the group has words 4s .. 4s+3)
__device__ __forceinline__ uint32_t task_word(const uint4& tq, int k, int gbase, unsigned gmask)
{
  const uint32_t c = (k & 3) == 0 ? tq.x : ((k & 3) == 1 ? tq.y : ((k & 3) == 2 ? tq.z : tq.w));
  return __shfl_sync(gmask, c, gbase + (k >> 2));
}
__device__ __forceinline__ double task_double(const uint4& tq, int k, int gbase, unsigned gmask)
{
  const int lo = (int)task_word(tq, k, gbase, gmask), hi = (int)task_word(tq, k + 1, gbase, gmask);
  return __hiloint2double(hi, lo);
}

// matcher.cpp:207-288 up to the start of the walk: pure per-thread math
__device__ inline void epi_geometry(const DevCam& cam, const RefFtr& f, const double* T_cur_ref, double d_estimate,
                                    double d_min, double d_max, const svob200_matcher_opts& o, EpiGeom* g)
{
  for (int k = 0; k < 7; ++k) g->T_cur_ref[k] = T_cur_ref[k];
  g->reject = 0; g->mode = EPI_MODE_NONE; g->n = 0; g->n_steps_report = 0; g->L = 0; g->epi_length = 0; g->warp_ok = 0;
  g->Bx0 = g->By0 = g->stepx = g->stepy = 0; g->px_mid[0] = g->px_mid[1] = 0; g->ex = g->ey = 0;
  g->a00 = g->a01 = g->a10 = g->a11 = g->pr0 = g->pr1 = g->dirx = g->diry = 0;
  const v3d f_ref = f.f;
  const v3d tA = se3_transform(T_cur_ref, {f_ref.x * d_min, f_ref.y * d_min, f_ref.z * d_min});
  const double Ax = tA.x / tA.z, Ay = tA.y / tA.z;
  const v3d tB = se3_transform(T_cur_ref, {f_ref.x * d_max, f_ref.y * d_max, f_ref.z * d_max});
  const double Bx = tB.x / tB.z, By = tB.y / tB.z;
  const double ex = Ax - Bx, ey = Ay - By;
  g->ex = ex; g->ey = ey;
  warp_matrix_affine(cam, f.px, f_ref, d_estimate, T_cur_ref, f.level, g->A);
  const double* A = g->A;
  if (f.type == 1 && o.epi_search_edgelet_filtering) {
    double gx = A[0] * f.grad[0] + A[1] * f.grad[1], gy = A[2] * f.grad[0] + A[3] * f.grad[1];
    { const double z = gx * gx + gy * gy; if (z > 0) { const double n = sqrt(z); gx /= n; gy /= n; } }
    double nx = ex, ny = ey;
    { const double z = nx * nx + ny * ny; if (z > 0) { const double n = sqrt(z); nx /= n; ny /= n; } }
    const double cosangle = fabs(gx * nx + gy * ny);
    if (cosangle < o.epi_search_edgelet_max_angle) { g->reject = 1; return; }
  }
  const int L = best_search_level(A, o.max_search_level);
  g->L = L;
  double pAx, pAy, pBx, pBy;
  world2cam_uv(cam, Ax, Ay, pAx, pAy);
  world2cam_uv(cam, Bx, By, pBx, pBy);
  { const double dx = pAx - pBx, dy = pAy - pBy; g->epi_length = sqrt(dx * dx + dy * dy) * pow2_inv(L); }   // / (1 << L), exactly
  // warpAffine prologue (matcher.cpp:92-102)
  {
    const double det = A[0] * A[3] - A[2] * A[1];
    const double invdet = 1.0 / det;
    g->a00 = (float)(A[3] * invdet); g->a01 = (float)(-A[1] * invdet);
    g->a10 = (float)(-A[2] * invdet); g->a11 = (float)(A[0] * invdet);
    g->warp_ok = isnan(g->a00) ? 0 : 1;
    g->pr0 = (float)f.px[0] * pow2_inv_f(f.level); g->pr1 = (float)f.px[1] * pow2_inv_f(f.level);   // / (float)(1 << level), exactly
  }
  {
    float dx = (float)(pAx - pBx), dy = (float)(pAy - pBy);
    const float z = dx * dx + dy * dy;
    if (z > 0.0f) { const float n = sqrtf(z); dx /= n; dy /= n; }
    g->dirx = dx; g->diry = dy;
  }
  g->px_mid[0] = (pAx + pBx) / 2.0; g->px_mid[1] = (pAy + pBy) / 2.0;
  if (g->epi_length < 2.0) { g->mode = EPI_MODE_DIRECT; return; }
  // x86 (size_t)(double): NaN / out of range -> 2^63 -> "skip epipolar search" (matcher.cpp:283-288).  The step count is
  // reported as the restatement's (int)n_steps: the low 32 bits, so 0 for 2^63
  const double q = g->epi_length / 0.7;
  if (!(q == q) || q >= 9.2e18) return;
  const unsigned long long n_steps = (unsigned long long)q;
  g->n_steps_report = (int)(uint32_t)n_steps;
  g->stepx = ex / (double)n_steps; g->stepy = ey / (double)n_steps;
  // the C ABI rejects a negative max_epi_search_steps, so n_steps <= INT_MAX here and n_steps + 1 fits 32 bits
  if (n_steps > (unsigned long long)o.max_epi_search_steps) return;
  g->n = (uint32_t)n_steps + 1u;
  g->Bx0 = Bx - g->stepx; g->By0 = By - g->stepy;
  g->mode = EPI_MODE_WALK;
}

// one 128-byte store of a refinement job by a group: lane s writes words 4s .. 4s+3 (pwb words come from shared memory)
__device__ __forceinline__ void emit_lk_job(LkJob* dst, const uint8_t* s_pwb, float u, float v, float dirx, float diry, int item,
                                            int image, int level_mode, int sub)
{
  const uint32_t* pw = reinterpret_cast<const uint32_t*>(s_pwb);
  uint4 q;
  if (sub < 6) q = make_uint4(pw[4 * sub], pw[4 * sub + 1], pw[4 * sub + 2], pw[4 * sub + 3]);
  else if (sub == 6) q = make_uint4(pw[24], __float_as_uint(u), __float_as_uint(v), __float_as_uint(dirx));
  else q = make_uint4(__float_as_uint(diry), (uint32_t)item, (uint32_t)image, (uint32_t)level_mode);
  reinterpret_cast<uint4*>(dst)[sub] = q;
}

// affine warp of the 10x10 reference patch (matcher.cpp:83-116) into shared memory by a group of 8 lanes
// R taps per lane in flight together (tap i = sub + 8 r); the tap's position (x - 5, y - 5) in the row-major 10x10 patch comes
// from a small shared-memory table (a running position with its wrap test cost four instructions per tap: 1.584 -> 1.544 ms per
// 3.1 M seeds together with the integer bounds test below).
// The four pixel loads of a tap are UNCONDITIONAL (an out-of-bounds tap reads the image's first 2x2 pixels and is discarded)
// and stay raw 32-bit values until the second loop, so that all 4R loads are issued before the first conversion waits for
// one (with a branch around the loads the compiler converted inside it and every tap waited for its own loads).
// one byte through the read-only path as an opaque 32-bit value: the compiler cannot fold the int -> float conversion into
// the load (it did, and then placed every tap's conversions — which wait for the data — before the next tap's loads)
__device__ __forceinline__ unsigned ldg_u8_raw(const uint8_t* p)
{
  unsigned v;
  asm("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// (x - 5, y - 5) of tap i of the row-major 10x10 patch, as floats, in shared memory: one LDS.64 per tap instead of a running
// position with its wrap test.  104 entries: the idle lanes of the tail round read 100..103.
constexpr int TAP_TABLE = 104;
__device__ __forceinline__ void fill_tap_table(float2* s_tap)
{
  for (int i = threadIdx.x; i < TAP_TABLE; i += blockDim.x) s_tap[i] = make_float2((float)(i % 10 - 5), (float)(i / 10 - 5));
}

// a00 .. a11 arrive multiplied by 2^L (exact), so (a00 * 2^L) * (x - 5) is the same float as the reference's a00 * ((x - 5) * 2^L).
template <int R, bool TAIL>
__device__ __forceinline__ void warp_patch_taps(const uint8_t* rimg, unsigned rp, unsigned xmax, unsigned ymax, float a00, float a01, float a10, float a11,
                                                float pr0, float pr1, uint8_t* s_pwb, int i0, const float2* tap)
{
  bool inb[R];
  float w00[R], w01[R], w10[R], w11[R];
  unsigned v00[R], v01[R], v10[R], v11[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const float2 t = tap[GL * r];
    const float qx = (a00 * t.x + a01 * t.y) + pr0;
    const float qy = (a10 * t.x + a11 * t.y) + pr1;
    // the reference's test !(qx < 0 || qy < 0 || qx >= cols - 1 || qy >= rows - 1) on the floored coordinates: for q >= 0
    // floor(q) < n <=> q < n (n an integer), a negative q floors below zero = a huge unsigned, NaN converts to 0 and passes,
    // as it passes the float comparisons.  vk::interpolateMat_8u (vision.h:19-36) floors too.
    const int ix = __float2int_rd(qx), iy = __float2int_rd(qy);
    inb[r] = (unsigned)ix < xmax && (unsigned)iy < ymax;
    if (TAIL) inb[r] = inb[r] && (i0 + GL * r < 100);
    const float sx = qx - ix, sy = qy - iy;
    w00[r] = (1.0f - sx) * (1.0f - sy);
    w01[r] = (1.0f - sx) * sy;
    w10[r] = sx * (1.0f - sy);
    w11[r] = 1.0f - w00[r] - w01[r] - w10[r];
    const unsigned off = inb[r] ? (unsigned)iy * rp + (unsigned)ix : 0u;
    const uint8_t* p = rimg + off;
    v00[r] = ldg_u8_raw(p); v10[r] = ldg_u8_raw(p + 1); v01[r] = ldg_u8_raw(p + rp); v11[r] = ldg_u8_raw(p + rp + 1);
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = i0 + GL * r;
    const float f = w00[r] * (float)(int)v00[r] + w01[r] * (float)(int)v01[r] + w10[r] * (float)(int)v10[r] + w11[r] * (float)(int)v11[r];
    if (!TAIL || i < 100) s_pwb[i] = inb[r] ? (uint8_t)f : (uint8_t)0;
  }
}

template <bool PREFETCH>
__device__ __forceinline__ void warp_patch_10x10(const uint8_t* rimg, int rp, int rc, int rr, float a00, float a01, float a10, float a11,
                                                 float pr0, float pr1, int L, uint8_t* s_pwb, int sub, const float2* s_tap)
{
  // 100 taps over 8 lanes = 12 full rounds + 4 taps: three passes of four rounds (the 16 pixel loads of a lane in flight
  // together) and ONE tail round, not a fourth pass whose last three rounds would be all-idle instructions
  const float sc = (float)(1 << L);
  // ptxas interleaves tap r's conversions (which wait for its pixels) with tap r+1's address arithmetic, so the ~11 image
  // rows of the window are 11 exposed cache misses in a row; PREFETCH touches both ends of every patch row up front (two
  // image rows each; lane `sub` takes patch row `sub`, lanes 0..3 also the ends of rows 8 and 9).  Measured per 4,096
  // sequences: match_prepare (nothing else to overlap the misses with) 0.182 -> 0.162 ms; the persistent search kernel, whose
  // other resident warps already cover them, 1.69 -> 1.77 ms — so only the former prefetches.
#pragma unroll
  for (int t = 0; PREFETCH && t < 3; ++t) {
    const float xmaxf = (float)(rc - 1), ymaxf = (float)(rr - 1);
    const int tx = t == 0 ? 0 : (t == 1 ? 9 : ((sub & 1) ? 9 : 0));
    const int ty = t < 2 ? sub : 8 + (sub >> 1);
    const float q0 = (float)(tx - 5) * sc, q1 = (float)(ty - 5) * sc;
    const float qx = (a00 * q0 + a01 * q1) + pr0, qy = (a10 * q0 + a11 * q1) + pr1;
    const bool ok = (t < 2 || sub < 4) && !(qx < 0 || qy < 0 || qx >= xmaxf || qy >= ymaxf);
    if (ok) {
      const uint8_t* p = rimg + ((unsigned)(int)qy * (unsigned)rp + (unsigned)(int)qx);
      asm volatile("prefetch.global.L1 [%0];" :: "l"(p));
      asm volatile("prefetch.global.L1 [%0];" :: "l"(p + rp));
    }
  }
  const unsigned xmax = rc > 1 ? (unsigned)(rc - 1) : 0u, ymax = rr > 1 ? (unsigned)(rr - 1) : 0u;
  const float b00 = a00 * sc, b01 = a01 * sc, b10 = a10 * sc, b11 = a11 * sc;      // exact: sc is a power of two
  const float2* tap = s_tap + sub;
#pragma unroll 1
  for (int r0 = 0; r0 < 12; r0 += 4)
    warp_patch_taps<4, false>(rimg, (unsigned)rp, xmax, ymax, b00, b01, b10, b11, pr0, pr1, s_pwb, sub + GL * r0, tap + GL * r0);
  warp_patch_taps<1, true>(rimg, (unsigned)rp, xmax, ymax, b00, b01, b10, b11, pr0, pr1, s_pwb, sub + GL * 12, tap + GL * 12);
}

constexpr int JOB_BATCH = 8;             // LK job slots a group reserves per atomicAdd

// matcher.cpp:251-340 minus the LK refinement, for ONE item whose packed task the group holds in `tq`: warp the patch, walk
// the epipolar segment, and hand the refinement to the thread-per-problem LK kernel as a job.  Executed by the 8 lanes of
// a group (gmask); the other groups of the warp run their own items in lockstep.
__device__ __forceinline__ void epi_search_item(const DevFrame* frames, int cur_slot, const DevCam& cam, const svob200_matcher_opts& o,
                                                const uint4& tq, int item, EpiGroupSmem* S, int sub, int gbase, unsigned gmask,
                                                LkJob* jobs, int* job_count, int& slot_base, int& slots_left, EpiSearch* search,
                                                SeedMatch* seed_match, svob200_epi_result* api_results, const float2* s_tap)
{
  const int flags = (int)task_word(tq, ST_FLAGS, gbase, gmask);
  const int mode = (flags >> ST_MODE_SHIFT) & 3;
  const int levels = (int)task_word(tq, ST_LEVELS, gbase, gmask);
  const int L = levels & 0xff, ref_level = (levels >> 8) & 0xff;
  const int cur_image = (int)task_word(tq, ST_CUR_IMAGE, gbase, gmask);
  EpiSearch out = epi_search_none();
  if (api_results) { for (int k = sub; k < 28; k += GL) reinterpret_cast<uint32_t*>(S->pwb)[k] = 0; __syncwarp(gmask); }
  if (flags & ST_WARP_OK) {
    const DevFrame& ref = frames[(int)task_word(tq, ST_REF_SLOT, gbase, gmask)];
    const int ref_image = (int)task_word(tq, ST_REF_IMAGE, gbase, gmask);
    const uint8_t* rimg = ref.lvl[ref_level] + (size_t)ref_image * ref.img_stride[ref_level];
    warp_patch_10x10<false>(rimg, ref.pitch[ref_level], ref.w[ref_level], ref.h[ref_level],
                     __uint_as_float(task_word(tq, ST_A00, gbase, gmask)), __uint_as_float(task_word(tq, ST_A01, gbase, gmask)),
                     __uint_as_float(task_word(tq, ST_A10, gbase, gmask)), __uint_as_float(task_word(tq, ST_A11, gbase, gmask)),
                     __uint_as_float(task_word(tq, ST_PR0, gbase, gmask)), __uint_as_float(task_word(tq, ST_PR1, gbase, gmask)), L, S->pwb, sub, s_tap);
  }
  __syncwarp(gmask);
  for (int k = sub; k < 64; k += GL) S->patch[k] = S->pwb[((k >> 3) + 1) * 10 + 1 + (k & 7)];
  __syncwarp(gmask);
  if (api_results) {
    svob200_epi_result* R = &api_results[item];
    for (int k = sub; k < 100; k += GL) R->patch_with_border[k] = S->pwb[k];
    for (int k = sub; k < 64; k += GL) R->patch[k] = S->patch[k];
  }
  bool want_job = false;
  double px0 = 0.0, px1 = 0.0;
  if (mode == EPI_MODE_DIRECT) {
    px0 = task_double(tq, ST_MIDX, gbase, gmask); px1 = task_double(tq, ST_MIDY, gbase, gmask);
    want_job = true;
  } else if (mode == EPI_MODE_WALK) {
    const DevFrame& cur = frames[cur_slot];
    const uint8_t* cimg = cur.lvl[L] + (size_t)cur_image * cur.img_stride[L];
    const int cpitch = cur.pitch[L];
    const uint32_t n = task_word(tq, ST_NSAMP, gbase, gmask);
    RefPatchRegs rpatch;
    load_ref_patch(S->patch, rpatch);
    unsigned long long best = ((unsigned long long)(2000 * 64) << 32);   // PatchScore::threshold(), strict <
    double best_u = 0.0, best_v = 0.0;
    int evals = 0;
    // the reference's running sums uv += step: x chain on lane 0 of the group, y chain on lane 1 (two independent DADD chains)
    // (task_word's k must be uniform over the group: the SOURCE lane picks the component with its own k)
    const double bx0 = task_double(tq, ST_BX0, gbase, gmask), by0 = task_double(tq, ST_BY0, gbase, gmask);
    const double stx = task_double(tq, ST_STEPX, gbase, gmask), sty = task_double(tq, ST_STEPY, gbase, gmask);
    double uv = (sub & 1) ? by0 : bx0;
    const double st = (sub & 1) ? sty : stx;
    const double inv_scale = pow2_inv(L);                                 // exact: dividing by 2^L == multiplying by 2^-L
    short2 last = make_short2(0, 0);                                     // last_checked_pxi(0,0)
    for (uint32_t base = 0; base < n; base += EPI_GCHUNK) {
      const int m = (int)min((uint32_t)EPI_GCHUNK, n - base);
      if (sub < 2) {
        double* dst = S->uv + sub;
        for (int i = 0; i < m; ++i, uv += st) dst[2 * i] = uv;
      }
      if (sub == 0) S->pxi[0] = last;
      __syncwarp(gmask);
      // pixel of every sample, in parallel: Vector2i(px/(1<<L) + 0.5) with the x86 truncating conversion
      for (int i = sub; i < m; i += GL) {
        const double ux = S->uv[2 * i], uy = S->uv[2 * i + 1];
        const double vx = (cam.fx * ux + cam.cx) * inv_scale + 0.5, vy = (cam.fy * uy + cam.cy) * inv_scale + 0.5;
        const int ix = (vx == vx) ? (vx >= 32767.0 ? 32767 : (vx <= -32768.0 ? -32768 : (int)vx)) : -32768;
        const int iy = (vy == vy) ? (vy >= 32767.0 ? 32767 : (vy <= -32768.0 ? -32768 : (int)vy)) : -32768;
        S->pxi[i + 1] = make_short2((short)ix, (short)iy);
      }
      __syncwarp(gmask);
      last = S->pxi[m];
      for (int i = sub; i < m; i += GL) {
        const short2 c = S->pxi[i + 1], prev = S->pxi[i];
        if (c.x == prev.x && c.y == prev.y) continue;
        if (!in_frame_level(cam, c.x, c.y, 8, L)) continue;
        const int z = zmssd_8x8(rpatch, cimg + (size_t)(c.y - 4) * cpitch + (c.x - 4), cpitch);
        ++evals;
        const unsigned long long key = ((unsigned long long)(unsigned)z << 32) | (base + (unsigned)i);
        if (key < best) { best = key; best_u = S->uv[2 * i]; best_v = S->uv[2 * i + 1]; }
      }
      __syncwarp(gmask);
    }
    unsigned long long gbest = best;
#pragma unroll
    for (int off = GL / 2; off > 0; off >>= 1) {
      const unsigned long long other = __shfl_xor_sync(gmask, gbest, off);
      if (other < gbest) gbest = other;
      evals += __shfl_xor_sync(gmask, evals, off);
    }
    out.n_evals = evals;
    const int zbest = (int)(gbest >> 32);
    out.zmssd_best = zbest;
    if (zbest < 2000 * 64) {
      // uv_best lives on the lane that evaluated the winning step (keys are unique: they contain the step index)
      const unsigned owner = __ffs(__ballot_sync(gmask, best == gbest) & gmask) - 1;
      const double ubx = __shfl_sync(gmask, best_u, owner), uby = __shfl_sync(gmask, best_v, owner);
      world2cam_uv(cam, ubx, uby, px0, px1);
      out.uv_best[0] = ubx; out.uv_best[1] = uby;
      if (!o.subpix_refinement) { out.px_cur[0] = px0; out.px_cur[1] = px1; out.px_cur_valid = 1; out.found = EPI_FOUND_UV_ONLY; }
      else want_job = true;
    }
  }
  if (want_job) { out.px_cur[0] = px0; out.px_cur[1] = px1; out.px_cur_valid = 1; }
  if (sub == 0) {
    if (seed_match) {
      SeedMatch m;
      m.found = out.found; m.zmssd_best = out.zmssd_best; m.n_evals = out.n_evals; m.xy_valid = out.px_cur_valid;
      const bool uv = out.found == EPI_FOUND_UV_ONLY;
      m.xy[0] = uv ? out.uv_best[0] : out.px_cur[0]; m.xy[1] = uv ? out.uv_best[1] : out.px_cur[1];
      seed_match[item] = m;
    } else search[item] = out;
  }
  if (!want_job) return;
  // hand over to the LK kernel: px_scaled = px_cur / (1 << L) (double), cast to float at the start of align1D/2D
  if (slots_left == 0) {
    if (sub == 0) slot_base = atomicAdd(job_count, JOB_BATCH);
    slot_base = __shfl_sync(gmask, slot_base, gbase);
    slots_left = JOB_BATCH;
  }
  const int slot = slot_base + (JOB_BATCH - slots_left);
  --slots_left;
  emit_lk_job(&jobs[slot], S->pwb, (float)(px0 * pow2_inv(L)), (float)(px1 * pow2_inv(L)), __uint_as_float(task_word(tq, ST_DIRX, gbase, gmask)),
              __uint_as_float(task_word(tq, ST_DIRY, gbase, gmask)), item, cur_image, L | ((o.align_1d ? 1 : 0) << 8), sub);
}

// matcher.cpp:269-276 / :341-351: triangulate from the matched pixel (per thread)
__device__ inline bool epi_finish(const DevCam& cam, v3d f_ref, const double* T_cur_ref, int found, double x0, double x1, double* depth)
{
  v3d fc;
  if (found == EPI_FOUND_REFINED) fc = cam2world(cam, x0, x1);               // x = the refined pixel
  else if (found == EPI_FOUND_UV_ONLY) fc = normalized3({x0, x1, 1.0});       // x = uv_best on the unit plane
  else return false;
  return depth_from_triangulation(T_cur_ref, f_ref, fc, depth);
}

// ---------------------------------------------------------------- the LK kernel: thread per job
// Where the result of a job goes (the consumers read plain arrays; no extra "finish" pass for the LK itself).
enum { LK_SINK_EPI = 0, LK_SINK_MATCH_COMPACT = 1, LK_SINK_MATCH_RESULT = 2, LK_SINK_ARRAYS = 3, LK_SINK_SEED = 4 };
struct LkSink {
  int kind;
  EpiSearch* search;              // LK_SINK_EPI: found / px_cur / h_inv of query `item`
  SeedMatch* seed_match;          // LK_SINK_SEED: found / xy of seed `item`
  double* px_out; int* ok_out;    // LK_SINK_MATCH_COMPACT (level-0 pixels) and LK_SINK_ARRAYS (pixels at the image's scale)
  svob200_match_result* mres;     // LK_SINK_MATCH_RESULT
  double* h_inv_out;              // LK_SINK_ARRAYS (may be null)
  const uint8_t* patches;         // LK_SINK_ARRAYS: caller-provided 8x8 reference patches, 64 B per job (else the centre of pwb)
};

__global__ void __launch_bounds__(LK_T, LK_CTAS) lk_refine_kernel(const DevFrame* frames, int cur_slot, const LkJob* jobs, const int* job_count,
                                                         int n_max, int n_iter, LkSink sink)
{
  __shared__ uint32_t s_d[64 * LK_T];
  const int j = blockIdx.x * LK_T + threadIdx.x;
  int n = n_max;
  if (job_count) { const int c = *job_count; n = c < n_max ? c : n_max; }
  if (j >= n) return;
  const uint4* q = reinterpret_cast<const uint4*>(&jobs[j]);
  uint32_t w[25];
  const uint4 a0 = q[0], a1 = q[1], a2 = q[2], a3 = q[3], a4 = q[4], a5 = q[5], a6 = q[6], a7 = q[7];
  w[0] = a0.x; w[1] = a0.y; w[2] = a0.z; w[3] = a0.w; w[4] = a1.x; w[5] = a1.y; w[6] = a1.z; w[7] = a1.w;
  w[8] = a2.x; w[9] = a2.y; w[10] = a2.z; w[11] = a2.w; w[12] = a3.x; w[13] = a3.y; w[14] = a3.z; w[15] = a3.w;
  w[16] = a4.x; w[17] = a4.y; w[18] = a4.z; w[19] = a4.w; w[20] = a5.x; w[21] = a5.y; w[22] = a5.z; w[23] = a5.w;
  w[24] = a6.x;
  float u = __uint_as_float(a6.y), v = __uint_as_float(a6.z);
  const float dirx = __uint_as_float(a6.w), diry = __uint_as_float(a7.x);
  const int item = (int)a7.y, image = (int)a7.z, level_mode = (int)a7.w;
  if (level_mode < 0) return;
  const int L = level_mode & 0xff, mode1d = (level_mode >> 8) & 1;
  uint32_t rp[16];
  if (sink.kind == LK_SINK_ARRAYS && sink.patches) {
    const uint4* pq = reinterpret_cast<const uint4*>(sink.patches + 64 * (size_t)j);
    const uint4 b0 = pq[0], b1 = pq[1], b2 = pq[2], b3 = pq[3];
    rp[0] = b0.x; rp[1] = b0.y; rp[2] = b0.z; rp[3] = b0.w; rp[4] = b1.x; rp[5] = b1.y; rp[6] = b1.z; rp[7] = b1.w;
    rp[8] = b2.x; rp[9] = b2.y; rp[10] = b2.z; rp[11] = b2.w; rp[12] = b3.x; rp[13] = b3.y; rp[14] = b3.z; rp[15] = b3.w;
  } else {
    // Matcher::createPatchFromPatchWithBorder (matcher.cpp:138-147): the 8x8 centre of the 10x10 template
#pragma unroll
    for (int y = 0; y < 8; ++y) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = (y + 1) * 10 + 1 + 4 * h;
        rp[2 * y + h] = (uint32_t)reg_byte(w, k) | ((uint32_t)reg_byte(w, k + 1) << 8) | ((uint32_t)reg_byte(w, k + 2) << 16) | ((uint32_t)reg_byte(w, k + 3) << 24);
      }
    }
  }
  const DevFrame& cur = frames[cur_slot];
  const uint8_t* img = cur.lvl[L] + (size_t)image * cur.img_stride[L];
  const int pitch = cur.pitch[L], cols = cur.w[L], rows = cur.h[L];
  uint32_t* sd = s_d + threadIdx.x;
  double h_inv = 0.0;
  bool ok;
  if (mode1d) ok = lk_align1d(img, pitch, cols, rows, dirx, diry, w, rp, n_iter, u, v, h_inv, sd);
  else ok = lk_align2d(img, pitch, cols, rows, w, rp, n_iter, u, v, sd);
  const double s = (double)(1 << L);
  if (sink.kind == LK_SINK_SEED) {
    if (ok) { SeedMatch* e = &sink.seed_match[item]; e->xy[0] = (double)u * s; e->xy[1] = (double)v * s; e->found = EPI_FOUND_REFINED; }
  } else if (sink.kind == LK_SINK_EPI) {
    EpiSearch* e = &sink.search[item];
    e->h_inv = h_inv;
    if (ok) { e->px_cur[0] = (double)u * s; e->px_cur[1] = (double)v * s; e->found = EPI_FOUND_REFINED; }
  } else if (sink.kind == LK_SINK_MATCH_COMPACT) {
    sink.px_out[2 * item] = (double)u * s; sink.px_out[2 * item + 1] = (double)v * s;      // written whether or not LK converged (matcher.cpp:200)
    sink.ok_out[item] = ok ? 1 : 0;
  } else if (sink.kind == LK_SINK_MATCH_RESULT) {
    svob200_match_result* R = &sink.mres[item];
    R->px_cur[0] = (double)u * s; R->px_cur[1] = (double)v * s; R->success = ok ? 1 : 0; R->h_inv = h_inv;
  } else {
    sink.px_out[2 * item] = (double)u; sink.px_out[2 * item + 1] = (double)v;
    sink.ok_out[item] = ok ? 1 : 0;
    if (sink.h_inv_out) sink.h_inv_out[item] = h_inv;
  }
}

cudaError_t launch_lk_refine(const DevFrame* d_frames, int cur_slot, const LkJob* d_jobs, const int* d_count, int n_max, int n_iter, const LkSink& sink,
                             cudaStream_t s, long long* launches)
{
  if (n_max <= 0) return cudaSuccess;
  lk_refine_kernel<<<(n_max + LK_T - 1) / LK_T, LK_T, 0, s>>>(d_frames, cur_slot, d_jobs, d_count, n_max, n_iter, sink);
  ++*launches;
  return cudaGetLastError();
}

// ---------------------------------------------------------------- depth filter: DepthFilter::updateSeeds loop body
// (depth_filter.cpp:250-340) as four kernels over all seeds: geometry (thread), search (8-lane group), LK (thread), update (thread).
//
// HBM traffic per seed is what bounds the two thread-per-seed kernels (ncu r1f: 1.46 + 1.27 GB per 3.1 M seeds, 73-89 % of the
// HBM peak), so the records are kept small:
//   * where a seed's reference feature lives is a template parameter: the caller's svob200_feature_ref records + one keyframe
//     pose per seed (svob200_seeds_update), or the tracker's 64-byte SeedRef + a table of relative poses indexed by
//     (keyframe, image), refreshed by one tiny kernel per step (the poses are shared by all the seeds of an image);
//   * the geometry kernel writes ONE record per seed, the search task; the finish kernel reads its 16-byte head (flags, levels,
//     epi_length) instead of a 128-byte cold record and a 32-byte pre record;
//   * the search / LK kernels hand over a 32-byte SeedMatch instead of the 64-byte EpiSearch.
// Per seed: geometry reads 64 + 20 B and writes 128 B; finish reads 64 + 20 + 32 + 32 B and writes 20 + 48 B.

// what a seed needs of the two frame poses
struct SeedPoses { double T_ref_cur[7], T_cur_ref[7], T_cur_ref_m[7]; double px_error_angle; };

// T_ref_cur = ref.T_f_w * cur.T_f_w^-1 (depth_filter.cpp:263), its inverse, the matcher's T_cur_ref = cur.T_f_w * ref.T_f_w^-1
// (matcher.cpp:216) and the pixel error angle of depth_filter.cpp:245-247
__device__ __forceinline__ void seed_relative_poses(const DevCam& cam, const double* T_ref_w, const double* T_cur_w, SeedPoses& P)
{
  double inv[7];
  se3_inverse(T_cur_w, inv);
  se3_mul(T_ref_w, inv, P.T_ref_cur);
  se3_inverse(P.T_ref_cur, P.T_cur_ref);
  se3_inverse(T_ref_w, inv);
  se3_mul(T_cur_w, inv, P.T_cur_ref_m);
  const double focal_length = fabs(cam.fx);
  P.px_error_angle = atan(1.0 / (2.0 * focal_length)) * 2.0;
}

// the caller's records (svob200_seeds_update): Feature as given, T_ref_w per seed; poses derived per seed
struct SeedSrcApi {
  const svob200_feature_ref* ftrs; const double* T_ref_w; const double* T_cur_w;
  __device__ __forceinline__ RefFtr get(int i) const { return ref_ftr_of(ftrs[i]); }
  __device__ __forceinline__ void poses(const DevCam& cam, int i, const RefFtr& f, SeedPoses& P) const
  {
    seed_relative_poses(cam, T_ref_w + 7 * (size_t)i, T_cur_w + 7 * (size_t)f.cur_image, P);
  }
  __device__ __forceinline__ int early_status(const RefFtr&) const { return 0; }
  __device__ __forceinline__ void erase(int) const {}
};
// the tracker's compact records: keyframe k of image b lives in frame slot kf_slot[k]; its poses relative to the current
// frame are row (k * batch + b) of the table seed_pose_table_kernel refreshed
struct SeedSrcCompact {
  SeedRef* refs; const SeedPoseRec* table; const int* kf_slot; int batch;
  const int* batch_counter;              // Seed::batch_counter of every sequence (one DepthFilter each), for the ageing rule
  int max_n_kfs;                         // DepthFilter::Options::max_n_kfs
  __device__ __forceinline__ RefFtr get(int i) const
  {
    const uint4* q = reinterpret_cast<const uint4*>(&refs[i]);
    const uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    RefFtr f;
    f.px[0] = __hiloint2double((int)a.y, (int)a.x); f.px[1] = __hiloint2double((int)a.w, (int)a.z);
    f.f = {__hiloint2double((int)b.y, (int)b.x), __hiloint2double((int)b.w, (int)b.z), __hiloint2double((int)c.y, (int)c.x)};
    f.ref_image = f.cur_image = (int)c.z;
    f.level = (int)(c.w & 0xffu); f.type = 0; f.grad[0] = 1.0; f.grad[1] = 0.0;
    f.kf = (int)((c.w >> 8) & 0xffu);
    f.batch_id = (int)(c.w >> 16);
    f.state = (int)(reinterpret_cast<const uint8_t*>(&refs[i])[48]);      // (plain load: the slot may have been filled since the last kernel)
    f.ref_slot = __ldg(&kf_slot[f.kf]);
    return f;
  }
  // -1: empty slot; SVOB200_SEED_TOO_OLD: "check if seed is not already too old" (depth_filter.cpp:258-261); 0: update it
  __device__ __forceinline__ int early_status(const RefFtr& f) const
  {
    if (f.state != 0) return -1;
    return (__ldg(&batch_counter[f.ref_image]) - f.batch_id) > max_n_kfs ? SVOB200_SEED_TOO_OLD : 0;
  }
  __device__ __forceinline__ void erase(int i) const { reinterpret_cast<uint8_t*>(&refs[i])[48] = 1; }
  __device__ __forceinline__ void poses(const DevCam&, int, const RefFtr& f, SeedPoses& P) const
  {
    // 176 bytes shared by all the seeds of an image: consecutive threads read the same row (L1 broadcast)
    const double2* q = reinterpret_cast<const double2*>(&table[(size_t)f.kf * batch + f.ref_image]);
    double v[22];
#pragma unroll
    for (int k = 0; k < 11; ++k) { const double2 d = __ldg(q + k); v[2 * k] = d.x; v[2 * k + 1] = d.y; }
#pragma unroll
    for (int k = 0; k < 7; ++k) { P.T_ref_cur[k] = v[k]; P.T_cur_ref[k] = v[7 + k]; P.T_cur_ref_m[k] = v[14 + k]; }
    P.px_error_angle = v[21];
  }
};

// one thread per (keyframe, image) of the range: the pose table of SeedSrcCompact
__global__ void seed_pose_table_kernel(DevCam cam, int batch, int n_kfs, int image0, int n_images, const double* T_kf_w, const double* T_cur_w,
                                       SeedPoseRec* table)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_kfs * n_images) return;
  const int k = i / n_images, b = image0 + (i - k * n_images);
  SeedPoses P;
  seed_relative_poses(cam, T_kf_w + 7 * ((size_t)k * batch + b), T_cur_w + 7 * (size_t)b, P);
  SeedPoseRec* r = &table[(size_t)k * batch + b];
  for (int j = 0; j < 7; ++j) { r->T_ref_cur[j] = P.T_ref_cur[j]; r->T_cur_ref[j] = P.T_cur_ref[j]; r->T_cur_ref_m[j] = P.T_cur_ref_m[j]; }
  r->px_error_angle = P.px_error_angle;
}

#ifndef SEEDS_GEOM_CTAS
#define SEEDS_GEOM_CTAS 6
#endif
// resident CTAs per SM (measured per 3.1 M seeds): geometry 6 CTAs (78 registers) 0.203 ms, 8 (64, spills) 0.204; finish 6 (76) 0.185 ms, 8 (64, 56 B of spills) 0.168
#ifndef SEEDS_FINISH_CTAS
#define SEEDS_FINISH_CTAS 8
#endif
// phase 1: thread per seed — visibility, inverse-depth range, epipolar geometry -> the search task
// (occupancy: capping the registers for 6 / 8 CTAs spills and measured slower; the kernel is bound by its record traffic)
template <class SRC>
__global__ void __launch_bounds__(128, SEEDS_GEOM_CTAS) seeds_geom_kernel(DevCam cam, int n, SRC src, svob200_matcher_opts o,
                                                         const svob200_seed* seeds, SearchTask* tasks, int* job_count)
{
  // the 128-byte task of a seed goes through shared memory (one padded slot per thread) so that a warp writes it as
  // 512-byte contiguous requests instead of 32 scattered 16-byte pieces per store instruction
  struct Slot { uint4 q[9]; };                                       // 8 used; 144-byte stride: conflict-free 16-byte accesses
  __shared__ Slot s_task[4][32];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (i == 0) *job_count = 0;                                        // consumed by the search kernel that follows on the stream
  const bool valid = i < n;
  bool has_geom = false;
  if (valid) {
    const RefFtr f = src.get(i);
    const svob200_seed s = seeds[i];
    SeedPoses P;
    int status = src.early_status(f);
    if (status == 0) {
      src.poses(cam, i, f, P);
      const double inv_mu = 1.0 / s.mu;
      const v3d xyz_f = se3_transform(P.T_cur_ref, {inv_mu * f.f.x, inv_mu * f.f.y, inv_mu * f.f.z});
      if (xyz_f.z < 0.0) status = SVOB200_SEED_BEHIND;
      else {
        double pxf, pyf;
        world2cam(cam, xyz_f, pxf, pyf);
        if (!in_frame(cam, (int)pxf, (int)pyf, 0)) status = SVOB200_SEED_NOT_IN_FRAME;
      }
    }
    if (status == 0) {
      const float z_inv_min = s.mu + sqrtf(s.sigma2);
      const float z_inv_max = fmaxf(s.mu - sqrtf(s.sigma2), 0.00000001f);
      EpiGeom g;
      epi_geometry(cam, f, P.T_cur_ref_m, 1.0 / s.mu, 1.0 / z_inv_min, 1.0 / z_inv_max, o, &g);
      store_geometry(g, f, !g.reject && g.mode != EPI_MODE_NONE, isnan(z_inv_min) ? ST_ZMIN_NAN : 0u, nullptr,
                     reinterpret_cast<SearchTask*>(&s_task[warp][lane]));
      has_geom = true;
    } else s_task[warp][lane].q[0] = make_uint4(status < 0 ? (uint32_t)ST_FREE : ((uint32_t)status << ST_STATUS_SHIFT), 0, 0, 0);   // nothing to search
  }
  const unsigned wrote = __ballot_sync(0xffffffffu, has_geom);
  const unsigned skip = __ballot_sync(0xffffffffu, valid && !has_geom);
  __syncwarp();                                                                // the slots written above are read by other lanes
  const size_t i0 = (size_t)(i - lane);                                        // first seed of this warp
  uint4* gtask = reinterpret_cast<uint4*>(tasks + i0);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int e = k * 32 + lane, r = e >> 3, j = e & 7;
    if (((wrote >> r) & 1u) || (((skip >> r) & 1u) && j == 0)) gtask[e] = s_task[warp][r].q[j];
  }
}

// geometry of stand-alone epipolar queries (svob200_epipolar_match): T_cur_ref and the depth range come from the caller
__global__ void __launch_bounds__(128) epi_geom_kernel(DevCam cam, int n, const svob200_feature_ref* ftrs, const double* d,
                                                       svob200_matcher_opts o, EpiCold* cold, SearchTask* tasks, int* job_count)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *job_count = 0;
  if (i >= n) return;
  const RefFtr f = ref_ftr_of(ftrs[i]);
  EpiGeom g;
  epi_geometry(cam, f, ftrs[i].T_cur_ref, d[3 * i], d[3 * i + 1], d[3 * i + 2], o, &g);
  store_geometry(g, f, !g.reject, 0u, &cold[i], &tasks[i]);           // stand-alone queries always warp the patch (unless rejected)
}

// phase 2: 8-lane group per item, PERSISTENT — the grid is sized to the machine and every group strides over the
// items; the packed task of the next item is fetched (one coalesced 128-byte load) while the current one is processed,
// and LK job slots are reserved JOB_BATCH at a time, so neither a DRAM round trip nor an atomic sits on the critical
// path of an item.  api_results != nullptr: stand-alone queries, which also return the warped patch.
__global__ void __launch_bounds__(128, SEARCH_CTAS) epi_search_kernel(const DevFrame* frames, int cur_slot, DevCam cam, int n, svob200_matcher_opts o,
                                                            const SearchTask* tasks, EpiSearch* search, SeedMatch* seed_match, LkJob* jobs,
                                                            int* job_count, svob200_epi_result* api_results)
{
  __shared__ EpiGroupSmem SM[4 * GPW];
  __shared__ float2 s_tap[TAP_TABLE];
  fill_tap_table(s_tap);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (GL - 1), grp = lane / GL, gbase = grp * GL;
  const unsigned gmask = ((1u << GL) - 1u) << gbase;
  EpiGroupSmem* S = &SM[warp * GPW + grp];
  const int stride = gridDim.x * 4 * GPW;              // items per sweep of the persistent grid
  int slot_base = 0, slots_left = 0;
  int i = (blockIdx.x * 4 + warp) * GPW + grp;
  // (an L2 prefetch of the NEXT item's reference window, issued one item ahead, was measured: 2.19 -> 2.41 ms; the kernel is
  //  bound by issue slots and dependent arithmetic at 6 resident CTAs per SM, not by the DRAM latency of the taps)
  uint4 next = (i < n) ? __ldg(reinterpret_cast<const uint4*>(&tasks[i]) + sub) : make_uint4(0, 0, 0, 0);
  for (; i < n; i += stride) {
    const uint4 tq = next;
    if (i + stride < n) next = __ldg(reinterpret_cast<const uint4*>(&tasks[i + stride]) + sub);
    if (!(task_word(tq, ST_FLAGS, gbase, gmask) & ST_ACTIVE)) continue;
    epi_search_item(frames, cur_slot, cam, o, tq, i, S, sub, gbase, gmask, jobs, job_count, slot_base, slots_left, search, seed_match, api_results, s_tap);
    __syncwarp(gmask);
  }
  // reserved but unused job slots become empty jobs
  for (int k = sub; k < slots_left; k += GL) jobs[slot_base + (JOB_BATCH - slots_left) + k].level_mode = -1;
}

// phase 4: thread per seed — triangulation, tau, Gaussian x Beta update, status
template <class SRC>
__global__ void __launch_bounds__(128, SEEDS_FINISH_CTAS) seeds_finish_kernel(DevCam cam, int n, SRC src, double conv_thresh,
                                                           const SearchTask* tasks, const SeedMatch* match, svob200_seed* seeds,
                                                           svob200_seed_obs* obs)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 head = __ldg(reinterpret_cast<const uint4*>(&tasks[i]));          // flags, levels, epi_length
  const uint32_t flags = head.x;
  const int status0 = (int)((flags >> ST_STATUS_SHIFT) & 7u);
  svob200_seed_obs ob;
  ob.status = status0; ob.search_level = 0; ob.zmssd_best = 2000 * 64; ob.n_evals = 0; ob.z = 0; ob.px_cur[0] = ob.px_cur[1] = 0; ob.epi_length = 0;
  if (status0 == SVOB200_SEED_TOO_OLD) src.erase(i);                          // it = seeds_.erase(it) (depth_filter.cpp:259)
  if (status0 == 0 && !(flags & ST_FREE)) {
    const RefFtr f = src.get(i);
    SeedMatch sr;
    if (flags & ST_ACTIVE) {
      const uint4* q = reinterpret_cast<const uint4*>(&match[i]);
      const uint4 a = q[0], b = q[1];
      sr.found = (int)a.x; sr.zmssd_best = (int)a.y; sr.n_evals = (int)a.z; sr.xy_valid = (int)a.w;
      sr.xy[0] = __hiloint2double((int)b.y, (int)b.x); sr.xy[1] = __hiloint2double((int)b.w, (int)b.z);
    } else { sr.found = EPI_FOUND_NONE; sr.zmssd_best = 2000 * 64; sr.n_evals = 0; sr.xy_valid = 0; sr.xy[0] = sr.xy[1] = 0; }
    svob200_seed s = seeds[i];
    ob.search_level = (int)(head.y & 0xffu); ob.zmssd_best = sr.zmssd_best; ob.n_evals = sr.n_evals;
    ob.epi_length = __hiloint2double((int)head.w, (int)head.z);
    if (sr.xy_valid) {
      if (sr.found == EPI_FOUND_UV_ONLY) world2cam_uv(cam, sr.xy[0], sr.xy[1], ob.px_cur[0], ob.px_cur[1]);
      else { ob.px_cur[0] = sr.xy[0]; ob.px_cur[1] = sr.xy[1]; }
    }
    SeedPoses P;
    src.poses(cam, i, f, P);
    double z = 0;
    if (!epi_finish(cam, f.f, P.T_cur_ref_m, sr.found, sr.xy[0], sr.xy[1], &z)) {
      s.b++;                                                         // depth_filter.cpp:286
      ob.status = SVOB200_SEED_NO_MATCH;
    } else {
      ob.z = z;
      const double tau = compute_tau(P.T_ref_cur, f.f, z, P.px_error_angle);
      const double zmt = z - tau;
      const double tau_inverse = 0.5 * (1.0 / (0.0000001 > zmt ? 0.0000001 : zmt) - 1.0 / (z + tau));
      update_seed((float)(1. / z), (float)(tau_inverse * tau_inverse), &s);
      if ((double)sqrtf(s.sigma2) < (double)s.z_range / conv_thresh) ob.status = SVOB200_SEED_CONVERGED;
      else if (flags & ST_ZMIN_NAN) ob.status = SVOB200_SEED_NAN_ERASED;
      else ob.status = SVOB200_SEED_UPDATED;
    }
    seeds[i] = s;
  }
  obs[i] = ob;
}

// stand-alone queries: triangulate and fill the scalar fields of svob200_epi_result (patches were written by the search kernel)
__global__ void __launch_bounds__(128) epi_result_kernel(DevCam cam, int n, const svob200_feature_ref* ftrs, const EpiCold* cold,
                                                         const EpiSearch* search, svob200_epi_result* results)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const svob200_feature_ref f = ftrs[i];
  const EpiCold* g = &cold[i];
  const EpiSearch sr = g->reject ? epi_search_none() : search[i];
  if (g->reject) {
    svob200_epi_result* R0 = &results[i];
    for (int k = 0; k < 100; ++k) R0->patch_with_border[k] = 0;
    for (int k = 0; k < 64; ++k) R0->patch[k] = 0;
  }
  double T_cur_ref[7];
  for (int k = 0; k < 7; ++k) T_cur_ref[k] = g->T_cur_ref[k];
  double depth = 0;
  const bool uv = sr.found == EPI_FOUND_UV_ONLY;
  const bool ok = epi_finish(cam, {f.f[0], f.f[1], f.f[2]}, T_cur_ref, sr.found, uv ? sr.uv_best[0] : sr.px_cur[0], uv ? sr.uv_best[1] : sr.px_cur[1], &depth);
  svob200_epi_result* R = &results[i];
  R->success = ok ? 1 : 0; R->search_level = g->L; R->reject = g->reject; R->zmssd_best = sr.zmssd_best;
  R->n_evals = sr.n_evals; R->n_steps = g->n_steps_report; R->depth = ok ? depth : 0.0;
  R->px_cur[0] = sr.px_cur[0]; R->px_cur[1] = sr.px_cur[1];
  R->epi_length = g->epi_length; R->h_inv = sr.h_inv;
  R->epi_dir[0] = g->ex; R->epi_dir[1] = g->ey;
  R->px_cur_valid = sr.px_cur_valid;
  for (int k = 0; k < 4; ++k) R->A_cur_ref[k] = g->A[k];
}

// ---------------------------------------------------------------- findMatchDirect: geometry (thread) + patch warp (warp) + LK job
struct MatchGeom {
  double A[4];                          // A_cur_ref (row-major)
  float a00, a01, a10, a11, pr0, pr1;   // A_ref_cur as float, px_ref at the reference level
  float dir0, dir1;                     // align1D direction for edgelets
  int L, flags;                         // search level; bit 0: in frame, bit 1: warp is finite
};

// matcher.cpp:156-183 up to warpAffine: in-frame test, affine warp matrix (FP64), search level.  Thread per candidate,
// so the double-precision geometry runs lane-parallel.  Candidates that fail the in-frame test get their final
// outputs here and an empty job.
__global__ void __launch_bounds__(128) match_geom_kernel(DevCam cam, int n, const svob200_feature_ref* ftrs, const double* depth_ref,
                                                         const double* px_in, svob200_matcher_opts o, MatchGeom* geom, LkJob* jobs,
                                                         svob200_match_result* results, double* px_out, int* ok_out,
                                                         const uint8_t* active, int* level_out, double* A_out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  MatchGeom g;
  g.A[0] = g.A[1] = g.A[2] = g.A[3] = 0; g.a00 = g.a01 = g.a10 = g.a11 = g.pr0 = g.pr1 = g.dir0 = g.dir1 = 0.f; g.L = 0; g.flags = 0;
  svob200_match_result* R = results ? &results[i] : nullptr;
  // candidates the caller masked out (reprojector: not in frame / no close view, matcher.cpp:161-162) fail without work;
  // their feature record is not read
  const bool is_active = !active || active[i];
  svob200_feature_ref f;
  if (is_active) f = ftrs[i]; else { f.level = 0; f.px[0] = f.px[1] = -1.0; }
  // ref_ftr_->px.cast<int>()/(1<<level), boundary halfpatch_size_+2 (matcher.cpp:165-167)
  const int pxi = (int)f.px[0] / (1 << f.level), pyi = (int)f.px[1] / (1 << f.level);
  if (!is_active || !in_frame_level(cam, pxi, pyi, 6, f.level)) {
    const double px0 = px_in[2 * i], px1 = px_in[2 * i + 1];
    jobs[i].level_mode = -1;
    if (level_out) { level_out[i] = 0; for (int k = 0; k < 4; ++k) A_out[4 * (size_t)i + k] = 0.0; }
    if (ok_out) { ok_out[i] = 0; px_out[2 * i] = px0; px_out[2 * i + 1] = px1; }
    if (R) {
      R->success = 0; R->search_level = 0; R->px_cur[0] = px0; R->px_cur[1] = px1; R->h_inv = 0;
      for (int k = 0; k < 4; ++k) R->A_cur_ref[k] = 0;
      for (int k = 0; k < 100; ++k) R->patch_with_border[k] = 0;
      for (int k = 0; k < 64; ++k) R->patch[k] = 0;
    }
    geom[i] = g;
    return;
  }
  g.flags = 1;
  warp_matrix_affine(cam, f.px, {f.f[0], f.f[1], f.f[2]}, depth_ref[i], f.T_cur_ref, f.level, g.A);
  g.L = best_search_level(g.A, o.max_search_level);
  const double det = g.A[0] * g.A[3] - g.A[2] * g.A[1];
  const double invdet = 1.0 / det;
  g.a00 = (float)(g.A[3] * invdet); g.a01 = (float)(-g.A[1] * invdet); g.a10 = (float)(-g.A[2] * invdet); g.a11 = (float)(g.A[0] * invdet);
  if (!isnan(g.a00)) g.flags |= 2;
  g.pr0 = (float)f.px[0] * pow2_inv_f(f.level); g.pr1 = (float)f.px[1] * pow2_inv_f(f.level);   // / (float)(1 << level), exactly
  if (f.type == 1) {
    double dx = g.A[0] * f.grad[0] + g.A[1] * f.grad[1], dy = g.A[2] * f.grad[0] + g.A[3] * f.grad[1];
    { const double z = dx * dx + dy * dy; if (z > 0) { const double nn = sqrt(z); dx /= nn; dy /= nn; } }
    g.dir0 = (float)dx; g.dir1 = (float)dy;
  }
  if (R) { R->search_level = g.L; R->h_inv = 0; for (int k = 0; k < 4; ++k) R->A_cur_ref[k] = g.A[k]; }
  if (level_out) { level_out[i] = g.L; for (int k = 0; k < 4; ++k) A_out[4 * (size_t)i + k] = g.A[k]; }
  geom[i] = g;
}

struct MatchSmem { __align__(16) uint8_t pwb[112]; };

// matcher.cpp:176-178: warpAffine of the 10x10 patch by a group of 8 lanes (four candidates per warp), then the LK job
__global__ void __launch_bounds__(128) match_prepare_kernel(const DevFrame* frames, int n, const svob200_feature_ref* ftrs,
                                                            const double* px_in, const MatchGeom* geom, LkJob* jobs,
                                                            svob200_match_result* results)
{
  __shared__ MatchSmem SM[4 * GPW];
  __shared__ float2 s_tap[TAP_TABLE];
  fill_tap_table(s_tap);
  __syncthreads();                                       // (before any thread leaves)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (GL - 1), grp = lane / GL;
  const unsigned gmask = ((1u << GL) - 1u) << (grp * GL);
  const int i = (blockIdx.x * 4 + warp) * GPW + grp;
  if (i >= n) return;
  const MatchGeom* gp = &geom[i];
  const int flags = gp->flags;
  if (!(flags & 1)) return;
  MatchSmem* S = &SM[warp * GPW + grp];
  const svob200_feature_ref* fp = &ftrs[i];
  const int level = fp->level, type = fp->type, ref_image = fp->ref_image, cur_image = fp->cur_image, L = gp->L;
  for (int k = sub; k < 28; k += GL) reinterpret_cast<uint32_t*>(S->pwb)[k] = 0;
  __syncwarp(gmask);
  if (flags & 2) {
    const DevFrame& ref = frames[(int)fp->ref_frame_id];
    const uint8_t* rimg = ref.lvl[level] + (size_t)ref_image * ref.img_stride[level];
    warp_patch_10x10<true>(rimg, ref.pitch[level], ref.w[level], ref.h[level], gp->a00, gp->a01, gp->a10, gp->a11, gp->pr0, gp->pr1, L, S->pwb, sub, s_tap);
  }
  __syncwarp(gmask);
  if (results) {
    svob200_match_result* R = &results[i];
    for (int k = sub; k < 100; k += GL) R->patch_with_border[k] = S->pwb[k];
    for (int k = sub; k < 64; k += GL) R->patch[k] = S->pwb[((k >> 3) + 1) * 10 + 1 + (k & 7)];
  }
  const double px0 = px_in[2 * i], px1 = px_in[2 * i + 1];
  emit_lk_job(&jobs[i], S->pwb, (float)(px0 * pow2_inv(L)), (float)(px1 * pow2_inv(L)), gp->dir0, gp->dir1, i, cur_image, L | ((type == 1 ? 1 : 0) << 8), sub);
}

// stand-alone align2D / align1D on caller-provided patches: thread per problem builds the job
__global__ void __launch_bounds__(128) align_jobs_kernel(int level, int n, const int* image, const uint8_t* pwb, const float* dir,
                                                         const double* px, LkJob* jobs)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  LkJob* J = &jobs[i];
  const uint32_t* src = reinterpret_cast<const uint32_t*>(pwb + 100 * (size_t)i);     // 100 * i is a multiple of 4
  uint32_t* dst = reinterpret_cast<uint32_t*>(J->pwb);
  for (int k = 0; k < 25; ++k) dst[k] = src[k];
  J->u = (float)px[2 * i]; J->v = (float)px[2 * i + 1];
  J->dirx = dir ? dir[2 * i] : 0.f; J->diry = dir ? dir[2 * i + 1] : 0.f;
  J->item = i; J->image = image[i]; J->level_mode = level | ((dir ? 1 : 0) << 8);
}

__global__ void update_seed_kernel(int n, const float* x, const float* tau2, svob200_seed* seeds)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  svob200_seed s = seeds[i];
  update_seed(x[i], tau2[i], &s);
  seeds[i] = s;
}

__global__ void compute_tau_kernel(int n, const double* T, const double* f, const double* z, double angle, double* out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = compute_tau(T + 7 * (size_t)i, {f[3 * i], f[3 * i + 1], f[3 * i + 2]}, z[i], angle);
}

// stand-alone warp::getWarpMatrixAffine (matcher.cpp:36-60): thread per item
__global__ void warp_matrix_kernel(DevCam cam, int n, const double* px_ref, const double* f_ref, const double* depth_ref,
                                   const double* T_cur_ref, const int* level_ref, double* A_out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double A[4];
  warp_matrix_affine(cam, px_ref + 2 * i, {f_ref[3 * i], f_ref[3 * i + 1], f_ref[3 * i + 2]}, depth_ref[i], T_cur_ref + 7 * (size_t)i, level_ref[i], A);
  for (int k = 0; k < 4; ++k) A_out[4 * (size_t)i + k] = A[k];
}

// stand-alone warp::warpAffine (matcher.cpp:83-116) for any halfpatch size: thread per patch pixel.
// Leaves the patch untouched when the warp is NaN, like the reference (:94-98).
__global__ void warp_affine_kernel(const uint8_t* img, int pitch, int cols, int rows, double A0, double A1, double A2, double A3,
                                   double px0, double px1, int level_ref, int search_level, int halfpatch, uint8_t* patch)
{
  const int ps = 2 * halfpatch;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ps * ps) return;
  const double det = A0 * A3 - A2 * A1;
  const double invdet = 1.0 / det;
  const float a00 = (float)(A3 * invdet), a01 = (float)(-A1 * invdet);
  const float a10 = (float)(-A2 * invdet), a11 = (float)(A0 * invdet);
  if (isnan(a00)) return;
  const float pr0 = (float)px0 / (float)(1 << level_ref), pr1 = (float)px1 / (float)(1 << level_ref);
  const int y = i / ps, x = i - y * ps;
  float p0 = (float)(x - halfpatch), p1 = (float)(y - halfpatch);
  p0 *= (float)(1 << search_level); p1 *= (float)(1 << search_level);
  const float qx = (a00 * p0 + a01 * p1) + pr0;
  const float qy = (a10 * p0 + a11 * p1) + pr1;
  uint8_t v = 0;
  if (!(qx < 0 || qy < 0 || qx >= cols - 1 || qy >= rows - 1)) v = (uint8_t)interpolate_8u(img, pitch, qx, qy);
  patch[i] = v;
}

// stand-alone depthFromTriangulation (matcher.cpp:123-136): thread per item
__global__ void triangulate_kernel(int n, const double* T, const double* f_ref, const double* f_cur, double* depth, int* ok)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double d = 0.0;
  const bool r = depth_from_triangulation(T + 7 * (size_t)i, {f_ref[3 * i], f_ref[3 * i + 1], f_ref[3 * i + 2]},
                                          {f_cur[3 * i], f_cur[3 * i + 1], f_cur[3 * i + 2]}, &d);
  ok[i] = r ? 1 : 0;
  if (r) depth[i] = d;
}

}  // namespace

// ---------------------------------------------------------------- launchers
static inline size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t lk_jobs_bytes(int n) { return up256((size_t)(n > 0 ? n : 1) * sizeof(LkJob)) + 256; }

cudaError_t launch_align_patches(const DevFrame* d_frames, int slot, int level, int n, const int* d_image, const uint8_t* d_pwb, const uint8_t* d_patch,
                                 const float* d_dir, int n_iter, double* d_px, int* d_converged, double* d_h_inv, void* d_scratch,
                                 cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  LkJob* jobs = static_cast<LkJob*>(d_scratch);
  align_jobs_kernel<<<(n + 127) / 128, 128, 0, s>>>(level, n, d_image, d_pwb, d_dir, d_px, jobs);
  ++*launches;
  if (cudaError_t e = cudaGetLastError()) return e;
  LkSink sink{};
  sink.kind = LK_SINK_ARRAYS; sink.px_out = d_px; sink.ok_out = d_converged; sink.h_inv_out = d_h_inv; sink.patches = d_patch;
  return launch_lk_refine(d_frames, slot, jobs, nullptr, n, n_iter, sink, s, launches);
}

size_t match_scratch_bytes(int n)
{
  const size_t m = (size_t)(n > 0 ? n : 1);
  return up256(m * sizeof(LkJob)) + up256(m * sizeof(MatchGeom)) + 256;
}

// Matcher::findMatchDirect for n candidates: geometry (thread) -> patch warp (warp) -> LK (thread).
// results: full records (API) or nullptr; px_out / ok_out: compact outputs (tracker) or nullptr.
// The scratch was sized for scratch_total candidates; this call covers [first, first + n) of it (all other
// pointers already point at candidate `first`).  marks: optional 2 events recorded between the three kernels.
cudaError_t launch_match_direct(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs,
                                const double* d_depth_ref, const double* d_px_in, svob200_matcher_opts opts, svob200_match_result* d_results,
                                double* d_px_out, int* d_ok_out, void* d_scratch, int scratch_total, int first, cudaStream_t s, long long* launches,
                                cudaEvent_t* marks, const uint8_t* d_active, int* d_level_out, double* d_A_out)
{
  if (n <= 0) return cudaSuccess;
  const size_t m = (size_t)(scratch_total > 0 ? scratch_total : 1);
  char* p = static_cast<char*>(d_scratch);
  LkJob* jobs = reinterpret_cast<LkJob*>(p) + first; p += up256(m * sizeof(LkJob));
  MatchGeom* geom = reinterpret_cast<MatchGeom*>(p) + first;
  match_geom_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_ftrs, d_depth_ref, d_px_in, opts, geom, jobs, d_results, d_px_out, d_ok_out,
                                                    d_active, d_level_out, d_A_out);
  if (marks) cudaEventRecord(marks[0], s);
  match_prepare_kernel<<<(n + 4 * GPW - 1) / (4 * GPW), 128, 0, s>>>(d_frames, n, d_ftrs, d_px_in, geom, jobs, d_results);
  *launches += 2;
  if (cudaError_t e = cudaGetLastError()) return e;
  if (marks) cudaEventRecord(marks[1], s);
  LkSink sink{};
  if (d_results) { sink.kind = LK_SINK_MATCH_RESULT; sink.mres = d_results; }
  else { sink.kind = LK_SINK_MATCH_COMPACT; sink.px_out = d_px_out; sink.ok_out = d_ok_out; }
  return launch_lk_refine(d_frames, cur_slot, jobs, nullptr, n, opts.align_max_iter, sink, s, launches);
}

// persistent grid of the search kernel: SEARCH_CTAS CTAs of 4 warps (16 groups) per SM
static int search_sms()
{
  // (initialised once, thread-safely: two contexts may be driven from two threads)
  static const int sms = [] { int dev = 0, n = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); return n > 0 ? n : 148; }();
  return sms;
}
// Grid of the search kernel = SEARCH_CTAS resident CTAs per SM times `waves`: 1 = persistent (every CTA lives for the whole kernel);
// more = CTAs that retire during the kernel, so that CTAs of a higher-priority stream (the tracking chain running beside an
// asynchronous depth filter) find free slots.  The LK job list (job_capacity) is sized for grids of up to SEARCH_MAX_WAVES waves:
// 4 leaves headroom over the 2 waves seeds_update_impl launches.
constexpr int SEARCH_MAX_WAVES = 4;
static int search_grid(int n, int waves = 1)
{
  const int want = (n + 4 * GPW - 1) / (4 * GPW), cap = search_sms() * SEARCH_CTAS * waves;
  return want < cap ? want : cap;
}
// LK jobs are compacted; a group reserves JOB_BATCH slots at a time, so the list can exceed n by the unused tail of every group
static size_t job_capacity(size_t m) { return m + (size_t)JOB_BATCH * 4 * GPW * ((size_t)search_sms() * 8 * SEARCH_MAX_WAVES + 8); }

size_t epipolar_scratch_bytes(int n)
{
  const size_t m = (size_t)(n > 0 ? n : 1);
  return up256(m * sizeof(EpiCold)) + up256(m * sizeof(SearchTask)) + up256(m * sizeof(EpiSearch)) + up256(job_capacity(m) * sizeof(LkJob)) + 512;
}

cudaError_t launch_epipolar(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs, const double* d_d,
                            svob200_matcher_opts opts, svob200_epi_result* d_results, void* d_scratch, cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  const size_t m = (size_t)n;
  char* p = static_cast<char*>(d_scratch);
  EpiCold* cold = reinterpret_cast<EpiCold*>(p); p += up256(m * sizeof(EpiCold));
  SearchTask* tasks = reinterpret_cast<SearchTask*>(p); p += up256(m * sizeof(SearchTask));
  EpiSearch* search = reinterpret_cast<EpiSearch*>(p); p += up256(m * sizeof(EpiSearch));
  LkJob* jobs = reinterpret_cast<LkJob*>(p); p += up256(job_capacity(m) * sizeof(LkJob));
  int* count = reinterpret_cast<int*>(p);
  epi_geom_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_ftrs, d_d, opts, cold, tasks, count);
  epi_search_kernel<<<search_grid(n), 128, 0, s>>>(d_frames, cur_slot, cam, n, opts, tasks, search, nullptr, jobs, count, d_results);
  *launches += 2;
  if (cudaError_t e = cudaGetLastError()) return e;
  LkSink sink{};
  sink.kind = LK_SINK_EPI; sink.search = search;
  if (cudaError_t e = launch_lk_refine(d_frames, cur_slot, jobs, count, (int)job_capacity(m), opts.align_max_iter, sink, s, launches)) return e;
  epi_result_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_ftrs, cold, search, d_results);
  ++*launches;
  return cudaGetLastError();
}

size_t seeds_scratch_bytes(int n)
{
  const size_t m = (size_t)(n > 0 ? n : 1);
  return up256(m * sizeof(SearchTask)) + up256(m * sizeof(SeedMatch)) + up256(job_capacity(m) * sizeof(LkJob)) + 512;
}

// DepthFilter::updateSeeds for n seeds: geometry (thread) -> search (group, persistent) -> LK (thread per job) -> update (thread).
// The scratch was sized for scratch_total seeds and is indexed by absolute seed number; `src`, d_seeds and d_obs already point at
// seed `first`.  marks: optional 3 events recorded between the four kernels.
template <class SRC>
static cudaError_t seeds_update_impl(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const SRC& src,
                                     svob200_matcher_opts opts, double conv_thresh, svob200_seed* d_seeds, svob200_seed_obs* d_obs, void* d_scratch,
                                     int scratch_total, int first, cudaStream_t s, long long* launches, cudaEvent_t* marks)
{
  if (n <= 0) return cudaSuccess;
  const size_t m = (size_t)(scratch_total > 0 ? scratch_total : 1);
  char* p = static_cast<char*>(d_scratch);
  SearchTask* tasks = reinterpret_cast<SearchTask*>(p) + first; p += up256(m * sizeof(SearchTask));
  SeedMatch* match = reinterpret_cast<SeedMatch*>(p) + first; p += up256(m * sizeof(SeedMatch));
  LkJob* jobs = reinterpret_cast<LkJob*>(p) + first; p += up256(job_capacity(m) * sizeof(LkJob));
  int* count = reinterpret_cast<int*>(p);
  seeds_geom_kernel<SRC><<<(n + 127) / 128, 128, 0, s>>>(cam, n, src, opts, d_seeds, tasks, count);
  if (marks) cudaEventRecord(marks[0], s);
  // small seed lists (the shard of an 8-GPU run): two waves of CTAs instead of a persistent grid, so that the tracking chain of the next
  // frame (higher-priority stream) gets SM slots while the search is running: 0.595 -> 0.564 ms per step at 512 sequences; bigger lists
  // fill the machine either way and lose 3-8 % to the extra CTA turnover, so they stay persistent
  const int waves = n <= 450000 ? 2 : 1;
  epi_search_kernel<<<search_grid(n, waves), 128, 0, s>>>(d_frames, cur_slot, cam, n, opts, tasks, nullptr, match, jobs, count, nullptr);
  if (marks) cudaEventRecord(marks[1], s);
  *launches += 2;
  if (cudaError_t e = cudaGetLastError()) return e;
  LkSink sink{};
  sink.kind = LK_SINK_SEED; sink.seed_match = match;
  if (cudaError_t e = launch_lk_refine(d_frames, cur_slot, jobs, count, (int)job_capacity((size_t)n), opts.align_max_iter, sink, s, launches)) return e;
  if (marks) cudaEventRecord(marks[2], s);
  seeds_finish_kernel<SRC><<<(n + 127) / 128, 128, 0, s>>>(cam, n, src, conv_thresh, tasks, match, d_seeds, d_obs);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_seeds_update(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, const svob200_feature_ref* d_ftrs,
                                const double* d_T_ref_w, const double* d_T_cur_w, svob200_matcher_opts opts, double conv_thresh,
                                svob200_seed* d_seeds, svob200_seed_obs* d_obs, void* d_scratch, int scratch_total, int first,
                                cudaStream_t s, long long* launches, cudaEvent_t* marks)
{
  SeedSrcApi src{d_ftrs, d_T_ref_w, d_T_cur_w};
  return seeds_update_impl(d_frames, cur_slot, cam, n, src, opts, conv_thresh, d_seeds, d_obs, d_scratch, scratch_total, first, s, launches, marks);
}

// rows (keyframe k, image b), b in [image0, image0 + n_images), of the pose table the compact seed kernels read
cudaError_t launch_seed_pose_table(const DevCam& cam, int batch, int n_kfs, int image0, int n_images, const double* d_T_kf_w, const double* d_T_cur_w,
                                   SeedPoseRec* d_pose_table, cudaStream_t s, long long* launches)
{
  const int rows = n_kfs * n_images;
  if (rows <= 0) return cudaSuccess;
  seed_pose_table_kernel<<<(rows + 127) / 128, 128, 0, s>>>(cam, batch, n_kfs, image0, n_images, d_T_kf_w, d_T_cur_w, d_pose_table);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_seeds_update_compact(const DevFrame* d_frames, int cur_slot, const DevCam& cam, int n, SeedRef* d_refs,
                                        const int* d_kf_slot, int batch, const SeedPoseRec* d_pose_table, const int* d_batch_counter, int max_n_kfs,
                                        svob200_matcher_opts opts, double conv_thresh,
                                        svob200_seed* d_seeds, svob200_seed_obs* d_obs, void* d_scratch, int scratch_total, int first,
                                        cudaStream_t s, long long* launches, cudaEvent_t* marks)
{
  SeedSrcCompact src{d_refs, d_pose_table, d_kf_slot, batch, d_batch_counter, max_n_kfs};
  return seeds_update_impl(d_frames, cur_slot, cam, n, src, opts, conv_thresh, d_seeds, d_obs, d_scratch, scratch_total, first, s, launches, marks);
}

cudaError_t launch_update_seed(int n, const float* d_x, const float* d_tau2, svob200_seed* d_seeds, cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  update_seed_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, d_x, d_tau2, d_seeds);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_compute_tau(int n, const double* d_T, const double* d_f, const double* d_z, double angle, double* d_out,
                               cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  compute_tau_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, d_T, d_f, d_z, angle, d_out);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_warp_matrix(const DevCam& cam, int n, const double* d_px_ref, const double* d_f_ref, const double* d_depth_ref,
                               const double* d_T_cur_ref, const int* d_level_ref, double* d_A_out, cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  warp_matrix_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_px_ref, d_f_ref, d_depth_ref, d_T_cur_ref, d_level_ref, d_A_out);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_warp_affine(const uint8_t* d_img, int pitch, int cols, int rows, const double* A, const double* px_ref, int level_ref,
                               int search_level, int halfpatch, uint8_t* d_patch, cudaStream_t s, long long* launches)
{
  const int n = 4 * halfpatch * halfpatch;
  if (n <= 0) return cudaSuccess;
  warp_affine_kernel<<<(n + 127) / 128, 128, 0, s>>>(d_img, pitch, cols, rows, A[0], A[1], A[2], A[3], px_ref[0], px_ref[1], level_ref,
                                                     search_level, halfpatch, d_patch);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_triangulate(int n, const double* d_T, const double* d_f_ref, const double* d_f_cur, double* d_depth, int* d_ok,
                               cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  triangulate_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, d_T, d_f_ref, d_f_cur, d_depth, d_ok);
  ++*launches;
  return cudaGetLastError();
}
