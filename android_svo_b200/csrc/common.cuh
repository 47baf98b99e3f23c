// common.cuh — shared device structs and math for libsvob200 (sm_100a).
//
// Parity rule for this library: it is compiled with -fmad=false and uses IEEE
// division / sqrt, and every float / double expression keeps the reference's
// operation order and float<->double promotions (the reference's x86-64 host
// build has no FMA).  That makes warped patches, residual terms, ZMSSD inputs
// and the whole geometry bit-identical to the CPU reference; only parallel
// reductions of doubles and libm transcendentals (sin/cos/acos/atan/exp) are
// tolerance-matched.  Reference paths are relative to
// /root/reference/app/src/main/cpp/svo.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/svob200.h"

#define SVOB_MAXL SVOB200_MAX_LEVELS

// Device pyramid of a frame batch.  Level l of image b starts at
// lvl[l] + b * img_stride[l]; rows are pitch[l] bytes apart (pitch is a multiple
// of 64 so every row start is sector- and uint4-aligned).
struct DevFrame {
  uint8_t* lvl[SVOB_MAXL];
  int w[SVOB_MAXL], h[SVOB_MAXL], pitch[SVOB_MAXL];
  unsigned long long img_stride[SVOB_MAXL];
  int n_levels, batch;
};

struct DevCam { int width, height; double fx, fy, cx, cy; };

__host__ __device__ inline int align_up_i(int v, int a) { return (v + a - 1) / a * a; }

// (int) of a double the way x86 cvttsd2si does it (NaN / out of range -> INT_MIN); Eigen's cast<int>() on the host
__device__ __forceinline__ int x86_d2i(double v) { return (v > -2147483649.0 && v < 2147483648.0) ? (int)v : (int)0x80000000; }

// Seed ctor depth_filter.cpp:36-45
__host__ __device__ inline svob200_seed seed_prior(float depth_mean, float depth_min)
{
  svob200_seed s;
  s.a = 10; s.b = 10; s.mu = (float)(1.0 / depth_mean); s.z_range = (float)(1.0 / depth_min); s.sigma2 = s.z_range * s.z_range / 36;
  return s;
}

// ---------------------------------------------------------------- SE3 / SO3 (SE3.h, SO3.h)
struct v3d { double x, y, z; };
__device__ __forceinline__ v3d v3_add(v3d a, v3d b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ v3d v3_neg(v3d a) { return {-a.x, -a.y, -a.z}; }
__device__ __forceinline__ v3d v3_scale(double s, v3d a) { return {s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ v3d v3_cross(v3d a, v3d b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

// SO3::operator*(Point3d) SO3.h:509-520
__device__ __forceinline__ v3d q_rot(const double* q, v3d p)
{
  const v3d qv = {q[0], q[1], q[2]};
  v3d uv = v3_cross(qv, p);
  uv = v3_add(uv, uv);
  return v3_add(v3_add(p, v3_scale(q[3], uv)), v3_cross(qv, uv));
}
// SO3::operator*(SO3) SO3.h:496-503
__device__ __forceinline__ void q_mul(const double* a, const double* b, double* o)
{
  const double x = a[0], y = a[1], z = a[2], w = a[3];
  o[0] = w * b[0] + x * b[3] + y * b[2] - z * b[1];
  o[1] = w * b[1] + y * b[3] + z * b[0] - x * b[2];
  o[2] = w * b[2] + z * b[3] + x * b[1] - y * b[0];
  o[3] = w * b[3] - x * b[0] - y * b[1] - z * b[2];
}
// SE3 * Vector3d  SE3.h:53-57
__device__ __forceinline__ v3d se3_transform(const double* T, v3d p)
{
  const v3d r = q_rot(T + 3, p);
  return {T[0] + r.x, T[1] + r.y, T[2] + r.z};
}
// SE3::operator* SE3.h:45-49
__device__ __forceinline__ void se3_mul(const double* A, const double* B, double* out)
{
  double q[4];
  q_mul(A + 3, B + 3, q);
  const v3d r = q_rot(A + 3, {B[0], B[1], B[2]});
  out[0] = A[0] + r.x; out[1] = A[1] + r.y; out[2] = A[2] + r.z;
  out[3] = q[0]; out[4] = q[1]; out[5] = q[2]; out[6] = q[3];
}
// SE3::inverse SE3.h:35-38
__device__ __forceinline__ void se3_inverse(const double* A, double* out)
{
  const double qi[4] = {-A[3], -A[4], -A[5], A[6]};
  const v3d r = v3_neg(q_rot(qi, {A[0], A[1], A[2]}));
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = qi[0]; out[4] = qi[1]; out[5] = qi[2]; out[6] = qi[3];
}
// SE3::exp SE3.h:153-182 (translation term divides by theta_sq unguarded, as the reference does)
__device__ inline void se3_exp(const double* l, double* out)
{
  const v3d p = {l[0], l[1], l[2]};
  const v3d r = {l[3], l[4], l[5]};
  const double theta_sq = r.x * r.x + r.y * r.y + r.z * r.z;
  const double theta = sqrt(theta_sq);
  const double half_theta = 0.5 * theta;
  double imag_factor, real_factor;
  if (theta < 1e-10) {
    const double theta_po4 = theta_sq * theta_sq;
    imag_factor = 0.5 - (1.0 / 48.0) * theta_sq + (1.0 / 3840.0) * theta_po4;
    real_factor = 1.0 - 0.5 * theta_sq + (1.0 / 384.0) * theta_po4;
  } else {
    double s, c;
    sincos(half_theta, &s, &c);                     // one argument reduction for both (same values as sin() and cos())
    imag_factor = s / theta;
    real_factor = c;
  }
  const v3d rxp = v3_cross(r, p);
  const v3d rxrxp = v3_cross(r, rxp);
  double sin_t, cos_t;
  sincos(theta, &sin_t, &cos_t);
  const double c1 = (1 - cos_t) / theta_sq;
  const double c2 = (theta - sin_t) / (theta_sq * theta);
  const v3d t = v3_add(v3_add(p, v3_scale(c1, rxp)), v3_scale(c2, rxrxp));
  out[0] = t.x; out[1] = t.y; out[2] = t.z;
  out[3] = imag_factor * r.x; out[4] = imag_factor * r.y; out[5] = imag_factor * r.z; out[6] = real_factor;
}
// SO3::getMatrix SO3.h:396-410, row-major
__device__ __forceinline__ void q_matrix(const double* q, double* m)
{
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  const double x2 = x * x, y2 = y * y, z2 = z * z, xy = x * y, xz = x * z, yz = y * z, wx = w * x, wy = w * y, wz = w * z;
  m[0] = 1.0 - 2.0 * (y2 + z2); m[1] = 2.0 * (xy - wz);       m[2] = 2.0 * (xz + wy);
  m[3] = 2.0 * (xy + wz);       m[4] = 1.0 - 2.0 * (x2 + z2); m[5] = 2.0 * (yz - wx);
  m[6] = 2.0 * (xz - wy);       m[7] = 2.0 * (yz + wx);       m[8] = 1.0 - 2.0 * (x2 + y2);
}

// Eigen 3.4 / SSE2 association of fixed-size-3 double reductions: one Packet2d + one scalar
__device__ __forceinline__ double dot3(v3d a, v3d b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ double norm3(v3d a) { return sqrt(dot3(a, a)); }
__device__ __forceinline__ v3d normalized3(v3d a)
{
  const double z = dot3(a, a);
  if (z > 0.0) { const double n = sqrt(z); return {a.x / n, a.y / n, a.z / n}; }
  return a;
}

// ---------------------------------------------------------------- pinhole camera
// PinholeCamera::cam2world pinhole_camera.cpp:48-66 (bearing vector of unit length)
__device__ __forceinline__ v3d cam2world(const DevCam& c, double u, double v)
{
  return normalized3({(u - c.cx) / c.fx, (v - c.cy) / c.fy, 1.0});
}
// world2cam(Vector2d uv) pinhole_camera.cpp:83-87
__device__ __forceinline__ void world2cam_uv(const DevCam& c, double u, double v, double& px, double& py)
{
  px = c.fx * u + c.cx;
  py = c.fy * v + c.cy;
}
// world2cam(Vector3d) = world2cam(project2d(xyz)) (math_utils.h:104-107)
__device__ __forceinline__ void world2cam(const DevCam& c, v3d p, double& px, double& py)
{
  world2cam_uv(c, p.x / p.z, p.y / p.z, px, py);
}
// AbstractCamera::isInFrame abstract_camera.h:58-72
__device__ __forceinline__ bool in_frame(const DevCam& c, int x, int y, int boundary)
{
  return x >= boundary && x < c.width - boundary && y >= boundary && y < c.height - boundary;
}
__device__ __forceinline__ bool in_frame_level(const DevCam& c, int x, int y, int boundary, int level)
{
  return x >= boundary && x < c.width / (1 << level) - boundary && y >= boundary && y < c.height / (1 << level) - boundary;
}

// 2^-L as a double, built from its bit pattern: x / (1 << L) == x * pow2_inv(L) bit for bit (a power-of-two scale is exact in
// both forms), without the ~40-instruction FP64 division the compiler emits for a run-time divisor
__device__ __forceinline__ double pow2_inv(int L) { return __longlong_as_double((long long)(1023 - L) << 52); }
__device__ __forceinline__ float pow2_inv_f(int L) { return __int_as_float((127 - L) << 23); }

// ---------------------------------------------------------------- warp helpers
__device__ __forceinline__ float warp_sum_f(float v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// byte k of a word as a float WITHOUT the conversion unit: PRMT builds the bit pattern of 2^23 + byte, one FADD removes the
// 2^23 (both exact).  I2F.U8 / I2F.S16 run on the quarter-rate XU pipe, which was the most loaded pipe of the LK kernel
// (~270 conversions per thread and iteration against ~1,000 FP32 operations).
__device__ __forceinline__ float byte_to_float(uint32_t w, int k) { return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + k)) - 8388608.0f; }

__device__ __forceinline__ int warp_sum_i(int v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// exclusive prefix sum over an NT-thread block (every thread calls it); *total = the block's sum.  It ends with a barrier, so
// one call may follow another (they share the partials).
template <int NT>
__device__ int block_exclusive_scan(int v, int* total)
{
  __shared__ int s_w[NT / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = v;
  for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) s_w[w] = x;
  __syncthreads();
  int before = 0, sum = 0;
  for (int k = 0; k < NT / 32; ++k) { if (k < w) before += s_w[k]; sum += s_w[k]; }
  *total = sum;
  __syncthreads();
  return before + x - v;
}
