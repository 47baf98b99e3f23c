// synth.cu — synthetic-sequence renderer for the bench (SURVEY.md §8d): a textured plane z = plane_z
// seen by a distortion-free pinhole camera.  Same float64 arithmetic and operation order as
// android_svo_b200/synth.py:render, so both produce identical bytes.  Bench/test support only —
// rendering is always outside the timed region.
#include "common.cuh"
#include "kernels.h"

namespace {
__global__ void synth_render_kernel(const uint8_t* tex, int size, double ppm, double plane_z, DevCam cam,
                                    const double* rc, uint8_t* out)
{
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, b = blockIdx.z;
  if (x >= cam.width || y >= cam.height) return;
  const double* R = rc + 12 * (size_t)b;
  const double* c = R + 9;
  const double X = ((double)x - cam.cx) / cam.fx, Y = ((double)y - cam.cy) / cam.fy;
  const double dx = R[0] * X + R[1] * Y + R[2];
  const double dy = R[3] * X + R[4] * Y + R[5];
  const double dz = R[6] * X + R[7] * Y + R[8];
  const double s = (plane_z - c[2]) / dz;
  const double u = (c[0] + s * dx) * ppm + (double)(size / 2);
  const double v = (c[1] + s * dy) * ppm + (double)(size / 2);
  const double uf = floor(u), vf = floor(v);
  const long long ui = (long long)uf, vi = (long long)vf;
  const double fu = u - uf, fv = v - vf;
  auto wrap = [size](long long a) { long long m = a % size; return (int)(m < 0 ? m + size : m); };
  const int u0 = wrap(ui), v0 = wrap(vi), u1 = wrap(ui + 1), v1 = wrap(vi + 1);
  const double t00 = tex[(size_t)v0 * size + u0], t01 = tex[(size_t)v0 * size + u1];
  const double t10 = tex[(size_t)v1 * size + u0], t11 = tex[(size_t)v1 * size + u1];
  const double val = (1 - fu) * (1 - fv) * t00 + fu * (1 - fv) * t01 + (1 - fu) * fv * t10 + fu * fv * t11;
  out[(size_t)b * cam.width * cam.height + (size_t)y * cam.width + x] = (uint8_t)floor(val + 0.5);
}
}  // namespace

cudaError_t launch_synth_render(const uint8_t* d_tex, int tex_size, double ppm, double plane_z, const DevCam& cam, int batch,
                                const double* d_rc, uint8_t* d_out, cudaStream_t s, long long* launches)
{
  dim3 blk(32, 8), grid((cam.width + 31) / 32, (cam.height + 7) / 8, batch);
  synth_render_kernel<<<grid, blk, 0, s>>>(d_tex, tex_size, ppm, plane_z, cam, d_rc, d_out);
  ++*launches;
  return cudaGetLastError();
}
