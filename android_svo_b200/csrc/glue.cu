// glue.cu — device-side marshalling between the operators so that a whole front-end step
// (pyramid -> sparse align -> reprojection refinement -> seed update) runs on one stream without a
// host round trip.  These are the small pieces of host code that sit between the operators in
// the reference:
//   Feature ctor                      f = cam.cam2world(px)                       (feature.h:43-51)
//   SparseImgAlign                    depth = |pos - ref_pos|, xyz_ref = f*depth  (sparse_img_align.cpp:132-134)
//   SparseImgAlign::run               cur.T_f_w = T_cur_from_ref * ref.T_f_w      (sparse_img_align.cpp:89)
//   Reprojector::reprojectMap         px = cur.w2c(point.pos)                     (reprojector.cpp:131-145)
//   Matcher::findMatchDirect          depth_ref = |ref.pos() - pt.pos|, T_cur_ref (matcher.cpp:169-173)
// Same operation order as the reference, unfused (library-wide -fmad=false) => bit-identical.
#include "common.cuh"
#include "kernels.h"

namespace {

// Frame::pos() = T_f_w.inverse().translation
__device__ __forceinline__ v3d frame_pos(const double* T_f_w)
{
  double inv[7];
  se3_inverse(T_f_w, inv);
  return {inv[0], inv[1], inv[2]};
}

__global__ void features_prepare_kernel(DevCam cam, int n, const double* px, const double* pt_world, const int* image,
                                        const double* T_ref_w, double* f_out, double* xyz_out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const v3d f = cam2world(cam, px[2 * i], px[2 * i + 1]);
  const v3d rp = frame_pos(T_ref_w + 7 * (size_t)image[i]);
  const v3d d = {pt_world[3 * i] - rp.x, pt_world[3 * i + 1] - rp.y, pt_world[3 * i + 2] - rp.z};
  const double depth = norm3(d);
  if (f_out) { f_out[3 * i] = f.x; f_out[3 * i + 1] = f.y; f_out[3 * i + 2] = f.z; }
  xyz_out[3 * i] = f.x * depth; xyz_out[3 * i + 1] = f.y * depth; xyz_out[3 * i + 2] = f.z * depth;
}

__global__ void compose_poses_kernel(int batch, const svob200_align_result* res, const double* T_ref_w, double* T_cur_w)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  double out[7];
  se3_mul(res[b].T_cur_ref, T_ref_w + 7 * (size_t)b, out);
  for (int k = 0; k < 7; ++k) T_cur_w[7 * (size_t)b + k] = out[k];
}

__global__ void reproject_prepare_kernel(DevCam cam, int n, svob200_feature_ref* ftrs, const double* pt_world,
                                         const double* T_kf_w /*7 per feature*/, const double* T_cur_w /*7 per image*/,
                                         double* depth_ref, double* px_cur)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* Tk = T_kf_w + 7 * (size_t)i;
  const double* Tc = T_cur_w + 7 * (size_t)ftrs[i].cur_image;
  double inv[7], Tcr[7];
  se3_inverse(Tk, inv);
  se3_mul(Tc, inv, Tcr);                                  // cur.T_f_w_ * ref.T_f_w_.inverse()
  for (int k = 0; k < 7; ++k) ftrs[i].T_cur_ref[k] = Tcr[k];
  const v3d p = {pt_world[3 * i], pt_world[3 * i + 1], pt_world[3 * i + 2]};
  const v3d kp = {inv[0], inv[1], inv[2]};                // ref frame pos()
  depth_ref[i] = norm3({kp.x - p.x, kp.y - p.y, kp.z - p.z});
  double u, v;
  world2cam(cam, se3_transform(Tc, p), u, v);             // Frame::w2c
  px_cur[2 * i] = u; px_cur[2 * i + 1] = v;
}

}  // namespace

cudaError_t launch_features_prepare(const DevCam& cam, int n, const double* d_px, const double* d_pt, const int* d_image,
                                    const double* d_T_ref_w, double* d_f, double* d_xyz, cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  features_prepare_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_px, d_pt, d_image, d_T_ref_w, d_f, d_xyz);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_compose_poses(int batch, const svob200_align_result* d_res, const double* d_T_ref_w, double* d_T_cur_w,
                                 cudaStream_t s, long long* launches)
{
  if (batch <= 0) return cudaSuccess;
  compose_poses_kernel<<<(batch + 127) / 128, 128, 0, s>>>(batch, d_res, d_T_ref_w, d_T_cur_w);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_reproject_prepare(const DevCam& cam, int n, svob200_feature_ref* d_ftrs, const double* d_pt, const double* d_T_kf_w,
                                     const double* d_T_cur_w, double* d_depth_ref, double* d_px_cur, cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  reproject_prepare_kernel<<<(n + 127) / 128, 128, 0, s>>>(cam, n, d_ftrs, d_pt, d_T_kf_w, d_T_cur_w, d_depth_ref, d_px_cur);
  ++*launches;
  return cudaGetLastError();
}
