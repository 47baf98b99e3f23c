// pyramid.cu — integer half-sampling image pyramid (reference: vk::halfSample
// vision.cpp:20-110, frame_utils::createImgPyramid frame.cpp:186-195).
//
// B200 design: the job is pure HBM streaming (read level 0 once, write every
// coarser level once: 408,000 B per VGA 4-level pyramid), so ONE fused kernel
// builds all levels: each CTA owns a 128x64 level-0 tile, pulls it with two
// coalesced uint8x16 loads per thread, reduces it with byte-SIMD integer ops in
// registers, and walks the remaining levels through shared memory.  No level is
// ever re-read from HBM.  Both reference roundings are implemented bit-exactly:
//   SSE2  : avg_epu8 of the row pair then avg_epu16 of neighbours (round-half-up twice)
//   TRUNC : (a+b+c+d)>>2  (scalar and NEON paths)
#include "common.cuh"
#include "kernels.h"

namespace {

// 8 level-0 bytes of the top row (t0,t1) + bottom row (b0,b1) -> 4 output bytes
__device__ __forceinline__ uint32_t half4_sse2(uint32_t t0, uint32_t t1, uint32_t b0, uint32_t b1)
{
  const uint32_t a0 = __vavgu4(t0, b0);              // (x+y+1)>>1 per byte == _mm_avg_epu8
  const uint32_t a1 = __vavgu4(t1, b1);
  const uint32_t e = __byte_perm(a0, a1, 0x6420);    // even bytes
  const uint32_t o = __byte_perm(a0, a1, 0x7531);    // odd bytes
  return __vavgu4(e, o);                             // == _mm_avg_epu16 on zero-extended lanes
}
__device__ __forceinline__ uint32_t half2_trunc(uint32_t t, uint32_t b)
{
  // 16-bit lanes: bytes (0,2) and (1,3) zero-extended, summed (max 1020), >>2
  const uint32_t s = __byte_perm(t, 0, 0x4240) + __byte_perm(t, 0, 0x4341) + __byte_perm(b, 0, 0x4240) + __byte_perm(b, 0, 0x4341);
  return (s >> 2) & 0x00FF00FFu;                     // results in bytes 0 and 2
}
__device__ __forceinline__ uint32_t half4_trunc(uint32_t t0, uint32_t t1, uint32_t b0, uint32_t b1)
{
  return __byte_perm(half2_trunc(t0, b0), half2_trunc(t1, b1), 0x6420);
}
__device__ __forceinline__ uint32_t half1(int a, int b, int c, int d, int mode)
{
  // a,b top pair; c,d bottom pair
  if (mode == SVOB200_ROUND_SSE2) return (uint32_t)(((((a + c + 1) >> 1) + ((b + d + 1) >> 1) + 1) >> 1));
  return (uint32_t)((a + b + c + d) >> 2);
}

__device__ __forceinline__ uint4 ldg_stream(const uint4* p)
{
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// ---------------------------------------------------------------- camera input stage (SURVEY §8f-3)
// YUV_420_888 -> RGBA (ImageProcess::GetCVImage / YUV2RGB, ../image_process.cpp:97-186) -> gray
// (cv::cvtColor(COLOR_RGBA2GRAY), ../svo_system.cpp:49-51; OpenCV 4.x RGB2Gray<uchar>: 15-bit fixed point on the
// channels in MEMORY order, i.e. c0 = the app's B, c1 = G, c2 = R).  Integer, bit-exact.  The chroma terms are
// shared by the 2x2 pixels of a chroma sample.
struct ChromaTerms { int rv, guv, bu; };
__device__ __forceinline__ ChromaTerms chroma_terms(int u, int v)
{
  const int nU = u - 128, nV = v - 128;
  return {1634 * nV, -833 * nV - 400 * nU, 2066 * nU};
}
__device__ __forceinline__ uint32_t yuv_gray1(int y, const ChromaTerms& c)
{
  const int yy = 1192 * max(y - 16, 0);
  const int r = min(max(yy + c.rv, 0), 262143) >> 10;
  const int g = min(max(yy + c.guv, 0), 262143) >> 10;
  const int b = min(max(yy + c.bu, 0), 262143) >> 10;
  return (uint32_t)((b * 9798 + g * 19235 + r * 3735 + (1 << 14)) >> 15);
}
// 16 bytes starting at p (any alignment); bytes at index >= valid are not read (returned as 0)
__device__ __forceinline__ uint4 load16_any(const uint8_t* p, int valid)
{
  if (valid >= 16 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) return ldg_stream(reinterpret_cast<const uint4*>(p));
  uint32_t w[4] = {0, 0, 0, 0};
  for (int k = 0; k < 16 && k < valid; ++k) w[k >> 2] |= (uint32_t)__ldg(p + k) << (8 * (k & 3));
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ int byte_of(const uint4& q, int k)
{
  const uint32_t w = k < 4 ? q.x : (k < 8 ? q.y : (k < 12 ? q.z : q.w));
  return (int)((w >> (8 * (k & 3))) & 0xffu);
}
// gray of 16 pixels of the row pair (y0, y0+1) starting at even x0; the planes as AImage hands them out
__device__ __forceinline__ void yuv_rows16(const YuvPlanes& s, int b, int x0, int y0, int w, int h, uint4& g0, uint4& g1)
{
  const int valid = min(16, w - x0);
  const uint8_t* py = s.y + (size_t)b * s.y_img_stride + (size_t)y0 * s.y_stride + x0;
  const uint4 ya = load16_any(py, valid);
  const uint4 yb = (y0 + 1 < h) ? load16_any(py + s.y_stride, valid) : make_uint4(0, 0, 0, 0);
  const size_t uvo = (size_t)b * s.uv_img_stride + (size_t)(y0 >> 1) * s.uv_stride + (size_t)(x0 >> 1) * s.uv_pixel_stride;
  const int nc = (valid + 1) >> 1;                 // chroma samples needed
  int cu[8], cv[8];
  if (s.uv_pixel_stride == 2 && (s.u == s.v + 1 || s.v == s.u + 1)) {
    // interleaved chroma (NV21 / NV12 views): one 16-byte window holds both planes
    const bool v_first = s.u == s.v + 1;
    const uint8_t* base = (v_first ? s.v : s.u) + uvo;
    const uint4 q = load16_any(base, 2 * nc);
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int a = byte_of(q, 2 * k), c = byte_of(q, 2 * k + 1); cu[k] = v_first ? c : a; cv[k] = v_first ? a : c; }
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const bool in = k < nc;
      cu[k] = in ? (int)__ldg(s.u + uvo + (size_t)k * s.uv_pixel_stride) : 128;
      cv[k] = in ? (int)__ldg(s.v + uvo + (size_t)k * s.uv_pixel_stride) : 128;
    }
  }
  uint32_t o0[4] = {0, 0, 0, 0}, o1[4] = {0, 0, 0, 0};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const ChromaTerms c = chroma_terms(cu[k], cv[k]);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int i = 2 * k + e;
      o0[i >> 2] |= yuv_gray1(byte_of(ya, i), c) << (8 * (i & 3));
      o1[i >> 2] |= yuv_gray1(byte_of(yb, i), c) << (8 * (i & 3));
    }
  }
  g0 = make_uint4(o0[0], o0[1], o0[2], o0[3]);
  g1 = make_uint4(o1[0], o1[1], o1[2], o1[3]);
}

// levels >= 2 of a tile, all sizes compile-time: src is a SW x SH tile in shared memory, dst its SW/2 x SH/2 half-sample.
// Four outputs per thread with the same byte-SIMD reduction as level 1 (two aligned 8-byte shared loads, one word to shared
// memory and one word to HBM; the pitch padding absorbs the tail of a row); tiles narrower than 4 fall back to one output per thread.
template <int SW_, int SH_, int NT_>
__device__ __forceinline__ void tile_level(const uint8_t* src, uint8_t* dst, int mode, uint8_t* gout, int pitch, int wl, int hl, int ox, int oy, int t)
{
  constexpr int DW = SW_ / 2, DH = SH_ / 2;
  if (DW >= 4) {
    constexpr int WPR = DW >= 4 ? DW / 4 : 1;            // words per output row of the tile (the branch is dead for narrower tiles)
    for (int i = t; i < DH * WPR; i += NT_) {
      const int ly = i / WPR, lw = i - ly * WPR;
      const uint2 top = *reinterpret_cast<const uint2*>(src + (2 * ly) * SW_ + 8 * lw);
      const uint2 bot = *reinterpret_cast<const uint2*>(src + (2 * ly + 1) * SW_ + 8 * lw);
      const uint32_t v = mode ? half4_sse2(top.x, top.y, bot.x, bot.y) : half4_trunc(top.x, top.y, bot.x, bot.y);
      *reinterpret_cast<uint32_t*>(dst + ly * DW + 4 * lw) = v;
      const int gx = ox + 4 * lw, gy = oy + ly;
      if (gx < wl && gy < hl) {
        uint8_t* o = gout + (size_t)gy * pitch + gx;
        if (gx + 4 <= pitch) *reinterpret_cast<uint32_t*>(o) = v;
        else for (int k = 0; k < 4 && gx + k < wl; ++k) o[k] = (uint8_t)((v >> (8 * k)) & 0xff);
      }
    }
  } else {
    for (int i = t; i < DH * DW; i += NT_) {
      const int ly = i / DW, lx = i - ly * DW;
      const uint8_t* p = src + (2 * ly) * SW_ + 2 * lx;
      const uint32_t v = half1(p[0], p[1], p[SW_], p[SW_ + 1], mode);
      dst[ly * DW + lx] = (uint8_t)v;
      const int gx = ox + lx, gy = oy + ly;
      if (gx < wl && gy < hl) gout[(size_t)gy * pitch + gx] = (uint8_t)v;
    }
  }
}

// One CTA = one 128x64 level-0 tile of one image; 256 threads; the pyramid depth NL is a template parameter, so every tile
// size, loop bound and index split below is a compile-time constant.
// (Measured alone, tools/pyr_probe.py, 4,096 VGA frames x 4 levels: 0.292 ms = 5.73 TB/s algorithmic = 0.876 of the copy peak.
// PERSISTENT CTAs walking the tiles with a grid stride, 8 or 6 per SM, measured 0.362 / 0.394 ms: a CTA that loops has a block
// barrier between tiles and nothing in flight across it, where the hardware scheduler starts the next short-lived CTA while the
// previous one's last warps drain.  A persistent TMA-load version reached the same bandwidth, lost inside the tracker step and
// was removed: DESIGN §8.)
// Thread t: 16-pixel segment (t&7) of row pair (t>>3).
// YUV = true: level 0 is PRODUCED here from the camera's YUV planes (and written once) instead of being read,
// so the input stage costs no extra pass over the frame.
constexpr int PTW = 128, PTH = 64, PNT = 256;
template <bool YUV, int NL>
__global__ void __launch_bounds__(PNT) pyramid_fused_kernel(DevFrame f, int modes_mask, YuvPlanes yuv)
{
  __shared__ __align__(16) uint8_t s_a[(PTH / 2) * (PTW / 2)];      // level-1 tile 64 x 32
  __shared__ __align__(16) uint8_t s_b[(PTH / 4) * (PTW / 4)];      // level-2 tile 32 x 16
  const int t = threadIdx.x;
  const int b = blockIdx.z;
  const int tx0 = blockIdx.x * PTW, ty0 = blockIdx.y * PTH;

  // ---- level 0 -> 1 (registers)
  {
    const int seg = t & 7, rp = t >> 3;
    const int x0 = tx0 + seg * 16, y0 = ty0 + rp * 2;
    const int w1 = f.w[1], h1 = f.h[1];
    const int x1 = x0 >> 1, y1 = y0 >> 1;
    uint32_t o0 = 0, o1 = 0;
    const bool act = (y1 < h1) && (x0 < f.pitch[0]) && (x1 < w1);
    if (YUV && !act && y0 < f.h[0] && x0 < f.w[0]) {
      // odd last row / column that the half-sampling drops: level 0 still has to be produced
      uint4 g0, g1;
      yuv_rows16(yuv, b, x0, y0, f.w[0], f.h[0], g0, g1);
      uint8_t* l0 = f.lvl[0] + (size_t)b * f.img_stride[0] + (size_t)y0 * f.pitch[0] + x0;
      *reinterpret_cast<uint4*>(l0) = g0;
      if (y0 + 1 < f.h[0]) *reinterpret_cast<uint4*>(l0 + f.pitch[0]) = g1;
    }
    if (act) {
      uint4 r0, r1;
      if (YUV) {
        yuv_rows16(yuv, b, x0, y0, f.w[0], f.h[0], r0, r1);
        uint8_t* l0 = f.lvl[0] + (size_t)b * f.img_stride[0] + (size_t)y0 * f.pitch[0] + x0;
        *reinterpret_cast<uint4*>(l0) = r0;                  // pitch is a multiple of 16: the tail lands in the padding
        *reinterpret_cast<uint4*>(l0 + f.pitch[0]) = r1;
      } else {
        const uint8_t* base = f.lvl[0] + (size_t)b * f.img_stride[0] + (size_t)y0 * f.pitch[0] + x0;
        r0 = ldg_stream(reinterpret_cast<const uint4*>(base));
        r1 = ldg_stream(reinterpret_cast<const uint4*>(base + f.pitch[0]));
      }
      if (modes_mask & 1) {
        o0 = half4_sse2(r0.x, r0.y, r1.x, r1.y);
        o1 = half4_sse2(r0.z, r0.w, r1.z, r1.w);
      } else {
        o0 = half4_trunc(r0.x, r0.y, r1.x, r1.y);
        o1 = half4_trunc(r0.z, r0.w, r1.z, r1.w);
      }
      uint8_t* out = f.lvl[1] + (size_t)b * f.img_stride[1] + (size_t)y1 * f.pitch[1] + x1;
      if (x1 + 8 <= f.pitch[1]) {
        *reinterpret_cast<uint2*>(out) = make_uint2(o0, o1);     // pitch padding absorbs the tail
      } else {
        for (int k = 0; k < 8 && x1 + k < w1; ++k) out[k] = (uint8_t)(((k < 4 ? o0 : o1) >> (8 * (k & 3))) & 0xff);
      }
    }
    if (NL > 2) *reinterpret_cast<uint2*>(&s_a[rp * (PTW / 2) + seg * 8]) = make_uint2(o0, o1);
  }
  if (NL <= 2) return;
  __syncthreads();
  // ---- levels 2.. (shared memory ping-pong): tile 64x32 -> 32x16 -> 16x8 -> 8x4 -> 4x2 -> 2x1
#define PYR_LEVEL(L, SW_, SH_, SRC, DST)                                                                                         \
  if (NL > (L)) {                                                                                                                \
    tile_level<SW_, SH_, PNT>(SRC, DST, (modes_mask >> ((L) - 1)) & 1, f.lvl[L] + (size_t)b * f.img_stride[L], f.pitch[L], f.w[L], \
                              f.h[L], tx0 >> (L), ty0 >> (L), t);                                                                \
    if (NL > (L) + 1) __syncthreads();                                                                                           \
  }
  PYR_LEVEL(2, 64, 32, s_a, s_b)
  PYR_LEVEL(3, 32, 16, s_b, s_a)
  PYR_LEVEL(4, 16, 8, s_a, s_b)
  PYR_LEVEL(5, 8, 4, s_b, s_a)
  PYR_LEVEL(6, 4, 2, s_a, s_b)
#undef PYR_LEVEL
}

// Generic single-level kernel: any size, both roundings, and the reference's scalar pointer
// walk for ODD input widths (vision.cpp:92-109: `top` advances 2*out_w per row, then += stride,
// so each output row starts one pixel early — reproduced through dense flat offsets).
__global__ void half_sample_generic_kernel(const uint8_t* in, int in_pitch, unsigned long long in_img_stride, int w, int h,
                                           uint8_t* out, int out_pitch, unsigned long long out_img_stride, int mode)
{
  const int ow = w / 2, oh = h / 2;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= ow || y >= oh) return;
  const uint8_t* img = in + (size_t)blockIdx.z * in_img_stride;
  int a, b, c, d;
  if ((w & 1) == 0 || mode == SVOB200_ROUND_SSE2) {
    const uint8_t* p = img + (size_t)(2 * y) * in_pitch + 2 * x;
    a = p[0]; b = p[1]; c = p[in_pitch]; d = p[in_pitch + 1];
  } else {
    // dense offsets of the scalar walk: row y starts at y*(2*w-1)
    const long long o = (long long)y * (2 * w - 1) + 2 * x;
    const long long idx[4] = {o, o + 1, o + w, o + w + 1};
    int v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = (int)(idx[k] / w), cc = (int)(idx[k] - (long long)r * w);
      v[k] = (r < h) ? img[(size_t)r * in_pitch + cc] : 0;
    }
    // the reference loop stops when `bottom` reaches the end of the image
    if ((long long)y * (2 * w - 1) + w >= (long long)w * h) return;
    a = v[0]; b = v[1]; c = v[2]; d = v[3];
  }
  out[(size_t)blockIdx.z * out_img_stride + (size_t)y * out_pitch + x] = (uint8_t)half1(a, b, c, d, mode);
}

// stand-alone input stage (frames the fused kernel does not take: odd level widths, > 7 levels, 1 level)
__global__ void __launch_bounds__(128) yuv_gray_kernel(DevFrame f, YuvPlanes yuv)
{
  const int b = blockIdx.z;
  const int x0 = (blockIdx.x * 32 + (threadIdx.x & 31)) * 16, y0 = (blockIdx.y * 4 + (threadIdx.x >> 5)) * 2;
  if (x0 >= f.w[0] || y0 >= f.h[0]) return;
  uint4 g0, g1;
  yuv_rows16(yuv, b, x0, y0, f.w[0], f.h[0], g0, g1);
  uint8_t* l0 = f.lvl[0] + (size_t)b * f.img_stride[0] + (size_t)y0 * f.pitch[0] + x0;
  *reinterpret_cast<uint4*>(l0) = g0;
  if (y0 + 1 < f.h[0]) *reinterpret_cast<uint4*>(l0 + f.pitch[0]) = g1;
}

}  // namespace

template <bool YUV>
static void launch_fused(const DevFrame& f, int mask, const YuvPlanes& yuv, cudaStream_t s)
{
  dim3 grid((f.w[0] + PTW - 1) / PTW, (f.h[0] + PTH - 1) / PTH, f.batch);
  switch (f.n_levels) {
    case 2: pyramid_fused_kernel<YUV, 2><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
    case 3: pyramid_fused_kernel<YUV, 3><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
    case 4: pyramid_fused_kernel<YUV, 4><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
    case 5: pyramid_fused_kernel<YUV, 5><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
    case 6: pyramid_fused_kernel<YUV, 6><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
    default: pyramid_fused_kernel<YUV, 7><<<grid, PNT, 0, s>>>(f, mask, yuv); break;
  }
}

static bool fused_ok(const DevFrame& f)
{
  bool odd = false;
  for (int l = 0; l + 1 < f.n_levels; ++l) odd |= (f.w[l] & 1) != 0;
  return !odd && f.n_levels >= 2 && f.n_levels <= 7;
}

// level 0 from YUV planes (+ all coarser levels); level 0 must be owned storage with a 16-byte pitch
int launch_pyramid_yuv(const DevFrame& f, const YuvPlanes& yuv, const int* modes, cudaStream_t s, long long* launches)
{
  if (fused_ok(f)) {
    int mask = 0;
    for (int l = 0; l + 1 < f.n_levels; ++l) if (modes[l] == SVOB200_ROUND_SSE2) mask |= 1 << l;
    launch_fused<true>(f, mask, yuv, s);
    ++*launches;
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
  }
  dim3 grid((f.w[0] + 511) / 512, (f.h[0] + 7) / 8, f.batch);
  yuv_gray_kernel<<<grid, 128, 0, s>>>(f, yuv);
  ++*launches;
  if (cudaGetLastError() != cudaSuccess) return -1;
  return launch_pyramid(f, modes, s, launches);
}

int launch_pyramid(const DevFrame& f, const int* modes, cudaStream_t s, long long* launches)
{
  if (f.n_levels <= 1) return 0;
  if (fused_ok(f)) {
    int mask = 0;
    for (int l = 0; l + 1 < f.n_levels; ++l) if (modes[l] == SVOB200_ROUND_SSE2) mask |= 1 << l;
    launch_fused<false>(f, mask, YuvPlanes{}, s);
    ++*launches;
  } else {
    for (int l = 0; l + 1 < f.n_levels; ++l) {
      dim3 blk(32, 8), grid((f.w[l + 1] + 31) / 32, (f.h[l + 1] + 7) / 8, f.batch);
      if (f.w[l + 1] == 0 || f.h[l + 1] == 0) break;
      half_sample_generic_kernel<<<grid, blk, 0, s>>>(f.lvl[l], f.pitch[l], f.img_stride[l], f.w[l], f.h[l],
                                                      f.lvl[l + 1], f.pitch[l + 1], f.img_stride[l + 1], modes[l]);
      ++*launches;
    }
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_half_sample_single(const uint8_t* in, int in_pitch, int w, int h, uint8_t* out, int out_pitch, int mode,
                              cudaStream_t s, long long* launches)
{
  if (w / 2 == 0 || h / 2 == 0) return 0;
  dim3 blk(32, 8), grid((w / 2 + 31) / 32, (h / 2 + 7) / 8, 1);
  half_sample_generic_kernel<<<grid, blk, 0, s>>>(in, in_pitch, 0, w, h, out, out_pitch, 0, mode);
  ++*launches;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
