// fast.cu — FAST-9/16 corners (threshold 10, 3x3 non-max suppression), Shi-Tomasi
// scoring and best-corner-per-grid-cell selection.
//
// reference: FastDetector::detect feature_detection.cpp:77-122; cv::FAST(img,kps,10,true) from
// OpenCV 4.5.4 features2d (fast.cpp / fast_score.cpp — third party, restated from the published
// algorithm and pinned against python cv2 in tests/golden); vk::shiTomasiScore vision.cpp:113-154.
//
// B200 design: one pass over each detected level, a CTA per 120x30 tile staged in shared memory.  Everything per-pixel is
// byte-SIMD on 16-bit lanes, FOUR pixels per thread, one warp per tile row, no data-dependent branch:
//   A. score of EVERY pixel.  The 7x12-byte neighbourhood of a 4-pixel group sits in 21 registers; ring position k of the four
//      pixels is one PRMT; X_k = 256 + v - ring_k on two lanes per word.  cv's cornerScore is S - 1 with
//         S = max( max over the 16 arcs of 9 of  min over the arc of (v - ring) ,  max over the arcs of  min of (ring - v) )
//      and the pixel is a FAST-9 corner iff S > t, so one sliding-window minimum AND maximum of X over the circular ring (3+3+3
//      taps with VIMNMX3.U16x2: min over an arc of (ring - v) = 256 - max over the arc of X) gives test and score at once.
//      A warp whose 128 pixels all fail OpenCV's necessary condition on four opposite pairs skips the rest (natural images).
//      The dense score tile holds S - 1 for every pixel; values below t mark non-corners and never win a comparison against
//      a corner's score (>= t), so the non-maximum suppression needs no mask.
//   C. strict 3x3 non-max suppression, again four pixels per thread on 16-bit lanes; survivors (>= t and > all 8 neighbours)
//      go to a compact keypoint list.
//   D. thread per keypoint: grid cell, occupancy, Shi-Tomasi by byte dot products (dp4a on funnel-shifted words: the
//      integer sums are exact, as the reference's float sums are), one 64-bit atomicMax per keypoint.
// The reference's sequential "first strictly-greater wins" rule over (level, y, x) order becomes
// a single 64-bit atomicMax per keypoint on key = (ordered(score) << 32) | ~(level,y,x), which is
// order-independent and therefore bit-identical to the sequential loop.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int TW = 120, TH = 30;                         // output tile: the score tile (1-px ring, rounded to groups) is 128 x 32
constexpr int HALO = 5;                                  // rows above / below (Shi-Tomasi reads y-5 .. y+4)
constexpr int XOFF = 8;                                  // the staged tile starts 8 columns left of the output tile (8-byte aligned chunks)
constexpr int PH = TH + 2 * HALO;                        // 40 staged rows
constexpr int PP = TW + 2 * XOFF;                        // 136 staged columns = 34 words
constexpr int PW = PP / 4;
constexpr int SG = 32;                                   // groups of 4 pixels per score row: columns ox-4 .. ox+123, one warp per row
constexpr int SW = 4 * SG, SH = TH + 2;                  // score tile 128 x 32
constexpr int NT = 256;
constexpr int COL0 = XOFF - 4, ROW0 = HALO - 1;          // staged-tile position of score-tile column 0 / row 0
static_assert(SH * SG == 4 * NT, "four groups per thread");

__device__ constexpr int c_ring_dx[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
__device__ constexpr int c_ring_dy[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};

__device__ __forceinline__ uint32_t ordered_bits(float f)
{
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float from_ordered_bits(uint32_t u)
{
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

// ring position K of a 4-pixel group as two words of 16-bit lanes: E = pixels 0 and 2, O = pixels 1 and 3.
// W[r][0..2] = the aligned words left of / at / right of the group on row y - 3 + r.
template <int K>
__device__ __forceinline__ void ring_lanes(const uint32_t (&W)[7][3], uint32_t& E, uint32_t& O)
{
  constexpr int dx = c_ring_dx[K], r = 3 + c_ring_dy[K];
  constexpr int start = 4 + dx;                                   // first byte inside the 12-byte row (left word = bytes 0..3)
  uint32_t v;
  if (dx == 0) v = W[r][1];
  else if (dx > 0) v = __byte_perm(W[r][1], W[r][2], (dx) | ((dx + 1) << 4) | ((dx + 2) << 8) | ((dx + 3) << 12));
  else v = __byte_perm(W[r][0], W[r][1], (start) | ((start + 1) << 4) | ((start + 2) << 8) | ((start + 3) << 12));
  E = v & 0x00ff00ffu;
  O = __byte_perm(v, 0u, 0x4341);                                 // (v >> 8) & 0x00ff00ff
}

template <int K> struct RingFill {
  static __device__ __forceinline__ void run(const uint32_t (&W)[7][3], uint32_t bE, uint32_t bO, uint32_t (&XE)[16], uint32_t (&XO)[16])
  {
    uint32_t e, o;
    ring_lanes<K>(W, e, o);
    XE[K] = bE - e; XO[K] = bO - o;                               // lane = 256 + v - ring_K in [1, 511]: no borrow between lanes
    RingFill<K + 1>::run(W, bE, bO, XE, XO);
  }
};
template <> struct RingFill<16> {
  static __device__ __forceinline__ void run(const uint32_t (&)[7][3], uint32_t, uint32_t, uint32_t (&)[16], uint32_t (&)[16]) {}
};

// S (two lanes, biased by 256) from the 16 biased differences of two pixels: max( max_arcs min_arc X , 512 - min_arcs max_arc X )
__device__ __forceinline__ uint32_t arc_score_lanes(const uint32_t (&X)[16])
{
  uint32_t lo3[16], hi3[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    lo3[k] = __vimin3_u16x2(X[k], X[(k + 1) & 15], X[(k + 2) & 15]);
    hi3[k] = __vimax3_u16x2(X[k], X[(k + 1) & 15], X[(k + 2) & 15]);
  }
  uint32_t a = 0u, b = 0xffffffffu;
#pragma unroll
  for (int k = 0; k < 16; k += 2) {
    const uint32_t m0 = __vimin3_u16x2(lo3[k], lo3[(k + 3) & 15], lo3[(k + 6) & 15]);
    const uint32_t m1 = __vimin3_u16x2(lo3[k + 1], lo3[(k + 4) & 15], lo3[(k + 7) & 15]);
    a = __vimax3_u16x2(a, m0, m1);
    const uint32_t n0 = __vimax3_u16x2(hi3[k], hi3[(k + 3) & 15], hi3[(k + 6) & 15]);
    const uint32_t n1 = __vimax3_u16x2(hi3[k + 1], hi3[(k + 4) & 15], hi3[(k + 7) & 15]);
    b = __vimin3_u16x2(b, n0, n1);
  }
  return __vmaxu2(a, 0x02000200u - b);
}

// necessary condition on four opposite pairs (0,8) (2,10) (4,12) (6,14): every pair needs a member < v - t (or every pair one
// > v + t).  In biased lanes: min over the pairs of max(X_k, X_k+8) > 256 + t, or max over the pairs of min(...) < 256 - t.
__device__ __forceinline__ bool group_may_have_corner(const uint32_t (&XE)[16], const uint32_t (&XO)[16], uint32_t thr_hi, uint32_t thr_lo)
{
  uint32_t f = 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const uint32_t (&X)[16] = h ? XO : XE;
    const uint32_t mx = __vimin3_u16x2(__vmaxu2(X[0], X[8]), __vmaxu2(X[2], X[10]), __vminu2(__vmaxu2(X[4], X[12]), __vmaxu2(X[6], X[14])));
    const uint32_t mn = __vimax3_u16x2(__vminu2(X[0], X[8]), __vminu2(X[2], X[10]), __vmaxu2(__vminu2(X[4], X[12]), __vminu2(X[6], X[14])));
    f |= ((mx | 0x80008000u) - thr_hi) | (thr_lo - mn);          // bit 15 / 31: mx >= 257 + t ; mn <= 255 - t
  }
  return (f & 0x80008000u) != 0;
}

// vk::shiTomasiScore vision.cpp:113-154 on the staged tile; p points at (u,v).  The reference's float sums of integer-valued
// terms are exact (< 2^24), so they are formed as byte dot products: with P / M / Z the 8 window columns shifted by +1 / -1 / 0,
//   dXX = sum P.P + M.M - 2 P.M     dYY = sum Zu.Zu + Zd.Zd - 2 Zu.Zd     dXY = sum (P - M).(Zu - Zd)     (u / d: row below / above)
__device__ __forceinline__ float shi_tomasi_smem(const uint8_t* p)
{
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(p - 5);
  const unsigned sh = (unsigned)(a0 & 3) * 8;
  const uint32_t* q0 = reinterpret_cast<const uint32_t*>(a0 & ~(uintptr_t)3);
  uint32_t Zl[3], Zh[3];                                   // rolling window: rows y'-1, y', y'+1
  uint32_t zz[3];
  uint32_t sxx = 0, sxy_pos = 0, sxy_neg = 0, syy = 0, pm = 0, zc = 0, Pl = 0, Ph = 0, Ml = 0, Mh = 0;
#pragma unroll
  for (int r = 0; r < 10; ++r) {                           // rows y - 5 .. y + 4
    const uint32_t* q = q0 + (r - 5) * PW;
    const uint32_t w0 = q[0], w1 = q[1], w2 = q[2], w3 = q[3];
    const uint32_t f0 = __funnelshift_r(w0, w1, sh), f1 = __funnelshift_r(w1, w2, sh), f2 = __funnelshift_r(w2, w3, sh);   // cols x-5 .. x+6
    const uint32_t zl = __byte_perm(f0, f1, 0x4321), zh = __byte_perm(f1, f2, 0x4321);                                    // cols x-4 .. x+3
    const int s = r % 3;
    Zl[s] = zl; Zh[s] = zh;
    zz[s] = __dp4a(zl, zl, __dp4a(zh, zh, 0u));
    if (r >= 2) {
      // centre row y' = row r - 1 (its P / M were formed in the previous round), below = row r, above = row r - 2
      const int u = s, d = (r - 2) % 3;
      sxx = __dp4a(Pl, Pl, sxx); sxx = __dp4a(Ph, Ph, sxx); sxx = __dp4a(Ml, Ml, sxx); sxx = __dp4a(Mh, Mh, sxx);
      pm = __dp4a(Pl, Ml, pm); pm = __dp4a(Ph, Mh, pm);
      syy += zz[u] + zz[d];
      zc = __dp4a(Zl[u], Zl[d], zc); zc = __dp4a(Zh[u], Zh[d], zc);
      sxy_pos = __dp4a(Pl, Zl[u], sxy_pos); sxy_pos = __dp4a(Ph, Zh[u], sxy_pos); sxy_pos = __dp4a(Ml, Zl[d], sxy_pos); sxy_pos = __dp4a(Mh, Zh[d], sxy_pos);
      sxy_neg = __dp4a(Pl, Zl[d], sxy_neg); sxy_neg = __dp4a(Ph, Zh[d], sxy_neg); sxy_neg = __dp4a(Ml, Zl[u], sxy_neg); sxy_neg = __dp4a(Mh, Zh[u], sxy_neg);
    }
    // P / M of this row, used when it is the centre row (next round): rows y - 4 .. y + 3
    Ml = f0; Mh = f1;                                                                                                      // cols x-5 .. x+2
    Pl = __byte_perm(f0, f1, 0x5432); Ph = __byte_perm(f1, f2, 0x5432);                                                    // cols x-3 .. x+4
  }
  float dXX = (float)(int)(sxx - 2u * pm);
  float dYY = (float)(int)(syy - 2u * zc);
  float dXY = (float)((int)sxy_pos - (int)sxy_neg);
  dXX = (float)((double)dXX / 128.0);
  dYY = (float)((double)dYY / 128.0);
  dXY = (float)((double)dXY / 128.0);
  const float tr = dXX + dYY;
  const float disc = tr * tr - 4 * (dXX * dYY - dXY * dXY);
  const double root = sqrt((double)disc);                  // ::sqrt(double) in the reference TU
  return (float)(0.5 * ((double)tr - root));
}

struct FastArgs {
  DevFrame f;
  int n_levels;            // detect levels
  int tiles_x[SVOB_MAXL], tile_begin[SVOB_MAXL + 1];   // flat tile index -> level (grid.x = tile_begin[n_levels], grid.y = batch)
  int cell, grid_cols, n_cells;
  float thr_f;
  const uint8_t* occupancy;
  const int* image_sel;    // optional: images with a negative entry are skipped
  unsigned long long* keys;
  // raw mode (svob200_fast_corners): single image / level, write score map instead of cells
  uint8_t* raw_scores; int raw_image, raw_level, raw_threshold, raw_nonmax;
};

// append `mine` entries per thread to a shared list: warp prefix sum + one atomic per warp; returns this thread's first slot
__device__ __forceinline__ int list_reserve(int mine, int* counter)
{
  const int lane = threadIdx.x & 31;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  int base = 0;
  if (lane == 31 && total) base = atomicAdd(counter, total);
  base = __shfl_sync(0xffffffffu, base, 31);
  return base + incl - mine;
}

__global__ void __launch_bounds__(NT, 3) fast_kernel(FastArgs A)
{
  __shared__ __align__(16) uint8_t s_px[PH * PP];
  __shared__ __align__(16) uint32_t s_scw[SH * SG];       // score tile, one word per group
  __shared__ unsigned short s_kp[TH * TW];                // keypoints: score-tile index
  __shared__ int s_n;
  const bool raw = A.raw_scores != nullptr;
  int level = 0;
  if (raw) level = A.raw_level;
  else { while (level + 1 < A.n_levels && (int)blockIdx.x >= A.tile_begin[level + 1]) ++level; }
  const int b = raw ? A.raw_image : (int)blockIdx.y;
  if (A.image_sel && A.image_sel[b] < 0) return;           // (uniform over the CTA)
  const int w = A.f.w[level], h = A.f.h[level], pitch = A.f.pitch[level];
  const int tile = (int)blockIdx.x - (raw ? 0 : A.tile_begin[level]);
  const int tiles_x = (w + TW - 1) / TW;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int ox = tx * TW, oy = ty * TH;
  const uint8_t* img = A.f.lvl[level] + (size_t)b * A.f.img_stride[level];
  const int threshold = raw ? A.raw_threshold : 10;

  // stage the tile: 8-byte chunks (ox is a multiple of 8, the pitch a multiple of 16 => chunks are aligned); a chunk that
  // starts left of the image, or a row outside it, is zero.  Bytes at gx >= w come from the row padding / the next row:
  // no corner, score or Shi-Tomasi window that is evaluated ever reads them (gx + 5 < w for every evaluated pixel).
  if (threadIdx.x == 0) s_n = 0;
  for (int i = threadIdx.x; i < PH * (PP / 8); i += NT) {
    const int r = i / (PP / 8), c8 = i - r * (PP / 8);
    const int gx = ox - XOFF + 8 * c8, gy = oy - HALO + r;
    uint2 v = make_uint2(0u, 0u);
    if (gx >= 0 && gy >= 0 && gx < pitch && gy < h) v = __ldg(reinterpret_cast<const uint2*>(img + (size_t)gy * pitch + gx));
    *reinterpret_cast<uint2*>(&s_px[r * PP + 8 * c8]) = v;
  }
  __syncthreads();

  // pass A: S - 1 of every pixel of the score tile, four pixels per thread.  Task (sr, sg): pixels gx = ox - 4 + 4 sg + {0..3},
  // gy = oy - 1 + sr; in the staged tile that is word COL0 / 4 + sg of row ROW0 + sr.  A warp = one score row.
  const uint32_t* s_w = reinterpret_cast<const uint32_t*>(s_px);
  const uint32_t thr_hi = (uint32_t)(257 + threshold) * 0x00010001u, thr_lo = (uint32_t)(255 - threshold) * 0x00010001u | 0x80008000u;
  const int sg = threadIdx.x & 31;
  const int gx0 = ox - 4 + 4 * sg;
  // pixels of the group inside [3, w - 3), as a byte mask of the score word
  uint32_t colmask = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) if (gx0 + k >= 3 && gx0 + k < w - 3) colmask |= 0xffu << (8 * k);
#pragma unroll 1
  for (int it = 0; it < 4; ++it) {
    const int sr = it * 8 + (threadIdx.x >> 5);
    const int gy = oy - 1 + sr;
    uint32_t word = 0;
    if (gy >= 3 && gy < h - 3 && colmask) {                // (uniform over the warp except for colmask at the image's right edge)
      uint32_t W[7][3];
      const uint32_t* q = s_w + (sr + ROW0 - 3) * PW + (COL0 / 4 - 1) + sg;      // row gy - 3, word left of the group
#pragma unroll
      for (int r = 0; r < 7; ++r) { W[r][0] = q[r * PW]; W[r][1] = q[r * PW + 1]; W[r][2] = q[r * PW + 2]; }
      const uint32_t c = W[3][1];
      const uint32_t bE = (c & 0x00ff00ffu) + 0x01000100u, bO = __byte_perm(c, 0u, 0x4341) + 0x01000100u;
      uint32_t XE[16], XO[16];
      RingFill<0>::run(W, bE, bO, XE, XO);
      if (__any_sync(__activemask(), group_may_have_corner(XE, XO, thr_hi, thr_lo))) {
        uint32_t sE = arc_score_lanes(XE), sO = arc_score_lanes(XO);
        sE = __vmaxu2(sE, 0x01010101u) - 0x01010101u;      // S - 1 (biased by 256 -> - 257), clamped at 0: <= 254 per lane
        sO = __vmaxu2(sO, 0x01010101u) - 0x01010101u;
        word = (sE | (sO << 8)) & colmask;
      }
    }
    s_scw[sr * SG + sg] = word;
  }
  __syncthreads();

  // pass C: strict 3x3 non-max suppression on 16-bit lanes, four pixels per thread.  Task (r, g): pixels gx = ox + 4 g + {0..3},
  // gy = oy + r = score-tile row r + 1, word g + 1.  keep <=> s >= t (a corner) and s > every neighbour.
  const uint32_t t_l = (uint32_t)threshold * 0x00010001u;
  for (int j = threadIdx.x; j < (TH * (TW / 4) + 31) / 32 * 32; j += NT) {         // (rounded up: whole warps reach the ballots below)
    uint32_t keepE = 0, keepO = 0, cE = 0, cO = 0;
    const int r = j / (TW / 4), g = j - r * (TW / 4);
    const bool live = j < TH * (TW / 4);
    if (live) {
      uint32_t LE[3], CE[3], CO[3], RO[3];
#pragma unroll
      for (int dr = 0; dr < 3; ++dr) {
        const uint32_t* q = s_scw + (r + dr) * SG + g;
        const uint32_t l = q[0], c = q[1], rr = q[2];
        CE[dr] = c & 0x00ff00ffu; CO[dr] = __byte_perm(c, 0u, 0x4341);
        LE[dr] = __byte_perm(__byte_perm(l, 0u, 0x4341), CO[dr], 0x5432);   // left neighbours of pixels 0, 2: pixel 3 of the left group, pixel 1
        RO[dr] = __byte_perm(CE[dr], rr & 0x00ff00ffu, 0x5432);             // right neighbours of pixels 1, 3: pixel 2, pixel 0 of the right group
      }
      cE = CE[1]; cO = CO[1];
      const uint32_t mE = __vmaxu2(__vimax3_u16x2(__vimax3_u16x2(LE[0], CE[0], CO[0]), LE[2], CE[2]), __vimax3_u16x2(CO[2], LE[1], CO[1]));
      const uint32_t mO = __vmaxu2(__vimax3_u16x2(__vimax3_u16x2(CE[0], CO[0], RO[0]), CE[2], CO[2]), __vimax3_u16x2(RO[2], CE[1], RO[1]));
      const bool nms = !raw || A.raw_nonmax;
      // bit 15 / 31: s >= t and (s >= m + 1 or no suppression)
      keepE = ((cE | 0x80008000u) - t_l) & (nms ? ((cE | 0x80008000u) - (mE + 0x00010001u)) : 0xffffffffu) & 0x80008000u;
      keepO = ((cO | 0x80008000u) - t_l) & (nms ? ((cO | 0x80008000u) - (mO + 0x00010001u)) : 0xffffffffu) & 0x80008000u;
      if (raw) {
        const int gy = oy + r;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int gx = ox + 4 * g + k;
          const uint32_t keep = (k & 1) ? keepO : keepE, sc = (k & 1) ? cO : cE;
          const int sh = (k & 2) ? 16 : 0;
          if (gx < w && gy < h) A.raw_scores[(size_t)gy * w + gx] = ((keep >> (sh + 15)) & 1u) ? (uint8_t)((sc >> sh) & 0xffu) : (uint8_t)0;
        }
        keepE = keepO = 0;
      }
    }
    const uint32_t any = keepE | (keepO >> 1);              // bits 15, 14, 31, 30: pixels 0, 1, 2, 3
    const int mine = __popc(any);
    if (__any_sync(0xffffffffu, mine != 0)) {
      int slot = list_reserve(mine, &s_n);
      const int base = (r + 1) * SW + 4 * (g + 1);
      if (any & (1u << 15)) s_kp[slot++] = (unsigned short)(base + 0);
      if (any & (1u << 14)) s_kp[slot++] = (unsigned short)(base + 1);
      if (any & (1u << 31)) s_kp[slot++] = (unsigned short)(base + 2);
      if (any & (1u << 30)) s_kp[slot++] = (unsigned short)(base + 3);
    }
  }
  __syncthreads();
  // pass D: grid cell, occupancy, Shi-Tomasi score and the cell's 64-bit atomicMax, one thread per keypoint
  const int n_kp = s_n;
  for (int j = threadIdx.x; j < n_kp; j += NT) {
    const int idx = s_kp[j];
    const int sr = idx / SW, c = idx - sr * SW;
    const int gx = ox - 4 + c, gy = oy - 1 + sr;
    if (gx >= w || gy >= h) continue;
    // cell index: xy is a cv::Point2f, scale an int, cell_size_ an int (feature_detection.cpp:99-100)
    const float scale = (float)(1 << level);
    const int k = (int)(((float)gy * scale) / (float)A.cell) * A.grid_cols + (int)(((float)gx * scale) / (float)A.cell);
    if (A.occupancy && A.occupancy[(size_t)b * A.n_cells + k]) continue;
    float score = 0.0f;
    if (!(gx - 4 < 1 || gx + 4 >= w - 1 || gy - 4 < 1 || gy + 4 >= h - 1))
      score = shi_tomasi_smem(&s_px[(sr + ROW0) * PP + (c + COL0)]);
    const uint32_t order = ((uint32_t)level << 28) | ((uint32_t)gy << 14) | (uint32_t)gx;
    const unsigned long long key = ((unsigned long long)ordered_bits(score) << 32) | (unsigned long long)(~order);
    atomicMax(&A.keys[(size_t)b * A.n_cells + k], key);
  }
}

__global__ void fast_init_keys_kernel(unsigned long long* keys, int n, float thr_f)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = ((unsigned long long)ordered_bits(thr_f) << 32) | 0xFFFFFFFFull;
}

// decode cell records; one CTA per image counts its features
__global__ void fast_finalize_kernel(const unsigned long long* keys, int n_cells, float thr_f, double thr,
                                     svob200_corner* cells, int* counts, const int* image_sel)
{
  const int b = blockIdx.x;
  if (image_sel && image_sel[b] < 0) { if (threadIdx.x == 0 && counts) counts[b] = 0; return; }
  int local = 0;
  for (int k = threadIdx.x; k < n_cells; k += blockDim.x) {
    const unsigned long long key = keys[(size_t)b * n_cells + k];
    svob200_corner c;
    if ((uint32_t)key == 0xFFFFFFFFu) { c.x = 0; c.y = 0; c.level = 0; c.score = thr_f; }
    else {
      const uint32_t order = ~(uint32_t)key;
      c.level = (int)(order >> 28);
      const int y = (int)((order >> 14) & 0x3FFF), x = (int)(order & 0x3FFF);
      c.x = x << c.level; c.y = y << c.level;
      c.score = from_ordered_bits((uint32_t)(key >> 32));
    }
    cells[(size_t)b * n_cells + k] = c;
    if ((double)c.score > thr) ++local;                        // feature_detection.cpp:117
  }
  local = warp_sum_i(local);
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(&s_cnt, local);
  __syncthreads();
  if (threadIdx.x == 0 && counts) counts[b] = s_cnt;
}

// stand-alone vk::shiTomasiScore(img, u, v) (vision.cpp:113-154) for n points of one image
__global__ void shi_tomasi_points_kernel(const uint8_t* img, int pitch, int cols, int rows, int n, const int* uv, float* out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int u = uv[2 * i], v = uv[2 * i + 1];
  const int halfbox = 4;
  if (u - halfbox < 1 || u + halfbox >= cols - 1 || v - halfbox < 1 || v + halfbox >= rows - 1) { out[i] = 0.f; return; }   // :129
  float dXX = 0.f, dYY = 0.f, dXY = 0.f;
  for (int y = -4; y < 4; ++y) {
    const uint8_t* r = img + (size_t)(v + y) * pitch + u;
    for (int x = -4; x < 4; ++x) {
      const float dx = (float)((int)r[x + 1] - (int)r[x - 1]);
      const float dy = (float)((int)r[x + pitch] - (int)r[x - pitch]);
      dXX += dx * dx; dYY += dy * dy; dXY += dx * dy;
    }
  }
  dXX = (float)((double)dXX / 128.0);
  dYY = (float)((double)dYY / 128.0);
  dXY = (float)((double)dXY / 128.0);
  const float tr = dXX + dYY;
  const float disc = tr * tr - 4 * (dXX * dYY - dXY * dXY);
  out[i] = (float)(0.5 * ((double)tr - sqrt((double)disc)));
}

}  // namespace

cudaError_t launch_fast_detect(const DevFrame& f, int n_detect_levels, int cell, int grid_cols, int grid_rows, double thr,
                               const uint8_t* d_occupancy, unsigned long long* d_keys, svob200_corner* d_cells, int* d_counts,
                               cudaStream_t s, long long* launches, const int* d_image_sel)
{
  const int n_cells = grid_cols * grid_rows;
  const int total = n_cells * f.batch;
  const float thr_f = (float)thr;
  fast_init_keys_kernel<<<(total + 255) / 256, 256, 0, s>>>(d_keys, total, thr_f);
  FastArgs A{};
  A.f = f; A.n_levels = n_detect_levels; A.cell = cell; A.grid_cols = grid_cols; A.n_cells = n_cells; A.thr_f = thr_f;
  A.occupancy = d_occupancy; A.image_sel = d_image_sel; A.keys = d_keys; A.raw_scores = nullptr;
  A.tile_begin[0] = 0;
  for (int l = 0; l < n_detect_levels; ++l) {
    A.tiles_x[l] = (f.w[l] + TW - 1) / TW;
    A.tile_begin[l + 1] = A.tile_begin[l] + A.tiles_x[l] * ((f.h[l] + TH - 1) / TH);
  }
  dim3 grid(A.tile_begin[n_detect_levels], f.batch);
  fast_kernel<<<grid, NT, 0, s>>>(A);
  fast_finalize_kernel<<<f.batch, 256, 0, s>>>(d_keys, n_cells, thr_f, thr, d_cells, d_counts, d_image_sel);
  *launches += 3;
  return cudaGetLastError();
}

cudaError_t launch_fast_raw(const DevFrame& f, int image, int level, int threshold, int nonmax, uint8_t* d_scores,
                            cudaStream_t s, long long* launches)
{
  FastArgs A{};
  A.f = f; A.n_levels = 1; A.raw_scores = d_scores; A.raw_image = image; A.raw_level = level;
  A.raw_threshold = threshold; A.raw_nonmax = nonmax;
  const int tiles = ((f.w[level] + TW - 1) / TW) * ((f.h[level] + TH - 1) / TH);
  fast_kernel<<<dim3(tiles, 1), NT, 0, s>>>(A);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_shi_tomasi_points(const uint8_t* d_img, int pitch, int cols, int rows, int n, const int* d_uv, float* d_out,
                                     cudaStream_t s, long long* launches)
{
  if (n <= 0) return cudaSuccess;
  shi_tomasi_points_kernel<<<(n + 127) / 128, 128, 0, s>>>(d_img, pitch, cols, rows, n, d_uv, d_out);
  ++*launches;
  return cudaGetLastError();
}
