// ctx_internal.h — context / frame-store internals shared by capi.cu and tracker.cu.
#pragma once
#include <cstdio>
#include <cstring>
#include <cstdarg>
#include <string>
#include <vector>
#include <unordered_map>
#include <mutex>
#include <algorithm>
#include "common.cuh"
#include "kernels.h"

constexpr int kMaxFrames = 4096;

struct FrameRec {
  DevFrame f;
  uint8_t* base = nullptr;       // owned allocation (all levels)
  size_t bytes = 0;              // its size
  uint8_t* own_l0 = nullptr;     // owned level-0 storage (f.lvl[0] may alias caller memory: frame_bind_level0)
  int own_pitch0 = 0;
  int slot = -1;
};

struct GrowBuf {
  void* p = nullptr; size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = std::max(n, (size_t)1 << 16);
    want = (want + (want >> 2) + 255) & ~(size_t)255;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct svob200_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  long long launches = 0;
  std::unordered_map<int64_t, FrameRec> frames;
  std::vector<int> free_slots;
  // allocations of released SMALL frames, kept for the next frame_create of the same size: a caller that mirrors one camera
  // frame per step (the C++ drop-in) would otherwise pay a cudaMalloc and a cudaFree per frame (~0.1 ms, more than the kernels)
  std::vector<std::pair<size_t, uint8_t*>> spare_frames;
  DevFrame* d_table = nullptr;
  // staging arenas (HOST mem mode)
  uint8_t* h_stage = nullptr; size_t h_cap = 0;
  GrowBuf d_stage, d_scratch, d_scratch2;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // streams on which work of this context may still be in flight after an asynchronous call returned (a tracker's
  // depth-filter stream): every synchronising entry point joins them into `stream` first (ctx_join_aux)
  std::vector<std::pair<cudaStream_t, cudaEvent_t>> aux;
  std::mutex mu;
};

inline int fail(svob200_ctx* c, int code, const char* fmt, ...)
{
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  if (c) c->err = buf;
  return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, SVOB200_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); } while (0)

// make ctx->stream wait for everything enqueued so far on the auxiliary streams
inline int ctx_join_aux(svob200_ctx* ctx)
{
  for (auto& a : ctx->aux) {
    CU(cudaEventRecord(a.second, a.first));
    CU(cudaStreamWaitEvent(ctx->stream, a.second, 0));
  }
  return 0;
}
inline int ctx_add_aux(svob200_ctx* ctx, cudaStream_t s)
{
  cudaEvent_t e = nullptr;
  CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  ctx->aux.push_back({s, e});
  return 0;
}
inline void ctx_remove_aux(svob200_ctx* ctx, cudaStream_t s)
{
  for (size_t i = 0; i < ctx->aux.size(); ++i)
    if (ctx->aux[i].first == s) { cudaEventDestroy(ctx->aux[i].second); ctx->aux.erase(ctx->aux.begin() + i); return; }
}

inline DevCam to_cam(const svob200_camera* c) { DevCam d; d.width = c->width; d.height = c->height; d.fx = c->fx; d.fy = c->fy; d.cx = c->cx; d.cy = c->cy; return d; }

inline FrameRec* find_frame(svob200_ctx* ctx, int64_t id)
{
  auto it = ctx->frames.find(id);
  return it == ctx->frames.end() ? nullptr : &it->second;
}

inline int ensure_host_stage(svob200_ctx* ctx, size_t n)
{
  if (n <= ctx->h_cap) return 0;
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  ctx->h_stage = nullptr; ctx->h_cap = 0;
  size_t want = std::max(n, (size_t)1 << 16);
  want = (want + (want >> 2) + 255) & ~(size_t)255;
  CU(cudaMallocHost((void**)&ctx->h_stage, want));
  ctx->h_cap = want;
  return 0;
}

// Three-region staging plan: IN | INOUT | OUT.  Device copies cover [0, end(INOUT)) on the way in
// and [begin(INOUT), end) on the way out — one cudaMemcpyAsync each way per call.
struct Stage {
  svob200_ctx* ctx; int mem;
  struct Item { const void* src; void* dst; size_t bytes, off; int kind; };   // kind 0 in, 1 inout, 2 out
  std::vector<Item> items;
  size_t total = 0, in_end = 0, io_begin = 0;
  bool pushed = false, drained = false;
  Stage(svob200_ctx* c, int m) : ctx(c), mem(m) {}
  // a call that fails between push() and download() must not leave its host->device copy in flight: the next call's upload()
  // writes the same pinned staging buffer
  ~Stage() { if (pushed && !drained) cudaStreamSynchronize(ctx->stream); }
  // returns an index; resolve() gives the device pointer
  int add(const void* src, void* dst, size_t bytes, int kind) { items.push_back({src, dst, bytes, 0, kind}); return (int)items.size() - 1; }
  int layout()
  {
    if (mem == SVOB200_MEM_DEVICE) return 0;
    size_t off = 0;
    for (int kind = 0; kind < 3; ++kind) {
      if (kind == 1) io_begin = off;
      for (auto& it : items) if (it.kind == kind) { it.off = off; off += (it.bytes + 255) & ~(size_t)255; }
      if (kind == 1) in_end = off;
    }
    total = off;
    if (int r = ensure_host_stage(ctx, total)) return r;
    if (ctx->d_stage.ensure(total) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "device staging alloc of %zu bytes failed", total);
    return 0;
  }
  template <class T> T* dev(int idx)
  {
    Item& it = items[idx];
    if (mem == SVOB200_MEM_DEVICE) return (T*)(it.kind == 2 ? it.dst : (it.kind == 1 ? it.dst : const_cast<void*>(it.src)));
    return reinterpret_cast<T*>(static_cast<uint8_t*>(ctx->d_stage.p) + it.off);
  }
  template <class T> T* host(int idx) { return reinterpret_cast<T*>(ctx->h_stage + items[idx].off); }   // staged host copy (HOST mode)
  int upload()
  {
    if (mem == SVOB200_MEM_DEVICE) return 0;
    for (auto& it : items) if (it.kind <= 1 && it.src && it.bytes) memcpy(ctx->h_stage + it.off, it.src, it.bytes);
    return 0;
  }
  int push()
  {
    if (mem == SVOB200_MEM_DEVICE || in_end == 0) return 0;
    pushed = true;
    CU(cudaMemcpyAsync(ctx->d_stage.p, ctx->h_stage, in_end, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
  }
  int download()
  {
    if (mem == SVOB200_MEM_DEVICE) return 0;
    if (total > io_begin)
      CU(cudaMemcpyAsync(ctx->h_stage + io_begin, static_cast<uint8_t*>(ctx->d_stage.p) + io_begin, total - io_begin, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    drained = true;
    for (auto& it : items) if (it.kind >= 1 && it.dst && it.bytes) memcpy(it.dst, ctx->h_stage + it.off, it.bytes);
    return 0;
  }
};

// Level 0 of a frame is its own storage or aliases a caller's device buffer; only these two switch it, and they rewrite the
// frame's row of the device table on ctx->stream.  Bind rejects (SVOB200_ERR_ARG, nothing changes) a buffer or stride that
// is not 16-byte aligned and a stride below the width; copy_pixels copies the aliased images into the frame's own storage.
int frame_bind_level0(svob200_ctx* ctx, FrameRec* r, const uint8_t* dev_gray, int stride);
int frame_own_level0(svob200_ctx* ctx, FrameRec* r, bool copy_pixels);

// rounding of every pyramid step l -> l+1: the caller's round_modes, or the reference's x86 dispatch on the level's width
inline void pyramid_round_modes(const DevFrame& f, const int* round_modes, int* modes)
{
  for (int l = 0; l + 1 < f.n_levels; ++l) modes[l] = round_modes ? round_modes[l] : svob200_round_mode_x86(f.w[l]);
}
