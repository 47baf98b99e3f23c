// capi.cu — the C ABI of libsvob200 (include/svob200.h): context, device-resident frame store,
// host<->device staging and the entry points that launch the kernels.  No compute happens on the
// host here; a missing / unusable GPU makes every call fail with SVOB200_ERR_CUDA.
#include "ctx_internal.h"

namespace {

// rewrite ref_frame_id -> frame-table slot in the staged copy of the feature records
int resolve_slots(svob200_ctx* ctx, svob200_feature_ref* staged, int n)
{
  int64_t last_id = 0; int last_slot = -1; bool have = false;
  for (int i = 0; i < n; ++i) {
    const int64_t id = staged[i].ref_frame_id;
    if (!have || id != last_id) {
      FrameRec* r = find_frame(ctx, id);
      if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "reference frame %lld of item %d is not resident", (long long)id, i);
      last_id = id; last_slot = r->slot; have = true;
    }
    staged[i].ref_frame_id = last_slot;
  }
  return 0;
}

}  // namespace

int frame_bind_level0(svob200_ctx* ctx, FrameRec* r, const uint8_t* dev_gray, int stride)
{
  if (stride < r->f.w[0] || (stride & 15) || (reinterpret_cast<uintptr_t>(dev_gray) & 15))
    return fail(ctx, SVOB200_ERR_ARG, "frame_bind: buffer and stride must be 16-byte aligned and stride >= width");
  r->f.lvl[0] = const_cast<uint8_t*>(dev_gray); r->f.pitch[0] = stride; r->f.img_stride[0] = (unsigned long long)stride * r->f.h[0];
  CU(cudaMemcpyAsync(ctx->d_table + r->slot, &r->f, sizeof(DevFrame), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int frame_own_level0(svob200_ctx* ctx, FrameRec* r, bool copy_pixels)
{
  if (r->f.lvl[0] == r->own_l0) return 0;
  if (copy_pixels)
    CU(cudaMemcpy2DAsync(r->own_l0, r->own_pitch0, r->f.lvl[0], r->f.pitch[0], r->f.w[0], (size_t)r->f.h[0] * r->f.batch, cudaMemcpyDeviceToDevice, ctx->stream));
  r->f.lvl[0] = r->own_l0; r->f.pitch[0] = r->own_pitch0; r->f.img_stride[0] = (unsigned long long)r->own_pitch0 * r->f.h[0];
  CU(cudaMemcpyAsync(ctx->d_table + r->slot, &r->f, sizeof(DevFrame), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

extern "C" {

int svob200_ctx_create(int device, svob200_ctx** out)
{
  if (!out) return SVOB200_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return SVOB200_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return SVOB200_ERR_CUDA;
  svob200_ctx* ctx = new svob200_ctx();
  ctx->device = device;
  // the context's stream carries the tracking chain; it gets the highest priority so that, beside a tracker's asynchronous
  // depth-filter stream (default priority), its CTAs are scheduled first when slots free up
  int prio_least = 0, prio_greatest = 0;
  cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
  if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) { delete ctx; return SVOB200_ERR_CUDA; }
  if (cudaMalloc((void**)&ctx->d_table, sizeof(DevFrame) * kMaxFrames) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return SVOB200_ERR_CUDA; }
  for (int i = kMaxFrames - 1; i >= 0; --i) ctx->free_slots.push_back(i);
  *out = ctx;
  return SVOB200_OK;
}

void svob200_ctx_destroy(svob200_ctx* ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  ctx_join_aux(ctx);
  cudaStreamSynchronize(ctx->stream);
  for (auto& a : ctx->aux) cudaEventDestroy(a.second);
  for (auto& kv : ctx->frames) if (kv.second.base) cudaFree(kv.second.base);
  for (auto& sp : ctx->spare_frames) cudaFree(sp.second);
  if (ctx->d_table) cudaFree(ctx->d_table);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  ctx->d_stage.release(); ctx->d_scratch.release(); ctx->d_scratch2.release();
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* svob200_last_error(const svob200_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (no usable CUDA device?)"; }
int svob200_ctx_sync(svob200_ctx* ctx)
{
  if (!ctx) return SVOB200_ERR_ARG;
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}
void* svob200_ctx_stream(svob200_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
long long svob200_ctx_launch_count(const svob200_ctx* ctx) { return ctx ? ctx->launches : 0; }

int svob200_ctx_timer_start(svob200_ctx* ctx)
{
  if (!ctx) return SVOB200_ERR_ARG;
  if (!ctx->ev0) { CU(cudaEventCreate(&ctx->ev0)); CU(cudaEventCreate(&ctx->ev1)); }
  CU(cudaEventRecord(ctx->ev0, ctx->stream));
  return 0;
}
int svob200_ctx_timer_stop_ms(svob200_ctx* ctx, float* ms)
{
  if (!ctx || !ms || !ctx->ev0) return SVOB200_ERR_ARG;
  if (int e = ctx_join_aux(ctx)) return e;            // the stop event covers work still in flight on a tracker's depth-filter stream
  CU(cudaEventRecord(ctx->ev1, ctx->stream));
  CU(cudaEventSynchronize(ctx->ev1));
  CU(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return 0;
}

// sizeof() of every struct that crosses the ABI, in header order, so bindings can verify their layout
int svob200_abi_sizes(int* sizes, int cap)
{
  const int v[] = {(int)sizeof(svob200_camera), (int)sizeof(svob200_corner), (int)sizeof(svob200_align_opts),
                   (int)sizeof(svob200_align_result), (int)sizeof(svob200_matcher_opts), (int)sizeof(svob200_feature_ref),
                   (int)sizeof(svob200_match_result), (int)sizeof(svob200_epi_result), (int)sizeof(svob200_seed),
                   (int)sizeof(svob200_seed_obs), (int)sizeof(svob200_step_stats), (int)sizeof(svob200_map_point),
                   (int)sizeof(svob200_reproj_result), (int)sizeof(svob200_reproj_stats), (int)sizeof(svob200_pose_opt_result),
                   (int)sizeof(svob200_pose_opt_opts)};
  const int n = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n && i < cap; ++i) sizes[i] = v[i];
  return n;
}

int svob200_round_mode_x86(int in_cols) { return (in_cols % 16) == 0 ? SVOB200_ROUND_SSE2 : SVOB200_ROUND_TRUNC; }

// ------------------------------------------------------------------ frames
int svob200_frame_create(svob200_ctx* ctx, int64_t frame_id, int batch, int w, int h, int n_levels)
{
  if (!ctx || batch <= 0 || w <= 0 || h <= 0 || n_levels < 1 || n_levels > SVOB200_MAX_LEVELS) return fail(ctx, SVOB200_ERR_ARG, "frame_create: bad arguments");
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (find_frame(ctx, frame_id)) return fail(ctx, SVOB200_ERR_ARG, "frame %lld already exists", (long long)frame_id);
  if (ctx->free_slots.empty()) return fail(ctx, SVOB200_ERR_NOMEM, "frame table full (%d)", kMaxFrames);
  FrameRec r;
  memset(&r.f, 0, sizeof(r.f));
  r.f.n_levels = n_levels; r.f.batch = batch;
  size_t total = 0;
  size_t off[SVOB200_MAX_LEVELS];
  int lw = w, lh = h;
  for (int l = 0; l < n_levels; ++l) {
    if (lw <= 0 || lh <= 0) return fail(ctx, SVOB200_ERR_ARG, "frame_create: level %d is empty", l);
    r.f.w[l] = lw; r.f.h[l] = lh; r.f.pitch[l] = align_up_i(lw, 64);
    r.f.img_stride[l] = (unsigned long long)r.f.pitch[l] * lh;
    off[l] = total;
    total += (size_t)r.f.img_stride[l] * batch;
    total = (total + 255) & ~(size_t)255;
    lw /= 2; lh /= 2;
  }
  total += 256;   // slack so word-granular reads at the very end stay inside the allocation
  for (size_t k = 0; k < ctx->spare_frames.size(); ++k)
    if (ctx->spare_frames[k].first == total) { r.base = ctx->spare_frames[k].second; ctx->spare_frames.erase(ctx->spare_frames.begin() + k); break; }
  if (!r.base && cudaMalloc((void**)&r.base, total) != cudaSuccess) { cudaGetLastError(); return fail(ctx, SVOB200_ERR_NOMEM, "frame_create: cudaMalloc(%zu) failed", total); }
  r.bytes = total;
  for (int l = 0; l < n_levels; ++l) r.f.lvl[l] = r.base + off[l];
  r.own_l0 = r.f.lvl[0]; r.own_pitch0 = r.f.pitch[0];
  r.slot = ctx->free_slots.back(); ctx->free_slots.pop_back();
  cudaError_t e = cudaMemsetAsync(r.base, 0, total, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_table + r.slot, &r.f, sizeof(DevFrame), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);      // r.f is a stack object
  if (e != cudaSuccess) {                                             // nothing is left behind: the allocation and the table slot go back
    cudaFree(r.base);
    ctx->free_slots.push_back(r.slot);
    return fail(ctx, SVOB200_ERR_CUDA, "frame_create: %s", cudaGetErrorString(e));
  }
  ctx->frames[frame_id] = r;
  return SVOB200_OK;
}

static int build_levels(svob200_ctx* ctx, FrameRec* r, const int* round_modes)
{
  int modes[SVOB200_MAX_LEVELS];
  pyramid_round_modes(r->f, round_modes, modes);
  if (launch_pyramid(r->f, modes, ctx->stream, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "pyramid launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return 0;
}

int svob200_frame_upload(svob200_ctx* ctx, int64_t frame_id, const uint8_t* gray, int stride, const int* round_modes, int mem)
{
  if (!ctx || !gray) return fail(ctx, SVOB200_ERR_ARG, "frame_upload: null argument");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (stride < r->f.w[0]) return fail(ctx, SVOB200_ERR_ARG, "frame_upload: stride < width");
  if (int e = frame_own_level0(ctx, r, false)) return e;
  CU(cudaMemcpy2DAsync(r->f.lvl[0], r->f.pitch[0], gray, stride, r->f.w[0], (size_t)r->f.h[0] * r->f.batch,
                       mem == SVOB200_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
  if (int e = build_levels(ctx, r, round_modes)) return e;
  if (mem == SVOB200_MEM_HOST) CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// Level 0 aliases the caller's device buffer (the reference's level 0 aliases the caller's cv::Mat,
// frame.cpp:189): no copy at all, the pyramid kernel reads the frame where it already is in HBM.
int svob200_frame_bind(svob200_ctx* ctx, int64_t frame_id, const uint8_t* dev_gray, int stride, const int* round_modes)
{
  if (!ctx || !dev_gray) return fail(ctx, SVOB200_ERR_ARG, "frame_bind: null argument");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (int e = frame_bind_level0(ctx, r, dev_gray, stride)) return e;
  return build_levels(ctx, r, round_modes);
}

int svob200_frame_download(svob200_ctx* ctx, int64_t frame_id, int image, int level, uint8_t* out, int out_stride)
{
  if (!ctx || !out) return fail(ctx, SVOB200_ERR_ARG, "frame_download: null argument");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (level < 0 || level >= r->f.n_levels || image < 0 || image >= r->f.batch || out_stride < r->f.w[level]) return fail(ctx, SVOB200_ERR_ARG, "frame_download: bad level/image/stride");
  CU(cudaMemcpy2DAsync(out, out_stride, r->f.lvl[level] + (size_t)image * r->f.img_stride[level], r->f.pitch[level], r->f.w[level], r->f.h[level],
                       cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

int svob200_frame_release(svob200_ctx* ctx, int64_t frame_id)
{
  if (!ctx) return SVOB200_ERR_ARG;
  std::lock_guard<std::mutex> lk(ctx->mu);
  auto it = ctx->frames.find(frame_id);
  if (it == ctx->frames.end()) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaStreamSynchronize(ctx->stream));
  // frames of up to 8 MB (single camera images with their pyramid) go to the spare list, at most kSpareFrames of them
  constexpr size_t kSpareFrames = 8, kSpareBytes = 8u << 20;
  if (it->second.bytes <= kSpareBytes && ctx->spare_frames.size() < kSpareFrames) ctx->spare_frames.push_back({it->second.bytes, it->second.base});
  else cudaFree(it->second.base);
  ctx->free_slots.push_back(it->second.slot);
  ctx->frames.erase(it);
  return SVOB200_OK;
}

int svob200_frame_info(svob200_ctx* ctx, int64_t frame_id, int* batch, int* w, int* h, int* n_levels)
{
  FrameRec* r = ctx ? find_frame(ctx, frame_id) : nullptr;
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (batch) *batch = r->f.batch;
  if (w) *w = r->f.w[0];
  if (h) *h = r->f.h[0];
  if (n_levels) *n_levels = r->f.n_levels;
  return SVOB200_OK;
}

int svob200_frame_slot(svob200_ctx* ctx, int64_t frame_id)
{
  FrameRec* r = ctx ? find_frame(ctx, frame_id) : nullptr;
  return r ? r->slot : fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
}

int svob200_half_sample(svob200_ctx* ctx, const uint8_t* in, int w, int h, int in_stride, uint8_t* out, int out_stride, int round_mode)
{
  if (!ctx || !in || !out || w < 2 || h < 2 || in_stride < w || out_stride < w / 2) return fail(ctx, SVOB200_ERR_ARG, "half_sample: bad arguments");
  const int ip = align_up_i(w, 64), op = align_up_i(w / 2, 64);
  const size_t in_b = (size_t)ip * h, out_b = (size_t)op * (h / 2);
  if (ctx->d_scratch.ensure(in_b + out_b + 512) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "half_sample: scratch alloc failed");
  uint8_t* d_in = static_cast<uint8_t*>(ctx->d_scratch.p);
  uint8_t* d_out = d_in + ((in_b + 255) & ~(size_t)255);
  CU(cudaMemcpy2DAsync(d_in, ip, in, in_stride, w, h, cudaMemcpyHostToDevice, ctx->stream));
  if (launch_half_sample_single(d_in, ip, w, h, d_out, op, round_mode, ctx->stream, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "half_sample launch failed");
  CU(cudaMemcpy2DAsync(out, out_stride, d_out, op, w / 2, h / 2, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// ------------------------------------------------------------------ FAST
int svob200_fast_detect(svob200_ctx* ctx, int64_t frame_id, int n_detect_levels, int cell_size, double thr,
                        const uint8_t* occupancy, svob200_corner* cells_out, int* n_features_out, int mem)
{
  if (!ctx || !cells_out || cell_size <= 0) return fail(ctx, SVOB200_ERR_ARG, "fast_detect: bad arguments");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (n_detect_levels < 1 || n_detect_levels > r->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "fast_detect: n_detect_levels out of range");
  if (r->f.w[0] >= 16384 || r->f.h[0] >= 16384) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "fast_detect: image larger than 16383");
  const int gc = (r->f.w[0] + cell_size - 1) / cell_size, gr = (r->f.h[0] + cell_size - 1) / cell_size;
  const size_t n_cells = (size_t)gc * gr, total = n_cells * r->f.batch;
  Stage st(ctx, mem);
  const int i_occ = occupancy ? st.add(occupancy, nullptr, total, 0) : -1;
  const int i_cells = st.add(nullptr, cells_out, total * sizeof(svob200_corner), 2);
  const int i_cnt = st.add(nullptr, n_features_out, sizeof(int) * r->f.batch, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(total * 8 + sizeof(int) * r->f.batch + 256) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "fast_detect: scratch alloc failed");
  unsigned long long* d_keys = static_cast<unsigned long long*>(ctx->d_scratch.p);
  int* d_cnt = (mem == SVOB200_MEM_DEVICE && !n_features_out) ? reinterpret_cast<int*>(d_keys + total) : st.dev<int>(i_cnt);
  if (launch_fast_detect(r->f, n_detect_levels, cell_size, gc, gr, thr, occupancy ? st.dev<uint8_t>(i_occ) : nullptr, d_keys,
                         st.dev<svob200_corner>(i_cells), d_cnt, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "fast_detect launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

int svob200_fast_corners(svob200_ctx* ctx, int64_t frame_id, int image, int level, int threshold, int nonmax, int cap,
                         int* xs, int* ys, int* scores)
{
  if (!ctx) return SVOB200_ERR_ARG;
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (level < 0 || level >= r->f.n_levels || image < 0 || image >= r->f.batch) return fail(ctx, SVOB200_ERR_ARG, "fast_corners: bad level/image");
  const int w = r->f.w[level], h = r->f.h[level];
  const size_t n = (size_t)w * h;
  if (ctx->d_scratch.ensure(n + 256) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "fast_corners: scratch alloc failed");
  uint8_t* d_sc = static_cast<uint8_t*>(ctx->d_scratch.p);
  threshold = std::min(std::max(threshold, 0), 255);
  if (launch_fast_raw(r->f, image, level, threshold, nonmax, d_sc, ctx->stream, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "fast_corners launch failed");
  std::vector<uint8_t> sc(n);
  CU(cudaMemcpyAsync(sc.data(), d_sc, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  int cnt = 0;   // row-major compaction of the device score map (output formatting only)
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) {
      const int s = sc[(size_t)y * w + x];
      if (!s) continue;
      if (cnt < cap) { if (xs) xs[cnt] = x; if (ys) ys[cnt] = y; if (scores) scores[cnt] = s; }
      ++cnt;
    }
  return cnt;
}

// ------------------------------------------------------------------ sparse alignment
int svob200_sparse_align(svob200_ctx* ctx, int64_t ref_frame_id, int64_t cur_frame_id, const svob200_camera* cam, int batch,
                         const int* ftr_offsets, const double* px, const double* xyz_ref, const uint8_t* has_point,
                         const double* T_cur_ref, const svob200_align_opts* opts, svob200_align_result* results, int mem)
{
  if (!ctx || !cam || !ftr_offsets || !opts || !results || batch <= 0) return fail(ctx, SVOB200_ERR_ARG, "sparse_align: bad arguments");
  FrameRec* ref = find_frame(ctx, ref_frame_id);
  FrameRec* cur = find_frame(ctx, cur_frame_id);
  if (!ref || !cur) return fail(ctx, SVOB200_ERR_NOFRAME, "sparse_align: frame not resident");
  if (batch > ref->f.batch || batch > cur->f.batch) return fail(ctx, SVOB200_ERR_ARG, "sparse_align: batch exceeds the frames' batch");
  if (opts->max_level >= ref->f.n_levels || opts->max_level >= cur->f.n_levels || opts->min_level < 0 || opts->min_level > opts->max_level)
    return fail(ctx, SVOB200_ERR_ARG, "sparse_align: level range [%d,%d] outside the pyramid", opts->min_level, opts->max_level);
  int total = 0, max_per = 0;
  if (mem == SVOB200_MEM_HOST) {
    total = ftr_offsets[batch];
    for (int b = 0; b < batch; ++b) max_per = std::max(max_per, ftr_offsets[b + 1] - ftr_offsets[b]);
  } else {
    // device-resident offsets: one small read-back of the final offset (the scratch size depends on it)
    CU(cudaMemcpyAsync(&total, ftr_offsets + batch, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    max_per = total;
  }
  Stage st(ctx, mem);
  const int i_off = st.add(ftr_offsets, nullptr, sizeof(int) * (batch + 1), 0);
  const int i_px = st.add(px, nullptr, sizeof(double) * 2 * total, 0);
  const int i_xyz = st.add(xyz_ref, nullptr, sizeof(double) * 3 * total, 0);
  const int i_hp = st.add(has_point, nullptr, (size_t)total, 0);
  const int i_T = st.add(T_cur_ref, nullptr, sizeof(double) * 7 * batch, 0);
  const int i_res = st.add(nullptr, results, sizeof(svob200_align_result) * batch, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(sparse_align_scratch_bytes(total)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "sparse_align: scratch alloc failed");
  if (launch_sparse_align(ref->f, cur->f, to_cam(cam), batch, total, max_per, st.dev<int>(i_off), st.dev<double>(i_px), st.dev<double>(i_xyz),
                          st.dev<uint8_t>(i_hp), st.dev<double>(i_T), *opts, st.dev<svob200_align_result>(i_res), ctx->d_scratch.p,
                          ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "sparse_align launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ feature alignment
int svob200_align_patches(svob200_ctx* ctx, int64_t frame_id, int level, int n, const int* image, const uint8_t* pwb,
                          const uint8_t* patch, const float* dir, int n_iter, double* px, int* converged, double* h_inv, int mem)
{
  if (!ctx || n < 0 || !image || !pwb || !patch || !px || !converged) return fail(ctx, SVOB200_ERR_ARG, "align_patches: bad arguments");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (level < 0 || level >= r->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "align_patches: bad level");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_img = st.add(image, nullptr, sizeof(int) * n, 0);
  const int i_pwb = st.add(pwb, nullptr, (size_t)100 * n, 0);
  const int i_pat = st.add(patch, nullptr, (size_t)64 * n, 0);
  const int i_dir = dir ? st.add(dir, nullptr, sizeof(float) * 2 * n, 0) : -1;
  const int i_px = st.add(px, px, sizeof(double) * 2 * n, 1);
  const int i_cv = st.add(nullptr, converged, sizeof(int) * n, 2);
  const int i_hi = h_inv ? st.add(nullptr, h_inv, sizeof(double) * n, 2) : -1;
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(lk_jobs_bytes(n)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "align_patches: scratch alloc failed");
  if (launch_align_patches(ctx->d_table, r->slot, level, n, st.dev<int>(i_img), st.dev<uint8_t>(i_pwb), st.dev<uint8_t>(i_pat), dir ? st.dev<float>(i_dir) : nullptr,
                           n_iter, st.dev<double>(i_px), st.dev<int>(i_cv), h_inv ? st.dev<double>(i_hi) : nullptr, ctx->d_scratch.p, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "align_patches launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ matcher
void svob200_matcher_opts_default(svob200_matcher_opts* o, int n_pyr_levels)
{
  o->align_1d = 0; o->align_max_iter = 10; o->max_epi_search_steps = 1000; o->subpix_refinement = 1;
  o->epi_search_edgelet_filtering = 1; o->epi_search_edgelet_max_angle = 0.7; o->max_search_level = n_pyr_levels - 1;
}

int svob200_match_direct(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n, const svob200_feature_ref* ftrs,
                         const double* depth_ref, const double* px_cur_in, const svob200_matcher_opts* opts,
                         svob200_match_result* results, int mem)
{
  if (!ctx || !cam || n < 0 || !ftrs || !depth_ref || !px_cur_in || !opts || !results) return fail(ctx, SVOB200_ERR_ARG, "match_direct: bad arguments");
  FrameRec* cur = find_frame(ctx, cur_frame_id);
  if (!cur) return fail(ctx, SVOB200_ERR_NOFRAME, "match_direct: current frame not resident");
  if (opts->max_search_level >= cur->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "match_direct: max_search_level outside the pyramid");
  if (opts->max_epi_search_steps < 0) return fail(ctx, SVOB200_ERR_ARG, "match_direct: negative max_epi_search_steps");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_f = st.add(ftrs, nullptr, sizeof(svob200_feature_ref) * n, 0);
  const int i_d = st.add(depth_ref, nullptr, sizeof(double) * n, 0);
  const int i_p = st.add(px_cur_in, nullptr, sizeof(double) * 2 * n, 0);
  const int i_r = st.add(nullptr, results, sizeof(svob200_match_result) * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (mem == SVOB200_MEM_HOST) if (int e = resolve_slots(ctx, st.host<svob200_feature_ref>(i_f), n)) return e;
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(match_scratch_bytes(n)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "match_direct: scratch alloc failed");
  if (launch_match_direct(ctx->d_table, cur->slot, to_cam(cam), n, st.dev<svob200_feature_ref>(i_f), st.dev<double>(i_d),
                          st.dev<double>(i_p), *opts, st.dev<svob200_match_result>(i_r), nullptr, nullptr, ctx->d_scratch.p, n, 0, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "match_direct launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

int svob200_epipolar_match(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n, const svob200_feature_ref* ftrs,
                           const double* d, const svob200_matcher_opts* opts, svob200_epi_result* results, int mem)
{
  if (!ctx || !cam || n < 0 || !ftrs || !d || !opts || !results) return fail(ctx, SVOB200_ERR_ARG, "epipolar_match: bad arguments");
  FrameRec* cur = find_frame(ctx, cur_frame_id);
  if (!cur) return fail(ctx, SVOB200_ERR_NOFRAME, "epipolar_match: current frame not resident");
  if (opts->max_search_level >= cur->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "epipolar_match: max_search_level outside the pyramid");
  if (opts->max_epi_search_steps < 0) return fail(ctx, SVOB200_ERR_ARG, "epipolar_match: negative max_epi_search_steps");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_f = st.add(ftrs, nullptr, sizeof(svob200_feature_ref) * n, 0);
  const int i_d = st.add(d, nullptr, sizeof(double) * 3 * n, 0);
  const int i_r = st.add(nullptr, results, sizeof(svob200_epi_result) * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (mem == SVOB200_MEM_HOST) if (int e = resolve_slots(ctx, st.host<svob200_feature_ref>(i_f), n)) return e;
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(epipolar_scratch_bytes(n)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "epipolar_match: scratch alloc failed");
  if (launch_epipolar(ctx->d_table, cur->slot, to_cam(cam), n, st.dev<svob200_feature_ref>(i_f), st.dev<double>(i_d), *opts,
                      st.dev<svob200_epi_result>(i_r), ctx->d_scratch.p, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "epipolar launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ depth filter
int svob200_seeds_update(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int n, const svob200_feature_ref* ftrs,
                         const double* T_ref_w, const double* T_cur_w, const svob200_matcher_opts* opts, double conv_thresh,
                         svob200_seed* seeds, svob200_seed_obs* obs, int mem)
{
  if (!ctx || !cam || n < 0 || !ftrs || !T_ref_w || !T_cur_w || !opts || !seeds || !obs) return fail(ctx, SVOB200_ERR_ARG, "seeds_update: bad arguments");
  FrameRec* cur = find_frame(ctx, cur_frame_id);
  if (!cur) return fail(ctx, SVOB200_ERR_NOFRAME, "seeds_update: current frame not resident");
  if (opts->max_search_level >= cur->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "seeds_update: max_search_level outside the pyramid");
  if (opts->max_epi_search_steps < 0) return fail(ctx, SVOB200_ERR_ARG, "seeds_update: negative max_epi_search_steps");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_f = st.add(ftrs, nullptr, sizeof(svob200_feature_ref) * n, 0);
  const int i_tr = st.add(T_ref_w, nullptr, sizeof(double) * 7 * n, 0);
  const int i_tc = st.add(T_cur_w, nullptr, sizeof(double) * 7 * cur->f.batch, 0);
  const int i_s = st.add(seeds, seeds, sizeof(svob200_seed) * n, 1);
  const int i_o = st.add(nullptr, obs, sizeof(svob200_seed_obs) * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (mem == SVOB200_MEM_HOST) if (int e = resolve_slots(ctx, st.host<svob200_feature_ref>(i_f), n)) return e;
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(seeds_scratch_bytes(n)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "seeds_update: scratch alloc failed");
  if (launch_seeds_update(ctx->d_table, cur->slot, to_cam(cam), n, st.dev<svob200_feature_ref>(i_f), st.dev<double>(i_tr),
                          st.dev<double>(i_tc), *opts, conv_thresh, st.dev<svob200_seed>(i_s), st.dev<svob200_seed_obs>(i_o),
                          ctx->d_scratch.p, n, 0, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "seeds_update launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

int svob200_update_seed(svob200_ctx* ctx, int n, const float* x, const float* tau2, svob200_seed* seeds)
{
  if (!ctx || n < 0 || !x || !tau2 || !seeds) return fail(ctx, SVOB200_ERR_ARG, "update_seed: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_x = st.add(x, nullptr, sizeof(float) * n, 0);
  const int i_t = st.add(tau2, nullptr, sizeof(float) * n, 0);
  const int i_s = st.add(seeds, seeds, sizeof(svob200_seed) * n, 1);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_update_seed(n, st.dev<float>(i_x), st.dev<float>(i_t), st.dev<svob200_seed>(i_s), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "update_seed launch failed");
  return st.download();
}

int svob200_debug_chi2_chain(svob200_ctx* ctx, int block, int n_features, const float* res, const uint8_t* visible, const uint8_t* contrib,
                             float* sums, int* counts)
{
  if (!ctx || n_features <= 0 || !res || !visible || !contrib || !sums || !counts) return fail(ctx, SVOB200_ERR_ARG, "debug_chi2_chain: bad arguments");
  if (block != 128 && block != 256 && block != 512) return fail(ctx, SVOB200_ERR_ARG, "debug_chi2_chain: block must be 128, 256 or 512");
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_r = st.add(res, nullptr, sizeof(float) * 16 * (size_t)n_features, 0);
  const int i_v = st.add(visible, nullptr, (size_t)n_features, 0);
  const int i_c = st.add(contrib, nullptr, (size_t)n_features, 0);
  const int i_s = st.add(nullptr, sums, sizeof(float) * 3, 2);
  const int i_n = st.add(nullptr, counts, sizeof(int) * 3, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_chi2_chain_test(block, st.dev<float>(i_r), st.dev<uint8_t>(i_v), st.dev<uint8_t>(i_c), n_features, st.dev<float>(i_s), st.dev<int>(i_n),
                             ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "debug_chi2_chain launch failed");
  return st.download();
}

int svob200_compute_tau(svob200_ctx* ctx, int n, const double* T_ref_cur, const double* f, const double* z, double px_error_angle, double* tau_out)
{
  if (!ctx || n < 0 || !T_ref_cur || !f || !z || !tau_out) return fail(ctx, SVOB200_ERR_ARG, "compute_tau: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_T = st.add(T_ref_cur, nullptr, sizeof(double) * 7 * n, 0);
  const int i_f = st.add(f, nullptr, sizeof(double) * 3 * n, 0);
  const int i_z = st.add(z, nullptr, sizeof(double) * n, 0);
  const int i_o = st.add(nullptr, tau_out, sizeof(double) * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_compute_tau(n, st.dev<double>(i_T), st.dev<double>(i_f), st.dev<double>(i_z), px_error_angle, st.dev<double>(i_o), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "compute_tau launch failed");
  return st.download();
}

// ------------------------------------------------------------------ glue between operators
int svob200_features_prepare(svob200_ctx* ctx, const svob200_camera* cam, int n, const double* px, const double* pt_world,
                             const int* image, int batch, const double* T_ref_w, double* f_out, double* xyz_ref_out, int mem)
{
  if (!ctx || !cam || n < 0 || !px || !pt_world || !image || !T_ref_w || !xyz_ref_out || batch <= 0) return fail(ctx, SVOB200_ERR_ARG, "features_prepare: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_px = st.add(px, nullptr, sizeof(double) * 2 * n, 0);
  const int i_pt = st.add(pt_world, nullptr, sizeof(double) * 3 * n, 0);
  const int i_im = st.add(image, nullptr, sizeof(int) * n, 0);
  const int i_T = st.add(T_ref_w, nullptr, sizeof(double) * 7 * batch, 0);
  const int i_f = f_out ? st.add(nullptr, f_out, sizeof(double) * 3 * n, 2) : -1;
  const int i_x = st.add(nullptr, xyz_ref_out, sizeof(double) * 3 * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_features_prepare(to_cam(cam), n, st.dev<double>(i_px), st.dev<double>(i_pt), st.dev<int>(i_im), st.dev<double>(i_T),
                              f_out ? st.dev<double>(i_f) : nullptr, st.dev<double>(i_x), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "features_prepare launch failed");
  return st.download();
}

int svob200_compose_poses(svob200_ctx* ctx, int batch, const svob200_align_result* results, const double* T_ref_w, double* T_cur_w, int mem)
{
  if (!ctx || batch <= 0 || !results || !T_ref_w || !T_cur_w) return fail(ctx, SVOB200_ERR_ARG, "compose_poses: bad arguments");
  Stage st(ctx, mem);
  const int i_r = st.add(results, nullptr, sizeof(svob200_align_result) * batch, 0);
  const int i_T = st.add(T_ref_w, nullptr, sizeof(double) * 7 * batch, 0);
  const int i_o = st.add(nullptr, T_cur_w, sizeof(double) * 7 * batch, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_compose_poses(batch, st.dev<svob200_align_result>(i_r), st.dev<double>(i_T), st.dev<double>(i_o), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "compose_poses launch failed");
  return st.download();
}

int svob200_reproject_prepare(svob200_ctx* ctx, const svob200_camera* cam, int n, svob200_feature_ref* ftrs, const double* pt_world,
                              const double* T_kf_w, int batch, const double* T_cur_w, double* depth_ref_out, double* px_cur_out, int mem)
{
  if (!ctx || !cam || n < 0 || !ftrs || !pt_world || !T_kf_w || !T_cur_w || !depth_ref_out || !px_cur_out || batch <= 0)
    return fail(ctx, SVOB200_ERR_ARG, "reproject_prepare: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_pt = st.add(pt_world, nullptr, sizeof(double) * 3 * n, 0);
  const int i_Tk = st.add(T_kf_w, nullptr, sizeof(double) * 7 * n, 0);
  const int i_Tc = st.add(T_cur_w, nullptr, sizeof(double) * 7 * batch, 0);
  const int i_f = st.add(ftrs, ftrs, sizeof(svob200_feature_ref) * n, 1);
  const int i_d = st.add(nullptr, depth_ref_out, sizeof(double) * n, 2);
  const int i_p = st.add(nullptr, px_cur_out, sizeof(double) * 2 * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_reproject_prepare(to_cam(cam), n, st.dev<svob200_feature_ref>(i_f), st.dev<double>(i_pt), st.dev<double>(i_Tk), st.dev<double>(i_Tc),
                               st.dev<double>(i_d), st.dev<double>(i_p), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "reproject_prepare launch failed");
  return st.download();
}

// one level of one image of a resident frame, copied verbatim from host memory: lets a host-side
// image pyramid (Frame::img_pyr_) be mirrored on the device exactly as the host holds it
int svob200_frame_upload_level(svob200_ctx* ctx, int64_t frame_id, int image, int level, const uint8_t* data, int stride)
{
  if (!ctx || !data) return fail(ctx, SVOB200_ERR_ARG, "frame_upload_level: null argument");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (level < 0 || level >= r->f.n_levels || image < 0 || image >= r->f.batch || stride < r->f.w[level]) return fail(ctx, SVOB200_ERR_ARG, "frame_upload_level: bad level/image/stride");
  if (level == 0) if (int e = frame_own_level0(ctx, r, false)) return e;
  CU(cudaMemcpy2DAsync(r->f.lvl[level] + (size_t)image * r->f.img_stride[level], r->f.pitch[level], data, stride, r->f.w[level], r->f.h[level],
                       cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// vk::shiTomasiScore (vision.cpp:113-154) for n pixels of a host image
int svob200_shi_tomasi(svob200_ctx* ctx, const uint8_t* img, int w, int h, int stride, int n, const int* uv, float* scores)
{
  if (!ctx || !img || w <= 0 || h <= 0 || stride < w || n < 0 || !uv || !scores) return fail(ctx, SVOB200_ERR_ARG, "shi_tomasi: bad arguments");
  if (n == 0) return SVOB200_OK;
  const int pitch = align_up_i(w, 64);
  const size_t img_b = ((size_t)pitch * h + 255) & ~(size_t)255, uv_b = ((size_t)n * 8 + 255) & ~(size_t)255;
  if (ctx->d_scratch.ensure(img_b + uv_b + (size_t)n * 4 + 256) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "shi_tomasi: scratch alloc failed");
  uint8_t* d_img = static_cast<uint8_t*>(ctx->d_scratch.p);
  int* d_uv = reinterpret_cast<int*>(d_img + img_b);
  float* d_out = reinterpret_cast<float*>(d_img + img_b + uv_b);
  CU(cudaMemcpy2DAsync(d_img, pitch, img, stride, w, h, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_uv, uv, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  if (launch_shi_tomasi_points(d_img, pitch, w, h, n, d_uv, d_out, ctx->stream, &ctx->launches)) return fail(ctx, SVOB200_ERR_CUDA, "shi_tomasi launch failed");
  CU(cudaMemcpyAsync(scores, d_out, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// warp::getWarpMatrixAffine (matcher.cpp:36-60) for n items; A_out row-major 2x2 per item
int svob200_warp_matrix_affine(svob200_ctx* ctx, const svob200_camera* cam, int n, const double* px_ref, const double* f_ref,
                               const double* depth_ref, const double* T_cur_ref, const int* level_ref, double* A_out, int mem)
{
  if (!ctx || !cam || n < 0 || !px_ref || !f_ref || !depth_ref || !T_cur_ref || !level_ref || !A_out) return fail(ctx, SVOB200_ERR_ARG, "warp_matrix_affine: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, mem);
  const int i_px = st.add(px_ref, nullptr, sizeof(double) * 2 * n, 0);
  const int i_f = st.add(f_ref, nullptr, sizeof(double) * 3 * n, 0);
  const int i_d = st.add(depth_ref, nullptr, sizeof(double) * n, 0);
  const int i_T = st.add(T_cur_ref, nullptr, sizeof(double) * 7 * n, 0);
  const int i_l = st.add(level_ref, nullptr, sizeof(int) * n, 0);
  const int i_A = st.add(nullptr, A_out, sizeof(double) * 4 * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_warp_matrix(to_cam(cam), n, st.dev<double>(i_px), st.dev<double>(i_f), st.dev<double>(i_d), st.dev<double>(i_T), st.dev<int>(i_l),
                         st.dev<double>(i_A), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "warp_matrix_affine launch failed");
  return st.download();
}

// warp::warpAffine (matcher.cpp:83-116) on a host image level; patch: (2*halfpatch)^2 bytes, in/out
// (left untouched when the warp matrix inverts to NaN, like the reference)
int svob200_warp_affine(svob200_ctx* ctx, const uint8_t* img, int w, int h, int stride, const double* A_cur_ref, const double* px_ref,
                        int level_ref, int search_level, int halfpatch_size, uint8_t* patch)
{
  if (!ctx || !img || w <= 0 || h <= 0 || stride < w || !A_cur_ref || !px_ref || halfpatch_size <= 0 || halfpatch_size > 64 || !patch
      || level_ref < 0 || level_ref > 30 || search_level < 0 || search_level > 30)
    return fail(ctx, SVOB200_ERR_ARG, "warp_affine: bad arguments");
  const int pitch = align_up_i(w, 64), np = 4 * halfpatch_size * halfpatch_size;
  const size_t img_b = ((size_t)pitch * h + 255) & ~(size_t)255;
  if (ctx->d_scratch.ensure(img_b + np + 256) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "warp_affine: scratch alloc failed");
  uint8_t* d_img = static_cast<uint8_t*>(ctx->d_scratch.p);
  uint8_t* d_patch = d_img + img_b;
  CU(cudaMemcpy2DAsync(d_img, pitch, img, stride, w, h, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_patch, patch, np, cudaMemcpyHostToDevice, ctx->stream));
  if (launch_warp_affine(d_img, pitch, w, h, A_cur_ref, px_ref, level_ref, search_level, halfpatch_size, d_patch, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "warp_affine launch failed");
  CU(cudaMemcpyAsync(patch, d_patch, np, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// depthFromTriangulation (matcher.cpp:123-136) for n items; depth is in/out (left untouched where ok = 0)
int svob200_depth_from_triangulation(svob200_ctx* ctx, int n, const double* T_search_ref, const double* f_ref, const double* f_cur,
                                     double* depth, int* ok)
{
  if (!ctx || n < 0 || !T_search_ref || !f_ref || !f_cur || !depth || !ok) return fail(ctx, SVOB200_ERR_ARG, "depth_from_triangulation: bad arguments");
  if (n == 0) return SVOB200_OK;
  Stage st(ctx, SVOB200_MEM_HOST);
  const int i_T = st.add(T_search_ref, nullptr, sizeof(double) * 7 * n, 0);
  const int i_a = st.add(f_ref, nullptr, sizeof(double) * 3 * n, 0);
  const int i_b = st.add(f_cur, nullptr, sizeof(double) * 3 * n, 0);
  const int i_d = st.add(depth, depth, sizeof(double) * n, 1);
  const int i_o = st.add(nullptr, ok, sizeof(int) * n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_triangulate(n, st.dev<double>(i_T), st.dev<double>(i_a), st.dev<double>(i_b), st.dev<double>(i_d), st.dev<int>(i_o), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "depth_from_triangulation launch failed");
  return st.download();
}

// ------------------------------------------------------------------ camera input stage (SURVEY §8f-3)
int svob200_frame_upload_yuv420(svob200_ctx* ctx, int64_t frame_id, const uint8_t* y, int y_stride, const uint8_t* u, const uint8_t* v,
                                int uv_stride, int uv_pixel_stride, size_t y_image_stride, size_t uv_image_stride, const int* round_modes, int mem)
{
  if (!ctx || !y || !u || !v) return fail(ctx, SVOB200_ERR_ARG, "frame_upload_yuv420: null argument");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  const int w = r->f.w[0], h = r->f.h[0], B = r->f.batch;
  if (y_stride < w || uv_pixel_stride < 1 || uv_pixel_stride > 2) return fail(ctx, SVOB200_ERR_ARG, "frame_upload_yuv420: bad strides");
  const int cw = (w + 1) / 2, ch = (h + 1) / 2;
  const int uv_row_bytes = (cw - 1) * uv_pixel_stride + 1;
  if (uv_stride < uv_row_bytes) return fail(ctx, SVOB200_ERR_ARG, "frame_upload_yuv420: uv_stride too small");
  if (int e = frame_own_level0(ctx, r, false)) return e;      // level 0 is produced here
  YuvPlanes P;
  if (mem == SVOB200_MEM_DEVICE) {
    P.y = y; P.u = u; P.v = v; P.y_stride = y_stride; P.uv_stride = uv_stride; P.uv_pixel_stride = uv_pixel_stride;
    P.y_img_stride = y_image_stride; P.uv_img_stride = uv_image_stride;
  } else {
    // stage the planes: Y with a 16-byte pitch; chroma either as ONE interleaved window (u, v are views of the same
    // buffer, pixel stride 2) or as two planes
    const bool inter = uv_pixel_stride == 2 && (u == v + 1 || v == u + 1);
    const size_t ypitch = (size_t)align_up_i(w, 16), cpitch = (size_t)align_up_i(inter ? 2 * cw : uv_row_bytes, 16);
    const size_t ybytes = ypitch * h * B, cbytes = cpitch * ch * B;
    const size_t total = ybytes + (inter ? cbytes : 2 * cbytes) + 64;
    if (ctx->d_stage.ensure(total) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "frame_upload_yuv420: staging alloc failed");
    uint8_t* dy = static_cast<uint8_t*>(ctx->d_stage.p);
    uint8_t* dc0 = dy + ybytes;
    uint8_t* dc1 = dc0 + cbytes;
    for (int b = 0; b < B; ++b) {
      CU(cudaMemcpy2DAsync(dy + (size_t)b * ypitch * h, ypitch, y + (size_t)b * y_image_stride, y_stride, w, h, cudaMemcpyHostToDevice, ctx->stream));
      if (inter) {
        const uint8_t* base = (u < v ? u : v) + (size_t)b * uv_image_stride;
        // the second plane's last sample sits one byte past 2*cw - 1 only when it is the +1 view: 2*cw bytes cover both
        CU(cudaMemcpy2DAsync(dc0 + (size_t)b * cpitch * ch, cpitch, base, uv_stride, std::min((size_t)2 * cw, (size_t)uv_stride), ch, cudaMemcpyHostToDevice, ctx->stream));
      } else {
        CU(cudaMemcpy2DAsync(dc0 + (size_t)b * cpitch * ch, cpitch, u + (size_t)b * uv_image_stride, uv_stride, uv_row_bytes, ch, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpy2DAsync(dc1 + (size_t)b * cpitch * ch, cpitch, v + (size_t)b * uv_image_stride, uv_stride, uv_row_bytes, ch, cudaMemcpyHostToDevice, ctx->stream));
      }
    }
    P.y = dy; P.y_stride = (int)ypitch; P.y_img_stride = ypitch * h;
    P.uv_stride = (int)cpitch; P.uv_pixel_stride = uv_pixel_stride; P.uv_img_stride = cpitch * ch;
    if (inter) { P.u = dc0 + (u > v ? 1 : 0); P.v = dc0 + (v > u ? 1 : 0); }
    else { P.u = dc0; P.v = dc1; }
  }
  int modes[SVOB200_MAX_LEVELS];
  pyramid_round_modes(r->f, round_modes, modes);
  if (launch_pyramid_yuv(r->f, P, modes, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "yuv pyramid launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (mem == SVOB200_MEM_HOST) CU(cudaStreamSynchronize(ctx->stream));
  return SVOB200_OK;
}

// ------------------------------------------------------------------ reprojector (SURVEY §8f-1)
int svob200_reproject_map(svob200_ctx* ctx, int64_t cur_frame_id, const svob200_camera* cam, int batch, const double* T_cur_w,
                          const int* point_offsets, int n_points, const svob200_map_point* points, int n_obs, const svob200_feature_ref* obs,
                          const double* T_obs_w, int cell_size, int max_fts, const svob200_matcher_opts* opts, svob200_reproj_result* results,
                          int* cell_winner, svob200_reproj_stats* stats, int mem)
{
  if (!ctx || !cam || batch <= 0 || !T_cur_w || !point_offsets || n_points < 0 || n_obs < 0 || !opts || !results || !cell_winner || !stats || cell_size <= 0)
    return fail(ctx, SVOB200_ERR_ARG, "reproject_map: bad arguments");
  if (n_points > 0 && (!points || !obs || !T_obs_w)) return fail(ctx, SVOB200_ERR_ARG, "reproject_map: null point / observation arrays");
  FrameRec* cur = find_frame(ctx, cur_frame_id);
  if (!cur) return fail(ctx, SVOB200_ERR_NOFRAME, "reproject_map: current frame not resident");
  if (batch != cur->f.batch) return fail(ctx, SVOB200_ERR_ARG, "reproject_map: batch differs from the frame's");
  if (opts->max_search_level >= cur->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "reproject_map: max_search_level outside the pyramid");
  if (opts->max_epi_search_steps < 0) return fail(ctx, SVOB200_ERR_ARG, "reproject_map: negative max_epi_search_steps");
  const int gc = (cam->width + cell_size - 1) / cell_size, gr = (cam->height + cell_size - 1) / cell_size;
  const size_t n_cells = (size_t)gc * gr;
  Stage st(ctx, mem);
  const int i_T = st.add(T_cur_w, nullptr, sizeof(double) * 7 * batch, 0);
  const int i_off = st.add(point_offsets, nullptr, sizeof(int) * (batch + 1), 0);
  const int i_p = st.add(points, nullptr, sizeof(svob200_map_point) * n_points, 0);
  const int i_o = st.add(obs, nullptr, sizeof(svob200_feature_ref) * n_obs, 0);
  const int i_To = st.add(T_obs_w, nullptr, sizeof(double) * 7 * n_obs, 0);
  const int i_r = st.add(nullptr, results, sizeof(svob200_reproj_result) * n_points, 2);
  const int i_w = st.add(nullptr, cell_winner, sizeof(int) * n_cells * batch, 2);
  const int i_s = st.add(nullptr, stats, sizeof(svob200_reproj_stats) * batch, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (mem == SVOB200_MEM_HOST && n_obs > 0) if (int e = resolve_slots(ctx, st.host<svob200_feature_ref>(i_o), n_obs)) return e;
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(match_scratch_bytes(n_points)) != cudaSuccess || ctx->d_scratch2.ensure(reproject_scratch_bytes(n_points)) != cudaSuccess)
    return fail(ctx, SVOB200_ERR_NOMEM, "reproject_map: scratch alloc failed");
  const int rc = launch_reproject_map(ctx->d_table, cur->slot, to_cam(cam), batch, st.dev<double>(i_T), st.dev<int>(i_off), n_points,
                                      st.dev<svob200_map_point>(i_p), st.dev<svob200_feature_ref>(i_o), st.dev<double>(i_To), cell_size, max_fts,
                                      *opts, st.dev<svob200_reproj_result>(i_r), st.dev<int>(i_w), st.dev<svob200_reproj_stats>(i_s),
                                      ctx->d_scratch2.p, ctx->d_scratch.p, nullptr, nullptr, nullptr, nullptr, nullptr, ctx->stream, &ctx->launches);
  if (rc == -2) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "reproject_map: grid of %zu cells exceeds the kernel's table (8192)", n_cells);
  if (rc) return fail(ctx, SVOB200_ERR_CUDA, "reproject_map launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ pose / structure optimisation (SURVEY §8f-2)
void svob200_pose_opt_opts_default(svob200_pose_opt_opts* o)
{
  o->reproj_thresh = 2.0;      // Config::poseOptimThresh (config.cpp)
  o->n_iter = 10;              // Config::poseOptimNumIter
  o->eps = 0.0000000001;       // svo::EPS global.h:91
  o->tukey_b = 8.6851f;        // TukeyWeightFunction::DEFAULT_B robust_cost.cpp:87
}

int svob200_pose_optimize(svob200_ctx* ctx, const svob200_camera* cam, int batch, const int* ftr_offsets, const double* f, const int* level,
                          const double* pos, const svob200_pose_opt_opts* opts, double* T_f_w, svob200_pose_opt_result* results,
                          uint8_t* outlier, int mem)
{
  if (!ctx || !cam || batch <= 0 || !ftr_offsets || !opts || !T_f_w || !results) return fail(ctx, SVOB200_ERR_ARG, "pose_optimize: bad arguments");
  int n = 0;
  if (mem == SVOB200_MEM_HOST) n = ftr_offsets[batch];
  else { CU(cudaMemcpyAsync(&n, ftr_offsets + batch, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); }
  if (n < 0 || (n > 0 && (!f || !level || !pos || !outlier))) return fail(ctx, SVOB200_ERR_ARG, "pose_optimize: null feature arrays");
  Stage st(ctx, mem);
  const int i_off = st.add(ftr_offsets, nullptr, sizeof(int) * (batch + 1), 0);
  const int i_f = st.add(f, nullptr, sizeof(double) * 3 * n, 0);
  const int i_l = st.add(level, nullptr, sizeof(int) * n, 0);
  const int i_p = st.add(pos, nullptr, sizeof(double) * 3 * n, 0);
  const int i_T = st.add(T_f_w, T_f_w, sizeof(double) * 7 * batch, 1);
  const int i_r = st.add(nullptr, results, sizeof(svob200_pose_opt_result) * batch, 2);
  const int i_o = st.add(nullptr, outlier, (size_t)n, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (ctx->d_scratch.ensure(sizeof(double) * (size_t)(n > 0 ? n : 1)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "pose_optimize: scratch alloc failed");
  const int* d_off = st.dev<int>(i_off);
  if (launch_pose_optimize(to_cam(cam), batch, d_off, d_off + 1, st.dev<double>(i_f), st.dev<int>(i_l), st.dev<double>(i_p), opts->reproj_thresh,
                           opts->n_iter, opts->eps, opts->tukey_b, st.dev<double>(i_T), st.dev<svob200_pose_opt_result>(i_r), st.dev<uint8_t>(i_o),
                           static_cast<double*>(ctx->d_scratch.p), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "pose_optimize launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

int svob200_points_optimize(svob200_ctx* ctx, int n, const int* obs_offsets, const double* T_f_w, const double* f, int n_iter, double eps,
                            double* pos, int* iters_out, int mem)
{
  if (!ctx || n < 0 || !obs_offsets || !pos) return fail(ctx, SVOB200_ERR_ARG, "points_optimize: bad arguments");
  if (n == 0) return SVOB200_OK;
  int m = 0;
  if (mem == SVOB200_MEM_HOST) m = obs_offsets[n];
  else { CU(cudaMemcpyAsync(&m, obs_offsets + n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); }
  if (m < 0 || (m > 0 && (!T_f_w || !f))) return fail(ctx, SVOB200_ERR_ARG, "points_optimize: null observation arrays");
  Stage st(ctx, mem);
  const int i_off = st.add(obs_offsets, nullptr, sizeof(int) * (n + 1), 0);
  const int i_T = st.add(T_f_w, nullptr, sizeof(double) * 7 * m, 0);
  const int i_f = st.add(f, nullptr, sizeof(double) * 3 * m, 0);
  const int i_p = st.add(pos, pos, sizeof(double) * 3 * n, 1);
  const int i_it = iters_out ? st.add(nullptr, iters_out, sizeof(int) * n, 2) : -1;
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  if (launch_points_optimize(n, st.dev<int>(i_off), st.dev<double>(i_T), st.dev<double>(i_f), n_iter, eps, st.dev<double>(i_p),
                             iters_out ? st.dev<int>(i_it) : nullptr, ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "points_optimize launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ seed initialisation (SURVEY §8f-4)
int svob200_seeds_initialize(svob200_ctx* ctx, int64_t frame_id, int n_detect_levels, int cell_size, double thr, const int* existing_offsets,
                             const double* existing_px, const float* depth_mean, const float* depth_min, svob200_corner* corners_out,
                             svob200_seed* seeds_out, int* counts, int mem)
{
  if (!ctx || cell_size <= 0 || !existing_offsets || !depth_mean || !depth_min || !corners_out || !seeds_out || !counts)
    return fail(ctx, SVOB200_ERR_ARG, "seeds_initialize: bad arguments");
  FrameRec* r = find_frame(ctx, frame_id);
  if (!r) return fail(ctx, SVOB200_ERR_NOFRAME, "frame %lld not found", (long long)frame_id);
  if (n_detect_levels < 1 || n_detect_levels > r->f.n_levels) return fail(ctx, SVOB200_ERR_ARG, "seeds_initialize: n_detect_levels out of range");
  if (r->f.w[0] >= 16384 || r->f.h[0] >= 16384) return fail(ctx, SVOB200_ERR_UNSUPPORTED, "seeds_initialize: image larger than 16383");
  const int B = r->f.batch;
  const int gc = (r->f.w[0] + cell_size - 1) / cell_size, gr = (r->f.h[0] + cell_size - 1) / cell_size;
  const size_t n_cells = (size_t)gc * gr, total = n_cells * B;
  int n = 0, max_per = 0;
  if (mem == SVOB200_MEM_HOST) { n = existing_offsets[B]; for (int b = 0; b < B; ++b) max_per = std::max(max_per, existing_offsets[b + 1] - existing_offsets[b]); }
  else { CU(cudaMemcpyAsync(&n, existing_offsets + B, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); max_per = n; }
  if (n < 0 || (n > 0 && !existing_px)) return fail(ctx, SVOB200_ERR_ARG, "seeds_initialize: null existing_px");
  Stage st(ctx, mem);
  const int i_off = st.add(existing_offsets, nullptr, sizeof(int) * (B + 1), 0);
  const int i_px = st.add(existing_px, nullptr, sizeof(double) * 2 * n, 0);
  const int i_dm = st.add(depth_mean, nullptr, sizeof(float) * B, 0);
  const int i_dn = st.add(depth_min, nullptr, sizeof(float) * B, 0);
  const int i_c = st.add(nullptr, corners_out, sizeof(svob200_corner) * total, 2);
  const int i_s = st.add(nullptr, seeds_out, sizeof(svob200_seed) * total, 2);
  const int i_n = st.add(nullptr, counts, sizeof(int) * B, 2);
  if (int e = st.layout()) return e;
  st.upload();
  if (int e = st.push()) return e;
  // scratch: cell keys (8 B) | cell records | occupancy | detector counts
  const size_t need = total * 8 + total * sizeof(svob200_corner) + ((total + 255) & ~(size_t)255) + sizeof(int) * B + 1024;
  if (ctx->d_scratch.ensure(need) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "seeds_initialize: scratch alloc failed");
  unsigned long long* d_keys = static_cast<unsigned long long*>(ctx->d_scratch.p);
  svob200_corner* d_cells = reinterpret_cast<svob200_corner*>(d_keys + total);
  uint8_t* d_occ = reinterpret_cast<uint8_t*>(d_cells + total);
  int* d_cnt = reinterpret_cast<int*>(d_occ + ((total + 255) & ~(size_t)255));
  CU(cudaMemsetAsync(d_occ, 0, total, ctx->stream));
  if (launch_occupancy(B, max_per, st.dev<int>(i_off), st.dev<double>(i_px), cell_size, gc, (int)n_cells, d_occ, ctx->stream, &ctx->launches) ||
      launch_fast_detect(r->f, n_detect_levels, cell_size, gc, gr, thr, d_occ, d_keys, d_cells, d_cnt, ctx->stream, &ctx->launches) ||
      launch_seeds_compact(B, d_cells, (int)n_cells, thr, st.dev<float>(i_dm), st.dev<float>(i_dn), st.dev<svob200_corner>(i_c),
                           st.dev<svob200_seed>(i_s), st.dev<int>(i_n), ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "seeds_initialize launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return st.download();
}

// ------------------------------------------------------------------ raw device helpers
int svob200_dev_alloc(svob200_ctx* ctx, size_t bytes, void** dptr)
{
  if (!ctx || !dptr) return SVOB200_ERR_ARG;
  if (cudaMalloc(dptr, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return fail(ctx, SVOB200_ERR_NOMEM, "dev_alloc(%zu) failed", bytes); }
  return SVOB200_OK;
}
int svob200_dev_free(svob200_ctx* ctx, void* dptr) { if (!ctx) return SVOB200_ERR_ARG; CU(cudaStreamSynchronize(ctx->stream)); CU(cudaFree(dptr)); return 0; }
int svob200_dev_upload(svob200_ctx* ctx, void* dptr, const void* host, size_t bytes)
{
  if (!ctx) return SVOB200_ERR_ARG;
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaMemcpyAsync(dptr, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int svob200_dev_download(svob200_ctx* ctx, void* host, const void* dptr, size_t bytes)
{
  if (!ctx) return SVOB200_ERR_ARG;
  if (int e = ctx_join_aux(ctx)) return e;
  CU(cudaMemcpyAsync(host, dptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int svob200_host_alloc_pinned(svob200_ctx* ctx, size_t bytes, void** hptr) { if (!ctx || !hptr) return SVOB200_ERR_ARG; CU(cudaMallocHost(hptr, bytes ? bytes : 1)); return 0; }
int svob200_host_free_pinned(svob200_ctx* ctx, void* hptr) { if (!ctx) return SVOB200_ERR_ARG; CU(cudaFreeHost(hptr)); return 0; }

int svob200_synth_render(svob200_ctx* ctx, const uint8_t* dev_texture, int tex_size, double ppm, double plane_z,
                         const svob200_camera* cam, int batch, const double* T_f_w, uint8_t* dev_out)
{
  if (!ctx || !dev_texture || !cam || !T_f_w || !dev_out || batch <= 0) return fail(ctx, SVOB200_ERR_ARG, "synth_render: bad arguments");
  // host: invert each pose into (R row-major, camera centre) — 12 doubles per image
  std::vector<double> rc((size_t)12 * batch);
  for (int b = 0; b < batch; ++b) {
    const double* T = T_f_w + 7 * (size_t)b;
    const double x = -T[3], y = -T[4], z = -T[5], w = T[6];     // inverse rotation
    double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                   2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                   2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)};
    for (int k = 0; k < 9; ++k) rc[12 * b + k] = R[k];
    for (int i = 0; i < 3; ++i) rc[12 * b + 9 + i] = -(R[3 * i] * T[0] + R[3 * i + 1] * T[1] + R[3 * i + 2] * T[2]);
  }
  if (ctx->d_scratch2.ensure(rc.size() * sizeof(double)) != cudaSuccess) return fail(ctx, SVOB200_ERR_NOMEM, "synth_render: scratch alloc failed");
  CU(cudaMemcpyAsync(ctx->d_scratch2.p, rc.data(), rc.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (launch_synth_render(dev_texture, tex_size, ppm, plane_z, to_cam(cam), batch, static_cast<const double*>(ctx->d_scratch2.p), dev_out,
                          ctx->stream, &ctx->launches))
    return fail(ctx, SVOB200_ERR_CUDA, "synth_render launch failed");
  return SVOB200_OK;
}

}  // extern "C"
