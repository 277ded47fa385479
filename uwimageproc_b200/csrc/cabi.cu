// cabi.cu - the C ABI declared in include/uwip.h: context, staging, and the reference-shaped entry
// points.  Host-pointer variants stage through the context workspace; `_dev` variants are stream
// ordered on device memory.  There is no CPU fallback anywhere in this file.
#include <stdarg.h>

#include <algorithm>
#include <mutex>

#include "common.cuh"
#include "e2e_schedule.h"

// Every entry point runs on the context's device and puts the caller's current device back when it returns (the library
// is used next to other CUDA code - torch, OpenCV - whose current device it must not change).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
static thread_local std::string g_create_err;

const char* uwip_set_err(uwip_ctx* ctx, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_err = buf;
  return ctx ? ctx->err.c_str() : g_create_err.c_str();
}

void* uwip_slot(uwip_ctx* ctx, int slot, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (ctx->slot_bytes[slot] >= bytes) return ctx->slot_ptr[slot];
  if (ctx->slot_ptr[slot]) {
    cudaStreamSynchronize(ctx->stream);  // growing a buffer that may still be in use
    cudaFree(ctx->slot_ptr[slot]);
    ctx->slot_ptr[slot] = nullptr;
    ctx->slot_bytes[slot] = 0;
  }
  size_t want = align_up(bytes, 1 << 20);
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    uwip_set_err(ctx, "cudaMalloc(%zu bytes) for workspace slot %d failed: %s", want, slot, cudaGetErrorString(e));
    cudaGetLastError();
    return nullptr;
  }
  ctx->slot_ptr[slot] = p;
  ctx->slot_bytes[slot] = want;
  return p;
}

void uwip_pre_launch(uwip_ctx* ctx, const char* tag) {
  if (!ctx->profiling) return;
  ProfRec r;
  r.tag = tag;
  cudaEventCreate(&r.e0);
  cudaEventCreate(&r.e1);
  cudaEventRecord(r.e0, ctx->stream);
  ctx->prof.push_back(r);
}
int uwip_post_launch(uwip_ctx* ctx, const char* tag) {
  ctx->launches++;
  if (ctx->profiling) cudaEventRecord(ctx->prof.back().e1, ctx->stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    uwip_set_err(ctx, "launch of %s failed: %s", tag, cudaGetErrorString(e));
    return UWIP_ERR_CUDA;
  }
  return UWIP_OK;
}

extern "C" {

int uwip_version(void) { return UWIP_VERSION; }

int uwip_create(int device, uwip_ctx** out) {
  if (!out) return UWIP_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    uwip_set_err(nullptr, "no CUDA device (%s); libuwip has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count 0");
    cudaGetLastError();
    return UWIP_ERR_CUDA;
  }
  if (device < 0 || device >= n) {
    uwip_set_err(nullptr, "device %d out of range (0..%d)", device, n - 1);
    return UWIP_ERR_INVALID;
  }
  cudaDeviceProp prop;
  DeviceGuard guard(device);   // the caller's current device is put back when uwip_create returns
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    uwip_set_err(nullptr, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    return UWIP_ERR_CUDA;
  }
  if (prop.major != 10) {
    uwip_set_err(nullptr, "device %d is sm_%d%d; libuwip is built for sm_100a only", device, prop.major, prop.minor);
    return UWIP_ERR_CUDA;
  }
  uwip_ctx* ctx = new uwip_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    uwip_set_err(nullptr, "cudaStreamCreate: %s", cudaGetErrorString(e));
    delete ctx;
    return UWIP_ERR_CUDA;
  }
  ctx->own_stream = true;
  if ((e = cudaMallocHost(&ctx->pinned, 1 << 16)) != cudaSuccess) {
    uwip_set_err(nullptr, "cudaMallocHost: %s", cudaGetErrorString(e));
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return UWIP_ERR_CUDA;
  }
  ctx->pinned_bytes = 1 << 16;
  *out = ctx;
  return UWIP_OK;
}

void uwip_destroy(uwip_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard guard(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& r : ctx->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  for (int i = 0; i < uwip_ctx::kSlots; i++)
    if (ctx->slot_ptr[i]) cudaFree(ctx->slot_ptr[i]);
  jpeg_io_destroy(ctx);
  jpeg_dec_destroy(ctx);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
  if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* uwip_last_error(const uwip_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int uwip_set_stream(uwip_ctx* ctx, void* s) {
  if (!ctx) return UWIP_ERR_INVALID;
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  ctx->own_stream = false;
  ctx->stream = (cudaStream_t)s;
  return UWIP_OK;
}
int uwip_synchronize(uwip_ctx* ctx) {
  if (!ctx) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}
int64_t uwip_launch_count(const uwip_ctx* ctx) { return ctx ? ctx->launches : 0; }

int uwip_profile(uwip_ctx* ctx, int enable) {
  if (!ctx) return UWIP_ERR_INVALID;
  cudaStreamSynchronize(ctx->stream);
  for (auto& r : ctx->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  ctx->prof.clear();
  ctx->profiling = enable != 0;
  return UWIP_OK;
}
int uwip_profile_read(uwip_ctx* ctx, const char* tag, double* total_ms, int64_t* launches) {
  if (!ctx || !tag) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  double tot = 0;
  int64_t n = 0;
  for (auto& r : ctx->prof) {
    if (!strstr(r.tag, tag)) continue;
    float ms = 0;
    UWIP_CUDA(ctx, cudaEventElapsedTime(&ms, r.e0, r.e1));
    tot += ms;
    n++;
  }
  if (total_ms) *total_ms = tot;
  if (launches) *launches = n;
  return UWIP_OK;
}

int uwip_device_alloc(uwip_ctx* ctx, size_t bytes, void** dptr) {
  if (!ctx || !dptr) return UWIP_ERR_INVALID;
  cudaError_t e = cudaMalloc(dptr, bytes ? bytes : 16);
  if (e != cudaSuccess) { uwip_set_err(ctx, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return UWIP_ERR_NOMEM; }
  return UWIP_OK;
}
int uwip_device_free(uwip_ctx* ctx, void* dptr) {
  if (!ctx) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  UWIP_CUDA(ctx, cudaFree(dptr));
  return UWIP_OK;
}
int uwip_host_alloc(uwip_ctx* ctx, size_t bytes, void** hptr) {
  if (!ctx || !hptr) return UWIP_ERR_INVALID;
  cudaError_t e = cudaMallocHost(hptr, bytes ? bytes : 16);
  if (e != cudaSuccess) { uwip_set_err(ctx, "cudaMallocHost(%zu): %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return UWIP_ERR_NOMEM; }
  return UWIP_OK;
}
int uwip_host_free(uwip_ctx* ctx, void* hptr) {
  if (!ctx) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaFreeHost(hptr));
  return UWIP_OK;
}
int uwip_copy_h2d(uwip_ctx* ctx, void* d, const void* h, size_t bytes) {
  if (!ctx) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return UWIP_OK;
}
int uwip_copy_d2h(uwip_ctx* ctx, void* h, const void* d, size_t bytes) {
  if (!ctx) return UWIP_ERR_INVALID;
  UWIP_CUDA(ctx, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return UWIP_OK;
}

// ---- preprocessing.cpp ---------------------------------------------------------------------------
int uwip_num_channel(char c) {
  if (c == 'R' || c == 'H' || c == 'h' || c == 'L' || c == 'Y') return 0;
  if (c == 'G' || c == 'S' || c == 's' || c == 'a' || c == 'C') return 1;
  if (c == 'B' || c == 'V' || c == 'l' || c == 'b' || c == 'X') return 2;
  return -1;
}
int uwip_num_space(char c) {
  if (c == 'R' || c == 'G' || c == 'B') return 0;
  if (c == 'H' || c == 'S' || c == 'V') return 1;
  if (c == 'h' || c == 's' || c == 'l') return 2;
  if (c == 'L' || c == 'a' || c == 'b') return 3;
  if (c == 'Y' || c == 'C' || c == 'X') return 4;
  return -1;
}

}  // extern "C"

// ---- staging helpers -----------------------------------------------------------------------------
static int stage_in(uwip_ctx* ctx, int slot, const uint8_t* src, size_t pitch, int w, int h, int ch, uint8_t** d) {
  size_t row = (size_t)w * ch;
  if (!src || w < 1 || h < 1 || pitch < row) { uwip_set_err(ctx, "bad image argument (w=%d h=%d pitch=%zu)", w, h, pitch); return UWIP_ERR_INVALID; }
  *d = (uint8_t*)uwip_slot(ctx, slot, row * h);
  if (!*d) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemcpy2DAsync(*d, row, src, pitch, row, h, cudaMemcpyHostToDevice, ctx->stream));
  return UWIP_OK;
}
static int stage_out(uwip_ctx* ctx, const uint8_t* d, uint8_t* dst, size_t pitch, int w, int h, int ch) {
  size_t row = (size_t)w * ch;
  if (!dst || pitch < row) { uwip_set_err(ctx, "bad output argument"); return UWIP_ERR_INVALID; }
  UWIP_CUDA(ctx, cudaMemcpy2DAsync(dst, pitch, d, row, row, h, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}
#define CTX_GUARD(ctx)                          \
  if (!(ctx)) return UWIP_ERR_INVALID;          \
  DeviceGuard uwip_device_guard__((ctx)->device)

static int check_percentiles(uwip_ctx* ctx, int lo, int hi) {
  if (!(0 <= lo && lo < hi && hi <= 100)) {
    uwip_set_err(ctx, "percentiles must satisfy 0 <= lo < hi <= 100 (preprocessing.h:60-64), got %d %d", lo, hi);
    return UWIP_ERR_INVALID;
  }
  return UWIP_OK;
}

static int32_t* flags_get(uwip_ctx* ctx, int n) {
  int32_t* f = (int32_t*)uwip_slot(ctx, SLOT_FLAGS, sizeof(int32_t) * (size_t)n);
  ctx->flags_n = f ? n : 0;
  return f;
}

// sub-batch size: the dehaze workspace is 60 B/px/frame (+ a 256 KB table; budgeted as 512 KB); keep it below 80 GB of the 180 GB
// (UWIP_WORKSPACE_GB overrides) and below 70 % of what the device has free plus what this context already holds, and among
// the sizes that fit take the one that wastes the fewest CTA waves of the marches (dehaze_sub_batch)
static int sub_batch(const uwip_ctx* ctx, int n, int w, int h) {
  size_t per_frame = (size_t)w * h * 60 + (512u << 10);
  double gb = 80.0;
  if (const char* e = getenv("UWIP_WORKSPACE_GB")) { double v = atof(e); if (v >= 1.0) gb = v; }
  size_t cap_bytes = (size_t)(gb * 1e9);
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
    size_t held = 0;
    for (int i = 0; i < uwip_ctx::kSlots; i++) held += ctx->slot_bytes[i];
    cap_bytes = std::min(cap_bytes, (size_t)(0.7 * (double)(free_b + held)));
  } else {
    cudaGetLastError();
  }
  size_t cap = std::max<size_t>(1, cap_bytes / per_frame);
  return dehaze_sub_batch(ctx, n, w, (int)std::min<size_t>(cap, (size_t)n));
}

// n device frames in sub-batches of sub_batch's size: fn(first, m, fs, flags + first) for each, stopping at the first error.
// One FrameState block of the largest sub-batch serves them all; the flags of the call are indexed by frame.
template <class Fn>
static int each_sub_batch(uwip_ctx* ctx, int n, int w, int h, Fn&& fn) {
  int nb = sub_batch(ctx, n, w, h);
  FrameState* fs = frame_state_get(ctx, nb);
  int32_t* flags = flags_get(ctx, n);
  if (!fs || !flags) return UWIP_ERR_NOMEM;
  for (int i = 0; i < n; i += nb) UWIP_CHECK(fn(i, std::min(nb, n - i), fs, flags + i));
  return UWIP_OK;
}

extern "C" {

int uwip_histogram_u8_dev(uwip_ctx* ctx, const uint8_t* d_plane, int w, int h, float* d_hist) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_plane && d_hist && w > 0 && h > 0, "bad argument");
  uint32_t* dh = (uint32_t*)uwip_slot(ctx, SLOT_HIST, 256 * 4);
  if (!dh) return UWIP_ERR_NOMEM;
  UWIP_CHECK(k_histogram_plane(ctx, d_plane, 1, (size_t)w * h, dh));
  return k_hist_to_float(ctx, dh, d_hist, 256);
}

int uwip_histogram_u8(uwip_ctx* ctx, const uint8_t* plane, int w, int h, size_t pitch, float hist[256]) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, hist, "null hist");
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, plane, pitch, w, h, 1, &d));
  float* dh = (float*)uwip_slot(ctx, SLOT_MISC, 256 * 4);
  if (!dh) return UWIP_ERR_NOMEM;
  UWIP_CHECK(uwip_histogram_u8_dev(ctx, d, w, h, dh));
  UWIP_CUDA(ctx, cudaMemcpyAsync(hist, dh, 256 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}

int uwip_channel_stretch_u8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int w, int h, int lo, int hi) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && w > 0 && h > 0, "bad argument");
  UWIP_CHECK(check_percentiles(ctx, lo, hi));
  uint32_t* dh = (uint32_t*)uwip_slot(ctx, SLOT_HIST, 256 * 4);
  uint8_t* dl = (uint8_t*)uwip_slot(ctx, SLOT_LUT, 1024);
  FrameState* fs = frame_state_get(ctx, 1);
  if (!dh || !dl || !fs) return UWIP_ERR_NOMEM;
  UWIP_CHECK(k_histogram_plane(ctx, d_src, 1, (size_t)w * h, dh));
  UWIP_CHECK(k_percentile_lut(ctx, dh, 1, w, h, lo, hi, fs, dl));
  return k_apply_lut_plane(ctx, d_src, d_dst, 1, (size_t)w * h, dl);
}

// pitched device planes (cv::cuda::GpuMat allocates with cudaMallocPitch: a 1920-wide plane has step 2048): the rows are
// gathered into the contiguous workspace, stretched there and scattered back, all on the context's stream
int uwip_channel_stretch_u8_dev_pitched(uwip_ctx* ctx, const uint8_t* d_src, size_t src_pitch, uint8_t* d_dst, size_t dst_pitch, int w, int h,
                                        int lo, int hi) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && w > 0 && h > 0 && src_pitch >= (size_t)w && dst_pitch >= (size_t)w, "bad argument");
  if (src_pitch == (size_t)w && dst_pitch == (size_t)w) return uwip_channel_stretch_u8_dev(ctx, d_src, d_dst, w, h, lo, hi);
  uint8_t* tmp = (uint8_t*)uwip_slot(ctx, SLOT_STAGE_IN, (size_t)w * h);
  if (!tmp) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemcpy2DAsync(tmp, (size_t)w, d_src, src_pitch, (size_t)w, (size_t)h, cudaMemcpyDeviceToDevice, ctx->stream));
  UWIP_CHECK(uwip_channel_stretch_u8_dev(ctx, tmp, tmp, w, h, lo, hi));
  UWIP_CUDA(ctx, cudaMemcpy2DAsync(d_dst, dst_pitch, tmp, (size_t)w, (size_t)w, (size_t)h, cudaMemcpyDeviceToDevice, ctx->stream));
  return UWIP_OK;
}

int uwip_channel_stretch_u8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst, size_t dp, int w, int h, int lo, int hi,
                            int* low_bin, int* high_bin) {
  CTX_GUARD(ctx);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, sp, w, h, 1, &d));
  UWIP_CHECK(uwip_channel_stretch_u8_dev(ctx, d, d, w, h, lo, hi));
  if (low_bin || high_bin) {
    FrameState* hs = (FrameState*)ctx->pinned;
    UWIP_CUDA(ctx, cudaMemcpyAsync(hs, frame_state_get(ctx, 1), sizeof(FrameState), cudaMemcpyDeviceToHost, ctx->stream));
    UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (low_bin) *low_bin = hs->low;
    if (high_bin) *high_bin = hs->high;
  }
  return stage_out(ctx, d, dst, dp, w, h, 1);
}

// ---- histretch CLI loop ----------------------------------------------------------------------------
int uwip_histretch_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const char* channels, int lo,
                            int hi, int order, int hsv_round) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && channels && n > 0 && w > 0 && h > 0, "bad argument");
  UWIP_REQUIRE(ctx, order == 0 || order == 1, "order must be 0 (intended) or 1 (literal)");
  UWIP_REQUIRE(ctx, hsv_round >= 0 && hsv_round <= 2, "bad hsv_round");
  UWIP_CHECK(check_percentiles(ctx, lo, hi));
  return histretch_frames_dev(ctx, d_src, d_dst, n, w, h, channels, lo, hi, order, hsv_round);
}
int uwip_histretch_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst, size_t dp, int w, int h, const char* channels,
                        int lo, int hi, int order, int hsv_round) {
  CTX_GUARD(ctx);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, sp, w, h, 3, &d));
  UWIP_CHECK(uwip_histretch_bgr8_dev(ctx, d, d, 1, w, h, channels, lo, hi, order, hsv_round));
  return stage_out(ctx, d, dst, dp, w, h, 3);
}

// ---- aclahe ------------------------------------------------------------------------------------------
int uwip_clahe_u8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst, "null pointer");
  return clahe_planes_dev(ctx, d_src, d_dst, n, w, h, clip, tx, ty);
}
int uwip_clahe_u8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst, size_t dp, int w, int h, double clip, int tx, int ty) {
  CTX_GUARD(ctx);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, sp, w, h, 1, &d));
  uint8_t* o = (uint8_t*)uwip_slot(ctx, SLOT_STAGE_OUT, (size_t)w * h);
  if (!o) return UWIP_ERR_NOMEM;
  UWIP_CHECK(clahe_planes_dev(ctx, d, o, 1, w, h, clip, tx, ty));
  return stage_out(ctx, o, dst, dp, w, h, 1);
}
int uwip_entropy_u8(uwip_ctx* ctx, const uint8_t* plane, int w, int h, size_t pitch, int flavour, float* entropy) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, entropy && (flavour == 0 || flavour == 1), "bad argument");
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, plane, pitch, w, h, 1, &d));
  uint32_t* dh = (uint32_t*)uwip_slot(ctx, SLOT_HIST, 256 * 4);
  float* de = (float*)uwip_slot(ctx, SLOT_MISC, 256);
  if (!dh || !de) return UWIP_ERR_NOMEM;
  UWIP_CHECK(k_histogram_plane(ctx, d, 1, (size_t)w * h, dh));
  UWIP_CHECK(k_entropy(ctx, dh, 1, w, h, flavour, de));
  UWIP_CUDA(ctx, cudaMemcpyAsync(entropy, de, 4, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}
int uwip_gaussian_blur3_u8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst, size_t dp, int w, int h) {
  CTX_GUARD(ctx);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, sp, w, h, 1, &d));
  uint8_t* o = (uint8_t*)uwip_slot(ctx, SLOT_STAGE_OUT, (size_t)w * h);
  if (!o) return UWIP_ERR_NOMEM;
  UWIP_CHECK(k_blur3(ctx, d, o, w, h));
  return stage_out(ctx, o, dst, dp, w, h, 1);
}
int uwip_clahe_entropy_sweep_u8(uwip_ctx* ctx, const uint8_t* plane, int w, int h, size_t pitch, int tiles, const double* clips,
                                int n_clips, int flavour, float* entropies) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, clips && entropies && (flavour == 0 || flavour == 1), "bad argument");
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, plane, pitch, w, h, 1, &d));
  return clahe_entropy_sweep_dev(ctx, d, w, h, tiles, clips, n_clips, flavour, entropies);
}
int uwip_clahe_entropy_sweep_u8_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, const int* grids, int n_grids,
                                    const double* clips, int n_clips, int flavour, float* entropies) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_planes && grids && clips && entropies && (flavour == 0 || flavour == 1), "bad argument");
  return clahe_entropy_sweep_batch_dev(ctx, d_planes, n, w, h, grids, n_grids, clips, n_clips, flavour, entropies);
}
int uwip_aclahe_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty,
                         int hsv_round) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && hsv_round >= 0 && hsv_round <= 2, "bad argument");
  return aclahe_frames_dev(ctx, d_src, d_dst, n, w, h, clip, tx, ty, hsv_round, nullptr, nullptr);
}
int uwip_aclahe_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst, size_t dp, int w, int h, double clip, int tx, int ty,
                     int hsv_round) {
  CTX_GUARD(ctx);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, sp, w, h, 3, &d));
  UWIP_CHECK(uwip_aclahe_bgr8_dev(ctx, d, d, 1, w, h, clip, tx, ty, hsv_round));
  return stage_out(ctx, d, dst, dp, w, h, 3);
}

// BS / CL outputs of the automatic calls: the caller's device arrays or the context's
static int auto_outputs(uwip_ctx* ctx, int n, int32_t*& d_bs, int32_t*& d_cl) {
  if (d_bs && d_cl) return UWIP_OK;
  int32_t* ws = (int32_t*)uwip_slot(ctx, SLOT_AUTO_BSCL, sizeof(int32_t) * 2 * (size_t)n);
  if (!ws) return UWIP_ERR_NOMEM;
  if (!d_bs) d_bs = ws;
  if (!d_cl) d_cl = ws + n;
  return UWIP_OK;
}

int uwip_aclahe_params_u8_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, int loop, int32_t* d_bs, int32_t* d_cl) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_planes && d_bs && d_cl && n > 0 && w > 0 && h > 0, "bad argument");
  int32_t* flags = flags_get(ctx, n);
  if (!flags) return UWIP_ERR_NOMEM;
  UWIP_CHECK(aclahe_params_planes_dev(ctx, d_planes, n, w, h, loop, d_bs, d_cl));
  return aclahe_nofit_flags(ctx, d_cl, n, flags, false);
}
int uwip_aclahe_bgr8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, int hsv_round,
                              double clip, int tx, int ty, int32_t* d_bs, int32_t* d_cl) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && n > 0 && w > 0 && h > 0 && hsv_round >= 0 && hsv_round <= 2, "bad argument");
  UWIP_CHECK(auto_outputs(ctx, n, d_bs, d_cl));
  int32_t* flags = flags_get(ctx, n);
  if (!flags) return UWIP_ERR_NOMEM;
  UWIP_CHECK(aclahe_frames_auto_dev(ctx, d_src, d_dst, n, w, h, loop, clip, tx, ty, hsv_round, nullptr, nullptr, d_bs, d_cl));
  return aclahe_nofit_flags(ctx, d_cl, n, flags, false);
}
int uwip_aclahe_u8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, double clip, int tx, int ty,
                            int32_t* d_bs, int32_t* d_cl) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && n > 0 && w > 0 && h > 0, "bad argument");
  UWIP_CHECK(auto_outputs(ctx, n, d_bs, d_cl));
  int32_t* flags = flags_get(ctx, n);
  if (!flags) return UWIP_ERR_NOMEM;
  UWIP_CHECK(aclahe_planes_auto_dev(ctx, d_src, d_dst, n, w, h, loop, clip, tx, ty, d_bs, d_cl));
  return aclahe_nofit_flags(ctx, d_cl, n, flags, false);
}

// ---- videostrip calcBlur ------------------------------------------------------------------------------
int uwip_calc_blur_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, int n, int w, int h, int aperture, double* d_mean_std) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_mean_std && n >= 1 && w >= 1 && h >= 1 && (aperture == 1 || aperture == 3), "bad argument");
  return calc_blur_frames_dev(ctx, d_src, n, w, h, aperture, d_mean_std, nullptr);
}
int uwip_calc_blur_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, int aperture, float* stdev, double* mean_std,
                        uint8_t* lap, size_t lap_pitch) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, stdev || mean_std || lap, "no output requested");
  UWIP_REQUIRE(ctx, aperture == 1 || aperture == 3, "aperture must be 1 or 3");
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, pitch, w, h, 3, &d));
  double* d_out = (double*)uwip_slot(ctx, SLOT_BLUROUT, 16);
  uint8_t* d_lap = lap ? (uint8_t*)uwip_slot(ctx, SLOT_STAGE_OUT, (size_t)w * h) : nullptr;
  if (!d_out || (lap && !d_lap)) return UWIP_ERR_NOMEM;
  UWIP_CHECK(calc_blur_frames_dev(ctx, d, 1, w, h, aperture, d_out, d_lap));
  double ms[2];
  UWIP_CUDA(ctx, cudaMemcpyAsync(ms, d_out, 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (lap) UWIP_CHECK(stage_out(ctx, d_lap, lap, lap_pitch, w, h, 1));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (stdev) *stdev = (float)ms[1];  // `return stdev.val[0];` from a float function
  if (mean_std) { mean_std[0] = ms[0]; mean_std[1] = ms[1]; }
  return UWIP_OK;
}

// ---- bgdehaze -----------------------------------------------------------------------------------------
void uwip_dehaze_defaults(uwip_dehaze_params* p) {
  if (!p) return;
  p->window = 15; p->radius = 40; p->eps = 1e-3; p->tmin = 0.2;
}
void uwip_chain_defaults(uwip_chain_params* p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  strcpy(p->channels, "V");
  p->lo = 1; p->hi = 99; p->order = UWIP_ORDER_INTENDED; p->hsv_round = UWIP_HSV_ROUND_CV2_4_13;
  p->clip = 2.0; p->tiles_x = 8; p->tiles_y = 8;
  uwip_dehaze_defaults(&p->dehaze);
}

static int dehaze_host(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, const uwip_dehaze_params* pp, int stop_after,
                       uint8_t* dst8, size_t dst_pitch, double B[3], int64_t idx[2], double* t_raw, double* t_ref, double* restored,
                       double* out) {
  uwip_dehaze_params p;
  if (pp) p = *pp; else uwip_dehaze_defaults(&p);
  uint8_t* d;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, src, pitch, w, h, 3, &d));
  size_t n_px = (size_t)w * h;
  uint8_t* o = (uint8_t*)uwip_slot(ctx, SLOT_STAGE_OUT, n_px * 3);
  double* f64 = (double*)uwip_slot(ctx, SLOT_F64OUT, n_px * 8 * 8);  // t_raw[2] t_ref[2] (restored|out)[3] + slack
  FrameState* fs = frame_state_get(ctx, 1);
  if (!o || !f64 || !fs) return UWIP_ERR_NOMEM;
  DehazeDebug dbg;
  dbg.t_raw = t_raw ? f64 : nullptr;
  dbg.t_ref = t_ref ? f64 + 2 * n_px : nullptr;
  dbg.restored = restored ? f64 + 4 * n_px : nullptr;
  dbg.out = out ? f64 + 4 * n_px : nullptr;
  dbg.stop_after = stop_after;
  UWIP_CHECK(frame_state_reset(ctx, fs, 1));
  UWIP_CHECK(dehaze_frames_dev(ctx, d, o, 1, w, h, p, false, fs, &dbg));
  FrameState* hs = (FrameState*)ctx->pinned;
  UWIP_CUDA(ctx, cudaMemcpyAsync(hs, fs, sizeof(FrameState), cudaMemcpyDeviceToHost, ctx->stream));
  if (t_raw) UWIP_CUDA(ctx, cudaMemcpyAsync(t_raw, dbg.t_raw, 2 * n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (t_ref) UWIP_CUDA(ctx, cudaMemcpyAsync(t_ref, dbg.t_ref, 2 * n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (restored) UWIP_CUDA(ctx, cudaMemcpyAsync(restored, dbg.restored, 3 * n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (out) UWIP_CUDA(ctx, cudaMemcpyAsync(out, dbg.out, 3 * n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (B) { B[0] = hs->B[0]; B[1] = hs->B[1]; B[2] = hs->B[2]; }
  if (idx) { idx[0] = hs->idx0; idx[1] = hs->idx1; }
  if (dst8) return stage_out(ctx, o, dst8, dst_pitch, w, h, 3);
  return UWIP_OK;
}

int uwip_background_light_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, int window, double B[3], int64_t idx[2]) {
  CTX_GUARD(ctx);
  uwip_dehaze_params p;
  uwip_dehaze_defaults(&p);
  p.window = window;
  return dehaze_host(ctx, src, pitch, w, h, &p, 1, nullptr, 0, B, idx, nullptr, nullptr, nullptr, nullptr);
}
int uwip_transmission_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, int window, double* t_blue, double* t_green) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, t_blue && t_green, "null output");
  UWIP_REQUIRE(ctx, window == 15, "transmission window other than 15 is not reachable in the reference chain (BGDehaze.py:52)");
  uwip_dehaze_params p;
  uwip_dehaze_defaults(&p);
  size_t n_px = (size_t)w * h;
  std::vector<double> tmp(2 * n_px);
  UWIP_CHECK(dehaze_host(ctx, src, pitch, w, h, &p, 2, nullptr, 0, nullptr, nullptr, tmp.data(), nullptr, nullptr, nullptr));
  memcpy(t_blue, tmp.data(), n_px * 8);
  memcpy(t_green, tmp.data() + n_px, n_px * 8);
  return UWIP_OK;
}
int uwip_refined_transmission_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, const uwip_dehaze_params* p,
                                   double* t_blue, double* t_green) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, t_blue && t_green, "null output");
  size_t n_px = (size_t)w * h;
  std::vector<double> tmp(2 * n_px);
  UWIP_CHECK(dehaze_host(ctx, src, pitch, w, h, p, 3, nullptr, 0, nullptr, nullptr, nullptr, tmp.data(), nullptr, nullptr));
  memcpy(t_blue, tmp.data(), n_px * 8);
  memcpy(t_green, tmp.data() + n_px, n_px * 8);
  return UWIP_OK;
}
int uwip_rc_correction_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t pitch, int w, int h, const uwip_dehaze_params* p, double* restored) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, restored, "null output");
  return dehaze_host(ctx, src, pitch, w, h, p, 4, nullptr, 0, nullptr, nullptr, nullptr, nullptr, restored, nullptr);
}
int uwip_bgdehaze_bgr8(uwip_ctx* ctx, const uint8_t* src, size_t sp, uint8_t* dst8, size_t dp, int w, int h, const uwip_dehaze_params* p,
                       double* out_f64) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, dst8, "null output");
  return dehaze_host(ctx, src, sp, w, h, p, 0, dst8, dp, nullptr, nullptr, nullptr, nullptr, nullptr, out_f64);
}

int uwip_boxfilter_f64(uwip_ctx* ctx, const double* src, int w, int h, int r, double* dst) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, src && dst && w >= 1 && h >= 1 && r >= 0, "bad argument");
  const size_t n_px = (size_t)w * h;
  double* d = (double*)uwip_slot(ctx, SLOT_F64OUT, n_px * 8 * 3);
  if (!d) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemcpyAsync(d, src, n_px * 8, cudaMemcpyHostToDevice, ctx->stream));
  UWIP_CHECK(boxfilter_f64_dev(ctx, d, d + n_px, d + 2 * n_px, w, h, r));
  UWIP_CUDA(ctx, cudaMemcpyAsync(dst, d + 2 * n_px, n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}
int uwip_guided_filter_u8(uwip_ctx* ctx, const uint8_t* guide, size_t pitch, int w, int h, int range, const double* p, int r, double eps,
                          double* q) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, guide && p && q, "null argument");
  uint8_t* d_g;
  UWIP_CHECK(stage_in(ctx, SLOT_STAGE_IN, guide, pitch, w, h, 3, &d_g));
  const size_t n_px = (size_t)w * h;
  double* d = (double*)uwip_slot(ctx, SLOT_F64OUT, n_px * 8 * 2);
  FrameState* fs = frame_state_get(ctx, 1);
  if (!d || !fs) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemcpyAsync(d, p, n_px * 8, cudaMemcpyHostToDevice, ctx->stream));
  UWIP_CHECK(guided_filter_u8_dev(ctx, d_g, d, d + n_px, w, h, range, r, eps, fs));
  FrameState* hs = (FrameState*)ctx->pinned;
  UWIP_CUDA(ctx, cudaMemcpyAsync(hs, fs, sizeof(FrameState), cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaMemcpyAsync(q, d + n_px, n_px * 8, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (hs->nan_flag & 2u) {
    uwip_set_err(ctx, "uwip_guided_filter_u8: p must lie in [0, 1.6] (the signals of the path do: transmission <= 1, exposure ratio <= 1.54)");
    return UWIP_ERR_INVALID;
  }
  return UWIP_OK;
}

int uwip_bgdehaze_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const uwip_dehaze_params* pp) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst && n > 0, "bad argument");
  uwip_dehaze_params p;
  if (pp) p = *pp; else uwip_dehaze_defaults(&p);
  const size_t fbytes = (size_t)w * h * 3;
  return each_sub_batch(ctx, n, w, h, [&](int i, int m, FrameState* fs, int32_t* flags) {
    UWIP_CHECK(frame_state_reset(ctx, fs, m));
    return dehaze_frames_dev(ctx, d_src + (size_t)i * fbytes, d_dst + (size_t)i * fbytes, m, w, h, p, false, fs, nullptr, flags);
  });
}

// ---- the chain ------------------------------------------------------------------------------------------
// automatic CLAHE parameters of a chain call (uwip_chain_bgr8_auto_dev): per-frame outputs of the frames it covers
struct ChainAuto {
  int loop;
  int32_t* d_bs;
  int32_t* d_cl;
};

static int chain_aclahe(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int m, int w, int h, const uwip_chain_params& p,
                        const uint8_t* d_prelut, FrameState* fs, const ChainAuto* au) {
  if (au)
    return aclahe_frames_auto_dev(ctx, d_src, d_dst, m, w, h, au->loop, p.clip, p.tiles_x, p.tiles_y, p.hsv_round, d_prelut, fs, au->d_bs,
                                  au->d_cl);
  return aclahe_frames_dev(ctx, d_src, d_dst, m, w, h, p.clip, p.tiles_x, p.tiles_y, p.hsv_round, d_prelut, fs);
}

static int chain_sub(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int m, int w, int h, const uwip_chain_params& p, FrameState* fs, int32_t* flags,
                     const ChainAuto* au = nullptr) {
  size_t fbytes = (size_t)w * h * 3;
  uint8_t* tmp = (uint8_t*)uwip_slot(ctx, SLOT_TMP_FRAME, fbytes * m);
  if (!tmp) return UWIP_ERR_NOMEM;
  UWIP_CHECK(frame_state_reset(ctx, fs, m));
  bool fused_head = (strcmp(p.channels, "V") == 0 && p.order == UWIP_ORDER_INTENDED);
  if (fused_head) {
    // P1: V histogram -> percentile LUT.  P2/P3 (inside aclahe_frames_dev): tile histograms of the
    // stretched, round-tripped V; CLAHE LUTs; one read+write pass doing stretch, both colour round
    // trips, CLAHE and the dehaze min/max.
    uint32_t* d_hist = (uint32_t*)uwip_slot(ctx, SLOT_HIST, (size_t)m * 256 * 4);
    uint8_t* d_lut = (uint8_t*)uwip_slot(ctx, SLOT_LUT, (size_t)m * 256 * 4);
    if (!d_hist || !d_lut) return UWIP_ERR_NOMEM;
    UWIP_CHECK(k_histogram_frame(ctx, d_src, m, w, h, CH_V, d_hist));
    UWIP_CHECK(k_percentile_lut(ctx, d_hist, m, w, h, p.lo, p.hi, fs, d_lut));
    UWIP_CHECK(chain_aclahe(ctx, d_src, tmp, m, w, h, p, d_lut, fs, au));
  } else {
    UWIP_CHECK(histretch_frames_dev(ctx, d_src, tmp, m, w, h, p.channels, p.lo, p.hi, p.order, p.hsv_round));
    UWIP_CHECK(chain_aclahe(ctx, tmp, tmp, m, w, h, p, nullptr, fs, au));
  }
  UWIP_CHECK(dehaze_frames_dev(ctx, tmp, d_dst, m, w, h, p.dehaze, true, fs, nullptr, flags));
  return au ? aclahe_nofit_flags(ctx, au->d_cl, m, flags, true) : UWIP_OK;
}

// size every workspace slot a sub-batch of m frames touches (the slots only grow: a later, smaller sub-batch reuses them)
static int chain_reserve(uwip_ctx* ctx, int m, int w, int h, const uwip_chain_params& p) {
  const size_t fbytes = (size_t)w * h * 3, n_pp = (size_t)((w + 3) & ~3) * h;
  const size_t ntile = (size_t)m * std::max(1, p.tiles_x) * std::max(1, p.tiles_y);
  const struct { int slot; size_t bytes; } want[] = {
      {SLOT_TMP_FRAME, fbytes * m}, {SLOT_HIST, (size_t)m * 256 * 4}, {SLOT_LUT, (size_t)m * 256 * 4},
      {SLOT_TILEHIST, ntile * 256 * 4}, {SLOT_TILELUT, ntile * 256 + 16}, {SLOT_MISC, 256},
      {SLOT_KQ, m * n_pp * 4}, {SLOT_MPLANES, m * n_pp}, {SLOT_YCC, m * n_pp * 4}, {SLOT_STAB, (size_t)m * 65536 * 8},
      {SLOT_SPLANE, m * n_pp * 4}, {SLOT_AB, m * n_pp * 32}, {SLOT_J, m * n_pp * 8}, {SLOT_REFS, m * n_pp * 4}};
  for (const auto& e : want)
    if (!uwip_slot(ctx, e.slot, e.bytes)) return UWIP_ERR_NOMEM;
  return UWIP_OK;
}

static int chain_check(uwip_ctx* ctx, const uwip_chain_params* p, int n, int w, int h) {
  UWIP_REQUIRE(ctx, p, "null params (use uwip_chain_defaults)");
  UWIP_REQUIRE(ctx, n > 0 && w > 0 && h > 0, "bad size");
  UWIP_REQUIRE(ctx, memchr(p->channels, 0, sizeof(p->channels)) != nullptr, "channels not terminated");
  UWIP_REQUIRE(ctx, p->order == 0 || p->order == 1, "bad order");
  UWIP_REQUIRE(ctx, p->hsv_round >= 0 && p->hsv_round <= 2, "bad hsv_round");
  return check_percentiles(ctx, p->lo, p->hi);
}

// the device-buffer chain on checked arguments; au: the automatic CLAHE outputs of the n frames, null for the fixed parameters
static int chain_batch_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const uwip_chain_params& p,
                           const ChainAuto* au) {
  ChainAuto a = au ? *au : ChainAuto{0, nullptr, nullptr};
  // before sub_batch: the BS / CL slot auto_outputs may grow counts toward what the context already holds
  if (au) UWIP_CHECK(auto_outputs(ctx, n, a.d_bs, a.d_cl));
  const size_t fbytes = (size_t)w * h * 3;
  return each_sub_batch(ctx, n, w, h, [&](int i, int m, FrameState* fs, int32_t* flags) {
    ChainAuto sub = a;
    if (au) { sub.d_bs += i; sub.d_cl += i; }
    return chain_sub(ctx, d_src + (size_t)i * fbytes, d_dst + (size_t)i * fbytes, m, w, h, p, fs, flags, au ? &sub : nullptr);
  });
}

int uwip_chain_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const uwip_chain_params* p) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst, "null pointer");
  UWIP_CHECK(chain_check(ctx, p, n, w, h));
  return chain_batch_dev(ctx, d_src, d_dst, n, w, h, *p, nullptr);
}

int uwip_chain_bgr8_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const uwip_chain_params* p, int loop,
                             int32_t* d_bs, int32_t* d_cl) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && d_dst, "null pointer");
  UWIP_CHECK(chain_check(ctx, p, n, w, h));
  UWIP_REQUIRE(ctx, loop == UWIP_ACLAHE_LOOP_REPAIRED || loop == UWIP_ACLAHE_LOOP_AS_COMMITTED, "bad loop");
  UWIP_CHECK(aclahe_check_auto_size(ctx, w, h));
  const ChainAuto au = {loop, d_bs, d_cl};
  return chain_batch_dev(ctx, d_src, d_dst, n, w, h, *p, &au);
}

// host buffers: H2D / compute / D2H pipelined over sub-batches with two staging buffers per direction
int uwip_chain_bgr8(uwip_ctx* ctx, const uint8_t* src, uint8_t* dst, int n, int w, int h, const uwip_chain_params* p) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, src && dst, "null pointer");
  UWIP_CHECK(chain_check(ctx, p, n, w, h));
  int nb = sub_batch(ctx, n, w, h);
  nb = std::max(1, std::min(nb, (n + 1) / 2));  // at least two sub-batches so copies overlap compute
  std::vector<int> sizes = e2e_schedule(n, nb, ctx->sm_count, dehaze_strips(w), dehaze_strips_narrow(w));
  if (const char* e = getenv("UWIP_E2E_SIZES")) {   // tuning: an explicit comma-separated schedule (used when it adds up to n)
    std::vector<int> v;
    long sum = 0;
    for (const char* q = e; *q;) {
      char* end = nullptr;
      long m = strtol(q, &end, 10);
      if (end == q || m <= 0) { v.clear(); break; }
      v.push_back((int)m); sum += m;
      q = (*end == ',') ? end + 1 : end;
      if (*end && *end != ',') { v.clear(); break; }
    }
    if (!v.empty() && sum == n && *std::max_element(v.begin(), v.end()) <= nb) sizes = v;
  }
  nb = *std::max_element(sizes.begin(), sizes.end());
  FrameState* fs = frame_state_get(ctx, nb);
  int32_t* flags = flags_get(ctx, n);
  size_t fbytes = (size_t)w * h * 3;
  uint8_t* din[2] = {(uint8_t*)uwip_slot(ctx, SLOT_CHAIN_IN0, fbytes * nb), (uint8_t*)uwip_slot(ctx, SLOT_CHAIN_IN1, fbytes * nb)};
  uint8_t* dout[2] = {(uint8_t*)uwip_slot(ctx, SLOT_CHAIN_OUT0, fbytes * nb), (uint8_t*)uwip_slot(ctx, SLOT_CHAIN_OUT1, fbytes * nb)};
  if (!fs || !flags || !din[0] || !din[1] || !dout[0] || !dout[1]) return UWIP_ERR_NOMEM;
  // copy streams and events live in the context (created on first use, destroyed with it)
  if (!ctx->s_in) UWIP_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
  if (!ctx->s_out) UWIP_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
  cudaStream_t s_in = ctx->s_in, s_out = ctx->s_out;
  int nsub = (int)sizes.size();
  while ((int)ctx->ev_pool.size() < 3 * nsub + 1) {
    cudaEvent_t e;
    UWIP_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ctx->ev_pool.push_back(e);
  }
  cudaEvent_t* ev_in = ctx->ev_pool.data();
  cudaEvent_t* ev_comp = ev_in + nsub;
  cudaEvent_t* ev_out = ev_comp + nsub;
  cudaEvent_t ev_start = ctx->ev_pool[3 * nsub];
  // the workspace of the largest sub-batch is sized before the pipeline starts: growing a slot synchronises and frees
  UWIP_CHECK(chain_reserve(ctx, nb, w, h, *p));
  int rc = UWIP_OK;
  cudaEventRecord(ev_start, ctx->stream);  // order after whatever the caller queued on the context stream
  cudaStreamWaitEvent(s_in, ev_start, 0);
  size_t first = 0;
  for (int i = 0; i < nsub && rc == UWIP_OK; i++) {
    int m = sizes[i];
    int b = i & 1;
    if (i >= 2) cudaStreamWaitEvent(s_in, ev_comp[i - 2], 0);       // in-buffer free again
    cudaMemcpyAsync(din[b], src + first * fbytes, fbytes * m, cudaMemcpyHostToDevice, s_in);
    cudaEventRecord(ev_in[i], s_in);
    cudaStreamWaitEvent(ctx->stream, ev_in[i], 0);
    if (i >= 2) cudaStreamWaitEvent(ctx->stream, ev_out[i - 2], 0);  // out-buffer drained
    rc = chain_sub(ctx, din[b], dout[b], m, w, h, *p, fs, flags + first);
    cudaEventRecord(ev_comp[i], ctx->stream);
    cudaStreamWaitEvent(s_out, ev_comp[i], 0);
    cudaMemcpyAsync(dst + first * fbytes, dout[b], fbytes * m, cudaMemcpyDeviceToHost, s_out);
    cudaEventRecord(ev_out[i], s_out);
    first += (size_t)m;
  }
  cudaError_t e1 = cudaStreamSynchronize(s_in), e2 = cudaStreamSynchronize(ctx->stream), e3 = cudaStreamSynchronize(s_out);
  if (rc != UWIP_OK) return rc;
  cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
  if (e != cudaSuccess) { uwip_set_err(ctx, "chain pipeline: %s", cudaGetErrorString(e)); return UWIP_ERR_CUDA; }
  return UWIP_OK;
}

// ---- JPEG files to and from the device (SURVEY 8f N3) ---------------------------------------------------------
int uwip_jpeg_info(uwip_ctx* ctx, const uint8_t* jpeg, size_t len, int* width, int* height) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, jpeg && len > 0 && width && height, "bad argument");
  return jpeg_info(ctx, jpeg, len, width, height);
}
int uwip_jpeg_decode_bgr8_dev(uwip_ctx* ctx, const uint8_t* jpeg, size_t len, uint8_t* d_bgr, int width, int height) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, jpeg && len > 0 && d_bgr && width > 0 && height > 0, "bad argument");
  int w = 0, h = 0;
  UWIP_CHECK(jpeg_info(ctx, jpeg, len, &w, &h));
  UWIP_REQUIRE(ctx, w == width && h == height, "the JPEG stream has another size (uwip_jpeg_info)");
  return jpeg_decode_dev(ctx, jpeg, len, d_bgr, w, h);
}
int uwip_jpeg_encode_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int width, int height, int quality, uint8_t* out, size_t cap, size_t* out_len) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_bgr && width > 0 && height > 0 && out_len && quality >= 1 && quality <= 100, "bad argument");
  return jpeg_encode_dev(ctx, d_bgr, width, height, quality, out, cap, out_len);
}
// JPEG in -> histretch -> aclahe -> bgdehaze on the device -> JPEG out: the file never exists as pixels on the host
int uwip_chain_jpeg(uwip_ctx* ctx, const uint8_t* jpeg_in, size_t len_in, const uwip_chain_params* p, int quality, uint8_t* jpeg_out,
                    size_t cap, size_t* len_out) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, jpeg_in && len_in > 0 && len_out, "bad argument");
  int w = 0, h = 0;
  UWIP_CHECK(jpeg_info(ctx, jpeg_in, len_in, &w, &h));
  UWIP_CHECK(chain_check(ctx, p, 1, w, h));
  const size_t fbytes = (size_t)w * h * 3;
  uint8_t* d_in = (uint8_t*)uwip_slot(ctx, SLOT_CHAIN_IN0, fbytes);
  uint8_t* d_out = (uint8_t*)uwip_slot(ctx, SLOT_CHAIN_OUT0, fbytes);
  if (!d_in || !d_out) return UWIP_ERR_NOMEM;
  UWIP_CHECK(each_sub_batch(ctx, 1, w, h, [&](int, int, FrameState* fs, int32_t* flags) {
    UWIP_CHECK(jpeg_decode_dev(ctx, jpeg_in, len_in, d_in, w, h));
    return chain_sub(ctx, d_in, d_out, 1, w, h, *p, fs, flags);
  }));
  return jpeg_encode_dev(ctx, d_out, w, h, quality, jpeg_out, cap, len_out);
}

size_t uwip_jpeg_encode_bound(int width, int height) {
  if (width < 1 || width > 65535 || height < 1 || height > 65535) return 0;
  return jpeg_encode_bound(width, height);
}
int uwip_jpeg_encode_bgr8_batch_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int n_frames, int width, int height, int quality, uint8_t* d_out,
                                    size_t out_stride, uint64_t* d_len) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_bgr && d_out && d_len && n_frames > 0, "bad argument");
  UWIP_REQUIRE(ctx, width >= 1 && width <= 65535 && height >= 1 && height <= 65535, "width and height must lie in 1..65535");
  UWIP_REQUIRE(ctx, quality >= 1 && quality <= 100, "quality must lie in 1..100");
  UWIP_REQUIRE(ctx, out_stride >= jpeg_encode_bound(width, height), "out_stride is below uwip_jpeg_encode_bound(width, height)");
  return jpeg_encode_batch_dev(ctx, d_bgr, n_frames, width, height, quality, d_out, out_stride, d_len);
}
size_t uwip_jpeg_encode_u8_bound(int width, int height) {
  if (width < 1 || width > 65535 || height < 1 || height > 65535) return 0;
  return jpeg_encode_u8_bound(width, height);
}
int uwip_jpeg_encode_u8_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n_frames, int width, int height, int quality, uint8_t* d_out,
                                  size_t out_stride, uint64_t* d_len) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_planes && d_out && d_len && n_frames > 0, "bad argument");
  UWIP_REQUIRE(ctx, width >= 1 && width <= 65535 && height >= 1 && height <= 65535, "width and height must lie in 1..65535");
  UWIP_REQUIRE(ctx, quality >= 1 && quality <= 100, "quality must lie in 1..100");
  UWIP_REQUIRE(ctx, out_stride >= jpeg_encode_u8_bound(width, height), "out_stride is below uwip_jpeg_encode_u8_bound(width, height)");
  return jpeg_encode_u8_batch_dev(ctx, d_planes, n_frames, width, height, quality, d_out, out_stride, d_len);
}

// the argument checks of the two batched readers (in the caller, whose name the messages carry)
#define DECODE_BATCH_REQUIRE(ctx, d_out)                                                                                         \
  UWIP_REQUIRE(ctx, jpegs && lens && d_out && n_frames > 0 && n_frames <= 65535, "bad argument (n_frames must lie in 1..65535)"); \
  UWIP_REQUIRE(ctx, width >= 1 && width <= 65500 && height >= 1 && height <= 65500, "width and height must lie in 1..65500");    \
  for (int f = 0; f < n_frames; f++) UWIP_REQUIRE(ctx, jpegs[f] && lens[f] > 0, "a file pointer is NULL or a length is 0")
int uwip_jpeg_decode_bgr8_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames, uint8_t* d_bgr, int width,
                                int height) {
  CTX_GUARD(ctx);
  DECODE_BATCH_REQUIRE(ctx, d_bgr);
  int32_t* flags = flags_get(ctx, n_frames);
  if (!flags) return UWIP_ERR_NOMEM;
  return jpeg_decode_batch(ctx, jpegs, lens, n_frames, d_bgr, width, height, flags, false, false);
}
int uwip_jpeg_decode_u8_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames, uint8_t* d_planes, int width,
                              int height) {
  CTX_GUARD(ctx);
  DECODE_BATCH_REQUIRE(ctx, d_planes);
  int32_t* flags = flags_get(ctx, n_frames);
  if (!flags) return UWIP_ERR_NOMEM;
  return jpeg_decode_batch(ctx, jpegs, lens, n_frames, d_planes, width, height, flags, true, false);
}
int uwip_jpeg_decode_bgr8_batch_oriented(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames, uint8_t* d_bgr,
                                         int width, int height) {
  CTX_GUARD(ctx);
  DECODE_BATCH_REQUIRE(ctx, d_bgr);
  int32_t* flags = flags_get(ctx, n_frames);
  if (!flags) return UWIP_ERR_NOMEM;
  return jpeg_decode_batch(ctx, jpegs, lens, n_frames, d_bgr, width, height, flags, false, true);
}
int uwip_jpeg_decode_u8_batch_oriented(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n_frames, uint8_t* d_planes,
                                       int width, int height) {
  CTX_GUARD(ctx);
  DECODE_BATCH_REQUIRE(ctx, d_planes);
  int32_t* flags = flags_get(ctx, n_frames);
  if (!flags) return UWIP_ERR_NOMEM;
  return jpeg_decode_batch(ctx, jpegs, lens, n_frames, d_planes, width, height, flags, true, true);
}
int uwip_jpeg_orientation(const uint8_t* jpeg, size_t len, int* orientation) {
  if (!jpeg || !len || !orientation) return UWIP_ERR_INVALID;
  return jpeg_orientation(jpeg, len, orientation);
}
int uwip_jpeg_decode_stats(uwip_ctx* ctx, int n, int32_t* stats_host) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, stats_host && n > 0, "bad argument");
  UWIP_REQUIRE(ctx, ctx->jdec_stats && n <= ctx->jdec_n, "more frames requested than the last batched JPEG decode processed");
  UWIP_CUDA(ctx, cudaMemcpyAsync(stats_host, ctx->jdec_stats, sizeof(int32_t) * 2 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}

int uwip_last_frame_flags(uwip_ctx* ctx, int n, int32_t* flags_host) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, flags_host && n > 0, "bad argument");
  UWIP_REQUIRE(ctx, n <= ctx->flags_n, "more frames requested than the last batched call processed");
  UWIP_CUDA(ctx, cudaMemcpyAsync(flags_host, ctx->slot_ptr[SLOT_FLAGS], sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UWIP_OK;
}

// ---- synthetic input ------------------------------------------------------------------------------------
int uwip_synth_bgr8_dev(uwip_ctx* ctx, uint8_t* d_dst, uint32_t seed, int first, int n, int w, int h) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_dst && n > 0 && w > 0 && h > 0 && first >= 0, "bad argument");
  return synth_frames_dev(ctx, d_dst, seed, first, n, w, h);
}
int uwip_checksum_bgr8_dev(uwip_ctx* ctx, const uint8_t* d_src, int n, int w, int h, uint64_t* sums_host) {
  CTX_GUARD(ctx);
  UWIP_REQUIRE(ctx, d_src && sums_host && n > 0, "bad argument");
  return checksum_frames_dev(ctx, d_src, n, w, h, sums_host);
}

}  // extern "C"
