// common.cuh - context, launch bookkeeping and the bit-exact colour arithmetic shared by all kernels.
// Target: sm_100a only.  No OpenCV, no torch.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/uwip.h"

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct ProfRec {
  const char* tag;
  cudaEvent_t e0, e1;
};

struct uwip_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  int64_t launches = 0;
  bool profiling = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;       // timing-disabled events of the host-buffer pipeline, created on demand, reused
  cudaStream_t s_in = nullptr, s_out = nullptr;   // copy streams of the host-buffer pipeline (created on first use)
  std::string err;
  // named, grow-only device buffers
  static const int kSlots = 33;
  void* slot_ptr[kSlots] = {};
  size_t slot_bytes[kSlots] = {};
  void* pinned = nullptr;  // small pinned scratch for scalar results
  size_t pinned_bytes = 0;
  int flags_n = 0;         // frames covered by SLOT_FLAGS (last batched chain / dehaze call)
  // opt-in dynamic shared memory already granted on THIS context's device, per kernel (cudaFuncSetAttribute is
  // per device: a process-global flag would leave the second device of a process without the opt-in)
  void* jpeg = nullptr;    // nvJPEG handles of the file entry points (jpegio.cu), created on first use
  // batched exact JPEG decoder (jpegdec.cu): pinned staging of the entropy-coded segments and tables, the event after the
  // copies that read it, and the per-frame statistics of the last call (device, 2 x int32 per frame)
  void* jdec_pinned = nullptr;
  size_t jdec_pinned_bytes = 0;
  cudaEvent_t jdec_ev = nullptr;
  int32_t* jdec_stats = nullptr;
  int jdec_n = 0;
  static const int kFuncs = 16;
  size_t func_smem[kFuncs] = {};
};

enum FuncId { FUNC_GF1A = 0, FUNC_GF1B, FUNC_GF2A, FUNC_GF2B, FUNC_WINDOW, FUNC_WINDOW15, FUNC_SWEEP, FUNC_GFQ };

// grant `bytes` of dynamic shared memory to `kern` on the context's device (once per context and size)
template <class K>
static inline cudaError_t uwip_func_smem(uwip_ctx* ctx, int id, K kern, size_t bytes) {
  if (bytes <= ctx->func_smem[id]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) ctx->func_smem[id] = bytes;
  return e;
}

enum Slot {
  SLOT_STAGE_IN = 0,  // host-API staging: input frames
  SLOT_STAGE_OUT,     // host-API staging: output frames
  SLOT_HIST,          // per-frame 256-bin histograms (u32)
  SLOT_LUT,           // per-frame stretch LUTs
  SLOT_TILEHIST,      // per-frame per-tile histograms (u32)
  SLOT_TILELUT,       // per-frame per-tile CLAHE LUTs (u8)
  SLOT_FSTATE,        // FrameState[n]
  SLOT_TMP_FRAME,     // intermediate bgr8 frames
  SLOT_MPLANES,       // dehaze: window-min plane of green (u8)
  SLOT_PARTIALS,      // dehaze: per-block arg-min partials
  SLOT_AB,            // dehaze: guided-filter coefficient planes (int32 fixed point x8)
  SLOT_J,             // dehaze: J_blue, J_green (f32 x2)
  SLOT_REFS,          // dehaze: refined exposure map (f32)
  SLOT_F64OUT,        // float64 outputs for the stage-wise host API
  SLOT_MISC,
  SLOT_CHAIN_IN0,
  SLOT_CHAIN_IN1,
  SLOT_CHAIN_OUT0,
  SLOT_CHAIN_OUT1,
  SLOT_SWEEP,
  SLOT_FLAGS,         // per-frame status words of the last chain / dehaze call (int32)
  SLOT_KQ,            // dehaze: packed k'_b k'_g k'_r m'_b (u32)
  SLOT_YCC,           // dehaze: packed Yi Cri Cbi Yj (u32)
  SLOT_STAB,          // dehaze: exposure-ratio table (u32 rint(S 2^28) x 65536 per frame)
  SLOT_SPLANE,        // dehaze: exposure ratio per pixel (u32 rint(S 2^28))
  SLOT_BLURSUMS,      // calcBlur: per-frame sum and sum of squares of the 8-bit Laplacian (u64 x2)
  SLOT_BLUROUT,       // calcBlur: per-frame mean, stdev (f64 x2)
  SLOT_APLANE,        // automatic CLAHE: V planes of the frames (u8)
  SLOT_ABLUR,         // automatic CLAHE: blurred planes (u8)
  SLOT_AUTO,          // automatic CLAHE: clip-curve derivatives, per-frame parameters, pick histograms and entropies
  SLOT_AUTO_BSCL,     // automatic CLAHE: BS, CL of the frames when the caller does not ask for them (int32 x2)
  SLOT_JPEGENC,       // batched JPEG encoder: tables, MCU bit offsets, block infos, int16 coefficients
  SLOT_JPEGDEC,       // batched JPEG decoder: tables, segments, compact streams, subsequence states, coefficients, sample planes
};

const char* uwip_set_err(uwip_ctx* ctx, const char* fmt, ...);
void* uwip_slot(uwip_ctx* ctx, int slot, size_t bytes);  // nullptr on failure (error text set)
void uwip_pre_launch(uwip_ctx* ctx, const char* tag);
int uwip_post_launch(uwip_ctx* ctx, const char* tag);

#define UWIP_CUDA(ctx, call)                                                                \
  do {                                                                                      \
    cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess) {                                                               \
      uwip_set_err((ctx), "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return UWIP_ERR_CUDA;                                                                 \
    }                                                                                       \
  } while (0)

#define UWIP_LAUNCH(ctx, tag, kern, grid, block, smem, ...)            \
  do {                                                                 \
    uwip_pre_launch((ctx), (tag));                                     \
    kern<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);     \
    int rc__ = uwip_post_launch((ctx), (tag));                         \
    if (rc__ != UWIP_OK) return rc__;                                  \
  } while (0)

#define UWIP_CHECK(expr)          \
  do {                            \
    int rc__ = (expr);            \
    if (rc__ != UWIP_OK) return rc__; \
  } while (0)

#define UWIP_REQUIRE(ctx, cond, msg)                       \
  do {                                                     \
    if (!(cond)) {                                         \
      uwip_set_err((ctx), "%s: %s", __func__, (msg));      \
      return UWIP_ERR_INVALID;                             \
    }                                                      \
  } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------
// per-frame device state: every frame-global reduction result lives here so that no pass needs a
// host round trip.  One struct per frame in a batch.
// ------------------------------------------------------------------------------------------------
struct FrameState {
  // histretch
  int low, high;               // percentile bins (preprocessing.cpp:89-94)
  // dehaze D0: joint min / max over all three channels (bgdehaze/main.py:17)
  unsigned int kmin, kmax;     // atomicMin / atomicMax targets
  // dehaze D1: arg-min results (first flat index) and background light
  unsigned int idx0, idx1;
  double B[3];                 // Background_light(normI, w)  (used by dehazed_BG, BGDehaze.py:51)
  double Bt[3];                // Background_light(normI, 15) (used inside transmission_map, :30,52)
  // dehaze D6: per-channel J min / max (ordered-uint encoding of the double) and fixed-point sums
  unsigned long long jmin_key[2], jmax_key[2];
  long long jsum_fix[2];       // sum of J * 2^32 (deterministic integer accumulation)
  // red channel statistics for D7 (min, max, sum of k' red)
  unsigned int rmin, rmax;
  unsigned long long rsum;
  // dehaze D8: joint min / max of the two YCrCb images (u8 arithmetic)
  unsigned int yi_min, yi_max, yj_min, yj_max;
  // final: min / max of OutputExp (ordered-uint encoding)
  unsigned long long omin_key, omax_key;
  unsigned int nan_flag;
  unsigned int pad;
};

// order preserving map double <-> uint64 (for atomicMin / atomicMax on doubles)
__host__ __device__ inline unsigned long long dkey(double d) {
  unsigned long long u;
#ifdef __CUDA_ARCH__
  u = (unsigned long long)__double_as_longlong(d);
#else
  memcpy(&u, &d, 8);
#endif
  return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__host__ __device__ inline double dunkey(unsigned long long k) {
  unsigned long long u = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)u);
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

// ------------------------------------------------------------------------------------------------
// colour arithmetic (SURVEY appendix A.3 - A.5); tables live in constant memory and are staged to
// shared memory by kernels whose index is thread-divergent.
// ------------------------------------------------------------------------------------------------
// sdiv[i] = rint((255<<12)/i), hdiv[i] = rint((180<<12)/(6i)); no exact .5 ties exist for i < 256,
// so round-half-up integer division reproduces OpenCV's tables.  Each CTA fills its own shared copy
// (the index is thread-divergent, which constant memory would serialise).
__device__ __forceinline__ int hsv_sdiv(int i) { return i ? ((255 << 12) * 2 + i) / (2 * i) : 0; }
__device__ __forceinline__ int hsv_hdiv(int i) { return i ? (2 * 122880 + i) / (2 * i) : 0; }

enum Channel {
  CH_B = 0, CH_G = 1, CH_R = 2, CH_H = 3, CH_S = 4, CH_V = 5, CH_Y = 6, CH_CR = 7, CH_CB = 8,
  CH_HLS_H = 9, CH_HLS_L = 10, CH_HLS_S = 11,  // planes 0, 1, 2 of BGR2HLS (letters 'h', 's', 'l': numChannel maps 's' -> 1, 'l' -> 2)
  CH_LAB_L = 12, CH_LAB_A = 13, CH_LAB_B = 14   // planes 0, 1, 2 of BGR2Lab (letters 'L', 'a', 'b')
};

__device__ __forceinline__ int imax3(int a, int b, int c) { return max(max(a, b), c); }
__device__ __forceinline__ int imin3(int a, int b, int c) { return min(min(a, b), c); }

// cvtColor(BGR2HSV) 8-bit, H in [0,180): integer, shift 12.  sdiv/hdiv: shared or constant tables.
__device__ __forceinline__ void bgr2hsv_u8(int b, int g, int r, const int* __restrict__ sdiv,
                                           const int* __restrict__ hdiv, int& h, int& s, int& v) {
  v = imax3(b, g, r);
  int d = v - imin3(b, g, r);
  s = (d * sdiv[v] + (1 << 11)) >> 12;
  int h0 = (v == r) ? (g - b) : ((v == g) ? (b - r + 2 * d) : (r - g + 4 * d));
  h = (h0 * hdiv[d] + (1 << 11)) >> 12;
  if (h < 0) h += 180;
}

// cvtColor(HSV2BGR) 8-bit.  trunc_mode: true = truncate (AVX2 body of cv2 4.13), false = rint.
__device__ __forceinline__ void hsv2bgr_u8(int H, int S, int V, bool trunc_mode, int& b, int& g,
                                           int& r) {
  const float hscale = 6.0f / 180.0f;
  const float k255 = 1.0f / 255.0f;
  float h = __fmul_rn((float)H, hscale);
  float s = __fmul_rn((float)S, k255);
  float v = __fmul_rn((float)V, k255);
  float fsec = floorf(h);
  float f = __fsub_rn(h, fsec);
  int sec = (int)fsec;
  if ((unsigned)sec >= 6u) {
    sec = 0;
    f = 0.f;
  }
  float t0 = v;
  float t1 = __fmul_rn(v, __fsub_rn(1.0f, s));
  float t2 = __fmul_rn(v, __fmaf_rn(-s, f, 1.0f));
  float t3 = __fmul_rn(v, __fmaf_rn(-s, __fsub_rn(1.0f, f), 1.0f));
  // sector table (b,g,r <- tab index): {1,3,0},{1,0,2},{3,0,1},{0,2,1},{0,1,3},{2,1,0}
  float fb, fg, fr;
  switch (sec) {
    case 0: fb = t1; fg = t3; fr = t0; break;
    case 1: fb = t1; fg = t0; fr = t2; break;
    case 2: fb = t3; fg = t0; fr = t1; break;
    case 3: fb = t0; fg = t2; fr = t1; break;
    case 4: fb = t0; fg = t1; fr = t3; break;
    default: fb = t2; fg = t1; fr = t0; break;
  }
  fb = __fmul_rn(fb, 255.0f);
  fg = __fmul_rn(fg, 255.0f);
  fr = __fmul_rn(fr, 255.0f);
  if (trunc_mode) {
    b = __float2int_rz(fb); g = __float2int_rz(fg); r = __float2int_rz(fr);
  } else {
    b = __float2int_rn(fb); g = __float2int_rn(fg); r = __float2int_rn(fr);
  }
  b = min(max(b, 0), 255);
  g = min(max(g, 0), 255);
  r = min(max(r, 0), 255);
}

// V channel of HSV2BGR(BGR2HSV(.)) after V was replaced by Vn: the max channel is tab0 = v.
__device__ __forceinline__ int hsv_roundtrip_v(int Vn, bool trunc_mode) {
  float v = __fmul_rn(__fmul_rn((float)Vn, 1.0f / 255.0f), 255.0f);
  int o = trunc_mode ? __float2int_rz(v) : __float2int_rn(v);
  return min(max(o, 0), 255);
}

// cvtColor(BGR2YCrCb) 8-bit: integer, shift 14; order Y, Cr, Cb.
__device__ __forceinline__ void bgr2ycrcb_u8(int b, int g, int r, int& Y, int& Cr, int& Cb) {
  Y = (4899 * r + 9617 * g + 1868 * b + 8192) >> 14;
  Cr = ((r - Y) * 11682 + 128 * 16384 + 8192) >> 14;
  Cb = ((b - Y) * 9241 + 128 * 16384 + 8192) >> 14;
  Cr = min(max(Cr, 0), 255);
  Cb = min(max(Cb, 0), 255);
}

// cvtColor(YCrCb2BGR) 8-bit: integer, shift 14, saturating (equal to cv2 4.13.0 on all 2^24 triples,
// tests/golden/kat.json: all_ycrcb2bgr_crc).
__device__ __forceinline__ void ycrcb2bgr_u8(int Y, int Cr, int Cb, int& b, int& g, int& r) {
  Cr -= 128; Cb -= 128;
  b = Y + ((Cb * 29049 + 8192) >> 14);
  g = Y + ((Cb * -5636 + Cr * -11698 + 8192) >> 14);
  r = Y + ((Cr * 22987 + 8192) >> 14);
  b = min(max(b, 0), 255);
  g = min(max(g, 0), 255);
  r = min(max(r, 0), 255);
}

// cvtColor(BGR2HLS) 8-bit (planes H in [0,180), L, S): float32 on k/255.  cv2 4.13.0 runs the first 8*floor(W/8)
// pixels of a row through a vector body and the rest through the scalar tail; they differ in the S denominator
// and in whether `h += 360` is fused with the product (oracle bgr2hls, pinned on all 2^24 triples for both).
__device__ __forceinline__ void bgr2hls_u8(int bi, int gi, int ri, bool body, int& H, int& L, int& S) {
  const float k255 = 1.0f / 255.0f;
  float b = __fmul_rn((float)bi, k255), g = __fmul_rn((float)gi, k255), r = __fmul_rn((float)ri, k255);
  float vmax = fmaxf(fmaxf(b, g), r), vmin = fminf(fminf(b, g), r);
  float diff = __fsub_rn(vmax, vmin), vs = __fadd_rn(vmax, vmin);
  float lum = __fmul_rn(vs, 0.5f);
  float hue = 0.f, sat = 0.f;
  if (diff > 1.1920928955078125e-07f) {  // FLT_EPSILON
    float den = body ? __fsub_rn(2.0f, vs) : __fsub_rn(__fsub_rn(2.0f, vmax), vmin);
    sat = __fdiv_rn(diff, lum < 0.5f ? vs : den);
    float dinv = __fdiv_rn(60.0f, diff);
    float d, add;
    if (vmax == r) { d = __fsub_rn(g, b); add = 0.f; }
    else if (vmax == g) { d = __fsub_rn(b, r); add = 120.f; }
    else { d = __fsub_rn(r, g); add = 240.f; }
    hue = (add == 0.f) ? __fmul_rn(d, dinv) : __fmaf_rn(d, dinv, add);
    if (hue < 0.f) hue = body ? __fmaf_rn(d, dinv, add + 360.f) : __fadd_rn(hue, 360.f);
  }
  H = min(max(__float2int_rn(__fmul_rn(hue, 0.5f)), 0), 255);
  L = min(max(__float2int_rn(__fmul_rn(lum, 255.0f)), 0), 255);
  S = min(max(__float2int_rn(__fmul_rn(sat, 255.0f)), 0), 255);
}

// cvtColor(HLS2BGR) 8-bit: float32, rint at the end (oracle hls2bgr; H >= 180 wraps the sector modulo 6).
__device__ __forceinline__ void hls2bgr_u8(int H, int L, int S, int& b, int& g, int& r) {
  const float k255 = 1.0f / 255.0f;
  float lum = __fmul_rn((float)L, k255);
  float fb = lum, fg = lum, fr = lum;
  if (S != 0) {
    float s = __fmul_rn((float)S, k255);
    float p2 = (lum <= 0.5f) ? __fmul_rn(lum, __fadd_rn(1.0f, s)) : __fsub_rn(__fadd_rn(lum, s), __fmul_rn(lum, s));
    float p1 = __fsub_rn(__fmul_rn(2.0f, lum), p2);
    float hh = __fmul_rn((float)H, 6.0f / 180.0f);
    float fsec = floorf(hh);
    float f = __fsub_rn(hh, fsec);
    int sec = ((int)fsec) % 6;
    float d = __fsub_rn(p2, p1);
    float t2 = __fadd_rn(p1, __fmul_rn(d, __fsub_rn(1.0f, f)));
    float t3 = __fadd_rn(p1, __fmul_rn(d, f));
    switch (sec) {  // (b,g,r) <- {p2,p1,t2,t3}: {1,3,0},{1,0,2},{3,0,1},{0,2,1},{0,1,3},{2,1,0}
      case 0: fb = p1; fg = t3; fr = p2; break;
      case 1: fb = p1; fg = p2; fr = t2; break;
      case 2: fb = t3; fg = p2; fr = p1; break;
      case 3: fb = p2; fg = t2; fr = p1; break;
      case 4: fb = p2; fg = p1; fr = t3; break;
      default: fb = t2; fg = p1; fr = p2; break;
    }
  }
  b = min(max(__float2int_rn(__fmul_rn(fb, 255.0f)), 0), 255);
  g = min(max(__float2int_rn(__fmul_rn(fg, 255.0f)), 0), 255);
  r = min(max(__float2int_rn(__fmul_rn(fr, 255.0f)), 0), 255);
}

// saturate_cast<uchar>(cvRound(x)) : NaN / inf -> INT_MIN -> 0
__device__ __forceinline__ int sat_rint_u8(float x) {
  if (!(fabsf(x) <= 3.0e9f)) return 0;  // NaN, inf (and absurdly large) -> cvRound gives INT_MIN
  int i = __float2int_rn(x);
  return min(max(i, 0), 255);
}

__device__ __forceinline__ unsigned int warp_reduce_min_u32(unsigned int v) {
  return __reduce_min_sync(0xffffffffu, v);
}
__device__ __forceinline__ unsigned int warp_reduce_max_u32(unsigned int v) {
  return __reduce_max_sync(0xffffffffu, v);
}

// ------------------------------------------------------------------------------------------------
// stage entry points implemented in the other translation units (device pointers, stream ordered)
// ------------------------------------------------------------------------------------------------
// histretch.cu
int k_histogram_plane(uwip_ctx* ctx, const uint8_t* d_plane, int n_planes, size_t n_px, uint32_t* d_hist);
int calc_blur_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, int n, int w, int h, int aperture, double* d_mean_std, uint8_t* d_lap);
int k_histogram_frame(uwip_ctx* ctx, const uint8_t* d_bgr, int n_frames, int w, int h, int channel, uint32_t* d_hist,
                      int hsv_round = UWIP_HSV_ROUND_CV2_4_13);
int k_percentile_lut(uwip_ctx* ctx, const uint32_t* d_hist, int n, int w, int h, int lo, int hi, FrameState* fs, uint8_t* d_lut);
int k_apply_lut_plane(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_planes, size_t n_px, const uint8_t* d_lut);
int k_apply_lut_frame(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_frames, int w, int h, int channel, const uint8_t* d_lut, bool use_lut, int hsv_round);
int k_hist_to_float(uwip_ctx* ctx, const uint32_t* d_hist, float* d_out, int n);
int k_entropy(uwip_ctx* ctx, const uint32_t* d_hist, int n_hists, int w, int h, int flavour, float* d_out);
int k_blur3(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int w, int h, int n = 1);   // n planes of w x h
int histretch_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const char* channels, int lo, int hi, int order, int hsv_round);

// clahe.cu
int clahe_planes_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty);
int aclahe_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty, int hsv_round, const uint8_t* d_prelut /*optional per-frame stretch LUT fused in front*/, FrameState* fs_minmax /*optional: accumulate dehaze D0 min/max of the output*/);
int clahe_entropy_sweep_dev(uwip_ctx* ctx, const uint8_t* d_plane, int w, int h, int tiles, const double* clips, int n_clips, int flavour, float* entropies_host);
int clahe_entropy_sweep_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, const int* grids, int n_grids, const double* clips, int n_clips, int flavour, float* entropies_host);
int aclahe_check_auto_size(uwip_ctx* ctx, int w, int h);   // UWIP_ERR_INVALID when a plane is too small for a grid of 2..32
int aclahe_params_planes_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, int loop, int* d_bs, int* d_cl);
int aclahe_frames_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, double clip, int tx, int ty, int hsv_round, const uint8_t* d_prelut, FrameState* fs_minmax, int* d_bs, int* d_cl);
int aclahe_planes_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, double clip, int tx, int ty, int* d_bs, int* d_cl);
int aclahe_nofit_flags(uwip_ctx* ctx, const int* d_cl, int n, int32_t* d_flags, bool keep);   // flags |= NOFIT where CL < 0

// aclahe_knee.cu
int k_aclahe_knees(uwip_ctx* ctx, const float* d_ent /*[5][n][n_clips]*/, int n, int n_clips, double* d_xd /*[2][49] scratch*/, int* d_cl);

// dehaze.cu
struct DehazeDebug {  // optional float64 stage outputs for the stage-wise host API (device pointers)
  double* t_raw = nullptr;    // [2][H*W] transmission_map
  double* t_ref = nullptr;    // [2][H*W] refined_t
  double* restored = nullptr; // [H*W*3]
  double* out = nullptr;      // [H*W*3]
  int stop_after = 0;         // 0 run all; 1 after background light; 2 after transmission; 3 after refined t; 4 after restored
};
int dehaze_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const uwip_dehaze_params& p, bool minmax_done, FrameState* fs, DehazeDebug* dbg, int32_t* d_flags = nullptr);
int frame_state_reset(uwip_ctx* ctx, FrameState* fs, int n);
int dehaze_strips(int w);         // strips of a frame in the wide layout of the marches (GF1b, GF2a, GF2b)
int dehaze_strips_narrow(int w);  // ... in the narrow layout (GF1a)
int dehaze_sub_batch(const uwip_ctx* ctx, int n, int w, int cap);  // sub-batch size <= cap that wastes the fewest CTA waves
FrameState* frame_state_get(uwip_ctx* ctx, int n);
int boxfilter_f64_dev(uwip_ctx* ctx, const double* d_src, double* d_tmp, double* d_dst, int w, int h, int r);
int guided_filter_u8_dev(uwip_ctx* ctx, const uint8_t* d_guide, const double* d_p, double* d_q, int w, int h, int range, int r, double eps, FrameState* fs);

// jpegio.cu
int jpeg_info(uwip_ctx* ctx, const uint8_t* data, size_t len, int* w, int* h);
int jpeg_decode_dev(uwip_ctx* ctx, const uint8_t* data, size_t len, uint8_t* d_bgr, int w, int h);
int jpeg_encode_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int w, int h, int quality, uint8_t* out, size_t cap, size_t* out_len);
void jpeg_io_destroy(uwip_ctx* ctx);

// jpegenc.cu
size_t jpeg_encode_bound(int w, int h);
size_t jpeg_encode_u8_bound(int w, int h);
int jpeg_encode_batch_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int n, int w, int h, int quality, uint8_t* d_out, size_t stride,
                          uint64_t* d_len);
int jpeg_encode_u8_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, int quality, uint8_t* d_out, size_t stride,
                             uint64_t* d_len);

// jpegdec.cu: d_out receives bgr8 frames, or grey planes (IMREAD_GRAYSCALE) when grey is set; orient: each frame turned by
// its Exif orientation (cv2.imdecode's default flags), w x h being the size after it; prog_ok: progressive files accepted
// too (uwip_jpeg_decode_batch_ex)
int jpeg_decode_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n, uint8_t* d_out, int w, int h,
                      int32_t* d_flags, bool grey, bool orient, bool prog_ok);
int jpeg_probe(const uint8_t* data, size_t len, int* width, int* height, int* orientation, int* progressive);
// the Exif orientation cv2.imdecode applies (1..8) from the host marker reader; its status when the header is refused
int jpeg_orientation(const uint8_t* data, size_t len, int* orientation);
void jpeg_dec_destroy(uwip_ctx* ctx);

// synth.cu
int synth_frames_dev(uwip_ctx* ctx, uint8_t* d_dst, uint32_t seed, int first, int n, int w, int h);
int checksum_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, int n, int w, int h, uint64_t* sums_host);
