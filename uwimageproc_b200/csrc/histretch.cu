// histretch.cu - getHistogram / imgChannelStretch / histretch channel loop for sm_100a.
//   reference: modules/common/preprocessing.cpp:25-34 (getHistogram), :74-105 (imgChannelStretch),
//              modules/histretch/src/histretch.cpp:219-254 (channel loop),
//              modules/aclahe/src/aclahe.cpp:228-248 (aclaheEntropy), aclahe/python/functions.py:14-19,
//              modules/aclahe/python/ACLAHE.py:15 (GaussianBlur 3x3)
// HBM-bound byte work: 16-byte vector loads (16 pixels = 3 x uint4), per-warp privatised shared
// histograms, block prefix scan for the percentile search, LUT apply fused with the colour round trip.
#include "common.cuh"
#include "lab_tables.inc"

// ---- 8-bit CIE Lab (cvtColor BGR2Lab / Lab2BGR; histretch letters L, a, b = transformation[2], histretch.cpp:155-156) ----
// OpenCV 4's bit-exact integer path (RGB2Lab_b / Lab2RGBinteger, D65, sRGB gamma): gamma table -> Q12 matrix ->
// cube-root table -> L, a, b; back through the L -> (y, f(y)) table, the cubic, the Q12 matrix and the inverse
// gamma table.  Equal to cv2 4.13.0 on all 2^24 triples in both directions (oracle bgr2lab / lab2bgr).
template <bool LAB>
struct LabSmem {};
template <>
struct LabSmem<true> {
  uint16_t gamma[256], cbrt[2048], yf[512];
  uint8_t invgamma[4096];
  __device__ void fill(bool fwd, bool inv) {
    if (fwd) {
      for (int i = threadIdx.x; i < 256; i += blockDim.x) gamma[i] = kLabGamma[i];
      for (int i = threadIdx.x; i < 2048; i += blockDim.x) cbrt[i] = kLabCbrt[i];
    }
    if (inv) {
      for (int i = threadIdx.x; i < 512; i += blockDim.x) yf[i] = kLabYF[i];
      for (int i = threadIdx.x; i < 4096; i += blockDim.x) invgamma[i] = kLabInvGamma[i];
    }
  }
};
__device__ __forceinline__ void bgr2lab_u8(int b, int g, int r, const LabSmem<true>& t, int& L, int& A, int& Bc) {
  constexpr int C[9] = LAB_FWD_COEFFS;
  const int R = t.gamma[r], G = t.gamma[g], B = t.gamma[b];
  const int fX = t.cbrt[(R * C[0] + G * C[1] + B * C[2] + 2048) >> 12];
  const int fY = t.cbrt[(R * C[3] + G * C[4] + B * C[5] + 2048) >> 12];
  const int fZ = t.cbrt[(R * C[6] + G * C[7] + B * C[8] + 2048) >> 12];
  constexpr int Lscale = (116 * 255 + 50) / 100, Lshift = -((16 * 255 * (1 << 15) + 50) / 100);
  L = min(max((Lscale * fY + Lshift + 16384) >> 15, 0), 255);
  A = min(max((500 * (fX - fY) + 128 * 32768 + 16384) >> 15, 0), 255);
  Bc = min(max((200 * (fY - fZ) + 128 * 32768 + 16384) >> 15, 0), 255);
}
__device__ __forceinline__ int lab_ab_to_xz(int i) {  // abToXZ_b as a function; integer division truncates toward zero
  constexpr int BASE = 1 << 14;
  return (i <= 3390) ? (i * 108) / 841 - BASE * 16 / 116 * 108 / 841 : (i * i / BASE) * i / BASE;
}
__device__ __forceinline__ void lab2bgr_u8(int L, int A, int Bc, const LabSmem<true>& t, int& b, int& g, int& r) {
  constexpr int C[9] = LAB_INV_COEFFS;
  constexpr int BASE = 1 << 14;
  const int y = t.yf[2 * L], ify = t.yf[2 * L + 1];
  const int adiv = ((5 * A * 53687 + (1 << 7)) >> 13) - 128 * BASE / 500;
  const int bdiv = ((Bc * 41943 + (1 << 4)) >> 9) - 128 * BASE / 200 + 1;
  const int x = lab_ab_to_xz(ify + adiv), z = lab_ab_to_xz(ify - bdiv);
  const int ro = min(max((C[0] * x + C[1] * y + C[2] * z + 8192) >> 14, 0), 4095);
  const int go = min(max((C[3] * x + C[4] * y + C[5] * z + 8192) >> 14, 0), 4095);
  const int bo = min(max((C[6] * x + C[7] * y + C[8] * z + 8192) >> 14, 0), 4095);
  r = t.invgamma[ro]; g = t.invgamma[go]; b = t.invgamma[bo];
}
template <int CH>
struct IsLab { static constexpr bool value = (CH == CH_LAB_L || CH == CH_LAB_A || CH == CH_LAB_B); };

// ---- helpers for 16-pixel (48 byte) groups ---------------------------------------------------
struct Px16 {
  uint32_t w[12];
};
__device__ __forceinline__ Px16 load_px16(const uint8_t* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
  Px16 r;
  r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w;
  r.w[4] = b.x; r.w[5] = b.y; r.w[6] = b.z; r.w[7] = b.w;
  r.w[8] = c.x; r.w[9] = c.y; r.w[10] = c.z; r.w[11] = c.w;
  return r;
}
__device__ __forceinline__ void store_px16(uint8_t* p, const Px16& r) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(r.w[0], r.w[1], r.w[2], r.w[3]);
  q[1] = make_uint4(r.w[4], r.w[5], r.w[6], r.w[7]);
  q[2] = make_uint4(r.w[8], r.w[9], r.w[10], r.w[11]);
}
__device__ __forceinline__ int px_byte(const Px16& r, int idx) {  // idx is a compile-time constant after unrolling
  return (r.w[idx >> 2] >> ((idx & 3) * 8)) & 0xff;
}
__device__ __forceinline__ void px_set(Px16& r, int idx, int v) {
  int sh = (idx & 3) * 8;
  r.w[idx >> 2] = (r.w[idx >> 2] & ~(0xffu << sh)) | ((uint32_t)v << sh);
}

template <int CH>
__device__ __forceinline__ int extract_channel(int b, int g, int r, const int* sdiv, const int* hdiv, bool hls_body,
                                               const LabSmem<IsLab<CH>::value>& lab) {
  if (CH == CH_B) return b;
  if (CH == CH_G) return g;
  if (CH == CH_R) return r;
  if (CH == CH_V) return imax3(b, g, r);
  if (CH == CH_Y || CH == CH_CR || CH == CH_CB) {
    int Y, Cr, Cb;
    bgr2ycrcb_u8(b, g, r, Y, Cr, Cb);
    return CH == CH_Y ? Y : (CH == CH_CR ? Cr : Cb);
  }
  if (CH == CH_HLS_H || CH == CH_HLS_L || CH == CH_HLS_S) {
    int H, L, S;
    bgr2hls_u8(b, g, r, hls_body, H, L, S);
    return CH == CH_HLS_H ? H : (CH == CH_HLS_L ? L : S);
  }
  if constexpr (IsLab<CH>::value) {
    int L, A, Bc;
    bgr2lab_u8(b, g, r, lab, L, A, Bc);
    return CH == CH_LAB_L ? L : (CH == CH_LAB_A ? A : Bc);
  }
  int h, s, v;
  bgr2hsv_u8(b, g, r, sdiv, hdiv, h, s, v);
  return CH == CH_H ? h : s;
}

// ---- histogram kernels -----------------------------------------------------------------------
constexpr int HIST_THREADS = 256;
constexpr int HIST_WARPS = HIST_THREADS / 32;

__device__ __forceinline__ void hist_flush(uint32_t (*sh)[256], uint32_t* gh) {
  __syncthreads();
  int t = threadIdx.x;
  uint32_t s = 0;
#pragma unroll
  for (int w = 0; w < HIST_WARPS; w++) s += sh[w][t];
  if (s) atomicAdd(&gh[t], s);
}

// planes: grid (blocks, n_planes); n_px per plane
__global__ void __launch_bounds__(HIST_THREADS) hist_plane_kernel(const uint8_t* __restrict__ src, size_t n_px,
                                                                  uint32_t* __restrict__ hist) {
  __shared__ uint32_t sh[HIST_WARPS][256];
  for (int i = threadIdx.x; i < HIST_WARPS * 256; i += HIST_THREADS) (&sh[0][0])[i] = 0;
  __syncthreads();
  const uint8_t* p = src + (size_t)blockIdx.y * n_px;
  uint32_t* myh = sh[threadIdx.x >> 5];
  bool vec = ((((uintptr_t)p) & 15) == 0);
  size_t n16 = vec ? n_px / 16 : 0;
  for (size_t g = (size_t)blockIdx.x * HIST_THREADS + threadIdx.x; g < n16; g += (size_t)gridDim.x * HIST_THREADS) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + g);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      atomicAdd(&myh[w[k] & 0xff], 1u);
      atomicAdd(&myh[(w[k] >> 8) & 0xff], 1u);
      atomicAdd(&myh[(w[k] >> 16) & 0xff], 1u);
      atomicAdd(&myh[w[k] >> 24], 1u);
    }
  }
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * HIST_THREADS + threadIdx.x; i < n_px; i += (size_t)gridDim.x * HIST_THREADS)
    atomicAdd(&myh[p[i]], 1u);
  hist_flush(sh, hist + (size_t)blockIdx.y * 256);
}

// frames: grid (blocks, n_frames); histogram of one channel (B,G,R,H,S,V) of a bgr8 frame
template <int CH>
__global__ void __launch_bounds__(HIST_THREADS) hist_frame_kernel(const uint8_t* __restrict__ src, size_t n_px,
                                                                  uint32_t* __restrict__ hist, int w, int hls_body_w) {
  constexpr bool HLS = (CH == CH_HLS_H || CH == CH_HLS_L || CH == CH_HLS_S);  // the only channels that depend on x
  __shared__ uint32_t sh[HIST_WARPS][256];
  __shared__ int s_sdiv[256], s_hdiv[256];
  __shared__ LabSmem<IsLab<CH>::value> s_lab;
  if constexpr (IsLab<CH>::value) s_lab.fill(true, false);
  for (int i = threadIdx.x; i < HIST_WARPS * 256; i += HIST_THREADS) (&sh[0][0])[i] = 0;
  if (CH == CH_H || CH == CH_S) {
    s_sdiv[threadIdx.x] = hsv_sdiv(threadIdx.x);
    s_hdiv[threadIdx.x] = hsv_hdiv(threadIdx.x);
  }
  __syncthreads();
  const uint8_t* p = src + (size_t)blockIdx.y * n_px * 3;
  uint32_t* myh = sh[threadIdx.x >> 5];
  bool vec = ((((uintptr_t)p) & 15) == 0);
  size_t n16 = vec ? n_px / 16 : 0;
  for (size_t g = (size_t)blockIdx.x * HIST_THREADS + threadIdx.x; g < n16; g += (size_t)gridDim.x * HIST_THREADS) {
    Px16 q = load_px16(p + g * 48);
    int x0 = HLS ? (int)((g * 16) % (size_t)w) : 0;
#pragma unroll
    for (int k = 0; k < 16; k++) {
      int xk = x0 + k;
      if (HLS && xk >= w) xk -= w;  // a 16-pixel group may straddle a row end
      int v = extract_channel<CH>(px_byte(q, 3 * k), px_byte(q, 3 * k + 1), px_byte(q, 3 * k + 2), s_sdiv, s_hdiv,
                                  HLS && xk < hls_body_w, s_lab);
      atomicAdd(&myh[v], 1u);
    }
  }
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * HIST_THREADS + threadIdx.x; i < n_px; i += (size_t)gridDim.x * HIST_THREADS) {
    int v = extract_channel<CH>(p[3 * i], p[3 * i + 1], p[3 * i + 2], s_sdiv, s_hdiv,
                                HLS && (int)(i % (size_t)w) < hls_body_w, s_lab);
    atomicAdd(&myh[v], 1u);
  }
  hist_flush(sh, hist + (size_t)blockIdx.y * 256);
}

static int hist_grid_x(uwip_ctx* ctx, size_t n_px, int n) {
  // enough blocks to fill the machine (multiples of the SM count), at most one 16-px group per thread
  size_t groups = (n_px + 15) / 16;
  int want = (int)((groups + HIST_THREADS - 1) / HIST_THREADS);
  int per_frame = (ctx->sm_count * 8 + n - 1) / n;
  int gx = want < per_frame ? want : per_frame;
  return gx < 1 ? 1 : gx;
}

int k_histogram_plane(uwip_ctx* ctx, const uint8_t* d_plane, int n_planes, size_t n_px, uint32_t* d_hist) {
  UWIP_CUDA(ctx, cudaMemsetAsync(d_hist, 0, (size_t)n_planes * 256 * 4, ctx->stream));
  dim3 grid(hist_grid_x(ctx, n_px, n_planes), n_planes);
  UWIP_LAUNCH(ctx, "hist_plane", hist_plane_kernel, grid, HIST_THREADS, 0, d_plane, n_px, d_hist);
  return UWIP_OK;
}

static int hls_body_width(int w, int hsv_round) { return hsv_round == UWIP_HSV_ROUND_CV2_4_13 ? 8 * (w / 8) : 0; }

int k_histogram_frame(uwip_ctx* ctx, const uint8_t* d_bgr, int n, int w, int h, int channel, uint32_t* d_hist, int hsv_round) {
  int hbw = hls_body_width(w, hsv_round);
  UWIP_CUDA(ctx, cudaMemsetAsync(d_hist, 0, (size_t)n * 256 * 4, ctx->stream));
  size_t n_px = (size_t)w * h;
  dim3 grid(hist_grid_x(ctx, n_px, n), n);
  switch (channel) {
    case CH_B: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_B>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_G: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_G>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_R: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_R>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_H: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_H>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_S: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_S>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_V: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_V>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_Y: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_Y>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_CR: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_CR>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_CB: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_CB>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_HLS_H: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_HLS_H>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_HLS_L: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_HLS_L>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_HLS_S: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_HLS_S>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_LAB_L: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_LAB_L>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_LAB_A: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_LAB_A>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    case CH_LAB_B: UWIP_LAUNCH(ctx, "hist_frame", hist_frame_kernel<CH_LAB_B>, grid, HIST_THREADS, 0, d_bgr, n_px, d_hist, w, hbw); break;
    default: uwip_set_err(ctx, "bad channel %d", channel); return UWIP_ERR_INVALID;
  }
  return UWIP_OK;
}

// ---- percentile search + stretch LUT (preprocessing.cpp:80-100) --------------------------------
// one block of 256 threads per histogram: block prefix scan, then the float32 while-loop's stopping
// bins are "number of bins whose exclusive prefix is below the threshold" - 1.
__global__ void __launch_bounds__(256) percentile_lut_kernel(const uint32_t* __restrict__ hist, int w, int h, int lo, int hi,
                                                             FrameState* fs, uint8_t* __restrict__ lut) {
  __shared__ uint32_t s_warp[8];
  __shared__ int s_lowhigh[2];
  int t = threadIdx.x, f = blockIdx.x;
  uint32_t c = hist[(size_t)f * 256 + t];
  uint32_t incl = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
    if ((t & 31) >= d) incl += o;
  }
  if ((t & 31) == 31) s_warp[t >> 5] = incl;
  __syncthreads();
  uint32_t base = 0;
#pragma unroll
  for (int k = 0; k < 8; k++)
    if (k < (t >> 5)) base += s_warp[k];
  incl += base;
  uint32_t excl = incl - c;
  uint32_t total = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) total += s_warp[k];

  float norm = (float)((double)(h * w) / 100.0);
  float lo_thr = __fmul_rn((float)lo, norm);
  float hi_thr = __fmul_rn((float)hi, norm);
  int low, high;
  if (total < (1u << 24)) {
    // every partial sum is an integer < 2^24: the float accumulator of the reference is exact
    int p_hi = ((float)excl < hi_thr);
    int p_lo = p_hi && ((float)excl < lo_thr);
    high = __syncthreads_count(p_hi) - 1;
    low = __syncthreads_count(p_lo) - 1;
  } else {
    // very large planes: replay the float32 accumulation literally
    if (t == 0) {
      float sum = 0.f;
      int l = -1, hh = -1, i = 0;
      while (sum < hi_thr && i < 256) {
        if (sum < lo_thr) l++;
        hh++;
        sum = __fadd_rn(sum, (float)hist[(size_t)f * 256 + i]);
        i++;
      }
      s_lowhigh[0] = l;
      s_lowhigh[1] = hh;
    }
    __syncthreads();
    low = s_lowhigh[0];
    high = s_lowhigh[1];
  }
  if (t == 0 && fs) {
    fs[f].low = low;
    fs[f].high = high;
  }
  int y = min(max(t - low, 0), 255);
  int d = high - low;
  int z = 0;
  if (d != 0) {
    float m = (float)(255.0 / (double)d);
    z = sat_rint_u8(__fmul_rn((float)y, m));
  }
  lut[(size_t)f * 256 + t] = (uint8_t)z;
}

int k_percentile_lut(uwip_ctx* ctx, const uint32_t* d_hist, int n, int w, int h, int lo, int hi, FrameState* fs, uint8_t* d_lut) {
  UWIP_LAUNCH(ctx, "percentile_lut", percentile_lut_kernel, n, 256, 0, d_hist, w, h, lo, hi, fs, d_lut);
  return UWIP_OK;
}

// ---- LUT apply ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) apply_lut_plane_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                              size_t n_px, const uint8_t* __restrict__ lut) {
  __shared__ uint8_t s_lut[256];
  s_lut[threadIdx.x] = lut[(size_t)blockIdx.y * 256 + threadIdx.x];
  __syncthreads();
  const uint8_t* p = src + (size_t)blockIdx.y * n_px;
  uint8_t* o = dst + (size_t)blockIdx.y * n_px;
  bool vec = (((((uintptr_t)p) | ((uintptr_t)o)) & 15) == 0);
  size_t n16 = vec ? n_px / 16 : 0;
  for (size_t g = (size_t)blockIdx.x * 256 + threadIdx.x; g < n16; g += (size_t)gridDim.x * 256) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + g);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++)
      w[k] = (uint32_t)s_lut[w[k] & 0xff] | ((uint32_t)s_lut[(w[k] >> 8) & 0xff] << 8) |
             ((uint32_t)s_lut[(w[k] >> 16) & 0xff] << 16) | ((uint32_t)s_lut[w[k] >> 24] << 24);
    reinterpret_cast<uint4*>(o)[g] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * 256 + threadIdx.x; i < n_px; i += (size_t)gridDim.x * 256) o[i] = s_lut[p[i]];
}

int k_apply_lut_plane(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n_planes, size_t n_px, const uint8_t* d_lut) {
  dim3 grid(hist_grid_x(ctx, n_px, n_planes), n_planes);
  UWIP_LAUNCH(ctx, "apply_lut_plane", apply_lut_plane_kernel, grid, 256, 0, d_src, d_dst, n_px, d_lut);
  return UWIP_OK;
}

// one pixel of the histretch channel loop: (optionally) convert, LUT one channel, convert back
template <int CH>
__device__ __forceinline__ void stretch_pixel(int& b, int& g, int& r, const uint8_t* s_lut, bool use_lut, bool trunc_mode,
                                              const int* sdiv, const int* hdiv, bool hls_body,
                                              const LabSmem<IsLab<CH>::value>& lab) {
  if (CH == CH_B) { if (use_lut) b = s_lut[b]; return; }
  if (CH == CH_G) { if (use_lut) g = s_lut[g]; return; }
  if (CH == CH_R) { if (use_lut) r = s_lut[r]; return; }
  if (CH == CH_Y || CH == CH_CR || CH == CH_CB) {  // transformation[3]: BGR2YCrCb / YCrCb2BGR (histretch.cpp:155-156)
    int Y, Cr, Cb;
    bgr2ycrcb_u8(b, g, r, Y, Cr, Cb);
    if (use_lut) {
      if (CH == CH_Y) Y = s_lut[Y];
      if (CH == CH_CR) Cr = s_lut[Cr];
      if (CH == CH_CB) Cb = s_lut[Cb];
    }
    ycrcb2bgr_u8(Y, Cr, Cb, b, g, r);
    return;
  }
  if (CH == CH_HLS_H || CH == CH_HLS_L || CH == CH_HLS_S) {  // transformation[1]: BGR2HLS / HLS2BGR
    int H, L, S;
    bgr2hls_u8(b, g, r, hls_body, H, L, S);
    if (use_lut) {
      if (CH == CH_HLS_H) H = s_lut[H];
      if (CH == CH_HLS_L) L = s_lut[L];
      if (CH == CH_HLS_S) S = s_lut[S];
    }
    hls2bgr_u8(H, L, S, b, g, r);
    return;
  }
  if constexpr (IsLab<CH>::value) {  // transformation[2]: BGR2Lab / Lab2BGR
    int L, A, Bc;
    bgr2lab_u8(b, g, r, lab, L, A, Bc);
    if (use_lut) {
      if (CH == CH_LAB_L) L = s_lut[L];
      if (CH == CH_LAB_A) A = s_lut[A];
      if (CH == CH_LAB_B) Bc = s_lut[Bc];
    }
    lab2bgr_u8(L, A, Bc, lab, b, g, r);
    return;
  }
  int h, s, v;
  bgr2hsv_u8(b, g, r, sdiv, hdiv, h, s, v);
  if (use_lut) {
    if (CH == CH_H) h = s_lut[h];
    if (CH == CH_S) s = s_lut[s];
    if (CH == CH_V) v = s_lut[v];
  }
  hsv2bgr_u8(h, s, v, trunc_mode, b, g, r);
}

// grid (blocks, n_frames).  body_w: pixels with x < body_w truncate in HSV2BGR, the others round.
template <int CH>
__global__ void __launch_bounds__(256) apply_lut_frame_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int w,
                                                              int h, const uint8_t* __restrict__ lut, int use_lut, int body_w, int hls_body_w) {
  __shared__ uint8_t s_lut[256];
  __shared__ int s_sdiv[256], s_hdiv[256];
  __shared__ LabSmem<IsLab<CH>::value> s_lab;
  if constexpr (IsLab<CH>::value) s_lab.fill(true, true);
  s_lut[threadIdx.x] = use_lut ? lut[(size_t)blockIdx.y * 256 + threadIdx.x] : (uint8_t)threadIdx.x;
  s_sdiv[threadIdx.x] = hsv_sdiv(threadIdx.x);
  s_hdiv[threadIdx.x] = hsv_hdiv(threadIdx.x);
  __syncthreads();
  size_t n_px = (size_t)w * h;
  const uint8_t* p = src + (size_t)blockIdx.y * n_px * 3;
  uint8_t* o = dst + (size_t)blockIdx.y * n_px * 3;
  bool vec = (((((uintptr_t)p) | ((uintptr_t)o)) & 15) == 0) && (w % 16 == 0);
  size_t n16 = vec ? n_px / 16 : 0;
  for (size_t gi = (size_t)blockIdx.x * 256 + threadIdx.x; gi < n16; gi += (size_t)gridDim.x * 256) {
    Px16 q = load_px16(p + gi * 48);
    int x0 = (int)((gi * 16) % (size_t)w);
#pragma unroll
    for (int k = 0; k < 16; k++) {
      int b = px_byte(q, 3 * k), g = px_byte(q, 3 * k + 1), r = px_byte(q, 3 * k + 2);
      stretch_pixel<CH>(b, g, r, s_lut, use_lut, (x0 + k) < body_w, s_sdiv, s_hdiv, (x0 + k) < hls_body_w, s_lab);
      px_set(q, 3 * k, b);
      px_set(q, 3 * k + 1, g);
      px_set(q, 3 * k + 2, r);
    }
    store_px16(o + gi * 48, q);
  }
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * 256 + threadIdx.x; i < n_px; i += (size_t)gridDim.x * 256) {
    int b = p[3 * i], g = p[3 * i + 1], r = p[3 * i + 2];
    int x = (int)(i % (size_t)w);
    stretch_pixel<CH>(b, g, r, s_lut, use_lut, x < body_w, s_sdiv, s_hdiv, x < hls_body_w, s_lab);
    o[3 * i] = (uint8_t)b;
    o[3 * i + 1] = (uint8_t)g;
    o[3 * i + 2] = (uint8_t)r;
  }
}

static int body_width(int w, int hsv_round) {
  if (hsv_round == UWIP_HSV_ROUND_TRUNC) return w;
  if (hsv_round == UWIP_HSV_ROUND_RINT) return 0;
  return 32 * (w / 32);
}

int k_apply_lut_frame(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int channel,
                      const uint8_t* d_lut, bool use_lut, int hsv_round) {
  size_t n_px = (size_t)w * h;
  dim3 grid(hist_grid_x(ctx, n_px, n), n);
  int bw = body_width(w, hsv_round);
  int ul = use_lut ? 1 : 0;
  int hbw = hls_body_width(w, hsv_round);
#define AL(CHX) UWIP_LAUNCH(ctx, "apply_lut_frame", apply_lut_frame_kernel<CHX>, grid, 256, 0, d_src, d_dst, w, h, d_lut, ul, bw, hbw)
  switch (channel) {
    case CH_B: AL(CH_B); break;
    case CH_G: AL(CH_G); break;
    case CH_R: AL(CH_R); break;
    case CH_H: AL(CH_H); break;
    case CH_S: AL(CH_S); break;
    case CH_V: AL(CH_V); break;
    case CH_Y: AL(CH_Y); break;
    case CH_CR: AL(CH_CR); break;
    case CH_CB: AL(CH_CB); break;
    case CH_HLS_H: AL(CH_HLS_H); break;
    case CH_HLS_L: AL(CH_HLS_L); break;
    case CH_HLS_S: AL(CH_HLS_S); break;
    case CH_LAB_L: AL(CH_LAB_L); break;
    case CH_LAB_A: AL(CH_LAB_A); break;
    case CH_LAB_B: AL(CH_LAB_B); break;
    default: uwip_set_err(ctx, "bad channel %d", channel); return UWIP_ERR_INVALID;
  }
#undef AL
  return UWIP_OK;
}

// ---- small utilities ----------------------------------------------------------------------------
__global__ void hist_to_float_kernel(const uint32_t* __restrict__ h, float* __restrict__ o, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = (float)h[i];
}
int k_hist_to_float(uwip_ctx* ctx, const uint32_t* d_hist, float* d_out, int n) {
  UWIP_LAUNCH(ctx, "hist_to_float", hist_to_float_kernel, cdiv(n, 256), 256, 0, d_hist, d_out, n);
  return UWIP_OK;
}

// entropy of 256-bin histograms.  flavour 0: aclaheEntropy (aclahe.cpp:228-248) - float p, double
// log2(p + 1e-5), product and accumulation in double stored back to a float accumulator each step
// (strictly sequential, so one thread replays it).  flavour 1: Entropia (functions.py:14-19) -
// float32 throughout, tree summation.
__global__ void __launch_bounds__(256) entropy_kernel(const uint32_t* __restrict__ hist, int w, int h, int flavour,
                                                      float* __restrict__ out) {
  __shared__ float s_v[256];
  int t = threadIdx.x;
  const uint32_t* hh = hist + (size_t)blockIdx.x * 256;
  if (flavour == 0) {
    if (t == 0) {
      float ent = 0.f;
      float n = (float)(w * h);
      for (int i = 0; i < 256; i++) {
        float p = __fdiv_rn((float)hh[i], n);
        double term = __dmul_rn((double)p, log2(__dadd_rn((double)p, 0.00001)));
        ent = (float)__dadd_rn((double)ent, term);
      }
      out[blockIdx.x] = -ent;
    }
    return;
  }
  // python flavour: hist / hist.sum() in float32 (sum of integer counts < 2^24 is exact)
  float tot = 0.f;
  s_v[t] = (float)hh[t];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (t < s) s_v[t] = __fadd_rn(s_v[t], s_v[t + s]);
    __syncthreads();
  }
  tot = s_v[0];
  __syncthreads();
  float p = __fdiv_rn((float)hh[t], tot);
  float lg = log2f(__fadd_rn(p, 0.00001f));
  s_v[t] = __fmul_rn(p, lg);
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (t < s) s_v[t] = __fadd_rn(s_v[t], s_v[t + s]);
    __syncthreads();
  }
  if (t == 0) out[blockIdx.x] = -s_v[0];
}
int k_entropy(uwip_ctx* ctx, const uint32_t* d_hist, int n_hists, int w, int h, int flavour, float* d_out) {
  UWIP_LAUNCH(ctx, "entropy", entropy_kernel, n_hists, 256, 0, d_hist, w, h, flavour, d_out);
  return UWIP_OK;
}

// GaussianBlur((3,3),0) on 8U: (sum [1 2 1]^T [1 2 1] p + 8) >> 4, reflect-101 border (ACLAHE.py:15); plane blockIdx.z
__global__ void blur3_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int w, int h) {
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  src += (size_t)blockIdx.z * w * h;
  dst += (size_t)blockIdx.z * w * h;
  auto rx = [&](int i) { return i < 0 ? -i : (i >= w ? 2 * w - 2 - i : i); };
  auto ry = [&](int i) { return i < 0 ? -i : (i >= h ? 2 * h - 2 - i : i); };
  int xs[3] = {w > 1 ? rx(x - 1) : 0, x, w > 1 ? rx(x + 1) : 0};
  int ys[3] = {h > 1 ? ry(y - 1) : 0, y, h > 1 ? ry(y + 1) : 0};
  const int k[3] = {1, 2, 1};
  int acc = 0;
#pragma unroll
  for (int j = 0; j < 3; j++)
#pragma unroll
    for (int i = 0; i < 3; i++) acc += k[j] * k[i] * src[(size_t)ys[j] * w + xs[i]];
  dst[(size_t)y * w + x] = (uint8_t)((acc + 8) >> 4);
}
int k_blur3(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int w, int h, int n) {
  dim3 block(32, 8), grid(cdiv(w, 32), cdiv(h, 8), n);
  UWIP_LAUNCH(ctx, "blur3", blur3_kernel, grid, block, 0, d_src, d_dst, w, h);
  return UWIP_OK;
}

// ---- the channel loop of the histretch CLI (histretch.cpp:219-254) on a batch of frames ----------
static int letter_channel(char c) {
  switch (c) {
    case 'R': return CH_B;  // numChannel('R') == 0 and plane 0 of an OpenCV image is BLUE
    case 'G': return CH_G;
    case 'B': return CH_R;  // numChannel('B') == 2 == red plane
    case 'H': return CH_H;
    case 'S': return CH_S;
    case 'V': return CH_V;
    case 'Y': return CH_Y;
    case 'C': return CH_CR;
    case 'X': return CH_CB;
    case 'h': return CH_HLS_H;
    case 's': return CH_HLS_L;  // numChannel('s') == 1 and plane 1 of BGR2HLS is L
    case 'l': return CH_HLS_S;  // numChannel('l') == 2 == the S plane
    case 'L': return CH_LAB_L;
    case 'a': return CH_LAB_A;
    case 'b': return CH_LAB_B;
  }
  return -1;
}

int histretch_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, const char* channels,
                         int lo, int hi, int order, int hsv_round) {
  size_t fbytes = (size_t)w * h * 3;
  uint32_t* d_hist = (uint32_t*)uwip_slot(ctx, SLOT_HIST, (size_t)n * 256 * 4);
  uint8_t* d_lut = (uint8_t*)uwip_slot(ctx, SLOT_LUT, (size_t)n * 256 * 4);
  if (!d_hist || !d_lut) return UWIP_ERR_NOMEM;
  const uint8_t* cur = d_src;
  bool any = false;
  for (const char* c = channels; *c; ++c) {
    int sp = uwip_num_space(*c);
    if (sp == -1) continue;  // "Option not recognized, skipping..."
    int ch = letter_channel(*c);
    bool literal_hsv = (sp != 0 && order == UWIP_ORDER_LITERAL);  // literal order: the frame becomes its colour-space round trip
    if (!literal_hsv) {
      UWIP_CHECK(k_histogram_frame(ctx, cur, n, w, h, ch, d_hist, hsv_round));
      UWIP_CHECK(k_percentile_lut(ctx, d_hist, n, w, h, lo, hi, nullptr, d_lut));
    }
    UWIP_CHECK(k_apply_lut_frame(ctx, cur, d_dst, n, w, h, ch, d_lut, !literal_hsv, hsv_round));
    cur = d_dst;
    any = true;
  }
  if (!any && d_src != d_dst) UWIP_CUDA(ctx, cudaMemcpyAsync(d_dst, d_src, fbytes * n, cudaMemcpyDeviceToDevice, ctx->stream));
  return UWIP_OK;
}
