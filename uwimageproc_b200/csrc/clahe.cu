// clahe.cu - cv::CLAHE::apply (8-bit) and the aclahe HSV frame wrapper for sm_100a.
//   reference call sites: modules/aclahe/src/aclahe.cpp:152-154 (BGR2HSV, split), :175-187 (apply),
//   modules/aclahe/python/functions.py:24-27, modules/aclahe/python/main.py:19-20.
//   The arithmetic itself is OpenCV's (not vendored in the reference); it is restated from SURVEY
//   appendix A.2 and pinned bit-exact against cv2 4.13.0 by tests/.
// Three passes: (1) per-tile histograms with per-warp privatised shared-memory atomics,
// (2) clip + redistribute + block prefix scan -> per-tile LUT, (3) bilinear blend of four tile LUTs,
// fused with the BGR<->HSV conversions (and, in the chain, with the histretch LUT in front and the
// dehaze min/max reduction behind).
#include <cuda_fp16.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

constexpr int TH_THREADS = 256;
constexpr int TH_WARPS = TH_THREADS / 32;

struct TileGeom {
  int W, H;      // image
  int EW, EH;    // extended (padded) size used for LUT building
  int tx, ty;    // grid
  int tw, th;    // tile size
};

__host__ __device__ static TileGeom make_geom(int W, int H, int tx, int ty) {
  TileGeom g;
  g.W = W; g.H = H; g.tx = tx; g.ty = ty;
  if (W % tx == 0 && H % ty == 0) {
    g.EW = W; g.EH = H;
  } else {  // OpenCV pads both dimensions (a full extra tile count when one of them divides evenly)
    g.EW = W + tx - W % tx;
    g.EH = H + ty - H % ty;
  }
  g.tw = g.EW / tx;
  g.th = g.EH / ty;
  return g;
}

// per-frame CLAHE parameters of the automatic path (grid, clip limit in counts, LUT scale), read by the PF instantiations
// of the three passes below: a CTA works on one frame, so its geometry stays uniform.  The workspaces of the PF passes
// hold `tpf` tiles per frame (the largest grid of the batch), CTAs beyond their frame's tile count exit.
struct FrameClahe {
  TileGeom g;
  int cl;
  float lut_scale;
};

__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
  return i;
}

// ---- pass 1: per-tile histograms ---------------------------------------------------------------
// FRAME=false: src is an 8U plane.  FRAME=true: src is bgr8 and the value is the HSV V channel
// (max(b,g,r)), optionally pushed through two 256-entry LUTs (trunc / rint flavour chosen by x) =
// the histretch stretch followed by the HSV->BGR->HSV round trip of its V channel.
template <bool FRAME, bool PF = false>
__global__ void __launch_bounds__(TH_THREADS) tilehist_kernel(const uint8_t* __restrict__ src, TileGeom g, int splits,
                                                              const uint8_t* __restrict__ prelut2 /*[n][2][256] or null*/,
                                                              int body_w, uint32_t* __restrict__ hist,
                                                              const FrameClahe* __restrict__ pf = nullptr, int tpf = 0) {
  __shared__ uint32_t sh[TH_WARPS][256];
  __shared__ uint8_t s_pre[2][256];
  int f = blockIdx.z;
  if (PF) {
    g = pf[f].g;
    if ((int)blockIdx.x >= g.tx * g.ty) return;
  }
  for (int i = threadIdx.x; i < TH_WARPS * 256; i += TH_THREADS) (&sh[0][0])[i] = 0;
  if (FRAME) {
    s_pre[0][threadIdx.x] = prelut2 ? prelut2[((size_t)f * 2 + 0) * 256 + threadIdx.x] : (uint8_t)threadIdx.x;
    s_pre[1][threadIdx.x] = prelut2 ? prelut2[((size_t)f * 2 + 1) * 256 + threadIdx.x] : (uint8_t)threadIdx.x;
  }
  __syncthreads();
  int tile = blockIdx.x;
  int tyi = tile / g.tx, txi = tile % g.tx;
  int rows_per = (g.th + splits - 1) / splits;
  int r0 = blockIdx.y * rows_per, r1 = min(r0 + rows_per, g.th);
  uint32_t* myh = sh[threadIdx.x >> 5];
  size_t n_px = (size_t)g.W * g.H;
  const uint8_t* base = src + (size_t)f * n_px * (FRAME ? 3 : 1);
  int x_begin = txi * g.tw, y_begin = tyi * g.th;
  bool vec = (g.EW == g.W) && (g.EH == g.H) && (g.tw % 16 == 0) && ((((uintptr_t)base) & 15) == 0);
  if (vec) {
    int gpr = g.tw / 16;  // 16-pixel groups per tile row
    int total = (r1 - r0) * gpr;
    for (int i = threadIdx.x; i < total; i += TH_THREADS) {
      int ry = i / gpr, gx = i - ry * gpr;
      int y = y_begin + r0 + ry, x = x_begin + gx * 16;
      if (FRAME) {
        const uint4* q = reinterpret_cast<const uint4*>(base + ((size_t)y * g.W + x) * 3);
        uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
        uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
#pragma unroll
        for (int k = 0; k < 16; k++) {
          int i0 = 3 * k, i1 = 3 * k + 1, i2 = 3 * k + 2;
          int bb = (w[i0 >> 2] >> ((i0 & 3) * 8)) & 0xff;
          int gg = (w[i1 >> 2] >> ((i1 & 3) * 8)) & 0xff;
          int rr = (w[i2 >> 2] >> ((i2 & 3) * 8)) & 0xff;
          int v = imax3(bb, gg, rr);
          v = s_pre[(x + k) < body_w ? 0 : 1][v];
          atomicAdd(&myh[v], 1u);
        }
      } else {
        uint4 a = __ldg(reinterpret_cast<const uint4*>(base + (size_t)y * g.W + x));
        uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
          atomicAdd(&myh[w[k] & 0xff], 1u);
          atomicAdd(&myh[(w[k] >> 8) & 0xff], 1u);
          atomicAdd(&myh[(w[k] >> 16) & 0xff], 1u);
          atomicAdd(&myh[w[k] >> 24], 1u);
        }
      }
    }
  } else {
    int total = (r1 - r0) * g.tw;
    for (int i = threadIdx.x; i < total; i += TH_THREADS) {
      int ry = i / g.tw, rx = i - ry * g.tw;
      int y = reflect101(y_begin + r0 + ry, g.H), x = reflect101(x_begin + rx, g.W);
      int v;
      if (FRAME) {
        const uint8_t* p = base + ((size_t)y * g.W + x) * 3;
        v = imax3(p[0], p[1], p[2]);
        v = s_pre[x < body_w ? 0 : 1][v];
      } else {
        v = base[(size_t)y * g.W + x];
      }
      atomicAdd(&myh[v], 1u);
    }
  }
  __syncthreads();
  uint32_t s = 0;
#pragma unroll
  for (int w = 0; w < TH_WARPS; w++) s += sh[w][threadIdx.x];
  if (s) atomicAdd(&hist[((PF ? (size_t)f * tpf : (size_t)f * g.tx * g.ty) + tile) * 256 + threadIdx.x], s);
}

// ---- pass 2: clip, redistribute, scan, LUT -------------------------------------------------------
__device__ __forceinline__ uint32_t block_incl_scan_256(uint32_t v, uint32_t* s_warp, uint32_t& total) {
  int t = threadIdx.x;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
    if ((t & 31) >= d) incl += o;
  }
  __syncthreads();  // protect s_warp reuse
  if ((t & 31) == 31) s_warp[t >> 5] = incl;
  __syncthreads();
  uint32_t base = 0;
  total = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint32_t x = s_warp[k];
    if (k < (t >> 5)) base += x;
    total += x;
  }
  return incl + base;
}

// one block per (tile, frame); `cl` = clip limit in counts (0: no clipping); n_cl > 1 builds LUTs for
// several clip limits at once (entropy sweep): lut layout [frame][tile][icl][256]
// PF: one clip limit per frame from pf[frame] (n_cl = 1), `tpf` tiles per frame of which the frame's grid uses the first
template <bool PF = false>
__global__ void __launch_bounds__(256) clahe_lut_kernel(const uint32_t* __restrict__ hist, const int* __restrict__ cls, int n_cl,
                                                        float lut_scale, uint8_t* __restrict__ lut,
                                                        const FrameClahe* __restrict__ pf = nullptr, int tpf = 0) {
  __shared__ uint32_t s_warp[8];
  int t = threadIdx.x;
  size_t tile = blockIdx.x;
  if (PF) {
    const FrameClahe& q = pf[blockIdx.x / tpf];
    if ((int)(blockIdx.x % tpf) >= q.g.tx * q.g.ty) return;
    lut_scale = q.lut_scale;
  }
  uint32_t h0 = hist[tile * 256 + t];
  for (int ic = 0; ic < n_cl; ic++) {
    int cl = PF ? pf[blockIdx.x / tpf].cl : cls[ic];
    uint32_t h = h0;
    if (cl > 0) {
      uint32_t excess = h > (uint32_t)cl ? h - cl : 0, clipped;
      block_incl_scan_256(excess, s_warp, clipped);
      h = min(h, (uint32_t)cl);
      uint32_t batch = clipped / 256, resid = clipped - batch * 256;
      h += batch;
      if (resid) {
        uint32_t step = max(256u / resid, 1u);
        if (t % step == 0 && t / step < resid) h++;
      }
    }
    uint32_t tot;
    uint32_t cum = block_incl_scan_256(h, s_warp, tot);
    lut[(tile * n_cl + ic) * 256 + t] = (uint8_t)sat_rint_u8(__fmul_rn((float)cum, lut_scale));
  }
}

// ---- pass 3: bilinear LUT interpolation ---------------------------------------------------------
struct Interp {
  int t1, t2;
  float a, a1;
};
__device__ __forceinline__ Interp interp_coord(int x, float inv_t, int ntile) {
  float f = __fsub_rn(__fmul_rn((float)x, inv_t), 0.5f);
  int t1 = (int)floorf(f);
  Interp r;
  r.a = __fsub_rn(f, (float)t1);
  r.a1 = __fsub_rn(1.0f, r.a);
  r.t2 = min(t1 + 1, ntile - 1);
  r.t1 = max(t1, 0);
  return r;
}
__device__ __forceinline__ int clahe_blend(float l11, float l12, float l21, float l22, const Interp& ix, const Interp& iy) {
  float top = __fadd_rn(__fmul_rn(l11, ix.a1), __fmul_rn(l12, ix.a));
  float bot = __fadd_rn(__fmul_rn(l21, ix.a1), __fmul_rn(l22, ix.a));
  float res = __fadd_rn(__fmul_rn(top, iy.a1), __fmul_rn(bot, iy.a));
  return __float_as_int(__fadd_rn(res, 8388608.0f)) & 0xff;   // rint of a blend of four bytes: in [0, 255], see ap_to_byte
}

// ---- colour arithmetic of the apply kernel: the same values as hsv2bgr_u8 / bgr2hsv_u8 (common.cuh), fewer instructions ----
// Float -> byte: the products below lie in [0, 256), so adding 2^23 leaves rint(x) (round to nearest even, as cvt.rni) or
// floor(x) (add rounding toward zero, as cvt.rzi on a non-negative value) in the low mantissa bits: one FADD instead of a
// conversion and two clamps.  The results keep the bit pattern of 2^23 as a common bias (AP_BIAS + k): maxima, minima and
// differences do not care, the byte is picked by PRMT when the words are packed.
constexpr int AP_BIAS = 0x4B000000;
__device__ __forceinline__ int ap_to_byte(float x, bool trunc_mode) {
  return __float_as_int(trunc_mode ? __fadd_rz(x, 8388608.0f) : __fadd_rn(x, 8388608.0f));
}
// sector table of cvtColor(HSV2BGR) as weights: channel = v * (1 - s * w), w = A + B * f with (A, B) = (0,0) for tab[0] = v,
// (1,0) for tab[1] = v(1-s), (0,1) for tab[2] = v(1-s f), (1,-1) for tab[3] = v(1-s(1-f)).  fma(B, f, A) and fma(-s, w, 1) round
// exactly like the subtractions of the scalar code (each is one rounding of the same real number), and the six-way
// branch on the sector disappears.  Row = sector, columns A_b B_b A_g B_g A_r B_r - -.
__device__ __forceinline__ void ap_fill_sector_table(float* tab /*[6][8]*/, int t) {
  if (t < 48) {
    const int sec = t >> 3, col = t & 7;
    // (b, g, r) <- tab index: {1,3,0},{1,0,2},{3,0,1},{0,2,1},{0,1,3},{2,1,0}
    // two bits per channel (b g r), six bits per sector
    const unsigned long long codes = 0x1cull | (0x12ull << 6) | (0x31ull << 12) | (0x09ull << 18) | (0x07ull << 24) | (0x24ull << 30);
    float val = 0.0f;
    if (col < 6) {
      const int k = (int)(codes >> (6 * sec + 2 * (2 - (col >> 1)))) & 3;
      const float A = (k == 1 || k == 3) ? 1.0f : 0.0f, B = (k == 2) ? 1.0f : (k == 3 ? -1.0f : 0.0f);
      val = (col & 1) ? B : A;
    }
    tab[t] = val;
  }
}
// H in [0, 180) (always true for the output of bgr2hsv), S, V bytes -> b, g, r carrying AP_BIAS
__device__ __forceinline__ void ap_hsv2bgr(int H, int S, int V, bool trunc_mode, const float* __restrict__ tab, int& b, int& g, int& r) {
  const float h = __fmul_rn((float)H, 6.0f / 180.0f);
  const float s = __fmul_rn((float)S, 1.0f / 255.0f);
  const float v = __fmul_rn((float)V, 1.0f / 255.0f);
  const float hz = __fadd_rz(h, 8388608.0f);            // 2^23 + floor(h)
  const float f = __fsub_rn(h, __fsub_rn(hz, 8388608.0f));
  const int sec = __float_as_int(hz) & 7;               // 0 .. 5
  const float4 w4 = *reinterpret_cast<const float4*>(tab + 8 * sec);
  const float2 w2 = *reinterpret_cast<const float2*>(tab + 8 * sec + 4);
  const float fb = __fmul_rn(v, __fmaf_rn(-s, __fmaf_rn(w4.y, f, w4.x), 1.0f));
  const float fg = __fmul_rn(v, __fmaf_rn(-s, __fmaf_rn(w4.w, f, w4.z), 1.0f));
  const float fr = __fmul_rn(v, __fmaf_rn(-s, __fmaf_rn(w2.y, f, w2.x), 1.0f));
  b = ap_to_byte(__fmul_rn(fb, 255.0f), trunc_mode);
  g = ap_to_byte(__fmul_rn(fg, 255.0f), trunc_mode);
  r = ap_to_byte(__fmul_rn(fr, 255.0f), trunc_mode);
}
// bgr2hsv_u8 on values that share an additive bias (0 or AP_BIAS); h, s, v come out plain
__device__ __forceinline__ void ap_bgr2hsv(int b, int g, int r, const int* __restrict__ sdiv, const int* __restrict__ hdiv, int& h, int& s, int& v) {
  const int vm = imax3(b, g, r);
  const int d = vm - imin3(b, g, r);
  v = vm & 0xff;
  s = (d * sdiv[v] + (1 << 11)) >> 12;
  const int h0 = (vm == r) ? (g - b) : ((vm == g) ? (b - r + 2 * d) : (r - g + 4 * d));
  h = (h0 * hdiv[d] + (1 << 11)) >> 12;
  if (h < 0) h += 180;
}
__device__ __forceinline__ uint32_t ap_pack4(int a, int b, int c, int d) {   // low bytes of four values
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

constexpr int AP_THREADS = 256;

// Processes `rows_per` image rows per block.  MODE 0: plane in / plane out.  MODE 1: bgr8 frame:
// [PRE: stretch LUT on V + HSV->BGR->HSV round trip] -> CLAHE on V -> HSV->BGR, and optional
// joint min/max of the output bytes into FrameState (dehaze D0, bgdehaze/main.py:17).
// A thread owns groups of four columns: the x interpolation of the four is formed once and reused down the band's rows,
// and the loop body is four pixels long (the former sixteen-pixel body was 60 KB of code: a third of the warp stalls
// were instruction fetches).
constexpr int AP_ROWS = 8;   // rows whose y interpolation is tabulated per block
template <int MODE, bool PRE, bool PF = false>
__global__ void __launch_bounds__(AP_THREADS) clahe_apply_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                                 TileGeom gp, int rows_per, const uint8_t* __restrict__ lut,
                                                                 const uint8_t* __restrict__ prelut /*[n][256], PRE only*/,
                                                                 int body_w, FrameState* fs,
                                                                 const FrameClahe* __restrict__ pf = nullptr, int tpf = 0) {
  extern __shared__ uint8_t s_lut[];  // [3][tx][256] when it fits
  __shared__ uint8_t s_pre[256];
  __shared__ int s_sdiv[256], s_hdiv[256];
  __shared__ Interp s_iy[AP_ROWS];
  __shared__ __align__(16) float s_sec[48];
  int f = blockIdx.y;
  const TileGeom g = PF ? pf[f].g : gp;
  int y0 = blockIdx.x * rows_per, y1 = min(y0 + rows_per, g.H);
  float inv_tw = __fdiv_rn(1.0f, (float)g.tw), inv_th = __fdiv_rn(1.0f, (float)g.th);
  const uint8_t* flut = lut + (PF ? (size_t)f * tpf : (size_t)f * g.tx * g.ty) * 256;
  // tile rows needed by this band
  int ty_lo = interp_coord(y0, inv_th, g.ty).t1;
  int ty_hi = interp_coord(y1 - 1, inv_th, g.ty).t2;
  bool staged = (ty_hi - ty_lo + 1) <= 3 && g.tx <= 32;
  if (staged) {
    int nbytes = (ty_hi - ty_lo + 1) * g.tx * 256;
    const uint32_t* s4 = reinterpret_cast<const uint32_t*>(flut + (size_t)ty_lo * g.tx * 256);
    for (int i = threadIdx.x; i < nbytes / 4; i += AP_THREADS) reinterpret_cast<uint32_t*>(s_lut)[i] = __ldg(s4 + i);
  }
  if (MODE == 1) {
    s_pre[threadIdx.x] = PRE ? prelut[(size_t)f * 256 + threadIdx.x] : (uint8_t)threadIdx.x;
    s_sdiv[threadIdx.x] = hsv_sdiv(threadIdx.x);
    s_hdiv[threadIdx.x] = hsv_hdiv(threadIdx.x);
    ap_fill_sector_table(s_sec, threadIdx.x);
  }
  if (threadIdx.x < AP_ROWS && y0 + (int)threadIdx.x < y1) s_iy[threadIdx.x] = interp_coord(y0 + threadIdx.x, inv_th, g.ty);
  __syncthreads();
  const uint8_t* L = staged ? s_lut : flut;
  int ty_off = staged ? ty_lo : 0;
  size_t n_px = (size_t)g.W * g.H;
  const uint8_t* in = src + (size_t)f * n_px * (MODE ? 3 : 1);
  uint8_t* out = dst + (size_t)f * n_px * (MODE ? 3 : 1);
  int mn = AP_BIAS + 255, mx = AP_BIAS;   // of the biased output bytes

  auto lookup = [&](int v, const Interp& ix, const Interp& iy) {
    const uint8_t* r1 = L + (size_t)(iy.t1 - ty_off) * g.tx * 256;
    const uint8_t* r2 = L + (size_t)(iy.t2 - ty_off) * g.tx * 256;
    float l11 = (float)r1[ix.t1 * 256 + v], l12 = (float)r1[ix.t2 * 256 + v];
    float l21 = (float)r2[ix.t1 * 256 + v], l22 = (float)r2[ix.t2 * 256 + v];
    return clahe_blend(l11, l12, l21, l22, ix, iy);
  };
  auto do_pixel = [&](int& b, int& gg, int& r, bool tr, const Interp& ix, const Interp& iy) {
    int h, s, v;
    if (PRE) {  // histretch on V (intended order) fused in front, incl. its colour round trip
      ap_bgr2hsv(b, gg, r, s_sdiv, s_hdiv, h, s, v);
      ap_hsv2bgr(h, s, s_pre[v], tr, s_sec, b, gg, r);
    }
    ap_bgr2hsv(b, gg, r, s_sdiv, s_hdiv, h, s, v);
    v = lookup(v, ix, iy);
    ap_hsv2bgr(h, s, v, tr, s_sec, b, gg, r);   // b, gg, r carry AP_BIAS from here on
    mn = min(mn, imin3(b, gg, r));
    mx = max(mx, imax3(b, gg, r));
  };

  const bool vec = (g.W % 4 == 0) && (((((uintptr_t)in) | ((uintptr_t)out)) & 3) == 0) && (body_w % 4 == 0);
  if (vec) {
    const int gpr = g.W / 4, wpr = MODE ? 3 * gpr : gpr;   // column groups, words per row
    for (int gx = threadIdx.x; gx < gpr; gx += AP_THREADS) {
      const int x = 4 * gx;
      const bool tr = x < body_w;
      Interp ix[4];
#pragma unroll
      for (int k = 0; k < 4; k++) ix[k] = interp_coord(x + k, inv_tw, g.tx);
      const uint32_t* q = reinterpret_cast<const uint32_t*>(in) + (size_t)y0 * wpr + (MODE ? 3 * gx : gx);
      uint32_t* o = reinterpret_cast<uint32_t*>(out) + (size_t)y0 * wpr + (MODE ? 3 * gx : gx);
      uint32_t n0 = __ldg(q), n1 = MODE ? __ldg(q + 1) : 0u, n2 = MODE ? __ldg(q + 2) : 0u;
#pragma unroll 1
      for (int y = y0; y < y1; y++) {
        const uint32_t w0 = n0, w1 = n1, w2 = n2;
        if (y + 1 < y1) {   // the next row's words are on their way while this row is worked on
          q += wpr;
          n0 = __ldg(q);
          if (MODE) { n1 = __ldg(q + 1); n2 = __ldg(q + 2); }
        }
        const Interp iy = (y - y0 < AP_ROWS) ? s_iy[y - y0] : interp_coord(y, inv_th, g.ty);
        if (MODE == 0) {
          const int v0 = lookup(w0 & 0xff, ix[0], iy), v1 = lookup((w0 >> 8) & 0xff, ix[1], iy);
          const int v2 = lookup((w0 >> 16) & 0xff, ix[2], iy), v3 = lookup(w0 >> 24, ix[3], iy);
          o[0] = (uint32_t)v0 | ((uint32_t)v1 << 8) | ((uint32_t)v2 << 16) | ((uint32_t)v3 << 24);
        } else {
          int b0 = w0 & 0xff, g0 = (w0 >> 8) & 0xff, r0 = (w0 >> 16) & 0xff, b1 = w0 >> 24;
          int g1 = w1 & 0xff, r1 = (w1 >> 8) & 0xff, b2 = (w1 >> 16) & 0xff, g2 = w1 >> 24;
          int r2 = w2 & 0xff, b3 = (w2 >> 8) & 0xff, g3 = (w2 >> 16) & 0xff, r3 = w2 >> 24;
          do_pixel(b0, g0, r0, tr, ix[0], iy);
          do_pixel(b1, g1, r1, tr, ix[1], iy);
          do_pixel(b2, g2, r2, tr, ix[2], iy);
          do_pixel(b3, g3, r3, tr, ix[3], iy);
          o[0] = ap_pack4(b0, g0, r0, b1);
          o[1] = ap_pack4(g1, r1, b2, g2);
          o[2] = ap_pack4(r2, b3, g3, r3);
        }
        o += wpr;
      }
    }
  } else {
    int total = (y1 - y0) * g.W;
    for (int i = threadIdx.x; i < total; i += AP_THREADS) {
      int ry = i / g.W, x = i - ry * g.W;
      int y = y0 + ry;
      Interp iy = interp_coord(y, inv_th, g.ty);
      Interp ix = interp_coord(x, inv_tw, g.tx);
      if (MODE == 0) {
        out[(size_t)y * g.W + x] = (uint8_t)lookup(in[(size_t)y * g.W + x], ix, iy);
      } else {
        const uint8_t* p = in + ((size_t)y * g.W + x) * 3;
        int b = p[0], gg = p[1], r = p[2];
        do_pixel(b, gg, r, x < body_w, ix, iy);
        uint8_t* o = out + ((size_t)y * g.W + x) * 3;
        o[0] = (uint8_t)b; o[1] = (uint8_t)gg; o[2] = (uint8_t)r;
      }
    }
  }
  if (MODE == 1 && fs) {
    const unsigned umn = warp_reduce_min_u32((unsigned)(mn & 0xff)), umx = warp_reduce_max_u32((unsigned)(mx & 0xff));
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&fs[f].kmin, umn);
      atomicMax(&fs[f].kmax, umx);
    }
  }
}

// composite LUTs for pass 1 of the fused histretch->aclahe head: V after stretch and after the
// HSV->BGR->HSV round trip, for the truncating body and the rounding tail of a row.
__global__ void prelut2_kernel(const uint8_t* __restrict__ lut1, uint8_t* __restrict__ lut2) {
  int f = blockIdx.x, t = threadIdx.x;
  int v = lut1[(size_t)f * 256 + t];
  lut2[((size_t)f * 2 + 0) * 256 + t] = (uint8_t)hsv_roundtrip_v(v, true);
  lut2[((size_t)f * 2 + 1) * 256 + t] = (uint8_t)hsv_roundtrip_v(v, false);
}

// ---- host-side drivers (device pointers) ----------------------------------------------------------
static int body_width(int w, int hsv_round) {
  if (hsv_round == UWIP_HSV_ROUND_TRUNC) return w;
  if (hsv_round == UWIP_HSV_ROUND_RINT) return 0;
  return 32 * (w / 32);
}

static int clip_count(double clip, int area) {
  if (!(clip > 0)) return 0;
  int cl = (int)(clip * area / 256.0);
  return cl < 1 ? 1 : cl;
}

static int pick_splits(uwip_ctx* ctx, const TileGeom& g, int n) {
  int tiles = g.tx * g.ty * n;
  int want = ctx->sm_count * 4;  // ~4 blocks per SM
  int s = (want + tiles - 1) / tiles;
  int max_s = (g.th + 7) / 8;
  if (s > max_s) s = max_s;
  return s < 1 ? 1 : s;
}

static int clahe_common(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty,
                        bool frame, int hsv_round, const uint8_t* d_prelut, FrameState* fs) {
  UWIP_REQUIRE(ctx, tx >= 1 && ty >= 1 && tx <= 256 && ty <= 256, "tile grid out of range");
  UWIP_REQUIRE(ctx, w >= 1 && h >= 1 && n >= 1, "bad size");
  TileGeom g = make_geom(w, h, tx, ty);
  UWIP_REQUIRE(ctx, (g.EW == w || 2 * w - 2 >= g.EW - 1 || w == 1) && (g.EH == h || 2 * h - 2 >= g.EH - 1 || h == 1),
               "image too small for this tile grid (reflect-101 padding undefined)");
  size_t ntile = (size_t)n * tx * ty;
  uint32_t* d_th = (uint32_t*)uwip_slot(ctx, SLOT_TILEHIST, ntile * 256 * 4);
  uint8_t* d_tl = (uint8_t*)uwip_slot(ctx, SLOT_TILELUT, ntile * 256 + 16);
  int* d_cl = (int*)uwip_slot(ctx, SLOT_MISC, 256);
  if (!d_th || !d_tl || !d_cl) return UWIP_ERR_NOMEM;
  uint8_t* d_pre2 = nullptr;
  int bw = body_width(w, hsv_round);
  if (d_prelut) {
    d_pre2 = (uint8_t*)uwip_slot(ctx, SLOT_LUT, (size_t)n * 256 * 4) + (size_t)n * 256;  // second half of the LUT slot
    UWIP_LAUNCH(ctx, "prelut2", prelut2_kernel, n, 256, 0, d_prelut, d_pre2);
  }
  UWIP_CUDA(ctx, cudaMemsetAsync(d_th, 0, ntile * 256 * 4, ctx->stream));
  int splits = pick_splits(ctx, g, n);
  dim3 grid1(tx * ty, splits, n);
  if (frame)
    UWIP_LAUNCH(ctx, "clahe_tilehist", tilehist_kernel<true>, grid1, TH_THREADS, 0, d_src, g, splits, d_pre2, bw, d_th);
  else
    UWIP_LAUNCH(ctx, "clahe_tilehist", tilehist_kernel<false>, grid1, TH_THREADS, 0, d_src, g, splits, (const uint8_t*)nullptr, bw, d_th);
  int cl = clip_count(clip, g.tw * g.th);
  UWIP_CUDA(ctx, cudaMemcpyAsync(d_cl, &cl, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  float lut_scale = 255.0f / (float)(g.tw * g.th);
  UWIP_LAUNCH(ctx, "clahe_lut", clahe_lut_kernel<false>, (unsigned)ntile, 256, 0, d_th, d_cl, 1, lut_scale, d_tl);
  int rows_per = 8;
  while (rows_per > 1 && (long long)cdiv(h, rows_per) * n < (long long)ctx->sm_count * 4) rows_per /= 2;
  dim3 grid3(cdiv(h, rows_per), n);
  size_t smem = (size_t)3 * (tx <= 32 ? tx : 0) * 256;
  if (frame && d_prelut)
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<1, true>), grid3, AP_THREADS, smem, d_src, d_dst, g, rows_per, d_tl, d_prelut, bw, fs);
  else if (frame)
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<1, false>), grid3, AP_THREADS, smem, d_src, d_dst, g, rows_per, d_tl, d_prelut, bw, fs);
  else
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<0, false>), grid3, AP_THREADS, smem, d_src, d_dst, g, rows_per, d_tl,
                (const uint8_t*)nullptr, bw, (FrameState*)nullptr);
  return UWIP_OK;
}

int clahe_planes_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty) {
  return clahe_common(ctx, d_src, d_dst, n, w, h, clip, tx, ty, false, 0, nullptr, nullptr);
}

int aclahe_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, double clip, int tx, int ty,
                      int hsv_round, const uint8_t* d_prelut, FrameState* fs) {
  return clahe_common(ctx, d_src, d_dst, n, w, h, clip, tx, ty, true, hsv_round, d_prelut, fs);
}

// ---- entropy sweep over clip limits (SURVEY 8f N1: aclahe.cpp:160-193, ACLAHE.py:20-47) ---------------------
// Tile histograms do not depend on the clip limit: build them once per grid, derive one LUT set per clip limit, then ONE
// pixel pass per grid accumulates the histogram of every CLAHE output without writing images.
//
// The pixel pass works per INTERPOLATION CELL: all pixels whose four neighbouring tiles are the same (t1x, t2x, t1y, t2y).
// A CTA owns a band of rows of one cell of one frame: the LUT sets of the four tiles for every clip limit are staged in
// shared memory as uchar4 (l11, l12, l21, l22) per (clip, value) - 4 x 51 x 256 B = 52 KB, the figure of SURVEY 8f - so
// one 32-bit shared load feeds a blend; the output histograms of the band ([n_cl][256] u32, another 52 KB) are
// accumulated in shared memory and flushed once.  Pixels come in as 32-bit words (4 per load).
constexpr int SW_MAX_CL = 64;
constexpr int SW_THREADS = 256;
__global__ void __launch_bounds__(SW_THREADS, 2) sweep_cell_kernel(const uint8_t* __restrict__ src, TileGeom g, int band_rows, int bands,
                                                                   const uint8_t* __restrict__ lut /*[frame][tile][n_cl][256]*/, int n_cl,
                                                                   uint32_t* __restrict__ out_hist /*[frame][n_cl][256]*/) {
  extern __shared__ __align__(16) uint32_t s_sw[];
  uint32_t* s_lut = s_sw;                 // [n_cl][256] packed (l11, l12, l21, l22)
  uint32_t* s_hist = s_sw + n_cl * 256;   // [n_cl][256]
  const int f = blockIdx.z;
  const int cell = blockIdx.x / bands, band = blockIdx.x - cell * bands;
  const int cx = cell % (g.tx + 1), cy = cell / (g.tx + 1);   // cell index = floor(coordinate / tile - 0.5) + 1
  const int t1x = max(cx - 1, 0), t2x = min(cx, g.tx - 1), t1y = max(cy - 1, 0), t2y = min(cy, g.ty - 1);
  const uint8_t* flut = lut + (size_t)f * g.tx * g.ty * n_cl * 256;
  const uint8_t* L11 = flut + (size_t)(t1y * g.tx + t1x) * n_cl * 256;
  const uint8_t* L12 = flut + (size_t)(t1y * g.tx + t2x) * n_cl * 256;
  const uint8_t* L21 = flut + (size_t)(t2y * g.tx + t1x) * n_cl * 256;
  const uint8_t* L22 = flut + (size_t)(t2y * g.tx + t2x) * n_cl * 256;
  for (int i = threadIdx.x; i < n_cl * 256; i += SW_THREADS) {
    s_lut[i] = (uint32_t)__ldg(L11 + i) | ((uint32_t)__ldg(L12 + i) << 8) | ((uint32_t)__ldg(L21 + i) << 16) | ((uint32_t)__ldg(L22 + i) << 24);
    s_hist[i] = 0;
  }
  __syncthreads();
  const float inv_tw = __fdiv_rn(1.0f, (float)g.tw), inv_th = __fdiv_rn(1.0f, (float)g.th);
  // the rectangle that surely contains the cell (two pixels of slack: the cell edges are decided by the float32 expression of
  // interp_coord, every pixel re-derives its cell and the CTA keeps only its own)
  // cell c covers the coordinates with floor(x / tile - 0.5) == c - 1, i.e. [(c - 0.5) tile, (c + 0.5) tile)
  const int xa = max(cx * g.tw - (g.tw + 1) / 2 - 2, 0) & ~3, xb = min(cx * g.tw + (g.tw + 1) / 2 + 2, g.W);
  const int ya0 = max(cy * g.th - (g.th + 1) / 2 - 2, 0), yb0 = min(cy * g.th + (g.th + 1) / 2 + 2, g.H);
  const int ya = ya0 + band * band_rows, yb = min(ya + band_rows, yb0);
  const uint8_t* img = src + (size_t)f * g.W * g.H;
  const int nwords = (xb - xa + 3) >> 2;
  const bool aligned = ((g.W & 3) == 0) && ((reinterpret_cast<uintptr_t>(img) & 3) == 0);
  if (xa < xb && ya < yb) {
    const int total = (yb - ya) * nwords;
    for (int i = threadIdx.x; i < total; i += SW_THREADS) {
      const int ry = i / nwords, wx = i - ry * nwords;
      const int y = ya + ry, x0 = xa + 4 * wx;
      const float fy = __fsub_rn(__fmul_rn((float)y, inv_th), 0.5f);
      const int ky = (int)floorf(fy);
      if (ky + 1 != cy) continue;
      const float ay = __fsub_rn(fy, (float)ky), ay1 = __fsub_rn(1.0f, ay);
      uint32_t w4;
      if (aligned && x0 + 3 < g.W) w4 = __ldg(reinterpret_cast<const uint32_t*>(img + (size_t)y * g.W + x0));
      else {
        w4 = 0;
        for (int k = 0; k < 4; k++) if (x0 + k < g.W) w4 |= (uint32_t)img[(size_t)y * g.W + x0 + k] << (8 * k);
      }
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int x = x0 + k;
        if (x >= xb) break;
        const float fx = __fsub_rn(__fmul_rn((float)x, inv_tw), 0.5f);
        const int kx = (int)floorf(fx);
        if (kx + 1 != cx) continue;
        const float ax = __fsub_rn(fx, (float)kx), ax1 = __fsub_rn(1.0f, ax);
        const uint32_t v = (w4 >> (8 * k)) & 255u;
        const uint32_t* lp = s_lut + v;
        uint32_t* hp = s_hist;
#pragma unroll 4
        for (int c = 0; c < n_cl; c++) {
          const uint32_t l = lp[c * 256];
          const float top = __fadd_rn(__fmul_rn((float)(l & 255u), ax1), __fmul_rn((float)((l >> 8) & 255u), ax));
          const float bot = __fadd_rn(__fmul_rn((float)((l >> 16) & 255u), ax1), __fmul_rn((float)(l >> 24), ax));
          const float res = __fadd_rn(__fmul_rn(top, ay1), __fmul_rn(bot, ay));
          const int o = min(max(__float2int_rn(res), 0), 255);   // the blend of four bytes is finite: sat_rint_u8 without its NaN test
          atomicAdd(hp + c * 256 + o, 1u);
        }
      }
    }
  }
  __syncthreads();
  uint32_t* oh = out_hist + (size_t)f * n_cl * 256;
  for (int i = threadIdx.x; i < n_cl * 256; i += SW_THREADS)
    if (s_hist[i]) atomicAdd(&oh[i], s_hist[i]);
}

static int check_sweep_size(uwip_ctx* ctx, int w, int h, const int* grids, int n_grids) {
  for (int gi = 0; gi < n_grids; gi++) {
    UWIP_REQUIRE(ctx, grids[gi] >= 1 && grids[gi] <= 256, "tile grid out of range");
    TileGeom g = make_geom(w, h, grids[gi], grids[gi]);
    UWIP_REQUIRE(ctx, (g.EW == w || 2 * w - 2 >= g.EW - 1) && (g.EH == h || 2 * h - 2 >= g.EH - 1), "image too small for grid");
  }
  return UWIP_OK;
}

// n planes x n_grids square grids x n_clips clip limits -> entropies on the device, layout [grid][frame][clip]; the
// pointer is workspace of the context (valid until the next sweep)
static int clahe_entropy_sweep_core(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, const int* grids, int n_grids,
                                    const double* clips, int n_clips, int flavour, float** d_ent_out) {
  UWIP_REQUIRE(ctx, n >= 1 && w >= 1 && h >= 1, "bad size");
  UWIP_REQUIRE(ctx, n_clips >= 1 && n_clips <= SW_MAX_CL, "1..64 clip limits per sweep");
  UWIP_REQUIRE(ctx, n_grids >= 1 && n_grids <= 16, "1..16 grids per sweep");
  UWIP_CHECK(check_sweep_size(ctx, w, h, grids, n_grids));
  size_t max_tiles = 0;
  for (int gi = 0; gi < n_grids; gi++) max_tiles = std::max(max_tiles, (size_t)grids[gi] * grids[gi]);
  uint32_t* d_th = (uint32_t*)uwip_slot(ctx, SLOT_TILEHIST, (size_t)n * max_tiles * 256 * 4);
  uint8_t* d_tl = (uint8_t*)uwip_slot(ctx, SLOT_TILELUT, (size_t)n * max_tiles * 256 * n_clips + 16);
  const size_t hist_bytes = (size_t)n * n_grids * n_clips * 256 * 4, ent_bytes = (size_t)n * n_grids * n_clips * 4;
  char* d_sw = (char*)uwip_slot(ctx, SLOT_SWEEP, 4096 + hist_bytes + ent_bytes);
  if (!d_th || !d_tl || !d_sw) return UWIP_ERR_NOMEM;
  int* d_cl_all = (int*)d_sw;   // [n_grids][n_clips] clip limits in counts
  uint32_t* d_oh = (uint32_t*)(d_sw + 4096);
  float* d_ent = (float*)(d_sw + 4096 + hist_bytes);
  std::vector<int> cls((size_t)n_grids * n_clips);
  for (int gi = 0; gi < n_grids; gi++) {
    TileGeom g = make_geom(w, h, grids[gi], grids[gi]);
    for (int i = 0; i < n_clips; i++) cls[(size_t)gi * n_clips + i] = clip_count(clips[i], g.tw * g.th);
  }
  UWIP_CUDA(ctx, cudaMemcpyAsync(d_cl_all, cls.data(), sizeof(int) * cls.size(), cudaMemcpyHostToDevice, ctx->stream));
  UWIP_CUDA(ctx, cudaMemsetAsync(d_oh, 0, hist_bytes, ctx->stream));
  const size_t smem = (size_t)n_clips * 256 * 8;
  UWIP_CUDA(ctx, uwip_func_smem(ctx, FUNC_SWEEP, sweep_cell_kernel, smem));
  for (int gi = 0; gi < n_grids; gi++) {
    const int tiles = grids[gi];
    TileGeom g = make_geom(w, h, tiles, tiles);
    const size_t ntile = (size_t)tiles * tiles;
    const int* d_cl = d_cl_all + (size_t)gi * n_clips;
    UWIP_CUDA(ctx, cudaMemsetAsync(d_th, 0, (size_t)n * ntile * 256 * 4, ctx->stream));
    int splits = pick_splits(ctx, g, n);
    dim3 grid1(tiles * tiles, splits, n);
    UWIP_LAUNCH(ctx, "clahe_tilehist", tilehist_kernel<false>, grid1, TH_THREADS, 0, d_planes, g, splits, (const uint8_t*)nullptr, 0, d_th);
    float lut_scale = 255.0f / (float)(g.tw * g.th);
    UWIP_LAUNCH(ctx, "clahe_lut", clahe_lut_kernel<false>, (unsigned)(ntile * n), 256, 0, d_th, d_cl, n_clips, lut_scale, d_tl);
    // bands of rows per cell: enough CTAs to fill the machine, at least 8 rows each
    const int cells = (tiles + 1) * (tiles + 1);
    const int cell_rows = g.th + 6;
    int bands = std::max(1, std::min(cdiv(ctx->sm_count * 4, cells * n), cdiv(cell_rows, 8)));
    const int band_rows = cdiv(cell_rows, bands);
    bands = cdiv(cell_rows, band_rows);
    dim3 grid3(cells * bands, 1, n);
    // device layout of the histograms and entropies: [grid][frame][clip]
    uint32_t* d_oh_g = d_oh + (size_t)gi * n * n_clips * 256;
    UWIP_LAUNCH(ctx, "clahe_sweep_hist", sweep_cell_kernel, grid3, SW_THREADS, smem, d_planes, g, band_rows, bands, d_tl, n_clips, d_oh_g);
  }
  UWIP_CHECK(k_entropy(ctx, d_oh, n * n_grids * n_clips, w, h, flavour, d_ent));
  *d_ent_out = d_ent;
  return UWIP_OK;
}

// n planes x n_grids square grids x n_clips clip limits -> entropies [n][n_grids][n_clips] (host pointer)
int clahe_entropy_sweep_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, const int* grids, int n_grids,
                                  const double* clips, int n_clips, int flavour, float* entropies_host) {
  float* d_ent = nullptr;
  UWIP_CHECK(clahe_entropy_sweep_core(ctx, d_planes, n, w, h, grids, n_grids, clips, n_clips, flavour, &d_ent));
  const size_t ent_bytes = (size_t)n * n_grids * n_clips * 4;
  std::vector<float> tmp((size_t)n * n_grids * n_clips);
  UWIP_CUDA(ctx, cudaMemcpyAsync(tmp.data(), d_ent, ent_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  UWIP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  // device layout [grid][frame][clip] -> caller layout [frame][grid][clip]
  for (int f = 0; f < n; f++)
    for (int gi = 0; gi < n_grids; gi++)
      memcpy(entropies_host + ((size_t)f * n_grids + gi) * n_clips, tmp.data() + ((size_t)gi * n + f) * n_clips, sizeof(float) * n_clips);
  return UWIP_OK;
}

int clahe_entropy_sweep_dev(uwip_ctx* ctx, const uint8_t* d_plane, int w, int h, int tiles, const double* clips, int n_clips,
                            int flavour, float* entropies_host) {
  return clahe_entropy_sweep_batch_dev(ctx, d_plane, 1, w, h, &tiles, 1, clips, n_clips, flavour, entropies_host);
}

// ---- automatic CLAHE parameters (ParametrosACLAHE, ACLAHE.py:9-129; SURVEY 8f N1) and CLAHE with per-frame parameters ----
static const int AUTO_GRIDS[5] = {2, 4, 8, 16, 32};   // ACLAHE.py:21
constexpr int AUTO_NCL = 50;                          // np.arange(0, 25, 0.5)
constexpr int AUTO_TPF = 32 * 32;                     // tiles per frame of the PF workspaces: the largest automatic grid

__device__ __forceinline__ int clip_count_dev(double clip, int area) {   // clip_count on the device
  if (!(clip > 0)) return 0;
  int cl = (int)(clip * area / 256.0);
  return cl < 1 ? 1 : cl;
}

// V plane of n bgr8 frames, optionally through the fused histretch head's two LUTs (the V of the intermediate frame)
__global__ void vplane_kernel(const uint8_t* __restrict__ src, int w, int h, const uint8_t* __restrict__ prelut2, int body_w,
                              uint8_t* __restrict__ dst) {
  const int f = blockIdx.y;
  const size_t n_px = (size_t)w * h;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += (size_t)gridDim.x * blockDim.x) {
    const uint8_t* p = src + (f * n_px + i) * 3;
    int v = imax3(p[0], p[1], p[2]);
    if (prelut2) v = prelut2[((size_t)f * 2 + ((int)(i % w) < body_w ? 0 : 1)) * 256 + v];
    dst[f * n_px + i] = (uint8_t)v;
  }
}

// the CLAHE parameters of grid `grid` at each frame's own clip limit (the block-size pick, ACLAHE.py:102-113)
__global__ void pick_params_kernel(const int* __restrict__ cl, int n, TileGeom g, FrameClahe* __restrict__ pf) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  FrameClahe q;
  q.g = g;
  q.cl = clip_count_dev((double)max(cl[f], 0), g.tw * g.th);
  q.lut_scale = 255.0f / (float)(g.tw * g.th);
  pf[f] = q;
}

// BS = the grid whose entropy, rounded to float16, is the last maximum (ACLAHE.py:102, 117-121); -1 with CL for a frame
// whose fit failed
__global__ void pick_bs_kernel(const float* __restrict__ ent /*[5][n]*/, int n, const int* __restrict__ cl, int* __restrict__ bs) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  int w = 0;
  float best = 0.f;
  for (int m = 0; m < 5; m++) {
    const float e = __half2float(__float2half_rn(ent[(size_t)m * n + f]));
    if (m == 0 || e >= best) { best = e; w = m; }
  }
  const int grids[5] = {2, 4, 8, 16, 32};
  bs[f] = cl[f] < 0 ? -1 : grids[w];
}

// per-frame parameters of the CLAHE apply: (BS, CL) or, for a frame whose fit failed, the caller's fixed ones
__global__ void auto_geom_kernel(const int* __restrict__ bs, const int* __restrict__ cl, int n, int w, int h, FrameClahe fallback,
                                 FrameClahe* __restrict__ pf) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  FrameClahe q = fallback;
  if (cl[f] >= 0) {
    q.g = make_geom(w, h, bs[f], bs[f]);
    q.cl = clip_count_dev((double)cl[f], q.g.tw * q.g.th);
    q.lut_scale = 255.0f / (float)(q.g.tw * q.g.th);
  }
  pf[f] = q;
}

__global__ void nofit_flags_kernel(const int* __restrict__ cl, int n, int32_t* __restrict__ flags, int keep) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  flags[f] = (keep ? flags[f] : 0) | (cl[f] < 0 ? UWIP_FRAME_ACLAHE_NOFIT : 0);
}

int aclahe_nofit_flags(uwip_ctx* ctx, const int* d_cl, int n, int32_t* d_flags, bool keep) {
  UWIP_LAUNCH(ctx, "aclahe_flags", nofit_flags_kernel, cdiv(n, 128), 128, 0, d_cl, n, d_flags, keep ? 1 : 0);
  return UWIP_OK;
}

int aclahe_check_auto_size(uwip_ctx* ctx, int w, int h) { return check_sweep_size(ctx, w, h, AUTO_GRIDS, 5); }

// ParametrosACLAHE on n equal-size planes: blur -> sweep (5 grids x 50 clip limits) -> knee per grid -> CL = max of the knees
// -> entropy of CLAHE(blurred, k, CL) per grid -> BS.  loop = 0 repaired, 1 as committed (CL = 0, ACLAHE.py:40-47 as it
// stands).  Stream ordered; d_bs, d_cl are device int32[n].
int aclahe_params_planes_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, int loop, int* d_bs, int* d_cl) {
  UWIP_REQUIRE(ctx, n >= 1 && w >= 1 && h >= 1, "bad size");
  UWIP_REQUIRE(ctx, loop == UWIP_ACLAHE_LOOP_REPAIRED || loop == UWIP_ACLAHE_LOOP_AS_COMMITTED, "bad loop");
  UWIP_CHECK(aclahe_check_auto_size(ctx, w, h));
  const size_t n_px = (size_t)w * h;
  uint8_t* d_blur = (uint8_t*)uwip_slot(ctx, SLOT_ABLUR, (size_t)n * n_px);
  const size_t pf_bytes = align_up(sizeof(FrameClahe) * 5 * n, 256), ent_bytes = align_up(sizeof(float) * 5 * n, 256);
  const size_t hist_bytes = (size_t)5 * n * 256 * 4;
  char* d_ws = (char*)uwip_slot(ctx, SLOT_AUTO, 256 * 8 + pf_bytes + ent_bytes + hist_bytes);
  if (!d_blur || !d_ws) return UWIP_ERR_NOMEM;
  double* d_xd = (double*)d_ws;                                 // derivatives of the clip curve [2][49]
  FrameClahe* d_pf = (FrameClahe*)(d_ws + 256 * 8);             // [5][n]
  float* d_pent = (float*)(d_ws + 256 * 8 + pf_bytes);          // [5][n]
  uint32_t* d_ph = (uint32_t*)(d_ws + 256 * 8 + pf_bytes + ent_bytes);   // [5][n][256]
  UWIP_CHECK(k_blur3(ctx, d_planes, d_blur, w, h, n));
  if (loop == UWIP_ACLAHE_LOOP_REPAIRED) {
    double clips[AUTO_NCL];
    for (int i = 0; i < AUTO_NCL; i++) clips[i] = 0.5 * i;
    float* d_ent = nullptr;
    UWIP_CHECK(clahe_entropy_sweep_core(ctx, d_blur, n, w, h, AUTO_GRIDS, 5, clips, AUTO_NCL, 1, &d_ent));
    UWIP_CHECK(k_aclahe_knees(ctx, d_ent, n, AUTO_NCL, d_xd, d_cl));
  } else {
    UWIP_CUDA(ctx, cudaMemsetAsync(d_cl, 0, sizeof(int) * n, ctx->stream));
  }
  // block size: the tile-histogram, LUT and sweep passes with one clip limit per frame
  uint32_t* d_th = (uint32_t*)uwip_slot(ctx, SLOT_TILEHIST, (size_t)n * AUTO_TPF * 256 * 4);
  uint8_t* d_tl = (uint8_t*)uwip_slot(ctx, SLOT_TILELUT, (size_t)n * AUTO_TPF * 256 + 16);
  if (!d_th || !d_tl) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemsetAsync(d_ph, 0, hist_bytes, ctx->stream));
  const size_t smem = (size_t)256 * 8;
  for (int gi = 0; gi < 5; gi++) {
    const int tiles = AUTO_GRIDS[gi];
    const TileGeom g = make_geom(w, h, tiles, tiles);
    const int ntile = tiles * tiles;
    FrameClahe* pf = d_pf + (size_t)gi * n;
    UWIP_LAUNCH(ctx, "aclahe_pick_params", pick_params_kernel, cdiv(n, 128), 128, 0, d_cl, n, g, pf);
    UWIP_CUDA(ctx, cudaMemsetAsync(d_th, 0, (size_t)n * ntile * 256 * 4, ctx->stream));
    const int splits = pick_splits(ctx, g, n);
    UWIP_LAUNCH(ctx, "clahe_tilehist", tilehist_kernel<false>, dim3(ntile, splits, n), TH_THREADS, 0, d_blur, g, splits,
                (const uint8_t*)nullptr, 0, d_th);
    UWIP_LAUNCH(ctx, "clahe_lut", clahe_lut_kernel<true>, (unsigned)(ntile * n), 256, 0, d_th, (const int*)nullptr, 1, 0.f, d_tl,
                (const FrameClahe*)pf, ntile);
    const int cells = (tiles + 1) * (tiles + 1), cell_rows = g.th + 6;
    int bands = std::max(1, std::min(cdiv(ctx->sm_count * 4, cells * n), cdiv(cell_rows, 8)));
    const int band_rows = cdiv(cell_rows, bands);
    bands = cdiv(cell_rows, band_rows);
    UWIP_LAUNCH(ctx, "clahe_sweep_hist", sweep_cell_kernel, dim3(cells * bands, 1, n), SW_THREADS, smem, d_blur, g, band_rows, bands,
                d_tl, 1, d_ph + (size_t)gi * n * 256);
  }
  UWIP_CHECK(k_entropy(ctx, d_ph, 5 * n, w, h, 1, d_pent));
  UWIP_LAUNCH(ctx, "aclahe_pick_bs", pick_bs_kernel, cdiv(n, 128), 128, 0, d_pent, n, d_cl, d_bs);
  return UWIP_OK;
}

// the refusals of the automatic calls: the fallback grid must suit the image and the image the five automatic grids
static int aclahe_auto_check(uwip_ctx* ctx, int n, int w, int h, int tx, int ty) {
  UWIP_REQUIRE(ctx, tx >= 1 && ty >= 1 && tx <= 256 && ty <= 256, "tile grid out of range");
  UWIP_REQUIRE(ctx, w >= 1 && h >= 1 && n >= 1, "bad size");
  const TileGeom gf = make_geom(w, h, tx, ty);
  UWIP_REQUIRE(ctx, (gf.EW == w || 2 * w - 2 >= gf.EW - 1 || w == 1) && (gf.EH == h || 2 * h - 2 >= gf.EH - 1 || h == 1),
               "image too small for this tile grid (reflect-101 padding undefined)");
  return aclahe_check_auto_size(ctx, w, h);
}

// The parameter search on the n planes d_search, then CLAHE of d_src into d_dst with each frame's own (BS, CL); frames
// whose fit fails (CL = -1) get the fixed clip / tx x ty.  FRAME: bgr8 frames, CLAHE on the V of HSV (optionally behind
// the fused histretch head: d_pre2, d_prelut, bw) with the dehaze min / max into fs; otherwise u8 planes.
template <bool FRAME>
static int aclahe_auto_core(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, const uint8_t* d_search, int n, int w, int h, int loop,
                            double clip, int tx, int ty, const uint8_t* d_pre2, const uint8_t* d_prelut, int bw, FrameState* fs,
                            int* d_bs, int* d_cl) {
  UWIP_CHECK(aclahe_params_planes_dev(ctx, d_search, n, w, h, loop, d_bs, d_cl));
  // per-frame geometry in the PF workspace: tpf tiles per frame
  const TileGeom gf = make_geom(w, h, tx, ty);
  const int tpf = std::max(AUTO_TPF, tx * ty);
  char* d_ws = (char*)uwip_slot(ctx, SLOT_AUTO, 0);   // the params call sized it: [2][49] doubles, then FrameClahe[5][n]
  FrameClahe* d_pf = (FrameClahe*)(d_ws + 256 * 8);   // reuses the pick's [0][n] block, consumed by then in stream order
  FrameClahe fb;
  fb.g = gf;
  fb.cl = clip_count(clip, gf.tw * gf.th);
  fb.lut_scale = 255.0f / (float)(gf.tw * gf.th);
  UWIP_LAUNCH(ctx, "aclahe_geom", auto_geom_kernel, cdiv(n, 128), 128, 0, d_bs, d_cl, n, w, h, fb, d_pf);
  uint32_t* d_th = (uint32_t*)uwip_slot(ctx, SLOT_TILEHIST, (size_t)n * tpf * 256 * 4);
  uint8_t* d_tl = (uint8_t*)uwip_slot(ctx, SLOT_TILELUT, (size_t)n * tpf * 256 + 16);
  if (!d_th || !d_tl) return UWIP_ERR_NOMEM;
  UWIP_CUDA(ctx, cudaMemsetAsync(d_th, 0, (size_t)n * tpf * 256 * 4, ctx->stream));
  // row splits sized for the coarsest grid (2 x 2: the tallest tiles); finer grids leave the upper splits idle
  const int splits = pick_splits(ctx, make_geom(w, h, 2, 2), n);
  UWIP_LAUNCH(ctx, "clahe_tilehist", (tilehist_kernel<FRAME, true>), dim3(tpf, splits, n), TH_THREADS, 0, d_src, gf, splits,
              d_pre2, bw, d_th, (const FrameClahe*)d_pf, tpf);
  UWIP_LAUNCH(ctx, "clahe_lut", clahe_lut_kernel<true>, (unsigned)((size_t)tpf * n), 256, 0, d_th, (const int*)nullptr, 1, 0.f, d_tl,
              (const FrameClahe*)d_pf, tpf);
  int rows_per = 8;
  while (rows_per > 1 && (long long)cdiv(h, rows_per) * n < (long long)ctx->sm_count * 4) rows_per /= 2;
  dim3 grid3(cdiv(h, rows_per), n);
  const size_t smem = (size_t)3 * 32 * 256;   // staged LUT rows of grids up to 32 tiles wide
  if (!FRAME)
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<0, false, true>), grid3, AP_THREADS, smem, d_src, d_dst, gf, rows_per, d_tl,
                d_prelut, bw, fs, (const FrameClahe*)d_pf, tpf);
  else if (d_prelut)
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<1, true, true>), grid3, AP_THREADS, smem, d_src, d_dst, gf, rows_per, d_tl, d_prelut,
                bw, fs, (const FrameClahe*)d_pf, tpf);
  else
    UWIP_LAUNCH(ctx, "clahe_apply", (clahe_apply_kernel<1, false, true>), grid3, AP_THREADS, smem, d_src, d_dst, gf, rows_per, d_tl,
                d_prelut, bw, fs, (const FrameClahe*)d_pf, tpf);
  return UWIP_OK;
}

// BGR->HSV, CLAHE on V with each frame's own (BS, CL), HSV->BGR on n frames (optionally behind the fused histretch head and
// with the dehaze min / max, like aclahe_frames_dev).  The parameters are found on the V plane of the frame that enters CLAHE;
// frames whose fit fails (CL = -1) get the fixed clip / tx x ty.
int aclahe_frames_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, double clip, int tx, int ty,
                           int hsv_round, const uint8_t* d_prelut, FrameState* fs, int* d_bs, int* d_cl) {
  UWIP_CHECK(aclahe_auto_check(ctx, n, w, h, tx, ty));
  const size_t n_px = (size_t)w * h;
  const int bw = body_width(w, hsv_round);
  uint8_t* d_v = (uint8_t*)uwip_slot(ctx, SLOT_APLANE, (size_t)n * n_px);
  if (!d_v) return UWIP_ERR_NOMEM;
  uint8_t* d_pre2 = nullptr;
  if (d_prelut) {
    d_pre2 = (uint8_t*)uwip_slot(ctx, SLOT_LUT, (size_t)n * 256 * 4) + (size_t)n * 256;  // second half of the LUT slot
    if (!d_pre2) return UWIP_ERR_NOMEM;
    UWIP_LAUNCH(ctx, "prelut2", prelut2_kernel, n, 256, 0, d_prelut, d_pre2);
  }
  UWIP_LAUNCH(ctx, "aclahe_vplane", vplane_kernel, dim3(std::max(1, std::min(cdiv((int)std::min<size_t>(n_px, 1 << 30), 256), 1024)), n), 256, 0,
              d_src, w, h, (const uint8_t*)d_pre2, bw, d_v);
  return aclahe_auto_core<true>(ctx, d_src, d_dst, d_v, n, w, h, loop, clip, tx, ty, d_pre2, d_prelut, bw, fs, d_bs, d_cl);
}

// main.py:18-20 on n u8 planes: the parameters of each plane (found on its blurred copy, ACLAHE.py:15), then CLAHE of the
// unblurred plane with them; planes whose fit fails get the fixed clip / tx x ty.
int aclahe_planes_auto_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int w, int h, int loop, double clip, int tx, int ty,
                           int* d_bs, int* d_cl) {
  UWIP_CHECK(aclahe_auto_check(ctx, n, w, h, tx, ty));
  return aclahe_auto_core<false>(ctx, d_src, d_dst, d_src, n, w, h, loop, clip, tx, ty, nullptr, nullptr, 0, nullptr, d_bs, d_cl);
}
