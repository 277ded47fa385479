// dehaze.cu - bgdehaze (Li et al. ICASSP-16 blue-green dehazing + red-channel correction + adaptive
// exposure map) for sm_100a.
//   reference: modules/bgdehaze/BGDehaze.py:14-89, modules/bgdehaze/guidedfilter.py:23-103,
//              modules/bgdehaze/main.py:16-19.  Stage names D0..D10 follow SURVEY.md 8a.
//
// Data flow per frame (all frame-global reductions land in FrameState, no host round trips):
//   minmax (D0)  ->  window: 15x15 window max / arg-min partials (D1), window min (D2), and the packed
//                    plane kq = (k'_b, k'_g, k'_r, m'_b) + plane m'_g that every later pass reads
//   -> GF1a: box sums of 17 moments + per-pixel 3x3 solve -> a,b planes (int32 fixed point x8)
//   -> GF1b: box(a,b) -> refined t (D3,D5) -> J (D6) + min/max/sum reductions -> J planes (f32 x2)
//   -> E: restored -> R8/I8 -> YCrCb joint min/max (D7,D8 first half); packed plane ycc = (Yi,Cri,Cbi,Yj)
//   -> S table (256x256 u32 per frame: the exposure ratio is a function of two bytes; rint(S 2^28)) -> S plane (u32)
//   -> GF2a: S + 13 moments + solve -> a,b (int32 fixed point x4)   -> GF2b: box(a,b) -> refined S, exposure min/max
//   -> final: normalise, x255, rint, saturate -> bgr8 (D8 second half, D10)
//
// The four GF passes are the guided-filter marches of gfpipe.cuh: per strip of columns, ACC threads keep the vertical
// running sums of a quad of columns, AUX warps form the prefixes over the strip, SOLVE threads take the window sums of two
// pixels and do the per-pixel work.  The solve works in "k units" (guide not divided by range) with eps_k = eps*range^2 on
// the exact integer numerators N*S_ij - S_i*S_j.  Details and measurements: DESIGN.md section 3.
#include <algorithm>

#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// frame state
// ------------------------------------------------------------------------------------------------
__global__ void fs_reset_kernel(FrameState* fs, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  FrameState s;
  memset(&s, 0, sizeof(s));
  s.kmin = 255; s.kmax = 0;
  s.jmin_key[0] = s.jmin_key[1] = ~0ull;
  s.jmax_key[0] = s.jmax_key[1] = 0ull;
  s.rmin = 255; s.rmax = 0;
  s.yi_min = s.yj_min = 255; s.yi_max = s.yj_max = 0;
  s.omin_key = ~0ull; s.omax_key = 0ull;
  fs[i] = s;
}
int frame_state_reset(uwip_ctx* ctx, FrameState* fs, int n) {
  UWIP_LAUNCH(ctx, "fs_reset", fs_reset_kernel, cdiv(n, 128), 128, 0, fs, n);
  return UWIP_OK;
}
FrameState* frame_state_get(uwip_ctx* ctx, int n) { return (FrameState*)uwip_slot(ctx, SLOT_FSTATE, sizeof(FrameState) * (size_t)n); }

#include "gfmarch.cuh"

int dehaze_gf1a_launch(uwip_ctx* ctx, const GfCommon& gc, int n, int W, int H, int r);   // dehaze_gf1a.cu (narrow strips)
int dehaze_gf1a_strips(int w);                                                               // strips of a frame in that layout

// ------------------------------------------------------------------------------------------------
// D0: joint min / max over all channels (bgdehaze/main.py:17)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) minmax_kernel(const uint8_t* __restrict__ src, size_t n_bytes, FrameState* fs) {
  const uint8_t* p = src + (size_t)blockIdx.y * n_bytes;
  unsigned int mn = 0x00ff00ffu, mx = 0;
  bool vec = ((((uintptr_t)p) & 15) == 0);
  size_t n16 = vec ? n_bytes / 16 : 0;
  for (size_t g = (size_t)blockIdx.x * 256 + threadIdx.x; g < n16; g += (size_t)gridDim.x * 256) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + g);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      unsigned int e = w[k] & 0x00ff00ffu, o = (w[k] >> 8) & 0x00ff00ffu;
      mn = __vminu2(mn, __vminu2(e, o));
      mx = __vmaxu2(mx, __vmaxu2(e, o));
    }
  }
  unsigned int smn = min(mn & 0xffffu, mn >> 16), smx = max(mx & 0xffffu, mx >> 16);
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * 256 + threadIdx.x; i < n_bytes; i += (size_t)gridDim.x * 256) {
    smn = min(smn, (unsigned)p[i]);
    smx = max(smx, (unsigned)p[i]);
  }
  smn = warp_reduce_min_u32(smn);
  smx = warp_reduce_max_u32(smx);
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&fs[blockIdx.y].kmin, smn);
    atomicMax(&fs[blockIdx.y].kmax, smx);
  }
}

// ------------------------------------------------------------------------------------------------
// D1 / D2: 15x15 window max (3 channels) -> arg-min partials; window min (blue, green); packed planes
// ------------------------------------------------------------------------------------------------
constexpr int WK_TX = 64, WK_TY = 32, WK_THREADS = 256;
constexpr int WK_MAXWIN = 33;
constexpr int WK_TWIN = 15;  // transmission window: always 15 (BGDehaze.py:52 drops w)

struct ArgPartial {
  double d0, d1;
  unsigned int i0, i1;
};

__device__ __forceinline__ bool lex_less(double a, unsigned ia, double b, unsigned ib) { return (a < b) || (a == b && ia < ib); }

// kq[y][x] = k'_b | k'_g<<8 | k'_r<<16 | m'_b<<24,  mg[y][x] = m'_g   (pitch Wp, pad columns zero)
//   k' = k - kmin (bgdehaze/main.py:17 numerator), m' = window min - kmin, 0 where the zero padding of
//   transmission_map (BGDehaze.py:32) reaches into the window.
__global__ void __launch_bounds__(WK_THREADS) window_kernel(const uint8_t* __restrict__ src, int W, int H, int Wp, int wmax,
                                                            const FrameState* __restrict__ fs, uint32_t* __restrict__ kq,
                                                            uint8_t* __restrict__ mgp, ArgPartial* __restrict__ partials) {
  extern __shared__ uint32_t s_w[];
  __shared__ double s_nrm[256];
  __shared__ ArgPartial s_part[WK_THREADS / 32];
  const int wmin = WK_TWIN;
  const int pmax = wmax / 2, pmin = wmin / 2;
  const int PL = max(pmax, pmin), PR = max(wmax - 1 - pmax, wmin - 1 - pmin);
  const int RW = WK_TX + PL + PR, RH = WK_TY + PL + PR;
  uint32_t* P0 = s_w;                 // (B | G<<16) of the input region, replicate border
  uint32_t* P1 = P0 + RW * RH;        // R
  uint32_t* HX0 = P1 + RW * RH;       // horizontal max (B,G)   [RH][WK_TX]
  uint32_t* HX1 = HX0 + RH * WK_TX;   // horizontal max R
  uint32_t* HN0 = HX1 + RH * WK_TX;   // horizontal min (B,G)
  int f = blockIdx.z;
  const uint8_t* img = src + (size_t)f * W * H * 3;
  int x0 = blockIdx.x * WK_TX, y0 = blockIdx.y * WK_TY;
  int kmin = fs[f].kmin, range = (int)fs[f].kmax - kmin;
  s_nrm[threadIdx.x] = (double)threadIdx.x / (double)range;  // normI value of k' (main.py:17)
  for (int i = threadIdx.x; i < RW * RH; i += WK_THREADS) {
    int ry = i / RW, rx = i - ry * RW;
    int y = min(max(y0 - PL + ry, 0), H - 1), x = min(max(x0 - PL + rx, 0), W - 1);
    const uint8_t* p = img + ((size_t)y * W + x) * 3;
    P0[i] = (uint32_t)p[0] | ((uint32_t)p[1] << 16);
    P1[i] = p[2];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < RH * WK_TX; i += WK_THREADS) {
    int ry = i / WK_TX, x = i - ry * WK_TX;
    const uint32_t* r0 = P0 + ry * RW + x + PL;
    const uint32_t* r1 = P1 + ry * RW + x + PL;
    uint32_t m0 = 0, m1 = 0, n0 = 0xffffffffu;
    for (int k = -pmax; k < wmax - pmax; k++) {
      m0 = __vmaxu2(m0, r0[k]);
      m1 = max(m1, r1[k]);
    }
    for (int k = -pmin; k < wmin - pmin; k++) n0 = __vminu2(n0, r0[k]);
    HX0[i] = m0; HX1[i] = m1; HN0[i] = n0;
  }
  __syncthreads();
  int x = threadIdx.x % WK_TX, rg = threadIdx.x / WK_TX;
  double bd0 = 0, bd1 = 0;
  unsigned bi0 = 0xffffffffu, bi1 = 0xffffffffu;
  bool have = false;
  int gx = x0 + x;
  uint32_t* kqf = kq + (size_t)f * Wp * H;
  uint8_t* mgf = mgp + (size_t)f * Wp * H;
  for (int j = 0; j < WK_TY / (WK_THREADS / WK_TX); j++) {
    int yy = rg * (WK_TY / (WK_THREADS / WK_TX)) + j;
    int gy = y0 + yy;
    if (gx >= Wp || gy >= H) continue;
    size_t ppix = (size_t)gy * Wp + gx;
    if (gx >= W) { kqf[ppix] = 0u; mgf[ppix] = 0; continue; }
    uint32_t m0 = 0, m1 = 0, n0 = 0xffffffffu;
    for (int k = -pmax; k < wmax - pmax; k++) {
      m0 = __vmaxu2(m0, HX0[(yy + PL + k) * WK_TX + x]);
      m1 = max(m1, HX1[(yy + PL + k) * WK_TX + x]);
    }
    for (int k = -pmin; k < wmin - pmin; k++) n0 = __vminu2(n0, HN0[(yy + PL + k) * WK_TX + x]);
    const int pw = WK_TWIN / 2;
    bool touches = (gx < pw) || (gy < pw) || (gx - pw + WK_TWIN - 1 >= W) || (gy - pw + WK_TWIN - 1 >= H);
    uint32_t c0 = P0[(yy + PL) * RW + x + PL], c1 = P1[(yy + PL) * RW + x + PL];
    uint32_t mb = touches ? 0u : (n0 & 0xffffu) - (uint32_t)kmin;
    uint32_t mg = touches ? 0u : (n0 >> 16) - (uint32_t)kmin;
    kqf[ppix] = ((c0 & 0xffffu) - kmin) | (((c0 >> 16) - kmin) << 8) | ((c1 - kmin) << 16) | (mb << 24);
    mgf[ppix] = (uint8_t)mg;
    // D (BGDehaze.py:20-21): max_R - max_B, max_R - max_G on the normalised image, in fp64
    double nr = s_nrm[(int)m1 - kmin];
    double d0 = nr - s_nrm[(int)(m0 & 0xffffu) - kmin];
    double d1 = nr - s_nrm[(int)(m0 >> 16) - kmin];
    unsigned idx = (unsigned)((size_t)gy * W + gx);
    if (!have) { bd0 = d0; bd1 = d1; bi0 = bi1 = idx; have = true; }
    else {
      if (d0 < bd0) { bd0 = d0; bi0 = idx; }
      if (d1 < bd1) { bd1 = d1; bi1 = idx; }
    }
  }
  // block reduction, lexicographic (value, flat index): first index of the minimum
  if (!have) { bd0 = bd1 = __longlong_as_double(0x7ff0000000000000ll); }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    double o0 = __shfl_xor_sync(0xffffffffu, bd0, d), o1 = __shfl_xor_sync(0xffffffffu, bd1, d);
    unsigned j0 = __shfl_xor_sync(0xffffffffu, bi0, d), j1 = __shfl_xor_sync(0xffffffffu, bi1, d);
    if (lex_less(o0, j0, bd0, bi0)) { bd0 = o0; bi0 = j0; }
    if (lex_less(o1, j1, bd1, bi1)) { bd1 = o1; bi1 = j1; }
  }
  if ((threadIdx.x & 31) == 0) { ArgPartial a; a.d0 = bd0; a.d1 = bd1; a.i0 = bi0; a.i1 = bi1; s_part[threadIdx.x >> 5] = a; }
  __syncthreads();
  if (threadIdx.x == 0) {
    ArgPartial a = s_part[0];
    for (int k = 1; k < WK_THREADS / 32; k++) {
      ArgPartial b = s_part[k];
      if (lex_less(b.d0, b.i0, a.d0, a.i0)) { a.d0 = b.d0; a.i0 = b.i0; }
      if (lex_less(b.d1, b.i1, a.d1, a.i1)) { a.d1 = b.d1; a.i1 = b.i1; }
    }
    partials[(size_t)f * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x] = a;
  }
}

// ---- fast path: both windows 15x15 (the reference's only reachable configuration unless -w is given) ----
// Tile 64 x 32 outputs, 256 threads, three CTAs per SM.  The window max / min of a run of outputs is formed in registers on
// 16-bit pairs with the three-input VIMNMX3.U16x2:  m3[i] = op(p[i], p[i+1], p[i+2]),  m9[i] = op(m3[i], m3[i+3], m3[i+6]),
// m15[i] = op(m9[i], m9[i+6])  - 3 + 18/N instructions per output of a run of N instead of 14.
// The arg-min of D is found in two steps: every pixel only feeds the packed integer differences (max_R - max_B,
// max_R - max_G; two instructions), and the fp64 value of BGDehaze.py:20-21 is evaluated for the pixels that reach the
// tile's integer minimum (one unit of the integer difference is 1/range, the fp64 rounding is far below that, so the fp64
// minimum is always among them).
constexpr int WF_TX = 64, WF_TY = 32, WF_R = 7, WF_RH = WF_TY + 2 * WF_R;   // region rows
constexpr int WF_VR = WF_TY / 4, WF_CTAS = 3;  // output rows per vertical run (four runs of 64 columns); CTAs per SM
constexpr int WF_RB = 8;    // region column c is image column x0 - WF_RB + c (80 columns: the 240 bytes of a row start on a word)
constexpr int WF_PP = 84;   // region pitch in words: 80 used; 21 x 16 bytes (odd) -> conflict-free 16-byte loads down a column of rows
constexpr int WF_HP = 68;   // pitch of the horizontal results: 17 x 16 bytes
constexpr int WF_HN = 16;   // outputs per horizontal task

template <int N, bool MAX, int OFF, int M>
__device__ __forceinline__ void win15(const uint32_t (&p)[M], uint32_t (&o)[N]) {
  static_assert(OFF + N + 14 <= M, "window run");
  uint32_t a[N + 12], b[N + 6];
#pragma unroll
  for (int i = 0; i < N + 12; i++)
    a[i] = MAX ? __vimax3_u16x2(p[OFF + i], p[OFF + i + 1], p[OFF + i + 2]) : __vimin3_u16x2(p[OFF + i], p[OFF + i + 1], p[OFF + i + 2]);
#pragma unroll
  for (int i = 0; i < N + 6; i++) b[i] = MAX ? __vimax3_u16x2(a[i], a[i + 3], a[i + 6]) : __vimin3_u16x2(a[i], a[i + 3], a[i + 6]);
#pragma unroll
  for (int i = 0; i < N; i++) o[i] = MAX ? __vmaxu2(b[i], b[i + 6]) : __vminu2(b[i], b[i + 6]);
}

__device__ __forceinline__ void wf_cp_async8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}

// rows of one vertical run: packs (B', G', R', min_B') and min_G' of every pixel (main.py:17's k' = k - kmin) and returns the
// packed minimum of the biased integer differences (low half max_R - max_B + 256, high half max_R - max_G + 256).
// FAST: all WF_VR rows lie inside the image and no window touches the border
template <bool FAST>
__device__ __forceinline__ uint32_t wf_emit_rows(const uint32_t (&mx0)[WF_VR], const uint32_t (&mx1)[WF_VR], const uint32_t (&mn0)[WF_VR],
                                                 const uint32_t* __restrict__ pc0, const uint32_t* __restrict__ pc1,
                                                 uint32_t* __restrict__ kqp, uint8_t* __restrict__ mgq, unsigned Wp, int nrows, int gy0, int H,
                                                 bool xt, bool inside, uint32_t km2) {
  uint32_t dmin2 = 0xffffffffu;
#pragma unroll
  for (int i = 0; i < WF_VR; i++) {
    if (!FAST && i >= nrows) break;
    const unsigned o = (unsigned)i * Wp;
    if (!FAST && !inside) { kqp[o] = 0u; mgq[o] = 0; continue; }
    const uint32_t t0 = pc0[i * WF_PP] - km2, t1 = pc1[i * WF_PP] - km2;   // (B', G'), (R', R')
    uint32_t tn = mn0[i] - km2;                                            // (min_B', min_G')
    if (!FAST) {
      const int gy = gy0 + i;
      if (xt || gy < WF_R || gy + WF_R >= H) tn = 0u;                       // the reference's min filter pads with 0 (BGDehaze.py:32)
    }
    kqp[o] = __byte_perm(__byte_perm(t0, t1, 0x4420), tn, 0x4210);          // B' | G' << 8 | R' << 16 | min_B' << 24
    mgq[o] = (uint8_t)(tn >> 16);
    dmin2 = __vminu2(dmin2, mx1[i] + 0x01000100u - mx0[i]);                 // D (BGDehaze.py:20-21) in units of 1/range
  }
  return dmin2;
}

// exact D of the pixels of a run whose integer difference is the tile's minimum: first index of the smallest fp64 value
template <int CH>
__device__ __forceinline__ void wf_exact(const uint32_t (&mx0)[WF_VR], const uint32_t (&mx1)[WF_VR], int nrows, uint32_t target, int kmin,
                                         const double* s_nrm, unsigned idx0, unsigned W, double& bd, unsigned& bi) {
#pragma unroll
  for (int i = 0; i < WF_VR; i++) {
    if (i >= nrows) break;
    const uint32_t mr = mx1[i] & 0xffffu, mc = CH ? (mx0[i] >> 16) : (mx0[i] & 0xffffu);
    if (mr + 256u - mc == target) {
      const double d = s_nrm[mr - kmin] - s_nrm[mc - kmin];
      if (d < bd) { bd = d; bi = idx0 + (unsigned)i * W; }   // rows go down: the index only grows
    }
  }
}

__global__ void __launch_bounds__(256, WF_CTAS) window15_kernel(const uint8_t* __restrict__ src, int W, int H, int Wp,
                                                          const FrameState* __restrict__ fs, uint32_t* __restrict__ kq,
                                                          uint8_t* __restrict__ mgp, ArgPartial* __restrict__ partials) {
  extern __shared__ __align__(16) uint32_t s_w[];
  __shared__ double s_nrm[256];
  __shared__ uint32_t s_wmin[8];
  __shared__ int s_cnt[2];
  uint32_t* P0 = s_w;                       // [WF_RH][84] (B | G<<16), replicate border
  uint32_t* P1 = P0 + WF_RH * WF_PP;        // [WF_RH][84] (R | R<<16)
  uint32_t* HX0 = P1 + WF_RH * WF_PP;       // [WF_RH][68] horizontal max (B,G)
  uint32_t* HX1 = HX0 + WF_RH * WF_HP;      // horizontal max (R,R)
  uint32_t* HN0 = HX1 + WF_RH * WF_HP;      // horizontal min (B,G)
  const int f = blockIdx.z, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint8_t* img = src + (size_t)f * W * H * 3;
  const int x0 = blockIdx.x * WF_TX, y0 = blockIdx.y * WF_TY;
  const int kmin = fs[f].kmin, range = (int)fs[f].kmax - kmin;
  s_nrm[tid] = (double)tid / (double)range;  // normI value of k' (main.py:17)
  if (tid < 2) s_cnt[tid] = 0;
  // region [y0-7, y0+WF_TY+7) x [x0-8, x0+72): WF_RH x 80 pixels.  The bytes of a region row come in as aligned 32-bit
  // words into a raw staging area that borrows HX0 (free until the horizontal phase), then get unpacked from shared
  uint32_t* RAW = HX0;  // [WF_RH][64] words
  const bool words = ((W & 3) == 0) && ((reinterpret_cast<uintptr_t>(img) & 3) == 0);  // rows start on 4-byte boundaries
  const bool dwords = ((W & 7) == 0) && ((reinterpret_cast<uintptr_t>(img) & 7) == 0);  // ... and the region rows of a tile on 8-byte ones
  if (dwords && x0 >= WF_RB && x0 - WF_RB + 80 <= W) {
    // no column clamp: the 240 bytes of a row are 30 aligned 8-byte copies (x0 * 3 - 24 is a multiple of 8), a warp per
    // row, then four pixels (three words) per unpack task
    const uint2* col = reinterpret_cast<const uint2*>(img + (size_t)(x0 - WF_RB) * 3);
#pragma unroll
    for (int k = 0; k < (WF_RH + 7) / 8; k++) {
      const int ry = warp + 8 * k;
      if (ry < WF_RH && lane < 30) {
        const int y = min(max(y0 - WF_R + ry, 0), H - 1);
        wf_cp_async8(reinterpret_cast<uint2*>(RAW + ry * 64) + lane, col + (size_t)y * (W * 3 / 8) + lane);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    for (int t = tid; t < WF_RH * 20; t += 256) {
      const int ry = t / 20, g = t - ry * 20;
      const uint32_t* w = RAW + ry * 64 + 3 * g;
      const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];   // B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
      uint4 bg, rr;
      bg.x = __byte_perm(w0, 0u, 0x4140); bg.y = __byte_perm(w0, w1, 0x0403) & 0x00ff00ffu;
      bg.z = __byte_perm(w1, 0u, 0x4342); bg.w = __byte_perm(w2, 0u, 0x4241);
      rr.x = __byte_perm(w0, 0u, 0x4242); rr.y = __byte_perm(w1, 0u, 0x4141);
      rr.z = __byte_perm(w2, 0u, 0x4040); rr.w = __byte_perm(w2, 0u, 0x4343);
      *reinterpret_cast<uint4*>(P0 + ry * WF_PP + 4 * g) = bg;
      *reinterpret_cast<uint4*>(P1 + ry * WF_PP + 4 * g) = rr;
    }
  } else if (words) {
    // frame's left / right edge: columns clamp (replicate border); bytes picked one by one
    const int xa = max(x0 - WF_RB, 0), xb = min(x0 - WF_RB + 79, W - 1);  // first / last image column of the region
    const int byte0 = (xa * 3) & ~3;
    const int nw = ((xb * 3 + 2) >> 2) - (byte0 >> 2) + 1;             // <= 61
#pragma unroll 4
    for (int idx = tid; idx < WF_RH * 64; idx += 256) {
      const int ry = idx >> 6, wi = idx & 63;
      if (wi < nw) {
        const int y = min(max(y0 - WF_R + ry, 0), H - 1);
        RAW[idx] = __ldg(reinterpret_cast<const uint32_t*>(img + (size_t)y * W * 3 + byte0) + wi);
      }
    }
    __syncthreads();
    if (tid < 240) {
      const int rx = tid % 80, rr = tid / 80;
      const int xc = min(max(x0 - WF_RB + rx, 0), W - 1);
      const uint8_t* rawb = reinterpret_cast<const uint8_t*>(RAW) + (xc * 3 - byte0);
#pragma unroll 7
      for (int ry = rr; ry < WF_RH; ry += 3) {
        const uint8_t* p = rawb + ry * 256;
        uint32_t b = p[0], g = p[1], r = p[2];
        P0[ry * WF_PP + rx] = b | (g << 16);
        P1[ry * WF_PP + rx] = r | (r << 16);
      }
    }
  } else if (tid < 240) {
    const int rx = tid % 80, rr = tid / 80;
    const int xc = min(max(x0 - WF_RB + rx, 0), W - 1);
    const uint8_t* col = img + (size_t)xc * 3;
#pragma unroll 7
    for (int ry = rr; ry < WF_RH; ry += 3) {
      const int y = min(max(y0 - WF_R + ry, 0), H - 1);
      const uint8_t* p = col + (size_t)y * W * 3;
      uint32_t b = __ldg(p), g = __ldg(p + 1), r = __ldg(p + 2);
      P0[ry * WF_PP + rx] = b | (g << 16);
      P1[ry * WF_PP + rx] = r | (r << 16);
    }
  }
  __syncthreads();
  // horizontal: task = (row, run of 16 outputs); consecutive lanes take consecutive rows.  Output column o is the window
  // of region columns o + 1 .. o + 15
  if (tid < WF_RH * (WF_TX / WF_HN)) {
    const int ry = tid % WF_RH, j = tid / WF_RH;
    uint32_t p[WF_HN + 16], o[WF_HN];
    const uint4* r0 = reinterpret_cast<const uint4*>(P0 + ry * WF_PP + WF_HN * j);
#pragma unroll
    for (int q = 0; q < (WF_HN + 16) / 4; q++) { const uint4 v = r0[q]; p[4 * q] = v.x; p[4 * q + 1] = v.y; p[4 * q + 2] = v.z; p[4 * q + 3] = v.w; }
    win15<WF_HN, true, 1>(p, o);
    uint4* h0 = reinterpret_cast<uint4*>(HX0 + ry * WF_HP + WF_HN * j);
#pragma unroll
    for (int q = 0; q < WF_HN / 4; q++) h0[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    win15<WF_HN, false, 1>(p, o);
    uint4* hn = reinterpret_cast<uint4*>(HN0 + ry * WF_HP + WF_HN * j);
#pragma unroll
    for (int q = 0; q < WF_HN / 4; q++) hn[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    const uint4* r1 = reinterpret_cast<const uint4*>(P1 + ry * WF_PP + WF_HN * j);
#pragma unroll
    for (int q = 0; q < (WF_HN + 16) / 4; q++) { const uint4 v = r1[q]; p[4 * q] = v.x; p[4 * q + 1] = v.y; p[4 * q + 2] = v.z; p[4 * q + 3] = v.w; }
    win15<WF_HN, true, 1>(p, o);
    uint4* h1 = reinterpret_cast<uint4*>(HX1 + ry * WF_HP + WF_HN * j);
#pragma unroll
    for (int q = 0; q < WF_HN / 4; q++) h1[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
  }
  __syncthreads();
  // vertical: thread = (column, run of WF_VR output rows)
  const int x = tid & 63, run = tid >> 6;
  const int gx = x0 + x, ry0 = run * WF_VR, gy0 = y0 + ry0;
  const int nrows = gx < Wp ? min(WF_VR, H - gy0) : 0;
  const bool inside = gx < W;
  uint32_t mx0[WF_VR], mx1[WF_VR], dmin2 = 0xffffffffu;
  if (nrows > 0) {
    uint32_t p[WF_VR + 14], mn0[WF_VR];
#pragma unroll
    for (int i = 0; i < WF_VR + 14; i++) p[i] = HX0[(ry0 + i) * WF_HP + x];
    win15<WF_VR, true, 0>(p, mx0);
#pragma unroll
    for (int i = 0; i < WF_VR + 14; i++) p[i] = HX1[(ry0 + i) * WF_HP + x];
    win15<WF_VR, true, 0>(p, mx1);
#pragma unroll
    for (int i = 0; i < WF_VR + 14; i++) p[i] = HN0[(ry0 + i) * WF_HP + x];
    win15<WF_VR, false, 0>(p, mn0);
    const size_t pix0 = (size_t)f * Wp * H + (size_t)gy0 * Wp + gx;
    const uint32_t* pc0 = P0 + (ry0 + WF_R) * WF_PP + x + WF_RB;
    const uint32_t* pc1 = P1 + (ry0 + WF_R) * WF_PP + x + WF_RB;
    const uint32_t km2 = (uint32_t)kmin * 0x10001u;
    const bool xt = (gx < WF_R) || (gx + WF_R >= W);
    if (!xt && gy0 >= WF_R && gy0 + WF_VR - 1 + WF_R < H)
      dmin2 = wf_emit_rows<true>(mx0, mx1, mn0, pc0, pc1, kq + pix0, mgp + pix0, (unsigned)Wp, nrows, gy0, H, xt, inside, km2);
    else
      dmin2 = wf_emit_rows<false>(mx0, mx1, mn0, pc0, pc1, kq + pix0, mgp + pix0, (unsigned)Wp, nrows, gy0, H, xt, inside, km2);
  }
  // the tile's integer minima of the two differences
  {
    const uint32_t m0 = __reduce_min_sync(0xffffffffu, dmin2 & 0xffffu), m1 = __reduce_min_sync(0xffffffffu, dmin2 >> 16);
    if (lane == 0) s_wmin[warp] = m0 | (m1 << 16);
  }
  __syncthreads();   // also: every read of HX0 / HX1 / HN0 is done, the candidate lists below borrow HX0
  double* cand_d = reinterpret_cast<double*>(HX0);          // [2][256]
  unsigned* cand_i = reinterpret_cast<unsigned*>(cand_d + 512);  // [2][256]
  uint32_t cm2 = s_wmin[0];
#pragma unroll
  for (int k = 1; k < 8; k++) cm2 = __vminu2(cm2, s_wmin[k]);
  if (inside && nrows > 0) {
    const unsigned idx0 = (unsigned)gy0 * (unsigned)W + (unsigned)gx;
    if ((dmin2 & 0xffffu) == (cm2 & 0xffffu)) {
      double bd = __longlong_as_double(0x7ff0000000000000ll); unsigned bi = 0xffffffffu;
      wf_exact<0>(mx0, mx1, nrows, cm2 & 0xffffu, kmin, s_nrm, idx0, (unsigned)W, bd, bi);
      const int slot = atomicAdd(&s_cnt[0], 1);
      cand_d[slot] = bd; cand_i[slot] = bi;
    }
    if ((dmin2 >> 16) == (cm2 >> 16)) {
      double bd = __longlong_as_double(0x7ff0000000000000ll); unsigned bi = 0xffffffffu;
      wf_exact<1>(mx0, mx1, nrows, cm2 >> 16, kmin, s_nrm, idx0, (unsigned)W, bd, bi);
      const int slot = atomicAdd(&s_cnt[1], 1);
      cand_d[256 + slot] = bd; cand_i[256 + slot] = bi;
    }
  }
  __syncthreads();
  // warp 0 finishes difference 0, warp 1 difference 1: lexicographic (value, index) minimum of the candidates.
  // A NaN D (range 0) never enters: the "nothing found" marker (inf, 0xffffffff) is left for bglight_finish_kernel
  if (warp < 2) {
    const int n = s_cnt[warp];
    double bd = __longlong_as_double(0x7ff0000000000000ll); unsigned bi = 0xffffffffu;
    for (int k = lane; k < n; k += 32) {
      const double d = cand_d[warp * 256 + k]; const unsigned i = cand_i[warp * 256 + k];
      if (lex_less(d, i, bd, bi)) { bd = d; bi = i; }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, bd, d); const unsigned oi = __shfl_xor_sync(0xffffffffu, bi, d);
      if (lex_less(od, oi, bd, bi)) { bd = od; bi = oi; }
    }
    if (lane == 0) {
      ArgPartial* a = partials + ((size_t)f * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x);
      if (bi == 0xffffffffu) bd = __longlong_as_double(0x7ff0000000000000ll);
      if (warp == 0) { a->d0 = bd; a->i0 = bi; } else { a->d1 = bd; a->i1 = bi; }
    }
  }
}

// finish the arg-min and form the background light B = mean of the two selected pixels (BGDehaze.py:22-26)
__global__ void __launch_bounds__(256) bglight_finish_kernel(const uint8_t* __restrict__ src, int W, int H,
                                                             const ArgPartial* __restrict__ partials, int n_part, FrameState* fs,
                                                             int write_B, int write_Bt) {
  __shared__ ArgPartial s_part[8];
  int f = blockIdx.x;
  const ArgPartial* pp = partials + (size_t)f * n_part;
  double bd0 = __longlong_as_double(0x7ff0000000000000ll), bd1 = bd0;
  unsigned bi0 = 0xffffffffu, bi1 = 0xffffffffu;
  for (int i = threadIdx.x; i < n_part; i += 256) {
    ArgPartial a = pp[i];
    if (lex_less(a.d0, a.i0, bd0, bi0)) { bd0 = a.d0; bi0 = a.i0; }
    if (lex_less(a.d1, a.i1, bd1, bi1)) { bd1 = a.d1; bi1 = a.i1; }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    double o0 = __shfl_xor_sync(0xffffffffu, bd0, d), o1 = __shfl_xor_sync(0xffffffffu, bd1, d);
    unsigned j0 = __shfl_xor_sync(0xffffffffu, bi0, d), j1 = __shfl_xor_sync(0xffffffffu, bi1, d);
    if (lex_less(o0, j0, bd0, bi0)) { bd0 = o0; bi0 = j0; }
    if (lex_less(o1, j1, bd1, bi1)) { bd1 = o1; bi1 = j1; }
  }
  if ((threadIdx.x & 31) == 0) { ArgPartial a; a.d0 = bd0; a.d1 = bd1; a.i0 = bi0; a.i1 = bi1; s_part[threadIdx.x >> 5] = a; }
  __syncthreads();
  if (threadIdx.x == 0) {
    ArgPartial a = s_part[0];
    for (int k = 1; k < 8; k++) {
      ArgPartial b = s_part[k];
      if (lex_less(b.d0, b.i0, a.d0, a.i0)) { a.d0 = b.d0; a.i0 = b.i0; }
      if (lex_less(b.d1, b.i1, a.d1, a.i1)) { a.d1 = b.d1; a.i1 = b.i1; }
    }
    FrameState& s = fs[f];
    int kmin = s.kmin;
    double range = (double)((int)s.kmax - kmin);
    if (a.i0 == 0xffffffffu || a.i1 == 0xffffffffu) {  // constant frame: every D is NaN; np.argmin -> 0
      a.i0 = a.i1 = 0;
      s.nan_flag = 1;
    }
    if (write_B) { s.idx0 = a.i0; s.idx1 = a.i1; }
    const uint8_t* img = src + (size_t)f * W * H * 3;
    for (int c = 0; c < 3; c++) {
      double v0 = (double)((int)img[(size_t)a.i0 * 3 + c] - kmin) / range;
      double v1 = (double)((int)img[(size_t)a.i1 * 3 + c] - kmin) / range;
      double b = (v0 + v1) / 2.0;
      if (write_B) s.B[c] = b;
      if (write_Bt) s.Bt[c] = b;
    }
  }
}

// transmission_map output for the stage-wise API: t = 1 - min_window(I_c / B_c), zero padded
__global__ void traw_kernel(const uint32_t* __restrict__ kq, const uint8_t* __restrict__ mgp, int W, int H, int Wp,
                            const FrameState* __restrict__ fs, double* __restrict__ t_raw) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  const FrameState& s = fs[0];
  double range = (double)((int)s.kmax - (int)s.kmin);
  size_t pp = (size_t)y * Wp + x, pix = (size_t)y * W + x;
  int mb = (int)(kq[pp] >> 24), mg = (int)mgp[pp];
  t_raw[pix] = 1.0 - ((double)mb / range) / s.Bt[0];
  t_raw[(size_t)W * H + pix] = 1.0 - ((double)mg / range) / s.Bt[1];
}

// -------------------------------------------------------------------------------------------------
// E: restored -> R8, I8 -> YCrCb joint min / max (BGDehaze.py:75-80); stores (Yi, Cri, Cbi, Yj)
// -------------------------------------------------------------------------------------------------
constexpr int DZ_ELEMENTWISE_CTAS = 4;   // resident CTAs per SM of the two element-wise fp64 kernels
__global__ void __launch_bounds__(256, DZ_ELEMENTWISE_CTAS) exposure_minmax_kernel(GfCommon g, int W, int H, int Wp, double* dbg_restored) {
  __shared__ ExpShared sh;
  int f = blockIdx.y;
  size_t n_pp = (size_t)Wp * H;
  exp_shared_init(&sh, g.fs[f], (double)W * (double)H);
  const uint32_t* kq = g.kq + (size_t)f * n_pp;
  const float* J = g.J + (size_t)f * 2 * n_pp;
  uint32_t* ycc = g.ycc + (size_t)f * n_pp;
  unsigned imn = 255, imx = 0, jmn = 255, jmx = 0;
  const int qpr = Wp / 4;
  const size_t n_q = (size_t)qpr * H;
  for (size_t qi = (size_t)blockIdx.x * 256 + threadIdx.x; qi < n_q; qi += (size_t)gridDim.x * 256) {
    int y = (int)(qi / qpr), x0 = (int)(qi - (size_t)y * qpr) * 4;
    size_t pp = (size_t)y * Wp + x0;
    uint4 kw = __ldg(reinterpret_cast<const uint4*>(kq + pp));
    float4 jb = __ldg(reinterpret_cast<const float4*>(J + pp)), jg = __ldg(reinterpret_cast<const float4*>(J + n_pp + pp));
    uint32_t out[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      out[c] = 0;
      if (x0 + c >= W) continue;
      uint32_t w = quad_get(kw, c);
      uint32_t kb = w & 255u, kg = (w >> 8) & 255u, kr = (w >> 16) & 255u;
      int r8b = restored_byte(quad_get(jb, c), sh.fc, 0), r8g = restored_byte(quad_get(jg, c), sh.fc, 1), r8r = sh.rt.red8[kr];
      if (dbg_restored && f == 0) {
        size_t pix = (size_t)y * W + x0 + c;
        dbg_restored[pix * 3] = norm_j(quad_get(jb, c), sh.fc, 0); dbg_restored[pix * 3 + 1] = norm_j(quad_get(jg, c), sh.fc, 1);
        dbg_restored[pix * 3 + 2] = sh.rt.redN[kr];
      }
      int Yi, Cri, Cbi, Yj, Crj, Cbj;
      bgr2ycrcb_u8(sh.rt.i8[kb], sh.rt.i8[kg], sh.rt.i8[kr], Yi, Cri, Cbi);
      imn = min(imn, (unsigned)imin3(Yi, Cri, Cbi)); imx = max(imx, (unsigned)imax3(Yi, Cri, Cbi));
      bgr2ycrcb_u8(r8b, r8g, r8r, Yj, Crj, Cbj);
      jmn = min(jmn, (unsigned)imin3(Yj, Crj, Cbj)); jmx = max(jmx, (unsigned)imax3(Yj, Crj, Cbj));
      out[c] = (uint32_t)Yi | ((uint32_t)Cri << 8) | ((uint32_t)Cbi << 16) | ((uint32_t)Yj << 24);
    }
    *reinterpret_cast<uint4*>(ycc + pp) = make_uint4(out[0], out[1], out[2], out[3]);
  }
  imn = warp_reduce_min_u32(imn); imx = warp_reduce_max_u32(imx);
  jmn = warp_reduce_min_u32(jmn); jmx = warp_reduce_max_u32(jmx);
  if ((threadIdx.x & 31) == 0) {
    FrameState& s = g.fs[f];
    atomicMin(&s.yi_min, imn); atomicMax(&s.yi_max, imx);
    atomicMin(&s.yj_min, jmn); atomicMax(&s.yj_max, jmx);
  }
}

// S (BGDehaze.py:83) as a table over (Yi - min, Yj - min): both are bytes.  grid (256, n), block 256.  The entry is what the
// marches consume - rint(min(S, 1.6) 2^28) as a 32-bit integer - or GP_S_NAN where S is 0/0 (a quarter of a megabyte per frame
// instead of half of one as doubles: the per-pixel gather of splane_kernel hits the caches more often and converts nothing)
constexpr uint32_t GP_S_NAN = 0xffffffffu;   // above every real entry (1.6 x 2^28 = 0x1999999a)
__global__ void __launch_bounds__(256) stab_kernel(const FrameState* __restrict__ fs, uint32_t* __restrict__ stab) {
  int f = blockIdx.y, gy = blockIdx.x, j = threadIdx.x;
  const FrameState& s = fs[f];
  double yi_rng = (double)((int)s.yi_max - (int)s.yi_min), yj_rng = (double)((int)s.yj_max - (int)s.yj_min);
  double yi = (double)gy / yi_rng, yj = (double)j / yj_rng;
  double yi2 = 0.3 * (yi * yi);
  const double S = (yj * yi + yi2) / (yj * yj + yi2);
  stab[(size_t)f * 65536 + gy * 256 + j] = (S == S) ? __double2uint_rn(fmin(S, GP_S_PMAX) * GP_PSCALE) : GP_S_NAN;
}

// S per pixel as a plane of the table's entries, rint(min(S, 1.6) 2^28) (0 where S is 0/0): GF2a then reads it through the
// same staged row copies as the guide instead of gathering from the table inside the march.
__global__ void __launch_bounds__(256) splane_kernel(GfCommon g, int H, int Wp) {
  int f = blockIdx.y;
  size_t n_pp = (size_t)Wp * H;
  const FrameState& s = g.fs[f];
  const uint32_t a = s.yi_min, b = s.yj_min;
  const uint32_t ysub = a | (a << 8) | (a << 16) | (b << 24);
  const uint32_t* ycc = g.ycc + (size_t)f * n_pp;
  const uint32_t* stab = g.stab + (size_t)f * 65536;
  uint32_t* sp = g.splane + (size_t)f * n_pp;
  const size_t n_q = n_pp / 4;
  bool nan_seen = false;
  for (size_t qi = (size_t)blockIdx.x * 256 + threadIdx.x; qi < n_q; qi += (size_t)gridDim.x * 256) {
    uint4 yw = __ldg(reinterpret_cast<const uint4*>(ycc) + qi);
    uint32_t o[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      uint32_t w = quad_get(yw, c);
      // pad columns hold zeros: keep them away from the table (their S is never used)
      const bool pad = (w & 255u) < a || (w >> 24) < b;
      w -= ysub;
      // S = 0/0 where Yi' = Yj' = 0 (SURVEY D9): the NaN reaches every output of the reference -> flag the frame
      const uint32_t S = pad ? 0u : __ldg(stab + (((w & 255u) << 8) | (w >> 24)));
      if (S == GP_S_NAN) nan_seen = true;
      o[c] = (S == GP_S_NAN) ? 0u : S;
    }
    reinterpret_cast<uint4*>(sp)[qi] = make_uint4(o[0], o[1], o[2], o[3]);
  }
  if (__any_sync(0xffffffffu, nan_seen) && (threadIdx.x & 31) == 0) atomicOr(&g.fs[f].nan_flag, 1u);
}

// final: (OutputExp - min)/(max - min) * 255 -> rint -> saturate (BGDehaze.py:88-89, main.py:19)
__global__ void __launch_bounds__(256, DZ_ELEMENTWISE_CTAS) final_kernel(GfCommon g, int W, int H, int Wp, uint8_t* __restrict__ dst, double* dbg_out, int32_t* __restrict__ flags) {
  __shared__ ExpShared sh;
  int f = blockIdx.y;
  size_t n_pp = (size_t)Wp * H;
  exp_shared_init(&sh, g.fs[f], (double)W * (double)H);
  const FrameState& s = g.fs[f];
  double omn = dunkey(s.omin_key), den = dunkey(s.omax_key) - omn;
  double scale = 255.0 / den;
  bool nan_frame = s.nan_flag != 0;
  if (flags && blockIdx.x == 0 && threadIdx.x == 0) flags[f] = nan_frame ? UWIP_FRAME_NAN : 0;
  const uint32_t* kq = g.kq + (size_t)f * n_pp;
  const float* J = g.J + (size_t)f * 2 * n_pp;
  const float* refS = g.refS + (size_t)f * n_pp;
  uint8_t* out = dst + (size_t)f * W * H * 3;
  const int qpr = Wp / 4;
  const size_t n_q = (size_t)qpr * H;
  const bool vec_ok = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
  for (size_t qi = (size_t)blockIdx.x * 256 + threadIdx.x; qi < n_q; qi += (size_t)gridDim.x * 256) {
    int y = (int)(qi / qpr), x0 = (int)(qi - (size_t)y * qpr) * 4;
    size_t pp = (size_t)y * Wp + x0;
    uint4 kw = __ldg(reinterpret_cast<const uint4*>(kq + pp));
    float4 jb = __ldg(reinterpret_cast<const float4*>(J + pp)), jg = __ldg(reinterpret_cast<const float4*>(J + n_pp + pp));
    float4 qs = __ldg(reinterpret_cast<const float4*>(refS + pp));
    uint8_t b[12];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      double rest[3];
      rest[0] = norm_j_fast(quad_get(jb, c), sh.fc, 0);
      rest[1] = norm_j_fast(quad_get(jg, c), sh.fc, 1);
      rest[2] = sh.rt.redN[(quad_get(kw, c) >> 16) & 255u];
      double q = (double)quad_get(qs, c);
#pragma unroll
      for (int ch = 0; ch < 3; ch++) {
        double v = (rest[ch] * q - omn) * scale;
        if (dbg_out && f == 0 && x0 + c < W) dbg_out[((size_t)y * W + x0 + c) * 3 + ch] = nan_frame ? __longlong_as_double(0x7ff8000000000000ll) : (rest[ch] * q - omn) / den;
        int bv = 0;
        if (!nan_frame && v == v && fabs(v) < 2.0e9) bv = min(max(__double2int_rn(v), 0), 255);
        b[c * 3 + ch] = (uint8_t)bv;
      }
    }
    uint8_t* o = out + ((size_t)y * W + x0) * 3;
    if (vec_ok) {
      uint32_t* o32 = reinterpret_cast<uint32_t*>(o);
      o32[0] = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
      o32[1] = (uint32_t)b[4] | ((uint32_t)b[5] << 8) | ((uint32_t)b[6] << 16) | ((uint32_t)b[7] << 24);
      o32[2] = (uint32_t)b[8] | ((uint32_t)b[9] << 8) | ((uint32_t)b[10] << 16) | ((uint32_t)b[11] << 24);
    } else {
      for (int c = 0; c < 4 && x0 + c < W; c++) { o[c * 3] = b[c * 3]; o[c * 3 + 1] = b[c * 3 + 1]; o[c * 3 + 2] = b[c * 3 + 2]; }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// driver
// -------------------------------------------------------------------------------------------------
// Batch size for which the strips of the one-CTA-per-SM marches make one full wave (4K: 148 SMs / 5 strips =
// 29 frames); the host-buffer pipeline cuts its sub-batches in multiples of it.
// strips of a frame in the two layouts of the marches (4K: 8 wide, 9 narrow)
int dehaze_strips(int w) {
  GfGeom g = gf_geometry(w, 4 * 40 + 2, 40);
  return cdiv(w, g.SW);
}
int dehaze_strips_narrow(int w) { return dehaze_gf1a_strips(w); }
// Sub-batch size of a device-resident batch of n frames when at most `cap` frames of workspace are wanted: the marches run
// one CTA per SM and strip for the whole height of a frame, so a launch costs ceil(frames * strips / SMs) CTA durations
// whatever the fill of its last wave.  Among the sizes in [cap/2, cap] take the one whose parts (k - 1 of that size and
// the remainder) need the fewest waves in total; ties go to the larger size.  (4K, 256 frames, cap 96: 92 + 92 + 72 frames =
// 14 waves of the wide layout; three equal parts of 86 are 15.)
int dehaze_sub_batch(const uwip_ctx* ctx, int n, int w, int cap) {
  cap = std::max(1, cap);
  if (n <= cap) return n;
  GfGeom g = gf_geometry(w, 4 * 40 + 2, 40);
  const long long sw = cdiv(w, g.SW), sn = dehaze_gf1a_strips(w), sms = std::max(1, ctx->sm_count);
  // a CTA of a layout with S strips lasts ~1/S of the layout's time per frame; GF1a (narrow strips) is about 0.36 of the
  // march time of a frame, the three wide marches 0.64
  auto waves = [&](long long frames, long long strips) { return (double)((frames * strips + sms - 1) / sms) / (double)strips; };
  double best_cost = -1.0;
  int best = cap;
  for (int m = cap; m >= std::max(1, cap / 2); m--) {
    const int full = n / m, rem = n - full * m;
    double cost = full * (0.64 * waves(m, sw) + 0.36 * waves(m, sn)) + (rem ? 0.64 * waves(rem, sw) + 0.36 * waves(rem, sn) : 0.0);
    if (best_cost < 0.0 || cost < best_cost - 1e-9) { best_cost = cost; best = m; }
  }
  return best;
}

int dehaze_frames_dev(uwip_ctx* ctx, const uint8_t* d_src, uint8_t* d_dst, int n, int W, int H, const uwip_dehaze_params& p,
                      bool minmax_done, FrameState* fs, DehazeDebug* dbg, int32_t* d_flags) {
  UWIP_REQUIRE(ctx, n >= 1 && W >= 1 && H >= 1, "bad size");
  UWIP_REQUIRE(ctx, p.window >= 1 && p.window <= WK_MAXWIN, "window must be 1..33");
  // (2r+1)^2 255^2 < 2^32: the 32-bit window sums of the guide moments stay exact (GP_MAX_RADIUS)
  UWIP_REQUIRE(ctx, p.radius >= 1 && p.radius <= GP_MAX_RADIUS, "radius must be 1..128");
  UWIP_REQUIRE(ctx, p.eps >= GP_MIN_EPS && p.tmin <= 1.0, "eps must be >= 1e-3 and tmin <= 1");
  UWIP_REQUIRE(ctx, (size_t)W * H < (1ull << 31), "frame too large");
  UWIP_REQUIRE(ctx, !dbg || n == 1, "stage outputs are single-frame");
  size_t n_px = (size_t)W * H;
  const int Wp = (W + 3) & ~3;
  size_t n_pp = (size_t)Wp * H;
  if (!minmax_done) {
    int want = (int)std::min<size_t>((n_px * 3 / 16 + 255) / 256, 1u << 16);
    int gxm = std::max(1, std::min(want, ctx->sm_count * 8 / n + 1));
    dim3 grid(gxm, n);
    UWIP_LAUNCH(ctx, "dz_minmax", minmax_kernel, grid, 256, 0, d_src, n_px * 3, fs);
  }
  uint32_t* d_kq = (uint32_t*)uwip_slot(ctx, SLOT_KQ, (size_t)n * n_pp * 4);
  uint8_t* d_mg = (uint8_t*)uwip_slot(ctx, SLOT_MPLANES, (size_t)n * n_pp);
  uint32_t* d_ycc = (uint32_t*)uwip_slot(ctx, SLOT_YCC, (size_t)n * n_pp * 4);
  uint32_t* d_stab = (uint32_t*)uwip_slot(ctx, SLOT_STAB, (size_t)n * 65536 * 4);
  uint32_t* d_sp = (uint32_t*)uwip_slot(ctx, SLOT_SPLANE, (size_t)n * n_pp * sizeof(uint32_t));
  dim3 gridw(cdiv(Wp, WK_TX), cdiv(H, WK_TY), n);    // generic-window kernel
  dim3 gridf(cdiv(Wp, WF_TX), cdiv(H, WF_TY), n);    // 15x15 kernel
  int n_part = gridw.x * gridw.y, n_partf = gridf.x * gridf.y;
  ArgPartial* d_part = (ArgPartial*)uwip_slot(ctx, SLOT_PARTIALS, (size_t)n * std::max(n_part, n_partf) * sizeof(ArgPartial));
  int32_t* d_ab = (int32_t*)uwip_slot(ctx, SLOT_AB, (size_t)n * 8 * n_pp * sizeof(int32_t));
  float* d_J = (float*)uwip_slot(ctx, SLOT_J, (size_t)n * 2 * n_pp * sizeof(float));
  float* d_refS = (float*)uwip_slot(ctx, SLOT_REFS, (size_t)n * n_pp * sizeof(float));
  if (!d_kq || !d_mg || !d_ycc || !d_stab || !d_sp || !d_part || !d_ab || !d_J || !d_refS) return UWIP_ERR_NOMEM;
  {
    const int wmax = p.window, wmin = WK_TWIN;
    if (wmax != WK_TWIN) {
      // Background_light(normI, w) for dehazed_BG's B (BGDehaze.py:51) uses the caller's window ...
      int PL = std::max(wmax / 2, wmin / 2), PR = std::max(wmax - 1 - wmax / 2, wmin - 1 - wmin / 2);
      int RW = WK_TX + PL + PR, RH = WK_TY + PL + PR;
      size_t smem = ((size_t)2 * RW * RH + (size_t)3 * RH * WK_TX) * 4;
      UWIP_CUDA(ctx, uwip_func_smem(ctx, FUNC_WINDOW, window_kernel, smem));
      UWIP_LAUNCH(ctx, "dz_window", window_kernel, gridw, WK_THREADS, smem, d_src, W, H, Wp, wmax, fs, d_kq, d_mg, d_part);
      UWIP_LAUNCH(ctx, "dz_bglight", bglight_finish_kernel, n, 256, 0, d_src, W, H, d_part, n_part, fs, 1, 0);
    }
    // ... but refined_t() is always called without w (BGDehaze.py:52): the transmission and the
    // background light inside transmission_map use the 15x15 window
    size_t smemf = ((size_t)2 * WF_RH * WF_PP + (size_t)3 * WF_RH * WF_HP) * 4;
    UWIP_CUDA(ctx, uwip_func_smem(ctx, FUNC_WINDOW15, window15_kernel, smemf));
    UWIP_LAUNCH(ctx, "dz_window", window15_kernel, gridf, 256, smemf, d_src, W, H, Wp, fs, d_kq, d_mg, d_part);
    UWIP_LAUNCH(ctx, "dz_bglight", bglight_finish_kernel, n, 256, 0, d_src, W, H, d_part, n_partf, fs, wmax == WK_TWIN ? 1 : 0, 1);
  }
  if (dbg && dbg->stop_after == 1) return UWIP_OK;
  if (dbg && dbg->t_raw) {
    dim3 g2(cdiv(W, 256), H);
    UWIP_LAUNCH(ctx, "dz_traw", traw_kernel, g2, 256, 0, d_kq, d_mg, W, H, Wp, fs, dbg->t_raw);
  }
  if (dbg && dbg->stop_after == 2) return UWIP_OK;

  GfCommon gc;
  gc.kq = d_kq; gc.mg = d_mg; gc.ycc = d_ycc; gc.stab = d_stab; gc.splane = d_sp; gc.ab = d_ab; gc.J = d_J; gc.refS = d_refS; gc.fs = fs;
  gc.eps = p.eps; gc.tmin = p.tmin; gc.dbg_tref = dbg ? dbg->t_ref : nullptr;
  UWIP_CHECK(dehaze_gf1a_launch(ctx, gc, n, W, H, p.radius));
  UWIP_CHECK(gp_launch<PipGF1b>(ctx, "dz_gf1b", FUNC_GF1B, gc, n, W, H, p.radius));
  if (dbg && dbg->stop_after == 3) return UWIP_OK;
  int gx = std::max(1, std::min((int)((n_pp / 4 + 1023) / 1024), std::max(1, ctx->sm_count * 24 / n)));
  dim3 grid_e(gx, n);
  UWIP_LAUNCH(ctx, "dz_exposure_minmax", exposure_minmax_kernel, grid_e, 256, 0, gc, W, H, Wp, dbg ? dbg->restored : (double*)nullptr);
  if (dbg && dbg->stop_after == 4) return UWIP_OK;
  dim3 grid_s(256, n);
  UWIP_LAUNCH(ctx, "dz_stab", stab_kernel, grid_s, 256, 0, fs, d_stab);
  UWIP_LAUNCH(ctx, "dz_splane", splane_kernel, grid_e, 256, 0, gc, H, Wp);
  UWIP_CHECK(gp_launch<PipGF2a>(ctx, "dz_gf2a", FUNC_GF2A, gc, n, W, H, p.radius));
  UWIP_CHECK(gp_launch<PipGF2b>(ctx, "dz_gf2b", FUNC_GF2B, gc, n, W, H, p.radius));
  UWIP_LAUNCH(ctx, "dz_final", final_kernel, grid_e, 256, 0, gc, W, H, Wp, d_dst, dbg ? dbg->out : (double*)nullptr, d_flags);
  return UWIP_OK;
}

// -------------------------------------------------------------------------------------------------
// stage entry points of guidedfilter.py (stage-wise parity; not on the throughput path)
// -------------------------------------------------------------------------------------------------
// boxfilter(I, r) guidedfilter.py:23-51: (2r+1)^2 window SUM, windows truncated at the borders; float64.  Two
// separable passes of direct sums (the reference takes differences of cumulative sums: 2e-11 relative apart).
__global__ void __launch_bounds__(256) box_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, int W, int H, int r) {
  const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  const double* row = src + (size_t)y * W;
  double s = 0.0;
  for (int k = max(x - r, 0); k <= min(x + r, W - 1); k++) s += row[k];
  dst[(size_t)y * W + x] = s;
}
__global__ void __launch_bounds__(256) box_cols_kernel(const double* __restrict__ src, double* __restrict__ dst, int W, int H, int r) {
  const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  double s = 0.0;
  for (int k = max(y - r, 0); k <= min(y + r, H - 1); k++) s += src[(size_t)k * W + x];
  dst[(size_t)y * W + x] = s;
}
int boxfilter_f64_dev(uwip_ctx* ctx, const double* d_src, double* d_tmp, double* d_dst, int W, int H, int r) {
  UWIP_REQUIRE(ctx, W >= 1 && H >= 1 && r >= 0, "bad size");
  dim3 grid(cdiv(W, 256), H);
  UWIP_LAUNCH(ctx, "box_rows", box_rows_kernel, grid, 256, 0, d_src, d_tmp, W, H, r);
  UWIP_LAUNCH(ctx, "box_cols", box_cols_kernel, grid, 256, 0, (const double*)d_tmp, d_dst, W, H, r);
  return UWIP_OK;
}

// guided_filter(I, p, r, eps) guidedfilter.py:54-103 for a guide of the form I = guide8 / range (every guide on the path
// is: main.py:17, BGDehaze.py:77-80).  The packed guide and the fixed-point p feed the same two marches as the third
// filter of adaptiveExp_map.
__global__ void __launch_bounds__(256) gfq_pack_kernel(const uint8_t* __restrict__ guide, const double* __restrict__ p, int W, int H, int Wp,
                                                       uint32_t* __restrict__ ycc, uint32_t* __restrict__ sp, FrameState* fs) {
  const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
  if (x >= Wp) return;
  uint32_t g = 0, P = 0;
  bool bad = false;
  if (x < W) {
    const uint8_t* q = guide + ((size_t)y * W + x) * 3;
    g = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16);
    const double v = p[(size_t)y * W + x];
    bad = !(v >= 0.0 && v <= GP_S_PMAX);
    P = bad ? 0u : __double2uint_rn(v * GP_PSCALE);
  }
  ycc[(size_t)y * Wp + x] = g;
  sp[(size_t)y * Wp + x] = P;
  if (bad) atomicOr(&fs[0].nan_flag, 2u);
}
__global__ void gfq_state_kernel(FrameState* fs, int range) {
  FrameState& s = fs[0];
  s.yi_min = 0; s.yi_max = (unsigned)range; s.yj_min = 0; s.yj_max = (unsigned)range;
  s.kmin = 0; s.kmax = (unsigned)range;
}
int guided_filter_u8_dev(uwip_ctx* ctx, const uint8_t* d_guide, const double* d_p, double* d_q, int W, int H, int range, int r, double eps,
                         FrameState* fs) {
  // (2r+1)^2 255^2 < 2^32 for r <= GP_MAX_RADIUS, as in dehaze_frames_dev
  UWIP_REQUIRE(ctx, W >= 1 && H >= 1 && r >= 1 && r <= GP_MAX_RADIUS && range >= 1 && range <= 255 && eps >= GP_MIN_EPS, "bad argument");
  const int Wp = (W + 3) & ~3;
  const size_t n_pp = (size_t)Wp * H;
  uint32_t* d_ycc = (uint32_t*)uwip_slot(ctx, SLOT_YCC, n_pp * 4);
  uint32_t* d_sp = (uint32_t*)uwip_slot(ctx, SLOT_SPLANE, n_pp * 4);
  int32_t* d_ab = (int32_t*)uwip_slot(ctx, SLOT_AB, 8 * n_pp * 4);
  if (!d_ycc || !d_sp || !d_ab) return UWIP_ERR_NOMEM;
  UWIP_CHECK(frame_state_reset(ctx, fs, 1));
  UWIP_LAUNCH(ctx, "gfq_state", gfq_state_kernel, 1, 1, 0, fs, range);
  dim3 grid(cdiv(Wp, 256), H);
  UWIP_LAUNCH(ctx, "gfq_pack", gfq_pack_kernel, grid, 256, 0, d_guide, d_p, W, H, Wp, d_ycc, d_sp, fs);
  GfCommon gc;
  memset(&gc, 0, sizeof(gc));
  gc.ycc = d_ycc; gc.splane = d_sp; gc.ab = d_ab; gc.fs = fs; gc.eps = eps; gc.tmin = 0.0; gc.dbg_tref = d_q;
  UWIP_CHECK(gp_launch<PipGF2a>(ctx, "dz_gf2a", FUNC_GF2A, gc, 1, W, H, r));
  UWIP_CHECK(gp_launch<PipGFq>(ctx, "gfq_out", FUNC_GFQ, gc, 1, W, H, r));
  return UWIP_OK;
}
