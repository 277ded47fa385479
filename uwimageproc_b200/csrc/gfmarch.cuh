// gfmarch.cuh - what the guided-filter marches (gfpipe.cuh) share with the rest of dehaze.cu: small fp64 / copy helpers, the plane
// bundle GfCommon, the strip geometry, frame constants, and the launcher.  Included by dehaze.cu (wide strips: GF1b, GF2a, GF2b, GFq)
// and by dehaze_gf1a.cu (GP_NARROW strips: GF1a), which differ only in the layout constants of gfpipe.cuh.
#pragma once
#include <algorithm>

#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// small fp64 helpers
// ------------------------------------------------------------------------------------------------
// exact uint32 -> double: one I2F on the conversion pipe (the 2^52 magic-add form costs three issue slots)
__device__ __forceinline__ double u2d(uint32_t u) { return __uint2double_rn(u); }
// 1/x to ~1 ulp (MUFU seed + two Newton steps).  Used where the result feeds continuous arithmetic
// only; every place whose result is truncated to a byte uses the IEEE division.
__device__ __forceinline__ double rcp_fast(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// cp.async (LDGSTS): global -> shared without a register in between
__device__ __forceinline__ void cp_async16(void* smem, const void* g) {
  unsigned a = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(a), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem, const void* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_wait_2() { asm volatile("cp.async.wait_group 2;" ::: "memory"); }
__device__ __forceinline__ void cp_async4(void* smem, const void* g) {
  unsigned a = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(a), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// mbarriers (the TMA bulk copies of gfpipe.cuh count their completion in bytes on them)
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}

// ------------------------------------------------------------------------------------------------
// guided-filter helpers
// ------------------------------------------------------------------------------------------------
// 3x3 symmetric system shared by GF1a / GF2a (gfpipe.cuh: gp_solve_rhs solves it for each signal).  Inputs are window sums
// in k units: si[0..2] (sum k_i), si[3..8] (sum k_i k_j: 00 01 02 11 12 22), N (window pixel count).
__device__ __forceinline__ void gf_build_M(const uint32_t* si, double N, double epsN2, double* M, double* Sd) {
  Sd[0] = u2d(si[0]); Sd[1] = u2d(si[1]); Sd[2] = u2d(si[2]);
  // exact: N*S_ij and S_i*S_j are integers < 2^53
  M[0] = fma(N, u2d(si[3]), -Sd[0] * Sd[0]) + epsN2;
  M[1] = fma(N, u2d(si[4]), -Sd[0] * Sd[1]);
  M[2] = fma(N, u2d(si[5]), -Sd[0] * Sd[2]);
  M[3] = fma(N, u2d(si[6]), -Sd[1] * Sd[1]) + epsN2;
  M[4] = fma(N, u2d(si[7]), -Sd[1] * Sd[2]);
  M[5] = fma(N, u2d(si[8]), -Sd[2] * Sd[2]) + epsN2;
}
// adjugate of the symmetric matrix [[m0 m1 m2],[m1 m3 m4],[m2 m4 m5]] and 1/det
__device__ __forceinline__ void gf_adjugate(const double* M, double* A, double& rdet) {
  A[0] = M[3] * M[5] - M[4] * M[4];
  A[1] = M[2] * M[4] - M[1] * M[5];
  A[2] = M[1] * M[4] - M[2] * M[3];
  A[3] = M[0] * M[5] - M[2] * M[2];
  A[4] = M[1] * M[2] - M[0] * M[4];
  A[5] = M[0] * M[3] - M[1] * M[1];
  double det = M[0] * A[0] + M[1] * A[1] + M[2] * A[2];
  rdet = rcp_fast(det);
}

struct GfCommon {
  const uint32_t* kq;     // [n][H][Wp] packed k'_b k'_g k'_r m'_b
  const uint8_t* mg;      // [n][H][Wp] m'_g
  uint32_t* ycc;          // [n][H][Wp] packed Yi Cri Cbi Yj
  const uint32_t* stab;   // [n][256][256] exposure ratio S(yi', yj') as rint(S 2^28), 0xffffffff where S is 0/0
  uint32_t* splane;       // [n][H][Wp] S per pixel as rint(S 2^28)
  int32_t* ab;            // [n][8][H][Wp] coefficient rows, int32 fixed point (gfpipe.cuh: coef_scale)
  float* J;               // [n][2][H][Wp]
  float* refS;            // [n][H][Wp]
  FrameState* fs;
  double eps, tmin;
  double* dbg_tref;       // optional [2][H*W] (frame 0 only)
};

// Largest guided-filter radius: SOLVE forms the window sums of the guide moments k_i k_j (k <= 255) as uint32
// (gp_window_pair), exact while a full window's (2r+1)^2 255^2 < 2^32 - up to r = 128 (4,294,836,225; r = 129 can reach
// 4,361,942,025).  The entry points refuse larger radii.
constexpr int GP_MAX_RADIUS = 128;
// Smallest eps: the stored b of a coefficient chunk is int32 fixed point with the exponent of coef_scale's proven bound
// 1.6 + 1.4 / sqrt(eps), so its step grows as eps shrinks (2^-24 at 1e-3, 2^-22 at 1e-4, 2^-19 at 1e-6).  Below 1e-3 the
// rounding of b alone puts outputs near zero (a step edge of p, t near 0 with tmin = 0) past 1e-5 of max(|q|, 1e-3).
constexpr double GP_MIN_EPS = 1e-3;

// strip geometry of one launch (see the file header)
struct GfGeom {
  int W, H, Wp;   // image size; pitch of the internal planes (multiple of 4)
  int r;          // box radius
  int HL;         // halo rounded up to a multiple of 4
  int SW;         // output columns per strip (multiple of 4)
  int NQ;         // quads per strip: one zero guard quad + (2*HL + SW)/4
  int seg_h;      // output rows per vertical segment
  int fast;       // r % 4 == 0: window edges fall on quad boundaries
};

// ---- shared per-CTA frame constants --------------------------------------------------------------
struct FrameConst {
  int kmin, range;
  double B[3], Bt[3];
  // restored-image parameters (valid after GF1b): J min / (max-min)
  double jmin[2], jinv[2], jrcp[2];
  int yi_min, yi_rng, yj_min, yj_rng;
};

__device__ __forceinline__ void load_frame_const(const FrameState& s, FrameConst& c) {
  c.kmin = s.kmin;
  c.range = (int)s.kmax - (int)s.kmin;
  c.B[0] = s.B[0]; c.B[1] = s.B[1]; c.B[2] = s.B[2];
  c.Bt[0] = s.Bt[0]; c.Bt[1] = s.Bt[1]; c.Bt[2] = s.Bt[2];
  for (int k = 0; k < 2; k++) {
    double mn = dunkey(s.jmin_key[k]), mx = dunkey(s.jmax_key[k]);
    c.jmin[k] = mn;
    c.jinv[k] = mx - mn;  // denominator; divisions are done where used
    c.jrcp[k] = 1.0 / (mx - mn);
  }
  c.yi_min = s.yi_min; c.yi_rng = (int)s.yi_max - (int)s.yi_min;
  c.yj_min = s.yj_min; c.yj_rng = (int)s.yj_max - (int)s.yj_min;
}

// red channel of `restored` (RC_correction, BGDehaze.py:61-64) as a function of k'_r, plus the
// truncated bytes R8 / I8 of adaptiveExp_map (BGDehaze.py:75-76).
struct RedTables {
  double redN[256];     // normRrec for k' = 0..255
  uint8_t red8[256];    // (normRrec*255).astype(uint8)
  uint8_t i8[256];      // (normI*255).astype(uint8) for k'
};
__device__ __forceinline__ int trunc_u8(double v) {  // numpy float64 -> uint8 cast for v in [0,255]; NaN -> 0
  if (!(v == v)) return 0;
  int i = (int)v;
  return i & 0xff;
}
static __device__ void build_red_tables(const FrameState& s, const FrameConst& fc, double n_px, RedTables* rt, int tid, int nthreads) {
  double range = (double)fc.range;
  double mean_b = ((double)s.jsum_fix[0] * (1.0 / 4294967296.0) / n_px - fc.jmin[0]) / fc.jinv[0];
  double mean_g = ((double)s.jsum_fix[1] * (1.0 / 4294967296.0) / n_px - fc.jmin[1]) / fc.jinv[1];
  double avgRr = 1.5 - mean_b - mean_g;
  double mean_r = ((double)s.rsum / n_px) / range;
  double coef = avgRr / mean_r;
  double ra = ((double)s.rmin / range) * coef, rb = ((double)s.rmax / range) * coef;
  double rmn = fmin(ra, rb), rmx = fmax(ra, rb);
  for (int k = tid; k < 256; k += nthreads) {
    double nk = (double)k / range;
    double v = (nk * coef - rmn) / (rmx - rmn);
    rt->redN[k] = v;
    rt->red8[k] = (uint8_t)trunc_u8(v * 255.0);
    rt->i8[k] = (uint8_t)trunc_u8(nk * 255.0);
  }
}

struct ExpShared {
  RedTables rt;
  FrameConst fc;
};
static __device__ void exp_shared_init(ExpShared* sh, const FrameState& s, double n_px) {
  if (threadIdx.x == 0) load_frame_const(s, sh->fc);
  __syncthreads();
  build_red_tables(s, sh->fc, n_px, &sh->rt, threadIdx.x, blockDim.x);
  __syncthreads();
}
// restored blue / green from the stored J value (dehazed_BG, BGDehaze.py:53-56).  The IEEE division is
// what the bytes R8 are truncated from; the reciprocal flavour feeds products only.
__device__ __forceinline__ double norm_j(float j, const FrameConst& fc, int c) { return ((double)j - fc.jmin[c]) / fc.jinv[c]; }
__device__ __forceinline__ double norm_j_fast(float j, const FrameConst& fc, int c) { return ((double)j - fc.jmin[c]) * fc.jrcp[c]; }
// (restored*255).astype(uint8) of BGDehaze.py:75: the byte is a truncation, so the quotient must be the
// IEEE one only where restored*255 sits next to an integer; everywhere else the reciprocal product (a few
// ulp off) truncates to the same byte.
__device__ __forceinline__ int restored_byte(float j, const FrameConst& fc, int c) {
  double v = norm_j_fast(j, fc, c) * 255.0;
  if (fabs(v - rint(v)) < 1.0e-9 || !(v == v)) v = norm_j(j, fc, c) * 255.0;
  return trunc_u8(v);
}

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}
__device__ __forceinline__ float warp_min_f32(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}
__device__ __forceinline__ float warp_max_f32(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}
__device__ __forceinline__ double warp_min_f64(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}
__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}

__device__ __forceinline__ uint32_t quad_get(const uint4& v, int c) { return c == 0 ? v.x : (c == 1 ? v.y : (c == 2 ? v.z : v.w)); }
__device__ __forceinline__ float quad_get(const float4& v, int c) { return c == 0 ? v.x : (c == 1 ? v.y : (c == 2 ? v.z : v.w)); }


// Coefficient rows (the a,b of a guided filter) are stored quad-interleaved: per image row, per quad of
// four pixels, NP/4 sixteen-byte chunks per pixel (chunk = a0,a1,a2,b of one filter) - 128 bytes per quad
// for GF1 (two filters), 64 for GF2.  The chunk order inside a quad is XOR-swizzled with the quad index
// so that the V-phase of the reader (one thread per quad, a 16-byte shared load per chunk) is free of
// bank conflicts although consecutive lanes are a whole quad apart.  Writer and reader are both ours.
template <int NP>
__device__ __forceinline__ int coef_chunk(int gq, int c, int j) {  // physical chunk of (pixel c, filter j) in quad gq
  if (NP == 8) return (2 * c + j) ^ (gq & 7);
  return c ^ ((gq >> 1) & 3);
}

// -------------------------------------------------------------------------------------------------
// the guided-filter marches: warp-specialised pipeline (gfpipe.cuh)
// -------------------------------------------------------------------------------------------------
#include "gfpipe.cuh"

// geometry + launch -------------------------------------------------------------------------------------
static GfGeom gf_geometry(int W, int H, int r) {
  GfGeom g;
  g.W = W; g.H = H; g.Wp = (W + 3) & ~3; g.r = r;
  g.HL = (r + 3) & ~3;
  int sw_max = std::min(4 * (GP_NTR - 1) - 2 * g.HL, GP_MAXSW);   // quads per strip (ACC) and pixel pairs per strip (SOLVE)
  int strips = cdiv(W, sw_max);
  g.SW = (cdiv(W, strips) + 3) & ~3;
  g.NQ = 1 + (2 * g.HL + g.SW) / 4;
  g.seg_h = H;
  g.fast = (r % 4 == 0) ? 1 : 0;
  return g;
}

template <class P>
static int gp_launch(uwip_ctx* ctx, const char* tag, int func_id, const GfCommon& gc, int n, int W, int H, int r) {
  GfGeom gg = gf_geometry(W, H, r);
  int strips = cdiv(W, gg.SW);
  // vertical segments: fill the machine (tail of the last wave) against the 2r warm-up rows per segment
  int slots = ctx->sm_count;
  int tasks = strips * n;
  int best = 1;
  double best_eff = 0.0;
  int max_segs = std::max(1, H / (4 * r + 2));
  for (int s = 1; s <= max_segs && s <= 64; s++) {
    int sh = cdiv(H, s), sc = cdiv(H, sh);
    double waves = (double)cdiv(tasks * sc, slots);
    double eff = ((double)tasks * sc / (waves * slots)) * ((double)sh / (double)(sh + 2 * r));
    if (eff > best_eff * 1.02) { best_eff = eff; best = s; }
  }
  gg.seg_h = cdiv(H, best);
  int segs = cdiv(H, gg.seg_h);
  static_assert(GpSmem<P>::bytes <= 227 * 1024, "shared memory");
  size_t smem = GpSmem<P>::bytes;
  UWIP_CUDA(ctx, uwip_func_smem(ctx, func_id, gp_kernel<P>, smem));
  dim3 grid(strips, segs, n);
  UWIP_LAUNCH(ctx, tag, gp_kernel<P>, grid, GP_THREADS, smem, gc, gg);
  return UWIP_OK;
}
