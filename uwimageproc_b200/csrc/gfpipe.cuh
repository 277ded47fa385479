// gfpipe.cuh - the guided-filter box sums of bgdehaze as a warp-specialised pipeline (included by gfmarch.cuh).
//   reference: modules/bgdehaze/guidedfilter.py:23-103 (boxfilter, guided_filter), BGDehaze.py:39-48,84.
//
// One CTA (one per SM) owns a strip of image columns plus a halo of r columns on both sides and walks down the rows.  Three
// roles hand rows to each other through mbarriers over a ring of published rows in shared memory (P::NSTAGE stages):
//   ACC   one thread per quad of four columns keeps the vertical running sums of every moment in registers (32-bit integers
//         for the guide moments, integer-valued doubles for the signal moments: exact) and publishes per output row the
//         inclusive prefix over its quad and the quad total.
//   AUX   turns the quad totals of a published row into prefixes over the strip; lane 0 of the first auxiliary warp is the
//         TMA producer of the coefficient rows of the plane readers.
//   SOLVE one thread per two adjacent output pixels forms their window sums from the published row, then does the per-pixel
//         work of the policy (3x3 solve / the filter output and its reductions).
// Warp order is issue priority (the scheduler prefers the highest warp id): SOLVE first, then ACC, the auxiliary warps last.
// The two strip layouts, the register budgets per role and the measurements behind them: DESIGN.md section 3.
#pragma once

#ifndef GP_NARROW
#define GP_NARROW 0             // 1: strips of 128 quads - four ACC warps in one warpgroup, four auxiliary warps in another with their own (small) register count
#endif
constexpr int GP_AUX_REGS = 88;   // GP_NARROW: registers of an auxiliary thread
constexpr int GP_GF1A_ACC_REGS = GP_NARROW ? 176 : 152;
constexpr int GP_GF2A_ACC_REGS = GP_NARROW ? 168 : 144;
constexpr int GP_B_ACC_REGS = GP_NARROW ? 128 : 136;

constexpr int GP_NT = GP_NARROW ? 128 : 160;   // quads of a strip (quad 0 is the zero guard) = ACC worker threads
constexpr int GP_NTR = GP_NT < 152 ? GP_NT : 152;   // quads of a strip that can hold data (gf_geometry keeps NQ within it): the pitch of the TMA ring rows
constexpr int GP_NAUX = GP_NARROW ? 4 : 3;      // auxiliary warps
constexpr int GP_SOLVE_THREADS = 256; // two warpgroups (threads 0..255)
constexpr int GP_ACC_THREADS = GP_NT + 32 * GP_NAUX;   // two warpgroups
constexpr int GP_THREADS = GP_ACC_THREADS + GP_SOLVE_THREADS;
constexpr int GP_MAXSW = 2 * GP_SOLVE_THREADS;   // output columns per strip
constexpr int GP_NSEG = 8, GP_SEGQ = 20;         // scan: 8 lanes per moment, 20 quads per lane (5 x 16 bytes of u32: odd -> conflict-free)
constexpr int GP_GP = GP_NSEG * GP_SEGQ;         // pitch of a quad-total row
// fp64 quad-total rows: a scan segment of 20 doubles is ten 16-byte chunks - an even number, so the eight lanes of a moment
// would start 2-way bank conflicted (segment stride 160 B = 8 banks x 5: lanes s and s + 4 share banks).  GP_SEG_PAD doubles of
// padding after every segment make the stride an odd number of chunks: every 16-byte access of the scan is conflict-free.
constexpr int GP_SEG_PAD = 2;
constexpr int GP_SEGD = GP_SEGQ + GP_SEG_PAD;    // segment stride of an fp64 quad-total row
constexpr int GP_GPD = GP_NSEG * GP_SEGD;        // pitch of an fp64 quad-total row
__device__ __forceinline__ int gp_dpos(int t) { return t + GP_SEG_PAD * (t / GP_SEGQ); }   // position of quad t in such a row
static_assert(GP_GP >= GP_NT, "thread layout");

// The filtered signal p (transmission, exposure ratio) is held as rint(p * 2^28): the guided filter amplifies a
// perturbation of p by up to ~10^3 (a = cov / (var + eps) with eps = 10^-3): a 2^-25 grid already costs 1.7e-5.
constexpr double GP_PSCALE = 268435456.0, GP_PINV = 1.0 / 268435456.0;
constexpr double GP_T_PMAX = 1.0, GP_S_PMAX = 1.6;
// registers left for a SOLVE thread when an ACC / AUX thread takes `acc` (pool = threads x launch registers), in units of 8
#define GP_SOLVE_REGS_FOR(acc) (GP_NARROW ? ((((65536 - 128 * (acc) - 128 * GP_AUX_REGS) / 256) / 8) * 8) : 256 - (acc))

// wait for the phase with the given parity; the suspend-time hint lets the hardware park the warp until the phase
// completes (or the time runs out) instead of re-issuing the test every few cycles
__device__ __forceinline__ void mbar_wait_park(uint64_t* bar, unsigned parity) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(a), "r"(parity), "r"(20000u) : "memory");
}
// L2 eviction policies for the coefficient rows of the plane readers: every row is read twice, 2r+1 march rows apart
__device__ __forceinline__ uint64_t l2_policy_evict_last(float fraction) {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, %1;" : "=l"(p) : "f"(fraction));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// TMA 1-D bulk copy global -> shared with an L2 cache policy, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s_hint(void* smem, const void* g, unsigned bytes, uint64_t* bar, uint64_t policy) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem), b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(d), "l"(g),
               "r"(bytes), "r"(b), "l"(policy) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}

// coefficient planes: int32 fixed point (a0, a1, a2, b) per pixel and filter.  |a_k| <= std(p)/sqrt(eps_k)
// (Cauchy-Schwarz on cov = E[(I-mu)(p-mu_p)] and (Sigma + eps)^-1 <= 1/eps), |b| <= max p + |a| |mean I|: the
// exponents below keep every stored value inside 2^30.  p <= 1.6 on both filters (transmission <= 1, S <= 1.54).
struct CoefScale { double sa, sb, isa, isb; };
__device__ __forceinline__ CoefScale coef_scale(double eps, double range) {
  double se = sqrt(eps);
  double amax = 0.8 / (range * se), bmax = 1.6 + 1.4 / se;
  int ea = 30 - (int)ceil(log2(amax)), eb = 30 - (int)ceil(log2(bmax));
  ea = min(max(ea, 0), 60); eb = min(max(eb, 0), 60);
  CoefScale c;
  c.sa = exp2((double)ea); c.sb = exp2((double)eb);
  c.isa = exp2((double)-ea); c.isb = exp2((double)-eb);
  if (!(range > 0.0) || !(eps > 0.0)) { c.sa = c.sb = c.isa = c.isb = 1.0; }
  return c;
}

// One scan task: GP_SEGQ consecutive quad totals of one moment -> inclusive prefix over the whole row.  The eight tasks
// of a moment sit in eight adjacent lanes; their segment totals are exchanged with shuffles.  The segment lives in
// registers between the load and the store (one pass over shared memory); the in-register prefix is done per group of
// four to keep the dependent chain short.
template <class T, class V4>
__device__ __forceinline__ void gp_scan_task(T* row, int seg, bool live) {
  constexpr int VW = sizeof(V4) / sizeof(T);  // 4 (u32) or 2 (f64)
  constexpr int NG = GP_SEGQ / 4;             // groups of four values
  T* p = row + seg * (VW == 2 ? GP_SEGD : GP_SEGQ);
  T v[GP_SEGQ];
#pragma unroll
  for (int i = 0; i < GP_SEGQ; i += VW) {
    V4 q;
    if (live) q = *reinterpret_cast<const V4*>(p + i);
    if constexpr (VW == 4) { v[i] = live ? q.x : T(0); v[i + 1] = live ? q.y : T(0); v[i + 2] = live ? q.z : T(0); v[i + 3] = live ? q.w : T(0); }
    else { v[i] = live ? q.x : T(0); v[i + 1] = live ? q.y : T(0); }
  }
  T gt[NG];
#pragma unroll
  for (int g = 0; g < NG; g++) {  // prefix inside each group of four (independent chains of three)
    v[4 * g + 1] += v[4 * g]; v[4 * g + 2] += v[4 * g + 1]; v[4 * g + 3] += v[4 * g + 2];
    gt[g] = v[4 * g + 3];
  }
#pragma unroll
  for (int g = 1; g < NG; g++) gt[g] += gt[g - 1];  // inclusive prefix of the group totals
  T incl = gt[NG - 1];
#pragma unroll
  for (int d = 1; d < GP_NSEG; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, incl, d, GP_NSEG);
    if (seg >= d) incl += o;
  }
  T run = __shfl_up_sync(0xffffffffu, incl, 1, GP_NSEG);  // exclusive offset of this segment
  if (seg == 0) run = 0;
  if (live) {
#pragma unroll
    for (int i = 0; i < GP_SEGQ; i += VW) {
      T off = run + (i >= 4 ? gt[i / 4 - 1] : T(0));
      V4 q;
      if constexpr (VW == 4) { q.x = v[i] + off; q.y = v[i + 1] + off; q.z = v[i + 2] + off; q.w = v[i + 3] + off; }
      else { q.x = v[i] + off; q.y = v[i + 1] + off; }
      *reinterpret_cast<V4*>(p + i) = q;
    }
  }
}

// layout of the fp64 in-quad prefixes: even / odd elements per array (six conflict-free 8-byte window loads per moment) for the
// policies with up to four fp64 moments, pairs per array (five loads, one of them two-way conflicted) for those with eight:
// measured per kernel (profiles/r2_summary.md)
#define GP_EVEN_ODD(nd) ((nd) <= 4)

// mbarrier indices (up to four stages / ring slots)
enum { GPB_FULL = 0, GPB_READY = 4, GPB_EMPTY = 8, GPB_TFULL = 12, GPB_TEMPTY = 16, GPB_COUNT = 20 };

template <class P>
struct GpSmem {
  static constexpr int NT = GP_NT, GP = GP_GP, NI = P::NI, ND = P::ND, NSTAGE = P::NSTAGE;
  // one published row: Pd [ND][NT] 4 x f64 (inclusive in-quad prefixes) | Gd [ND][GP] f64 | Pi [NI][NT] uint4 | Gi [NI][GP] u32
  // (Pd = two arrays: Pa [ND][NT] (p0, p1) and, 64 bytes past a multiple of 128 further, Pb [ND][NT] (p2, p3): consecutive
  // threads publish consecutive 16 bytes, and the 16-byte loads of the two halves of a quad fall into different banks)
  static constexpr size_t off_pb = (((size_t)ND * NT * 16 + 127) & ~(size_t)127) + 64;
  static constexpr size_t off_gd = (off_pb + (size_t)ND * NT * 16 + 127) & ~(size_t)127;
  static constexpr size_t off_pi = off_gd + (size_t)ND * GP_GPD * 8;
  static constexpr size_t off_gi = off_pi + (size_t)NI * NT * 16;
  static constexpr size_t stage_bytes = (off_gi + (size_t)NI * GP * 4 + 127) & ~(size_t)127;
  static constexpr size_t off_sh = NSTAGE * stage_bytes;
  static constexpr size_t off_in = (off_sh + sizeof(typename P::Shared) + 127) & ~(size_t)127;  // ACC input staging
  static constexpr size_t off_bar = off_in + P::IN_BYTES;
  static constexpr size_t off_sin = (off_bar + 8 * GPB_COUNT + 15) & ~(size_t)15;   // SOLVE input staging: 3 row slots x 8-byte fields x threads
  static constexpr size_t bytes = off_sin + (size_t)3 * P::SOLVE_FIELDS * GP_SOLVE_THREADS * 8 + 16;
};

struct GpStage {
  double2* Pa; double2* Pb; double* Gd; uint4* Pi; uint32_t* Gi;   // in-quad prefixes per quad and moment: Pa = (p0, p1), Pb = (p2, p3 = quad total); policies with few fp64 moments: (p0, p2), (p1, p3)
};
template <class P>
__device__ __forceinline__ GpStage gp_stage(unsigned char* smem, int s) {
  typedef GpSmem<P> L;
  unsigned char* b = smem + (size_t)s * L::stage_bytes;
  GpStage g;
  g.Pa = reinterpret_cast<double2*>(b);
  g.Pb = reinterpret_cast<double2*>(b + L::off_pb);
  g.Gd = reinterpret_cast<double*>(b + L::off_gd);
  g.Pi = reinterpret_cast<uint4*>(b + L::off_pi);
  g.Gi = reinterpret_cast<uint32_t*>(b + L::off_gi);
  return g;
}
// position in the ring of published rows: stage index and the parity of its current use
struct GpRing {
  int s; unsigned ph;
  __device__ __forceinline__ GpRing() : s(0), ph(0) {}
  template <int NSTAGE> __device__ __forceinline__ void next() { if (++s == NSTAGE) { s = 0; ph ^= 1u; } }
};

// geometry shared by the roles
struct GpGeo {
  int W, H, Wp, r, rho, HL, SW, NQ, fast;
  int xs;                  // first output column of the strip
  int ys, ye;              // output rows of the segment
  int y_first, y_begin, y_end;
};
__device__ __forceinline__ GpGeo gp_geo(const GfGeom& gg) {
  GpGeo g;
  g.W = gg.W; g.H = gg.H; g.Wp = gg.Wp; g.r = gg.r; g.rho = gg.r >> 2; g.HL = gg.HL; g.SW = gg.SW; g.NQ = gg.NQ; g.fast = gg.fast;
  g.xs = blockIdx.x * gg.SW;
  g.ys = blockIdx.y * gg.seg_h; g.ye = min(g.ys + gg.seg_h, gg.H);
  g.y_first = max(g.ys - gg.r, 0);
  g.y_begin = g.ys - gg.r; g.y_end = g.ye + gg.r;
  return g;
}

// ------------------------------------------------------------------------------------------------
// ACC role
// ------------------------------------------------------------------------------------------------
template <class P>
__device__ __forceinline__ void gp_acc_worker(const GfCommon& gc, const GfGeom& gg, unsigned char* smem) {
  constexpr int NI = P::NI, ND = P::ND, NT = GP_NT, GP = GP_GP, NSTAGE = P::NSTAGE;
  constexpr int NIa = NI > 0 ? NI : 1;
  typedef GpSmem<P> L;
  typedef typename P::Acc Acc;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  unsigned char* stage_in = smem + L::off_in;
  const GpGeo g = gp_geo(gg);
  const int t = threadIdx.x - GP_SOLVE_THREADS;
  const int gx = g.xs - g.HL - 4 + 4 * t;     // image column of this thread's quad (multiple of 4)
  const int tdp = gp_dpos(t);                 // position of its quad total in an fp64 quad-total row
  const bool qact = t < g.NQ;
  unsigned cmask = 0;                         // columns of the quad that are image columns; quad 0 is the zero guard
  if (qact && t > 0) {
#pragma unroll
    for (int c = 0; c < 4; c++) if (gx + c >= 0 && gx + c < g.W) cmask |= 1u << c;
  }
  const bool qload = cmask != 0;              // then 0 <= gx < Wp: the whole quad is readable
  Acc acc;
  acc.init(gc, blockIdx.z, reinterpret_cast<typename P::Shared*>(smem + L::off_sh), gg);

  uint32_t Vi[4][NIa];
  double Vl[4][ND];
#pragma unroll
  for (int c = 0; c < 4; c++) {
#pragma unroll
    for (int k = 0; k < NIa; k++) Vi[c][k] = 0;
#pragma unroll
    for (int k = 0; k < ND; k++) Vl[c][k] = 0;
  }
  // first quad of this strip that lies inside the padded image (the TMA rows start there)
  const int tA = max(1, (g.HL + 4 - g.xs) >> 2);

  // a-kernels: the raw quads of the next march row land in this thread's own shared-memory slots (cp.async, no register
  // held meanwhile)
  if constexpr (!P::PLANE_READER) {
    const int yl = g.y_begin - 2 * g.r - 1;
    if (qload && g.y_begin >= 0 && g.y_begin < g.H) acc.stage_issue(stage_in, 0, g.y_begin, gx, t);
    if (qload && yl >= g.y_first) acc.stage_issue(stage_in, 1, yl, gx, t);
    cp_async_commit();
  }
  GpRing ring, tring;
  int rows_out = 0;
  for (int yin = g.y_begin; yin < g.y_end; ++yin) {
    const int yli = yin - 2 * g.r - 1;
    const bool enter = (yin >= 0 && yin < g.H), leave = (yli >= g.y_first);
    if constexpr (!P::PLANE_READER) {
      const int yn = yin + 1, yln = yli + 1;
      const int par = (yin - g.y_begin) & 1;
      cp_async_wait_all();
      if (qload && yn < g.y_end) {
        if (yn >= 0 && yn < g.H) acc.stage_issue(stage_in, 2 * (par ^ 1), yn, gx, t);
        if (yln >= g.y_first) acc.stage_issue(stage_in, 2 * (par ^ 1) + 1, yln, gx, t);
      }
      cp_async_commit();
      typename Acc::Raw rw;
      if (qload && enter) {
        acc.stage_read(stage_in, 2 * par, rw, t);
        if (cmask == 0xfu) acc.template accum<+1, true>(rw, cmask, Vi, Vl);  // whole quad inside the image: straight-line code
        else acc.template accum<+1, false>(rw, cmask, Vi, Vl);
      }
      if (qload && leave) {
        acc.stage_read(stage_in, 2 * par + 1, rw, t);
        if (cmask == 0xfu) acc.template accum<-1, true>(rw, cmask, Vi, Vl);
        else acc.template accum<-1, false>(rw, cmask, Vi, Vl);
      }
    } else {
      // the entering and the leaving coefficient row of this march row sit in slot `tring.s` of the TMA ring (auxiliary warp 0)
      mbar_wait_park(bars + GPB_TFULL + tring.s, tring.ph);
      if (qload && (enter || leave)) {
        const int4* slot = reinterpret_cast<const int4*>(stage_in) + ((size_t)tring.s * 2 * GP_NTR + (t - tA)) * P::NP;
        acc.accum_staged(slot, slot + (size_t)GP_NTR * P::NP, gx >> 2, enter, leave, cmask, Vl);
      }
      mbar_arrive(bars + GPB_TEMPTY + tring.s);
      tring.template next<P::NRING>();
    }
    if (yin - g.r >= g.ys) {
      if (rows_out >= NSTAGE) mbar_wait_park(bars + GPB_EMPTY + ring.s, ring.ph ^ 1u);  // SOLVE has left the row that used this stage
      rows_out++;
      const GpStage st = gp_stage<P>(smem, ring.s);
      if (qact) {
#pragma unroll
        for (int k = 0; k < NI; k++) {
          uint32_t p0 = Vi[0][k], p1 = p0 + Vi[1][k], p2 = p1 + Vi[2][k], p3 = p2 + Vi[3][k];
          st.Pi[k * NT + t] = make_uint4(p0, p1, p2, p3);
          st.Gi[k * GP + t] = p3;
        }
#pragma unroll
        for (int k = 0; k < ND; k++) {
          const double p0 = Vl[0][k], p1 = p0 + Vl[1][k], p2 = p1 + Vl[2][k], p3 = p2 + Vl[3][k];
          if constexpr (GP_EVEN_ODD(ND)) {
            st.Pa[k * NT + t] = make_double2(p0, p2);   // even elements
            st.Pb[k * NT + t] = make_double2(p1, p3);   // odd elements
          } else {
            st.Pa[k * NT + t] = make_double2(p0, p1);
            st.Pb[k * NT + t] = make_double2(p2, p3);
          }
          st.Gd[k * GP_GPD + tdp] = p3;
        }
      }
      mbar_arrive(bars + GPB_FULL + ring.s);
      ring.template next<NSTAGE>();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// AUX role: prefix over the quad totals of every published row; TMA producer of the plane readers
// ------------------------------------------------------------------------------------------------
template <class P>
__device__ __forceinline__ void gp_aux(const GfCommon& gc, const GfGeom& gg, unsigned char* smem) {
  constexpr int NI = P::NI, ND = P::ND, GP = GP_GP, NSTAGE = P::NSTAGE;
  constexpr int NIa = NI > 0 ? NI : 1;
  typedef GpSmem<P> L;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  const GpGeo g = gp_geo(gg);
  const int lane = threadIdx.x & 31;
  const int aw = (threadIdx.x - GP_SOLVE_THREADS - GP_NT) >> 5;   // 0..GP_NAUX-1
  const int tA = max(1, (g.HL + 4 - g.xs) >> 2), tB = min(g.NQ, (g.Wp - g.xs + g.HL + 4) >> 2);
  uint64_t pol_enter = 0, pol_leave = 0;
  if constexpr (P::PLANE_READER) { pol_enter = l2_policy_evict_last(P::L2_FRAC); pol_leave = l2_policy_evict_first(); }
  (void)pol_enter; (void)pol_leave;
  auto tma_rows = [&](int yi, int j) {   // march row yi into ring slot j
    if constexpr (P::PLANE_READER) {
      if (yi >= g.y_end) return;
      const int yli = yi - 2 * g.r - 1;
      const bool en = (yi >= 0 && yi < g.H), le = (yli >= g.y_first);
      const unsigned row_bytes = (unsigned)(tB - tA) * 16u * P::NP;
      uint64_t* bar = bars + GPB_TFULL + j;
      mbar_arrive_expect_tx(bar, ((en ? 1u : 0u) + (le ? 1u : 0u)) * row_bytes);
      int4* slot = reinterpret_cast<int4*>(smem + L::off_in) + (size_t)j * 2 * GP_NTR * P::NP;
      const int gqa = (g.xs - g.HL - 4 + 4 * tA) >> 2;   // global quad index of strip quad tA
      const int4* rows = reinterpret_cast<const int4*>(P::coef_rows(gc, blockIdx.z, gg));
      const size_t qpr = (size_t)(g.Wp >> 2);
      if (en) tma_bulk_g2s_hint(slot, rows + ((size_t)yi * qpr + gqa) * P::NP, row_bytes, bar, pol_enter);
      if (le) tma_bulk_g2s_hint(slot + (size_t)GP_NTR * P::NP, rows + ((size_t)yli * qpr + gqa) * P::NP, row_bytes, bar, pol_leave);
    }
  };
  GpRing ring, tring;
  if constexpr (P::PLANE_READER) {
    if (aw == 0 && lane == 0) {
      for (int j = 0; j < P::NRING; j++) tma_rows(g.y_begin + j, j);
    }
  }
  for (int yin = g.y_begin; yin < g.y_end; ++yin) {
    if constexpr (P::PLANE_READER) {
      // the ring slot of march row yin is free once every worker has consumed it: request row yin + NRING into it
      if (aw == 0) {
        if (yin + P::NRING < g.y_end) {
          mbar_wait_park(bars + GPB_TEMPTY + tring.s, tring.ph);
          if (lane == 0) tma_rows(yin + P::NRING, tring.s);
        }
        tring.template next<P::NRING>();
      }
    }
    if (yin - g.r < g.ys) continue;
    mbar_wait_park(bars + GPB_FULL + ring.s, ring.ph);
    const GpStage st = gp_stage<P>(smem, ring.s);
    // four moments per round (8 lanes each, GP_SEGQ quads per lane); the rounds are dealt out over the auxiliary warps
    const int seg = lane & 7, mq = lane >> 3;
    constexpr int RI = (NI + 3) / 4, RD = (ND + 3) / 4;
#pragma unroll
    for (int rd = 0; rd < RI + RD; rd++) {
      if (rd % GP_NAUX != aw) continue;
      if (rd < RI) { const int k0 = 4 * rd; gp_scan_task<uint32_t, uint4>(st.Gi + min(k0 + mq, NIa - 1) * GP, seg, k0 + mq < NI); }
      else { const int k0 = 4 * (rd - RI); gp_scan_task<double, double2>(st.Gd + min(k0 + mq, ND - 1) * GP_GPD, seg, k0 + mq < ND); }
    }
    mbar_arrive(bars + GPB_READY + ring.s);
    ring.template next<NSTAGE>();
  }
}

// ------------------------------------------------------------------------------------------------
// SOLVE role
// ------------------------------------------------------------------------------------------------
// window sums of one pixel pair (half h of strip quad tq) from the published row
template <class P>
__device__ __forceinline__ void gp_window_pair(const GpStage& st, const GpGeo& g, int tq, int h, uint32_t (&si)[2][P::NI > 0 ? P::NI : 1],
                                               double (&sd)[2][P::ND]) {
  constexpr int NI = P::NI, ND = P::ND, NT = GP_NT, GP = GP_GP;
  if (g.fast) {
    const int tlo = tq - g.rho, thi = tq + g.rho;
    const int dhi = gp_dpos(thi - 1), dlo = gp_dpos(tlo - 1);   // loop invariants of the caller's row loop
#pragma unroll
    for (int k = 0; k < NI; k++) {
      const uint32_t Wq = st.Gi[k * GP + thi - 1] - st.Gi[k * GP + tlo - 1];
      const uint32_t* pl = reinterpret_cast<const uint32_t*>(st.Pi + k * NT + tlo);
      const uint2 b = reinterpret_cast<const uint2*>(st.Pi + k * NT + thi)[h];
      const uint32_t a0 = pl[h], a1 = pl[2 * h];   // h = 0: (unused, a.x)   h = 1: (a.y, a.z)
      si[0][k] = Wq - (h ? a0 : 0u) + b.x;
      si[1][k] = Wq - a1 + b.y;
    }
    // pixel c of the quad: (G[thi-1] - G[tlo-1]) - p_tlo[c-1] + p_thi[c].  This thread has c = 2h, 2h+1: the pair of quad thi is
    // one 16-byte load, p_tlo[2h] one 8-byte load, and p_tlo[2h-1] is p_tlo[1] for h = 1 and element 0 of quad 0 - the zero
    // guard of every moment row - for h = 0: the same instructions for both halves, no branch between the moments, all
    // addresses a per-thread base plus a constant (a branch per moment kept the loads of the moments from overlapping)
    if constexpr (GP_EVEN_ODD(ND)) {
      // Pa holds the even elements (p0, p2) of a quad, Pb the odd ones (p1, p3): element 2h of a quad is Pa[quad] component h, so
      // the two halves of a quad read consecutive 8 bytes (an 8-byte load at a 16-byte stride is two-way bank conflicted);
      // six conflict-free 8-byte loads per moment
      const double* ev = reinterpret_cast<const double*>(st.Pa) + h;
      const double* od = reinterpret_cast<const double*>(st.Pb) + h;
      const double* lo0_p = h ? reinterpret_cast<const double*>(st.Pb + tlo) : reinterpret_cast<const double*>(st.Pa);   // p1 of tlo / zero guard
#pragma unroll
      for (int k = 0; k < ND; k++) {
        const double Wq = st.Gd[k * GP_GPD + dhi] - st.Gd[k * GP_GPD + dlo];
        sd[0][k] = (Wq - lo0_p[k * NT * 2]) + ev[(k * NT + thi) * 2];
        sd[1][k] = (Wq - ev[(k * NT + tlo) * 2]) + od[(k * NT + thi) * 2];
      }
    } else {
      // Pa = (p0, p1), Pb = (p2, p3): five loads per moment, the pair of quad thi in one 16-byte load (p_tlo[2h] stays a
      // two-way conflicted 8-byte load; with eight moments the sixth load instruction costs more than the conflict)
      const double2* half = h ? st.Pb : st.Pa;
      const double2* hi_p = half + thi;
      const double* lo1_p = reinterpret_cast<const double*>(half + tlo);
      const double* lo0_p = h ? reinterpret_cast<const double*>(st.Pa + tlo) + 1 : reinterpret_cast<const double*>(st.Pa);
#pragma unroll
      for (int k = 0; k < ND; k++) {
        const double Wq = st.Gd[k * GP_GPD + dhi] - st.Gd[k * GP_GPD + dlo];
        const double2 b = hi_p[k * NT];
        sd[0][k] = (Wq - lo0_p[k * NT * 2]) + b.x;
        sd[1][k] = (Wq - lo1_p[k * NT * 2]) + b.y;
      }
    }
  } else {
    const uint32_t* Pis = reinterpret_cast<const uint32_t*>(st.Pi);
    const double* Pa = reinterpret_cast<const double*>(st.Pa);
#pragma unroll
    for (int cc = 0; cc < 2; cc++) {
      const int z = 4 * tq + 2 * h + cc;
      const int zl = z - g.r, zh = z + g.r + 1;   // window = strip columns [zl, zh)
#pragma unroll
      for (int k = 0; k < NI; k++) {
        uint32_t fl = st.Gi[k * GP + (zl >> 2) - 1] + ((zl & 3) ? Pis[k * NT * 4 + zl - 1] : 0u);
        uint32_t fh = st.Gi[k * GP + (zh >> 2) - 1] + ((zh & 3) ? Pis[k * NT * 4 + zh - 1] : 0u);
        si[cc][k] = fh - fl;
      }
#pragma unroll
      for (int k = 0; k < ND; k++) {
        // prefix element (z&3)-1 of quad z>>2
        const int el = (zl & 3) - 1, eh = (zh & 3) - 1;
        // element e of a quad: even / odd layout: array e & 1, component e / 2; pair layout: array e / 2, component e & 1
        const double* Pb = reinterpret_cast<const double*>(st.Pb);
        constexpr bool EO = GP_EVEN_ODD(ND);
        double pl = (el < 0) ? 0.0 : (((EO ? (el & 1) : (el >> 1)) ? Pb : Pa)[(k * NT + (zl >> 2)) * 2 + (EO ? (el >> 1) : (el & 1))]);
        double ph = (eh < 0) ? 0.0 : (((EO ? (eh & 1) : (eh >> 1)) ? Pb : Pa)[(k * NT + (zh >> 2)) * 2 + (EO ? (eh >> 1) : (eh & 1))]);
        sd[cc][k] = (st.Gd[k * GP_GPD + gp_dpos((zh >> 2) - 1)] + ph) - (st.Gd[k * GP_GPD + gp_dpos((zl >> 2) - 1)] + pl);
      }
    }
  }
}

template <class P>
__device__ __forceinline__ void gp_solve(const GfCommon& gc, const GfGeom& gg, unsigned char* smem) {
  constexpr int NI = P::NI, ND = P::ND, NSTAGE = P::NSTAGE;
  constexpr int NIa = NI > 0 ? NI : 1;
  typedef GpSmem<P> L;
  typedef typename P::Solve Solve;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  const GpGeo g = gp_geo(gg);
  const int v = threadIdx.x;                    // 0..255
  const int h = v & 1;                          // which half of the quad
  const int q = v >> 1;                         // output quad of the strip
  const int tq = g.HL / 4 + 1 + q;              // its strip quad
  const int gx = g.xs + 4 * q + 2 * h;          // image column of the first pixel
  const bool act = (q < g.SW / 4) && (gx < g.W);
  const bool second = gx + 1 < g.W;
  const int nx0 = min(gx + g.r, g.W - 1) - max(gx - g.r, 0) + 1;
  const int nx1 = max(min(gx + 1 + g.r, g.W - 1) - max(gx + 1 - g.r, 0) + 1, 1);
  Solve sol;
  sol.init(gc, blockIdx.z, reinterpret_cast<typename P::Shared*>(smem + L::off_sh), gg);
  // policies with SOLVE_FIELDS > 0: the per-pixel inputs of SOLVE (packed guide, J) are requested two rows ahead - one row
  // (about 1 us) did not cover the DRAM latency under load: a fifth of the SOLVE samples of GF2b waited on the first use of
  // the prefetched word.  They land in this thread's own slots of a three-row staging ring in shared memory (cp.async): no
  // register is tied to a load in flight, and no barrier is needed (the thread reads back only what it requested itself)
  unsigned char* sin = smem + L::off_sin + (size_t)v * 8;
  constexpr int SLOT = P::SOLVE_FIELDS * GP_SOLVE_THREADS * 8;
  if constexpr (P::SOLVE_FIELDS > 0) {
    if (act) sol.row_prefetch(g.ys, gx, sin);
    cp_async_commit();
    if (act && g.ys + 1 < g.ye) sol.row_prefetch(g.ys + 1, gx, sin + SLOT);
    cp_async_commit();
  } else {
    if (act) sol.row_prefetch(g.ys, gx, nullptr);   // register prefetch, one row ahead
  }
  int slot = 0;
  GpRing ring;
  // All eight warps work on the same row.  Two alternatives were built and measured slower (profiles/r2_summary.md): the
  // window sums of the next row requested before the per-pixel work of this one (software pipeline over rows), and two
  // groups of four warps on alternate rows with two pixel pairs per thread.
  for (int yo = g.ys; yo < g.ye; ++yo) {
    mbar_wait_park(bars + GPB_READY + ring.s, ring.ph);
    uint32_t si[2][NIa];
    double sd[2][ND];
    if (act) gp_window_pair<P>(gp_stage<P>(smem, ring.s), g, tq, h, si, sd);
    mbar_arrive(bars + GPB_EMPTY + ring.s);   // everything this thread needs of the stage is in registers
    ring.template next<NSTAGE>();
    if (act) {
      if constexpr (P::SOLVE_FIELDS > 0) {
        const int s2 = slot >= 1 ? slot - 1 : 2;   // (slot + 2) % 3
        if (yo + 2 < g.ye) sol.row_prefetch(yo + 2, gx, sin + s2 * SLOT);
        cp_async_commit();
        cp_async_wait_2();
        sol.row_pickup(sin + slot * SLOT);
        slot = slot == 2 ? 0 : slot + 1;
      } else {
        sol.row_pickup(nullptr);
        if (yo + 1 < g.ye) sol.row_prefetch(yo + 1, gx, nullptr);
      }
      const int ny = min(yo + g.r, g.H - 1) - max(yo - g.r, 0) + 1;
      // both pixels in straight-line code (no branch between them: the scheduler interleaves the two dependent chains);
      // the second one is a pad column only in the last pair of an odd-width image: computed, not stored / reduced
      sol.column(0, yo, gx, ny * nx0, si[0], sd[0], true);
      sol.column(1, yo, gx + 1, ny * nx1, si[1], sd[1], second);
      sol.store_pair(yo, gx, second);
    }
  }
  sol.finish();
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
// register budget of the calling warpgroup; the kernel starts with GP_LAUNCH_REGS for every thread
constexpr int GP_LAUNCH_REGS = 128;   // 65536 / GP_THREADS
template <int R>
__device__ __forceinline__ void gp_set_regs() {
  if constexpr (R > GP_LAUNCH_REGS) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R));
  else if constexpr (R < GP_LAUNCH_REGS) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R));
}

template <class P>
__global__ void __launch_bounds__(GP_THREADS, 1) gp_kernel(GfCommon gc, GfGeom gg) {
  typedef GpSmem<P> L;
  static_assert((GP_NARROW ? GP_NT * P::ACC_REGS + 32 * GP_NAUX * GP_AUX_REGS : GP_ACC_THREADS * P::ACC_REGS) + GP_SOLVE_THREADS * P::SOLVE_REGS <=
                        GP_THREADS * GP_LAUNCH_REGS && P::SOLVE_REGS <= 255 && P::ACC_REGS <= 255 && P::NSTAGE >= 2 && P::NSTAGE <= 4,
                "register pool / ring");
  static_assert(!GP_NARROW || (GP_NT == 128 && GP_NAUX == 4), "narrow layout: one warpgroup of ACC workers, one of auxiliary warps");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L::off_bar);
  const int t = threadIdx.x;
  // the quad-total rows are scanned over their whole length: keep the unused tail finite
  for (int s = 0; s < P::NSTAGE; s++) {
    const GpStage st = gp_stage<P>(smem_raw, s);
    for (int i = t; i < GP_GP; i += GP_THREADS) {
#pragma unroll
      for (int k = 0; k < P::NI; k++) st.Gi[k * GP_GP + i] = 0u;
#pragma unroll
      for (int k = 0; k < P::ND; k++) st.Gd[k * GP_GPD + i] = 0.0;
    }
    for (int i = GP_GP + t; i < GP_GPD; i += GP_THREADS) {
#pragma unroll
      for (int k = 0; k < P::ND; k++) st.Gd[k * GP_GPD + i] = 0.0;
    }
  }
  if (t == 0) {
    for (int s = 0; s < P::NSTAGE; s++) {
      mbar_init(bars + GPB_FULL + s, GP_NT);
      mbar_init(bars + GPB_READY + s, 32 * GP_NAUX);
      mbar_init(bars + GPB_EMPTY + s, GP_SOLVE_THREADS);
    }
    for (int s = 0; s < 4; s++) {
      mbar_init(bars + GPB_TFULL + s, 1);
      mbar_init(bars + GPB_TEMPTY + s, GP_NT);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  P::init_shared(gc, blockIdx.z, reinterpret_cast<typename P::Shared*>(smem_raw + L::off_sh), gg);  // ends with __syncthreads()
  if (t < GP_SOLVE_THREADS) {
    gp_set_regs<P::SOLVE_REGS>();
    gp_solve<P>(gc, gg, smem_raw);
  } else if constexpr (GP_NARROW) {
    if (t < GP_SOLVE_THREADS + GP_NT) {
      gp_set_regs<P::ACC_REGS>();
      gp_acc_worker<P>(gc, gg, smem_raw);
    } else {
      gp_set_regs<GP_AUX_REGS>();
      gp_aux<P>(gc, gg, smem_raw);
    }
  } else {
    gp_set_regs<P::ACC_REGS>();
    if (t < GP_SOLVE_THREADS + GP_NT) gp_acc_worker<P>(gc, gg, smem_raw);
    else gp_aux<P>(gc, gg, smem_raw);
  }
}

// ------------------------------------------------------------------------------------------------
// policies
// ------------------------------------------------------------------------------------------------
// 1 / (pixels in the window) of the two pixels of a SOLVE thread: the count changes only in the first and last r rows of the
// image, so the a-kernels keep the reciprocal (MUFU seed + two Newton steps) from row to row (in the plane readers the
// branch costs more than it saves: it breaks the straight-line interleave of the two pixels)
struct GpInvN {
  int n[2]; double inv[2];
  __device__ __forceinline__ GpInvN() { n[0] = n[1] = 0; inv[0] = inv[1] = 0.0; }
  __device__ __forceinline__ double get(int cc, int Ncnt) {
    if (Ncnt != n[cc]) { n[cc] = Ncnt; inv[cc] = rcp_fast(u2d((uint32_t)Ncnt)); }
    return inv[cc];
  }
};

// 3x3 symmetric solve for one right-hand side; the signal sums carry the 2^pbits scale of the fixed-point signal,
// rdetP = pinv / det(M) takes it out of a, the product with pinv = 2^-pbits out of b.
__device__ __forceinline__ void gp_solve_rhs(const double* A, double rdetP, const double* Sd, double N, double invN, double pinv, double Sp,
                                             const double* Sip, double* a, double& b) {
  double C0 = fma(N, Sip[0], -Sd[0] * Sp), C1 = fma(N, Sip[1], -Sd[1] * Sp), C2 = fma(N, Sip[2], -Sd[2] * Sp);
  a[0] = (C0 * A[0] + C1 * A[1] + C2 * A[2]) * rdetP;
  a[1] = (C0 * A[1] + C1 * A[3] + C2 * A[4]) * rdetP;
  a[2] = (C0 * A[2] + C1 * A[4] + C2 * A[5]) * rdetP;
  b = (fma(Sp, pinv, -a[0] * Sd[0]) - a[1] * Sd[1] - a[2] * Sd[2]) * invN;
}
__device__ __forceinline__ int4 coef_pack_fix(const double* a, double b, double sa, double sb) {
  return make_int4(__double2int_rn(a[0] * sa), __double2int_rn(a[1] * sa), __double2int_rn(a[2] * sa), __double2int_rn(b * sb));
}

// GF1a: guide = normI (k units), p = max(t_blue, tmin) and max(t_green, tmin) (BGDehaze.py:39-48, guidedfilter.py:62-93)
struct PipGF1a {
  static constexpr int NI = 9, ND = 8, NSTAGE = 3, ACC_REGS = GP_GF1A_ACC_REGS, SOLVE_REGS = GP_SOLVE_REGS_FOR(GP_GF1A_ACC_REGS);
  static constexpr bool PLANE_READER = false;
  static constexpr int IN_BYTES = 4 * GP_NT * 20;   // per worker: 4 cp.async slots (2 buffers x enter / leave) of one uint4 + one u32
  static constexpr int SOLVE_FIELDS = 0;   // 8-byte words of per-pixel-pair input SOLVE reads per row (staged by cp.async)
  struct Shared {
    double pT[2][256];    // rint(p_c * 2^28) as a function of the window-min k' (an exact integer-valued double)
    FrameConst fc;
    double epsN_k;        // eps * range^2
    double pinv;          // 2^-pbits
    CoefScale cs;
  };
  static __device__ void init_shared(const GfCommon& g, int f, Shared* sh, const GfGeom& gg) {
    if (threadIdx.x == 0) load_frame_const(g.fs[f], sh->fc);
    __syncthreads();
    const double range = (double)sh->fc.range;
    for (int i = threadIdx.x; i < 512; i += blockDim.x) {
      const int c = i >> 8, k = i & 255;
      double t = 1.0 - ((double)k / range) / sh->fc.Bt[c];     // transmission_map (BGDehaze.py:35-36)
      double p = (t < g.tmin) ? g.tmin : t;                      // np.maximum(t, tmin): NaN stays NaN
      // p is NaN only for 0/0 (k' = 0 with B_c = 0) or a constant frame; k' = 0 occurs in every frame (the zero
      // padding of transmission_map reaches every border pixel), so the NaN always reaches the sums: flag the frame
      if (!(p == p)) { p = 0.0; if (blockIdx.x == 0 && blockIdx.y == 0) atomicOr(&g.fs[f].nan_flag, 1u); }
      sh->pT[c][k] = rint(fmin(p, GP_T_PMAX) * GP_PSCALE);   // tmin <= 1 is checked on the host
    }
    if (threadIdx.x == 0) {
      sh->epsN_k = g.eps * range * range; sh->cs = coef_scale(g.eps, range);
      sh->pinv = GP_PINV;
    }
    __syncthreads();
  }
  struct Acc {
    struct Raw { uint4 k; uint32_t m; };
    const Shared* sh; int Wp;
    const uint32_t* kq; const uint8_t* mg;
    __device__ __forceinline__ void init(const GfCommon& g, int f, Shared* s, const GfGeom& gg) {
      sh = s; Wp = gg.Wp;
      const size_t n_pp = (size_t)gg.Wp * gg.H;
      kq = g.kq + (size_t)f * n_pp;
      mg = g.mg + (size_t)f * n_pp;
    }
    // staging slot s (0..3 = 2 buffers x enter / leave) of worker t: one uint4 + one u32, filled by cp.async
    __device__ __forceinline__ void stage_issue(unsigned char* st, int s, int y, int gx, int t) const {
      const size_t o = (size_t)y * Wp + gx;
      cp_async16(st + ((size_t)s * GP_NT + t) * 16, kq + o);
      cp_async4(st + (size_t)4 * GP_NT * 16 + ((size_t)s * GP_NT + t) * 4, mg + o);
    }
    __device__ __forceinline__ void stage_read(const unsigned char* st, int s, Raw& r, int t) const {
      r.k = *reinterpret_cast<const uint4*>(st + ((size_t)s * GP_NT + t) * 16);
      r.m = *reinterpret_cast<const uint32_t*>(st + (size_t)4 * GP_NT * 16 + ((size_t)s * GP_NT + t) * 4);
    }
    // The leaving row is the entering row with negated k: every update is one multiply-add in place - IMAD for the 32-bit
    // guide moments, DFMA for the signal moments (k and rint(p 2^28) are integers: products and sums are exact in fp64).
    // A 64-bit integer multiply-add costs three instructions on this machine (IMAD.WIDE + IADD3 + IADD3.X) against one DFMA.
    // Every signal term is an integer below 2^38 and the sums stay below 2^53: exact.
    template <int SIGN, bool FULL>
    __device__ __forceinline__ void accum(const Raw& r, unsigned cmask, uint32_t (&Vi)[4][NI], double (&Vl)[4][ND]) const {
#pragma unroll
      for (int c = 0; c < 4; c++) {
        const uint32_t w = quad_get(r.k, c);
        const int kb = (int)(w & 255u), kg = (int)((w >> 8) & 255u), kr = (int)((w >> 16) & 255u);
        const uint32_t mb = w >> 24, mgv = (r.m >> (8 * c)) & 255u;
        const int sb = SIGN > 0 ? kb : -kb, sg = SIGN > 0 ? kg : -kg, sr = SIGN > 0 ? kr : -kr;
        Vi[c][0] += (uint32_t)sb; Vi[c][1] += (uint32_t)sg; Vi[c][2] += (uint32_t)sr;
        Vi[c][3] += (uint32_t)(sb * kb); Vi[c][4] += (uint32_t)(sb * kg); Vi[c][5] += (uint32_t)(sb * kr);
        Vi[c][6] += (uint32_t)(sg * kg); Vi[c][7] += (uint32_t)(sg * kr); Vi[c][8] += (uint32_t)(sr * kr);
        if (FULL || (cmask & (1u << c))) {
          const double pb = sh->pT[0][mb], pg = sh->pT[1][mgv];
          Vl[c][0] += SIGN > 0 ? pb : -pb; Vl[c][1] += SIGN > 0 ? pg : -pg;
          const double db = (double)sb, dg = (double)sg, dr = (double)sr;
          Vl[c][2] = fma(db, pb, Vl[c][2]); Vl[c][3] = fma(dg, pb, Vl[c][3]); Vl[c][4] = fma(dr, pb, Vl[c][4]);
          Vl[c][5] = fma(db, pg, Vl[c][5]); Vl[c][6] = fma(dg, pg, Vl[c][6]); Vl[c][7] = fma(dr, pg, Vl[c][7]);
        }
      }
    }
  };
  struct Solve {
    const Shared* sh; int Wp; int32_t* ab;
    GpInvN cinv;
    __device__ __forceinline__ void init(const GfCommon& g, int f, Shared* s, const GfGeom& gg) {
      sh = s; Wp = gg.Wp;
      ab = g.ab + (size_t)f * 8 * (size_t)gg.Wp * gg.H;
    }
    __device__ __forceinline__ void row_prefetch(int, int, unsigned char*) {}
    __device__ __forceinline__ void row_pickup(const unsigned char*) {}
    // results go out pixel by pixel: two 16-byte chunks (one per filter) into the swizzled quad block
    __device__ __forceinline__ void column(int cc, int y, int x, int Ncnt, const uint32_t* si, const double* sd, bool valid) {
      const double N = u2d((uint32_t)Ncnt), invN = cinv.get(cc, Ncnt);
      double M[6], Sd[3], A[6], rdet;
      gf_build_M(si, N, sh->epsN_k * N * N, M, Sd);
      gf_adjugate(M, A, rdet);
      const double pinv = sh->pinv;
      rdet *= pinv;
      double a0[3], b0, a1[3], b1;
      const int gq = x >> 2, c = x & 3;
      int4* blk = reinterpret_cast<int4*>(ab) + ((size_t)y * (Wp >> 2) + gq) * 8;
      gp_solve_rhs(A, rdet, Sd, N, invN, pinv, sd[0], sd + 2, a0, b0);
      gp_solve_rhs(A, rdet, Sd, N, invN, pinv, sd[1], sd + 5, a1, b1);
      if (valid) {
        blk[coef_chunk<8>(gq, c, 0)] = coef_pack_fix(a0, b0, sh->cs.sa, sh->cs.sb);
        blk[coef_chunk<8>(gq, c, 1)] = coef_pack_fix(a1, b1, sh->cs.sa, sh->cs.sb);
      }
    }
    __device__ __forceinline__ void store_pair(int, int, bool) {}
    __device__ __forceinline__ void finish() {}
  };
};

// GF2a: guide = normYiCrCb (k units), p = S (BGDehaze.py:83-84)
struct PipGF2a {
  static constexpr int NI = 9, ND = 4, NSTAGE = 3, ACC_REGS = GP_GF2A_ACC_REGS, SOLVE_REGS = GP_SOLVE_REGS_FOR(GP_GF2A_ACC_REGS);
  static constexpr bool PLANE_READER = false;
  static constexpr int IN_BYTES = 4 * GP_NT * 32;
  static constexpr int SOLVE_FIELDS = 0;   // 8-byte words of per-pixel-pair input SOLVE reads per row (staged by cp.async)
  struct Shared { FrameConst fc; double epsN_k, pinv; CoefScale cs; };
  static __device__ void init_shared(const GfCommon& g, int f, Shared* sh, const GfGeom& gg) {
    if (threadIdx.x == 0) {
      load_frame_const(g.fs[f], sh->fc);
      const double rng = (double)sh->fc.yi_rng;
      sh->epsN_k = g.eps * rng * rng;
      sh->cs = coef_scale(g.eps, rng);
      sh->pinv = GP_PINV;
    }
    __syncthreads();
  }
  struct Acc {
    struct Raw { uint4 y; uint4 s; };
    int Wp; const uint32_t* ycc; const uint32_t* sp;
    uint32_t ysub;   // (yi_min, yi_min, yi_min, yj_min): no byte can borrow
    __device__ __forceinline__ void init(const GfCommon& g, int f, Shared* s, const GfGeom& gg) {
      Wp = gg.Wp;
      const size_t n_pp = (size_t)gg.Wp * gg.H;
      ycc = g.ycc + (size_t)f * n_pp;
      sp = g.splane + (size_t)f * n_pp;
      const uint32_t a = (uint32_t)s->fc.yi_min, b = (uint32_t)s->fc.yj_min;
      ysub = a | (a << 8) | (a << 16) | (b << 24);
    }
    __device__ __forceinline__ void stage_issue(unsigned char* st, int s, int y, int gx, int t) const {
      const size_t o = (size_t)y * Wp + gx;
      // (32 bytes per worker: splitting the two quads into two arrays, 16 bytes apart per worker, measured 2 % slower)
      cp_async16(st + ((size_t)s * GP_NT + t) * 32, ycc + o);
      cp_async16(st + ((size_t)s * GP_NT + t) * 32 + 16, sp + o);
    }
    __device__ __forceinline__ void stage_read(const unsigned char* st, int s, Raw& r, int t) const {
      r.y = *reinterpret_cast<const uint4*>(st + ((size_t)s * GP_NT + t) * 32);
      r.s = *reinterpret_cast<const uint4*>(st + ((size_t)s * GP_NT + t) * 32 + 16);
    }
    template <int SIGN, bool FULL>
    __device__ __forceinline__ void accum(const Raw& r, unsigned cmask, uint32_t (&Vi)[4][NI], double (&Vl)[4][ND]) const {
#pragma unroll
      for (int c = 0; c < 4; c++) {
        if (FULL || (cmask & (1u << c))) {
          const uint32_t w = quad_get(r.y, c) - ysub;
          const int g0 = (int)(w & 255u), g1 = (int)((w >> 8) & 255u), g2 = (int)((w >> 16) & 255u);
          const double S = u2d(quad_get(r.s, c));   // rint(S 2^28) < 2^29
          const int s0 = SIGN > 0 ? g0 : -g0, s1 = SIGN > 0 ? g1 : -g1, s2 = SIGN > 0 ? g2 : -g2;
          Vi[c][0] += (uint32_t)s0; Vi[c][1] += (uint32_t)s1; Vi[c][2] += (uint32_t)s2;
          Vi[c][3] += (uint32_t)(s0 * g0); Vi[c][4] += (uint32_t)(s0 * g1); Vi[c][5] += (uint32_t)(s0 * g2);
          Vi[c][6] += (uint32_t)(s1 * g1); Vi[c][7] += (uint32_t)(s1 * g2); Vi[c][8] += (uint32_t)(s2 * g2);
          Vl[c][0] += SIGN > 0 ? S : -S;
          Vl[c][1] = fma((double)s0, S, Vl[c][1]); Vl[c][2] = fma((double)s1, S, Vl[c][2]); Vl[c][3] = fma((double)s2, S, Vl[c][3]);
        }
      }
    }
  };
  struct Solve {
    const Shared* sh; int Wp; int32_t* ab;
    GpInvN cinv;
    __device__ __forceinline__ void init(const GfCommon& g, int f, Shared* s, const GfGeom& gg) {
      sh = s; Wp = gg.Wp;
      ab = g.ab + (size_t)f * 8 * (size_t)gg.Wp * gg.H;
    }
    __device__ __forceinline__ void row_prefetch(int, int, unsigned char*) {}
    __device__ __forceinline__ void row_pickup(const unsigned char*) {}
    __device__ __forceinline__ void column(int cc, int y, int x, int Ncnt, const uint32_t* si, const double* sd, bool valid) {
      const double N = u2d((uint32_t)Ncnt), invN = cinv.get(cc, Ncnt);
      double M[6], Sd[3], A[6], rdet, a[3], b;
      gf_build_M(si, N, sh->epsN_k * N * N, M, Sd);
      gf_adjugate(M, A, rdet);
      const double pinv = sh->pinv;
      rdet *= pinv;
      gp_solve_rhs(A, rdet, Sd, N, invN, pinv, sd[0], sd + 1, a, b);
      const int gq = x >> 2;
      int4* blk = reinterpret_cast<int4*>(ab) + ((size_t)y * (Wp >> 2) + gq) * 4;
      if (valid) blk[coef_chunk<4>(gq, x & 3, 0)] = coef_pack_fix(a, b, sh->cs.sa, sh->cs.sb);
    }
    __device__ __forceinline__ void store_pair(int, int, bool) {}
    __device__ __forceinline__ void finish() {}
  };
};

// ---- plane readers -------------------------------------------------------------------------------
__device__ __forceinline__ int4 lds128i(unsigned addr) {
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
// add the entering coefficient row to the running sums and drop the leaving one (int32 fixed point summed as doubles: exact)
template <int NP, bool ENTER, bool LEAVE, bool FULL>
__device__ __forceinline__ void gp_accum_coef_case(const int4* be_p, const int4* bl_p, int gq, unsigned cmask, double (&Vl)[4][NP]) {
  // quad blocks are NP*16 bytes and block-aligned, so (logical chunk ^ swizzle) * 16 is the block address with the
  // swizzle folded in, XOR a compile-time constant: one LOP3 per load
  const unsigned swz = (unsigned)coef_chunk<NP>(gq, 0, 0) << 4;
  const unsigned be = (unsigned)__cvta_generic_to_shared(be_p) + swz;
  const unsigned bl = (unsigned)__cvta_generic_to_shared(bl_p) + swz;
#pragma unroll
  for (int c = 0; c < 4; c++) {
#pragma unroll
    for (int j = 0; j < NP / 4; j++) {
      const unsigned q16 = (unsigned)(NP == 8 ? 2 * c + j : c) << 4;
      int4 e = make_int4(0, 0, 0, 0), l = make_int4(0, 0, 0, 0);
      if (ENTER) e = lds128i(be ^ q16);
      if (LEAVE) l = lds128i(bl ^ q16);
      if (FULL || (cmask & (1u << c))) {   // |coefficient| < 2^30: the difference cannot wrap; integer-valued doubles: exact
        Vl[c][4 * j + 0] += (double)(e.x - l.x); Vl[c][4 * j + 1] += (double)(e.y - l.y);
        Vl[c][4 * j + 2] += (double)(e.z - l.z); Vl[c][4 * j + 3] += (double)(e.w - l.w);
      }
    }
  }
}
template <int NP>
__device__ __forceinline__ void gp_accum_coef(const int4* be, const int4* bl, int gq, bool enter, bool leave, unsigned cmask, double (&Vl)[4][NP]) {
  if (enter && leave) {   // steady state (both rows, all four columns inside the image) is the straight-line case
    if (cmask == 0xfu) gp_accum_coef_case<NP, true, true, true>(be, bl, gq, cmask, Vl);
    else gp_accum_coef_case<NP, true, true, false>(be, bl, gq, cmask, Vl);
  } else if (enter) {
    gp_accum_coef_case<NP, true, false, false>(be, bl, gq, cmask, Vl);
  } else if (leave) {
    gp_accum_coef_case<NP, false, true, false>(be, bl, gq, cmask, Vl);
  }
}

// GF1b: q = (box(a).k + box(b))/N for blue and green (guidedfilter.py:99-101) -> J (dehazed_BG, BGDehaze.py:53-56) + reductions
struct PipGF1b {
  // fraction of the entering coefficient rows kept in L2 (evict_last) until they leave the window: 81 rows x 148 strips
  // are 216 MB, keep half of it resident in the 126 MB L2
  static constexpr float L2_FRAC = 0.5f;
  static constexpr int NI = 0, ND = 8, NP = 8, NSTAGE = 2, NRING = 3, ACC_REGS = GP_B_ACC_REGS, SOLVE_REGS = GP_SOLVE_REGS_FOR(GP_B_ACC_REGS);
  static constexpr bool PLANE_READER = true;
  static constexpr int IN_BYTES = NRING * 2 * GP_NTR * NP * 16;   // ring slots x (entering, leaving) row
  static constexpr int SOLVE_FIELDS = 0;   // the one word per row stays a register prefetch (the staged copy measured 5 % slower here)
  struct Shared {
    double inv_range;   // I_c = k / range as k * (1 / range): one ulp from the quotient, far inside J's 1e-5 (a 256-entry table of
                        // the exact quotients cost four bank-conflicted gathers per thread and row)
    FrameConst fc;
    CoefScale cs;
  };
  static __device__ void init_shared(const GfCommon& g, int f, Shared* sh, const GfGeom&) {
    if (threadIdx.x == 0) {
      load_frame_const(g.fs[f], sh->fc); sh->cs = coef_scale(g.eps, (double)sh->fc.range);
      sh->inv_range = 1.0 / (double)sh->fc.range;   // range 0 (constant frame): inf, and 0 * inf = NaN like 0 / 0
    }
    __syncthreads();
  }
  static __device__ __forceinline__ const void* coef_rows(const GfCommon& g, int f, const GfGeom& gg) {
    return g.ab + (size_t)f * 8 * (size_t)gg.Wp * gg.H;
  }
  struct Acc {
    __device__ __forceinline__ void init(const GfCommon&, int, Shared*, const GfGeom&) {}
    __device__ __forceinline__ void accum_staged(const int4* be, const int4* bl, int gq, bool enter, bool leave, unsigned cmask, double (&Vl)[4][ND]) const {
      gp_accum_coef<NP>(be, bl, gq, enter, leave, cmask, Vl);
    }
  };
  struct Solve {
    const Shared* sh; GfCommon g; int W, Wp, H, f;
    const uint32_t* kq; float* J;
    float jmn[2], jmx[2];
    long long jsum[2];   // sum of bits(J*2^32 + 1.5*2^52): exact 2^-32 fixed point, independent of the partition
    unsigned cnt, rmn, rmx, rsum, nanf;
    uint2 knext, kcur;
    float o[2][2];
    double* dbg;   // stage-wise API only: refined t of frame 0
    __device__ __forceinline__ void init(const GfCommon& gc, int frame, Shared* s, const GfGeom& gg) {
      g = gc; sh = s; W = gg.W; Wp = gg.Wp; H = gg.H; f = frame;
      dbg = (frame == 0) ? gc.dbg_tref : nullptr;
      const size_t n_pp = (size_t)Wp * H;
      kq = g.kq + (size_t)f * n_pp;
      J = g.J + (size_t)f * 2 * n_pp;
      jmn[0] = jmn[1] = __int_as_float(0x7f800000); jmx[0] = jmx[1] = -__int_as_float(0x7f800000);
      jsum[0] = jsum[1] = 0;
      cnt = 0; rmn = 255; rmx = 0; rsum = 0; nanf = 0;
      o[0][0] = o[0][1] = o[1][0] = o[1][1] = 0.f;
    }
    __device__ __forceinline__ void row_prefetch(int y, int x, unsigned char*) { knext = __ldg(reinterpret_cast<const uint2*>(kq + (size_t)y * Wp + x)); }
    __device__ __forceinline__ void row_pickup(const unsigned char*) { kcur = knext; }
    __device__ __forceinline__ void column(int cc, int y, int x, int Ncnt, const uint32_t*, const double* sd, bool valid) {
      const double invN = rcp_fast(u2d((uint32_t)Ncnt));
      const uint32_t w = cc ? kcur.y : kcur.x;
      const uint32_t k[3] = {w & 255u, (w >> 8) & 255u, (w >> 16) & 255u};
      const double kd[3] = {u2d(k[0]), u2d(k[1]), u2d(k[2])};
      const double isa = sh->cs.isa * invN, isb = sh->cs.isb * invN;
#pragma unroll
      for (int c = 0; c < 2; c++) {
        const double* s = sd + 4 * c;
        const double q = (s[0] * kd[0] + s[1] * kd[1] + s[2] * kd[2]) * isa + s[3] * isb;   // guidedfilter.py:100-101
        if (dbg && valid) dbg[(size_t)c * W * H + (size_t)y * W + x] = q;
        const double Bc = sh->fc.B[c];
        const double Jv = (kd[c] * sh->inv_range - Bc) * rcp_fast(q) + Bc;            // BGDehaze.py:53,55 (I_c = k / range)
        float Jf = (float)Jv;
        o[cc][c] = Jf;
        if (valid) {
          if (!(fabsf(Jf) < 262144.0f)) { nanf |= 1u; Jf = 0.f; }
          jmn[c] = fminf(jmn[c], Jf);
          jmx[c] = fmaxf(jmx[c], Jf);
          jsum[c] += __double_as_longlong(fma((double)Jf, 4294967296.0, 6755399441055744.0));
        }
      }
      if (valid) {
        cnt++;
        rmn = min(rmn, k[2]); rmx = max(rmx, k[2]); rsum += k[2];
      }
    }
    __device__ __forceinline__ void store_pair(int y, int x, bool second) {
      const size_t n_pp = (size_t)Wp * H, pp = (size_t)y * Wp + x;
      if (!second) { o[1][0] = 0.f; o[1][1] = 0.f; }
      *reinterpret_cast<float2*>(J + pp) = make_float2(o[0][0], o[1][0]);
      *reinterpret_cast<float2*>(J + n_pp + pp) = make_float2(o[0][1], o[1][1]);
    }
    __device__ __forceinline__ void finish() {
      FrameState& s = g.fs[f];
      for (int c = 0; c < 2; c++) {
        float a = warp_min_f32(jmn[c]), b = warp_max_f32(jmx[c]);
        long long sm = warp_sum_i64(jsum[c] - (long long)cnt * __double_as_longlong(6755399441055744.0));
        if ((threadIdx.x & 31) == 0) {
          if (a <= b) {
            atomicMin(&s.jmin_key[c], dkey((double)a));
            atomicMax(&s.jmax_key[c], dkey((double)b));
          }
          atomicAdd((unsigned long long*)&s.jsum_fix[c], (unsigned long long)sm);
        }
      }
      unsigned a = warp_reduce_min_u32(rmn), b = warp_reduce_max_u32(rmx);
      unsigned rs = __reduce_add_sync(0xffffffffu, rsum);
      unsigned nf = __reduce_or_sync(0xffffffffu, nanf);
      if ((threadIdx.x & 31) == 0) {
        atomicMin(&s.rmin, a);
        atomicMax(&s.rmax, b);
        atomicAdd(&s.rsum, (unsigned long long)rs);
        if (nf) atomicOr(&s.nan_flag, nf);
      }
    }
  };
};

// GF2b: refined S -> exposure product -> min / max (BGDehaze.py:84-89)
struct PipGF2b {
  static constexpr float L2_FRAC = 1.0f;   // as PipGF1b: 108 MB, all of it
  static constexpr int NI = 0, ND = 4, NP = 4, NSTAGE = 3, NRING = 4, ACC_REGS = GP_B_ACC_REGS, SOLVE_REGS = GP_SOLVE_REGS_FOR(GP_B_ACC_REGS);
  static constexpr bool PLANE_READER = true;
  static constexpr int IN_BYTES = NRING * 2 * GP_NTR * NP * 16;
  static constexpr int SOLVE_FIELDS = 4;   // 8-byte words of per-pixel-pair input SOLVE reads per row (staged by cp.async)
  struct Shared { ExpShared e; CoefScale cs; };
  static __device__ void init_shared(const GfCommon& g, int f, Shared* sh, const GfGeom& gg) {
    exp_shared_init(&sh->e, g.fs[f], (double)gg.W * (double)gg.H);
    if (threadIdx.x == 0) sh->cs = coef_scale(g.eps, (double)sh->e.fc.yi_rng);
    __syncthreads();
  }
  static __device__ __forceinline__ const void* coef_rows(const GfCommon& g, int f, const GfGeom& gg) {
    return g.ab + (size_t)f * 8 * (size_t)gg.Wp * gg.H;
  }
  struct Acc {
    __device__ __forceinline__ void init(const GfCommon&, int, Shared*, const GfGeom&) {}
    __device__ __forceinline__ void accum_staged(const int4* be, const int4* bl, int gq, bool enter, bool leave, unsigned cmask, double (&Vl)[4][ND]) const {
      gp_accum_coef<NP>(be, bl, gq, enter, leave, cmask, Vl);
    }
  };
  struct Solve {
    const Shared* sh; GfCommon g; int Wp, H, f;
    const uint32_t* kq; const uint32_t* ycc; const float* J; float* refS;
    double omn, omx; unsigned nanf;
    uint2 kc, yc; float2 jbc, jgc;
    float o[2];
    __device__ __forceinline__ void init(const GfCommon& gc, int frame, Shared* s, const GfGeom& gg) {
      g = gc; sh = s; Wp = gg.Wp; H = gg.H; f = frame;
      const size_t n_pp = (size_t)Wp * H;
      kq = g.kq + (size_t)f * n_pp;
      ycc = g.ycc + (size_t)f * n_pp;
      J = g.J + (size_t)f * 2 * n_pp;
      refS = g.refS + (size_t)f * n_pp;
      omn = __longlong_as_double(0x7ff0000000000000ll); omx = -omn; nanf = 0;
      o[0] = o[1] = 0.f;
    }
    static constexpr int FLD = GP_SOLVE_THREADS * 8;   // field pitch of a staging slot
    __device__ __forceinline__ void row_prefetch(int y, int x, unsigned char* st) {
      const size_t n_pp = (size_t)Wp * H, p = (size_t)y * Wp + x;
      cp_async8(st, kq + p);
      cp_async8(st + FLD, ycc + p);
      cp_async8(st + 2 * FLD, J + p);
      cp_async8(st + 3 * FLD, J + n_pp + p);
    }
    __device__ __forceinline__ void row_pickup(const unsigned char* st) {
      kc = *reinterpret_cast<const uint2*>(st); yc = *reinterpret_cast<const uint2*>(st + FLD);
      jbc = *reinterpret_cast<const float2*>(st + 2 * FLD); jgc = *reinterpret_cast<const float2*>(st + 3 * FLD);
    }
    __device__ __forceinline__ void column(int cc, int, int, int Ncnt, const uint32_t*, const double* sd, bool valid) {
      const double invN = rcp_fast(u2d((uint32_t)Ncnt));
      const uint32_t yw = cc ? yc.y : yc.x;
      const uint32_t ymin = (uint32_t)sh->e.fc.yi_min;
      const double g0 = u2d((yw & 255u) - ymin), g1 = u2d(((yw >> 8) & 255u) - ymin), g2 = u2d(((yw >> 16) & 255u) - ymin);
      const double q = ((sd[0] * g0 + sd[1] * g1 + sd[2] * g2) * sh->cs.isa + sd[3] * sh->cs.isb) * invN;
      const float qf = (float)q;
      o[cc] = qf;
      const double qr = (double)qf;
      const double rb = norm_j_fast(cc ? jbc.y : jbc.x, sh->e.fc, 0), rg = norm_j_fast(cc ? jgc.y : jgc.x, sh->e.fc, 1);
      const double rr = sh->e.rt.redN[((cc ? kc.y : kc.x) >> 16) & 255u];
      // min / max over the three channels of restored * refinedS
      const double o0 = rb * qr, o1 = rg * qr, o2 = rr * qr;
      const double os = (o0 + o1) + o2;
      if (!valid) {}
      else if (!(os == os) || fabs(os) > 1.0e300) { nanf = 1u; }  // any NaN / inf poisons the sum
      else {  // plain compare-selects: no NaN in here, fmin/fmax would pay for their NaN rules
        double lo = o0 < o1 ? o0 : o1, hi = o0 < o1 ? o1 : o0;
        lo = o2 < lo ? o2 : lo; hi = o2 > hi ? o2 : hi;
        omn = lo < omn ? lo : omn;
        omx = hi > omx ? hi : omx;
      }
    }
    __device__ __forceinline__ void store_pair(int y, int x, bool second) {
      if (!second) o[1] = 0.f;
      *reinterpret_cast<float2*>(refS + (size_t)y * Wp + x) = make_float2(o[0], o[1]);
    }
    __device__ __forceinline__ void finish() {
      const double a = warp_min_f64(omn), b = warp_max_f64(omx);
      const unsigned nf = __reduce_or_sync(0xffffffffu, nanf);
      if ((threadIdx.x & 31) == 0) {
        if (a <= b) {
          atomicMin(&g.fs[f].omin_key, dkey(a));
          atomicMax(&g.fs[f].omax_key, dkey(b));
        }
        if (nf) atomicOr(&g.fs[f].nan_flag, 1u);
      }
    }
  };
};

// GFq: the filter output itself, q = (box(a).I + box(b))/N (guidedfilter.py:99-101), as a float64 plane: the second half
// of the stand-alone guided_filter stage entry (first half = PipGF2a on a packed 8-bit guide and a fixed-point p)
struct PipGFq {
  static constexpr float L2_FRAC = 1.0f;
  static constexpr int NI = 0, ND = 4, NP = 4, NSTAGE = 3, NRING = 4, ACC_REGS = GP_B_ACC_REGS, SOLVE_REGS = GP_SOLVE_REGS_FOR(GP_B_ACC_REGS);
  static constexpr bool PLANE_READER = true;
  static constexpr int IN_BYTES = NRING * 2 * GP_NTR * NP * 16;
  static constexpr int SOLVE_FIELDS = 1;   // 8-byte words of per-pixel-pair input SOLVE reads per row (staged by cp.async)
  struct Shared { FrameConst fc; CoefScale cs; };
  static __device__ void init_shared(const GfCommon& g, int f, Shared* sh, const GfGeom&) {
    if (threadIdx.x == 0) { load_frame_const(g.fs[f], sh->fc); sh->cs = coef_scale(g.eps, (double)sh->fc.yi_rng); }
    __syncthreads();
  }
  static __device__ __forceinline__ const void* coef_rows(const GfCommon& g, int f, const GfGeom& gg) {
    return g.ab + (size_t)f * 8 * (size_t)gg.Wp * gg.H;
  }
  struct Acc {
    __device__ __forceinline__ void init(const GfCommon&, int, Shared*, const GfGeom&) {}
    __device__ __forceinline__ void accum_staged(const int4* be, const int4* bl, int gq, bool enter, bool leave, unsigned cmask, double (&Vl)[4][ND]) const {
      gp_accum_coef<NP>(be, bl, gq, enter, leave, cmask, Vl);
    }
  };
  struct Solve {
    const Shared* sh; int W, Wp;
    const uint32_t* ycc; double* q_out;
    uint2 yc;
    __device__ __forceinline__ void init(const GfCommon& g, int f, Shared* s, const GfGeom& gg) {
      sh = s; W = gg.W; Wp = gg.Wp;
      ycc = g.ycc + (size_t)f * (size_t)gg.Wp * gg.H;
      q_out = g.dbg_tref + (size_t)f * (size_t)gg.W * gg.H;
    }
    __device__ __forceinline__ void row_prefetch(int y, int x, unsigned char* st) { cp_async8(st, ycc + (size_t)y * Wp + x); }
    __device__ __forceinline__ void row_pickup(const unsigned char* st) { yc = *reinterpret_cast<const uint2*>(st); }
    __device__ __forceinline__ void column(int cc, int y, int x, int Ncnt, const uint32_t*, const double* sd, bool valid) {
      const double invN = rcp_fast(u2d((uint32_t)Ncnt));
      const uint32_t yw = cc ? yc.y : yc.x;
      const uint32_t ymin = (uint32_t)sh->fc.yi_min;
      const double g0 = u2d((yw & 255u) - ymin), g1 = u2d(((yw >> 8) & 255u) - ymin), g2 = u2d(((yw >> 16) & 255u) - ymin);
      if (valid) q_out[(size_t)y * W + x] = ((sd[0] * g0 + sd[1] * g1 + sd[2] * g2) * sh->cs.isa + sd[3] * sh->cs.isb) * invN;
    }
    __device__ __forceinline__ void store_pair(int, int, bool) {}
    __device__ __forceinline__ void finish() {}
  };
};
