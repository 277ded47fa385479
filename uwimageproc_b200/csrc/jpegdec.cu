// jpegdec.cu - batched sequential JPEG decoder whose pixels equal cv2.imdecode(file, IMREAD_COLOR) or
// cv2.imdecode(file, IMREAD_GRAYSCALE) / libjpeg-turbo (SURVEY 8f row N3, the read half of the device path).  The arithmetic is csrc/jpegdec.h; this file spreads it over the GPU.  The
// headers are parsed on the host (the files come from there): per-frame tables and geometry go to the device in one copy, the
// entropy-coded segments, concatenated in a pinned staging buffer, in another.  Then every launch covers all n frames:
//   destuff  a CTA per frame: the segment without the 0x00 after each 0xFF, fill bytes and RST markers, and the byte offset
//            of every restart interval; then the subsequences: each interval is cut into pieces of SUB_BITS bits
//   sync     a thread per subsequence decodes it from an entry state (bit position, block of the MCU, coefficient index) and
//            records its exit state, the first codeword start at or past its end.  An interval's first subsequence starts in
//            the known state, the others guess (block 0, DC); inside a CTA each takes its left neighbour's exit state as its
//            entry until none changes (Weissenberger & Schmidt, ICPP 2018 / HiPC 2021).  The decode of the final round
//            also counts the blocks each subsequence completes and sums its DC differences per component.
//   fixup    a thread per frame walks the CTA boundaries in order and re-decodes from the true exit state until it meets a
//            recorded entry state.  Every loop is bounded by the subsequence count: a stream that never synchronises is
//            decoded sequentially, not wrongly.
//   scan     a CTA per frame: exclusive scans of the counts and DC sums, restarted at each restart interval, give each
//            subsequence its first block and its DC predictors (DC prediction as a segmented scan per component and interval)
//   huff     a thread per subsequence decodes it once more from its true state and writes the int16 coefficients of its
//            blocks in natural order, DC as values
//   idct     a thread per block: jpeg_idct_islow into the padded sample planes
//   color    a thread per output pixel: upsampling with its one-row / one-column context and YCbCr -> B,G,R, cropped to W x H
// Grey output (IMREAD_GRAYSCALE) runs the same passes up to huff; then the idct of the component-0 blocks only and a grey
// pass that crops the Y plane (jdcolor.c grayscale_convert: no chroma IDCT, upsampling or colour conversion).
// The oriented readers apply each frame's Exif orientation (cv2.imdecode's default flags) in the output pass only: the
// oriented pass replaces color / grey with a CTA per 32 x 32 output tile that forms the tile's stored pixels in shared memory
// from rows of the sample planes and writes them out as rows of the output (a column of stored pixels for 5..8).
// Bad entropy-coded data (an invalid code, a coefficient past 63, the data ending before the last block, the wrong number of
// RST markers) leaves the frame all zeros and sets UWIP_FRAME_JPEG_BAD.  A frame's pixels do not depend on the batch it is in.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "jpegdec.h"

namespace {

using jpegdec::Bits;
using jpegdec::DTbl;
using jpegdec::Geo;
using jpegdec::Step;

constexpr int SUB_BITS = 1024;     // bits per subsequence
constexpr int SYNC_T = 128;        // subsequences per CTA of the sync and huff passes
constexpr int CTA_T = 1024;        // destuff and scan passes
constexpr int DESTUFF_BYTES = 16;  // per thread and tile
constexpr int IDCT_T = 128;
constexpr int COLOR_T = 256;
constexpr int TILE = 32;           // output tile edge of the oriented pass

struct FrameTab {
  Geo g;
  uint16_t q[3][64];           // quantisers of the components, natural order
  DTbl dc[3], ac[3];           // decoding tables of the components
  uint64_t seg_off;            // the segment in the staging copy, and its compact stream (16-byte aligned)
  uint64_t seg_len;
  uint64_t blk_off, smp_off;   // first block of the coefficient store, first byte of the sample planes
  uint64_t sub_off, int_off;   // first subsequence slot, first interval slot (nint + 1 of them)
  uint32_t sub_cap;            // subsequence slots (a multiple of SYNC_T)
  int32_t orient;              // Exif orientation applied by the oriented pass, 1..8
};

struct Sub {
  uint32_t start, end, lim;    // bits of the compact stream: the piece, and the end of its restart interval's data
  uint32_t k;                  // restart interval | 1 << 31 for the interval's first piece
};

__host__ __device__ inline uint64_t pack(uint32_t p, int blk, int z) { return ((uint64_t)p << 16) | ((uint64_t)blk << 8) | (uint64_t)z; }

// exclusive prefix sum over the CTA; returns the CTA total
template <class T>
__device__ __forceinline__ T cta_exclusive_scan(T v, T& excl, T* s_warp) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  T x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) s_warp[wid] = x;
  __syncthreads();
  if (wid == 0) {
    T s = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : T(0);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const T y = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += y;
    }
    s_warp[lane] = s;
  }
  __syncthreads();
  excl = x - v + (wid ? s_warp[wid - 1] : T(0));
  const T total = s_warp[(blockDim.x >> 5) - 1];
  __syncthreads();
  return total;
}

__global__ void __launch_bounds__(CTA_T) jpeg_dec_destuff_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ stage,
                                                                   uint8_t* __restrict__ comp, uint32_t* __restrict__ istart,
                                                                   uint32_t* __restrict__ ibase, Sub* __restrict__ subs,
                                                                   int* __restrict__ nsub, int32_t* __restrict__ flags) {
  __shared__ unsigned long long s_warp[32];
  __shared__ unsigned long long s_end;
  const int f = blockIdx.x;
  const FrameTab& t = tabs[f];
  const uint64_t len = t.seg_len;
  const int nint = t.g.nint;
  const uint8_t* seg = stage + t.seg_off;
  uint8_t* cs = comp + t.seg_off;
  uint32_t* ist = istart + t.int_off;
  if (threadIdx.x == 0) s_end = len;
  __syncthreads();
  unsigned long long carry = 0;   // kept bytes | RST markers << 40
  constexpr unsigned long long KEEP = (1ull << 40) - 1;
  uint64_t stop = len;   // the segment ends at the first marker other than RSTn (read once per tile, after the barrier)
  for (uint64_t t0 = 0; t0 < stop; t0 += (uint64_t)DESTUFF_BYTES * CTA_T) {
    const uint64_t i0 = t0 + (uint64_t)DESTUFF_BYTES * threadIdx.x;
    uint8_t v[DESTUFF_BYTES];
    *reinterpret_cast<uint4*>(v) = i0 < len ? *reinterpret_cast<const uint4*>(seg + i0) : make_uint4(0, 0, 0, 0);
    int prev = i0 > 0 && i0 <= len ? seg[i0 - 1] : -1;
    const int after = i0 + DESTUFF_BYTES < len ? seg[i0 + DESTUFF_BYTES] : -1;
    uint8_t kind[DESTUFF_BYTES];
#pragma unroll
    for (int j = 0; j < DESTUFF_BYTES; j++) {
      const uint64_t i = i0 + j;
      kind[j] = 1;
      if (i < len) {
        const int next = j + 1 < DESTUFF_BYTES ? (i + 1 < len ? v[j + 1] : -1) : after;
        kind[j] = (uint8_t)jpegdec::byte_kind(prev, v[j], next);
        if (kind[j] == 3) atomicMin(&s_end, (unsigned long long)i);
      }
      prev = v[j];
    }
    __syncthreads();
    const uint64_t e = s_end;
    unsigned long long cnt = 0;
#pragma unroll
    for (int j = 0; j < DESTUFF_BYTES; j++) {
      if (i0 + j < e) cnt += kind[j] == 0 ? 1ull : (kind[j] == 2 ? 1ull << 40 : 0ull);
    }
    unsigned long long excl;
    const unsigned long long tot = cta_exclusive_scan(cnt, excl, s_warp);
    unsigned long long pos = (carry & KEEP) + (excl & KEEP);
    unsigned long long r = (carry >> 40) + (excl >> 40);
#pragma unroll
    for (int j = 0; j < DESTUFF_BYTES; j++) {
      if (i0 + j < e) {
        if (kind[j] == 0) cs[pos++] = v[j];
        if (kind[j] == 2 && ++r < (unsigned long long)nint) ist[r] = (uint32_t)pos;
      }
    }
    carry += tot;
    stop = e;
  }
  const uint32_t ncomp_bytes = (uint32_t)(carry & KEEP);
  const bool bad = (carry >> 40) != (unsigned long long)(nint - 1);
  if (threadIdx.x == 0) {
    ist[0] = 0;
    ist[nint] = ncomp_bytes;
  }
  __syncthreads();
  if (bad) {   // the wrong number of restart markers
    if (threadIdx.x == 0) {
      nsub[f] = 0;
      atomicOr(flags + f, UWIP_FRAME_JPEG_BAD);
    }
    return;
  }
  // the subsequences: ceil(bits / SUB_BITS) per interval (at least one)
  Sub* sb = subs + t.sub_off;
  uint32_t* ib = ibase + t.int_off;
  unsigned long long carry2 = 0;
  for (int kb = 0; kb < nint; kb += CTA_T) {
    const int k = kb + threadIdx.x;
    unsigned long long nk = 0;
    uint32_t a = 0, b = 0;
    if (k < nint) {
      a = ist[k] * 8u;
      b = ist[k + 1] * 8u;
      nk = b > a ? (b - a + SUB_BITS - 1) / SUB_BITS : 1;
    }
    unsigned long long excl;
    const unsigned long long tot = cta_exclusive_scan(nk, excl, s_warp);
    if (k < nint) {
      const unsigned long long base = carry2 + excl;
      ib[k] = (uint32_t)base;
      for (unsigned long long i = 0; i < nk && base + i < t.sub_cap; i++) {
        Sub s;
        s.start = a + (uint32_t)i * SUB_BITS;
        s.end = s.start + SUB_BITS < b ? s.start + SUB_BITS : b;
        s.lim = b;
        s.k = (uint32_t)k | (i == 0 ? 0x80000000u : 0u);
        sb[base + i] = s;
      }
    }
    carry2 += tot;
  }
  if (threadIdx.x == 0) {
    if (carry2 > t.sub_cap) {
      nsub[f] = 0;
      atomicOr(flags + f, UWIP_FRAME_JPEG_BAD);
    } else {
      nsub[f] = (int)carry2;
    }
  }
}

// decode one subsequence from entry state e: exit state, blocks completed, DC differences per component
__device__ __forceinline__ uint64_t decode_sub(const Geo& g, const DTbl* dc, const DTbl* ac, const uint8_t* cs, const Sub& s, uint64_t e,
                                               int4& cd) {
  Bits b;
  b.init(cs, (uint32_t)(e >> 16));
  int blk = (int)((e >> 8) & 255), z = (int)(e & 255);
  int cnt = 0, d0 = 0, d1 = 0, d2 = 0;
  while (b.p < s.end) {
    const int c = jpegdec::block_comp(g, blk);
    Step st;
    jpegdec::decode_step(dc[c], ac[c], b, z, st);
    if (st.kind == 0) {
      if (c == 0) d0 += st.v;
      else if (c == 1) d1 += st.v;
      else d2 += st.v;
    }
    if (st.done) {
      cnt++;
      z = 0;
      blk = blk + 1 == g.bpm ? 0 : blk + 1;
    }
  }
  cd = make_int4(cnt, d0, d1, d2);
  return pack(b.p, blk, z);
}

__device__ __forceinline__ void load_tables(const FrameTab& t, DTbl* s_dc, DTbl* s_ac) {
  const int nc = t.g.ncomp;
  const int words = (int)(sizeof(DTbl) / 4);
  for (int i = threadIdx.x; i < nc * words; i += blockDim.x) {
    reinterpret_cast<uint32_t*>(s_dc)[i] = reinterpret_cast<const uint32_t*>(t.dc)[i];
    reinterpret_cast<uint32_t*>(s_ac)[i] = reinterpret_cast<const uint32_t*>(t.ac)[i];
  }
  __syncthreads();
}

__global__ void __launch_bounds__(SYNC_T) jpeg_dec_sync_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ comp,
                                                                const Sub* __restrict__ subs, const int* __restrict__ nsub,
                                                                uint64_t* __restrict__ entry, uint64_t* __restrict__ exitst,
                                                                int4* __restrict__ cd, int32_t* __restrict__ stats) {
  __shared__ DTbl s_dc[3], s_ac[3];
  __shared__ uint64_t s_ex[SYNC_T];
  const int f = blockIdx.y;
  const int ns = nsub[f];
  const int j0 = blockIdx.x * SYNC_T;
  if (j0 >= ns) return;
  const FrameTab& t = tabs[f];
  load_tables(t, s_dc, s_ac);
  const Geo g = t.g;
  const uint8_t* cs = comp + t.seg_off;
  const int j = j0 + threadIdx.x;
  const bool active = j < ns;
  Sub s = {0, 0, 0, 0x80000000u};
  if (active) s = subs[t.sub_off + j];
  const bool first = (s.k >> 31) != 0;
  uint64_t e = pack(s.start, 0, 0), ex = 0;
  int4 c4 = make_int4(0, 0, 0, 0);
  int redecodes = 0;
  for (int it = 0; it <= SYNC_T; it++) {
    if (active) ex = decode_sub(g, s_dc, s_ac, cs, s, e, c4);
    s_ex[threadIdx.x] = ex;
    __syncthreads();
    bool changed = false;
    if (active && !first && threadIdx.x > 0 && s_ex[threadIdx.x - 1] != e) {
      e = s_ex[threadIdx.x - 1];
      changed = true;
      redecodes++;
    }
    if (!__syncthreads_or(changed)) break;
  }
  if (active) {
    entry[t.sub_off + j] = e;
    exitst[t.sub_off + j] = ex;
    cd[t.sub_off + j] = c4;
    if (redecodes) atomicAdd(stats + 2 * f, redecodes);
  }
}

__global__ void jpeg_dec_fixup_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ comp, const Sub* __restrict__ subs,
                                      const int* __restrict__ nsub, uint64_t* __restrict__ entry, uint64_t* __restrict__ exitst,
                                      int4* __restrict__ cd, int32_t* __restrict__ stats, int n) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const FrameTab& t = tabs[f];
  const int ns = nsub[f];
  const uint8_t* cs = comp + t.seg_off;
  const uint64_t o = t.sub_off;
  int steps = 0;
  for (int j0 = SYNC_T; j0 < ns; j0 += SYNC_T) {
    for (int j = j0; j < ns; j++) {
      const Sub s = subs[o + j];
      if (s.k >> 31) break;   // an interval starts in the known state
      const uint64_t e = exitst[o + j - 1];
      if (e == entry[o + j]) break;
      int4 c4;
      entry[o + j] = e;
      exitst[o + j] = decode_sub(t.g, t.dc, t.ac, cs, s, e, c4);
      cd[o + j] = c4;
      steps++;
    }
  }
  stats[2 * f + 1] = steps;
}

// first block and DC predictors of every subsequence: scans over the frame's subsequences minus the value at the first
// subsequence of the restart interval
__global__ void __launch_bounds__(CTA_T) jpeg_dec_scan_kernel(const FrameTab* __restrict__ tabs, const Sub* __restrict__ subs,
                                                               const int* __restrict__ nsub, const uint32_t* __restrict__ ibase,
                                                               int4* __restrict__ cd, int4* __restrict__ px) {
  __shared__ int s_warp[32];
  const int f = blockIdx.x;
  const FrameTab& t = tabs[f];
  const int ns = nsub[f];
  const uint64_t o = t.sub_off;
  int4 carry = make_int4(0, 0, 0, 0);
  for (int base = 0; base < ns; base += CTA_T) {
    const int j = base + threadIdx.x;
    const int4 v = j < ns ? cd[o + j] : make_int4(0, 0, 0, 0);
    int4 ex, tot;
    tot.x = cta_exclusive_scan(v.x, ex.x, s_warp);
    tot.y = cta_exclusive_scan(v.y, ex.y, s_warp);
    tot.z = cta_exclusive_scan(v.z, ex.z, s_warp);
    tot.w = cta_exclusive_scan(v.w, ex.w, s_warp);
    if (j < ns) px[o + j] = make_int4(carry.x + ex.x, carry.y + ex.y, carry.z + ex.z, carry.w + ex.w);
    carry = make_int4(carry.x + tot.x, carry.y + tot.y, carry.z + tot.z, carry.w + tot.w);
  }
  __syncthreads();
  const int per_int = t.g.ri ? t.g.ri * t.g.bpm : 0;
  for (int j = threadIdx.x; j < ns; j += CTA_T) {
    const uint32_t k = subs[o + j].k & 0x7fffffffu;
    const int4 p = px[o + j], h = px[o + ibase[t.int_off + k]];
    cd[o + j] = make_int4((int)k * per_int + (p.x - h.x), p.y - h.y, p.z - h.z, p.w - h.w);
  }
}

__global__ void __launch_bounds__(SYNC_T) jpeg_dec_huff_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ comp,
                                                                const Sub* __restrict__ subs, const int* __restrict__ nsub,
                                                                const uint64_t* __restrict__ entry, const int4* __restrict__ cd,
                                                                int16_t* __restrict__ coef, int32_t* __restrict__ flags) {
  __shared__ DTbl s_dc[3], s_ac[3];
  const int f = blockIdx.y;
  const int ns = nsub[f];
  const int j0 = blockIdx.x * SYNC_T;
  if (j0 >= ns) return;
  const FrameTab& t = tabs[f];
  load_tables(t, s_dc, s_ac);
  const int j = j0 + threadIdx.x;
  if (j >= ns) return;
  const Geo g = t.g;
  const Sub s = subs[t.sub_off + j];
  const uint64_t e = entry[t.sub_off + j];
  const int4 c4 = cd[t.sub_off + j];
  const int k = (int)(s.k & 0x7fffffffu);
  const int iend = (g.ri ? min((k + 1) * g.ri, g.nmcu) : g.nmcu) * g.bpm;
  int G = c4.x;
  int pred[3] = {c4.y, c4.z, c4.w};
  int16_t* cf = coef + t.blk_off * 64;
  Bits b;
  b.init(comp + t.seg_off, (uint32_t)(e >> 16));
  int blk = (int)((e >> 8) & 255), z = (int)(e & 255);
  bool bad = false;
  while (G < iend && b.p < s.end) {
    const int c = jpegdec::block_comp(g, blk);
    Step st;
    if (!jpegdec::decode_step(s_dc[c], s_ac[c], b, z, st) || b.p > s.lim) {
      bad = true;
      break;
    }
    if (st.kind == 0) {
      pred[c] += st.v;
      cf[(size_t)G * 64] = (int16_t)pred[c];
    } else if (st.kind == 1) {
      cf[(size_t)G * 64 + jpegdec::natural_order(st.zz)] = (int16_t)st.v;
    }
    if (st.done) {
      G++;
      z = 0;
      blk = blk + 1 == g.bpm ? 0 : blk + 1;
    }
  }
  if (s.end == s.lim && G < iend) bad = true;   // the interval's data ended before its last block
  if (bad) atomicOr(flags + f, UWIP_FRAME_JPEG_BAD);
}

// Y_ONLY: the blocks of component 0 (grey output); the chroma blocks' threads exit
template <bool Y_ONLY>
__global__ void __launch_bounds__(IDCT_T) jpeg_dec_idct_kernel(const FrameTab* __restrict__ tabs, const int16_t* __restrict__ coef,
                                                                uint8_t* __restrict__ smp) {
  __shared__ uint16_t s_q[3][64];
  const int f = blockIdx.y;
  const FrameTab& t = tabs[f];
  for (int i = threadIdx.x; i < 192; i += blockDim.x) s_q[i >> 6][i & 63] = t.q[i >> 6][i & 63];
  __syncthreads();
  const Geo g = t.g;
  const size_t blk = (size_t)blockIdx.x * IDCT_T + threadIdx.x;
  if (blk >= g.nblocks) return;
  const int m = (int)(blk / g.bpm), bi = (int)(blk % g.bpm);
  int c, bx, by;
  jpegdec::block_pos(g, m, bi, c, bx, by);
  if (Y_ONLY && c != 0) return;
  int16_t cb[64];
  const uint4* src = reinterpret_cast<const uint4*>(coef + (t.blk_off + blk) * 64);
#pragma unroll
  for (int i = 0; i < 8; i++) reinterpret_cast<uint4*>(cb)[i] = __ldg(src + i);
  jpegdec::idct_islow(cb, s_q[c], smp + t.smp_off + g.poff[c] + (size_t)8 * by * g.pw[c] + 8 * bx, g.pw[c]);
}

__global__ void __launch_bounds__(COLOR_T) jpeg_dec_color_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ smp,
                                                                  const int32_t* __restrict__ flags, uint8_t* __restrict__ out, int w,
                                                                  int h) {
  const int f = blockIdx.y;
  const size_t i = (size_t)blockIdx.x * COLOR_T + threadIdx.x;
  if (i >= (size_t)w * h) return;
  uint8_t* o = out + ((size_t)f * w * h + i) * 3;
  if (flags[f] & UWIP_FRAME_JPEG_BAD) {
    o[0] = o[1] = o[2] = 0;
    return;
  }
  const FrameTab& t = tabs[f];
  const Geo g = t.g;
  jpegdec::pixel(g, smp + t.smp_off, (int)(i % w), (int)(i / w), o);
}

__global__ void __launch_bounds__(COLOR_T) jpeg_dec_grey_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ smp,
                                                                 const int32_t* __restrict__ flags, uint8_t* __restrict__ out, int w,
                                                                 int h) {
  const int f = blockIdx.y;
  const size_t i = (size_t)blockIdx.x * COLOR_T + threadIdx.x;
  if (i >= (size_t)w * h) return;
  uint8_t* o = out + (size_t)f * w * h + i;
  if (flags[f] & UWIP_FRAME_JPEG_BAD) {
    *o = 0;
    return;
  }
  const FrameTab& t = tabs[f];
  *o = smp[t.smp_off + (i / w) * t.g.pw[0] + i % w];
}

// The output pass of the oriented readers (GREY: the Y plane, else B,G,R), a CTA per TILE x TILE tile of the w x h output.
// The stored pixels the tile shows (the tile, flipped and, for orientations 5..8, transposed) are formed along rows of the
// sample planes into shared memory; then each warp writes a row of the output tile.  Loads and stores stay coalesced for
// every orientation, and the column reads of the transposing orientations hit distinct banks (row pitch TILE + 1 words).
template <bool GREY>
__global__ void __launch_bounds__(COLOR_T) jpeg_dec_oriented_kernel(const FrameTab* __restrict__ tabs, const uint8_t* __restrict__ smp,
                                                                     const int32_t* __restrict__ flags, uint8_t* __restrict__ out,
                                                                     int w, int h, int tiles_x) {
  constexpr int CH = GREY ? 1 : 3, ROWS = COLOR_T / TILE;
  __shared__ uint32_t s_px[TILE][TILE + 1];
  const int f = blockIdx.y;
  const int x0 = (int)(blockIdx.x % tiles_x) * TILE, y0 = (int)(blockIdx.x / tiles_x) * TILE;
  const int tw = min(TILE, w - x0), th = min(TILE, h - y0);
  const int tx = threadIdx.x % TILE, ty = threadIdx.x / TILE;
  const FrameTab& t = tabs[f];
  const int o = t.orient;
  const bool bad = (flags[f] & UWIP_FRAME_JPEG_BAD) != 0;
  int ax, ay, bx, by;   // the stored pixels of two opposite corners: the stored rectangle starts at their minimum
  jpegdec::oriented_src(o, w, h, x0, y0, ax, ay);
  jpegdec::oriented_src(o, w, h, x0 + tw - 1, y0 + th - 1, bx, by);
  const int sx0 = min(ax, bx), sy0 = min(ay, by);
  if (!bad) {
    const int sw = o >= 5 ? th : tw, sh = o >= 5 ? tw : th;
    const Geo g = t.g;
    const uint8_t* p = smp + t.smp_off;
    for (int v = ty; v < sh; v += ROWS) {
      if (tx >= sw) continue;
      uint32_t px;
      if (GREY) {
        px = p[(size_t)(sy0 + v) * g.pw[0] + sx0 + tx];
      } else {
        uint8_t c[3];
        jpegdec::pixel(g, p, sx0 + tx, sy0 + v, c);
        px = c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16;
      }
      s_px[v][tx] = px;
    }
    __syncthreads();
  }
  for (int ly = ty; ly < th; ly += ROWS) {
    if (tx >= tw) continue;
    uint32_t px = 0;
    if (!bad) {
      int sx, sy;
      jpegdec::oriented_src(o, w, h, x0 + tx, y0 + ly, sx, sy);
      px = s_px[sy - sy0][sx - sx0];
    }
    uint8_t* q = out + ((size_t)f * w * h + (size_t)(y0 + ly) * w + x0 + tx) * CH;
    q[0] = (uint8_t)px;
    if (!GREY) {
      q[1] = (uint8_t)(px >> 8);
      q[2] = (uint8_t)(px >> 16);
    }
  }
}

size_t a16(size_t x) { return (x + 15) / 16 * 16; }

}  // namespace

void jpeg_dec_destroy(uwip_ctx* ctx) {
  if (ctx->jdec_ev) cudaEventSynchronize(ctx->jdec_ev), cudaEventDestroy(ctx->jdec_ev);
  if (ctx->jdec_pinned) cudaFreeHost(ctx->jdec_pinned);
  ctx->jdec_ev = nullptr;
  ctx->jdec_pinned = nullptr;
  ctx->jdec_pinned_bytes = 0;
}

int jpeg_orientation(const uint8_t* data, size_t len, int* orientation) {
  jpegdec::Header hd;
  const int rc = jpegdec::parse_header(data, len, hd);
  if (rc == jpegdec::OK) *orientation = hd.orientation;
  return rc;
}

int jpeg_decode_batch(uwip_ctx* ctx, const uint8_t* const* jpegs, const size_t* lens, int n, uint8_t* d_out, int w, int h,
                      int32_t* d_flags, bool grey, bool orient) {
  const char* fn = grey ? orient ? "uwip_jpeg_decode_u8_batch_oriented" : "uwip_jpeg_decode_u8_batch"
                        : orient ? "uwip_jpeg_decode_bgr8_batch_oriented" : "uwip_jpeg_decode_bgr8_batch";
  // ---- parse every header on the host
  std::vector<FrameTab> tabs((size_t)n);
  jpegdec::Header hd;
  size_t seg_total = 0, int_total = 0, sub_total = 0, blk_total = 0, smp_total = 0;
  uint32_t max_cap = 0;
  size_t max_blocks = 0;
  for (int f = 0; f < n; f++) {
    const int rc = jpegdec::parse_header(jpegs[f], lens[f], hd);
    if (rc != jpegdec::OK) {
      uwip_set_err(ctx, "%s: file %d: %s", fn, f,
                   rc == jpegdec::UNSUPPORTED ? "coding not supported (progressive, arithmetic, lossless, 12-bit, multi-scan, CMYK, RGB "
                                                "or sampling other than 4:4:4 / 4:2:2 / 4:4:0 / 4:2:0 / grey)"
                                              : "malformed or truncated header");
      return rc;
    }
    const int o = orient ? hd.orientation : 1;   // the stored size is the output size, transposed for 5..8
    if (hd.width != (o >= 5 ? h : w) || hd.height != (o >= 5 ? w : h)) {
      if (o == 1) uwip_set_err(ctx, "%s: file %d is %d x %d, not %d x %d", fn, f, hd.width, hd.height, w, h);
      else uwip_set_err(ctx, "%s: file %d is %d x %d with Exif orientation %d, which does not turn it into %d x %d", fn, f, hd.width, hd.height, o, w, h);
      return UWIP_ERR_INVALID;
    }
    FrameTab& t = tabs[f];
    t.g = jpegdec::geometry(hd);
    t.orient = o;
    for (int c = 0; c < hd.ncomp; c++) {
      memcpy(t.q[c], hd.q[hd.comp[c].tq], sizeof(t.q[c]));
      if (!jpegdec::make_derived(hd.dc[hd.comp[c].td], true, t.dc[c]) || !jpegdec::make_derived(hd.ac[hd.comp[c].ta], false, t.ac[c])) {
        uwip_set_err(ctx, "%s: file %d: bad Huffman table", fn, f);
        return UWIP_ERR_INVALID;
      }
    }
    t.seg_len = lens[f] - hd.scan_off;
    if (t.seg_len > (size_t)0x1FFFFFF0) {
      uwip_set_err(ctx, "%s: file %d: entropy-coded segment above 512 MB", fn, f);
      return UWIP_ERR_INVALID;
    }
    t.seg_off = seg_total;
    seg_total += a16(t.seg_len) + 16;
    t.int_off = int_total;
    int_total += (size_t)t.g.nint + 1;
    const uint64_t cap = (t.seg_len * 8 + SUB_BITS - 1) / SUB_BITS + (uint64_t)t.g.nint;
    t.sub_cap = (uint32_t)((cap + SYNC_T - 1) / SYNC_T * SYNC_T);
    t.sub_off = sub_total;
    sub_total += t.sub_cap;
    t.blk_off = blk_total;
    blk_total += t.g.nblocks;
    t.smp_off = smp_total;
    smp_total += a16(t.g.nsamples);
    max_cap = std::max(max_cap, t.sub_cap);
    max_blocks = std::max(max_blocks, t.g.nblocks);
  }
  // ---- device workspace: tables | staged segments | compact streams | interval starts, first subsequences | nsub | stats |
  //      subsequences | entry states | exit states | counts / DC | prefixes | coefficients | sample planes
  const size_t b_tab = a16((size_t)n * sizeof(FrameTab)), b_seg = a16(seg_total + 16), b_int = a16(int_total * 4);
  const size_t b_ns = a16((size_t)n * 4), b_st = a16((size_t)n * 8), b_sub = sub_total * sizeof(Sub), b_e = sub_total * 8,
               b_cd = sub_total * 16, b_coef = blk_total * 128;
  const size_t total = b_tab + 2 * b_seg + 2 * b_int + b_ns + b_st + b_sub + 2 * b_e + 2 * b_cd + b_coef + smp_total;
  uint8_t* ws = (uint8_t*)uwip_slot(ctx, SLOT_JPEGDEC, total);
  if (!ws) return UWIP_ERR_NOMEM;
  uint8_t* p = ws;
  auto take = [&](size_t b) { uint8_t* r = p; p += b; return r; };
  FrameTab* d_tab = (FrameTab*)take(b_tab);
  uint8_t* d_seg = take(b_seg);
  uint8_t* d_comp = take(b_seg);
  uint32_t* d_ist = (uint32_t*)take(b_int);
  uint32_t* d_ibase = (uint32_t*)take(b_int);
  int* d_nsub = (int*)take(b_ns);
  int32_t* d_stats = (int32_t*)take(b_st);
  int4* d_cd = (int4*)take(b_cd);
  int4* d_px = (int4*)take(b_cd);
  Sub* d_sub = (Sub*)take(b_sub);
  uint64_t* d_entry = (uint64_t*)take(b_e);
  uint64_t* d_exit = (uint64_t*)take(b_e);
  int16_t* d_coef = (int16_t*)take(b_coef);
  uint8_t* d_smp = take(smp_total);
  ctx->jdec_stats = d_stats;
  ctx->jdec_n = n;
  // ---- pinned staging: segments then tables; the copies of the previous call must have read it
  const size_t pin_bytes = seg_total + 16 + b_tab;
  if (ctx->jdec_ev) UWIP_CUDA(ctx, cudaEventSynchronize(ctx->jdec_ev));
  else UWIP_CUDA(ctx, cudaEventCreateWithFlags(&ctx->jdec_ev, cudaEventDisableTiming));
  if (ctx->jdec_pinned_bytes < pin_bytes) {
    if (ctx->jdec_pinned) cudaFreeHost(ctx->jdec_pinned);
    ctx->jdec_pinned = nullptr;
    ctx->jdec_pinned_bytes = 0;
    const size_t want = align_up(pin_bytes, 1 << 20);
    cudaError_t e = cudaMallocHost(&ctx->jdec_pinned, want);
    if (e != cudaSuccess) {
      uwip_set_err(ctx, "cudaMallocHost(%zu bytes) for the JPEG staging buffer failed: %s", want, cudaGetErrorString(e));
      cudaGetLastError();
      return UWIP_ERR_NOMEM;
    }
    ctx->jdec_pinned_bytes = want;
  }
  uint8_t* pin = (uint8_t*)ctx->jdec_pinned;
  for (int f = 0; f < n; f++) memcpy(pin + tabs[f].seg_off, jpegs[f] + (lens[f] - tabs[f].seg_len), tabs[f].seg_len);
  memcpy(pin + seg_total + 16, tabs.data(), (size_t)n * sizeof(FrameTab));
  UWIP_CUDA(ctx, cudaMemcpyAsync(d_seg, pin, seg_total, cudaMemcpyHostToDevice, ctx->stream));
  UWIP_CUDA(ctx, cudaMemcpyAsync(d_tab, pin + seg_total + 16, (size_t)n * sizeof(FrameTab), cudaMemcpyHostToDevice, ctx->stream));
  UWIP_CUDA(ctx, cudaEventRecord(ctx->jdec_ev, ctx->stream));
  UWIP_CUDA(ctx, cudaMemsetAsync(d_flags, 0, (size_t)n * 4, ctx->stream));
  UWIP_CUDA(ctx, cudaMemsetAsync(d_stats, 0, (size_t)n * 8, ctx->stream));
  UWIP_CUDA(ctx, cudaMemsetAsync(d_coef, 0, b_coef, ctx->stream));
  // ---- the passes
  const unsigned ny = (unsigned)n;
  UWIP_LAUNCH(ctx, "jpeg_dec_destuff", jpeg_dec_destuff_kernel, n, CTA_T, 0, (const FrameTab*)d_tab, (const uint8_t*)d_seg, d_comp, d_ist,
              d_ibase, d_sub, d_nsub, d_flags);
  const dim3 gsub(max_cap / SYNC_T, ny);
  UWIP_LAUNCH(ctx, "jpeg_dec_sync", jpeg_dec_sync_kernel, gsub, SYNC_T, 0, (const FrameTab*)d_tab, (const uint8_t*)d_comp,
              (const Sub*)d_sub, (const int*)d_nsub, d_entry, d_exit, d_cd, d_stats);
  UWIP_LAUNCH(ctx, "jpeg_dec_fixup", jpeg_dec_fixup_kernel, (n + 31) / 32, 32, 0, (const FrameTab*)d_tab, (const uint8_t*)d_comp,
              (const Sub*)d_sub, (const int*)d_nsub, d_entry, d_exit, d_cd, d_stats, n);
  UWIP_LAUNCH(ctx, "jpeg_dec_scan", jpeg_dec_scan_kernel, n, CTA_T, 0, (const FrameTab*)d_tab, (const Sub*)d_sub, (const int*)d_nsub,
              (const uint32_t*)d_ibase, d_cd, d_px);
  UWIP_LAUNCH(ctx, "jpeg_dec_huff", jpeg_dec_huff_kernel, gsub, SYNC_T, 0, (const FrameTab*)d_tab, (const uint8_t*)d_comp,
              (const Sub*)d_sub, (const int*)d_nsub, (const uint64_t*)d_entry, (const int4*)d_cd, d_coef, d_flags);
  const dim3 gblk((unsigned)((max_blocks + IDCT_T - 1) / IDCT_T), ny), gpix((unsigned)(((size_t)w * h + COLOR_T - 1) / COLOR_T), ny);
  if (grey) UWIP_LAUNCH(ctx, "jpeg_dec_idct_y", jpeg_dec_idct_kernel<true>, gblk, IDCT_T, 0, (const FrameTab*)d_tab, (const int16_t*)d_coef, d_smp);
  else UWIP_LAUNCH(ctx, "jpeg_dec_idct", jpeg_dec_idct_kernel<false>, gblk, IDCT_T, 0, (const FrameTab*)d_tab, (const int16_t*)d_coef, d_smp);
  if (orient) {
    const int tiles_x = (w + TILE - 1) / TILE;
    const dim3 gtile((unsigned)((size_t)tiles_x * ((h + TILE - 1) / TILE)), ny);
    if (grey)
      UWIP_LAUNCH(ctx, "jpeg_dec_grey_oriented", jpeg_dec_oriented_kernel<true>, gtile, COLOR_T, 0, (const FrameTab*)d_tab,
                  (const uint8_t*)d_smp, (const int32_t*)d_flags, d_out, w, h, tiles_x);
    else
      UWIP_LAUNCH(ctx, "jpeg_dec_color_oriented", jpeg_dec_oriented_kernel<false>, gtile, COLOR_T, 0, (const FrameTab*)d_tab,
                  (const uint8_t*)d_smp, (const int32_t*)d_flags, d_out, w, h, tiles_x);
  } else if (grey) {
    UWIP_LAUNCH(ctx, "jpeg_dec_grey", jpeg_dec_grey_kernel, gpix, COLOR_T, 0, (const FrameTab*)d_tab, (const uint8_t*)d_smp,
                (const int32_t*)d_flags, d_out, w, h);
  } else {
    UWIP_LAUNCH(ctx, "jpeg_dec_color", jpeg_dec_color_kernel, gpix, COLOR_T, 0, (const FrameTab*)d_tab, (const uint8_t*)d_smp,
                (const int32_t*)d_flags, d_out, w, h);
  }
  return UWIP_OK;
}
