// jpegenc.cu - batched baseline JPEG encoder whose files are byte-identical to cv2.imwrite / libjpeg-turbo (SURVEY 8f row N3,
// the file half of the device path).  The arithmetic is csrc/jpegenc.h; this file spreads it over the GPU.  Every 8 x 8 block
// is independent except for the DC difference (a neighbour subtraction) and its bit offset (a prefix sum of code lengths), so
// the work splits into five launches, each covering all n frames:
//   setup   one thread: quantiser reciprocals, Huffman code tables and the header (they depend only on W, H and quality)
//   blocks  a CTA per 32 MCUs: colour conversion, edge expansion and h2v2 in shared memory, one thread per block runs islow,
//           quantises and stores the zig-zag int16 coefficients, their non-zero mask, the quantised DC and the AC code bits.
//           A grey plane (one component, an MCU of one block) has its own load: a thread per block reads its 8 x 8 samples
//           with the edges replicated, then codes the block the same way.
//   scan    a CTA per frame: MCU code lengths (DC differences taken across MCUs here) -> exclusive prefix sum = bit offsets
//   emit    a thread per MCU writes its bits at its offset into the frame's bit buffer; only the words two MCUs share are
//           combined with atomicOr (the scan zeroed them)
//   stuff   a CTA per frame: header, the scan bytes with 0x00 after every 0xFF, EOI, and the file length
// The unstuffed bit buffer of frame f lives in the tail of its own output slot (jpegenc::raw_capacity), so the only workspace
// is the coefficient store of the blocks pass (about 3 B/px, 2 B/px grey).  A frame's bytes do not depend on the batch it is
// in.  The scan, emit and stuff passes and the host sequence take the component count NC (3: 4:2:0, 1: grey) as a template
// parameter: blocks per MCU, their tables and the header length follow from it (jpegenc.h).
#include <algorithm>

#include "common.cuh"
#include "jpegenc.h"

namespace {

using jpegenc::Geometry;
using jpegenc::Huff;
using jpegenc::Recip;

constexpr int MCUS_PER_CTA = 32;         // blocks pass: 32 MCUs x 6 blocks = 192 threads
constexpr int SCAN_THREADS = 1024;
constexpr int EMIT_THREADS = 128;
constexpr int STUFF_BYTES = 16;          // per thread and tile of the stuffing pass
constexpr int GREY_BLOCKS_T = 128;       // blocks pass of a grey plane: a thread per block

struct Tables {
  Recip q[2][64];   // natural order; 0 luma, 1 chroma
  Huff hf[4];       // DC0, AC0, DC1, AC1
  uint8_t header[jpegenc::HEADER_BYTES];   // the longer of the two headers
};

struct BlockInfo {
  unsigned long long mask;   // bit k: zig-zag coefficient k (1..63) is non-zero
  int dc;                    // quantised DC (a dummy block's is copied from its neighbour, jccoefct.c)
  unsigned acbits;           // bits of the AC codes, EOB included
};

// the frame's unstuffed bit buffer: 16-byte aligned, after room for the header and the stuffed copy of everything before it
template <int NC>
__host__ __device__ inline uint8_t* raw_buffer(uint8_t* out_f, size_t raw_cap) {
  return (uint8_t*)(((uintptr_t)out_f + jpegenc::header_bytes(NC) + raw_cap + 2 + 15) & ~(uintptr_t)15);
}

__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }

template <int NC>
__global__ void jpe_setup_kernel(Tables* __restrict__ t, int w, int h, int quality) {
  const int i = threadIdx.x;
  if (i < 128) t->q[i >> 6][i & 63] = jpegenc::compute_reciprocal((unsigned)jpegenc::quant_value(i >> 6, i & 63, quality) << 3);
  if (i < 4) jpegenc::make_derived(i, t->hf[i]);
  if (i == 4) jpegenc::write_header(t->header, w, h, quality, NC);
}

// 16 pixels of row y from column x0 (clamped at the right edge), as 48 bytes
__device__ __forceinline__ void load_row16(const uint8_t* __restrict__ frame, const Geometry& g, int x0, int y, uint8_t* px) {
  const uint8_t* row = frame + (size_t)y * g.w * 3;
  const uint8_t* p = row + (size_t)x0 * 3;
  if (x0 + 16 <= g.w && ((uintptr_t)p & 15) == 0) {
    const uint4* v = reinterpret_cast<const uint4*>(p);
#pragma unroll
    for (int k = 0; k < 3; k++) reinterpret_cast<uint4*>(px)[k] = __ldg(v + k);
  } else {
#pragma unroll
    for (int j = 0; j < 16; j++) {
      const int x = min(x0 + j, g.w - 1);
      px[3 * j] = row[3 * x]; px[3 * j + 1] = row[3 * x + 1]; px[3 * j + 2] = row[3 * x + 2];
    }
  }
}

// islow, quantisation and the zig-zag store (to cb) of one block whose samples minus 128 are d; its quantised DC goes to dc,
// its non-zero mask, DC and AC code bits (acs: AC code lengths of its table) to bi
__device__ __forceinline__ void code_block(int (&d)[64], const Recip* q, const uint8_t* acs, short* cb, int& dc, BlockInfo* bi) {
#pragma unroll
  for (int r = 0; r < 8; r++) jpegenc::fdct_1d(d + 8 * r, 1, true);
#pragma unroll
  for (int c = 0; c < 8; c++) jpegenc::fdct_1d(d + c, 8, false);
  int zz[64];
#pragma unroll
  for (int k = 0; k < 64; k++) zz[k] = jpegenc::quantize(d[jpegenc::natural_order(k)], q[jpegenc::natural_order(k)]);
  unsigned long long mask = 0;
  unsigned bits = 0;
  int run = 0;
#pragma unroll
  for (int k = 1; k < 64; k++) {
    if (zz[k] == 0) {
      run++;
    } else {
      mask |= 1ull << k;
      while (run > 15) { bits += acs[0xF0]; run -= 16; }
      const int nb = jpegenc::nbits(zz[k]);
      bits += acs[(run << 4) | nb] + nb;
      run = 0;
    }
  }
  if (run) bits += acs[0];
  uint4* cw = reinterpret_cast<uint4*>(cb);
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint32_t v[4];
#pragma unroll
    for (int j = 0; j < 4; j++) v[j] = (uint32_t)(uint16_t)zz[8 * k + 2 * j] | ((uint32_t)(uint16_t)zz[8 * k + 2 * j + 1] << 16);
    cw[k] = make_uint4(v[0], v[1], v[2], v[3]);
  }
  dc = zz[0];
  bi->mask = mask;
  bi->dc = zz[0];
  bi->acbits = bits;
}

__global__ void __launch_bounds__(MCUS_PER_CTA * 6) jpe_blocks_kernel(const uint8_t* __restrict__ src, int n, Geometry g,
                                                                        const Tables* __restrict__ tab, short* __restrict__ coef,
                                                                        BlockInfo* __restrict__ info) {
  __shared__ uint8_t s_y[MCUS_PER_CTA][256], s_cb[MCUS_PER_CTA][256], s_cr[MCUS_PER_CTA][256];
  __shared__ Recip s_q[2][64];
  __shared__ uint8_t s_acsize[2][256];
  __shared__ int s_dc[MCUS_PER_CTA][6];
  const int tid = threadIdx.x;
  const int nmcu = g.mcux * g.mcuy;
  for (int i = tid; i < 128; i += blockDim.x) s_q[i >> 6][i & 63] = tab->q[i >> 6][i & 63];
  for (int i = tid; i < 512; i += blockDim.x) s_acsize[i >> 8][i & 255] = tab->hf[1 + 2 * (i >> 8)].size[i & 255];
  const int m0 = blockIdx.x * MCUS_PER_CTA;
  for (int f = blockIdx.y; f < n; f += gridDim.y) {
    const uint8_t* frame = src + (size_t)f * g.w * g.h * 3;
    __syncthreads();
    // colour conversion of the 16 x 16 pixels of each MCU: Y from the edge-replicated row, Cb / Cr from the row that feeds
    // the chroma of that position (jcprepct.c pads to an even row count, then the downsampled plane to whole blocks)
    for (int r = tid; r < MCUS_PER_CTA * 16; r += blockDim.x) {
      const int lm = r >> 4, m = m0 + lm;
      if (m >= nmcu) continue;
      const int x0 = 16 * (m % g.mcux), y = 16 * (m / g.mcux) + (r & 15);
      const int yl = min(y, g.h - 1), yc = jpegenc::chroma_src_row(g, y);
      uint8_t px[48];
      load_row16(frame, g, x0, yl, px);
      uint8_t* oy = &s_y[lm][(r & 15) * 16];
      uint8_t* ob = &s_cb[lm][(r & 15) * 16];
      uint8_t* orr = &s_cr[lm][(r & 15) * 16];
#pragma unroll
      for (int j = 0; j < 16; j++) {
        int Y, cb, cr;
        jpegenc::rgb_ycc(px[3 * j], px[3 * j + 1], px[3 * j + 2], Y, cb, cr);
        oy[j] = (uint8_t)Y; ob[j] = (uint8_t)cb; orr[j] = (uint8_t)cr;
      }
      if (yc != yl) {
        load_row16(frame, g, x0, yc, px);
#pragma unroll
        for (int j = 0; j < 16; j++) {
          int Y, cb, cr;
          jpegenc::rgb_ycc(px[3 * j], px[3 * j + 1], px[3 * j + 2], Y, cb, cr);
          ob[j] = (uint8_t)cb; orr[j] = (uint8_t)cr;
        }
      }
    }
    __syncthreads();
    const int lm = tid / 6, b = tid % 6, m = m0 + lm;
    const int mx = m % g.mcux, my = m / g.mcux;
    const bool luma = b < 4;
    const bool real = m < nmcu && (!luma || (2 * mx + (b & 1) < g.ybw && 2 * my + (b >> 1) < g.ybh));
    BlockInfo* bi = info + ((size_t)f * nmcu + m) * 6 + b;
    if (real) {
      int d[64];
      if (luma) {
        const uint8_t* s = &s_y[lm][(b >> 1) * 128 + (b & 1) * 8];
#pragma unroll
        for (int i = 0; i < 64; i++) d[i] = (int)s[(i >> 3) * 16 + (i & 7)] - 128;
      } else {
        const uint8_t* s = b == 4 ? s_cb[lm] : s_cr[lm];
#pragma unroll
        for (int i = 0; i < 64; i++) {
          const int o = (i >> 3) * 32 + (i & 7) * 2;
          d[i] = jpegenc::h2v2(s[o], s[o + 1], s[o + 16], s[o + 17], i) - 128;
        }
      }
      code_block(d, s_q[luma ? 0 : 1], s_acsize[luma ? 0 : 1], coef + (((size_t)f * nmcu + m) * 6 + b) * 64, s_dc[lm][b], bi);
    }
    __syncthreads();
    if (m < nmcu && !real) {   // compress_data: right of the edge the DC on the left, below it the DC of the MCU's block 1
      const bool real1 = 2 * mx + 1 < g.ybw;
      const int dc1 = real1 ? s_dc[lm][1] : s_dc[lm][0];
      const bool bottom = 2 * my + (b >> 1) >= g.ybh;
      bi->mask = 0;
      bi->dc = bottom ? dc1 : s_dc[lm][b - 1];
      bi->acbits = s_acsize[0][0];
    }
  }
}

// a grey plane: a thread per block (= MCU) loads its 8 x 8 samples, the column and row past the edge replicated (jcsample.c
// expand_right_edge, jcprepct.c expand_bottom_edge), and codes it with table 0
__global__ void __launch_bounds__(GREY_BLOCKS_T) jpe_blocks_u8_kernel(const uint8_t* __restrict__ src, int n, Geometry g,
                                                                      const Tables* __restrict__ tab, short* __restrict__ coef,
                                                                      BlockInfo* __restrict__ info) {
  __shared__ Recip s_q[64];
  __shared__ uint8_t s_acsize[256];
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_q[i] = tab->q[0][i];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_acsize[i] = tab->hf[1].size[i];
  __syncthreads();
  const int nblk = g.mcux * g.mcuy;
  const int m = blockIdx.x * GREY_BLOCKS_T + threadIdx.x;
  if (m >= nblk) return;
  const int x0 = 8 * (m % g.mcux), y0 = 8 * (m / g.mcux);
  for (int f = blockIdx.y; f < n; f += gridDim.y) {
    const uint8_t* plane = src + (size_t)f * g.w * g.h;
    int d[64];
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const uint8_t* row = plane + (size_t)min(y0 + r, g.h - 1) * g.w;
      if (x0 + 8 <= g.w && ((uintptr_t)(row + x0) & 7) == 0) {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(row + x0));
#pragma unroll
        for (int j = 0; j < 4; j++) {
          d[8 * r + j] = (int)((v.x >> (8 * j)) & 255u) - 128;
          d[8 * r + 4 + j] = (int)((v.y >> (8 * j)) & 255u) - 128;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; j++) d[8 * r + j] = (int)row[min(x0 + j, g.w - 1)] - 128;
      }
    }
    int dc;
    code_block(d, s_q, s_acsize, coef + ((size_t)f * nblk + m) * 64, dc, info + (size_t)f * nblk + m);
  }
}

// exclusive prefix sum over the CTA (blockDim.x == SCAN_THREADS); returns the CTA total
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
    s_warp[lane] = s;   // inclusive totals of the warps
  }
  __syncthreads();
  excl = x - v + (wid ? s_warp[wid - 1] : T(0));
  const T total = s_warp[(blockDim.x >> 5) - 1];
  __syncthreads();
  return total;
}

template <int NC>
__global__ void __launch_bounds__(SCAN_THREADS) jpe_scan_kernel(const BlockInfo* __restrict__ info, int nmcu, const Tables* __restrict__ tab,
                                                                 unsigned long long* __restrict__ offs, unsigned long long* __restrict__ total,
                                                                 uint8_t* __restrict__ out, size_t stride, size_t raw_cap) {
  constexpr int NB = jpegenc::blocks_per_mcu(NC);
  __shared__ unsigned long long s_warp[32];
  __shared__ uint8_t s_dcsize[2][12];
  const int f = blockIdx.x;
  if (threadIdx.x < 24) s_dcsize[threadIdx.x / 12][threadIdx.x % 12] = tab->hf[2 * (threadIdx.x / 12)].size[threadIdx.x % 12];
  __syncthreads();
  const BlockInfo* fi = info + (size_t)f * nmcu * NB;
  uint32_t* raw = reinterpret_cast<uint32_t*>(raw_buffer<NC>(out + (size_t)f * stride, raw_cap));
  unsigned long long carry = 0;
  for (int base = 0; base < nmcu; base += SCAN_THREADS) {
    const int m = base + threadIdx.x;
    unsigned long long bits = 0;
    if (m < nmcu) {
      const BlockInfo* b = fi + (size_t)m * NB;
      int pred[NC];   // DC predictors: the last block of each component in the MCU before
#pragma unroll
      for (int c = 0; c < NC; c++) pred[c] = m > 0 ? b[c - NC].dc : 0;
      unsigned s = 0;
#pragma unroll
      for (int k = 0; k < NB; k++) {
        const int c = jpegenc::block_comp(k);
        const int nb = jpegenc::nbits(b[k].dc - pred[c]);
        s += b[k].acbits + s_dcsize[jpegenc::block_table(k)][nb] + nb;
        pred[c] = b[k].dc;
      }
      bits = s;
    }
    unsigned long long excl;
    const unsigned long long tot = cta_exclusive_scan(bits, excl, s_warp);
    if (m < nmcu) {
      const unsigned long long o = carry + excl;
      offs[(size_t)f * nmcu + m] = o;
      raw[o >> 5] = 0u;   // the word holding the MCU's first bit may be shared with the MCU before it
    }
    carry += tot;
  }
  if (threadIdx.x == 0) {
    total[f] = carry;
    raw[carry >> 5] = 0u;   // the last word: the end of the scan and its 1-bit padding
  }
}

struct BitOut {
  uint32_t* raw;
  unsigned long long word;   // index of the word being filled
  unsigned long long first;  // the MCU's first word (shared with the MCU before unless it starts on a word boundary)
  bool first_shared;
  unsigned long long acc;
  int nacc;
  __device__ __forceinline__ void put(uint32_t code, int size) {
    acc = (acc << size) | code;
    nacc += size;
    if (nacc >= 32) {
      nacc -= 32;
      const uint32_t v = bswap32((uint32_t)(acc >> nacc));
      if (word == first && first_shared) atomicOr(raw + word, v);
      else raw[word] = v;
      word++;
    }
  }
  __device__ __forceinline__ void finish() {
    if (nacc) atomicOr(raw + word, bswap32((uint32_t)(acc << (32 - nacc))));
  }
};

template <int NC>
__global__ void __launch_bounds__(EMIT_THREADS) jpe_emit_kernel(const BlockInfo* __restrict__ info, const short* __restrict__ coef, int n,
                                                                 int nmcu, const Tables* __restrict__ tab,
                                                                 const unsigned long long* __restrict__ offs,
                                                                 const unsigned long long* __restrict__ total, uint8_t* __restrict__ out,
                                                                 size_t stride, size_t raw_cap) {
  __shared__ uint16_t s_code[4][256];
  __shared__ uint8_t s_size[4][256];
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
    s_code[i >> 8][i & 255] = tab->hf[i >> 8].code[i & 255];
    s_size[i >> 8][i & 255] = tab->hf[i >> 8].size[i & 255];
  }
  __syncthreads();
  constexpr int NB = jpegenc::blocks_per_mcu(NC);
  const int m = blockIdx.x * EMIT_THREADS + threadIdx.x;
  if (m >= nmcu) return;
  for (int f = blockIdx.y; f < n; f += gridDim.y) {
    const size_t mi = (size_t)f * nmcu + m;
    const BlockInfo* b = info + mi * NB;
    const short* c = coef + mi * NB * 64;
    const unsigned long long off = offs[mi];
    BitOut o;
    o.raw = reinterpret_cast<uint32_t*>(raw_buffer<NC>(out + (size_t)f * stride, raw_cap));
    o.word = o.first = off >> 5;
    o.first_shared = (off & 31) != 0;
    o.acc = 0;
    o.nacc = (int)(off & 31);   // leading bits of the first word belong to the MCU before: zeros here
    int pred[NC];
#pragma unroll
    for (int k = 0; k < NC; k++) pred[k] = m > 0 ? b[k - NC].dc : 0;
    for (int k = 0; k < NB; k++) {
      const int comp = jpegenc::block_comp(k), t = 2 * jpegenc::block_table(k);
      const BlockInfo bk = b[k];
      const int diff = bk.dc - pred[comp];
      pred[comp] = bk.dc;
      int nb = jpegenc::nbits(diff);
      o.put(((uint32_t)s_code[t][nb] << nb) | ((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << nb) - 1u)), s_size[t][nb] + nb);
      unsigned long long mask = bk.mask;
      int last = 0;
      const short* ck = c + k * 64;
      while (mask) {
        const int z = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        int run = z - last - 1;
        while (run > 15) { o.put(s_code[t + 1][0xF0], s_size[t + 1][0xF0]); run -= 16; }
        const int v = ck[z];
        nb = jpegenc::nbits(v);
        const int sym = (run << 4) | nb;
        o.put(((uint32_t)s_code[t + 1][sym] << nb) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << nb) - 1u)), s_size[t + 1][sym] + nb);
        last = z;
      }
      if (last != 63) o.put(s_code[t + 1][0], s_size[t + 1][0]);
    }
    if (m == nmcu - 1) {   // flush_bits: the last byte is padded with 1-bits
      const int pad = (int)((8 - (total[f] & 7)) & 7);
      if (pad) o.put((1u << pad) - 1u, pad);
    }
    o.finish();
  }
}

template <int NC>
__global__ void __launch_bounds__(SCAN_THREADS) jpe_stuff_kernel(const Tables* __restrict__ tab, const unsigned long long* __restrict__ total,
                                                                  uint8_t* __restrict__ out, size_t stride, size_t raw_cap,
                                                                  unsigned long long* __restrict__ len) {
  constexpr int HEADER = jpegenc::header_bytes(NC);
  __shared__ unsigned long long s_warp[32];
  const int f = blockIdx.x;
  uint8_t* o = out + (size_t)f * stride;
  const uint8_t* raw = raw_buffer<NC>(o, raw_cap);
  for (int i = threadIdx.x; i < HEADER; i += blockDim.x) o[i] = tab->header[i];
  const unsigned long long nraw = (total[f] + 7) >> 3;
  uint8_t* dst = o + HEADER;
  unsigned long long carry = 0;   // 0x00 bytes inserted so far
  // Tile by tile: every thread reads its 16 bytes before any thread writes (the scan below synchronises), and a tile's
  // output ends below the raw bytes of the next tile (raw_buffer leaves room for the stuffed copy of everything before it).
  for (unsigned long long t0 = 0; t0 < nraw; t0 += (unsigned long long)STUFF_BYTES * SCAN_THREADS) {
    const unsigned long long i0 = t0 + (unsigned long long)STUFF_BYTES * threadIdx.x;
    uint8_t v[STUFF_BYTES];
    *reinterpret_cast<uint4*>(v) = i0 < nraw ? *reinterpret_cast<const uint4*>(raw + i0) : make_uint4(0, 0, 0, 0);
    const int nv = i0 < nraw ? (int)min((unsigned long long)STUFF_BYTES, nraw - i0) : 0;
    unsigned long long cnt = 0;
#pragma unroll
    for (int j = 0; j < STUFF_BYTES; j++) cnt += (j < nv && v[j] == 0xFF);
    unsigned long long excl;
    const unsigned long long tot = cta_exclusive_scan(cnt, excl, s_warp);
    unsigned long long p = i0 + carry + excl;
#pragma unroll
    for (int j = 0; j < STUFF_BYTES; j++) {
      if (j < nv) {
        dst[p++] = v[j];
        if (v[j] == 0xFF) dst[p++] = 0;
      }
    }
    carry += tot;
  }
  if (threadIdx.x == 0) {
    dst[nraw + carry] = 0xFF;
    dst[nraw + carry + 1] = 0xD9;
    len[f] = HEADER + nraw + carry + 2;
  }
}

// the five passes over n frames (NC = 3: bgr8 frames as 4:2:0, NC = 1: grey planes)
template <int NC>
int encode_batch(uwip_ctx* ctx, const uint8_t* d_src, int n, int w, int h, int quality, uint8_t* d_out, size_t stride, uint64_t* d_len) {
  constexpr int NB = jpegenc::blocks_per_mcu(NC);
  const Geometry g = jpegenc::geometry(w, h, NC);
  const size_t nmcu = (size_t)g.mcux * g.mcuy;
  const size_t raw_cap = jpegenc::raw_capacity(w, h, NC);
  // workspace: tables | MCU bit offsets | per-frame totals | block infos | coefficients
  const size_t b_tab = align_up(sizeof(Tables), 256);
  const size_t b_off = align_up((size_t)n * nmcu * 8, 256), b_tot = align_up((size_t)n * 8, 256);
  const size_t b_info = align_up((size_t)n * nmcu * NB * sizeof(BlockInfo), 256);
  const size_t b_coef = (size_t)n * nmcu * NB * 64 * sizeof(short);
  uint8_t* ws = (uint8_t*)uwip_slot(ctx, SLOT_JPEGENC, b_tab + b_off + b_tot + b_info + b_coef);
  if (!ws) return UWIP_ERR_NOMEM;
  Tables* tab = (Tables*)ws;
  unsigned long long* offs = (unsigned long long*)(ws + b_tab);
  unsigned long long* tot = (unsigned long long*)(ws + b_tab + b_off);
  BlockInfo* info = (BlockInfo*)(ws + b_tab + b_off + b_tot);
  short* coef = (short*)(ws + b_tab + b_off + b_tot + b_info);
  const int ny = std::min(n, 65535);
  UWIP_LAUNCH(ctx, "jpeg_enc_setup", jpe_setup_kernel<NC>, 1, 128, 0, tab, w, h, quality);
  if (NC == 3)
    UWIP_LAUNCH(ctx, "jpeg_enc_blocks", jpe_blocks_kernel, dim3((unsigned)((nmcu + MCUS_PER_CTA - 1) / MCUS_PER_CTA), ny),
                MCUS_PER_CTA * 6, 0, d_src, n, g, (const Tables*)tab, coef, info);
  else
    UWIP_LAUNCH(ctx, "jpeg_enc_blocks_u8", jpe_blocks_u8_kernel, dim3((unsigned)((nmcu + GREY_BLOCKS_T - 1) / GREY_BLOCKS_T), ny),
                GREY_BLOCKS_T, 0, d_src, n, g, (const Tables*)tab, coef, info);
  UWIP_LAUNCH(ctx, "jpeg_enc_scan", jpe_scan_kernel<NC>, n, SCAN_THREADS, 0, (const BlockInfo*)info, (int)nmcu, (const Tables*)tab, offs,
              tot, d_out, stride, raw_cap);
  UWIP_LAUNCH(ctx, "jpeg_enc_emit", jpe_emit_kernel<NC>, dim3((unsigned)((nmcu + EMIT_THREADS - 1) / EMIT_THREADS), ny), EMIT_THREADS, 0,
              (const BlockInfo*)info, (const short*)coef, n, (int)nmcu, (const Tables*)tab, (const unsigned long long*)offs,
              (const unsigned long long*)tot, d_out, stride, raw_cap);
  UWIP_LAUNCH(ctx, "jpeg_enc_stuff", jpe_stuff_kernel<NC>, n, SCAN_THREADS, 0, (const Tables*)tab, (const unsigned long long*)tot, d_out,
              stride, raw_cap, (unsigned long long*)d_len);
  return UWIP_OK;
}

}  // namespace

size_t jpeg_encode_bound(int w, int h) { return jpegenc::encode_bound(w, h); }
size_t jpeg_encode_u8_bound(int w, int h) { return jpegenc::encode_bound(w, h, 1); }

int jpeg_encode_batch_dev(uwip_ctx* ctx, const uint8_t* d_bgr, int n, int w, int h, int quality, uint8_t* d_out, size_t stride,
                          uint64_t* d_len) {
  return encode_batch<3>(ctx, d_bgr, n, w, h, quality, d_out, stride, d_len);
}
int jpeg_encode_u8_batch_dev(uwip_ctx* ctx, const uint8_t* d_planes, int n, int w, int h, int quality, uint8_t* d_out, size_t stride,
                             uint64_t* d_len) {
  return encode_batch<1>(ctx, d_planes, n, w, h, quality, d_out, stride, d_len);
}
