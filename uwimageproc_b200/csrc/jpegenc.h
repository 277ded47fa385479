// jpegenc.h - the baseline JPEG encoder of libjpeg-turbo 3.1.2 (the codec behind cv2.imwrite / cv2.imencode of cv2 4.13.0)
// restated in plain C++ that compiles for the host and the device: the standard Annex K quantisation tables scaled by
// quality, the standard Annex K Huffman tables, no restart markers, no optimised Huffman tables, not progressive.  Two
// component layouts, `nc` below: a bgr8 frame is written as YCbCr 4:2:0 (nc = 3: Y 2x2, Cb and Cr 1x1, an MCU of six blocks),
// a grey plane as one component (nc = 1, jpeg_set_colorspace(JCS_GRAYSCALE): an MCU of one block).  csrc/jpegenc.cu runs
// this arithmetic batched on the GPU; encode_frame() and encode_grey_frame() below are the scalar references for one frame,
// which only the host test compiles.
//
// The bytes of a file are: SOI, APP0 (JFIF 1.01, density 1x1, no thumbnail), DQT 0 [, DQT 1], SOF0, DHT DC0, AC0 [, DC1, AC1],
// SOS, the entropy-coded segment, EOI; the bracketed tables only for nc = 3.  Every function names the libjpeg-turbo
// function it restates.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define JPEG_HD __host__ __device__
#else
#define JPEG_HD
#endif

namespace jpegenc {

// SOI .. SOS of the layout above (write_file_header, write_frame_header, write_scan_header)
JPEG_HD constexpr int header_bytes(int nc) { return nc == 3 ? 623 : 328; }
constexpr int HEADER_BYTES = header_bytes(3);
constexpr int GREY_HEADER_BYTES = header_bytes(1);
// blocks of an MCU, and the component and table pair (0 luma, 1 chroma) of block b: Y Y Y Y Cb Cr, or one grey block
JPEG_HD constexpr int blocks_per_mcu(int nc) { return nc == 3 ? 6 : 1; }
JPEG_HD constexpr int block_comp(int b) { return b < 4 ? 0 : b - 3; }
JPEG_HD constexpr int block_table(int b) { return b < 4 ? 0 : 1; }

// jpeg_natural_order (jutils.c): natural index of zig-zag position k
JPEG_HD constexpr int natural_order(int k) {
  constexpr int t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                         41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                         30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
  return t[k];
}

// std_luminance_quant_tbl / std_chrominance_quant_tbl (jcparam.c), natural order
JPEG_HD constexpr int std_quant(int table, int i) {
  constexpr unsigned char lum[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                     14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                     18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
  constexpr unsigned char chr[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
                                     99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
  return table == 0 ? lum[i] : chr[i];
}

// jpeg_quality_scaling (jcparam.c)
JPEG_HD inline int quality_scaling(int quality) {
  if (quality <= 0) quality = 1;
  if (quality > 100) quality = 100;
  return quality < 50 ? 5000 / quality : 200 - quality * 2;
}

// jpeg_add_quant_table with force_baseline = TRUE (jcparam.c): quantiser of natural index i
JPEG_HD inline int quant_value(int table, int i, int quality) {
  long t = ((long)std_quant(table, i) * quality_scaling(quality) + 50L) / 100L;
  if (t <= 0L) t = 1L;
  if (t > 255L) t = 255L;
  return (int)t;
}

// compute_reciprocal (jcdctmgr.c) for a 16-bit DCTELEM and divisor = quantiser << 3 (the SIMD build): reciprocal, correction
// and shift such that quantize() below equals the library's rounding division.  divisor >= 8 here, so the divisor == 1 case
// of the library never arises.
struct Recip {
  uint16_t recip, corr;
  int16_t shift;   // total right shift of (|x| + corr) * recip
};
JPEG_HD inline Recip compute_reciprocal(unsigned divisor) {
  int b = 0;
  while ((divisor >> (b + 1)) != 0u) b++;   // flss(divisor) - 1
  int r = 16 + b;
  uint32_t fq = (1u << r) / divisor, fr = (1u << r) % divisor;
  uint32_t c = divisor / 2u;
  if (fr == 0u) {   // power of two
    fq >>= 1;
    r--;
  } else if (fr <= divisor / 2u) {
    c++;
  } else {
    fq++;
  }
  Recip q;
  q.recip = (uint16_t)fq;
  q.corr = (uint16_t)c;
  q.shift = (int16_t)r;   // the SIMD build's two high-half multiplies, by recip and by scale = 1 << (32 - r): one shift by r
  return q;
}

// quantize (jcdctmgr.c), per coefficient
JPEG_HD inline int quantize(int x, Recip q) {
  const uint32_t a = (uint32_t)(x < 0 ? -x : x);
  const int p = (int)(((a + q.corr) * (uint32_t)q.recip) >> q.shift);
  return x < 0 ? -p : p;
}

// rgb_ycc_convert (jccolor.c): FIX(x) = (int)(x * 2^16 + 0.5), ONE_HALF = 2^15, CBCR_OFFSET = 128 << 16
JPEG_HD inline void rgb_ycc(int b, int g, int r, int& y, int& cb, int& cr) {
  y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
  cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
  cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// h2v2_downsample (jcsample.c): output column oc of the row pair, bias 1, 2, 1, 2 ... along the row
JPEG_HD inline int h2v2(int a, int b, int c, int d, int oc) { return (a + b + c + d + 1 + (oc & 1)) >> 2; }

// jpeg_fdct_islow (jfdctint.c): CONST_BITS 13, PASS1_BITS 2; data = samples - 128, in place, output scaled by 8
JPEG_HD inline int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }
JPEG_HD inline void fdct_1d(int* d, int stride, bool first) {
  const int t0 = d[0] + d[7 * stride], t7 = d[0] - d[7 * stride];
  const int t1 = d[stride] + d[6 * stride], t6 = d[stride] - d[6 * stride];
  const int t2 = d[2 * stride] + d[5 * stride], t5 = d[2 * stride] - d[5 * stride];
  const int t3 = d[3 * stride] + d[4 * stride], t4 = d[3 * stride] - d[4 * stride];
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  const int s = first ? 13 - 2 : 13 + 2;
  if (first) {
    d[0] = (t10 + t11) * 4;
    d[4 * stride] = (t10 - t11) * 4;
  } else {
    d[0] = descale(t10 + t11, 2);
    d[4 * stride] = descale(t10 - t11, 2);
  }
  const int z1 = (t12 + t13) * 4433;                         // FIX_0_541196100
  d[2 * stride] = descale(z1 + t13 * 6270, s);               // FIX_0_765366865
  d[6 * stride] = descale(z1 + t12 * -15137, s);             // FIX_1_847759065
  const int z5 = (t4 + t6 + t5 + t7) * 9633;                 // FIX_1_175875602
  const int a1 = (t4 + t7) * -7373, a2 = (t5 + t6) * -20995; // FIX_0_899976223, FIX_2_562915447
  const int a3 = (t4 + t6) * -16069 + z5, a4 = (t5 + t7) * -3196 + z5;   // FIX_1_961570560, FIX_0_390180644
  d[7 * stride] = descale(t4 * 2446 + a1 + a3, s);           // FIX_0_298631336
  d[5 * stride] = descale(t5 * 16819 + a2 + a4, s);          // FIX_2_053119869
  d[3 * stride] = descale(t6 * 25172 + a2 + a3, s);          // FIX_3_072711026
  d[1 * stride] = descale(t7 * 12299 + a1 + a4, s);          // FIX_1_501321110
}
JPEG_HD inline void fdct_islow(int* data) {
  for (int r = 0; r < 8; r++) fdct_1d(data + 8 * r, 1, true);
  for (int c = 0; c < 8; c++) fdct_1d(data + c, 8, false);
}

// std_huff_tables (jstdhuff.c): bits[1..16] and values of DC 0, AC 0, DC 1, AC 1
JPEG_HD constexpr int std_huff_bits(int t, int l /*1..16*/) {
  constexpr unsigned char bits[4][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                                         {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                                         {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},
                                         {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
  return bits[t][l - 1];
}
JPEG_HD constexpr int std_huff_val(int t, int i) {
  constexpr unsigned char ac_lum[162] = {
      0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
      0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
      0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
      0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
      0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
      0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
      0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
      0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
  constexpr unsigned char ac_chr[162] = {
      0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
      0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
      0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
      0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
      0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
      0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
      0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
      0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
  return (t & 1) ? (t == 1 ? ac_lum[i] : ac_chr[i]) : i;   // the DC tables list the categories 0 .. 11 in order
}

// jpeg_make_c_derived_tbl (jchuff.c): code and length of every symbol of table t (0 DC0, 1 AC0, 2 DC1, 3 AC1); a symbol the
// table lacks has length 0 (never emitted by a baseline 8-bit scan)
struct Huff {
  uint16_t code[256];
  uint8_t size[256];
};
JPEG_HD inline void make_derived(int t, Huff& h) {
  for (int i = 0; i < 256; i++) { h.code[i] = 0; h.size[i] = 0; }
  unsigned code = 0;
  int k = 0;
  for (int l = 1; l <= 16; l++) {
    for (int i = 0; i < std_huff_bits(t, l); i++, k++) {
      const int v = std_huff_val(t, k);
      h.code[v] = (uint16_t)code++;
      h.size[v] = (uint8_t)l;
    }
    code <<= 1;
  }
}

// the magnitude category of a coefficient or DC difference (jchuff.c: nbits = JPEG_NBITS(temp))
JPEG_HD inline int nbits(int v) {
  unsigned a = (unsigned)(v < 0 ? -v : v);
  int n = 0;
  while (a) { n++; a >>= 1; }
  return n;
}

// geometry of a frame: MCUs of 16 x 16 pixels (4:2:0) or 8 x 8 (grey), luma blocks of the padded plane, chroma rows after
// h2v2.  A grey scan has no dummy blocks: its MCUs are the blocks.
struct Geometry {
  int w, h, mcux, mcuy, ybw, ybh, ch;
};
JPEG_HD inline Geometry geometry(int w, int h, int nc = 3) {
  Geometry g;
  g.w = w; g.h = h;
  g.ybw = (w + 7) / 8; g.ybh = (h + 7) / 8;
  g.mcux = nc == 3 ? (w + 15) / 16 : g.ybw;
  g.mcuy = nc == 3 ? (h + 15) / 16 : g.ybh;
  g.ch = (h + 1) / 2;
  return g;
}

// Largest entropy-coded bits of one MCU: per block the longest DC code plus category 11 (luma 9 + 11, chroma 11 + 11)
// and 63 AC codes of the longest length (16) plus category 10; an AC magnitude stays below 2^10 because quantiser << 3
// >= 8 divides an islow output below 2^13.  Every byte may be 0xFF and then be followed by a stuffed 0x00.
JPEG_HD constexpr long mcu_max_bits(int nc) {
  return nc == 3 ? 4L * (9 + 11 + 63 * (16 + 10)) + 2L * (11 + 11 + 63 * (16 + 10)) : 9 + 11 + 63 * (16 + 10);
}
constexpr long MCU_MAX_BITS = mcu_max_bits(3);

// bytes of the unstuffed entropy-coded segment reserved at the end of an output slot (whole 16-byte lines, one spare)
JPEG_HD inline size_t raw_capacity(int w, int h, int nc = 3) {
  const Geometry g = geometry(w, h, nc);
  const size_t bits = (size_t)g.mcux * g.mcuy * (size_t)mcu_max_bits(nc);
  return ((bits + 7) / 8 + 16 + 15) / 16 * 16;
}

// worst-case file size: header, every scan byte doubled by stuffing, EOI.  The batched encoder keeps the unstuffed scan in
// the last raw_capacity() bytes of the slot (16-byte aligned, hence the 16 spare bytes) while it stuffs it into the front.
JPEG_HD inline size_t encode_bound(int w, int h, int nc = 3) {
  return (size_t)header_bytes(nc) + 2 * raw_capacity(w, h, nc) + 2 + 16;
}

// write_file_header, write_frame_header, write_scan_header (jcmarker.c): SOI .. SOS, header_bytes(nc) bytes.  Only the
// tables the components use are written (emit_dqt per component's table, emit_dht per table the scan names).
JPEG_HD inline int write_header(uint8_t* o, int w, int h, int quality, int nc = 3) {
  int n = 0;
  auto b = [&](int v) { o[n++] = (uint8_t)v; };
  auto w16 = [&](int v) { b(v >> 8); b(v & 255); };
  const int ntab = nc == 3 ? 2 : 1;
  b(0xFF); b(0xD8);                                                 // SOI
  b(0xFF); b(0xE0); w16(16);                                        // APP0: JFIF 1.01, density unit 0, 1 x 1, no thumbnail
  b('J'); b('F'); b('I'); b('F'); b(0); b(1); b(1); b(0); w16(1); w16(1); b(0); b(0);
  for (int t = 0; t < ntab; t++) {                                  // emit_dqt: 8-bit precision, zig-zag order
    b(0xFF); b(0xDB); w16(67); b(t);
    for (int k = 0; k < 64; k++) b(quant_value(t, natural_order(k), quality));
  }
  b(0xFF); b(0xC0); w16(8 + 3 * nc); b(8); w16(h); w16(w); b(nc);   // emit_sof(M_SOF0): id, h << 4 | v, quantisation table
  for (int c = 0; c < nc; c++) { b(c + 1); b(nc == 3 && c == 0 ? 0x22 : 0x11); b(c ? 1 : 0); }
  for (int t = 0; t < 2 * ntab; t++) {                              // emit_dht in the order the scan header sends them
    int count = 0;
    for (int l = 1; l <= 16; l++) count += std_huff_bits(t, l);
    b(0xFF); b(0xC4); w16(2 + 1 + 16 + count); b(((t & 1) << 4) | (t >> 1));
    for (int l = 1; l <= 16; l++) b(std_huff_bits(t, l));
    for (int i = 0; i < count; i++) b(std_huff_val(t, i));
  }
  b(0xFF); b(0xDA); w16(6 + 2 * nc); b(nc);                         // emit_sos: id, DC << 4 | AC table; Ss 0, Se 63, Ah Al 0
  for (int c = 0; c < nc; c++) { b(c + 1); b(c ? 0x11 : 0x00); }
  b(0); b(63); b(0);
  return n;
}

// colour conversion and edge expansion of one MCU position: Y sample and the h2v2 chroma sample of the padded planes
// (jcprepct.c expand_bottom_edge, jcsample.c expand_right_edge).  bgr: the frame, w * h * 3 bytes.
JPEG_HD inline int luma_at(const uint8_t* bgr, const Geometry& g, int x, int y) {
  x = x < g.w ? x : g.w - 1;
  y = y < g.h ? y : g.h - 1;
  const uint8_t* p = bgr + ((size_t)y * g.w + x) * 3;
  int Y, cb, cr;
  rgb_ycc(p[0], p[1], p[2], Y, cb, cr);
  return Y;
}
// the full-resolution row that feeds chroma row y: rows past the even-padded height repeat the last downsampled row
JPEG_HD inline int chroma_src_row(const Geometry& g, int y) {
  if (y >= 2 * g.ch) y = 2 * g.ch - 2 + (y & 1);
  return y < g.h ? y : g.h - 1;
}

// Scalar reference encoder of one frame (encode_mcu_huff of jchuff.c over compress_data of jccoefct.c).  Returns the file
// length; `out` must hold encode_bound(w, h) bytes.  Host only: the tests compile it with g++.
struct BitSink {
  uint8_t* o;
  size_t n;
  uint64_t acc;
  int nacc;
  JPEG_HD void put(uint32_t code, int size) {
    acc = (acc << size) | (code & ((1u << size) - 1u));
    nacc += size;
    while (nacc >= 8) {
      const uint8_t v = (uint8_t)(acc >> (nacc - 8));
      nacc -= 8;
      o[n++] = v;
      if (v == 0xFF) o[n++] = 0;
    }
  }
  JPEG_HD void flush() {   // flush_bits: pad the last byte with 1-bits
    if (nacc) put((1u << (8 - nacc)) - 1u, 8 - nacc);
  }
};

JPEG_HD inline void encode_block(BitSink& s, const int* zz, int& pred, const Huff& dc, const Huff& ac) {
  const int diff = zz[0] - pred;
  pred = zz[0];
  int nb = nbits(diff);
  s.put(dc.code[nb], dc.size[nb]);
  if (nb) s.put((uint32_t)(diff < 0 ? diff - 1 : diff), nb);
  int run = 0;
  for (int k = 1; k < 64; k++) {
    const int v = zz[k];
    if (v == 0) { run++; continue; }
    while (run > 15) { s.put(ac.code[0xF0], ac.size[0xF0]); run -= 16; }
    nb = nbits(v);
    const int sym = (run << 4) | nb;
    s.put(ac.code[sym], ac.size[sym]);
    s.put((uint32_t)(v < 0 ? v - 1 : v), nb);
    run = 0;
  }
  if (run) s.put(ac.code[0], ac.size[0]);
}

// quantised zig-zag coefficients of the 8 x 8 block whose samples `smp` are (natural order, 0..255)
JPEG_HD inline void block_coefs(const int* smp, const Recip* q, int* zz) {
  int d[64];
  for (int i = 0; i < 64; i++) d[i] = smp[i] - 128;
  fdct_islow(d);
  for (int k = 0; k < 64; k++) {
    const int i = natural_order(k);
    zz[k] = quantize(d[i], q[i]);
  }
}

#ifndef __CUDA_ARCH__
inline size_t encode_frame(const uint8_t* bgr, int w, int h, int quality, uint8_t* out) {
  const Geometry g = geometry(w, h);
  Recip q[2][64];
  for (int t = 0; t < 2; t++)
    for (int i = 0; i < 64; i++) q[t][i] = compute_reciprocal((unsigned)quant_value(t, i, quality) << 3);
  static Huff hf[4];
  for (int t = 0; t < 4; t++) make_derived(t, hf[t]);
  BitSink s{out, (size_t)write_header(out, w, h, quality), 0, 0};
  int pred[3] = {0, 0, 0};
  for (int my = 0; my < g.mcuy; my++)
    for (int mx = 0; mx < g.mcux; mx++) {
      int zz[6][64], smp[64];
      for (int b = 0; b < 4; b++) {   // compress_data: blocks past the right edge copy the DC on their left, past the bottom
        const int bx = 2 * mx + (b & 1), by = 2 * my + (b >> 1);   // the DC of the MCU's last block above
        if (bx < g.ybw && by < g.ybh) {
          for (int i = 0; i < 64; i++) smp[i] = luma_at(bgr, g, 8 * bx + (i & 7), 8 * by + (i >> 3));
          block_coefs(smp, q[0], zz[b]);
        } else {
          for (int k = 0; k < 64; k++) zz[b][k] = 0;
          zz[b][0] = by < g.ybh ? zz[b - 1][0] : zz[1][0];
        }
      }
      for (int c = 0; c < 2; c++) {
        for (int i = 0; i < 64; i++) {
          const int ox = 8 * mx + (i & 7), oy = 8 * my + (i >> 3);
          const int y0 = chroma_src_row(g, 2 * oy), y1 = chroma_src_row(g, 2 * oy + 1);
          const int x0 = 2 * ox < w ? 2 * ox : w - 1, x1 = 2 * ox + 1 < w ? 2 * ox + 1 : w - 1;
          int v[4];
          const int xs[4] = {x0, x1, x0, x1}, ys[4] = {y0, y0, y1, y1};
          for (int j = 0; j < 4; j++) {
            const uint8_t* p = bgr + ((size_t)ys[j] * w + xs[j]) * 3;
            int Y, cb, cr;
            rgb_ycc(p[0], p[1], p[2], Y, cb, cr);
            v[j] = c == 0 ? cb : cr;
          }
          smp[i] = h2v2(v[0], v[1], v[2], v[3], ox);
        }
        block_coefs(smp, q[1], zz[4 + c]);
      }
      for (int b = 0; b < 4; b++) encode_block(s, zz[b], pred[0], hf[0], hf[1]);
      encode_block(s, zz[4], pred[1], hf[2], hf[3]);
      encode_block(s, zz[5], pred[2], hf[2], hf[3]);
    }
  s.flush();
  out[s.n++] = 0xFF;
  out[s.n++] = 0xD9;
  return s.n;
}

// The grey twin (nc = 1): grayscale_convert copies the plane, expand_right_edge / expand_bottom_edge replicate the last column
// and row into the padded blocks, and every block is an MCU.  plane: w * h bytes; `out` must hold encode_bound(w, h, 1).
inline size_t encode_grey_frame(const uint8_t* plane, int w, int h, int quality, uint8_t* out) {
  const Geometry g = geometry(w, h, 1);
  Recip q[64];
  for (int i = 0; i < 64; i++) q[i] = compute_reciprocal((unsigned)quant_value(0, i, quality) << 3);
  static Huff hf[2];
  for (int t = 0; t < 2; t++) make_derived(t, hf[t]);
  BitSink s{out, (size_t)write_header(out, w, h, quality, 1), 0, 0};
  int pred = 0;
  for (int by = 0; by < g.ybh; by++)
    for (int bx = 0; bx < g.ybw; bx++) {
      int zz[64], smp[64];
      for (int i = 0; i < 64; i++) {
        const int x = 8 * bx + (i & 7), y = 8 * by + (i >> 3);
        smp[i] = plane[(size_t)(y < h ? y : h - 1) * w + (x < w ? x : w - 1)];
      }
      block_coefs(smp, q, zz);
      encode_block(s, zz, pred, hf[0], hf[1]);
    }
  s.flush();
  out[s.n++] = 0xFF;
  out[s.n++] = 0xD9;
  return s.n;
}
#endif

}  // namespace jpegenc
