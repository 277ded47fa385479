// jpegdec.h - the sequential Huffman JPEG decoder of libjpeg-turbo 3.1.2 (the codec behind cv2.imread / cv2.imdecode of
// cv2 4.13.0) as OpenCV drives it - JDCT_ISLOW, do_fancy_upsampling = TRUE, output JCS_EXT_BGR (IMREAD_COLOR) or
// JCS_GRAYSCALE (IMREAD_GRAYSCALE) - restated in plain C++ that compiles for the host and the device.  csrc/jpegdec.cu runs
// this arithmetic batched on the GPU; decode_frame() below is the scalar reference for one frame, which only the host test
// compiles.  Every function names the libjpeg-turbo function it restates.
//
// Grey output of a YCbCr file is its Y component and nothing else: jdcolor.c's grayscale_convert copies component 0 and
// marks Cb and Cr as not needed, so their blocks are entropy-decoded (the scan interleaves them) but never transformed,
// upsampled or converted.  A different thing from cvtColor(BGR2GRAY) of the colour pixels.
//
// Accepted: baseline or extended sequential Huffman (SOF0, SOF1), 8-bit samples, one interleaved scan, one component (grey)
// or three YCbCr components with Cb = Cr = 1x1 and Y 1x1, 2x1, 1x2 or 2x2 (4:4:4, 4:2:2, 4:4:0, 4:2:0), any restart
// interval, any quantisation and Huffman tables.  Refused as unsupported: progressive, arithmetic, lossless, 12-bit,
// other sampling factors, multi-scan, four components, RGB-coded three-component files.
//
// Exif orientation: parse_header records the value cv2 4.13.0's Exif reader reports (exif_orientation below), and
// oriented_src() maps an output pixel to its stored pixel as cv2's ApplyExifOrientation flips and transposes.  A reader
// that applies it equals cv2.imdecode with its default flags; one that does not gives the stored orientation
// (cv2.IMREAD_IGNORE_ORIENTATION), which is also what cv2.imdecode returns for every file without an orientation tag.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define JPEG_HD __host__ __device__
#else
#define JPEG_HD
#endif

namespace jpegdec {

enum Status { OK = 0, INVALID = -1, UNSUPPORTED = -3 };   // the values of UWIP_OK, UWIP_ERR_INVALID, UWIP_ERR_UNSUPPORTED

constexpr int LOOK = 9;   // lookahead bits of the decoding tables (libjpeg's HUFF_LOOKAHEAD is 8; the result is the same)

// jpeg_natural_order (jutils.c): natural index of zig-zag position k
JPEG_HD inline int natural_order(int k) {
  constexpr unsigned char t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                   41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                   30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
  return t[k];
}

// ---- the marker reader (jdmarker.c) ------------------------------------------------------------------------------------
struct HuffSpec {   // a DHT table: bits[1..16], values
  uint8_t bits[17];
  uint8_t val[256];
  bool defined;
};
struct Component {
  int id, h, v, tq, td, ta;
};
struct Header {
  int width, height, ncomp;
  Component comp[4];
  uint16_t q[4][64];   // natural order
  bool qdef[4];
  HuffSpec dc[4], ac[4];
  int restart;         // restart interval in MCUs, 0: none
  bool jfif, adobe;
  int adobe_transform;
  size_t scan_off;     // first byte of the entropy-coded segment (after the SOS header)
  int orientation;     // the Exif orientation cv2 applies, 1..8 (1: none, or a value cv2 ignores)
};

struct Reader {
  const uint8_t* d;
  size_t len, pos;
  bool ok;
  int u8() {
    if (pos >= len) { ok = false; return 0; }
    return d[pos++];
  }
  int u16() { const int a = u8(); return (a << 8) | u8(); }
};

// The orientation cv2 4.13.0 takes from the payload of one APP1 segment (OpenCV's ExifReader over the TIFF structure after
// "Exif\0\0", as it behaves, not as TIFF specifies): -1 when the segment gives no orientation entry, so that the next Exif
// APP1 is read; otherwise the entry's value, which cv2 applies only when it lies in 1..8.
//  - The byte order is little-endian for "II" and big-endian for anything else, "MM" or not; the next u16 must be 42.
//  - IFD0 is wherever the u32 at offset 4 points; IFD1 and later directories are not read.
//  - Entries are read in order; the first orientation tag (0x0112) wins, whatever its type and count: its value is the u16 at
//    the entry's value field, so a LONG value reads as 0 in a big-endian file.
//  - Every read must lie inside the payload, or the segment gives nothing from that read on (an entry count running past the
//    segment is harmless when the orientation tag comes first).
inline int exif_orientation(const uint8_t* p, size_t n) {
  if (n < 6 || memcmp(p, "Exif\0\0", 6) != 0) return -1;
  p += 6;
  n -= 6;
  const bool le = n >= 2 && p[0] == 'I' && p[1] == 'I';
  auto u16 = [&](uint64_t o) -> int { return o + 2 > n ? -1 : le ? p[o] | p[o + 1] << 8 : p[o] << 8 | p[o + 1]; };
  if (u16(2) != 42 || n < 8) return -1;
  const uint64_t ifd = le ? (uint32_t)p[4] | (uint32_t)p[5] << 8 | (uint32_t)p[6] << 16 | (uint32_t)p[7] << 24
                          : (uint32_t)p[4] << 24 | (uint32_t)p[5] << 16 | (uint32_t)p[6] << 8 | (uint32_t)p[7];
  const int count = u16(ifd);
  for (int k = 0; k < count; k++) {
    const uint64_t e = ifd + 2 + 12 * (uint64_t)k;
    const int tag = u16(e);
    if (tag < 0) return -1;
    if (tag == 0x0112) return u16(e + 8);
  }
  return -1;
}

// read_markers / first_marker / next_marker / get_sof / get_sos / get_dht / get_dqt / get_dri / examine_app0 / examine_app14 /
// skip_variable, then the colour-space decision of default_decompress_parms (jdapimin.c) and the checks of initial_setup
// (jdinput.c) and jinit_upsampler (jdsample.c) that this decoder restricts further.  Stops after the first SOS.
inline int parse_header(const uint8_t* data, size_t len, Header& hd) {
  memset(&hd, 0, sizeof(hd));
  hd.orientation = 1;
  bool exif = false;   // an Exif APP1 gave an orientation entry: later ones are not read
  Reader r{data, len, 0, true};
  if (r.u8() != 0xFF || r.u8() != 0xD8 || !r.ok) return INVALID;   // first_marker: SOI
  bool sof = false;
  for (;;) {
    int c = r.u8();
    while (r.ok && c != 0xFF) c = r.u8();   // next_marker: garbage before a marker is skipped
    do { c = r.u8(); } while (r.ok && c == 0xFF);
    if (!r.ok) return INVALID;
    if (c == 0xC0 || c == 0xC1) {   // get_sof: baseline / extended sequential Huffman
      if (sof) return INVALID;
      sof = true;
      const int length = r.u16() - 2;
      const int prec = r.u8();
      hd.height = r.u16();
      hd.width = r.u16();
      hd.ncomp = r.u8();
      if (!r.ok) return INVALID;
      if (prec != 8) return UNSUPPORTED;
      if (hd.height <= 0 || hd.width <= 0 || hd.ncomp <= 0) return INVALID;
      if (length != hd.ncomp * 3 + 6) return INVALID;
      if (hd.width > 65500 || hd.height > 65500) return INVALID;   // JPEG_MAX_DIMENSION
      if (hd.ncomp > 4) return UNSUPPORTED;
      for (int i = 0; i < hd.ncomp; i++) {
        hd.comp[i].id = r.u8();
        const int hv = r.u8();
        hd.comp[i].h = hv >> 4;
        hd.comp[i].v = hv & 15;
        hd.comp[i].tq = r.u8();
        if (hd.comp[i].h < 1 || hd.comp[i].h > 4 || hd.comp[i].v < 1 || hd.comp[i].v > 4 || hd.comp[i].tq > 3) return INVALID;
      }
      if (!r.ok) return INVALID;
    } else if (c == 0xC2 || c == 0xC3 || (c >= 0xC5 && c <= 0xC7) || (c >= 0xC9 && c <= 0xCB) || (c >= 0xCD && c <= 0xCF)) {
      return UNSUPPORTED;   // progressive, lossless, differential, arithmetic
    } else if (c == 0xC4) {   // get_dht
      int length = r.u16() - 2;
      while (length > 16) {
        int index = r.u8();
        uint8_t bits[17];
        bits[0] = 0;
        int count = 0;
        for (int i = 1; i <= 16; i++) { bits[i] = (uint8_t)r.u8(); count += bits[i]; }
        length -= 1 + 16;
        if (!r.ok || count > 256 || count > length) return INVALID;
        HuffSpec* t;
        if (index & 0x10) { index -= 0x10; t = hd.ac; } else { t = hd.dc; }
        if (index < 0 || index >= 4) return INVALID;
        memcpy(t[index].bits, bits, 17);
        memset(t[index].val, 0, 256);
        for (int i = 0; i < count; i++) t[index].val[i] = (uint8_t)r.u8();
        t[index].defined = true;
        length -= count;
        if (!r.ok) return INVALID;
      }
      if (length != 0) return INVALID;
    } else if (c == 0xDB) {   // get_dqt
      int length = r.u16() - 2;
      while (length > 0) {
        const int n = r.u8();
        const int prec = n >> 4, t = n & 15;
        length--;
        if (!r.ok || t >= 4 || length < (prec ? 128 : 64)) return INVALID;
        for (int i = 0; i < 64; i++) hd.q[t][natural_order(i)] = (uint16_t)(prec ? r.u16() : r.u8());
        hd.qdef[t] = true;
        length -= prec ? 128 : 64;
        if (!r.ok) return INVALID;
      }
      if (length != 0) return INVALID;
    } else if (c == 0xDD) {   // get_dri
      if (r.u16() != 4) return INVALID;
      hd.restart = r.u16();
      if (!r.ok) return INVALID;
    } else if (c == 0xDA) {   // get_sos
      if (!sof) return INVALID;
      const int length = r.u16();
      const int ns = r.u8();
      if (!r.ok || length != ns * 2 + 6 || ns < 1 || ns > 4) return INVALID;
      bool seen[4] = {false, false, false, false};
      for (int i = 0; i < ns; i++) {
        const int id = r.u8(), t = r.u8();
        int ci = 0;
        while (ci < hd.ncomp && (hd.comp[ci].id != id || seen[ci])) ci++;
        if (ci == hd.ncomp) return INVALID;
        seen[ci] = true;
        hd.comp[ci].td = t >> 4;
        hd.comp[ci].ta = t & 15;
        if (hd.comp[ci].td > 3 || hd.comp[ci].ta > 3) return INVALID;
      }
      r.u8(); r.u8(); r.u8();   // Ss, Se, Ah/Al: a sequential scan takes them as 0, 63, 0
      if (!r.ok) return INVALID;
      hd.scan_off = r.pos;
      // default_decompress_parms
      if (hd.ncomp == 3) {
        bool rgb;
        if (hd.jfif) rgb = false;
        else if (hd.adobe) rgb = hd.adobe_transform == 0;
        else rgb = hd.comp[0].id == 82 && hd.comp[1].id == 71 && hd.comp[2].id == 66;
        if (rgb) return UNSUPPORTED;
      } else if (hd.ncomp != 1) {
        return UNSUPPORTED;   // CMYK / YCCK and other component counts
      }
      if (ns != hd.ncomp) return UNSUPPORTED;   // a multi-scan sequential file
      if (hd.ncomp == 3) {
        const int hy = hd.comp[0].h, vy = hd.comp[0].v;
        for (int i = 1; i < 3; i++)
          if (hd.comp[i].h != 1 || hd.comp[i].v != 1) return UNSUPPORTED;
        if (hy > 2 || vy > 2) return UNSUPPORTED;
      }
      for (int i = 0; i < hd.ncomp; i++) {   // latch_quant_tables, jpeg_make_d_derived_tbl's missing-table check
        if (!hd.qdef[hd.comp[i].tq] || !hd.dc[hd.comp[i].td].defined || !hd.ac[hd.comp[i].ta].defined) return INVALID;
      }
      return OK;
    } else if (c == 0xD9) {   // EOI before any scan: no image
      return INVALID;
    } else if (c == 0xE0 || c == 0xEE) {   // examine_app0 / examine_app14
      const int length = r.u16() - 2;
      if (!r.ok || length < 0 || r.pos + (size_t)length > len) return INVALID;
      const uint8_t* p = data + r.pos;
      if (c == 0xE0 && length >= 14 && p[0] == 'J' && p[1] == 'F' && p[2] == 'I' && p[3] == 'F' && p[4] == 0) hd.jfif = true;
      if (c == 0xEE && length >= 12 && p[0] == 'A' && p[1] == 'd' && p[2] == 'o' && p[3] == 'b' && p[4] == 'e') {
        hd.adobe = true;
        hd.adobe_transform = p[11];
      }
      r.pos += length;
    } else if ((c >= 0xE1 && c <= 0xEF) || c == 0xFE || c == 0xCC || c == 0xDC) {   // APPn, COM, DAC, DNL: skip_variable
      const int length = r.u16() - 2;
      if (!r.ok || length < 0 || r.pos + (size_t)length > len) return INVALID;
      if (c == 0xE1 && !exif) {
        const int o = exif_orientation(data + r.pos, (size_t)length);
        exif = o >= 0;
        if (o >= 1 && o <= 8) hd.orientation = o;
      }
      r.pos += length;
    } else if ((c >= 0xD0 && c <= 0xD7) || c == 0x01) {   // RSTn, TEM: no parameters
    } else {
      return INVALID;   // JERR_UNKNOWN_MARKER (SOI again, JPG, reserved codes)
    }
  }
}

// ---- jpeg_make_d_derived_tbl (jdhuff.c) --------------------------------------------------------------------------------
// look[c]: (length << 8) | symbol of the code that the LOOK-bit prefix c starts with, 0 when the code is longer.
// maxcode[l]: the largest code of length l (-1: none); valoff[l]: value index minus code for length l.
struct DTbl {
  uint16_t look[1 << LOOK];
  int32_t maxcode[18];
  int32_t valoff[18];
  uint8_t val[256];
};

inline bool make_derived(const HuffSpec& s, bool is_dc, DTbl& t) {
  uint8_t size[257];
  uint32_t code[257];
  int p = 0;
  for (int l = 1; l <= 16; l++) {
    const int i = s.bits[l];
    if (p + i > 256) return false;
    for (int k = 0; k < i; k++) size[p++] = (uint8_t)l;
  }
  size[p] = 0;
  const int nsym = p;
  uint32_t c = 0;
  int si = size[0];
  p = 0;
  while (size[p]) {
    while (size[p] == si) { code[p++] = c; c++; }
    if (c >= (1u << si)) return false;   // no code may be all ones
    c <<= 1;
    si++;
  }
  p = 0;
  for (int l = 1; l <= 16; l++) {
    if (s.bits[l]) {
      t.valoff[l] = p - (int32_t)code[p];
      p += s.bits[l];
      t.maxcode[l] = (int32_t)code[p - 1];
    } else {
      t.valoff[l] = 0;
      t.maxcode[l] = -1;
    }
  }
  t.valoff[0] = t.maxcode[0] = 0;
  t.valoff[17] = 0;
  t.maxcode[17] = 0xFFFFF;
  memcpy(t.val, s.val, 256);
  memset(t.look, 0, sizeof(t.look));
  p = 0;
  for (int l = 1; l <= LOOK; l++)
    for (int i = 1; i <= s.bits[l]; i++, p++) {
      const uint32_t base = code[p] << (LOOK - l);
      for (uint32_t k = 0; k < (1u << (LOOK - l)); k++) t.look[base + k] = (uint16_t)((l << 8) | s.val[p]);
    }
  if (is_dc)
    for (int i = 0; i < nsym; i++)
      if (s.val[i] > 15) return false;
  return true;
}

// ---- bit reader over a destuffed stream (fill_bit_buffer without markers: they were taken out) ---------------------------
// The stream is read in aligned big-endian 32-bit words; its buffer must be 4-byte aligned and readable 16 bytes past the
// last bit a decode may look at.
JPEG_HD inline uint32_t be32(const uint8_t* p) {
#ifdef __CUDA_ARCH__
  return __byte_perm(__ldg(reinterpret_cast<const unsigned int*>(p)), 0, 0x0123);
#else
  return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
#endif
}
struct Bits {
  const uint8_t* s;
  uint64_t acc;   // the next n bits, MSB-aligned
  int n;
  uint32_t w;     // next word
  uint32_t p;     // bit position of acc's top bit
  JPEG_HD void init(const uint8_t* base, uint32_t bit) {
    s = base;
    w = bit >> 5;
    acc = ((uint64_t)be32(s + 4 * (size_t)w) << 32) | be32(s + 4 * (size_t)w + 4);
    w += 2;
    acc <<= (bit & 31);
    n = 64 - (int)(bit & 31);
    p = bit;
  }
  JPEG_HD uint32_t peek(int k) const { return (uint32_t)(acc >> (64 - k)); }   // 1 <= k <= 32
  JPEG_HD void skip(int k) {                                                    // 0 <= k <= 32
    acc <<= k;
    n -= k;
    p += k;
    if (n < 32) {
      acc |= (uint64_t)be32(s + 4 * (size_t)w) << (32 - n);
      w++;
      n += 32;
    }
  }
};

// jpeg_huff_decode / HUFF_DECODE: the symbol, or -1 for a bit pattern no code of the table starts
JPEG_HD inline int huff_decode(const DTbl& t, Bits& b) {
  const int e = t.look[b.peek(LOOK)];
  if (e) {
    b.skip(e >> 8);
    return e & 255;
  }
  const uint32_t c16 = b.peek(16);
  for (int l = LOOK + 1; l <= 16; l++) {
    const int32_t c = (int32_t)(c16 >> (16 - l));
    if (c <= t.maxcode[l]) {
      b.skip(l);
      return t.val[(c + t.valoff[l]) & 255];
    }
  }
  return -1;
}

// HUFF_EXTEND (jdhuff.c)
JPEG_HD inline int huff_extend(int x, int s) { return x < (1 << (s - 1)) ? x + (int)((~0u << s) + 1u) : x; }

// One step of decode_mcu (jdhuff.c): the codeword (and its extra bits) that starts at b.p in state (block of the MCU `blk`,
// coefficient index z: 0 = DC, 1..63 = the next AC position).  Outputs: what was decoded (kind 0: DC difference `v`,
// kind 1: AC coefficient `v` at zig-zag `zz`, kind 2: nothing stored) and whether the block is complete.  Returns false for
// an invalid code (one bit is then skipped so that a speculative decode goes on deterministically) or a coefficient past 63.
struct Step {
  int kind, v, zz;
  bool done;
};
JPEG_HD inline bool decode_step(const DTbl& dc, const DTbl& ac, Bits& b, int& z, Step& st) {
  st.done = false;
  st.kind = 2;
  if (z == 0) {
    const int s = huff_decode(dc, b);
    if (s < 0) { b.skip(1); return false; }
    int v = 0;
    if (s) { v = huff_extend((int)b.peek(s), s); b.skip(s); }
    st.kind = 0;
    st.v = v;
    z = 1;
    return true;
  }
  const int sym = huff_decode(ac, b);
  if (sym < 0) { b.skip(1); return false; }
  const int r = sym >> 4, s = sym & 15;
  if (s) {
    z += r;
    const int v = huff_extend((int)b.peek(s), s);
    b.skip(s);
    if (z > 63) { st.done = true; z = 64; return false; }
    st.kind = 1;
    st.v = v;
    st.zz = z;
    z++;
  } else if (r == 15) {
    z += 16;
  } else {
    z = 64;   // EOB
  }
  if (z >= 64) st.done = true;
  return true;
}

// ---- jpeg_idct_islow (jidctint.c) with the dequantisation and IDCT_range_limit ------------------------------------------
JPEG_HD inline int range_limit(int x) {   // sample_range_limit + CENTERJSAMPLE, indexed by x & RANGE_MASK (jdmaster.c)
  x &= 1023;
  if (x >= 512) x -= 1024;
  x += 128;
  return x < 0 ? 0 : (x > 255 ? 255 : x);
}
JPEG_HD inline void idct_1d(int64_t d0, int64_t d1, int64_t d2, int64_t d3, int64_t d4, int64_t d5, int64_t d6, int64_t d7,
                            int shift, int64_t* o) {
  // even part
  int64_t z2 = d2, z3 = d6;
  int64_t z1 = (z2 + z3) * 4433;                 // FIX_0_541196100
  const int64_t tmp2 = z1 + z3 * -15137;         // FIX_1_847759065
  const int64_t tmp3 = z1 + z2 * 6270;           // FIX_0_765366865
  const int64_t tmp0 = (d0 + d4) * 8192, tmp1 = (d0 - d4) * 8192;
  const int64_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
  // odd part
  int64_t t0 = d7, t1 = d5, t2 = d3, t3 = d1;
  z1 = t0 + t3;
  z2 = t1 + t2;
  z3 = t0 + t2;
  int64_t z4 = t1 + t3;
  const int64_t z5 = (z3 + z4) * 9633;           // FIX_1_175875602
  t0 *= 2446;                                    // FIX_0_298631336
  t1 *= 16819;                                   // FIX_2_053119869
  t2 *= 25172;                                   // FIX_3_072711026
  t3 *= 12299;                                   // FIX_1_501321110
  z1 *= -7373;                                   // FIX_0_899976223
  z2 *= -20995;                                  // FIX_2_562915447
  z3 = z3 * -16069 + z5;                         // FIX_1_961570560
  z4 = z4 * -3196 + z5;                          // FIX_0_390180644
  t0 += z1 + z3;
  t1 += z2 + z4;
  t2 += z2 + z3;
  t3 += z1 + z4;
  const int64_t r = (int64_t)1 << (shift - 1);
  o[0] = (tmp10 + t3 + r) >> shift;
  o[7] = (tmp10 - t3 + r) >> shift;
  o[1] = (tmp11 + t2 + r) >> shift;
  o[6] = (tmp11 - t2 + r) >> shift;
  o[2] = (tmp12 + t1 + r) >> shift;
  o[5] = (tmp12 - t1 + r) >> shift;
  o[3] = (tmp13 + t0 + r) >> shift;
  o[4] = (tmp13 - t0 + r) >> shift;
}
// coef: 64 int16 coefficients in natural order; q: quantisers in natural order; out: 8 rows of 8 samples, row stride `stride`
JPEG_HD inline void idct_islow(const int16_t* coef, const uint16_t* q, uint8_t* out, size_t stride) {
  int32_t ws[64];   // the workspace is int
  for (int c = 0; c < 8; c++) {   // pass 1: columns, CONST_BITS - PASS1_BITS
    int64_t o[8];
    idct_1d((int64_t)coef[c] * q[c], (int64_t)coef[8 + c] * q[8 + c], (int64_t)coef[16 + c] * q[16 + c],
            (int64_t)coef[24 + c] * q[24 + c], (int64_t)coef[32 + c] * q[32 + c], (int64_t)coef[40 + c] * q[40 + c],
            (int64_t)coef[48 + c] * q[48 + c], (int64_t)coef[56 + c] * q[56 + c], 13 - 2, o);
    for (int r = 0; r < 8; r++) ws[8 * r + c] = (int32_t)o[r];
  }
  for (int r = 0; r < 8; r++) {   // pass 2: rows, CONST_BITS + PASS1_BITS + 3
    const int32_t* w = ws + 8 * r;
    int64_t o[8];
    idct_1d(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], 13 + 2 + 3, o);
    for (int c = 0; c < 8; c++) out[(size_t)r * stride + c] = (uint8_t)range_limit((int)o[c]);
  }
}

// ---- frame geometry (jdinput.c initial_setup, per_scan_setup) ----------------------------------------------------------
// Blocks are numbered in decoding order: MCU after MCU, inside an MCU the hy x vy luma blocks row by row, then Cb, then Cr
// (grey: one block per MCU).  The sample planes are padded to whole MCUs; dw, dh are the real (downsampled) sizes.
struct Geo {
  int w, h, ncomp, hy, vy, bpm, mcux, mcuy, nmcu, ri, nint;
  int pw[3], ph[3], dw[3], dh[3];
  size_t poff[3], nblocks, nsamples;
};
inline Geo geometry(const Header& hd) {
  Geo g;
  memset(&g, 0, sizeof(g));
  g.w = hd.width;
  g.h = hd.height;
  g.ncomp = hd.ncomp;
  if (hd.ncomp == 1) {   // a non-interleaved scan: the MCU is one block whatever the sampling factors
    g.hy = g.vy = 1;
    g.bpm = 1;
    g.mcux = (g.w + 7) / 8;
    g.mcuy = (g.h + 7) / 8;
    g.pw[0] = 8 * g.mcux;
    g.ph[0] = 8 * g.mcuy;
    g.dw[0] = g.w;
    g.dh[0] = g.h;
  } else {
    g.hy = hd.comp[0].h;
    g.vy = hd.comp[0].v;
    g.bpm = g.hy * g.vy + 2;
    g.mcux = (g.w + 8 * g.hy - 1) / (8 * g.hy);
    g.mcuy = (g.h + 8 * g.vy - 1) / (8 * g.vy);
    g.pw[0] = 8 * g.hy * g.mcux;
    g.ph[0] = 8 * g.vy * g.mcuy;
    g.dw[0] = g.w;
    g.dh[0] = g.h;
    for (int c = 1; c < 3; c++) {
      g.pw[c] = 8 * g.mcux;
      g.ph[c] = 8 * g.mcuy;
      g.dw[c] = (g.w + g.hy - 1) / g.hy;   // downsampled_width = ceil(W * h / max_h)
      g.dh[c] = (g.h + g.vy - 1) / g.vy;
    }
  }
  g.nmcu = g.mcux * g.mcuy;
  g.ri = hd.restart;
  g.nint = g.ri ? (g.nmcu + g.ri - 1) / g.ri : 1;
  g.nblocks = (size_t)g.nmcu * g.bpm;
  size_t o = 0;
  for (int c = 0; c < g.ncomp; c++) {
    g.poff[c] = o;
    o += (size_t)g.pw[c] * g.ph[c];
  }
  g.nsamples = o;
  return g;
}
// component of block b of an MCU
JPEG_HD inline int block_comp(const Geo& g, int b) { return b < g.hy * g.vy ? 0 : b - g.hy * g.vy + 1; }
// sample-plane position (in blocks) of block b of MCU m
JPEG_HD inline void block_pos(const Geo& g, int m, int b, int& c, int& bx, int& by) {
  const int mx = m % g.mcux, my = m / g.mcux;
  c = block_comp(g, b);
  if (c == 0) {
    bx = mx * g.hy + b % g.hy;
    by = my * g.vy + b / g.hy;
  } else {
    bx = mx;
    by = my;
  }
}

// ---- upsampling (jdsample.c) and colour conversion (jdcolor.c) of one output pixel --------------------------------------
// The chroma sample of output pixel (x, y) for the upsampler jinit_upsampler picks: fullsize_upsample (4:4:4);
// h2v1_fancy_upsample, h1v2_fancy_upsample, h2v2_fancy_upsample with the context rows of jdmainct.c (the first and last real
// rows replicated); h2v1_upsample / h2v2_upsample when downsampled_width <= 2.  p: the plane, stride pw.
JPEG_HD inline int chroma_at(const uint8_t* p, int pw, int dw, int dh, int hy, int vy, int x, int y) {
  if (hy == 1 && vy == 1) return p[(size_t)y * pw + x];
  const bool fancy = hy == 1 || dw > 2;   // h1v2 is fancy at every width
  if (!fancy) return p[(size_t)(y / vy) * pw + x / hy];
  if (vy == 1) {   // h2v1_fancy_upsample
    const uint8_t* s = p + (size_t)y * pw;
    const int i = x >> 1;
    if ((x & 1) == 0) return i == 0 ? s[0] : (3 * s[i] + s[i - 1] + 1) >> 2;
    return i == dw - 1 ? s[i] : (3 * s[i] + s[i + 1] + 2) >> 2;
  }
  const int j = y >> 1;
  const int jn = (y & 1) ? (j + 1 < dh ? j + 1 : dh - 1) : (j > 0 ? j - 1 : 0);
  const uint8_t* s0 = p + (size_t)j * pw;
  const uint8_t* s1 = p + (size_t)jn * pw;
  if (hy == 1) return (3 * s0[x] + s1[x] + ((y & 1) ? 2 : 1)) >> 2;   // h1v2_fancy_upsample
  const int i = x >> 1;                                                // h2v2_fancy_upsample
  const int c = 3 * s0[i] + s1[i];
  if ((x & 1) == 0) return i == 0 ? (4 * c + 8) >> 4 : (3 * c + 3 * s0[i - 1] + s1[i - 1] + 8) >> 4;
  return i == dw - 1 ? (4 * c + 7) >> 4 : (3 * c + 3 * s0[i + 1] + s1[i + 1] + 7) >> 4;
}
// build_ycc_rgb_table + ycc_rgb_convert (SCALEBITS 16) into B, G, R
JPEG_HD inline void ycc_bgr(int y, int cb, int cr, uint8_t* o) {
  cb -= 128;
  cr -= 128;
  const int r = y + ((91881 * cr + 32768) >> 16);
  const int g = y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
  const int b = y + ((116130 * cb + 32768) >> 16);
  o[0] = (uint8_t)(b < 0 ? 0 : (b > 255 ? 255 : b));
  o[1] = (uint8_t)(g < 0 ? 0 : (g > 255 ? 255 : g));
  o[2] = (uint8_t)(r < 0 ? 0 : (r > 255 ? 255 : r));
}
// output pixel (x, y) of the frame whose sample planes start at `smp` (gray_rgb_convert for one component)
JPEG_HD inline void pixel(const Geo& g, const uint8_t* smp, int x, int y, uint8_t* o) {
  const int Y = smp[(size_t)y * g.pw[0] + x];
  if (g.ncomp == 1) {
    o[0] = o[1] = o[2] = (uint8_t)Y;
    return;
  }
  const int cb = chroma_at(smp + g.poff[1], g.pw[1], g.dw[1], g.dh[1], g.hy, g.vy, x, y);
  const int cr = chroma_at(smp + g.poff[2], g.pw[2], g.dw[2], g.dh[2], g.hy, g.vy, x, y);
  ycc_bgr(Y, cb, cr, o);
}

// ---- Exif orientation (OpenCV's ApplyExifOrientation) ---------------------------------------------------------------------
// The stored pixel (sx, sy) that output pixel (x, y) of orientation o shows; w x h is the output size (the stored size is
// w x h for o = 1..4 and h x w for 5..8).  2: flip(1), 3: flip(-1), 4: flip(0); 5: transpose, 6: transpose + flip(1),
// 7: transpose + flip(-1), 8: transpose + flip(0).
JPEG_HD inline void oriented_src(int o, int w, int h, int x, int y, int& sx, int& sy) {
  const int fx = o == 2 || o == 3 || o == 6 || o == 7 ? w - 1 - x : x;
  const int fy = o == 3 || o == 4 || o == 7 || o == 8 ? h - 1 - y : y;
  if (o >= 5) {
    sx = fy;
    sy = fx;
  } else {
    sx = fx;
    sy = fy;
  }
}

// ---- destuffing: the bytes fill_bit_buffer hands to the decoder -----------------------------------------------------------
// Kind of byte i of the entropy-coded segment s[0..len): 0 data, 1 dropped (stuffed 0x00, fill 0xFF, RSTn marker), 2 RSTn
// code byte (dropped; a restart interval ends before it), 3 the 0xFF of any other marker: the segment ends there.
JPEG_HD inline int byte_kind(int prev, int b, int next) {   // prev / next: -1 outside the segment
  if (b == 0xFF) {
    if (next == 0x00) return 0;
    if (next == 0xFF || (next >= 0xD0 && next <= 0xD7)) return 1;
    return 3;
  }
  if (prev == 0xFF) {
    if (b == 0x00) return 1;
    if (b >= 0xD0 && b <= 0xD7) return 2;
  }
  return 0;
}

#ifndef __CUDA_ARCH__
// The scalar reference of one frame: decode_mcu over the whole scan with process_restart, decompress_onepass's IDCTs, then
// upsampling and colour conversion.  out: w * h * 3 bytes, or w * h for grey (IMREAD_GRAYSCALE: the IDCTs of component 0
// only, cropped).  orient: the frame is then turned by the Exif orientation (h x w for 5..8), as cv2.imdecode's default
// flags do.  Returns OK, INVALID, UNSUPPORTED, or 1 for bad entropy-coded data (the frame is then all zeros, as the batched
// decoder leaves it).
inline int decode_frame(const uint8_t* data, size_t len, uint8_t* out, bool grey = false, bool orient = false) {
  Header hd;
  int rc = parse_header(data, len, hd);
  if (rc != OK) return rc;
  if (orient && hd.orientation != 1) {
    const int ch = grey ? 1 : 3, o = hd.orientation, w = o >= 5 ? hd.height : hd.width, h = o >= 5 ? hd.width : hd.height;
    uint8_t* st = new uint8_t[(size_t)hd.width * hd.height * ch];
    rc = decode_frame(data, len, st, grey, false);
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        int sx, sy;
        oriented_src(o, w, h, x, y, sx, sy);
        memcpy(out + ((size_t)y * w + x) * ch, st + ((size_t)sy * hd.width + sx) * ch, ch);
      }
    delete[] st;
    return rc;
  }
  static DTbl dct[3], act[3];
  for (int c = 0; c < hd.ncomp; c++)
    if (!make_derived(hd.dc[hd.comp[c].td], true, dct[c]) || !make_derived(hd.ac[hd.comp[c].ta], false, act[c])) return INVALID;
  const Geo g = geometry(hd);
  // destuff, recording where each restart interval starts
  const uint8_t* seg = data + hd.scan_off;
  const size_t slen = len - hd.scan_off;
  uint8_t* cs = new uint8_t[slen + 32]();
  size_t* istart = new size_t[g.nint + 1];
  size_t n = 0;
  int nrst = 0;
  bool bad = false;
  istart[0] = 0;
  for (size_t i = 0; i < slen; i++) {
    const int k = byte_kind(i ? seg[i - 1] : -1, seg[i], i + 1 < slen ? seg[i + 1] : -1);
    if (k == 3) break;
    if (k == 0) cs[n++] = seg[i];
    if (k == 2) {
      if (++nrst < g.nint) istart[nrst] = n;
    }
  }
  if (nrst != g.nint - 1) bad = true;
  istart[g.nint] = n;
  uint8_t* smp = new uint8_t[g.nsamples]();
  int16_t blk[64];
  for (int k = 0; k < g.nint && !bad; k++) {
    const uint32_t lim = (uint32_t)(istart[k + 1] * 8);
    Bits b;
    b.init(cs, (uint32_t)(istart[k] * 8));
    int pred[3] = {0, 0, 0};
    const int m1 = g.ri ? (k + 1) * g.ri < g.nmcu ? (k + 1) * g.ri : g.nmcu : g.nmcu;
    for (int m = g.ri ? k * g.ri : 0; m < m1 && !bad; m++)
      for (int bi = 0; bi < g.bpm && !bad; bi++) {
        int c, bx, by;
        block_pos(g, m, bi, c, bx, by);
        for (int i = 0; i < 64; i++) blk[i] = 0;
        int z = 0;
        Step st;
        do {
          if (!decode_step(dct[c], act[c], b, z, st) || b.p > lim) { bad = true; break; }
          if (st.kind == 0) { pred[c] += st.v; blk[0] = (int16_t)pred[c]; }
          if (st.kind == 1) blk[natural_order(st.zz)] = (int16_t)st.v;
        } while (!st.done);
        if (!bad && (!grey || c == 0)) idct_islow(blk, hd.q[hd.comp[c].tq], smp + g.poff[c] + (size_t)8 * by * g.pw[c] + 8 * bx, g.pw[c]);
      }
  }
  if (bad) {
    memset(out, 0, (size_t)g.w * g.h * (grey ? 1 : 3));
  } else if (grey) {
    for (int y = 0; y < g.h; y++) memcpy(out + (size_t)y * g.w, smp + (size_t)y * g.pw[0], g.w);
  } else {
    for (int y = 0; y < g.h; y++)
      for (int x = 0; x < g.w; x++) pixel(g, smp, x, y, out + ((size_t)y * g.w + x) * 3);
  }
  delete[] cs;
  delete[] istart;
  delete[] smp;
  return bad ? 1 : OK;
}
#endif

}  // namespace jpegdec
