"""CPU oracle for the histretch -> aclahe -> bgdehaze path (pure numpy).

TEST INFRASTRUCTURE ONLY.  Nothing in the product path (uwimageproc_b200/, include/,
the C-ABI library) may import, call or link this file.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs use it,
and there only as the checker or as the timed CPU baseline.

It restates, in plain numpy, the algorithm the reference runs on the CPU:

  * modules/common/preprocessing.cpp:25-34   getHistogram
  * modules/common/preprocessing.cpp:74-105  imgChannelStretch
  * modules/common/preprocessing.cpp:147-161 numChannel / numSpace
  * modules/histretch/src/histretch.cpp:153-156,219-254  channel loop (literal + intended)
  * modules/aclahe/src/aclahe.cpp:152-193,228-248        HSV wrapper, sweep, aclaheEntropy
  * modules/aclahe/python/functions.py:14-27             Entropia, CLAHE
  * modules/aclahe/python/ACLAHE.py:15                   GaussianBlur 3x3 pre-filter
  * modules/bgdehaze/BGDehaze.py:14-89, guidedfilter.py:23-103, main.py:16-19

The pixel arithmetic of the first two modules lives in a third-party dependency that is
NOT vendored in the reference: OpenCV (documented pin 3.4.6, INSTALL.md:3,47-62; the
only OpenCV that can be executed in this image is the cv2 4.13.0 wheel).  The OpenCV
calls on the path (calcHist, Mat += / *=, cvtColor BGR<->HSV / BGR2YCrCb, CLAHE::apply,
GaussianBlur) are restated here from their published algorithm (SURVEY.md appendix A)
and PINNED against cv2 4.13.0 outputs: tests/golden/*.json|npz are produced by
oracle/make_golden.py (cv2 + the reference's own .py files imported from
/root/reference) and tests/test_oracle_*.py replays them; when cv2 is importable the
tests also compare live.

Float conventions: "f32" means every operation rounds to IEEE binary32 with no FMA
contraction unless fma is written; rint = round-half-to-even; sat = clamp to [0,255].
"""
from __future__ import annotations

import math
import zlib

import numpy as np

F32 = np.float32

# ----------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------


def crc32(a: np.ndarray) -> str:
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


def _sat_u8_from_rint(x: np.ndarray) -> np.ndarray:
    """saturate_cast<uchar>(cvRound(x)) for float input; NaN / +-inf -> INT_MIN -> 0."""
    x = np.asarray(x)
    bad = ~np.isfinite(x)
    r = np.rint(np.where(bad, 0, x))
    r = np.clip(r, 0, 255)
    r = np.where(bad, 0, r)
    return r.astype(np.uint8)


# ----------------------------------------------------------------------------------------
# histretch  (preprocessing.cpp)
# ----------------------------------------------------------------------------------------


def num_channel(c: str) -> int:
    """preprocessing.cpp:147-152 (note 'R'->0 and 'B'->2 although planes are B,G,R)."""
    if c in "RHhLY":
        return 0
    if c in "GSsaC":
        return 1
    if c in "BVlbX":
        return 2
    return -1


def num_space(c: str) -> int:
    """preprocessing.cpp:154-161: 0 BGR, 1 HSV, 2 HLS, 3 Lab, 4 YCrCb, -1 unknown."""
    if c in "RGB":
        return 0
    if c in "HSV":
        return 1
    if c in "hsl":
        return 2
    if c in "Lab":
        return 3
    if c in "YCX":
        return 4
    return -1


def get_histogram(plane: np.ndarray) -> np.ndarray:
    """preprocessing.cpp:25-34: 256-bin calcHist of an 8U plane, returned as float32[256]."""
    plane = np.asarray(plane)
    assert plane.dtype == np.uint8
    return np.bincount(plane.ravel(), minlength=256).astype(F32)


def percentile_bins(hist: np.ndarray, width: int, height: int, lo: int, hi: int):
    """The float32 while-loop of preprocessing.cpp:80-94.  Returns (low, high) as ints;
    low == -1 when lo == 0.  The reference reads past bin 255 (UB) if the threshold is never
    reached; here the loop stops at i == 256."""
    norm = F32(height * width / 100.0)
    lo_thr = F32(F32(lo) * norm)
    hi_thr = F32(F32(hi) * norm)
    s = F32(0.0)
    low = -1
    high = -1
    i = 0
    while s < hi_thr and i < 256:
        if s < lo_thr:
            low += 1
        high += 1
        s = F32(s + F32(hist[i]))
        i += 1
    return low, high


def stretch_lut(low: int, high: int) -> np.ndarray:
    """Net effect of `img += b; img *= m` (preprocessing.cpp:96-100) as a 256-entry LUT:
    y = sat(x + b) (cv::add with an integral scalar), z = sat(rint(f32(y) * m))
    (Mat::convertTo(-1, m): one float32 multiply)."""
    x = np.arange(256, dtype=np.int32)
    y = np.clip(x - low, 0, 255)
    d = float(high - low)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        m = F32(np.float64(255.0) / np.float64(d)) if d != 0 else F32(np.inf)
        z = y.astype(F32) * m
    return _sat_u8_from_rint(z)


def img_channel_stretch(plane: np.ndarray, lo: int = 0, hi: int = 100) -> np.ndarray:
    """imgChannelStretch (preprocessing.cpp:74-105) on one 8U plane; returns the new plane."""
    h, w = plane.shape
    low, high = percentile_bins(get_histogram(plane), w, h, lo, hi)
    return stretch_lut(low, high)[plane]


# ----------------------------------------------------------------------------------------
# colour conversions (OpenCV 8-bit paths, SURVEY appendix A.3-A.5)
# ----------------------------------------------------------------------------------------

_HSV_SHIFT = 12
_i = np.arange(1, 256, dtype=np.float64)
SDIV = np.zeros(256, np.int32)
HDIV = np.zeros(256, np.int32)
SDIV[1:] = np.rint((255 << _HSV_SHIFT) / _i).astype(np.int32)
HDIV[1:] = np.rint((180 << _HSV_SHIFT) / (6.0 * _i)).astype(np.int32)


def bgr2hsv(bgr: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_BGR2HSV) on 8UC3, H in [0,180): pure integer, shift 12 (A.4)."""
    b = bgr[..., 0].astype(np.int32)
    g = bgr[..., 1].astype(np.int32)
    r = bgr[..., 2].astype(np.int32)
    v = np.maximum(np.maximum(b, g), r)
    vmin = np.minimum(np.minimum(b, g), r)
    d = v - vmin
    s = (d * SDIV[v] + (1 << 11)) >> 12
    h0 = np.where(v == r, g - b, np.where(v == g, b - r + 2 * d, r - g + 4 * d))
    h = (h0 * HDIV[d] + (1 << 11)) >> 12
    h = np.where(h < 0, h + 180, h)
    return np.stack([h, s, v], axis=-1).astype(np.uint8)


_SECTOR = np.array(
    [[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]], dtype=np.int64
)


def hsv2bgr(hsv: np.ndarray, rounding: str = "cv2") -> np.ndarray:
    """cvtColor(COLOR_HSV2BGR) on 8UC3 (A.3).  rounding: 'trunc', 'rint', or 'cv2' = what the
    cv2 4.13.0 build in this image does: truncation for pixels x < 32*floor(W/32) of each row
    (AVX2 body) and rint for the scalar tail."""
    hsv = np.asarray(hsv)
    shape = hsv.shape
    H = hsv[..., 0].astype(F32)
    S = hsv[..., 1].astype(F32)
    V = hsv[..., 2].astype(F32)
    h = H * F32(6.0 / 180.0)
    s = S * F32(1.0 / 255.0)
    v = V * F32(1.0 / 255.0)
    sec = np.floor(h)
    f = (h - sec).astype(F32)
    sec = sec.astype(np.int64)
    oob = (sec < 0) | (sec > 5)
    sec = np.where(oob, 0, sec)
    f = np.where(oob, F32(0), f).astype(F32)
    one = F32(1.0)
    LD = np.longdouble  # 64-bit mantissa: s*f (48 bits) and 1 - s*f (<= 60 bits) are exact

    def fma_neg(sv, fv):  # fma(-s, f, 1) with a single rounding to f32
        return (LD(1.0) - sv.astype(LD) * fv.astype(LD)).astype(F32)

    tab = np.empty(shape[:-1] + (4,), F32)
    tab[..., 0] = v
    tab[..., 1] = v * (one - s)
    tab[..., 2] = v * fma_neg(s, f)
    tab[..., 3] = v * fma_neg(s, (one - f).astype(F32))
    idx = _SECTOR[sec]  # (..., 3) -> tab index for b, g, r
    out = np.take_along_axis(tab, idx, axis=-1) * F32(255.0)
    tr = np.clip(np.trunc(out), 0, 255).astype(np.uint8)
    if rounding == "trunc":
        return tr
    rn = np.clip(np.rint(out), 0, 255).astype(np.uint8)
    if rounding == "rint":
        return rn
    assert rounding == "cv2" and hsv.ndim == 3
    W = shape[1]
    body = 32 * (W // 32)
    res = tr.copy()
    res[:, body:] = rn[:, body:]
    return res


def bgr2ycrcb(bgr: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_BGR2YCrCb) on 8UC3: integer, shift 14; channel order Y, Cr, Cb (A.5)."""
    b = bgr[..., 0].astype(np.int32)
    g = bgr[..., 1].astype(np.int32)
    r = bgr[..., 2].astype(np.int32)
    Y = (4899 * r + 9617 * g + 1868 * b + 8192) >> 14
    Cr = np.clip(((r - Y) * 11682 + 128 * 16384 + 8192) >> 14, 0, 255)
    Cb = np.clip(((b - Y) * 9241 + 128 * 16384 + 8192) >> 14, 0, 255)
    return np.stack([Y, Cr, Cb], axis=-1).astype(np.uint8)


def ycrcb2bgr(ycc: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_YCrCb2BGR) on 8UC3: integer, shift 14, saturating (checked against cv2 4.13.0 on all
    2^24 triples by oracle/make_golden.py)."""
    Y = ycc[..., 0].astype(np.int32)
    Cr = ycc[..., 1].astype(np.int32) - 128
    Cb = ycc[..., 2].astype(np.int32) - 128
    b = np.clip(Y + ((Cb * 29049 + 8192) >> 14), 0, 255)
    g = np.clip(Y + ((Cb * -5636 + Cr * -11698 + 8192) >> 14), 0, 255)
    r = np.clip(Y + ((Cr * 22987 + 8192) >> 14), 0, 255)
    return np.stack([b, g, r], axis=-1).astype(np.uint8)


def _fma32(a, b, c):
    """float32 fused multiply-add: the product of two float32 is exact in float64, one rounding at the end."""
    return (a.astype(np.float64) * b.astype(np.float64) + np.asarray(c, dtype=np.float64)).astype(np.float32)


def bgr2hls(bgr: np.ndarray, simd: str = "cv2") -> np.ndarray:
    """cvtColor(COLOR_BGR2HLS) on 8UC3 (H in [0,180), order H, L, S): float32 arithmetic on k/255.
    cv2 4.13.0 here runs the first 8*floor(W/8) pixels of every row through a vector body and the rest through
    the scalar tail; the two differ in two places (found by fitting against all 2^24 triples, make_golden.py):
      body: S denominator 2 - (vmax + vmin); `h += 360` fused with the product (one rounding)
      tail: S denominator (2 - vmax) - vmin;  `h += 360` on the rounded value
    In both, `(x - y)*d + 120|240` is one fused multiply-add.  simd='cv2': body/tail split; 'scalar': tail model
    everywhere (what the C++ source says without vectorisation)."""
    f32 = np.float32
    b = bgr[..., 0].astype(f32) * f32(1 / 255.0)
    g = bgr[..., 1].astype(f32) * f32(1 / 255.0)
    r = bgr[..., 2].astype(f32) * f32(1 / 255.0)
    vmax = np.maximum(np.maximum(b, g), r)
    vmin = np.minimum(np.minimum(b, g), r)
    diff = vmax - vmin
    vs = vmax + vmin
    lum = vs * f32(0.5)
    W = bgr.shape[-2]
    body = np.zeros(bgr.shape[:-1], bool)
    if simd == "cv2":
        body[..., : 8 * (W // 8)] = True
    with np.errstate(all="ignore"):
        den = np.where(body, f32(2) - vs, (f32(2) - vmax) - vmin)
        sat = np.where(lum < f32(0.5), diff / vs, diff / den)
        dinv = f32(60.0) / diff

        def hsel(d1, d2, add):
            hh = (d1 - d2) * dinv if add == 0 else _fma32(d1 - d2, dinv, add)
            wrapped = np.where(body, _fma32(d1 - d2, dinv, add + 360.0), hh + f32(360.0))
            return np.where(hh < 0, wrapped, hh)

        hue = np.where(vmax == r, hsel(g, b, 0), np.where(vmax == g, hsel(b, r, 120.0), hsel(r, g, 240.0)))
    gray = diff <= np.finfo(np.float32).eps
    hue = np.where(gray, f32(0), hue)
    sat = np.where(gray, f32(0), sat)
    H = np.clip(np.rint(hue * f32(0.5)), 0, 255)
    L = np.clip(np.rint(lum * f32(255.0)), 0, 255)
    S = np.clip(np.rint(sat * f32(255.0)), 0, 255)
    return np.stack([H, L, S], axis=-1).astype(np.uint8)


_HLS_SECTOR = np.array([[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]])


def hls2bgr(hls: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_HLS2BGR) on 8UC3: float32, rint at the end; equal to cv2 4.13.0 on all 180*2^16 triples
    (and for H >= 180, which a stretched H plane can hold: the sector index wraps modulo 6)."""
    f32 = np.float32
    h = hls[..., 0].astype(f32)
    lum = hls[..., 1].astype(f32) * f32(1 / 255.0)
    s = hls[..., 2].astype(f32) * f32(1 / 255.0)
    p2 = np.where(lum <= f32(0.5), lum * (f32(1) + s), lum + s - lum * s)
    p1 = f32(2) * lum - p2
    hh = h * f32(6 / 180.0)
    sec = np.floor(hh)
    fr = hh - sec
    sec = sec.astype(np.int32) % 6
    d = p2 - p1
    tab = np.stack([p2, p1, p1 + d * (f32(1) - fr), p1 + d * fr], 0).reshape(4, -1)
    idx = np.arange(h.size)
    secf = sec.reshape(-1)
    out = np.stack([tab[_HLS_SECTOR[secf, k], idx].reshape(h.shape) for k in range(3)], axis=-1)
    out = np.where((hls[..., 2] == 0)[..., None], lum[..., None], out)
    return np.clip(np.rint(out * f32(255.0)), 0, 255).astype(np.uint8)



# ---- 8-bit CIE Lab (cvtColor BGR2Lab / Lab2BGR, D65, sRGB gamma): OpenCV 4's bit-exact integer path ----
# Restated from the published algorithm (imgproc color_lab.cpp: RGB2Lab_b / Lab2RGBinteger) and pinned against cv2
# 4.13.0 on all 2^24 triples in both directions (tests/golden/kat.json: lab).  Position independent (no body/tail split).
_LAB_SHIFT, _GAMMA_SHIFT, _LAB_SHIFT2, _LAB_BASE, _INV_GAMMA_SIZE, _LAB_MIN_AB = 12, 3, 15, 1 << 14, 1 << 12, -8145
_LAB_WHITE = (0.950456, 1.0, 1.088754)
_SRGB2XYZ = (0.412453, 0.357580, 0.180423, 0.212671, 0.715160, 0.072169, 0.019334, 0.119193, 0.950227)
_XYZ2SRGB = (3.240479, -1.53715, -0.498535, -0.969256, 1.875991, 0.041556, 0.055648, -0.204043, 1.057311)


def lab_tables():
    """The lookup tables of the 8-bit Lab conversions: (gamma[256], cbrt[3072], fwd coeffs[9], LabToYF[512], invgamma[4096],
    inv coeffs[9]).  Table values are rint() of float32 products like the source computes them.  The cube-root table is
    rint(2^15 cbrt(x)) with cbrt in double from the float32 abscissa, except entry 49 (true value 9454.5004, the source's
    soft-float cbrt lands below the tie: 9454) - fixed by the exhaustive comparison; 8-bit inputs reach entries 0..2040 only."""
    f32 = np.float32
    i = np.arange(256)
    x = i.astype(f32) / f32(255)
    xd = x.astype(np.float64)
    g = np.where(xd <= 0.04045, xd / 12.92, ((xd + 0.055) / 1.055) ** 2.4).astype(f32)
    gamma = np.rint(f32(255 * (1 << _GAMMA_SHIFT)) * g).astype(np.int64)
    n = 256 * 3 // 2 * (1 << _GAMMA_SHIFT)
    xi = (f32(1) / (f32(255) * f32(1 << _GAMMA_SHIFT))) * np.arange(n).astype(f32)
    xd = xi.astype(np.float64)
    lin = (xd * np.float64(f32(841 / 108.0)) + np.float64(f32(16 / 116.0))).astype(f32).astype(np.float64)
    cb = np.where(xi < f32(216 / 24389.0), lin, np.cbrt(xd))
    cbrt = np.rint((1 << _LAB_SHIFT2) * cb).astype(np.int64)
    cbrt[49] = 9454
    fwd = np.array([int(np.rint((1 << _LAB_SHIFT) * _SRGB2XYZ[k * 3 + j] / _LAB_WHITE[k])) for k in range(3) for j in range(3)], np.int64)
    ytab = np.zeros(512, np.int64)
    B = _LAB_BASE
    for L in range(256):
        if L <= 20:
            y = np.rint(f32(L * B * 20 * 9) / f32(17 * 29 * 29 * 29))
            ify = np.rint(f32(B) * (f32(16) / f32(116) + f32(L * 5) / f32(3 * 17 * 29)))
        else:
            fy = f32(L * 100 * B) / f32(255 * 116) + f32(16 * B) / f32(116)
            ify = np.rint(fy)
            y = np.rint(fy * fy * fy / f32(B * B))
        ytab[2 * L], ytab[2 * L + 1] = int(y), int(ify)
    xg = (f32(1) / f32(_INV_GAMMA_SIZE)) * np.arange(_INV_GAMMA_SIZE).astype(f32)
    xd = xg.astype(np.float64)
    ig = np.where(xd <= 0.0031308, xd * 12.92, np.power(xd, 1 / 2.4) * 1.055 - 0.055).astype(f32)
    invgamma = np.rint(f32(255) * ig).astype(np.int64)
    inv = np.array([int(np.rint((1 << _LAB_SHIFT) * _XYZ2SRGB[r * 3 + k] * _LAB_WHITE[k])) for r in range(3) for k in range(3)], np.int64)
    return gamma, cbrt, fwd, ytab, invgamma, inv


_LAB_T = None


def _lab_t():
    global _LAB_T
    if _LAB_T is None:
        _LAB_T = lab_tables()
    return _LAB_T


def _descale(v, s):
    return (v + (1 << (s - 1))) >> s


def lab_ab_to_xz(i):
    """abToXZ_b as a function (the source tabulates it over [-8145, 28719)): C integer division truncates toward zero."""
    i = np.asarray(i, np.int64)
    t = i * 108
    lo = np.where(t >= 0, t // 841, -((-t) // 841)) - (_LAB_BASE * 16 // 116 * 108 // 841)
    hi = (i * i // _LAB_BASE) * i // _LAB_BASE
    return np.where(i <= 3390, lo, hi)


def bgr2lab(bgr: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_BGR2Lab) on 8UC3 (planes L*255/100, a+128, b+128)."""
    gamma, cbrt, C, _, _, _ = _lab_t()
    B, G, R = gamma[bgr[..., 0]], gamma[bgr[..., 1]], gamma[bgr[..., 2]]
    fX = cbrt[_descale(R * C[0] + G * C[1] + B * C[2], _LAB_SHIFT)]
    fY = cbrt[_descale(R * C[3] + G * C[4] + B * C[5], _LAB_SHIFT)]
    fZ = cbrt[_descale(R * C[6] + G * C[7] + B * C[8], _LAB_SHIFT)]
    Lscale = (116 * 255 + 50) // 100
    Lshift = -((16 * 255 * (1 << _LAB_SHIFT2) + 50) // 100)
    L = _descale(Lscale * fY + Lshift, _LAB_SHIFT2)
    a = _descale(500 * (fX - fY) + 128 * (1 << _LAB_SHIFT2), _LAB_SHIFT2)
    b = _descale(200 * (fY - fZ) + 128 * (1 << _LAB_SHIFT2), _LAB_SHIFT2)
    return np.clip(np.stack([L, a, b], axis=-1), 0, 255).astype(np.uint8)


def lab2bgr(lab: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_Lab2BGR) on 8UC3."""
    _, _, _, ytab, invgamma, C = _lab_t()
    LL, aa, bb = (lab[..., k].astype(np.int64) for k in range(3))
    y, ify = ytab[2 * LL], ytab[2 * LL + 1]
    adiv = ((5 * aa * 53687 + (1 << 7)) >> 13) - 128 * _LAB_BASE // 500
    bdiv = ((bb * 41943 + (1 << 4)) >> 9) - 128 * _LAB_BASE // 200 + 1
    x, z = lab_ab_to_xz(ify + adiv), lab_ab_to_xz(ify - bdiv)
    shift = _LAB_SHIFT + (14 - 12)
    ch = [invgamma[np.clip(_descale(C[3 * r] * x + C[3 * r + 1] * y + C[3 * r + 2] * z, shift), 0, _INV_GAMMA_SIZE - 1)] for r in range(3)]
    return np.stack([ch[2], ch[1], ch[0]], axis=-1).astype(np.uint8)


# ----------------------------------------------------------------------------------------
# histretch CLI channel loop (histretch.cpp:219-254)
# ----------------------------------------------------------------------------------------


def histretch_frame(
    bgr: np.ndarray,
    channels: str = "V",
    lo: int = 2,
    hi: int = 98,
    order: str = "intended",
    hsv_rounding: str = "cv2",
) -> np.ndarray:
    """Channel loop of the histretch CLI.  Supports every letter of the CLI (BGR, HSV, HLS, Lab, YCrCb).  Note the letter -> plane map of numChannel: in HLS (plane order H, L, S) the letter 's' is
    plane 1 = L and 'l' is plane 2 = S, exactly as the reference indexes them.
    order='intended': convert -> stretch -> merge -> convert back (modules/histretch/README.md:4)
    order='literal' : histretch.cpp:232-240 as written - the back-conversion runs on the
                      UNstretched converted image, so the frame becomes its HSV round trip."""
    src = np.array(bgr, copy=True)
    for c in channels:
        ch, sp = num_channel(c), num_space(c)
        if sp == -1:
            continue  # "Option not recognized, skipping..." (histretch.cpp:252)
        if sp == 0:
            src[..., ch] = img_channel_stretch(src[..., ch], lo, hi)
        elif sp == 1:
            dst = bgr2hsv(src)
            if order == "literal":
                src = hsv2bgr(dst, hsv_rounding)
            else:
                dst[..., ch] = img_channel_stretch(dst[..., ch], lo, hi)
                src = hsv2bgr(dst, hsv_rounding)
        elif sp == 2:  # h, s, l: transformation[1] = BGR2HLS / HLS2BGR
            dst = bgr2hls(src, "scalar" if hsv_rounding in ("trunc", "rint") else "cv2")
            if order != "literal":
                dst[..., ch] = img_channel_stretch(dst[..., ch], lo, hi)
            src = hls2bgr(dst)
        elif sp == 3:  # L, a, b: transformation[2] = BGR2Lab / Lab2BGR
            dst = bgr2lab(src)
            if order != "literal":
                dst[..., ch] = img_channel_stretch(dst[..., ch], lo, hi)
            src = lab2bgr(dst)
        elif sp == 4:  # Y, C, X: transformation[3] = BGR2YCrCb / YCrCb2BGR (histretch.cpp:155-156)
            dst = bgr2ycrcb(src)
            if order != "literal":
                dst[..., ch] = img_channel_stretch(dst[..., ch], lo, hi)
            src = ycrcb2bgr(dst)
    return src


# ----------------------------------------------------------------------------------------
# videostrip calcBlur (videostrip.cpp:170-184) - SURVEY 8f row N4
# ----------------------------------------------------------------------------------------


def bgr2gray(bgr: np.ndarray) -> np.ndarray:
    """cvtColor(COLOR_BGR2GRAY) on 8UC3 as cv2 4.13.0 computes it: Q15 (9798 R + 19235 G + 3735 B + 2^14) >> 15
    (equal on all 2^24 triples; OpenCV 3.4.6 documents the Q14 triple 4899/9617/1868, which differs by one level on
    0.26 % of the triples)."""
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    return ((9798 * r + 19235 * g + 3735 * b + 16384) >> 15).astype(np.uint8)


def _reflect101(n: int) -> np.ndarray:
    idx = np.arange(-1, n + 1)
    if n == 1:
        return np.zeros_like(idx)
    return np.where(idx < 0, -idx, np.where(idx >= n, 2 * n - 2 - idx, idx))


def laplacian3_u8(grey: np.ndarray, aperture: int = 3) -> np.ndarray:
    """Laplacian(grey, dst, CV_8U, ksize=3) - what `Laplacian(grey, laplacian, grey.type(), CV_16S)` at
    videostrip.cpp:175 asks for (third argument = depth CV_8U, fourth = aperture, CV_16S == 3):
    kernel [2 0 2; 0 -8 0; 2 0 2], BORDER_REFLECT_101, saturated to 8 bits.  aperture=1: [0 1 0; 1 -4 1; 0 1 0],
    the kernel calcBlurGPU requests from cv::cuda::createLaplacianFilter (videostrip.cpp:48)."""
    h, w = grey.shape
    P = grey.astype(np.int64)[np.ix_(_reflect101(h), _reflect101(w))]
    if aperture == 3:
        L = 2 * (P[:-2, :-2] + P[:-2, 2:] + P[2:, :-2] + P[2:, 2:]) - 8 * P[1:-1, 1:-1]
    else:
        L = P[:-2, 1:-1] + P[2:, 1:-1] + P[1:-1, :-2] + P[1:-1, 2:] - 4 * P[1:-1, 1:-1]
    return np.clip(L, 0, 255).astype(np.uint8)


def mean_stddev_u8(plane: np.ndarray):
    """cv::meanStdDev on 8U: integer sums, then scale = 1/N, mean = s*scale, var = max(sq*scale - mean^2, 0)."""
    p = plane.astype(np.int64)
    scale = 1.0 / p.size
    mean = float(int(p.sum())) * scale
    var = max(float(int((p * p).sum())) * scale - mean * mean, 0.0)
    return mean, float(np.sqrt(var))


def golden_frame(key: str) -> np.ndarray:
    """Input frame of a golden-vector case named `<synth|rand>_<seed hex>_<frame>_<W>x<H>` (tests/golden/kat.json)."""
    kind, seed, f, size = key.split("_")
    W, H = map(int, size.split("x"))
    if kind == "synth":
        return synth_frame(int(seed, 16), int(f), W, H)
    return np.random.default_rng(int(seed, 16)).integers(0, 256, (H, W, 3), dtype=np.uint8)


def golden_pixels(a: np.ndarray, px: np.ndarray) -> np.ndarray:
    """Values of an (H, W) or (H, W, C) map at the flat pixel indices `px`: the float maps of tests/golden/dehaze_literal.npz
    are stored at such a sample of pixels (its `px` key), compared maps are taken there."""
    a = np.asarray(a)
    return a.reshape((-1,) + a.shape[2:])[px]


def calc_blur(bgr: np.ndarray, aperture: int = 3) -> np.float32:
    """float calcBlur(Mat frame), videostrip.cpp:170-184: the standard deviation of the Laplacian, returned as float."""
    return np.float32(mean_stddev_u8(laplacian3_u8(bgr2gray(bgr), aperture))[1])


# ----------------------------------------------------------------------------------------
# CLAHE (cv::CLAHE::apply, 8-bit; SURVEY appendix A.2)
# ----------------------------------------------------------------------------------------


def clahe_luts(plane: np.ndarray, clip: float, tiles_x: int, tiles_y: int) -> np.ndarray:
    """Per-tile LUTs [tiles_y, tiles_x, 256] uint8."""
    H, W = plane.shape
    src = plane
    if W % tiles_x or H % tiles_y:
        src = np.pad(
            plane,
            ((0, tiles_y - H % tiles_y), (0, tiles_x - W % tiles_x)),
            mode="reflect",
        )
    EH, EW = src.shape
    tw, th = EW // tiles_x, EH // tiles_y
    area = tw * th
    cl = max(int(clip * area / 256.0), 1) if clip > 0 else 0
    lut_scale = F32(255.0) / F32(area)
    t = src.reshape(tiles_y, th, tiles_x, tw).transpose(0, 2, 1, 3).reshape(tiles_y * tiles_x, area)
    nt = t.shape[0]
    offs = (np.arange(nt, dtype=np.int64) * 256)[:, None]
    hist = np.bincount((t.astype(np.int64) + offs).ravel(), minlength=nt * 256).reshape(nt, 256)
    hist = hist.astype(np.int64)
    if cl > 0:
        clipped = np.maximum(hist - cl, 0).sum(axis=1)
        hist = np.minimum(hist, cl)
        batch = clipped // 256
        resid = clipped - batch * 256
        hist = hist + batch[:, None]
        step = np.maximum(256 // np.maximum(resid, 1), 1)
        k = np.arange(256, dtype=np.int64)[None, :]
        inc = (resid[:, None] > 0) & (k % step[:, None] == 0) & (k // step[:, None] < resid[:, None])
        hist = hist + inc
    cum = np.cumsum(hist, axis=1)
    lut = _sat_u8_from_rint(cum.astype(F32) * lut_scale)
    return lut.reshape(tiles_y, tiles_x, 256)


def clahe_apply(plane: np.ndarray, clip: float = 40.0, tiles_x: int = 8, tiles_y: int = 8) -> np.ndarray:
    """cv2.createCLAHE(clip, (tiles_x, tiles_y)).apply(plane) for an 8U plane."""
    H, W = plane.shape
    lut = clahe_luts(plane, clip, tiles_x, tiles_y).astype(F32)
    if W % tiles_x == 0 and H % tiles_y == 0:
        EW, EH = W, H
    else:  # OpenCV pads BOTH dimensions (a full extra tile count when one divides evenly)
        EW, EH = W + tiles_x - W % tiles_x, H + tiles_y - H % tiles_y
    tw, th = EW // tiles_x, EH // tiles_y
    inv_tw = F32(1.0) / F32(tw)
    inv_th = F32(1.0) / F32(th)

    def coords(n, inv, ntile):
        f = np.arange(n).astype(F32) * inv - F32(0.5)
        t1 = np.floor(f).astype(np.int64)
        a = (f - t1.astype(F32)).astype(F32)
        a1 = (F32(1.0) - a).astype(F32)
        t2 = np.minimum(t1 + 1, ntile - 1)
        t1 = np.maximum(t1, 0)
        return t1, t2, a, a1

    tx1, tx2, xa, xa1 = coords(W, inv_tw, tiles_x)
    ty1, ty2, ya, ya1 = coords(H, inv_th, tiles_y)
    v = plane.astype(np.int64)
    Y1, Y2 = ty1[:, None], ty2[:, None]
    X1, X2 = tx1[None, :], tx2[None, :]
    l11 = lut[Y1, X1, v]
    l12 = lut[Y1, X2, v]
    l21 = lut[Y2, X1, v]
    l22 = lut[Y2, X2, v]
    xa_, xa1_ = xa[None, :], xa1[None, :]
    ya_, ya1_ = ya[:, None], ya1[:, None]
    top = (l11 * xa1_ + l12 * xa_).astype(F32)
    bot = (l21 * xa1_ + l22 * xa_).astype(F32)
    res = ((top * ya1_).astype(F32) + (bot * ya_).astype(F32)).astype(F32)
    return _sat_u8_from_rint(res)


def aclahe_frame(bgr, clip=2.0, tiles_x=8, tiles_y=8, hsv_rounding="cv2"):
    """aclahe.cpp:152-154 wrapper + the intended (stubbed, :214-218) tail: BGR->HSV, CLAHE on V,
    merge, HSV->BGR."""
    hsv = bgr2hsv(bgr)
    hsv[..., 2] = clahe_apply(hsv[..., 2], clip, tiles_x, tiles_y)
    return hsv2bgr(hsv, hsv_rounding)


def entropy_cpp(plane: np.ndarray) -> np.float32:
    """aclaheEntropy (aclahe.cpp:228-248): float p, double log2(p + 1e-5), product and running
    sum evaluated in double then stored to the float accumulator each iteration."""
    h, w = plane.shape
    hist = get_histogram(plane)
    ent = F32(0)
    n = F32(w * h)
    for i in range(256):
        p = F32(hist[i] / n)
        ent = F32(np.float64(ent) + np.float64(p) * math.log2(np.float64(p) + 0.00001))
    return F32(-ent)


def entropy_py(plane: np.ndarray) -> np.float32:
    """Entropia (functions.py:14-19): float32 throughout."""
    hist = get_histogram(plane)
    p = (hist / hist.sum(dtype=F32)).astype(F32)
    lg = np.log2(p + F32(0.00001)).astype(F32)
    return F32(-1) * (p * lg).sum(dtype=F32)


def gaussian_blur3(plane: np.ndarray) -> np.ndarray:
    """cv2.GaussianBlur(plane, (3,3), 0) on 8U (ACLAHE.py:15): (sum [1 2 1]^T[1 2 1] p + 8) >> 4,
    reflect-101 border."""
    p = np.pad(plane.astype(np.int32), 1, mode="reflect")
    hsum = p[:, :-2] + 2 * p[:, 1:-1] + p[:, 2:]
    vsum = hsum[:-2] + 2 * hsum[1:-1] + hsum[2:]
    return ((vsum + 8) >> 4).astype(np.uint8)


# ----------------------------------------------------------------------------------------
# bgdehaze (BGDehaze.py, guidedfilter.py) - float64, vectorised
# ----------------------------------------------------------------------------------------


def _aclahe_knee(x: np.ndarray, y: np.ndarray) -> int:
    """DerivadaY / DerivadaX / Curvatura of modules/aclahe/python/functions.py:49-93: double-exponential fit of the 49
    samples, cubic spline through 25 points of the fit, curvature |x'y'' - y'x''| / (x'^2 + y'^2)^1.5 at 49 points,
    index of its maximum (used directly as the clip limit, ACLAHE.py:92-96)."""
    from scipy.interpolate import splev, splrep
    from scipy.optimize import curve_fit

    def f(t, p0, p1, p2, p3):
        return p0 * np.exp(-p1 * t) + p2 * np.exp(-p3 * t)

    u = np.linspace(1, 49, 49)
    x22 = np.linspace(1, 25, 25)
    x222 = np.linspace(1, 25, 49)
    d = []
    for v in (y, x):
        popt, _ = curve_fit(f, u, v, (7, 0.4, 0.9, 5))
        tck = splrep(x22, f(x22, *popt))
        d.append((splev(x222, tck, der=1), splev(x222, tck, der=2)))
    (y1, y2), (x1, x2) = d
    k = np.sqrt((x1 * y2 - y1 * x2) ** 2) / np.sqrt((x1 ** 2 + y1 ** 2) ** 3)
    return int(np.argmax(k))


def parametros_aclahe(img: np.ndarray, loop: str = "repaired"):
    """ParametrosACLAHE of modules/aclahe/python/ACLAHE.py:9-129 -> (BS, CL, entropies[5][50]).
    loop='as_committed': the sweep body as it stands in the file (lines 42-45 outside `for i in cl`): the curves handed to
    the knee search are all zero, the clip limit degenerates to 0.  loop='repaired': every clip limit evaluated."""
    import warnings

    blur = gaussian_blur3(img)                                     # ACLAHE.py:15
    bl = (2, 4, 8, 16, 32)
    cl = np.arange(0, 25, 0.5)
    ent = np.zeros((5, 50), np.float32)
    if loop == "repaired":
        knees = []
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for j, k in enumerate(bl):
                ent[j] = [entropy_py(clahe_apply(blur, float(c), k, k)) for c in cl]
                row_x = np.zeros(51, np.float32)
                row_y = np.zeros(51, np.float32)
                row_x[1:51] = cl
                row_y[1:51] = ent[j]
                knees.append(_aclahe_knee(row_x[2:51], row_y[2:51]))   # graficar drops the first two columns
        d = max(knees)
    elif loop == "as_committed":
        d = 0
    else:
        raise ValueError(loop)
    res = np.zeros((2, 5), np.float16)                             # ACLAHE.py:102: float16 table
    for m, k in enumerate(bl):
        res[0, m] = k
        res[1, m] = entropy_py(clahe_apply(blur, float(d), k, k))
    w = int(np.flatnonzero(res[1] == res[1].max())[-1])            # last arg-max wins (ACLAHE.py:117-121)
    return int(round(float(res[0, w]))), d, ent


def _window_reduce(a: np.ndarray, w: int, op, pad_value) -> np.ndarray:
    """w x w window reduction centred like `padded[y:y+w, x:x+w]` with padwidth floor(w/2)."""
    pw = w // 2
    H, W = a.shape
    p = np.full((H + 2 * pw, W + 2 * pw), pad_value, dtype=a.dtype)
    p[pw : pw + H, pw : pw + W] = a
    acc = p[:, 0:W].copy()
    for k in range(1, w):
        acc = op(acc, p[:, k : k + W])
    out = acc[0:H].copy()
    for k in range(1, w):
        out = op(out, acc[k : k + H])
    return out


def normalize_frame(I8: np.ndarray) -> np.ndarray:
    """bgdehaze/main.py:17: (I - I.min()) / (I.max() - I.min()), uint8 subtract, float64 divide."""
    mn, mx = I8.min(), I8.max()
    with np.errstate(divide="ignore", invalid="ignore"):
        return (I8 - mn) / np.uint8(mx - mn)


def background_light(normI: np.ndarray, w: int = 15, return_idx: bool = False):
    """BGDehaze.py:14-26.  Tie rule: FIRST flat index of the minimum (np.argmin); the reference's
    `argsort(axis=0)[:1]` is an unstable sort whose choice among ties is machine dependent."""
    M, N, _ = normI.shape
    mx = [_window_reduce(normI[..., c], w, np.maximum, 0.0) for c in range(3)]
    D0 = (mx[2] - mx[0]).ravel()
    D1 = (mx[2] - mx[1]).ravel()
    i0, i1 = int(np.argmin(D0)), int(np.argmin(D1))
    flatI = normI.reshape(M * N, 3)
    B = np.average(flatI.take([i0, i1], axis=0), axis=0)
    return (B, (i0, i1)) if return_idx else B


def transmission_map(normI: np.ndarray, w: int = 15, B=None) -> np.ndarray:
    """BGDehaze.py:28-37: 1 - min_{w x w}(I_c / B_c), zero padded, c = blue, green."""
    if B is None:
        B = background_light(normI, w)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = normI / B
    t = np.empty(normI.shape[:2] + (2,), np.float64)
    for c in range(2):
        t[..., c] = 1 - _window_reduce(q[..., c], w, np.minimum, 0.0)
    return t


def boxfilter(I: np.ndarray, r: int) -> np.ndarray:
    """guidedfilter.py:23-51: (2r+1)^2 window sum, windows truncated at the borders."""
    M, N = I.shape
    c = np.zeros((M + 1, N), np.float64)
    np.cumsum(I, axis=0, out=c[1:])
    lo = np.clip(np.arange(M) - r, 0, M)
    hi = np.clip(np.arange(M) + r + 1, 0, M)
    v = c[hi] - c[lo]
    c2 = np.zeros((M, N + 1), np.float64)
    np.cumsum(v, axis=1, out=c2[:, 1:])
    lo = np.clip(np.arange(N) - r, 0, N)
    hi = np.clip(np.arange(N) + r + 1, 0, N)
    return c2[:, hi] - c2[:, lo]


def guided_filter(I: np.ndarray, p: np.ndarray, r: int = 40, eps: float = 1e-3) -> np.ndarray:
    """guidedfilter.py:54-103: colour-guide guided filter (He et al. ECCV-10 eqs 14-16)."""
    M, N = p.shape
    base = boxfilter(np.ones((M, N)), r)
    means = [boxfilter(I[..., i], r) / base for i in range(3)]
    mean_p = boxfilter(p, r) / base
    means_IP = [boxfilter(I[..., i] * p, r) / base for i in range(3)]
    cov = [means_IP[i] - means[i] * mean_p for i in range(3)]
    var = {}
    for i in range(3):
        for j in range(i, 3):
            var[i, j] = boxfilter(I[..., i] * I[..., j], r) / base - means[i] * means[j]
    Sigma = np.empty((M, N, 3, 3), np.float64)
    for i in range(3):
        for j in range(3):
            Sigma[..., i, j] = var[min(i, j), max(i, j)]
    Sigma += eps * np.eye(3)
    covv = np.stack(cov, axis=-1)
    bad = ~np.isfinite(Sigma).all(axis=(-1, -2))
    if bad.any():
        Sigma[bad] = np.eye(3)
    inv = np.linalg.inv(Sigma)
    a = np.einsum("...j,...jk->...k", covv, inv)
    if bad.any():
        a[bad] = np.nan
    b = mean_p - a[..., 0] * means[0] - a[..., 1] * means[1] - a[..., 2] * means[2]
    q = (
        boxfilter(a[..., 0], r) * I[..., 0]
        + boxfilter(a[..., 1], r) * I[..., 1]
        + boxfilter(a[..., 2], r) * I[..., 2]
        + boxfilter(b, r)
    ) / base
    return q


def refined_t(normI, w=15, tmin=0.2, r=40, eps=1e-3, B=None):
    """BGDehaze.py:39-48.  (The reference's dehazed_BG calls this WITHOUT w, so w is always 15.)"""
    t = transmission_map(normI, w, B)
    tb = np.maximum(t[..., 0], tmin)
    tg = np.maximum(t[..., 1], tmin)
    return guided_filter(normI, tb, r, eps), guided_filter(normI, tg, r, eps)


def _minmax_norm(x):
    with np.errstate(divide="ignore", invalid="ignore"):
        return (x - x.min()) / (x.max() - x.min())


def dehazed_bg(normI, w=15, stages=None, r=40, eps=1e-3, tmin=0.2):
    """BGDehaze.py:50-57; r, eps and tmin are the reference's fixed values (BGDehaze.py:41) unless given."""
    B = background_light(normI, w)
    B15 = B if w == 15 else background_light(normI, 15)
    rb, rg = refined_t(normI, 15, tmin, r, eps, B=B15)
    with np.errstate(divide="ignore", invalid="ignore"):
        Jb = (normI[..., 0] - B[0]) / rb + B[0]
        Jg = (normI[..., 1] - B[1]) / rg + B[1]
    if stages is not None:
        stages.update(B=B, t_blue=rb, t_green=rg, J_blue=Jb, J_green=Jg)
    return _minmax_norm(Jb), _minmax_norm(Jg)


def rc_correction(normI, w=15, stages=None, r=40, eps=1e-3, tmin=0.2):
    """BGDehaze.py:59-69."""
    nb, ng = dehazed_bg(normI, w, stages, r, eps, tmin)
    avgRr = 1.5 - np.average(nb.ravel()) - np.average(ng.ravel())
    with np.errstate(divide="ignore", invalid="ignore"):
        coef = avgRr / np.average(normI[..., 2].ravel())
    Rrec = normI[..., 2] * coef
    restored = np.zeros(normI.shape)
    restored[..., 0] = nb
    restored[..., 1] = ng
    restored[..., 2] = _minmax_norm(Rrec)
    if stages is not None:
        stages.update(restored=restored)
    return restored


def adaptive_exp_map(normI, w=15, stages=None, r=40, eps=1e-3, tmin=0.2):
    """BGDehaze.py:71-89; r and eps (fixed at 40 and 1e-3 at BGDehaze.py:72) serve all three guided filters."""
    restored = rc_correction(normI, w, stages, r, eps, tmin)
    with np.errstate(invalid="ignore"):
        R = (restored * 255).astype(np.uint8)
        I = (normI * 255).astype(np.uint8)
    Yj = bgr2ycrcb(R)
    Yi = bgr2ycrcb(I)
    with np.errstate(divide="ignore", invalid="ignore"):
        nYj = (Yj - Yj.min()) / np.uint8(Yj.max() - Yj.min())
        nYi = (Yi - Yi.min()) / np.uint8(Yi.max() - Yi.min())
        yi, yj = nYi[..., 0], nYj[..., 0]
        S = (yj * yi + 0.3 * yi**2) / (yj**2 + 0.3 * yi**2)
    refS = guided_filter(nYi, S, r, eps)
    out = restored * refS[..., None]
    if stages is not None:
        stages.update(S=S, refinedS=refS, out_exp=out)
    return _minmax_norm(out)


def bgdehaze_frame(bgr8: np.ndarray, w: int = 15, stages=None, r=40, eps=1e-3, tmin=0.2):
    """bgdehaze/main.py:16-19 minus file I/O: returns (float64 HxWx3 in [0,1], uint8 HxWx3 =
    what imwrite hands to the encoder: sat(rint(restored * 255)), NaN -> 0).  r, eps, tmin: the guided filters'
    radius and regulariser and the floor of the raw transmission (uwip_dehaze_params)."""
    normI = normalize_frame(bgr8)
    out = adaptive_exp_map(normI, w, stages, r, eps, tmin)
    return out, _sat_u8_from_rint(out * 255)


# ----------------------------------------------------------------------------------------
# the chain
# ----------------------------------------------------------------------------------------


def chain_frame(bgr8, lo=1, hi=99, clip=2.0, tiles_x=8, tiles_y=8, w=15, hsv_rounding="cv2"):
    """histretch -c=V (intended order) -> aclahe (fixed BS/CL) -> bgdehaze; each stage hands an
    8UC3 BGR frame to the next exactly as running the three tools back to back would."""
    a = histretch_frame(bgr8, "V", lo, hi, "intended", hsv_rounding)
    b = aclahe_frame(a, clip, tiles_x, tiles_y, hsv_rounding)
    return bgdehaze_frame(b, w)[1]


# ----------------------------------------------------------------------------------------
# deterministic synthetic underwater-like frames (integer only; CUDA twin in csrc/synth.cu)
# ----------------------------------------------------------------------------------------

_M32 = np.uint64(0xFFFFFFFF)


def _lowbias32(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64) & _M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & _M32
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & _M32
    x ^= x >> np.uint64(16)
    return x


def _tri(t: np.ndarray, period: int) -> np.ndarray:
    p = t % period
    v = (p * 510) // period
    return np.where(v > 255, 510 - v, v)


def _value_noise(seed, f, X, Y, cell, salt):
    cx, cy = X // cell, Y // cell
    fx = ((X % cell) * 256) // cell
    fy = ((Y % cell) * 256) // cell

    def lat(ix, iy):
        k = (
            np.uint64(seed)
            + np.uint64(salt) * np.uint64(0x9E3779B1)
            + np.uint64(f) * np.uint64(0x85EBCA77)
            + ix.astype(np.uint64) * np.uint64(0xC2B2AE3D)
            + iy.astype(np.uint64) * np.uint64(0x27D4EB2F)
        )
        return (_lowbias32(k) & np.uint64(255)).astype(np.int64)

    h00, h10 = lat(cx, cy), lat(cx + 1, cy)
    h01, h11 = lat(cx, cy + 1), lat(cx + 1, cy + 1)
    top = h00 * (256 - fx) + h10 * fx
    bot = h01 * (256 - fx) + h11 * fx
    return (top * (256 - fy) + bot * fy) >> 16


SYNTH_BASE = (120, 140, 30)
SYNTH_GAIN = (60, 50, -25)
SYNTH_TEXGAIN = (40, 36, 16)


def synth_frame(seed: int, f: int, width: int, height: int) -> np.ndarray:
    """pixel(seed,f,y,x,c) = clamp_u8(base_c + ((depth*gain_c)>>8) + ((tex*texgain_c)>>8) + noise)."""
    Y, X = np.meshgrid(np.arange(height, dtype=np.int64), np.arange(width, dtype=np.int64), indexing="ij")
    px, py = max(width // 2, 2), max(height // 3, 2)
    depth = (_tri(X + 7 * f, px) + _tri(Y + 5 * f, py)) >> 1
    tex = 2 * _value_noise(seed, f, X, Y, 32, 1) + _value_noise(seed, f, X, Y, 8, 2) - 384
    out = np.empty((height, width, 3), np.uint8)
    for c in range(3):
        k = (
            np.uint64(seed)
            + np.uint64(f) * np.uint64(0x85EBCA77)
            + Y.astype(np.uint64) * np.uint64(0x27D4EB2F)
            + X.astype(np.uint64) * np.uint64(0xC2B2AE3D)
            + np.uint64(c + 1) * np.uint64(0x165667B1)
        )
        noise = (_lowbias32(k) & np.uint64(7)).astype(np.int64) - 3
        val = SYNTH_BASE[c] + ((depth * SYNTH_GAIN[c]) >> 8) + ((tex * SYNTH_TEXGAIN[c]) >> 8) + noise
        out[..., c] = np.clip(val, 0, 255).astype(np.uint8)
    return out
