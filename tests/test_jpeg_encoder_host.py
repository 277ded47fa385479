"""The JPEG encoder arithmetic of csrc/jpegenc.h (what the GPU's batched encoder runs), compiled with g++ for the host: whole
files byte-identical to cv2.imencode (libjpeg-turbo, baseline 4:2:0, standard tables) across sizes, qualities and content;
compute_reciprocal against a direct evaluation of the formula; worst-case output within uwip_jpeg_encode_bound."""
import os
import shutil
import subprocess

import cv2
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

DRIVER_SRC = r"""
#include <cstdio>
#include <vector>
#include "jpegenc.h"
// stdin, one job per line:
//   enc <w> <h> <quality> <in.raw> <out.jpg>   encode the bgr8 frame in in.raw, print the file length
//   recip <divisor>                            print recip corr shift
//   bound <w> <h>                              print encode_bound and HEADER_BYTES
int main() {
  char op[16];
  while (scanf("%15s", op) == 1) {
    if (op[0] == 'e') {
      int w, h, q;
      char in[4096], out[4096];
      if (scanf("%d %d %d %4095s %4095s", &w, &h, &q, in, out) != 5) return 1;
      std::vector<uint8_t> px((size_t)w * h * 3), o(jpegenc::encode_bound(w, h));
      FILE* f = fopen(in, "rb");
      if (!f || fread(px.data(), 1, px.size(), f) != px.size()) return 2;
      fclose(f);
      const size_t n = jpegenc::encode_frame(px.data(), w, h, q, o.data());
      f = fopen(out, "wb");
      fwrite(o.data(), 1, n, f);
      fclose(f);
      printf("%zu\n", n);
    } else if (op[0] == 'r') {
      unsigned d;
      if (scanf("%u", &d) != 1) return 1;
      const jpegenc::Recip r = jpegenc::compute_reciprocal(d);
      printf("%u %u %d\n", r.recip, r.corr, r.shift);
    } else {
      int w, h;
      if (scanf("%d %d", &w, &h) != 2) return 1;
      printf("%zu %d\n", jpegenc::encode_bound(w, h), jpegenc::HEADER_BYTES);
    }
    fflush(stdout);
  }
  return 0;
}
"""

SIZES = [(1, 1), (1, 29), (23, 1), (7, 9), (8, 8), (15, 17), (16, 16), (17, 16), (53, 37), (481, 270)]   # (w, h)
QUALITIES = [1, 10, 50, 75, 90, 95, 100]


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("jpegenc")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(DRIVER_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)],
                   check=True)
    return str(exe), d


def _run(driver, lines):
    exe, _ = driver
    out = subprocess.run([exe], input="\n".join(lines) + "\n", check=True, capture_output=True, text=True).stdout
    return out.split("\n")[:len(lines)]


def _encode(driver, frames, q):
    """frames: list of (H, W, 3) uint8 -> list of the driver's file bytes."""
    _, d = driver
    lines, outs = [], []
    for i, f in enumerate(frames):
        src, dst = d / ("f%d.raw" % i), d / ("f%d.jpg" % i)
        src.write_bytes(np.ascontiguousarray(f).tobytes())
        lines.append("enc %d %d %d %s %s" % (f.shape[1], f.shape[0], q, src, dst))
        outs.append(dst)
    lens = _run(driver, lines)
    got = [p.read_bytes() for p in outs]
    assert [len(g) for g in got] == [int(n) for n in lens]
    return got


def _cv2(f, q):
    ok, b = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(b)


def contents(w, h, seed):
    """noise, two gradients, constant 0 / 128 / 255, saturated colour edges"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    out = {
        "noise": rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
        "gradient": np.stack([xx * 255 // max(w - 1, 1), yy * 255 // max(h - 1, 1), ((xx + yy) * 7) % 256], -1).astype(np.uint8),
        "diagonal": np.stack([(xx * 3 + yy) % 256, (255 - xx) % 256, (yy * 5) % 256], -1).astype(np.uint8),
        "zero": np.zeros((h, w, 3), np.uint8),
        "grey": np.full((h, w, 3), 128, np.uint8),
        "white": np.full((h, w, 3), 255, np.uint8),
    }
    edges = np.zeros((h, w, 3), np.uint8)
    cols = np.array([[0, 0, 255], [0, 255, 0], [255, 0, 0], [255, 255, 255], [0, 0, 0], [255, 0, 255]], np.uint8)
    edges[:] = cols[((xx // 3) + (yy // 5)) % len(cols)]
    out["edges"] = edges
    return out


@pytest.mark.parametrize("q", QUALITIES)
def test_files_equal_cv2_imencode(driver, q):
    frames, names = [], []
    for (w, h) in SIZES:
        for name, f in contents(w, h, 1000 * w + h).items():
            frames.append(f)
            names.append("%dx%d %s" % (w, h, name))
    got = _encode(driver, frames, q)
    bad = [n for n, f, g in zip(names, frames, got) if g != _cv2(f, q)]
    assert not bad, "q=%d: %d of %d files differ: %s" % (q, len(bad), len(frames), bad[:8])


@pytest.mark.parametrize("q", [75, 95])
def test_full_hd_frame_equals_cv2_imencode(driver, q):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    assert img.shape == (1080, 1920, 3)
    (got,) = _encode(driver, [img], q)
    assert got == _cv2(img, q)


def test_compute_reciprocal_every_quantiser(driver):
    """compute_reciprocal (jcdctmgr.c) for every divisor q << 3 that any quality produces, against the formula evaluated here;
    and over the whole range of |islow output| the quantisation it drives equals the rounding division (|x| + d/2) / d."""
    qs = sorted({int(v) for t in (0, 1) for quality in range(1, 101) for v in _qtable(t, quality)})
    divisors = [q << 3 for q in qs]
    rows = _run(driver, ["recip %d" % d for d in divisors])
    for d, row in zip(divisors, rows):
        recip, corr, shift = (int(v) for v in row.split())
        b = d.bit_length() - 1
        r = 16 + b
        fq, fr, c = (1 << r) // d, (1 << r) % d, d // 2
        if fr == 0:
            fq, r = fq >> 1, r - 1
        elif fr <= d // 2:
            c += 1
        else:
            fq += 1
        assert (recip, corr, shift) == (fq, c, r), d
        a = np.arange(0, 8 * 1024 * 8 + 1, dtype=np.int64)
        assert (((a + corr) * recip) >> shift == (a + d // 2) // d).all(), d


def _qtable(t, quality):
    lum = [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
           18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112,
           100, 103, 99]
    chrom = [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99,
             99, 99] + [99] * 32
    s = 5000 // quality if quality < 50 else 200 - 2 * quality
    return np.clip([(b * s + 50) // 100 for b in (lum if t == 0 else chrom)], 1, 255)


def encode_bound(w, h):
    """Python mirror of uwip_jpeg_encode_bound (jpegenc::encode_bound)."""
    mcu_bits = 4 * (9 + 11 + 63 * (16 + 10)) + 2 * (11 + 11 + 63 * (16 + 10))
    bits = ((w + 15) // 16) * ((h + 15) // 16) * mcu_bits
    raw = ((bits + 7) // 8 + 16 + 15) // 16 * 16
    return 623 + 2 * raw + 2 + 16


def test_bound_holds_for_quality_100_noise(driver):
    sizes = [(1, 1), (8, 8), (17, 16), (53, 37), (256, 128)]
    rows = _run(driver, ["bound %d %d" % s for s in sizes])
    for (w, h), row in zip(sizes, rows):
        bound, header = (int(v) for v in row.split())
        assert bound == encode_bound(w, h) and header == 623
    rng = np.random.default_rng(7)
    frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for (w, h) in sizes]
    # alternating extremes make the largest coefficients the tables allow
    frames += [((np.indices((h, w)).sum(0) % 2) * 255).astype(np.uint8)[..., None].repeat(3, -1) for (w, h) in sizes]
    got = _encode(driver, frames, 100)
    for f, g in zip(frames, got):
        assert g == _cv2(f, 100)
        assert len(g) <= encode_bound(f.shape[1], f.shape[0])
