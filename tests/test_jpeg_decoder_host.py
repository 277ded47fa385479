"""The JPEG decoder arithmetic of csrc/jpegdec.h (what the GPU's batched decoder runs), compiled with g++ for the host: the
pixels of decode_frame() equal cv2.imdecode(file, IMREAD_COLOR) (libjpeg-turbo, islow, fancy upsampling) across sizes,
sampling factors, grey, qualities, restart intervals, optimised tables and content; the golden 1920 x 1080 frame; the files of
the project's own encoder; and the refusals (progressive, 4:1:1, arithmetic, 12-bit, truncated headers)."""
import os
import shutil
import subprocess

import cv2
import numpy as np
import pytest

from test_jpeg_encoder_host import contents

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

DRIVER_SRC = r"""
#include <cstdio>
#include <vector>
#include "jpegdec.h"
#include "jpegenc.h"
// stdin, one job per line:
//   dec <in.jpg> <out.raw>                       print status width height; out.raw: the bgr8 frame when status is 0 or 1
//   enc <w> <h> <quality> <in.raw> <out.jpg>     the project's encoder (jpegenc.h)
static std::vector<uint8_t> slurp(const char* p) {
  std::vector<uint8_t> d;
  FILE* f = fopen(p, "rb");
  if (!f) return d;
  int c;
  while ((c = fgetc(f)) != EOF) d.push_back((uint8_t)c);
  fclose(f);
  return d;
}
int main() {
  char op[16], in[4096], out[4096];
  while (scanf("%15s", op) == 1) {
    if (op[0] == 'd') {
      if (scanf("%4095s %4095s", in, out) != 2) return 1;
      std::vector<uint8_t> d = slurp(in);
      jpegdec::Header hd;
      int rc = jpegdec::parse_header(d.data(), d.size(), hd);
      if (rc == 0) {
        std::vector<uint8_t> px((size_t)hd.width * hd.height * 3);
        rc = jpegdec::decode_frame(d.data(), d.size(), px.data());
        FILE* f = fopen(out, "wb");
        fwrite(px.data(), 1, px.size(), f);
        fclose(f);
      }
      printf("%d %d %d\n", rc, hd.width, hd.height);
    } else {
      int w, h, q;
      if (scanf("%d %d %d %4095s %4095s", &w, &h, &q, in, out) != 5) return 1;
      std::vector<uint8_t> px = slurp(in), o(jpegenc::encode_bound(w, h));
      const size_t n = jpegenc::encode_frame(px.data(), w, h, q, o.data());
      FILE* f = fopen(out, "wb");
      fwrite(o.data(), 1, n, f);
      fclose(f);
      printf("%zu\n", n);
    }
    fflush(stdout);
  }
  return 0;
}
"""

SIZES = [(1, 1), (1, 29), (23, 1), (2, 2), (3, 5), (4, 7), (5, 3), (7, 9), (8, 8), (15, 17), (16, 16), (17, 16), (53, 37), (481, 270)]
SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420}
EXTRAS = {"plain": [], "rst1": [cv2.IMWRITE_JPEG_RST_INTERVAL, 1], "rst7": [cv2.IMWRITE_JPEG_RST_INTERVAL, 7],
          "optimize": [cv2.IMWRITE_JPEG_OPTIMIZE, 1]}


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("jpegdec")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(DRIVER_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)],
                   check=True)
    return str(exe), d


def _run(driver, lines):
    exe, _ = driver
    out = subprocess.run([exe], input="\n".join(lines) + "\n", check=True, capture_output=True, text=True).stdout
    return out.split("\n")[:len(lines)]


def decode(driver, files):
    """files: list of bytes -> list of (status, frame or None)."""
    _, d = driver
    lines = []
    for i, b in enumerate(files):
        (d / ("d%d.jpg" % i)).write_bytes(b)
        lines.append("dec %s %s" % (d / ("d%d.jpg" % i), d / ("d%d.raw" % i)))
    res = []
    for i, row in enumerate(_run(driver, lines)):
        rc, w, h = (int(v) for v in row.split())
        px = np.fromfile(str(d / ("d%d.raw" % i)), np.uint8).reshape(h, w, 3) if rc in (0, 1) else None
        res.append((rc, px))
    return res


def imencode(img, q, sampling=None, extra=()):
    p = [cv2.IMWRITE_JPEG_QUALITY, q] + ([cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]] if sampling else []) + list(extra)
    ok, b = cv2.imencode(".jpg", img, p)
    assert ok
    return bytes(b)


def _check(driver, files, names):
    got = decode(driver, files)
    bad = []
    for name, b, (rc, px) in zip(names, files, got):
        want = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)
        if rc != 0 or px.shape != want.shape or not (px == want).all():
            bad.append(name)
    assert not bad, "%d of %d files differ from cv2.imdecode: %s" % (len(bad), len(files), bad[:8])


@pytest.mark.parametrize("sampling", ["444", "422", "440", "420", "grey"])
@pytest.mark.parametrize("q", [1, 50, 95, 100])
def test_pixels_equal_cv2_imdecode(driver, sampling, q):
    files, names = [], []
    for (w, h) in SIZES:
        for cname, f in contents(w, h, 1000 * w + h).items():
            for ename, extra in EXTRAS.items():
                if sampling == "grey":
                    files.append(imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), q, None, extra))
                else:
                    files.append(imencode(f, q, sampling, extra))
                names.append("%dx%d %s %s" % (w, h, cname, ename))
    _check(driver, files, names)


def test_upsampling_fallback_widths(driver):
    """h2v1 / h2v2 fancy upsampling needs downsampled_width > 2: widths 1 to 5 cover both sides of the fallback."""
    files, names = [], []
    for w in range(1, 6):
        for h in (1, 2, 3, 6):
            for s in ("422", "420", "440"):
                f = contents(w, h, 31 * w + h)["noise"]
                files.append(imencode(f, 90, s))
                names.append("%dx%d %s" % (w, h, s))
    _check(driver, files, names)


def test_luma_quality_differs_from_chroma(driver):
    files, names = [], []
    for (w, h) in [(17, 16), (53, 37), (481, 270)]:
        for cname, f in contents(w, h, w + h).items():
            for lq, cq in [(95, 30), (20, 90)]:
                for s in ("420", "444"):
                    files.append(imencode(f, 75, s, [cv2.IMWRITE_JPEG_LUMA_QUALITY, lq, cv2.IMWRITE_JPEG_CHROMA_QUALITY, cq]))
                    names.append("%dx%d %s %d/%d %s" % (w, h, cname, lq, cq, s))
    _check(driver, files, names)


def test_full_hd_golden_frame(driver):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    files = [imencode(img, q, s) for q in (75, 95) for s in ("420", "444")] + [imencode(img, 95, "420", EXTRAS["rst7"])]
    _check(driver, files, ["q%d %s" % (q, s) for q in (75, 95) for s in ("420", "444")] + ["rst7"])


def test_files_of_the_project_encoder(driver):
    """The files csrc/jpegenc.h writes (byte-identical to cv2.imencode) decode to cv2.imdecode's pixels."""
    _, d = driver
    lines, names = [], []
    for (w, h) in [(1, 1), (7, 9), (53, 37), (481, 270)]:
        for cname, f in contents(w, h, 5 * w + h).items():
            raw = d / ("e%d.raw" % len(names))
            raw.write_bytes(np.ascontiguousarray(f).tobytes())
            lines.append("enc %d %d 95 %s %s" % (w, h, raw, d / ("e%d.jpg" % len(names))))
            names.append("%dx%d %s" % (w, h, cname))
    _run(driver, lines)
    files = [(d / ("e%d.jpg" % i)).read_bytes() for i in range(len(names))]
    _check(driver, files, names)


def _segments(b):
    """(marker, offset of its 0xFF) of the header segments up to SOS"""
    out, i = [], 2
    while i < len(b):
        m = b[i + 1]
        out.append((m, i))
        if m == 0xDA:
            break
        i += 2 + int.from_bytes(b[i + 2:i + 4], "big")
    return out


def test_refusals(driver):
    f = contents(40, 24, 3)["gradient"]
    base = imencode(f, 90, "420")
    ok, prog = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    assert ok
    s411 = imencode(f, 90, None, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])
    sof = dict(_segments(base))[0xC0]
    sof9 = bytearray(base)
    sof9[sof + 1] = 0xC9
    bit12 = bytearray(base)
    bit12[sof + 4] = 12
    dht = dict(_segments(base))[0xC4]
    files = [bytes(prog), s411, bytes(sof9), bytes(bit12), base[:dht + 10], base[:sof + 6], b"\xff\xd8", b"not a jpeg", base]
    got = [rc for rc, _ in decode(driver, files)]
    assert got == [-3, -3, -3, -3, -1, -1, -1, -1, 0]


def test_truncated_scan_is_bad_data(driver):
    f = contents(64, 48, 9)["noise"]
    b = imencode(f, 95, "420")
    sos = dict(_segments(b))[0xDA]
    cut = b[:sos + 14 + (len(b) - sos) // 2]
    (rc, px), = decode(driver, [cut])
    assert rc == 1 and px is not None and not px.any()
