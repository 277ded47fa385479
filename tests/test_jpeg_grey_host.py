"""The grey halves of csrc/jpegenc.h and csrc/jpegdec.h (what the GPU's batched grey writer and reader run), compiled with g++
for the host: encode_grey_frame() writes the bytes of cv2.imencode(".jpg", plane) for a 2-D plane (one component, one block
per MCU) across sizes, qualities and content, within uwip_jpeg_encode_u8_bound; decode_frame(.., grey) gives
cv2.imdecode(file, IMREAD_GRAYSCALE) for grey and YCbCr files of every accepted sampling, restart interval and table choice,
and refuses what the colour reader refuses."""
import os
import shutil
import subprocess

import cv2
import numpy as np
import pytest

from test_jpeg_decoder_host import EXTRAS, SAMPLING, _segments, imencode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

DRIVER_SRC = r"""
#include <cstdio>
#include <vector>
#include "jpegdec.h"
#include "jpegenc.h"
// stdin, one job per line:
//   enc <w> <h> <quality> <in.raw> <out.jpg>   encode the grey plane in in.raw, print the file length
//   dec <in.jpg> <out.raw>                     print status width height; out.raw: the grey plane when status is 0 or 1
//   bound <w> <h>                              print encode_bound(w, h, 1) and GREY_HEADER_BYTES
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
    if (op[0] == 'e') {
      int w, h, q;
      if (scanf("%d %d %d %4095s %4095s", &w, &h, &q, in, out) != 5) return 1;
      std::vector<uint8_t> px = slurp(in), o(jpegenc::encode_bound(w, h, 1));
      const size_t n = jpegenc::encode_grey_frame(px.data(), w, h, q, o.data());
      FILE* f = fopen(out, "wb");
      fwrite(o.data(), 1, n, f);
      fclose(f);
      printf("%zu\n", n);
    } else if (op[0] == 'd') {
      if (scanf("%4095s %4095s", in, out) != 2) return 1;
      std::vector<uint8_t> d = slurp(in);
      jpegdec::Header hd;
      int rc = jpegdec::parse_header(d.data(), d.size(), hd);
      if (rc == 0) {
        std::vector<uint8_t> px((size_t)hd.width * hd.height);
        rc = jpegdec::decode_frame(d.data(), d.size(), px.data(), true);
        FILE* f = fopen(out, "wb");
        fwrite(px.data(), 1, px.size(), f);
        fclose(f);
      }
      printf("%d %d %d\n", rc, hd.width, hd.height);
    } else {
      int w, h;
      if (scanf("%d %d", &w, &h) != 2) return 1;
      printf("%zu %d\n", jpegenc::encode_bound(w, h, 1), jpegenc::GREY_HEADER_BYTES);
    }
    fflush(stdout);
  }
  return 0;
}
"""

SIZES = [(1, 1), (1, 29), (23, 1), (7, 9), (8, 8), (15, 17), (17, 16), (53, 37), (481, 270)]   # (w, h)
QUALITIES = [1, 10, 50, 75, 90, 95, 100]


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("jpeggrey")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(DRIVER_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)],
                   check=True)
    return str(exe), d


def _run(driver, lines):
    exe, _ = driver
    out = subprocess.run([exe], input="\n".join(lines) + "\n", check=True, capture_output=True, text=True).stdout
    return out.split("\n")[:len(lines)]


def _encode(driver, planes, q):
    _, d = driver
    lines, outs = [], []
    for i, p in enumerate(planes):
        src, dst = d / ("g%d.raw" % i), d / ("g%d.jpg" % i)
        src.write_bytes(np.ascontiguousarray(p).tobytes())
        lines.append("enc %d %d %d %s %s" % (p.shape[1], p.shape[0], q, src, dst))
        outs.append(dst)
    lens = _run(driver, lines)
    got = [p.read_bytes() for p in outs]
    assert [len(g) for g in got] == [int(n) for n in lens]
    return got


def _decode(driver, files):
    _, d = driver
    lines = []
    for i, b in enumerate(files):
        (d / ("r%d.jpg" % i)).write_bytes(b)
        lines.append("dec %s %s" % (d / ("r%d.jpg" % i), d / ("r%d.raw" % i)))
    res = []
    for i, row in enumerate(_run(driver, lines)):
        rc, w, h = (int(v) for v in row.split())
        px = np.fromfile(str(d / ("r%d.raw" % i)), np.uint8).reshape(h, w) if rc in (0, 1) else None
        res.append((rc, px))
    return res


def _cv2(p, q):
    ok, b = cv2.imencode(".jpg", p, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(b)


def planes(w, h, seed):
    """flat 0 / 128 / 255, two gradients, noise"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    return {
        "zero": np.zeros((h, w), np.uint8),
        "flat": np.full((h, w), 128, np.uint8),
        "white": np.full((h, w), 255, np.uint8),
        "gradient": ((xx * 255 // max(w - 1, 1) + yy * 3) % 256).astype(np.uint8),
        "diagonal": ((xx * 3 + yy * 5) % 256).astype(np.uint8),
        "noise": rng.integers(0, 256, (h, w), dtype=np.uint8),
    }


def grey_bound(w, h):
    """Python mirror of uwip_jpeg_encode_u8_bound (jpegenc::encode_bound(w, h, 1))."""
    bits = ((w + 7) // 8) * ((h + 7) // 8) * (9 + 11 + 63 * (16 + 10))
    raw = ((bits + 7) // 8 + 16 + 15) // 16 * 16
    return 328 + 2 * raw + 2 + 16


@pytest.mark.parametrize("q", QUALITIES)
def test_grey_files_equal_cv2_imencode(driver, q):
    ps, names = [], []
    for (w, h) in SIZES:
        for name, p in planes(w, h, 1000 * w + h).items():
            ps.append(p)
            names.append("%dx%d %s" % (w, h, name))
    got = _encode(driver, ps, q)
    bad = [n for n, p, g in zip(names, ps, got) if g != _cv2(p, q)]
    assert not bad, "q=%d: %d of %d files differ: %s" % (q, len(bad), len(ps), bad[:8])


def test_grey_header_and_bound(driver):
    sizes = [(1, 1), (8, 8), (17, 16), (53, 37), (256, 128)]
    rows = _run(driver, ["bound %d %d" % s for s in sizes])
    for (w, h), row in zip(sizes, rows):
        bound, header = (int(v) for v in row.split())
        assert bound == grey_bound(w, h) and header == 328
        assert bytes(_cv2(np.zeros((h, w), np.uint8), 95)).find(b"\xff\xda") + 10 == 328
    rng = np.random.default_rng(7)
    ps = [rng.integers(0, 256, (h, w), dtype=np.uint8) for (w, h) in sizes]
    ps += [((np.indices((h, w)).sum(0) % 2) * 255).astype(np.uint8) for (w, h) in sizes]
    got = _encode(driver, ps, 100)
    for p, g in zip(ps, got):
        assert g == _cv2(p, 100)
        assert len(g) <= grey_bound(p.shape[1], p.shape[0])


def _check(driver, files, names):
    got = _decode(driver, files)
    bad = []
    for name, b, (rc, px) in zip(names, files, got):
        want = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_GRAYSCALE)
        if rc != 0 or px.shape != want.shape or not (px == want).all():
            bad.append(name)
    assert not bad, "%d of %d files differ from cv2.imdecode(.., IMREAD_GRAYSCALE): %s" % (len(bad), len(files), bad[:8])


@pytest.mark.parametrize("sampling", ["444", "422", "440", "420", "grey"])
def test_grey_planes_equal_cv2_imdecode(driver, sampling):
    files, names = [], []
    rng = np.random.default_rng(5)
    for (w, h) in SIZES:
        for q in (50, 95):
            for ename, extra in EXTRAS.items():
                f = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
                if sampling == "grey":
                    files.append(imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), q, None, extra))
                else:
                    files.append(imencode(f, q, sampling, extra))
                names.append("%dx%d q%d %s" % (w, h, q, ename))
    _check(driver, files, names)


def test_grey_plane_of_colour_file_is_not_cvtcolor(driver):
    """IMREAD_GRAYSCALE of a YCbCr file is its Y component, which cvtColor of the colour pixels does not give back."""
    f = np.random.default_rng(3).integers(0, 256, (48, 64, 3), dtype=np.uint8)
    b = imencode(f, 50, "444")
    ((rc, px),) = _decode(driver, [b])
    assert rc == 0
    assert (px == cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_GRAYSCALE)).all()
    assert (px != cv2.cvtColor(cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR), cv2.COLOR_BGR2GRAY)).any()


def test_grey_full_hd_golden_frame(driver):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    files = [imencode(img, q, s) for q in (75, 95) for s in ("420", "444")] + [imencode(img, 95, "420", EXTRAS["rst7"]),
                                                                             imencode(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), 95)]
    _check(driver, files, ["q75 420", "q75 444", "q95 420", "q95 444", "rst7", "grey"])


def test_grey_files_of_the_project_encoder(driver):
    ps, names = [], []
    for (w, h) in [(1, 1), (7, 9), (53, 37), (481, 270)]:
        for name, p in planes(w, h, 5 * w + h).items():
            ps.append(p)
            names.append("%dx%d %s" % (w, h, name))
    _check(driver, _encode(driver, ps, 95), names)


def test_grey_refusals(driver):
    f = np.random.default_rng(1).integers(0, 256, (24, 40, 3), dtype=np.uint8)
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
    got = [rc for rc, _ in _decode(driver, files)]
    assert got == [-3, -3, -3, -3, -1, -1, -1, -1, 0]


def test_grey_truncated_scan_is_bad_data(driver):
    b = imencode(np.random.default_rng(9).integers(0, 256, (48, 64, 3), dtype=np.uint8), 95, "420")
    sos = dict(_segments(b))[0xDA]
    ((rc, px),) = _decode(driver, [b[:sos + 14 + (len(b) - sos) // 2]])
    assert rc == 1 and px is not None and not px.any()
