"""The progressive half of csrc/jpegdec.h (what the GPU's progressive passes run), compiled with g++ for the host: the
whole-file marker reader parse_file and decode_frame_ex give cv2.imdecode(file, IMREAD_COLOR) and
cv2.imdecode(file, IMREAD_GRAYSCALE), with and without the Exif orientation, for progressive files written by cv2 and by
Pillow across sizes, samplings, qualities and restart intervals, and the golden 1920 x 1080 frame.  Baseline files decode as
decode_frame does.  The refusals: incomplete progressions (cut after a scan, EOI appended), an Ah that is not the previous
Al, bad Ss / Se / Ah / Al, SOF10 and progressive 4:1:1; a file cut inside a scan is bad data."""
import io
import os
import re
import shutil
import subprocess

import cv2
import numpy as np
import pytest

from test_jpeg_decoder_host import SAMPLING
from test_jpeg_orientation_host import frame, tag

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

DRIVER_SRC = r"""
#include <cstdio>
#include <vector>
#include "jpegdec.h"
// stdin, one job per line:  <in.jpg> <out.raw> <grey 0|1> <orient 0|1> <ex 0|1>
// ex = 1: decode_frame_ex, ex = 0: decode_frame.  Prints: status progressive scans out_width out_height; out.raw holds the
// pixels when the status is 0 or 1
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
  char in[4096], out[4096];
  int grey, orient, ex;
  static jpegdec::Prog pg;
  while (scanf("%4095s %4095s %d %d %d", in, out, &grey, &orient, &ex) == 5) {
    std::vector<uint8_t> d = slurp(in);
    jpegdec::Header hd;
    int rc = jpegdec::parse_file(d.data(), d.size(), hd, &pg);
    const bool t = orient && hd.orientation >= 5;
    const int w = t ? hd.height : hd.width, h = t ? hd.width : hd.height;
    if (rc == 0) {
      std::vector<uint8_t> px((size_t)w * h * (grey ? 1 : 3));
      rc = ex ? jpegdec::decode_frame_ex(d.data(), d.size(), px.data(), grey != 0, orient != 0)
              : jpegdec::decode_frame(d.data(), d.size(), px.data(), grey != 0, orient != 0);
      FILE* f = fopen(out, "wb");
      fwrite(px.data(), 1, px.size(), f);
      fclose(f);
    }
    printf("%d %d %d %d %d\n", rc, pg.nscans > 0, pg.nscans, w, h);
    fflush(stdout);
  }
  return 0;
}
"""


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("jpegprog")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(DRIVER_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)],
                   check=True)
    return str(exe), d


def decode(driver, files, grey=False, orient=False, ex=True):
    """[(status, progressive, scans, pixels or None)] of decode_frame_ex (ex) or decode_frame over the files"""
    exe, d = driver
    lines = []
    for i, b in enumerate(files):
        (d / ("p%d.jpg" % i)).write_bytes(b)
        lines.append("%s %s %d %d %d" % (d / ("p%d.jpg" % i), d / ("p%d.raw" % i), grey, orient, ex))
    rows = subprocess.run([exe], input="\n".join(lines) + "\n", check=True, capture_output=True, text=True).stdout.split("\n")
    res = []
    for i, row in enumerate(rows[:len(files)]):
        rc, prog, ns, w, h = (int(v) for v in row.split())
        shape = (h, w) if grey else (h, w, 3)
        res.append((rc, prog, ns, np.fromfile(str(d / ("p%d.raw" % i)), np.uint8).reshape(shape) if rc in (0, 1) else None))
    return res


def cv2_prog(img, q, sampling=None, rst=0):
    """cv2.imwrite's progressive file (libjpeg-turbo's jpeg_simple_progression)"""
    p = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
    if sampling:
        p += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    if rst:
        p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    ok, b = cv2.imencode(".jpg", img, p)
    assert ok
    return bytes(b)


def pil_prog(img, q, sampling):
    """Pillow's progressive file: bgr8 or grey img; sampling 444 / 422 / 420 / grey"""
    from PIL import Image

    buf = io.BytesIO()
    if sampling == "grey":
        Image.fromarray(img if img.ndim == 2 else cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)).save(buf, "JPEG", quality=q, progressive=True)
    else:
        sub = {"444": 0, "422": 1, "420": 2}[sampling]
        Image.fromarray(img[..., ::-1].copy()).save(buf, "JPEG", quality=q, progressive=True, subsampling=sub)
    return buf.getvalue()


def prog_file(w, h, sampling, q, rst=0, seed=1):
    f = frame(w, h, seed)
    if sampling == "grey":
        return cv2_prog(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), q, None, rst)
    return cv2_prog(f, q, sampling, rst)


def cv2_decode(b, grey=False, orient=False):
    flags = (cv2.IMREAD_GRAYSCALE if grey else cv2.IMREAD_COLOR) | (0 if orient else cv2.IMREAD_IGNORE_ORIENTATION)
    return cv2.imdecode(np.frombuffer(b, np.uint8), flags)


def _check(driver, files, grey=False, orient=False):
    got = decode(driver, files, grey, orient)
    bad = []
    for i, (b, (rc, prog, _, px)) in enumerate(zip(files, got)):
        want = cv2_decode(b, grey, orient)
        if rc != 0 or px.shape != want.shape or not (px == want).all():
            bad.append((i, rc, None if px is None else int(np.abs(px.astype(int) - want).max()) if px.shape == want.shape else px.shape))
    assert not bad, bad[:10]
    return got


# ---- the marker-level structure of a progressive file -------------------------------------------------------------------
def sos_offsets(b):
    """byte offsets of every SOS marker (0xFF 0xDA cannot occur inside entropy-coded data)"""
    return [m.start() for m in re.finditer(rb"\xff\xda", b)]


def scan_end(b, sos):
    """the offset of the marker that ends the scan whose SOS is at `sos`"""
    start = sos + 2 + int.from_bytes(b[sos + 2:sos + 4], "big")
    return re.compile(rb"\xff[^\x00\xd0-\xd7\xff]").search(b, start).start()


def set_scan(b, k, ss=None, se=None, ah=None, al=None):
    """the file with scan k's Ss, Se, Ah, Al replaced"""
    sos = sos_offsets(b)[k]
    n = b[sos + 4]
    p = sos + 5 + 2 * n
    s = bytearray(b)
    s0, s1, a = s[p], s[p + 1], s[p + 2]
    s[p] = s0 if ss is None else ss
    s[p + 1] = s1 if se is None else se
    s[p + 2] = ((a >> 4 if ah is None else ah) << 4) | (a & 15 if al is None else al)
    return bytes(s)


SIZES = [(1, 1), (7, 5), (8, 8), (17, 9), (40, 24), (481, 270)]
SAMPLINGS = ["444", "422", "440", "420", "grey"]


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_cv2_progressive_equal_cv2(driver, sampling):
    files = []
    for i, (w, h) in enumerate(SIZES):
        for j, q in enumerate((1, 50, 95, 100)):
            files.append(prog_file(w, h, sampling, q, (0, 1, 7)[(i + j) % 3], seed=10 * i + j))
    got = _check(driver, files)
    assert all(prog == 1 and ns >= 6 for _, prog, ns, _ in got)
    _check(driver, files, grey=True)


@pytest.mark.parametrize("sampling", ["444", "422", "420", "grey"])
def test_pillow_progressive_equal_cv2(driver, sampling):
    # Pillow's own output buffer is too small for 481 x 270 at 4:4:4 and high qualities, so that size stops at q50
    files = [pil_prog(frame(w, h, 7 + i), q if w < 400 else min(q, 50), sampling) for i, (w, h) in enumerate(SIZES) for q in (1, 50, 95, 100)]
    got = _check(driver, files)
    assert all(prog == 1 for _, prog, _, _ in got)
    _check(driver, files, grey=True)


@pytest.mark.parametrize("rst", [1, 7])
def test_restart_intervals(driver, rst):
    files = [prog_file(w, h, s, 90, rst, seed=i) for i, (w, h) in enumerate([(40, 24), (481, 270), (17, 9)]) for s in SAMPLINGS]
    _check(driver, files)
    _check(driver, files, grey=True)


def test_exif_orientation(driver):
    files = [tag(prog_file(40, 24, s, 90, (0, 7)[o % 2], seed=o), o, le=o % 2 == 0) for o in range(1, 9) for s in ("420", "grey", "422")]
    for grey in (False, True):
        _check(driver, files, grey, orient=True)
        _check(driver, files, grey, orient=False)


def test_full_hd_golden_frame(driver):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    assert img.shape == (1080, 1920, 3)
    files = [cv2_prog(img, 95, "420"), cv2_prog(img, 75, "444", 7), pil_prog(img, 90, "420")]
    _check(driver, files)
    _check(driver, files, grey=True)


def test_baseline_as_decode_frame(driver):
    from test_jpeg_decoder_host import imencode

    files = [imencode(frame(w, h, i), q, s, ([cv2.IMWRITE_JPEG_RST_INTERVAL, 3] if i % 2 else [])) for i, (w, h) in enumerate(SIZES)
             for q, s in ((90, "420"), (50, "444"), (95, "422"))]
    for grey in (False, True):
        a, b = decode(driver, files, grey, ex=True), decode(driver, files, grey, ex=False)
        assert all(x[0] == 0 and x[1] == 0 and y[0] == 0 and (x[3] == y[3]).all() for x, y in zip(a, b))


# ---- refusals and bad data ---------------------------------------------------------------------------------------------
def test_incomplete_progressions_unsupported(driver):
    for b in (prog_file(40, 24, "420", 90), prog_file(40, 24, "grey", 90), prog_file(17, 9, "444", 50, 1)):
        sos = sos_offsets(b)
        cut = [b[:scan_end(b, sos[k])] + b"\xff\xd9" for k in range(len(sos) - 1)]
        for k in {0, 1, 4, 5, len(sos) - 2} & set(range(len(cut))):
            assert cv2.imdecode(np.frombuffer(cut[k], np.uint8), cv2.IMREAD_COLOR) is not None   # cv2 smooths them
        assert [r[0] for r in decode(driver, cut)] == [-3] * len(cut)
        assert decode(driver, [b[:scan_end(b, sos[-1])] + b"\xff\xd9"])[0][0] == 0   # every scan: complete


def test_ah_al_mismatch_unsupported(driver):
    b = prog_file(40, 24, "420", 90)
    last = len(sos_offsets(b)) - 1   # Y 1..63 refined from Al 1 to 0
    assert decode(driver, [set_scan(b, last, ah=2, al=1)])[0][0] == -3
    assert decode(driver, [set_scan(b, 1, ah=1, al=0)])[0][0] == -3   # a first AC scan that claims to refine


@pytest.mark.parametrize("edit", [dict(ss=0, se=5), dict(ss=6, se=5), dict(se=64), dict(al=14), dict(ah=3, al=1)],
                         ids=["dc_se", "ss_gt_se", "se_64", "al_14", "ah_al"])
def test_bad_progression_parameters_invalid(driver, edit):
    b = prog_file(40, 24, "420", 90)
    k = 1 if "ss" in edit or "se" in edit else len(sos_offsets(b)) - 1
    if edit == dict(ss=0, se=5):
        k = 0   # a DC scan with Se 5
        edit = dict(se=5)
    assert decode(driver, [set_scan(b, k, **edit)])[0][0] == -1


def test_multi_component_ac_scan_invalid(driver):
    b = prog_file(40, 24, "420", 90)
    assert decode(driver, [set_scan(b, 0, ss=1, se=5)])[0][0] == -1   # the 3-component first scan made an AC scan


def test_sof10_and_411_unsupported(driver):
    b = prog_file(40, 24, "420", 90)
    i = b.index(b"\xff\xc2")
    sof10 = b[:i] + b"\xff\xca" + b[i + 2:]
    ok, f411 = cv2.imencode(".jpg", frame(40, 24, 3), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                                        cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])
    assert [r[0] for r in decode(driver, [sof10, bytes(f411)])] == [-3, -3]


def test_cut_inside_a_scan_is_bad_data(driver):
    b = prog_file(481, 270, "420", 95)
    sos = sos_offsets(b)
    inside = [b[:(sos[k] + scan_end(b, sos[k])) // 2] for k in (0, 4, len(sos) - 1)] + [b[:len(b) - 40]]
    for grey in (False, True):
        got = decode(driver, inside, grey)
        assert [r[0] for r in got] == [1] * len(inside)
        assert not any(r[3].any() for r in got)
