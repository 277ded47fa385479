"""The Exif orientation of csrc/jpegdec.h (what the GPU's oriented readers run), compiled with g++ for the host: parse_header
records the orientation cv2.imdecode applies and decode_frame(.., grey, orient = true) gives cv2.imdecode(file, IMREAD_COLOR)
and cv2.imdecode(file, IMREAD_GRAYSCALE) with their default flags, for all eight orientations in both TIFF byte orders, every
accepted sampling, grey files, edge sizes and restart intervals.  The marker reader's Exif rules are checked against cv2
itself on files built to probe them (cv2 writes no Exif, so the APP1 segments are spliced in), and through the library's
uwip_jpeg_orientation.  decode_frame(.., orient = false) keeps the stored orientation."""
import ctypes as C
import os
import shutil
import struct
import subprocess

import cv2
import numpy as np
import pytest

from test_jpeg_decoder_host import SAMPLING, imencode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DRIVER_SRC = r"""
#include <cstdio>
#include <vector>
#include "jpegdec.h"
// stdin, one job per line:  <in.jpg> <out.raw> <grey 0|1> <orient 0|1>
// prints: status orientation out_width out_height; out.raw holds the pixels when the status is 0 or 1
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
  int grey, orient;
  while (scanf("%4095s %4095s %d %d", in, out, &grey, &orient) == 4) {
    std::vector<uint8_t> d = slurp(in);
    jpegdec::Header hd;
    int rc = jpegdec::parse_header(d.data(), d.size(), hd);
    const bool t = orient && hd.orientation >= 5;
    const int w = t ? hd.height : hd.width, h = t ? hd.width : hd.height;
    if (rc == 0) {
      std::vector<uint8_t> px((size_t)w * h * (grey ? 1 : 3));
      rc = jpegdec::decode_frame(d.data(), d.size(), px.data(), grey != 0, orient != 0);
      FILE* f = fopen(out, "wb");
      fwrite(px.data(), 1, px.size(), f);
      fclose(f);
    }
    printf("%d %d %d %d\n", rc, hd.orientation, w, h);
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
    d = tmp_path_factory.mktemp("jpegorient")
    src, exe = d / "drv.cpp", d / "drv"
    src.write_text(DRIVER_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)],
                   check=True)
    return str(exe), d


def decode(driver, files, grey=False, orient=True):
    """[(status, orientation, pixels or None)] of decode_frame over the files"""
    exe, d = driver
    lines = []
    for i, b in enumerate(files):
        (d / ("o%d.jpg" % i)).write_bytes(b)
        lines.append("%s %s %d %d" % (d / ("o%d.jpg" % i), d / ("o%d.raw" % i), grey, orient))
    rows = subprocess.run([exe], input="\n".join(lines) + "\n", check=True, capture_output=True, text=True).stdout.split("\n")
    res = []
    for i, row in enumerate(rows[:len(files)]):
        rc, o, w, h = (int(v) for v in row.split())
        shape = (h, w) if grey else (h, w, 3)
        res.append((rc, o, np.fromfile(str(d / ("o%d.raw" % i)), np.uint8).reshape(shape) if rc in (0, 1) else None))
    return res


# ---- Exif APP1 segments, built field by field so that each of cv2's rules can be probed ------------------------------
def app1(payload):
    return b"\xff\xe1" + struct.pack(">H", len(payload) + 2) + payload


def tiff(o, le=True, typ=3, count=1, ifd=8, before=0, bom=None, entries=None, cut=None):
    """A TIFF structure whose IFD0 holds `before` ASCII entries, then the orientation tag (value o, of type typ: 3 SHORT,
    4 LONG); entries: the entry count written (default: the real one); cut: keep only the first `cut` bytes."""
    e = "<" if le else ">"
    t = (bom or (b"II" if le else b"MM")) + struct.pack(e + "HI", 42, ifd) + b"\0" * (ifd - 8)
    ents = b"".join(struct.pack(e + "HHI", 0x010F + k, 2, 4) + b"abc\0" for k in range(before))
    ents += struct.pack(e + "HHII", 0x0112, 4, count, o) if typ == 4 else struct.pack(e + "HHIHH", 0x0112, typ, count, o, 0)
    t += struct.pack(e + "H", before + 1 if entries is None else entries) + ents + struct.pack(e + "I", 0)
    return t[:cut] if cut else t


def exif(o, **k):
    return app1(b"Exif\0\0" + tiff(o, **k))


def splice(data, seg, at=2):
    """the file with `seg` inserted at byte `at` (default: right after SOI)"""
    return data[:at] + seg + data[at:]


def tag(data, o, le=True):
    return splice(data, exif(o, le=le))


def cv2_decode(b, grey=False, ignore=False):
    flags = (cv2.IMREAD_GRAYSCALE if grey else cv2.IMREAD_COLOR) | (cv2.IMREAD_IGNORE_ORIENTATION if ignore else 0)
    return cv2.imdecode(np.frombuffer(b, np.uint8), flags)


def cv2_orientation(b):
    """the orientation cv2.imdecode applied to file b: which flip / transpose of the stored image it returned"""
    stored, got = cv2_decode(b, ignore=True), cv2_decode(b)
    t = cv2.transpose(stored)
    cands = {1: stored, 2: cv2.flip(stored, 1), 3: cv2.flip(stored, -1), 4: cv2.flip(stored, 0),
             5: t, 6: cv2.flip(t, 1), 7: cv2.flip(t, -1), 8: cv2.flip(t, 0)}
    hits = [o for o, c in cands.items() if c.shape == got.shape and (c == got).all()]
    assert len(hits) == 1, "the probe image must tell all eight orientations apart"
    return hits[0]


def frame(w, h, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    f = np.stack([(xx * 7 + yy * 3) % 256, (yy * 11 + 40) % 256, (xx * yy) % 256], -1) + rng.integers(0, 24, (h, w, 3))
    return np.clip(f, 0, 255).astype(np.uint8)


def base_file(w, h, sampling, seed=1, extra=()):
    f = frame(w, h, seed)
    if sampling == "grey":
        return imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), 90, None, extra)
    return imencode(f, 90, sampling, extra)


def _check_against_cv2(driver, files):
    for grey in (False, True):
        got = decode(driver, files, grey=grey)
        for i, (b, (rc, _, px)) in enumerate(zip(files, got)):
            want = cv2_decode(b, grey)
            assert rc == 0, "file %d: status %d" % (i, rc)
            assert px.shape == want.shape and (px == want).all(), "file %d (grey=%s) differs from cv2.imdecode" % (i, grey)


@pytest.mark.parametrize("size", [(1, 1), (1, 7), (7, 1), (17, 9), (481, 270)], ids=lambda s: "%dx%d" % s)
@pytest.mark.parametrize("sampling", list(SAMPLING) + ["grey"])
def test_every_orientation_and_byte_order_equals_cv2(driver, sampling, size):
    b = base_file(size[0], size[1], sampling, seed=size[0] * 31 + size[1])
    _check_against_cv2(driver, [tag(b, o, le) for le in (True, False) for o in range(1, 9)])


def test_restart_interval_file(driver):
    for extra in ([cv2.IMWRITE_JPEG_RST_INTERVAL, 1], [cv2.IMWRITE_JPEG_RST_INTERVAL, 7, cv2.IMWRITE_JPEG_OPTIMIZE, 1]):
        b = base_file(53, 37, "420", seed=5, extra=extra)
        _check_against_cv2(driver, [tag(b, o, le) for le in (True, False) for o in range(1, 9)])


def test_orient_false_is_the_stored_image(driver):
    b = base_file(17, 9, "420")
    files = [tag(b, o) for o in range(1, 9)]
    for grey in (False, True):
        for rc, o, px in decode(driver, files, grey=grey, orient=False):
            assert rc == 0 and o in range(1, 9)
            assert (px == cv2_decode(b, grey)).all()
    assert [o for _, o, _ in decode(driver, files)] == list(range(1, 9))


def _probes(b):
    """files probing each rule of cv2's Exif reader: name -> bytes"""
    xmp = app1(b"http://ns.adobe.com/xap/1.0/\0<x:xmpmeta/>")
    sof = b.index(b"\xff\xc0")
    eoi = len(b) - 2
    dup = lambda first: app1(b"Exif\0\0II" + struct.pack("<HIH", 42, 8, 2) + struct.pack("<HHIHH", 0x0112, 3, 1, first, 0)
                             + struct.pack("<HHIHH", 0x0112, 3, 1, 3, 0) + struct.pack("<I", 0))
    ifd1 = app1(b"Exif\0\0II" + struct.pack("<HIH", 42, 8, 1) + struct.pack("<HHIHH", 0x0128, 3, 1, 2, 0) + struct.pack("<I", 26)
                + struct.pack("<H", 1) + struct.pack("<HHIHH", 0x0112, 3, 1, 6, 0) + struct.pack("<I", 0))
    no_tag = app1(b"Exif\0\0" + tiff(6, before=1, entries=1))
    return {
        "xmp_before_exif": splice(b, xmp + exif(6)),
        "xmp_after_exif": splice(b, exif(6) + xmp),
        "not_exif_identifier": splice(b, app1(b"Exix\0\0" + tiff(6))),
        "identifier_without_nulls": splice(b, app1(b"Exif" + tiff(6))),
        "value_0": splice(b, exif(0)),
        "value_9": splice(b, exif(9)),
        "long_le": splice(b, exif(6, typ=4)),
        "long_be": splice(b, exif(6, typ=4, le=False)),
        "count_2": splice(b, exif(6, count=2)),
        "count_0": splice(b, exif(6, count=0)),
        "ifd0_at_20": splice(b, exif(6, ifd=20)),
        "ifd0_at_9": splice(b, exif(7, ifd=9, le=False)),
        "ifd0_past_the_end": splice(b, app1(b"Exif\0\0II*\0\xff\xff\xff\xff") + exif(3)),
        "entries_before_the_tag": splice(b, exif(6, before=3)),
        "tiff_cut_inside_ifd0": splice(b, exif(6, cut=14)),
        "tiff_cut_inside_the_value": splice(b, exif(6, cut=19)),
        "tiff_cut_after_the_value": splice(b, exif(6, cut=20)),
        "cut_before_the_tag_then_3": splice(b, exif(6, cut=14) + exif(3)),
        "cut_after_the_tag_then_3": splice(b, exif(6, cut=20) + exif(3)),
        "bom_XX_big_endian": splice(b, exif(6, le=False, bom=b"XX")),
        "bom_IM_big_endian": splice(b, exif(6, le=False, bom=b"IM")),
        "bom_XX_little_endian": splice(b, exif(6, bom=b"XX")),
        "bom_II_big_endian_body": splice(b, exif(6, le=False, bom=b"II")),
        "not_42": splice(b, app1(b"Exif\0\0II\x2b\0" + tiff(6)[4:])),
        "not_42_then_6": splice(b, app1(b"Exif\0\0II\x2b\0" + tiff(3)[4:]) + exif(6)),
        "after_dqt_before_sof": splice(b, exif(6), at=sof),
        "after_the_scan": splice(b, exif(6), at=eoi),
        "two_exif_6_3": splice(b, exif(6) + exif(3)),
        "two_exif_3_6": splice(b, exif(3) + exif(6)),
        "two_exif_0_6": splice(b, exif(0) + exif(6)),
        "empty_exif_then_6": splice(b, app1(b"Exif\0\0") + exif(6)),
        "exif_without_the_tag_then_3": splice(b, no_tag + exif(3)),
        "exif_with_no_entries_then_3": splice(b, exif(6, entries=0) + exif(3)),
        "entry_count_past_the_segment": splice(b, exif(6, entries=50)),
        "entry_count_past_the_segment_cut": splice(b, exif(6, entries=50, cut=22)),
        "tag_only_in_ifd1": splice(b, ifd1),
        "tag_twice_in_ifd0_6_3": splice(b, dup(6)),
        "tag_twice_in_ifd0_0_3": splice(b, dup(0)),
    }


def test_exif_rules_equal_cv2(driver):
    b = base_file(24, 16, "420", seed=3)
    probes = _probes(b)
    want = {name: cv2_orientation(f) for name, f in probes.items()}
    got = dict(zip(probes, decode(driver, list(probes.values()))))
    assert {name: o for name, (_, o, _) in got.items()} == want
    for name, f in probes.items():   # and the pixels, colour and grey
        rc, _, px = got[name]
        assert rc == 0 and (px == cv2_decode(f)).all(), name
    _check_against_cv2(driver, [probes[k] for k in ("long_le", "ifd0_at_9", "two_exif_3_6", "after_dqt_before_sof")])
    # the rules the probes above pin, as cv2 4.13.0 behaves
    assert want["xmp_before_exif"] == want["xmp_after_exif"] == 6
    assert want["not_exif_identifier"] == want["value_0"] == want["value_9"] == want["long_be"] == want["tiff_cut_inside_ifd0"] == 1
    assert want["long_le"] == want["count_2"] == want["ifd0_at_20"] == want["entries_before_the_tag"] == want["bom_XX_big_endian"] == 6
    assert want["after_dqt_before_sof"] == 6 and want["after_the_scan"] == 1


def test_library_reports_the_same_orientation(driver):
    from uwimageproc_b200 import _lib

    lib = _lib.load()
    b = base_file(24, 16, "420", seed=3)
    probes = _probes(b)
    for name, f in probes.items():
        buf = np.frombuffer(f, np.uint8)
        o = C.c_int(-1)
        assert lib.uwip_jpeg_orientation(buf.ctypes.data, buf.size, C.byref(o)) == 0, name
        assert o.value == cv2_orientation(f), name
    o = C.c_int(-1)
    bad = np.frombuffer(b"\xff\xd8\xff\xe1\x00", np.uint8)
    assert lib.uwip_jpeg_orientation(bad.ctypes.data, bad.size, C.byref(o)) == -1 and o.value == -1
