"""Pins oracle/uwip_oracle.py (pure numpy) to the golden vectors that oracle/make_golden.py produced
from cv2 4.13.0 and the reference's own Python files (SURVEY 8c).  CPU only."""
import json
import os

import numpy as np
import pytest

from oracle import uwip_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_k0_by_hand():
    # SURVEY 8c K0: 10x10 plane holding 0..99 once each, lo=2, hi=98
    p = np.arange(100, dtype=np.uint8).reshape(10, 10)
    low, high = O.percentile_bins(O.get_histogram(p), 10, 10, 2, 98)
    assert (low, high) == (1, 97)
    exp = np.clip(np.rint(np.maximum(p.astype(np.float32) - 1, 0) * np.float32(2.65625)), 0, 255)
    assert (O.img_channel_stretch(p, 2, 98) == exp.astype(np.uint8)).all()


def test_k1_stretch(kat, k1_plane):
    assert O.crc32(k1_plane) == kat["K1_plane_crc"] == "74187490"
    assert O.crc32(O.get_histogram(k1_plane)) == kat["K1_hist_crc"]
    for lo, hi in [(2, 98), (1, 99), (0, 100), (5, 50)]:
        g = kat["K1_stretch_%d_%d" % (lo, hi)]
        assert O.percentile_bins(O.get_histogram(k1_plane), 1920, 1080, lo, hi) == (g["low"], g["high"])
        assert O.crc32(O.img_channel_stretch(k1_plane, lo, hi)) == g["crc"]
    assert kat["K1_stretch_2_98"]["crc"] == "cb2c9c00" and kat["K1_stretch_1_99"]["crc"] == "e4f7741e"


def test_stretch_edge_cases(kat):
    const = np.full((40, 50), 77, np.uint8)
    out = O.img_channel_stretch(const, 2, 98)
    assert O.crc32(out) == kat["stretch_edge"]["const"]["out_crc"] and out.max() == 0
    c2 = const.copy()
    c2[0, :10] = 200
    out = O.img_channel_stretch(c2, 40, 60)
    assert O.crc32(out) == kat["stretch_edge"]["const_plus"]["out_crc"]


@pytest.mark.parametrize("tiles", [2, 4, 8, 16, 32])
def test_k1_clahe(kat, k1_plane, tiles):
    for clip in [0.0, 0.5, 2.0, 4.0, 24.5, 40.0]:
        assert O.crc32(O.clahe_apply(k1_plane, clip, tiles, tiles)) == kat["K1_clahe_%g_%d" % (clip, tiles)]


def test_blur3(kat, k1_plane):
    assert O.crc32(O.gaussian_blur3(k1_plane)) == kat["K1_blur3_crc"]


def test_odd_sizes(kat):
    for key, e in kat["odd"].items():
        W, H = map(int, key.split("x"))
        b = np.random.default_rng(H * 10007 + W).integers(0, 256, (H, W, 3), dtype=np.uint8)
        assert O.crc32(b) == e["bgr_crc"]
        hsv = O.bgr2hsv(b)
        assert O.crc32(hsv) == e["hsv_crc"]
        assert O.crc32(O.hsv2bgr(hsv, "cv2")) == e["hsv2bgr_crc"]
        assert O.crc32(O.bgr2ycrcb(b)) == e["ycrcb_crc"]
        for k, crc in e["clahe"].items():
            clip, tiles = k.split("_")
            got = O.clahe_apply(np.ascontiguousarray(b[..., 1]), float(clip), int(tiles), int(tiles))
            assert O.crc32(got) == crc, (key, k)


def test_k2_conversions(kat):
    bgr = np.random.default_rng(1).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    assert O.crc32(bgr) == kat["K2"]["bgr_crc"] == "9525bd44"
    hsv = O.bgr2hsv(bgr)
    assert O.crc32(hsv) == kat["K2"]["hsv_crc"] == "0ff6a727"
    assert O.crc32(O.hsv2bgr(hsv)) == kat["K2"]["hsv2bgr_crc"] == "46d8170b"
    assert O.crc32(O.bgr2ycrcb(bgr)) == kat["K2"]["ycrcb_crc"] == "249772e2"
    assert O.crc32(O.ycrcb2bgr(O.bgr2ycrcb(bgr))) == kat["K2"]["ycrcb2bgr_crc"]


def test_histretch_ycrcb_letters(kat):
    """Y, C, X letters (histretch.cpp:155-156, transformation[3]); goldens made with cv2 doing the conversions."""
    fr = O.synth_frame(0x5EED0001, 2, 479, 321)
    for letter in "YCX":
        assert O.crc32(O.histretch_frame(fr, letter, 2, 98)) == kat["histretch_ycrcb"][letter]
    assert O.crc32(O.histretch_frame(fr, "X", 2, 98, order="literal")) == kat["histretch_ycrcb"]["literal"]


def test_hls_conversions_and_letters(kat):
    """h, s, l letters (histretch.cpp:155-156, transformation[1]); goldens made with cv2 doing the conversions."""
    e = kat["hls"]
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8)
    body = trip.reshape(4096, 4096, 3)
    tail = trip[: 7 * ((1 << 24) // 7)].reshape(-1, 7, 3)
    assert O.crc32(O.bgr2hls(body)) == e["all_bgr2hls_body_crc"]
    assert O.crc32(O.bgr2hls(tail)) == e["all_bgr2hls_tail7_crc"]
    assert O.crc32(O.hls2bgr(body)) == e["all_hls2bgr_body_crc"]
    assert O.crc32(O.hls2bgr(tail)) == e["all_hls2bgr_tail7_crc"]
    bgr = np.random.default_rng(1).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    assert O.crc32(O.bgr2hls(bgr)) == e["K2_hls_crc"]
    assert O.crc32(O.hls2bgr(O.bgr2hls(bgr))) == e["K2_hls2bgr_crc"]
    for key, v in e["histretch"].items():
        W, H = map(int, key.split("x"))
        fr = O.synth_frame(0x5EED0001, 2, W, H)
        for letter in "hsl":
            assert O.crc32(O.histretch_frame(fr, letter, 2, 98)) == v[letter], (key, letter)
        assert O.crc32(O.histretch_frame(fr, "l", 2, 98, order="literal")) == v["literal"]


def test_lab_conversions_and_letters(kat):
    """L, a, b letters (histretch.cpp:155-156, transformation[2]); goldens made with cv2 doing the conversions."""
    e = kat["lab"]
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    assert O.crc32(O.bgr2lab(trip)) == e["all_bgr2lab_crc"]
    assert O.crc32(O.lab2bgr(trip)) == e["all_lab2bgr_crc"]
    assert O.crc32(O.bgr2lab(trip.reshape(-1, 3)[: 7 * 100000].reshape(-1, 7, 3))) == e["tail7_bgr2lab_crc"]
    for key, v in e["histretch"].items():
        W, H = map(int, key.split("x"))
        fr = O.synth_frame(0x5EED0001, 2, W, H)
        for letter in "Lab":
            assert O.crc32(O.histretch_frame(fr, letter, 2, 98)) == v[letter], (key, letter)
        assert O.crc32(O.histretch_frame(fr, "a", 2, 98, order="literal")) == v["literal"]


def test_calcblur_goldens(kat):
    """calcBlur (videostrip.cpp:170-184): goldens made by cv2 (cvtColor, Laplacian, meanStdDev); exact, doubles included."""
    e = kat["calcblur"]
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    assert O.crc32(O.bgr2gray(trip)) == e["all_bgr2gray_crc"]
    for key, v in e["frames"].items():
        fr = O.golden_frame(key)
        assert O.crc32(fr) == v["frame_crc"]
        for ap in (1, 3):
            lap = O.laplacian3_u8(O.bgr2gray(fr), ap)
            assert O.crc32(lap) == v["ap%d" % ap]["lap_crc"], (key, ap)
            assert O.mean_stddev_u8(lap) == (v["ap%d" % ap]["mean"], v["ap%d" % ap]["stdev"]), (key, ap)
            assert float(O.calc_blur(fr, ap)) == v["ap%d" % ap]["calcBlur"]


def test_exhaustive_colour_tables(kat):
    g = np.arange(1 << 24, dtype=np.uint32)
    allbgr = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    assert O.crc32(O.bgr2hsv(allbgr)) == kat["all_bgr2hsv_crc"]
    assert O.crc32(O.bgr2ycrcb(allbgr)) == kat["all_bgr2ycrcb_crc"]
    assert O.crc32(O.ycrcb2bgr(allbgr)) == kat["all_ycrcb2bgr_crc"]
    g = np.arange(180 * 65536, dtype=np.uint32)
    allhsv = np.stack([(g >> 16), (g >> 8) & 255, g & 255], axis=-1).astype(np.uint8).reshape(180 * 64, 1024, 3)
    assert O.crc32(O.hsv2bgr(allhsv, "cv2")) == kat["all_hsv2bgr_trunc_crc"]
    tail = allhsv.reshape(-1, 3)[: 31 * 380000].reshape(380000, 31, 3)
    assert O.crc32(O.hsv2bgr(tail, "cv2")) == kat["hsv2bgr_tail31_crc"]


def test_entropy_and_crowd(kat, k1_plane):
    assert abs(float(O.entropy_py(k1_plane)) - kat["entropy"]["K1"]) < 2e-6
    hist = np.array(kat["entropy"]["crowd_hist"], dtype=np.float32)
    p = hist / hist.sum(dtype=np.float32)
    e = -(p * np.log2(p + np.float32(1e-5))).sum(dtype=np.float32)
    assert abs(float(e) - kat["entropy"]["crowd"]) < 2e-6 and abs(kat["entropy"]["crowd"] - 6.1331363) < 1e-6
    z = np.load(os.path.join(GOLD, "crowd_crop.npz"))
    img = z["img"]
    assert abs(float(O.entropy_py(img)) - float(z["entropia"])) < 2e-6
    # the C++ flavour (float p, double log2) agrees with the float32 python flavour to ~1e-6
    assert abs(float(O.entropy_cpp(img)) - float(z["entropia"])) < 1e-5
    assert (O.clahe_apply(O.gaussian_blur3(img), 7, 4, 4) == z["clahe_4_7"]).all()
    assert (O.clahe_apply(img, 2.0, 8, 8) == z["clahe_8_2"]).all()


def test_dehaze_vs_literal_reference():
    z = np.load(os.path.join(GOLD, "dehaze_literal.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    assert len(names) == 5
    for name in names:
        fr = z[name + "/frame"]
        px = z[name + "/px"]   # the float maps are stored at these pixels
        st = {}
        out, out8 = O.bgdehaze_frame(fr, 15, st)
        assert np.allclose(st["B"], z[name + "/B"], rtol=0, atol=1e-15)
        # the (restored*255).astype(uint8) truncation (BGDehaze.py:75) makes the final map
        # discontinuous: a 1e-16 change can flip a byte of R8 and move `out` by ~1e-5
        assert np.abs(O.golden_pixels(out, px) - z[name + "/out"]).max() < 5e-5
        ref8 = O._sat_u8_from_rint(z[name + "/out"] * 255).astype(int)
        assert np.abs(O.golden_pixels(out8, px).astype(int) - ref8).max() <= 1
        if name + "/t_blue" in z.files:
            assert np.abs(O.transmission_map(O.normalize_frame(fr), 15) - z[name + "/tmap"]).max() == 0
            assert np.abs(O.golden_pixels(st["t_blue"], px) - z[name + "/t_blue"]).max() < 1e-12
            assert np.abs(O.golden_pixels(st["t_green"], px) - z[name + "/t_green"]).max() < 1e-12
            assert np.abs(O.golden_pixels(st["restored"], px) - z[name + "/restored"]).max() < 1e-12


def test_chain_goldens(kat):
    for key, e in kat["chain"].items():
        wh, f = key.split("_f")
        W, H = map(int, wh.split("x"))
        fr = O.synth_frame(0x5EED0004, int(f), W, H)
        assert O.crc32(fr) == e["synth_crc"]
        a = O.histretch_frame(fr, "V", 1, 99)
        assert O.crc32(a) == e["histretch_crc"]
        b = O.aclahe_frame(a, 2.0, 8, 8)
        assert O.crc32(b) == e["aclahe_crc"]


def test_histretch_literal_order_is_hsv_round_trip():
    fr = O.synth_frame(0x5EED0001, 0, 96, 64)
    lit = O.histretch_frame(fr, "V", 2, 98, order="literal")
    assert (lit == O.hsv2bgr(O.bgr2hsv(fr))).all()
    # default CLI letter 'r' is not recognised -> no-op (histretch.cpp:71, preprocessing.cpp:147)
    assert (O.histretch_frame(fr, "r") == fr).all()
    # 'R' maps to plane 0 which is BLUE in OpenCV's BGR order
    out = O.histretch_frame(fr, "R", 2, 98)
    assert (out[..., 0] == O.img_channel_stretch(fr[..., 0], 2, 98)).all() and (out[..., 1:] == fr[..., 1:]).all()


def test_parametros_aclahe_k4():
    """SURVEY K4: the oracle's restatement of ACLAHE.py:9-129 against what the reference's own ACLAHE.py / functions.py
    returned in the build container for crowd.png (tests/golden/crowd_full.npz, oracle/make_golden_aclahe.py)."""
    pytest.importorskip("scipy")
    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    img = z["img"]
    assert O.crc32(img) == json.load(open(os.path.join(GOLD, "kat.json")))["entropy"]["crowd_crc"]
    bs, cl, _ = O.parametros_aclahe(img, "as_committed")
    assert (bs, cl) == tuple(int(v) for v in z["as_committed"]) == (8, 0)
    bs, cl, ent = O.parametros_aclahe(img, "repaired")
    assert np.abs(ent - z["entropies"]).max() < 2e-6
    assert (bs, cl) == tuple(int(v) for v in z["repaired"]) == (4, 7)


def test_k3_background_light_full_fixture(kat):
    """SURVEY K3 on the CPU: the oracle's Background_light (first-index tie rule) on the full-resolution fixture frame shipped
    by oracle/make_golden_k3.py reproduces the B and indices make_golden.py stored from the reference's decoded image."""
    z = np.load(os.path.join(GOLD, "k3_pis_full.npz"))
    for key in z.files:
        name = key.split("/")[0]
        img = z[key]
        assert O.crc32(img) == kat["K3"][name]["decoded_crc"]
        B, idx = O.background_light(O.normalize_frame(img), 15, True)
        assert [float(v) for v in B] == kat["K3"][name]["B_first_index"]
        assert [int(i) for i in idx] == kat["K3"][name]["idx"]
