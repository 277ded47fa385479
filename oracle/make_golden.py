#!/usr/bin/env python3
"""Generate tests/golden/* from the REAL reference stack available in the build container.

TEST INFRASTRUCTURE ONLY (see oracle/uwip_oracle.py header).  Run in the container that has
/root/reference mounted:

    python oracle/make_golden.py

It executes
  * cv2 4.13.0 (the only executable OpenCV in this image) for every OpenCV call on the path,
  * the reference's own Python files imported unmodified from /root/reference
    (modules/bgdehaze/BGDehaze.py, guidedfilter.py; modules/aclahe/python/functions.py with a
    matplotlib stub),
and stores small input/output vectors.  The only intervention in the reference code is the
arg-min tie rule of Background_light (BGDehaze.py:24 uses an unstable argsort whose choice among
ties is machine dependent, SURVEY 8a-D1): the oracle's first-index rule is injected, and the
literal (machine-dependent) B is stored next to it for information.

The GPU box has no /root/reference; the tests only read the files written here.
"""
import json
import os
import sys
import types

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = "/root/reference/modules"

import cv2  # noqa: E402
import numpy as np  # noqa: E402

from oracle import uwip_oracle as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
os.makedirs(GOLD, exist_ok=True)
assert cv2.useOptimized(), "oracle must run with cv2 optimisations on (SURVEY 8c)"


DEHAZE_PX = 3072   # pixels per bgdehaze case at which its float maps are stored: keeps dehaze_literal.npz under 1 MB


def sample_dehaze_case(case):
    """One case of dehaze_literal.npz with its full-size float maps (out, t_blue, t_green, restored) reduced to the pixels
    listed in `px`: DEHAZE_PX flat indices drawn without replacement from a fixed seed, ascending.  frame, B and tmap stay whole."""
    H, W = case["frame"].shape[:2]
    px = np.sort(np.random.default_rng(0x5EED).choice(H * W, DEHAZE_PX, replace=False)).astype(np.int32)
    out = dict(case, px=px)
    for k in ("out", "t_blue", "t_green", "restored"):
        if k in case:
            out[k] = O.golden_pixels(case[k], px)
    return out


def k1_plane():
    rng = np.random.default_rng(0)
    mu = rng.uniform(60, 180)
    sd = rng.uniform(10, 60)
    return np.clip(rng.normal(mu, sd, (1080, 1920)), 0, 255).astype(np.uint8)


def cv_stretch(ch, lo, hi):
    """imgChannelStretch through cv2 calls (calcHist, add, convertTo)."""
    hist = cv2.calcHist([ch], [0], None, [256], [0, 256]).ravel()
    low, high = O.percentile_bins(hist, ch.shape[1], ch.shape[0], lo, hi)
    b = -float(low)
    with np.errstate(divide="ignore"):
        m = float(np.float32(np.float64(255.0) / np.float64(high - low))) if high != low else float("inf")
    y = cv2.add(ch, b)
    z = cv2.convertScaleAbs(y, alpha=m) if np.isfinite(m) else None
    return low, high, y, z


def hls_goldens(kat):
    """HLS letters h, s, l of histretch (transformation[1], histretch.cpp:155-156): cv2 does every conversion."""
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8)
    body = trip.reshape(4096, 4096, 3)  # W % 8 == 0: every pixel through the vector body
    tail = trip[: 7 * ((1 << 24) // 7)].reshape(-1, 7, 3)  # W < 8: every pixel through the scalar tail
    hls = {
        "all_bgr2hls_body_crc": O.crc32(cv2.cvtColor(body, cv2.COLOR_BGR2HLS)),
        "all_bgr2hls_tail7_crc": O.crc32(cv2.cvtColor(tail, cv2.COLOR_BGR2HLS)),
        # the same 2^24 triples read as (H, L, S), H up to 255 (a stretched H plane can hold that)
        "all_hls2bgr_body_crc": O.crc32(cv2.cvtColor(body, cv2.COLOR_HLS2BGR)),
        "all_hls2bgr_tail7_crc": O.crc32(cv2.cvtColor(tail, cv2.COLOR_HLS2BGR)),
    }
    letters = {}
    for (W, H) in ((479, 321), (640, 360)):
        fr = O.synth_frame(0x5EED0001, 2, W, H)
        e = {}
        for letter, ch in (("h", 0), ("s", 1), ("l", 2)):
            d = cv2.cvtColor(fr, cv2.COLOR_BGR2HLS)
            d[..., ch] = O.img_channel_stretch(np.ascontiguousarray(d[..., ch]), 2, 98)
            e[letter] = O.crc32(cv2.cvtColor(d, cv2.COLOR_HLS2BGR))
        e["literal"] = O.crc32(cv2.cvtColor(cv2.cvtColor(fr, cv2.COLOR_BGR2HLS), cv2.COLOR_HLS2BGR))
        letters["%dx%d" % (W, H)] = e
    hls["histretch"] = letters
    bgr = np.random.default_rng(1).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    hls["K2_hls_crc"] = O.crc32(cv2.cvtColor(bgr, cv2.COLOR_BGR2HLS))
    hls["K2_hls2bgr_crc"] = O.crc32(cv2.cvtColor(cv2.cvtColor(bgr, cv2.COLOR_BGR2HLS), cv2.COLOR_HLS2BGR))
    kat["hls"] = hls


def blur_goldens(kat):
    """calcBlur (videostrip.cpp:170-184) with cv2 doing cvtColor, Laplacian and meanStdDev."""
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    out = {"all_bgr2gray_crc": O.crc32(cv2.cvtColor(trip, cv2.COLOR_BGR2GRAY)), "frames": {}}
    cases = [("synth", 0x5EED0002, 1, 1920, 1080), ("synth", 0x5EED0002, 3, 479, 321), ("rand", 11, 0, 333, 100),
             ("rand", 12, 0, 1, 1), ("rand", 13, 0, 5, 1), ("rand", 14, 0, 1, 7), ("rand", 15, 0, 31, 2), ("synth", 0x5EED0004, 0, 3840, 2160)]
    for kind, seed, f, W, H in cases:
        fr = O.synth_frame(seed, f, W, H) if kind == "synth" else np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
        grey = cv2.cvtColor(fr, cv2.COLOR_BGR2GRAY)
        e = {"frame_crc": O.crc32(fr)}
        for ap in (1, 3):
            lap = cv2.Laplacian(grey, cv2.CV_8U, ksize=ap)  # aperture 3 is what videostrip.cpp:175 passes as CV_16S
            m, sd = cv2.meanStdDev(lap)
            e["ap%d" % ap] = {"lap_crc": O.crc32(lap), "mean": float(m[0, 0]), "stdev": float(sd[0, 0]),
                              "calcBlur": float(np.float32(sd[0, 0]))}
        out["frames"]["%s_%x_%d_%dx%d" % (kind, seed, f, W, H)] = e
    kat["calcblur"] = out


def lab_goldens(kat):
    """Lab letters L, a, b of histretch (transformation[2], histretch.cpp:155-156): cv2 does every conversion."""
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    lab = {
        "all_bgr2lab_crc": O.crc32(cv2.cvtColor(trip, cv2.COLOR_BGR2Lab)),
        "all_lab2bgr_crc": O.crc32(cv2.cvtColor(trip, cv2.COLOR_Lab2BGR)),  # the same triples read as (L, a, b)
        "tail7_bgr2lab_crc": O.crc32(cv2.cvtColor(trip.reshape(-1, 3)[: 7 * 100000].reshape(-1, 7, 3), cv2.COLOR_BGR2Lab)),
    }
    letters = {}
    for (W, H) in ((479, 321), (640, 360)):
        fr = O.synth_frame(0x5EED0001, 2, W, H)
        e = {}
        for letter, ch in (("L", 0), ("a", 1), ("b", 2)):
            d = cv2.cvtColor(fr, cv2.COLOR_BGR2Lab)
            d[..., ch] = O.img_channel_stretch(np.ascontiguousarray(d[..., ch]), 2, 98)
            e[letter] = O.crc32(cv2.cvtColor(d, cv2.COLOR_Lab2BGR))
        e["literal"] = O.crc32(cv2.cvtColor(cv2.cvtColor(fr, cv2.COLOR_BGR2Lab), cv2.COLOR_Lab2BGR))
        letters["%dx%d" % (W, H)] = e
    lab["histretch"] = letters
    kat["lab"] = lab


def main():
    kat = {"cv2": cv2.__version__, "numpy": np.__version__}

    # ---- K1 family ------------------------------------------------------------------
    ch = k1_plane()
    kat["K1_plane_crc"] = O.crc32(ch)
    kat["K1_hist_crc"] = O.crc32(cv2.calcHist([ch], [0], None, [256], [0, 256]).ravel())
    for lo, hi in [(2, 98), (1, 99), (0, 100), (5, 50)]:
        low, high, y, z = cv_stretch(ch, lo, hi)
        kat["K1_stretch_%d_%d" % (lo, hi)] = {"low": low, "high": high, "crc": O.crc32(z)}
    for clip in [0.0, 0.5, 2.0, 4.0, 24.5, 40.0]:
        for tiles in [2, 4, 8, 16, 32]:
            out = cv2.createCLAHE(clip, (tiles, tiles)).apply(ch)
            kat["K1_clahe_%g_%d" % (clip, tiles)] = O.crc32(out)
    kat["K1_blur3_crc"] = O.crc32(cv2.GaussianBlur(ch, (3, 3), 0))

    # ---- odd sizes (CLAHE pad branch, HSV tail rounding) ------------------------------
    odd = {}
    for (H, W) in [(479, 641), (33, 33), (600, 800), (7, 100), (135, 240), (100, 1000)]:
        b = np.random.default_rng(H * 10007 + W).integers(0, 256, (H, W, 3), dtype=np.uint8)
        hsv = cv2.cvtColor(b, cv2.COLOR_BGR2HSV)
        e = {
            "bgr_crc": O.crc32(b),
            "hsv_crc": O.crc32(hsv),
            "hsv2bgr_crc": O.crc32(cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)),
            "ycrcb_crc": O.crc32(cv2.cvtColor(b, cv2.COLOR_BGR2YCrCb)),
            "clahe": {},
        }
        for tiles in [2, 4, 8, 16]:
            if tiles > min(H, W):
                continue
            for clip in [0.0, 2.0, 40.0]:
                e["clahe"]["%g_%d" % (clip, tiles)] = O.crc32(
                    cv2.createCLAHE(clip, (tiles, tiles)).apply(b[..., 1].copy())
                )
        odd["%dx%d" % (W, H)] = e
    kat["odd"] = odd

    # ---- K2: colour conversions on random 1080p ---------------------------------------
    bgr = np.random.default_rng(1).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    hsv = cv2.cvtColor(bgr, cv2.COLOR_BGR2HSV)
    kat["K2"] = {
        "bgr_crc": O.crc32(bgr),
        "hsv_crc": O.crc32(hsv),
        "hsv2bgr_crc": O.crc32(cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)),
        "ycrcb_crc": O.crc32(cv2.cvtColor(bgr, cv2.COLOR_BGR2YCrCb)),
        "ycrcb2bgr_crc": O.crc32(cv2.cvtColor(cv2.cvtColor(bgr, cv2.COLOR_BGR2YCrCb), cv2.COLOR_YCrCb2BGR)),
    }

    # ---- exhaustive tables ------------------------------------------------------------
    # all 2^24 BGR triples -> HSV, YCrCb ; all 180*256*256 HSV triples -> BGR (trunc body: W%32==0)
    g = np.arange(1 << 24, dtype=np.uint32)
    allbgr = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)
    kat["all_bgr2hsv_crc"] = O.crc32(cv2.cvtColor(allbgr, cv2.COLOR_BGR2HSV))
    kat["all_bgr2ycrcb_crc"] = O.crc32(cv2.cvtColor(allbgr, cv2.COLOR_BGR2YCrCb))
    kat["all_ycrcb2bgr_crc"] = O.crc32(cv2.cvtColor(allbgr, cv2.COLOR_YCrCb2BGR))  # the same 2^24 triples read as Y,Cr,Cb
    g = np.arange(180 * 65536, dtype=np.uint32)
    allhsv = np.stack([(g >> 16), (g >> 8) & 255, g & 255], axis=-1).astype(np.uint8).reshape(180 * 64, 1024, 3)
    kat["all_hsv2bgr_trunc_crc"] = O.crc32(cv2.cvtColor(allhsv, cv2.COLOR_HSV2BGR))
    # width 31 (<32): every pixel goes through the scalar tail -> rint everywhere
    tail = allhsv.reshape(-1, 3)[: 31 * 380000].reshape(380000, 31, 3)
    kat["hsv2bgr_tail31_crc"] = O.crc32(cv2.cvtColor(tail, cv2.COLOR_HSV2BGR))

    # ---- stretch edge cases -----------------------------------------------------------
    edge = {}
    const = np.full((40, 50), 77, np.uint8)
    low, high, y, z = cv_stretch(const, 2, 98)
    # high == low -> m = inf: run the real convertTo with an infinite scale
    zinf = cv2.convertScaleAbs(y, alpha=float("inf"))
    y2 = const.copy()
    y2[0, :10] = 200  # a few pixels above the single dominant bin
    low2, high2, yy, _ = cv_stretch(y2, 40, 60)
    zinf2 = cv2.convertScaleAbs(yy, alpha=float("inf"))
    edge["const"] = {"low": low, "high": high, "out_crc": O.crc32(zinf), "out_max": int(zinf.max())}
    edge["const_plus"] = {"low": low2, "high": high2, "out_crc": O.crc32(zinf2), "out_max": int(zinf2.max())}
    kat["stretch_edge"] = edge
    # NOTE convertScaleAbs == |x| then saturate; identical to convertTo for non-negative input.
    # Cross-check convertTo semantics through numpy-visible API: Mat *= m is convertTo(-1, m).
    for lo, hi in [(2, 98), (1, 99)]:
        low, high, y, z = cv_stretch(ch, lo, hi)
        m = float(np.float32(255.0 / (high - low)))
        alt = cv2.multiply(y, np.array([m]))  # NOT equivalent in general (SURVEY A.1) - recorded only
        kat["K1_multiply_differs_%d_%d" % (lo, hi)] = int((alt != z).sum())

    # ---- aclahe python reference functions --------------------------------------------
    sys.modules.setdefault("matplotlib", types.ModuleType("matplotlib"))
    sys.modules.setdefault("matplotlib.pyplot", types.ModuleType("matplotlib.pyplot"))
    sys.path.insert(0, os.path.join(REF, "aclahe", "python"))
    import functions as AF  # the reference's functions.py

    ent = {"K1": float(AF.Entropia(ch))}
    crowd = cv2.imread(os.path.join(REF, "aclahe", "python", "crowd.png"), 0)
    ent["crowd_shape"] = list(crowd.shape)
    ent["crowd_crc"] = O.crc32(crowd)
    ent["crowd"] = float(AF.Entropia(crowd))
    ent["crowd_hist"] = [int(v) for v in np.bincount(crowd.ravel(), minlength=256)]
    blur = cv2.GaussianBlur(crowd, (3, 3), 0)
    ent["crowd_blur_crc"] = O.crc32(blur)
    sweep = {}
    for bs in [2, 4, 8, 16, 32]:
        for cl in [0.0, 0.5, 2.0, 7.0, 24.5]:
            sweep["%d_%g" % (bs, cl)] = float(AF.Entropia(AF.CLAHE(blur, bs, cl)))
    ent["crowd_sweep"] = sweep
    kat["entropy"] = ent
    # a 200x152 crop of crowd.png travels as the small input fixture for the entropy/CLAHE tests
    crop = np.ascontiguousarray(crowd[200:352, 300:500])
    np.savez_compressed(
        os.path.join(GOLD, "crowd_crop.npz"),
        img=crop,
        entropia=np.float32(AF.Entropia(crop)),
        clahe_4_7=AF.CLAHE(cv2.GaussianBlur(crop, (3, 3), 0), 4, 7),
        clahe_8_2=AF.CLAHE(crop, 8, 2.0),
    )

    # ---- bgdehaze: literal reference on small frames ----------------------------------
    sys.path.insert(0, os.path.join(REF, "bgdehaze"))
    import BGDehaze as RB  # the reference's BGDehaze.py, unmodified

    literal_BL = RB.Background_light
    cases = {}
    frames = {
        "synth_128x96": O.synth_frame(0x5EED0003, 0, 128, 96),
        "synth_112x88": O.synth_frame(0x5EED0003, 1, 112, 88),
    }
    k3 = {}
    for name in ["BUL_T1A_0028", "BUL_T1A_0209", "PIS_T1A_259"]:
        img = cv2.imread(os.path.join(REF, "bgdehaze", "img", name + ".jpg"))
        normI = O.normalize_frame(img)
        B, idx = O.background_light(normI, 15, True)
        k3[name] = {"decoded_crc": O.crc32(img), "B_first_index": [float(v) for v in B], "idx": list(idx)}
        # a 144x82 area-resampled copy keeps the underwater colour cast of the real fixture
        small = cv2.resize(img, (144, 82), interpolation=cv2.INTER_AREA)
        frames["fixture_%s_144x82" % name] = small
    kat["K3"] = k3

    for name, fr in frames.items():
        normI = O.normalize_frame(fr)
        B_lit = literal_BL(normI, 15)
        RB.Background_light = lambda n, w=15: O.background_light(n, w)
        try:
            B = RB.Background_light(normI, 15)
            tmap = RB.transmission_map(normI, 15)
            tb, tg = RB.refined_t(normI)
            nb, ng = RB.dehazed_BG(normI, 15)
            restored = RB.RC_correction(normI, 15)
            out = RB.adaptiveExp_map(normI, 15)
        finally:
            RB.Background_light = literal_BL
        assert not np.isnan(out).any(), name
        cases[name] = dict(frame=fr, B=B, B_literal_unstable=B_lit, out=out)
        if name == "synth_128x96":  # full stage dump for one case only (keeps the fixture small)
            cases[name].update(tmap=tmap, t_blue=tb, t_green=tg, restored=restored)
        mine = O.bgdehaze_frame(fr, 15)[0]
        print("dehaze", name, "oracle vs literal reference maxabs", np.abs(mine - out).max())
        cases[name] = sample_dehaze_case(cases[name])
    flat = {}
    for name, d in cases.items():
        for k, v in d.items():
            flat[name + "/" + k] = v
    np.savez_compressed(os.path.join(GOLD, "dehaze_literal.npz"), **flat)

    # ---- chain CRCs on synthetic frames (oracle output, pinned so GPU and CPU boxes agree) ----
    chain = {}
    for (W, H, f) in [(160, 120, 0), (480, 270, 3)]:
        fr = O.synth_frame(0x5EED0004, f, W, H)
        a = O.histretch_frame(fr, "V", 1, 99)
        a_cv = cv2.cvtColor(fr, cv2.COLOR_BGR2HSV)
        a_cv[..., 2] = cv_stretch(np.ascontiguousarray(a_cv[..., 2]), 1, 99)[3]
        a_cv = cv2.cvtColor(a_cv, cv2.COLOR_HSV2BGR)
        assert (a == a_cv).all()
        b_cv = cv2.cvtColor(a_cv, cv2.COLOR_BGR2HSV)
        b_cv[..., 2] = cv2.createCLAHE(2.0, (8, 8)).apply(np.ascontiguousarray(b_cv[..., 2]))
        b_cv = cv2.cvtColor(b_cv, cv2.COLOR_HSV2BGR)
        assert (O.aclahe_frame(a, 2.0, 8, 8) == b_cv).all()
        chain["%dx%d_f%d" % (W, H, f)] = {
            "synth_crc": O.crc32(fr),
            "histretch_crc": O.crc32(a_cv),
            "aclahe_crc": O.crc32(b_cv),
            "chain_crc": O.crc32(O.bgdehaze_frame(b_cv, 15)[1]),
        }
    kat["chain"] = chain
    # ---- histretch on the YCrCb letters with cv2 doing the conversions (histretch.cpp:232-240, intended order)
    ycx = {}
    fr = O.synth_frame(0x5EED0001, 2, 479, 321)
    for letter, ch in (("Y", 0), ("C", 1), ("X", 2)):
        d = cv2.cvtColor(fr, cv2.COLOR_BGR2YCrCb)
        d[..., ch] = O.img_channel_stretch(np.ascontiguousarray(d[..., ch]), 2, 98)
        ycx[letter] = O.crc32(cv2.cvtColor(d, cv2.COLOR_YCrCb2BGR))
    ycx["literal"] = O.crc32(cv2.cvtColor(cv2.cvtColor(fr, cv2.COLOR_BGR2YCrCb), cv2.COLOR_YCrCb2BGR))
    kat["histretch_ycrcb"] = ycx
    kat["synth_1080p_f0_crc"] = O.crc32(O.synth_frame(0x5EED0003, 0, 1920, 1080))
    hls_goldens(kat)
    blur_goldens(kat)
    lab_goldens(kat)

    with open(os.path.join(GOLD, "kat.json"), "w") as f:
        json.dump(kat, f, indent=1, sort_keys=True)
    print("wrote", GOLD)


if __name__ == "__main__":
    if any(a.startswith("--only-") for a in sys.argv):  # add vectors to an existing kat.json without re-running the rest
        path = os.path.join(GOLD, "kat.json")
        with open(path) as f:
            kat = json.load(f)
        if "--only-hls" in sys.argv:
            hls_goldens(kat)
        if "--only-blur" in sys.argv:
            blur_goldens(kat)
        if "--only-lab" in sys.argv:
            lab_goldens(kat)
        with open(path, "w") as f:
            json.dump(kat, f, indent=1, sort_keys=True)
    else:
        main()
