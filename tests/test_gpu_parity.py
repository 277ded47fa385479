"""Parity of the CUDA path (through the C ABI, libuwip.so) against the oracle and the golden vectors.
Bit-exact for histogram / percentile / LUT / colour / CLAHE work; stated tolerances for bgdehaze."""
import os

import numpy as np
import pytest

from oracle import uwip_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def rand_frame(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


# ---- histretch ---------------------------------------------------------------------------------
def test_histogram_and_stretch_k1(ctx, kat, k1_plane):
    hist = ctx.histogram(k1_plane)
    assert hist.dtype == np.float32 and (hist == O.get_histogram(k1_plane)).all()
    assert O.crc32(hist) == kat["K1_hist_crc"]
    for lo, hi in [(2, 98), (1, 99), (0, 100), (5, 50)]:
        out, low, high = ctx.channel_stretch(k1_plane, lo, hi, return_bins=True)
        g = kat["K1_stretch_%d_%d" % (lo, hi)]
        assert (low, high) == (g["low"], g["high"])
        assert O.crc32(out) == g["crc"]


def test_stretch_edge_cases(ctx, kat):
    const = np.full((40, 50), 77, np.uint8)
    assert O.crc32(ctx.channel_stretch(const, 2, 98)) == kat["stretch_edge"]["const"]["out_crc"]
    c2 = const.copy()
    c2[0, :10] = 200
    assert O.crc32(ctx.channel_stretch(c2, 40, 60)) == kat["stretch_edge"]["const_plus"]["out_crc"]
    # ragged sizes, pitched input
    for (h, w) in [(1, 1), (3, 5), (17, 31), (100, 333)]:
        p = np.random.default_rng(h * w).integers(0, 256, (h, w + 7), dtype=np.uint8)[:, :w]
        assert (ctx.channel_stretch(p, 2, 98) == O.img_channel_stretch(np.ascontiguousarray(p), 2, 98)).all()
        assert (ctx.histogram(p) == O.get_histogram(np.ascontiguousarray(p))).all()
    import uwimageproc_b200 as u

    with pytest.raises(u.UwipError):
        ctx.channel_stretch(const, 50, 50)
    with pytest.raises(u.UwipError):
        ctx.channel_stretch(const, -1, 50)


@pytest.mark.parametrize("shape", [(1080, 1920), (135, 240), (64, 33), (50, 100), (479, 641)])
def test_histretch_frame(ctx, shape):
    h, w = shape
    for fr in (O.synth_frame(0x5EED0001, 2, w, h), rand_frame(h + w, h, w)):
        for ch in ["V", "S", "H", "R", "G", "B", "HV", "VS", "xV", "r", "Y", "C", "X", "YV", "CX", "h", "s", "l", "hl", "sV", "L", "a", "b", "La", "bV"]:
            got = ctx.histretch(fr, ch, 2, 98)
            assert (got == O.histretch_frame(fr, ch, 2, 98)).all(), (shape, ch)
        got = ctx.histretch(fr, "V", 1, 99, order="literal")
        assert (got == O.histretch_frame(fr, "V", 1, 99, order="literal")).all()
        got = ctx.histretch(fr, "Y", 1, 99, order="literal")
        assert (got == O.histretch_frame(fr, "Y", 1, 99, order="literal")).all()
        got = ctx.histretch(fr, "s", 1, 99, order="literal")
        assert (got == O.histretch_frame(fr, "s", 1, 99, order="literal")).all()
        assert (ctx.histretch(fr, "l", 1, 99, hsv_round="rint") == O.histretch_frame(fr, "l", 1, 99, hsv_rounding="rint")).all()
        for mode in ["trunc", "rint"]:
            assert (ctx.histretch(fr, "V", 1, 99, hsv_round=mode) == O.histretch_frame(fr, "V", 1, 99, hsv_rounding=mode)).all()


def test_histretch_hls_all_triples(ctx):
    """Every BGR triple through BGR2HLS -> HLS2BGR (literal order) and through the 'l' (S plane) stretch, on a width
    that is all vector body (4096) and one that is all scalar tail (7): the two cv2 code paths of appendix A."""
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8)
    for fr in (trip.reshape(4096, 4096, 3), trip[: 7 * 300000].reshape(-1, 7, 3)):
        assert (ctx.histretch(fr, "h", 2, 98, order="literal") == O.histretch_frame(fr, "h", 2, 98, order="literal")).all()
        for letter in "hsl":
            assert (ctx.histretch(fr, letter, 5, 90) == O.histretch_frame(fr, letter, 5, 90)).all(), letter


def test_calcblur(ctx, kat):
    """calcBlur (videostrip.cpp:170-184): 8-bit Laplacian bit-exact, mean / stdev equal to cv::meanStdDev's doubles."""
    for key, v in kat["calcblur"]["frames"].items():
        fr = O.golden_frame(key)
        for ap in (1, 3):
            sd, (mean, std), lap = ctx.calc_blur(fr, return_all=True, aperture=ap)
            e = v["ap%d" % ap]
            assert O.crc32(lap) == e["lap_crc"], (key, ap)
            assert (mean, std) == (e["mean"], e["stdev"]), (key, ap)
            assert float(sd) == e["calcBlur"] == float(O.calc_blur(fr, ap))
    # pitched input, ragged width (strip of 240 columns + 1) and the batch entry point on device memory
    big = rand_frame(77, 70, 250)
    view = big[3:67, 5:246]
    assert float(ctx.calc_blur(view)) == float(O.calc_blur(np.ascontiguousarray(view)))
    import uwimageproc_b200 as u

    with pytest.raises(u.UwipError):
        ctx.calc_blur(view, aperture=5)


def test_calcblur_batch_4k(ctx):
    torch = pytest.importorskip("torch")
    n, W, H = 6, 3840, 2160
    d = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, 2), dtype=torch.float64, device="cuda")
    ctx.synth_dev(d.data_ptr(), 0x5EED0004, 0, n, W, H)
    ctx.calc_blur_dev(d.data_ptr(), n, W, H, out.data_ptr())
    ctx.synchronize()
    got = out.cpu().numpy()
    for f in (0, n - 1):
        fr = d[f].cpu().numpy()
        assert tuple(got[f]) == O.mean_stddev_u8(O.laplacian3_u8(O.bgr2gray(fr)))


def test_histretch_lab_all_triples(ctx):
    """Every BGR triple through BGR2Lab -> Lab2BGR (literal order) and through the L, a, b stretches (SURVEY 8f N2)."""
    g = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(g & 255), (g >> 8) & 255, (g >> 16) & 255], axis=-1).astype(np.uint8)
    for fr in (trip.reshape(4096, 4096, 3), trip[: 7 * 300000].reshape(-1, 7, 3)):
        assert (ctx.histretch(fr, "L", 2, 98, order="literal") == O.histretch_frame(fr, "L", 2, 98, order="literal")).all()
        for letter in "Lab":
            assert (ctx.histretch(fr, letter, 5, 90) == O.histretch_frame(fr, letter, 5, 90)).all(), letter


def test_histretch_every_letter_of_the_cli(ctx):
    """-c=RGBHSVhslLabYCX (histretch.cpp:68-74): all fifteen letters in one call, plus unknown ones that are skipped."""
    fr = O.synth_frame(0x5EED0001, 5, 641, 479)
    letters = "RGBHSVhslLabYCX"
    assert (ctx.histretch(fr, letters, 2, 98) == O.histretch_frame(fr, letters, 2, 98)).all()
    assert (ctx.histretch(fr, "r?Lz", 2, 98) == O.histretch_frame(fr, "L", 2, 98)).all()


# ---- aclahe --------------------------------------------------------------------------------------
@pytest.mark.parametrize("tiles", [2, 4, 8, 16, 32])
def test_clahe_k1(ctx, kat, k1_plane, tiles):
    for clip in [0.0, 0.5, 2.0, 4.0, 24.5, 40.0]:
        assert O.crc32(ctx.clahe(k1_plane, clip, (tiles, tiles))) == kat["K1_clahe_%g_%d" % (clip, tiles)]


def test_clahe_odd_sizes(ctx, kat):
    for key, e in kat["odd"].items():
        W, H = map(int, key.split("x"))
        b = np.random.default_rng(H * 10007 + W).integers(0, 256, (H, W, 3), dtype=np.uint8)
        for k, crc in e["clahe"].items():
            clip, tiles = k.split("_")
            got = ctx.clahe(np.ascontiguousarray(b[..., 1]), float(clip), (int(tiles), int(tiles)))
            assert O.crc32(got) == crc, (key, k)
    p = np.random.default_rng(5).integers(0, 256, (90, 160), dtype=np.uint8)
    assert (ctx.clahe(p, 3.0, (4, 2)) == O.clahe_apply(p, 3.0, 4, 2)).all()  # non-square grid


@pytest.mark.parametrize("shape", [(1080, 1920), (270, 480), (100, 100), (479, 641)])
def test_aclahe_frame(ctx, shape):
    h, w = shape
    for fr in (O.synth_frame(0x5EED0002, 1, w, h), rand_frame(h * 3 + w, h, w)):
        for clip in [0.0, 2.0, 40.0]:
            assert (ctx.aclahe(fr, clip, (8, 8)) == O.aclahe_frame(fr, clip, 8, 8)).all(), (shape, clip)


def test_entropy_blur_sweep(ctx, kat, k1_plane):
    assert abs(float(ctx.entropy(k1_plane, "py")) - kat["entropy"]["K1"]) < 1e-5
    assert abs(float(ctx.entropy(k1_plane, "cpp")) - float(O.entropy_cpp(k1_plane))) < 1e-5
    assert O.crc32(ctx.gaussian_blur3(k1_plane)) == kat["K1_blur3_crc"]
    z = np.load(os.path.join(GOLD, "crowd_crop.npz"))
    img = z["img"]
    assert abs(float(ctx.entropy(img, "py")) - float(z["entropia"])) < 1e-5
    assert (ctx.clahe(ctx.gaussian_blur3(img), 7, (4, 4)) == z["clahe_4_7"]).all()
    clips = np.arange(0, 25.5, 0.5)
    for tiles in [2, 8]:
        got = ctx.clahe_entropy_sweep(img, tiles, clips, "py")
        want = np.array([O.entropy_py(O.clahe_apply(img, c, tiles, tiles)) for c in clips])
        assert np.abs(got - want).max() < 1e-5


# ---- synthetic generator ---------------------------------------------------------------------------
def test_synth_matches_oracle(ctx, kat):
    import torch

    for (w, h, first, n) in [(1920, 1080, 0, 1), (240, 135, 3, 4), (97, 61, 10, 2)]:
        buf = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        ctx.synth_dev(buf, 0x5EED0003, first, n, w, h)
        ctx.synchronize()
        got = buf.cpu().numpy()
        for i in range(n):
            assert (got[i] == O.synth_frame(0x5EED0003, first + i, w, h)).all()
        import uwimageproc_b200 as u

        assert (ctx.checksum_dev(buf, n, w, h) == u.host_checksum(got)).all()
    assert O.crc32(O.synth_frame(0x5EED0003, 0, 1920, 1080)) == kat["synth_1080p_f0_crc"]


# ---- bgdehaze ------------------------------------------------------------------------------------------
# Tolerance of the FINAL float map: 1 LSB of the 8-bit output (1/255), the same bar as the bytes.  The
# continuous stages before it are held to 1e-5; adaptiveExp_map itself is discontinuous in them:
# `(restored*255).astype(uint8)` (BGDehaze.py:75) truncates, and the red channel of `restored` is
# (k' - rmin)/(rmax - rmin) mathematically, i.e. EXACTLY on an integer boundary times 1/255 for every pixel when
# rmax - rmin = 255 - which side it falls on is decided by the last bits of mean(Jb), mean(Jg) (a numpy pairwise
# sum in the reference).  One flipped byte at the extreme of the YCrCb images moves the joint min-max
# normalisation by one level (0.3-0.4 %), which stays inside 1 LSB of the output but not inside 2e-4.
OUT_TOL = 1.0 / 255.0


def _dehaze_case(ctx, fr, tag):
    st = {}
    out, out8 = O.bgdehaze_frame(fr, 15, st)
    normI = O.normalize_frame(fr)
    B, idx = ctx.background_light(fr, 15)
    Bo, idxo = O.background_light(normI, 15, True)
    assert idx == idxo and np.abs(B - Bo).max() < 1e-15, tag
    tb, tg = ctx.transmission(fr)
    t = O.transmission_map(normI, 15, Bo)
    assert np.abs(tb - t[..., 0]).max() < 1e-14 and np.abs(tg - t[..., 1]).max() < 1e-14, tag
    rb, rg = ctx.refined_transmission(fr)
    # float intermediates: <= 1e-5 relative (BASELINE north_star)
    assert (np.abs(rb - st["t_blue"]) / np.abs(st["t_blue"])).max() < 1e-5, tag
    assert (np.abs(rg - st["t_green"]) / np.abs(st["t_green"])).max() < 1e-5, tag
    rest = ctx.rc_correction(fr)
    assert np.abs(rest - st["restored"]).max() < 1e-5, tag
    got8, gotf = ctx.bgdehaze(fr, return_float=True)
    assert np.abs(gotf - out).max() < OUT_TOL, tag
    d = np.abs(got8.astype(int) - out8.astype(int))
    assert d.max() <= 1, (tag, d.max())  # max abs <= 1 LSB on the 8-bit output
    return (d > 0).mean()


@pytest.mark.parametrize("size", [(128, 96), (240, 135), (480, 270), (641, 479)])
def test_dehaze_synth(ctx, size):
    w, h = size
    frac = _dehaze_case(ctx, O.synth_frame(0x5EED0003, 0, w, h), size)
    assert frac < 0.02


def test_dehaze_golden_literal(ctx):
    """Against the literal reference outputs stored by oracle/make_golden.py."""
    z = np.load(os.path.join(GOLD, "dehaze_literal.npz"))
    for name in sorted({k.split("/")[0] for k in z.files}):
        fr = z[name + "/frame"]
        px = z[name + "/px"]   # the float maps are stored at these pixels
        B, _ = ctx.background_light(fr, 15)
        assert np.abs(B - z[name + "/B"]).max() < 1e-15
        got8, gotf = ctx.bgdehaze(fr, return_float=True)
        assert np.abs(O.golden_pixels(gotf, px) - z[name + "/out"]).max() < OUT_TOL, name
        ref8 = O._sat_u8_from_rint(z[name + "/out"] * 255).astype(int)
        assert np.abs(O.golden_pixels(got8, px).astype(int) - ref8).max() <= 1, name
        if name + "/t_blue" in z.files:
            rb, rg = ctx.refined_transmission(fr)
            assert (np.abs(O.golden_pixels(rb, px) - z[name + "/t_blue"]) / np.abs(z[name + "/t_blue"])).max() < 1e-5
            assert (np.abs(O.golden_pixels(rg, px) - z[name + "/t_green"]) / np.abs(z[name + "/t_green"])).max() < 1e-5


def test_dehaze_1080p(ctx):
    frac = _dehaze_case(ctx, O.synth_frame(0x5EED0003, 0, 1920, 1080), "1080p")
    assert frac < 0.02


def test_dehaze_window_param(ctx):
    fr = O.synth_frame(0x5EED0003, 4, 200, 150)
    normI = O.normalize_frame(fr)
    for w in [7, 15, 21]:
        B, idx = ctx.background_light(fr, w)
        Bo, idxo = O.background_light(normI, w, True)
        assert idx == idxo and np.abs(B - Bo).max() < 1e-15
    out8 = ctx.bgdehaze(fr, ctx.dehaze_params(window=21))
    want = O.bgdehaze_frame(fr, 21)[1]
    assert np.abs(out8.astype(int) - want.astype(int)).max() <= 1


# ---- chain ------------------------------------------------------------------------------------------------
def test_chain_small(ctx, kat):
    for key, e in kat["chain"].items():
        wh, f = key.split("_f")
        W, H = map(int, wh.split("x"))
        fr = O.synth_frame(0x5EED0004, int(f), W, H)
        assert O.crc32(ctx.histretch(fr, "V", 1, 99)) == e["histretch_crc"]
        assert O.crc32(ctx.aclahe(ctx.histretch(fr, "V", 1, 99), 2.0, (8, 8))) == e["aclahe_crc"]
        got = ctx.chain(fr)
        want = O.chain_frame(fr)
        assert np.abs(got.astype(int) - want.astype(int)).max() <= 1


def test_chain_batch_matches_single_and_device_path(ctx):
    import torch

    W, H, n = 320, 180, 5
    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in range(n)])
    host = ctx.chain(frames)
    singles = np.stack([ctx.chain(frames[i]) for i in range(n)])
    assert (host == singles).all()
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    ctx.chain_dev(d_in, d_out, n, W, H)
    ctx.synchronize()
    assert (d_out.cpu().numpy() == host).all()
    # un-fused head (generic channel string) agrees with the fused V head
    p = ctx.chain_params(channels="xV")
    assert (ctx.chain(frames, p) == host).all()
    # staged pieces == chain
    staged = np.stack([ctx.bgdehaze(ctx.aclahe(ctx.histretch(f, "V", 1, 99), 2.0, (8, 8))) for f in frames])
    assert (staged == host).all()
    want = np.stack([O.chain_frame(f) for f in frames])
    assert np.abs(host.astype(int) - want.astype(int)).max() <= 1
    assert (ctx.last_frame_flags(n) == 0).all()


def test_bench_dump_outputs_are_the_chain_outputs(ctx, tmp_path):
    """`bench.py --dump-outputs DIR` writes what its timed chain step returned: the batch is small enough to be written
    whole, so frames.npy must equal the chain of the same synthetic frames, and frame_flags.npy their flags."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    W, H, n = 320, 180, 2
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--frames", str(n), "--width", str(W), "--height", str(H),
                        "--steps", "1", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 1
    frames = np.stack([O.synth_frame(0x5EED0004, f, W, H) for f in range(n)])   # bench.py's SEED, rank 0's frames
    want = ctx.chain(frames)
    got = np.load(tmp_path / "frames.npy")
    assert got.dtype == np.float32 and (got == want).all()
    flags = np.load(tmp_path / "frame_flags.npy")
    assert flags.dtype == np.float32 and (flags == ctx.last_frame_flags(n)).all()


def test_chain_host_schedule(ctx, monkeypatch):
    """uwip_chain_bgr8 cuts the batch into sub-batches (csrc/e2e_schedule.h; UWIP_E2E_SIZES replaces the schedule): whatever
    the cut, the bytes are those of the device-resident call, and the per-frame flags line up with the frames."""
    import torch

    W, H, n = 160, 120, 12
    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in range(n)])
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    ctx.chain_dev(d_in, d_out, n, W, H)
    ctx.synchronize()
    want = d_out.cpu().numpy()
    want_flags = np.asarray(ctx.last_frame_flags(n)).copy()
    for sizes in (None, "1,2,4,3,2", "6,6", "2,6,4", "1,1,1,1,1,1,1,1,1,1,1,1", "3,3", "12"):   # the last two are ignored: "3,3" does not add up, "12" is one sub-batch (no copy could overlap)
        if sizes is None:
            monkeypatch.delenv("UWIP_E2E_SIZES", raising=False)
        else:
            monkeypatch.setenv("UWIP_E2E_SIZES", sizes)
        got = ctx.chain(frames)
        assert (got == want).all(), sizes
        assert (np.asarray(ctx.last_frame_flags(n)) == want_flags).all(), sizes
    monkeypatch.delenv("UWIP_E2E_SIZES", raising=False)


def test_chain_nan_frame_matches_reference(ctx):
    """D9: where Yi = Yj = 0 the reference's S is 0/0 and the whole frame turns NaN (imwrite stores zeros).
    The CUDA path must flag exactly the frames the oracle does."""
    W, H = 320, 180
    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in range(3, 8)])  # frame 5 is a NaN frame
    got = ctx.chain(frames)
    flags = ctx.last_frame_flags(len(frames))
    assert flags[2] == 1 and flags.sum() == 1
    for i, fr in enumerate(frames):
        b = O.aclahe_frame(O.histretch_frame(fr, "V", 1, 99), 2.0, 8, 8)
        out, out8 = O.bgdehaze_frame(b, 15)
        assert bool(flags[i] & 1) == bool(np.isnan(out).any()), i
        assert np.abs(got[i].astype(int) - out8.astype(int)).max() <= 1


def test_chain_full_size_properties(ctx):
    """BASELINE config sizes: size-independent properties instead of a full oracle run."""
    import torch

    import uwimageproc_b200 as u

    W, H, n = 3840, 2160, 3
    d_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d_in, 0x5EED0004, 0, n, W, H)
    d_out = torch.empty_like(d_in)
    ctx.chain_dev(d_in, d_out, n, W, H)
    ctx.synchronize()
    out = d_out.cpu().numpy()
    flags = ctx.last_frame_flags(n)
    # the final min-max normalisation pins the extremes of every frame; a frame on which the reference's
    # exposure map is NaN (S = 0/0, SURVEY 8a-D9) comes out all zero, as imwrite would store it
    for i in range(n):
        if flags[i] & 1:
            assert out[i].max() == 0
        else:
            assert out[i].min() == 0 and out[i].max() == 255
    assert (flags & 1).sum() < n
    # determinism + batch independence: frame 1 alone gives the same bytes
    d_o1 = torch.empty_like(d_in[1:2])
    ctx.chain_dev(d_in[1:2].contiguous(), d_o1, 1, W, H)
    ctx.synchronize()
    assert (d_o1.cpu().numpy()[0] == out[1]).all()
    assert (ctx.checksum_dev(d_out, n, W, H) == u.host_checksum(out)).all()
    # head of the chain bit-exact at 4K against the oracle (cheap stages)
    fr = d_in[0].cpu().numpy()
    a = ctx.histretch(fr, "V", 1, 99)
    assert (a == O.histretch_frame(fr, "V", 1, 99)).all()
    assert (ctx.aclahe(a, 2.0, (8, 8)) == O.aclahe_frame(a, 2.0, 8, 8)).all()


def test_chain_4k_against_oracle(ctx):
    """The headline configuration itself (BASELINE configs[3]: 3840x2160, seed 0x5EED0004 - frames 0 and 1 are the first
    two frames bench.py processes) against the fp64 oracle: 8-bit output <= 1 LSB, refined transmission <= 1e-5 relative.
    The oracle needs about half a minute per 4K frame."""
    W, H = 3840, 2160
    frames = np.stack([O.synth_frame(0x5EED0004, f, W, H) for f in (0, 1)])
    got = ctx.chain(frames)
    flags = ctx.last_frame_flags(2)
    checked = 0
    for i in range(2):
        head = O.aclahe_frame(O.histretch_frame(frames[i], "V", 1, 99), 2.0, 8, 8)
        st = {}
        ref, ref8 = O.bgdehaze_frame(head, 15, st)
        assert bool(flags[i] & 1) == bool(np.isnan(ref).any()), i
        d = np.abs(got[i].astype(int) - ref8.astype(int))
        assert d.max() <= 1, (i, d.max())
        assert (d > 0).mean() < 0.02
        if i == 0:
            # float stage at full size: refined t of the frame the dehaze stage sees
            assert (ctx.aclahe(ctx.histretch(frames[i], "V", 1, 99), 2.0, (8, 8)) == head).all()
            rb, rg = ctx.refined_transmission(head)
            assert (np.abs(rb - st["t_blue"]) / np.abs(st["t_blue"])).max() < 1e-5
            assert (np.abs(rg - st["t_green"]) / np.abs(st["t_green"])).max() < 1e-5
        checked += 1
    assert checked == 2


# ---- frame-batch sharding (SURVEY 8e): ranks are emulated one after the other on one GPU ------------------------
def test_sharded_stream_equals_single_gpu(ctx):
    import torch

    from uwimageproc_b200.shard import batches, frame_range

    W, H, total = 480, 270, 11
    d_in = torch.empty((total, H, W, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d_in, 0x5EED0005, 0, total, W, H)
    d_out = torch.empty_like(d_in)
    ctx.chain_dev(d_in, d_out, total, W, H)
    ctx.synchronize()
    single = ctx.checksum_dev(d_out, total, W, H)
    for world in (2, 4):
        got = np.zeros(total, np.uint64)
        for rank in range(world):
            first, count = frame_range(rank, world, total)
            for f, n in batches(first, count, 2):  # each rank generates ITS frames and runs them in batches of 2
                b_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
                ctx.synth_dev(b_in, 0x5EED0005, f, n, W, H)
                b_out = torch.empty_like(b_in)
                ctx.chain_dev(b_in, b_out, n, W, H)
                ctx.synchronize()
                got[f:f + n] = ctx.checksum_dev(b_out, n, W, H)
        assert (got == single).all(), world


def test_cpp_shims_on_device():
    """The reference-shaped C++ entry points (uwimageproc_b200/shims) against K0 of SURVEY 8c."""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "uwimageproc_b200", "shims", "shim_test")
    if not os.path.exists(exe):
        subprocess.run(["bash", os.path.join(root, "uwimageproc_b200", "shims", "check.sh")], check=True, capture_output=True)
    r = subprocess.run([exe, "gpu"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize("radius", [3, 4, 7, 10, 16, 40, 63, 64, 65, 100, 128])
def test_refined_transmission_other_radii(ctx, radius):
    """The guided-filter radius is a parameter of the ABI (the reference fixes r=40, BGDehaze.py:41): radii that
    are multiples of 4 take the quad path, the others the scalar window path; windows wider than 127 pixels (r >= 64)
    recompute the per-column pixel counts per row instead of unpacking them; all against the oracle."""
    fr = O.synth_frame(0x5EED0003, 2, 213, 118)   # width not a multiple of 4: pad columns are exercised too
    normI = O.normalize_frame(fr)
    for eps, tmin in [(1e-3, 0.2), (1e-2, 0.35)]:
        rb, rg = ctx.refined_transmission(fr, ctx.dehaze_params(radius=radius, eps=eps, tmin=tmin))
        tb, tg = O.refined_t(normI, 15, tmin, radius, eps)
        assert (np.abs(rb - tb) / np.abs(tb)).max() < 1e-5, (radius, eps)
        assert (np.abs(rg - tg) / np.abs(tg)).max() < 1e-5, (radius, eps)


def test_dehaze_degenerate_frames(ctx):
    """Constant frame (range 0: every normalised value is 0/0) and a two-level frame: the reference turns the
    constant frame into NaN (imwrite stores zeros); the CUDA path must flag it and write zeros, not crash."""
    const = np.full((64, 80, 3), 93, np.uint8)
    out = ctx.bgdehaze(const)
    assert out.shape == const.shape and out.max() == 0
    two = const.copy()
    two[:, 40:] = (30, 200, 120)
    got = ctx.bgdehaze(two)
    ref, ref8 = O.bgdehaze_frame(two, 15)
    if np.isnan(ref).any():
        assert got.max() == 0
    else:
        assert np.abs(got.astype(int) - ref8.astype(int)).max() <= 1


def test_result_independent_of_batch_split(ctx):
    """A frame's bytes must not depend on how the batch is cut (sub-batches, vertical segments of the guided
    filter march, GPU count): every value entering a running sum sits on a power-of-two grid, so the sums are
    exact.  1080p frames alone (many vertical segments) against the same frames inside a batch of 12 (one)."""
    import torch

    W, H, n = 1920, 1080, 12
    d_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d_in, 0x5EED0006, 0, n, W, H)
    d_out = torch.empty_like(d_in)
    ctx.chain_dev(d_in, d_out, n, W, H)
    ctx.synchronize()
    whole = ctx.checksum_dev(d_out, n, W, H)
    for i in (0, 5, 11):
        one = torch.empty_like(d_in[i:i + 1])
        ctx.chain_dev(d_in[i:i + 1].contiguous(), one, 1, W, H)
        ctx.synchronize()
        assert ctx.checksum_dev(one, 1, W, H)[0] == whole[i], i
    # host-buffer path (ramped sub-batches) == device path
    host = ctx.chain(d_in.cpu().numpy())
    assert (host == d_out.cpu().numpy()).all()


def test_abi_error_statuses(ctx):
    """What the reference leaves undefined (preprocessing.h:60-64) or prints-and-skips becomes a status code."""
    import ctypes as C

    import uwimageproc_b200 as u

    lib = ctx.lib
    plane = np.zeros((16, 16), np.uint8)
    out = np.zeros_like(plane)
    hist = (C.c_float * 256)()
    # null pointers, bad sizes, pitch smaller than a row
    assert lib.uwip_histogram_u8(ctx.h, None, 16, 16, 16, hist) == -1
    assert lib.uwip_histogram_u8(ctx.h, plane.ctypes.data, 0, 16, 16, hist) == -1
    assert lib.uwip_histogram_u8(ctx.h, plane.ctypes.data, 16, 16, 8, hist) == -1
    assert b"pitch" in lib.uwip_last_error(ctx.h) or b"bad image" in lib.uwip_last_error(ctx.h)
    # percentiles outside 0 <= lo < hi <= 100
    for lo, hi in [(-1, 50), (50, 50), (60, 40), (0, 101)]:
        assert lib.uwip_channel_stretch_u8(ctx.h, plane.ctypes.data, 16, out.ctypes.data, 16, 16, 16, lo, hi, None, None) == -1
    # dehaze parameter ranges
    fr = np.zeros((32, 32, 3), np.uint8) + np.arange(32, dtype=np.uint8)[None, :, None] * 7
    for kw in (dict(window=0), dict(window=35), dict(radius=0), dict(radius=129), dict(radius=161)):
        with pytest.raises(u.UwipError) as e:
            ctx.bgdehaze(fr, ctx.dehaze_params(**kw))
        assert e.value.status == -1
    # radius 129: a full window's sum of k_i k_j can pass 2^32 (guided_filter_u8_dev's 32-bit moment sums)
    for r in (0, 129):
        with pytest.raises(u.UwipError) as e:
            ctx.guided_filter_u8(fr, 255, np.full(fr.shape[:2], 0.5), r, 1e-3)
        assert e.value.status == -1
    # a call after an error works (the context stays usable)
    assert (ctx.histogram(plane) == O.get_histogram(plane)).all()
    # frame flags: asking for more frames than the last call processed is refused
    ctx.chain(fr[None])
    with pytest.raises(u.UwipError):
        ctx.last_frame_flags(5)
