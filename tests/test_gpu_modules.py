"""GPU tests of the reference-facing Python mirrors (uwimageproc_b200/modules/*) and of the batch `_dev` entry points
called directly with n > 1.  Everything goes through libuwip.so; the oracle / the golden files are the checkers."""
import os

import numpy as np
import pytest

from oracle import uwip_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
OUT_TOL = 1.0 / 255.0  # see tests/test_gpu_parity.py


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.default_context()
    yield c


# ---- modules/bgdehaze: BGDehaze.py function names on normI ------------------------------------------------
def test_bgdehaze_module_against_literal_reference(ctx):
    """adaptiveExp_map(normI) and the five helpers of BGDehaze.py:14-89 through the mirror module, against the outputs
    the reference's own BGDehaze.py produced in the build container (tests/golden/dehaze_literal.npz)."""
    from uwimageproc_b200.modules import bgdehaze as M

    z = np.load(os.path.join(GOLD, "dehaze_literal.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    assert names
    for name in names:
        fr = z[name + "/frame"]
        px = z[name + "/px"]   # the float maps are stored at these pixels
        normI = O.normalize_frame(fr)
        assert (M._as_u8(normI) == fr - fr.min()).all()   # the 8-bit frame behind normI (k - kmin: same normalisation)
        assert np.abs(M.Background_light(normI) - z[name + "/B"]).max() < 1e-15
        out = M.adaptiveExp_map(normI)
        assert out.shape == normI.shape and out.dtype == np.float64
        assert np.abs(O.golden_pixels(out, px) - z[name + "/out"]).max() < OUT_TOL, name
        if name + "/t_blue" in z.files:
            tb, tg = M.refined_t(normI)
            assert (np.abs(O.golden_pixels(tb, px) - z[name + "/t_blue"]) / np.abs(z[name + "/t_blue"])).max() < 1e-5
            assert (np.abs(O.golden_pixels(tg, px) - z[name + "/t_green"]) / np.abs(z[name + "/t_green"])).max() < 1e-5
        # stage functions against the oracle (first-index tie rule of the arg-min, as the module documents)
        st = {}
        O.bgdehaze_frame(fr, 15, st)
        t = M.transmission_map(normI)
        Bo = O.background_light(normI, 15)
        assert np.abs(t - O.transmission_map(normI, 15, Bo)).max() < 1e-14
        rest = M.RC_correction(normI)
        assert np.abs(rest - st["restored"]).max() < 1e-5
        jb, jg = M.dehazed_BG(normI)
        assert np.abs(jb - st["restored"][..., 0]).max() < 1e-5 and np.abs(jg - st["restored"][..., 1]).max() < 1e-5
        got8 = M.generate_results(fr)
        ref8 = O._sat_u8_from_rint(z[name + "/out"] * 255).astype(int)
        assert np.abs(O.golden_pixels(got8, px).astype(int) - ref8).max() <= 1


def test_bgdehaze_module_rejects_non_8bit_sources():
    from uwimageproc_b200.modules import bgdehaze as M

    bad = np.random.default_rng(3).random((8, 8, 3))
    bad[0, 0] = 0.0
    bad[1, 1] = 1.0
    with pytest.raises(ValueError):
        M.adaptiveExp_map(bad)


def test_guided_filter_and_boxfilter_stage_entries(ctx):
    """guidedfilter.py:23,54 as stage entry points: boxfilter on a float64 plane, guided_filter with an 8-bit BGR guide
    (normI) and with a YCrCb guide - the third filter of adaptiveExp_map (BGDehaze.py:84) - both <= 1e-5."""
    from uwimageproc_b200.modules import guidedfilter as G

    fr = O.synth_frame(0x5EED0003, 5, 232, 150)
    rng = np.random.default_rng(11)
    plane = rng.random((150, 232))
    for r in (3, 40):
        got = G.boxfilter(plane, r)
        want = O.boxfilter(plane, r)
        assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()
    normI = O.normalize_frame(fr)
    p = np.clip(0.2 + 0.8 * normI[..., 0] ** 2 + 0.05 * rng.random(normI.shape[:2]), 0.0, 1.0)
    q = G.guided_filter(normI, p, 40, 1e-3)
    want = O.guided_filter(normI, p, 40, 1e-3)
    assert (np.abs(q - want) / np.maximum(np.abs(want), 1e-3)).max() < 1e-5
    # YCrCb guide, normalised jointly over its three channels exactly like BGDehaze.py:77-80
    ycc = O.bgr2ycrcb(fr).astype(np.float64)
    guide = (ycc - ycc.min()) / (ycc.max() - ycc.min())
    S = np.clip(0.3 + normI[..., 1] + 0.02 * rng.random(normI.shape[:2]), 0.0, 1.5)
    q = G.guided_filter(guide, S, 40, 1e-3)
    want = O.guided_filter(guide, S, 40, 1e-3)
    assert (np.abs(q - want) / np.maximum(np.abs(want), 1e-3)).max() < 1e-5


# ---- modules/aclahe: the automatic parameter search (SURVEY K4) ---------------------------------------------
def test_parametros_aclahe_on_crowd(ctx):
    """ParametrosACLAHE (ACLAHE.py:9-129) on the reference's crowd.png pixels: (8, 0) as the file is committed,
    (4, 7) with the sweep loop repaired; the 5 x 50 entropy table against the reference's own functions.py."""
    from uwimageproc_b200.modules import aclahe as A

    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    img = z["img"]
    assert img.shape == (600, 800)
    assert abs(float(A.Entropia(img)) - 6.1331363) < 1e-5
    blur = ctx.gaussian_blur3(img)
    cl = np.arange(0, 25, 0.5)
    for j, bs in enumerate(A.BLOCK_SIZES):   # all five grids, every clip limit, one device pass per grid
        got = ctx.clahe_entropy_sweep(blur, bs, cl, "py")
        assert np.abs(got - z["entropies"][j]).max() < 1e-5, bs
    assert tuple(A.ParametrosACLAHE(img, loop="as_committed")) == tuple(int(v) for v in z["as_committed"]) == (8, 0)
    assert tuple(A.ParametrosACLAHE(img, loop="repaired")) == tuple(int(v) for v in z["repaired"]) == (4, 7)
    out = A.main(img)
    assert (out == O.clahe_apply(img, 7.0, 4, 4)).all()   # aclahe/python/main.py:18-20 with the repaired parameters


def test_sweep_batch_matches_single(ctx):
    """The batched sweep entry (frames x grids in one call) equals the one-grid calls."""
    import torch

    z = np.load(os.path.join(GOLD, "crowd_crop.npz"))
    base = z["img"]
    planes = np.stack([base, np.ascontiguousarray(base[::-1]), np.ascontiguousarray(base[:, ::-1])])
    clips = np.arange(0, 25.5, 0.5)
    grids = [2, 4, 8, 16, 32]
    d = torch.from_numpy(planes).cuda()
    got = ctx.clahe_entropy_sweep_dev(d, planes.shape[0], base.shape[1], base.shape[0], grids, clips, "py")
    assert got.shape == (3, 5, len(clips))
    for f in range(3):
        for j, g in enumerate(grids):
            want = ctx.clahe_entropy_sweep(planes[f], g, clips, "py")
            assert np.abs(got[f, j] - want).max() < 1e-6, (f, g)
    want0 = np.array([O.entropy_py(O.clahe_apply(base, c, 16, 16)) for c in clips])
    assert np.abs(got[0, 3] - want0).max() < 1e-5


# ---- modules/preprocessing, modules/videostrip -----------------------------------------------------------
def test_preprocessing_and_videostrip_modules(ctx):
    from uwimageproc_b200.modules import preprocessing as P
    from uwimageproc_b200.modules import videostrip as V

    fr = O.synth_frame(0x5EED0001, 0, 322, 200)
    plane = np.ascontiguousarray(fr[..., 1])
    assert (P.getHistogram(plane) == O.get_histogram(plane)).all()
    want = O.img_channel_stretch(plane, 2, 98)
    assert (P.imgChannelStretch(plane, None, 2, 98) == want).all()
    inplace = plane.copy()
    P.imgChannelStretchGPU(inplace, inplace, 2, 98)   # every reference caller passes the same plane twice
    assert (inplace == want).all()
    for c in "RGBHSVhslLabYCXr?":
        assert P.numChannel(c) == O.num_channel(c) and P.numSpace(c) == O.num_space(c)
    for letters in ("V", "HSV", "B", "Lab"):
        assert (P.histretch(fr, letters) == O.histretch_frame(fr, letters, 2, 98)).all(), letters
    assert (P.histretch(fr, "V", literal=True) == O.histretch_frame(fr, "V", 2, 98, order="literal")).all()
    assert abs(float(V.calcBlur(fr)) - float(O.calc_blur(fr))) < 1e-4
    assert abs(float(V.calcBlurGPU(fr)) - float(O.calc_blur(fr, aperture=1))) < 1e-4


# ---- batch `_dev` entry points called directly with n > 1 ---------------------------------------------------
def test_batch_dev_entry_points(ctx):
    import torch

    n, w, h = 5, 322, 200
    frames = np.stack([O.synth_frame(0x5EED0002, f, w, h) for f in range(n)])
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    ctx.histretch_dev(d_in, d_out, n, w, h, "HV", 2, 98)
    ctx.synchronize()
    got = d_out.cpu().numpy()
    for f in range(n):
        assert (got[f] == O.histretch_frame(frames[f], "HV", 2, 98)).all(), f
    ctx.aclahe_dev(d_in, d_out, n, w, h, 2.0, (8, 8))
    ctx.synchronize()
    got = d_out.cpu().numpy()
    for f in range(n):
        assert (got[f] == O.aclahe_frame(frames[f], 2.0, 8, 8)).all(), f
    planes = np.ascontiguousarray(frames[..., 2])
    dp_in = torch.from_numpy(planes).cuda()
    dp_out = torch.empty_like(dp_in)
    ctx.clahe_dev(dp_in, dp_out, n, w, h, 3.0, (4, 8))
    ctx.synchronize()
    got = dp_out.cpu().numpy()
    for f in range(n):
        assert (got[f] == O.clahe_apply(planes[f], 3.0, 4, 8)).all(), f
    ctx.bgdehaze_dev(d_in, d_out, n, w, h)
    ctx.synchronize()
    got = d_out.cpu().numpy()
    flags = ctx.last_frame_flags(n)
    for f in range(n):
        ref, ref8 = O.bgdehaze_frame(frames[f], 15)
        if np.isnan(ref).any():
            assert flags[f] != 0 and got[f].max() == 0
        else:
            assert flags[f] == 0
            assert np.abs(got[f].astype(int) - ref8.astype(int)).max() <= 1, f


def test_k3_background_light_on_fixture_frames(ctx):
    """SURVEY K3: Background_light (BGDehaze.py:14-31, first-index tie rule) on a full-resolution bgdehaze fixture of the
    reference: PIS_T1A_259.jpg as decoded by cv2.imread in the build container (oracle/make_golden_k3.py ->
    k3_pis_full.npz); B and the two arg-min indices are the ones oracle/make_golden.py stored in kat.json."""
    import json

    kat = json.load(open(os.path.join(GOLD, "kat.json")))
    z = np.load(os.path.join(GOLD, "k3_pis_full.npz"))
    checked = 0
    for name, e in kat["K3"].items():
        if name + "/full" not in z.files:
            continue
        B, idx = ctx.background_light(z[name + "/full"], 15)
        assert [int(i) for i in idx] == [int(i) for i in e["idx"]]
        assert np.abs(np.asarray(B, np.float64) - np.array(e["B_first_index"])).max() < 1e-15
        checked += 1
    assert checked >= 1


# ---- two contexts on two devices in one process (ADVICE r1: per-device kernel attributes) -----------------
def test_two_devices_in_one_process():
    import torch

    import uwimageproc_b200 as u

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    fr = O.synth_frame(0x5EED0004, 0, 320, 180)
    outs = []
    for dev in (0, 1):
        c = u.Context(dev)
        outs.append(c.chain(fr))
        c.close()
    assert (outs[0] == outs[1]).all()
    torch.cuda.set_device(0)


# ---- command-line shims (histretch.cpp:61-271, aclahe.cpp:64-226, bgdehaze/main.py:22-33) --------------------
def _write_ppm(path, bgr):
    with open(path, "wb") as f:
        f.write(b"P6\n%d %d\n255\n" % (bgr.shape[1], bgr.shape[0]))
        f.write(np.ascontiguousarray(bgr[..., ::-1]).tobytes())


def _read_ppm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"P6"
        w, h = map(int, f.readline().split())
        assert f.readline().strip() == b"255"
        return np.frombuffer(f.read(), np.uint8).reshape(h, w, 3)[..., ::-1].copy()


def test_cpp_cli_shims(tmp_path):
    """The histretch / aclahe binaries built by shims/check.sh (stand-in OpenCV: imread / imwrite speak PPM)."""
    import subprocess

    shims = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "uwimageproc_b200", "shims")
    exe = os.path.join(shims, "histretch")
    if not os.path.exists(exe):
        subprocess.run(["bash", os.path.join(shims, "check.sh")], check=True, capture_output=True)
    fr = O.synth_frame(0x5EED0001, 3, 200, 120)
    src, dst = str(tmp_path / "in.ppm"), str(tmp_path / "out.ppm")
    _write_ppm(src, fr)
    r = subprocess.run([exe, src, dst, "-c=HV", "-cuda=1", "-time=1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Execution Time GPU :" in r.stdout and "Channel[1]: V" in r.stdout and "hS: saving to disk" in r.stdout
    assert (_read_ppm(dst) == O.histretch_frame(fr, "HV", 2, 98)).all()
    r = subprocess.run([exe, src, dst, "-literal=1", "-c=Vr"], capture_output=True, text=True)   # as written + an unknown letter
    assert r.returncode == 0 and "Option r not recognized, skipping..." in r.stdout
    assert (_read_ppm(dst) == O.histretch_frame(fr, "V", 2, 98, order="literal")).all()
    r = subprocess.run([exe, src, dst], capture_output=True, text=True)                          # default -c=r: no-op (SURVEY H3)
    assert r.returncode == 0 and (_read_ppm(dst) == fr).all()
    exe = os.path.join(shims, "aclahe")
    r = subprocess.run([exe, src, dst, "-bs=8", "-cl=2"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    table = [l.split() for l in r.stdout.splitlines() if len(l.split()) == 51]
    assert len(table) == 5
    v = fr.max(axis=2)
    for i, bs in enumerate((2, 4, 8, 16, 32)):
        for j in (0, 4, 50):
            want = float(O.entropy_cpp(O.clahe_apply(v, 0.5 * j, bs, bs)))
            assert abs(float(table[i][j]) - want) < 2e-5, (bs, j)
    assert (_read_ppm(dst) == O.aclahe_frame(fr, 2.0, 8, 8)).all()


def test_python_cli_shims(tmp_path, capsys):
    cv2 = pytest.importorskip("cv2")
    from uwimageproc_b200.cli import aclahe as CA
    from uwimageproc_b200.cli import bgdehaze_main as CB
    from uwimageproc_b200.cli import histretch as CH

    fr = O.synth_frame(0x5EED0001, 4, 240, 136)
    src, dst = str(tmp_path / "in.png"), str(tmp_path / "out.png")
    cv2.imwrite(src, fr)
    assert CH.main([src, dst, "-c=V", "-time=1", "-cuda=0"]) == 0
    out = capsys.readouterr().out
    assert "Execution Time GPU :" in out and "Channel: V" in out and "no CPU path" in out
    assert (cv2.imread(dst) == O.histretch_frame(fr, "V", 2, 98)).all()
    assert CH.main([src]) == 0 and "Complete options are:" in capsys.readouterr().out
    z = np.load(os.path.join(GOLD, "crowd_crop.npz"))
    g_src = str(tmp_path / "grey.png")
    cv2.imwrite(g_src, z["img"])
    assert CA.main([g_src, dst, "-grey=1", "-loop=as_committed"]) == 0
    assert "BS = " in capsys.readouterr().out
    d_dst = str(tmp_path / "res" / "dehazed.png")
    assert CB.main(["--src", src, "--dest", d_dst, "-w", "15"]) == 0
    assert np.abs(cv2.imread(d_dst).astype(int) - O.bgdehaze_frame(fr, 15)[1].astype(int)).max() <= 1


# ---- JPEG files to and from the device (SURVEY 8f N3) ----------------------------------------------------------
def test_jpeg_device_io(ctx):
    """nvJPEG decode -> chain -> nvJPEG encode without the pixels touching the host.  nvJPEG's IDCT is not libjpeg-turbo's:
    the decoded pixels are compared with cv2.imdecode (max 4 levels apart on this frame, chroma upsampling differs: bounded here by
    8 levels and a mean of 1); the chain is then checked against the oracle on the
    pixels nvJPEG produced, and the encoded result by decoding it again."""
    cv2 = pytest.importorskip("cv2")
    fr = O.synth_frame(0x5EED0004, 2, 640, 360)
    ok, enc = cv2.imencode(".jpg", fr, [cv2.IMWRITE_JPEG_QUALITY, 95])
    assert ok
    data = enc.tobytes()
    assert ctx.jpeg_info(data) == (640, 360)
    d = ctx.jpeg_decode_dev(data)
    dec = d.cpu().numpy()
    ref = cv2.imdecode(enc, cv2.IMREAD_COLOR)
    diff = np.abs(dec.astype(int) - ref.astype(int))
    assert diff.max() <= 8 and diff.mean() < 1.0, (diff.max(), diff.mean())
    out_jpeg = ctx.chain_jpeg(data, quality=95)
    got = cv2.imdecode(np.frombuffer(out_jpeg, np.uint8), cv2.IMREAD_COLOR)
    assert got.shape == fr.shape
    want = O.chain_frame(dec)                      # the oracle on nvJPEG's pixels
    direct = ctx.chain(dec)                        # the chain on the same pixels, no JPEG on the way out
    assert np.abs(direct.astype(int) - want.astype(int)).max() <= 1
    mse = np.mean((got.astype(float) - direct.astype(float)) ** 2)
    psnr = 10 * np.log10(255.0 ** 2 / max(mse, 1e-9))
    assert psnr > 30.0, psnr                       # quality-95 4:2:0 JPEG of the result
    rt = ctx.jpeg_encode_dev(d, 640, 360, 95)
    back = cv2.imdecode(np.frombuffer(rt, np.uint8), cv2.IMREAD_COLOR)
    assert 10 * np.log10(255.0 ** 2 / np.mean((back.astype(float) - dec.astype(float)) ** 2)) > 30.0
