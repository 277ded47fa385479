"""The grey prototype (modules/aclahe/python/main.py) on the device: the grey JPEG writer (uwip_jpeg_encode_u8_batch_dev)
against cv2.imencode, the grey reader (uwip_jpeg_decode_u8_batch) against cv2.imdecode(.., IMREAD_GRAYSCALE), automatic
CLAHE on planes (uwip_aclahe_u8_auto_dev) against the oracle's ParametrosACLAHE and cv2's CLAHE, and `aclahe -grey=1
-device=1` on a file and on a directory."""
import os
import warnings

import cv2
import numpy as np
import pytest

from oracle import uwip_oracle as O
from test_jpeg_decoder_host import EXTRAS, _segments, imencode
from test_jpeg_grey_host import planes as grey_planes

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
H, W = 180, 320
NOFIT, JPEG_BAD = 2, 4
NOTE_NOFIT = "note: the entropy curve fit failed for this frame (the reference raises); the fixed 8x8 grid and clip 2 were used"


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _cv2(p, q):
    ok, b = cv2.imencode(".jpg", p, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(b)


def _encode(ctx, ps, q):
    import torch

    return ctx.jpeg_encode_grey_batch_dev(torch.from_numpy(np.ascontiguousarray(ps)).cuda(), q)


# ---- writer ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("q", [1, 50, 95, 100])
def test_writer_equals_cv2_across_sizes(ctx, q):
    for (w, h) in [(1, 1), (1, 29), (23, 1), (7, 9), (8, 8), (15, 17), (17, 16), (53, 37), (481, 270)]:
        ps = np.stack(list(grey_planes(w, h, w * 7 + h).values()))
        got = _encode(ctx, ps, q)
        assert got == [_cv2(p, q) for p in ps], (w, h)


def test_writer_4k_batch_and_alone(ctx):
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:2160, 0:3840]
    v = O.bgr2hsv(O.synth_frame(0x5EED0004, 3, 3840, 2160))[..., 2]
    ps = np.stack([v, rng.integers(0, 256, (2160, 3840), dtype=np.uint8), ((xx + 2 * yy) % 256).astype(np.uint8)])
    got = _encode(ctx, ps, 95)
    assert got == [_cv2(p, 95) for p in ps]
    assert _encode(ctx, ps[1:2], 95) == got[1:2]
    assert ctx.jpeg_encode_grey(ps[2], 95) == got[2]


def test_writer_refusals(ctx):
    import torch

    from uwimageproc_b200._lib import UwipError

    d = torch.zeros((1, 16, 16), dtype=torch.uint8, device="cuda")
    out = torch.empty(ctx.jpeg_encode_grey_bound(16, 16), dtype=torch.uint8, device="cuda")
    ln = torch.empty(1, dtype=torch.int64, device="cuda")
    for q, stride in [(0, out.numel()), (101, out.numel()), (95, out.numel() - 1)]:
        with pytest.raises(UwipError):
            ctx._ck(ctx.lib.uwip_jpeg_encode_u8_batch_dev(ctx.h, d.data_ptr(), 1, 16, 16, q, out.data_ptr(), stride, ln.data_ptr()))
    assert ctx.jpeg_encode_grey_bound(0, 5) == 0 and ctx.jpeg_encode_grey_bound(65536, 5) == 0


# ---- reader ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sampling", ["444", "422", "440", "420", "grey"])
def test_reader_equals_cv2_imdecode_grayscale(ctx, sampling):
    rng = np.random.default_rng(2)
    for (w, h) in [(1, 1), (7, 9), (53, 37), (481, 270)]:
        files = []
        for ename, extra in EXTRAS.items():
            f = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            files.append(imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), 90, None, extra) if sampling == "grey" else imencode(f, 90, sampling, extra))
        got = ctx.jpeg_decode_grey(files)
        for name, b, g in zip(EXTRAS, files, got):
            assert (g == cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_GRAYSCALE)).all(), (w, h, name)
        assert not ctx.last_frame_flags(len(files)).any()


def test_reader_truncated_file_in_a_batch(ctx):
    fs = [imencode(O.synth_frame(0x5EED0004, i, 160, 96), 95, "420") for i in range(3)]
    sos = dict(_segments(fs[1]))[0xDA]
    fs[1] = fs[1][:sos + 14 + (len(fs[1]) - sos) // 2]
    got = ctx.jpeg_decode_grey(fs)
    flags = ctx.last_frame_flags(3)
    assert flags.tolist() == [0, JPEG_BAD, 0]
    assert not got[1].any()
    for i in (0, 2):
        assert (got[i] == cv2.imdecode(np.frombuffer(fs[i], np.uint8), cv2.IMREAD_GRAYSCALE)).all()
        assert (ctx.jpeg_decode_grey(fs[i]) == got[i]).all()


# ---- automatic CLAHE on planes ---------------------------------------------------------------------------------------
def _oracle_params(plane, loop="repaired"):
    try:
        bs, cl, _ = O.parametros_aclahe(plane, loop)
        return bs, cl
    except RuntimeError:
        return -1, -1


def _auto(ctx, ps, loop="repaired"):
    """main_batch runs on the module's default context: its flags are read there"""
    from uwimageproc_b200.api import default_context
    from uwimageproc_b200.modules import aclahe as A

    out, bs, cl = A.main_batch(ps, loop)
    return out, list(zip(bs.tolist(), cl.tolist())), default_context().last_frame_flags(len(ps))


def test_crowd_full_both_loops(ctx):
    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    img = z["img"]
    for loop in ("repaired", "as_committed"):
        out, params, flags = _auto(ctx, img[None], loop)
        assert params == [tuple(z[loop])] and flags[0] == 0
        bs, cl = params[0]
        assert (out[0] == cv2.createCLAHE(float(cl), (bs, bs)).apply(img)).all()
    assert [tuple(z["repaired"]), tuple(z["as_committed"])] == [(4, 7), (8, 0)]


def test_corpus_matches_parametros_aclahe_and_cv2_clahe(ctx):
    from uwimageproc_b200.modules import aclahe as A

    crowd = np.load(os.path.join(GOLD, "crowd_full.npz"))["img"][200:200 + H, 300:300 + W]
    yy, xx = np.mgrid[0:H, 0:W]
    grad = ((xx * 255) // (W - 1) * 0.7 + (yy * 255) // (H - 1) * 0.3).astype(np.uint8)
    uni = np.random.default_rng(3).integers(0, 256, (H, W), dtype=np.uint8)
    synth = [O.bgr2hsv(O.synth_frame(0x5EED0004, i, W, H))[..., 2].copy() for i in (6, 9)]
    ps = np.stack([crowd, grad, uni] + synth)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = [_oracle_params(p) for p in ps]
        mirror = [A.ParametrosACLAHE(p) for i, p in enumerate(ps) if want[i] != (-1, -1)]
    assert want[2] == (-1, -1)
    assert mirror == [w for w in want if w != (-1, -1)]
    out, params, flags = _auto(ctx, ps)
    assert params == want
    for i, (p, (bs, cl)) in enumerate(zip(ps, params)):
        if bs < 0:
            assert flags[i] == NOFIT
            ref = cv2.createCLAHE(2.0, (8, 8)).apply(p)
        else:
            assert flags[i] == 0
            ref = cv2.createCLAHE(float(cl), (bs, bs)).apply(p)
        assert (out[i] == ref).all(), i
    # a plane's output does not depend on its batch
    one, p1, _ = _auto(ctx, ps[4:5])
    assert p1 == params[4:5] and (one[0] == out[4]).all()


def test_refuses_planes_too_small_for_the_search(ctx):
    from uwimageproc_b200._lib import UwipError
    from uwimageproc_b200.modules import aclahe as A

    with pytest.raises(UwipError):
        A.main_batch(np.zeros((1, 10, 10), np.uint8))   # 10 px cannot be reflect-101 padded to a 32 x 32 grid


# ---- command line ----------------------------------------------------------------------------------------------------
def _cli(argv):
    from uwimageproc_b200.cli import aclahe as cli

    assert cli.main(argv) == 0


def test_cli_single_file_is_the_reference_file(ctx, tmp_path, capsys):
    crowd = np.load(os.path.join(GOLD, "crowd_full.npz"))["img"]
    src = tmp_path / "crowd.png"
    cv2.imwrite(str(src), crowd)
    for loop, (bs, cl) in (("repaired", (4, 7)), ("as_committed", (8, 0))):
        out = tmp_path / ("clahe_2_%s.jpg" % loop)
        capsys.readouterr()
        _cli([str(src), str(out), "-grey=1", "-device=1", "-loop=" + loop])
        assert "BS = %d, CL = %d\n" % (bs, cl) in capsys.readouterr().out
        want = tmp_path / "want.jpg"
        cv2.imwrite(str(want), cv2.createCLAHE(float(cl), (bs, bs)).apply(crowd))
        assert out.read_bytes() == want.read_bytes()
    # a JPEG input goes through the grey reader: the pixels of cv2.imread(.., 0)
    jin = tmp_path / "crowd.jpg"
    cv2.imwrite(str(jin), crowd)
    _cli([str(jin), str(tmp_path / "from_jpeg.png"), "-grey=1", "-device=1"])
    grey = cv2.imread(str(jin), 0)
    res, bs, cl = _main_batch(grey)
    assert bs > 0 and (cv2.imread(str(tmp_path / "from_jpeg.png"), 0) == res).all()
    assert (res == cv2.createCLAHE(float(cl), (bs, bs)).apply(grey)).all()


def test_cli_directory_mode(ctx, tmp_path, capsys):
    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    dst.mkdir()
    names = {"a.jpg": O.synth_frame(0x5EED0004, 24, W, H), "b.jpg": O.synth_frame(0x5EED0004, 26, W, H),
             "c.jpg": np.random.default_rng(5).integers(0, 256, (H, W), dtype=np.uint8), "d.jpg": O.synth_frame(0x5EED0004, 6, 160, 96)}
    for n, img in names.items():
        (src / n).write_bytes(imencode(img, 95, "420") if img.ndim == 3 else _cv2(img, 95))
    capsys.readouterr()
    _cli([str(src), str(dst), "-grey=1", "-device=1", "-batch=2"])
    out = capsys.readouterr().out
    lines = []
    for n in sorted(names):
        g = cv2.imread(str(src / n), 0)
        res, bs, cl = _main_batch(g)
        if bs < 0:
            res = cv2.createCLAHE(2.0, (8, 8)).apply(g)
        assert (dst / n).read_bytes() == _cv2(res, 95), n
        lines += ["%s: BS = %d, CL = %d" % (n, bs, cl)] + ([NOTE_NOFIT] if bs < 0 else []) + ["saved %s" % (dst / n)]
    assert out.split("\n")[-len(lines) - 1:] == lines + [""]


def _main_batch(p):
    from uwimageproc_b200.modules import aclahe as A

    out, bs, cl = A.main_batch(p[None])
    return out[0], int(bs[0]), int(cl[0])
