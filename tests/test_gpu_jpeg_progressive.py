"""The progressive-capable device JPEG reader (uwip_jpeg_decode_batch_ex, `progressive=True`): every frame equal to
cv2.imdecode for batches that mix progressive and baseline files, samplings, qualities and restart intervals, in colour, grey
and oriented forms; 4K progressive files; batch-split independence; a file cut inside a scan in the middle of a batch; the
refusals through the C ABI and uwip_jpeg_probe; and `chain` / `aclahe` over directories that mix progressive and baseline
files."""
import ctypes as C
import os

import cv2
import numpy as np
import pytest

from oracle import uwip_oracle as O
from test_jpeg_decoder_host import imencode
from test_jpeg_orientation_host import frame, tag
from test_jpeg_progressive_host import cv2_decode, cv2_prog, pil_prog, scan_end, set_scan, sos_offsets

pytestmark = pytest.mark.gpu
SAMPLINGS = ["420", "444", "422", "440", "grey"]


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _file(i, w, h):
    """file i of a mixed batch: progressive (cv2 or Pillow) or baseline, every sampling, qualities 1..100, restart 0 / 1 / 7"""
    f = frame(w, h, 200 + i)
    s = SAMPLINGS[i % 5]
    img = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) if s == "grey" else f
    q = (1, 50, 95, 100)[i % 4]
    rst = (0, 1, 7)[i % 3]
    kind = i % 3
    if kind == 0:
        return imencode(img, q, None if s == "grey" else s, [cv2.IMWRITE_JPEG_RST_INTERVAL, rst] if rst else [])
    if kind == 1 or s == "440":
        return cv2_prog(img, q, None if s == "grey" else s, rst)
    return pil_prog(img, min(q, 90), s)


def _check(ctx, files, grey, orient=False):
    got = (ctx.jpeg_decode_grey if grey else ctx.jpeg_decode)(files, orientation=orient, progressive=True)
    want = np.stack([cv2_decode(b, grey, orient) for b in files])
    assert got.shape == want.shape
    bad = [i for i in range(len(files)) if not (got[i] == want[i]).all()]
    assert not bad, "frames %s of %d differ from cv2.imdecode" % (bad[:10], len(files))
    assert not ctx.last_frame_flags(len(files)).any()


@pytest.mark.parametrize("grey", [False, True], ids=["bgr8", "u8"])
@pytest.mark.parametrize("n", [1, 7, 60])
def test_mixed_batches_equal_cv2(ctx, n, grey):
    files = [_file(i + (1 if n == 1 else 0), 97, 45) for i in range(n)]
    _check(ctx, files, grey)


@pytest.mark.parametrize("grey", [False, True], ids=["bgr8", "u8"])
def test_mixed_orientations_equal_cv2(ctx, grey):
    files = []
    for i in range(16):
        o = 1 + i % 8
        b = _file(i, 45, 97) if o >= 5 else _file(i, 97, 45)
        files.append(tag(b, o, le=i % 2 == 0))
    _check(ctx, files, grey, orient=True)
    ws = [ctx.jpeg_probe(b) for b in files]
    assert all(p[:2] == (97, 45) and p[2] == 1 + i % 8 for i, p in enumerate(ws))


@pytest.mark.parametrize("grey", [False, True], ids=["bgr8", "u8"])
def test_4k_progressive(ctx, grey):
    f0, f1 = O.synth_frame(0x5EED0004, 5, 3840, 2160), O.synth_frame(0x5EED0004, 6, 3840, 2160)
    files = [cv2_prog(f0, 95, "420"), imencode(f1, 95, "420"), cv2_prog(f1, 90, "444", 7), pil_prog(f0, 85, "420")]
    _check(ctx, files, grey)


def test_batch_split_independence(ctx):
    files = [_file(i, 61, 33) for i in range(13)]
    for grey in (False, True):
        dec = ctx.jpeg_decode_grey if grey else ctx.jpeg_decode
        whole = dec(files, progressive=True)
        parts = np.concatenate([dec(files[:4], progressive=True), dec(files[4:5], progressive=True), dec(files[5:], progressive=True)])
        singles = np.stack([dec(b, progressive=True) for b in files])
        assert (whole == parts).all() and (whole == singles).all()


def test_cut_inside_a_scan_in_a_batch(ctx):
    files = [cv2_prog(frame(96, 64, 300 + i), 95, "420", (0, 7)[i % 2]) if i % 2 else imencode(frame(96, 64, 300 + i), 90, "420")
             for i in range(8)]
    b = files[3]
    sos = sos_offsets(b)
    cuts = [b[:(sos[k] + scan_end(b, sos[k])) // 2] for k in (2, len(sos) - 1)]
    for cut in cuts:
        batch = files[:3] + [cut] + files[4:]
        for grey in (False, True):
            got = (ctx.jpeg_decode_grey if grey else ctx.jpeg_decode)(batch, progressive=True)
            assert ctx.last_frame_flags(8).tolist() == [0, 0, 0, 4, 0, 0, 0, 0]
            assert not got[3].any()
            assert all((got[i] == cv2_decode(batch[i], grey)).all() for i in range(8) if i != 3)


def test_refusals_through_the_c_abi(ctx):
    import torch

    from uwimageproc_b200 import UwipError

    b = cv2_prog(frame(40, 24, 1), 90, "420")
    base = imencode(frame(40, 24, 2), 90, "420")
    sos = sos_offsets(b)
    incomplete = b[:scan_end(b, sos[4])] + b"\xff\xd9"
    mismatch = set_scan(b, len(sos) - 1, ah=2, al=1)
    bad_al = set_scan(b, len(sos) - 1, al=14)
    i = b.index(b"\xff\xc2")
    sof10 = b[:i] + b"\xff\xca" + b[i + 2:]
    d = torch.empty((2, 24, 40, 3), dtype=torch.uint8, device="cuda")

    def call(files, flags=0):
        bufs = [np.frombuffer(x, np.uint8) for x in files]
        ptrs, lens = (C.c_void_p * 2)(*[x.ctypes.data for x in bufs]), (C.c_size_t * 2)(*[x.size for x in bufs])
        return ctx.lib.uwip_jpeg_decode_batch_ex(ctx.h, ptrs, lens, 2, d.data_ptr(), 40, 24, flags)

    assert call([base, b]) == 0
    ctx.synchronize()
    assert (d[1].cpu().numpy() == cv2_decode(b)).all() and (d[0].cpu().numpy() == cv2_decode(base)).all()
    assert [call([base, x]) for x in (incomplete, mismatch, sof10)] == [-3, -3, -3]
    assert call([base, bad_al]) == -1
    assert call([base, b], 4) == -1   # an unknown flag
    for x, rc in ((incomplete, -3), (mismatch, -3), (sof10, -3), (bad_al, -1)):
        with pytest.raises(UwipError) as e:
            ctx.jpeg_probe(x)
        assert e.value.status == rc
    # the existing readers and their defaults still refuse progressive files
    with pytest.raises(UwipError) as e:
        ctx.jpeg_decode([base, b])
    assert e.value.status == -3
    assert ctx.jpeg_probe(b) == (40, 24, 1, True) and ctx.jpeg_probe(base) == (40, 24, 1, False)


# ---- command lines ---------------------------------------------------------------------------------------------------
def _dir_files(n, w=160, h=96):
    out = {}
    for i in range(n):
        f = O.synth_frame(0x5EED0004, 60 + i, w if i != 4 else 128, h)
        out["f%d.jpg" % i] = (cv2_prog(f, 95, "420"), imencode(f, 95, "420"), pil_prog(f, 90, "444"), cv2_prog(f, 80, "422", 7))[i % 4]
    return out


def test_chain_cli_mixed_directory(ctx, tmp_path):
    from uwimageproc_b200.cli import chain

    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    dst.mkdir()
    files = _dir_files(9)
    files["r6.jpg"] = tag(cv2_prog(O.synth_frame(0x5EED0004, 90, 96, 160), 95, "420"), 6)
    for name, b in files.items():
        (src / name).write_bytes(b)
    for exif in (False, True):
        args = ["-decoder=exact", "-encoder=exact", "-batch=3"] + (["-orientation=exif"] if exif else [])
        assert chain.main([str(src), str(dst)] + args) == 0
        for name, b in files.items():
            d_in = ctx.jpeg_decode_batch_dev(b, orientation=exif, progressive=True)
            d_out = d_in.clone()
            n, h, w = d_in.shape[:3]
            ctx.chain_dev(d_in, d_out, n, w, h)
            assert (dst / name).read_bytes() == ctx.jpeg_encode_batch_dev(d_out, 95)[0], name
            assert (dst / name).read_bytes() == bytes(cv2.imencode(".jpg", ctx.chain(cv2_decode(b, orient=exif)))[1]), name


def test_aclahe_cli_mixed_directory(ctx, tmp_path):
    from uwimageproc_b200.cli import aclahe as cli
    from uwimageproc_b200.modules import aclahe as A

    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    dst.mkdir()
    files = _dir_files(6)
    for name, b in files.items():
        (src / name).write_bytes(b)
    assert cli.main([str(src), str(dst), "-grey=1", "-device=1", "-batch=4"]) == 0
    for name, b in files.items():
        g = ctx.jpeg_decode_grey(b, progressive=True)
        out, bs, cl = A.main_batch(g[None])
        assert (g == cv2_decode(b, grey=True)).all()
        assert (dst / name).read_bytes() == bytes(cv2.imencode(".jpg", out[0], [cv2.IMWRITE_JPEG_QUALITY, 95])[1]), name
