"""The oriented device JPEG readers (uwip_jpeg_decode_bgr8_batch_oriented, uwip_jpeg_decode_u8_batch_oriented): every frame
equal to cv2.imdecode(file, IMREAD_COLOR) / cv2.imdecode(file, IMREAD_GRAYSCALE) with the Exif orientation applied, in
batches that mix orientations 1 to 8 (stored landscape for 1..4, stored portrait for 5..8), samplings and byte orders; 4K at
the rotating orientations; bad data inside an oriented batch; batch-split independence; the size refusal; untagged files
read alike by both readers; and `chain` / `aclahe` with -orientation=exif."""
import os

import cv2
import numpy as np
import pytest

from oracle import uwip_oracle as O
from test_jpeg_decoder_host import imencode
from test_jpeg_orientation_host import cv2_decode, frame, tag

pytestmark = pytest.mark.gpu
MIX = [("420", []), ("444", [cv2.IMWRITE_JPEG_RST_INTERVAL, 1]), ("422", [cv2.IMWRITE_JPEG_OPTIMIZE, 1]), ("440", []), ("grey", []),
       ("420", [cv2.IMWRITE_JPEG_RST_INTERVAL, 3])]


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _plain(i, w, h):
    """an untagged w x h file of the mix"""
    f = frame(w, h, 100 + i)
    s, extra = MIX[i % len(MIX)]
    return imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), 90, None, extra) if s == "grey" else imencode(f, (50, 95)[i % 2], s, extra)


def _file(i, w, h, o=None):
    """file i of a batch whose output is w x h: orientation o (default 1 + i % 8), stored h x w for 5..8"""
    o = 1 + i % 8 if o is None else o
    return tag(_plain(i, h, w) if o >= 5 else _plain(i, w, h), o, le=(i // 8) % 2 == 0)


def _check(ctx, files, grey):
    got = (ctx.jpeg_decode_grey if grey else ctx.jpeg_decode)(files, orientation=True)
    want = np.stack([cv2_decode(b, grey) for b in files])
    assert got.shape == want.shape
    bad = [i for i in range(len(files)) if not (got[i] == want[i]).all()]
    assert not bad, "frames %s of %d differ from cv2.imdecode" % (bad[:10], len(files))
    assert not ctx.last_frame_flags(len(files)).any()


@pytest.mark.parametrize("grey", [False, True], ids=["bgr8", "u8"])
@pytest.mark.parametrize("n", [1, 3, 149])
def test_mixed_orientations_equal_cv2(ctx, n, grey):
    files = [_file(i, 53, 37, 6 if n == 1 else None) for i in range(n)]
    _check(ctx, files, grey)


@pytest.mark.parametrize("grey", [False, True], ids=["bgr8", "u8"])
def test_4k_rotated(ctx, grey):
    f = O.synth_frame(0x5EED0004, 3, 2160, 3840)   # stored portrait: 3840 x 2160 once turned
    b = imencode(f, 95, "420")
    files = [tag(b, 6), tag(b, 8, le=False)]
    _check(ctx, files, grey)
    assert ctx.jpeg_size(files[0]) == (3840, 2160) and ctx.jpeg_size(files[0], orientation=False) == (2160, 3840)


def test_bad_data_in_an_oriented_batch(ctx):
    files = [_file(i, 96, 64) for i in range(8)]
    cut = files[5][:len(files[5]) * 2 // 3]   # orientation 6: stored 64 x 96
    batch = files[:5] + [cut] + files[6:]
    keep = [0, 1, 2, 3, 4, 6, 7]
    for grey in (False, True):
        got = (ctx.jpeg_decode_grey if grey else ctx.jpeg_decode)(batch, orientation=True)
        assert ctx.last_frame_flags(8).tolist() == [0, 0, 0, 0, 0, 4, 0, 0]
        assert got.shape[1:3] == (64, 96) and not got[5].any()
        assert all((got[i] == cv2_decode(batch[i], grey)).all() for i in keep)


def test_batch_split_independence(ctx):
    files = [_file(i, 97, 45) for i in range(11)]
    for grey in (False, True):
        dec = ctx.jpeg_decode_grey if grey else ctx.jpeg_decode
        whole = dec(files, orientation=True)
        parts = np.concatenate([dec(files[:4], orientation=True), dec(files[4:5], orientation=True), dec(files[5:], orientation=True)])
        singles = np.stack([dec(b, orientation=True) for b in files])
        assert (whole == parts).all() and (whole == singles).all()


def test_size_refusal(ctx):
    import ctypes as C

    import torch

    from uwimageproc_b200 import UwipError

    land, port = imencode(frame(40, 24, 1), 90, "420"), imencode(frame(24, 40, 2), 90, "420")
    with pytest.raises(UwipError) as e:   # 24 x 40 stored, orientation 1: not 40 x 24
        ctx.jpeg_decode([tag(land, 3), tag(port, 1)], orientation=True)
    assert e.value.status == -1 and "file 1 is 24 x 40" in str(e.value)
    with pytest.raises(UwipError) as e:   # 40 x 24 stored, orientation 6: 24 x 40
        ctx.jpeg_decode_grey([tag(land, 1), tag(land, 6)], orientation=True)
    assert e.value.status == -1 and "file 1 is 40 x 24 with Exif orientation 6" in str(e.value)
    files = [tag(land, 2), tag(port, 7)]
    bufs = [np.frombuffer(b, np.uint8) for b in files]
    ptrs, lens = (C.c_void_p * 2)(*[b.ctypes.data for b in bufs]), (C.c_size_t * 2)(*[b.size for b in bufs])
    d = torch.empty((2, 24, 40, 3), dtype=torch.uint8, device="cuda")
    assert ctx.lib.uwip_jpeg_decode_bgr8_batch_oriented(ctx.h, ptrs, lens, 2, d.data_ptr(), 24, 40) == -1
    assert ctx.lib.uwip_jpeg_decode_bgr8_batch_oriented(ctx.h, ptrs, lens, 2, d.data_ptr(), 40, 24) == 0
    ctx.synchronize()
    assert all((d[i].cpu().numpy() == cv2_decode(files[i])).all() for i in range(2))
    ok, prog = cv2.imencode(".jpg", frame(40, 24, 1), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    with pytest.raises(UwipError) as e:
        ctx.jpeg_decode([tag(land, 1), tag(bytes(prog), 3)], orientation=True)
    assert e.value.status == -3


def test_untagged_files_read_alike(ctx):
    files = [_plain(i, 53, 37) for i in range(12)]
    assert all(ctx.jpeg_orientation(b) == 1 for b in files)
    for grey in (False, True):
        dec = ctx.jpeg_decode_grey if grey else ctx.jpeg_decode
        assert (dec(files) == dec(files, orientation=True)).all()


# ---- command lines ---------------------------------------------------------------------------------------------------
def _cv2_chain_route(ctx, src_bytes, q=95):
    out = ctx.chain(cv2_decode(src_bytes))
    return bytes(cv2.imencode(".jpg", out, [cv2.IMWRITE_JPEG_QUALITY, q])[1])


def _tagged(i, o, w=160, h=96):
    sw, sh = (h, w) if o >= 5 else (w, h)
    return tag(imencode(O.synth_frame(0x5EED0004, 40 + i, sw, sh), 95, ("420", "444")[i % 2]), o, le=i % 2 == 0)


def test_chain_cli_exif(ctx, tmp_path):
    from uwimageproc_b200.cli import chain

    exact = ["-decoder=exact", "-encoder=exact", "-orientation=exif"]
    src, dst = tmp_path / "in.jpg", tmp_path / "out.jpg"
    src.write_bytes(_tagged(0, 6))
    assert chain.main([str(src), str(dst)] + exact) == 0
    assert dst.read_bytes() == _cv2_chain_route(ctx, src.read_bytes())
    assert cv2.imread(str(dst)).shape == (96, 160, 3)
    assert chain.main([str(src), str(dst), "-orientation=exif"]) == -1                       # nvJPEG does not read Exif
    assert chain.main([str(src), str(dst), "-decoder=nvjpeg", "-orientation=exif"]) == -1
    assert chain.main([str(src), str(dst), "-decoder=exact", "-orientation=upright"]) == -1
    # the default keeps the stored orientation: the bytes of the run without the flag
    assert chain.main([str(src), str(dst), "-decoder=exact", "-encoder=exact"]) == 0
    stored = bytes(cv2.imencode(".jpg", ctx.chain(cv2_decode(src.read_bytes(), ignore=True)), [cv2.IMWRITE_JPEG_QUALITY, 95])[1])
    assert dst.read_bytes() == stored
    assert chain.main([str(src), str(dst), "-decoder=exact", "-encoder=exact", "-orientation=ignore"]) == 0
    assert dst.read_bytes() == stored
    assert chain.main([str(src), str(dst)]) == 0
    assert dst.read_bytes() == ctx.chain_jpeg(src.read_bytes(), quality=95)


def test_chain_cli_exif_directory(ctx, tmp_path):
    from uwimageproc_b200.cli import chain

    exact = ["-decoder=exact", "-encoder=exact", "-orientation=exif"]
    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    dst.mkdir()
    orients = [1, 6, 3, 8, 5, 2, 7, 4, 1]
    for i, o in enumerate(orients):
        (src / ("f%d.jpg" % i)).write_bytes(_tagged(i, o))
    (src / "g.jpg").write_bytes(_tagged(20, 1, 97, 45))
    assert chain.main([str(src), str(dst), "-batch=4"] + exact) == 0
    for name in sorted(os.listdir(src)):
        assert (dst / name).read_bytes() == _cv2_chain_route(ctx, (src / name).read_bytes()), name


def test_aclahe_cli_exif(ctx, tmp_path):
    from uwimageproc_b200.cli import aclahe as cli
    from uwimageproc_b200.modules import aclahe as A

    def want(path):
        g = cv2.imread(str(path), 0)   # the host route's reader: orientation applied
        out, bs, cl = A.main_batch(g[None])
        return bytes(cv2.imencode(".jpg", out[0], [cv2.IMWRITE_JPEG_QUALITY, 95])[1]), int(bs[0]), int(cl[0])

    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    dst.mkdir()
    for i, o in enumerate([6, 1, 8, 3]):
        (src / ("p%d.jpg" % i)).write_bytes(_tagged(30 + i, o))
    one = tmp_path / "one.jpg"
    assert cli.main([str(src / "p0.jpg"), str(one), "-grey=1", "-device=1", "-orientation=exif"]) == 0
    w0 = want(src / "p0.jpg")
    assert one.read_bytes() == w0[0] and cv2.imread(str(one), 0).shape == (96, 160)
    assert cli.main([str(src), str(dst), "-grey=1", "-device=1", "-orientation=exif", "-batch=3"]) == 0
    for name in sorted(os.listdir(src)):
        assert (dst / name).read_bytes() == want(src / name)[0], name
    assert cli.main([str(src / "p0.jpg"), str(one), "-grey=1", "-orientation=exif"]) == -1   # the flag needs -device=1
    assert cli.main([str(src / "p0.jpg"), str(one), "-grey=1", "-device=1", "-orientation=sideways"]) == -1
    # the default keeps the stored orientation, as before
    assert cli.main([str(src / "p0.jpg"), str(one), "-grey=1", "-device=1"]) == 0
    g = cv2.imread(str(src / "p0.jpg"), cv2.IMREAD_GRAYSCALE | cv2.IMREAD_IGNORE_ORIENTATION)
    out, bs, cl = A.main_batch(g[None])
    assert one.read_bytes() == bytes(cv2.imencode(".jpg", out[0], [cv2.IMWRITE_JPEG_QUALITY, 95])[1])
