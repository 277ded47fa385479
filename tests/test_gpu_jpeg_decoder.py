"""The batched device JPEG decoder (uwip_jpeg_decode_bgr8_batch, csrc/jpegdec.cu): every frame equal to
cv2.imdecode(file, IMREAD_COLOR) across batch sizes that mix sampling, quality, restart interval and optimised tables, every
size of the host matrix, 4K frames, the golden frame and streams that stress the subsequence synchronisation; a frame's pixels
independent of its batch; a truncated file in the middle of a batch; refusals; and `chain -decoder=exact`."""
import os

import cv2
import numpy as np
import pytest

from oracle import uwip_oracle as O
from test_jpeg_decoder_host import SIZES, imencode
from test_jpeg_encoder_host import contents

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
MIX = [("420", []), ("444", [cv2.IMWRITE_JPEG_RST_INTERVAL, 1]), ("422", [cv2.IMWRITE_JPEG_OPTIMIZE, 1]),
       ("440", [cv2.IMWRITE_JPEG_RST_INTERVAL, 7]), ("grey", []), ("420", [cv2.IMWRITE_JPEG_RST_INTERVAL, 3, cv2.IMWRITE_JPEG_OPTIMIZE, 1])]


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _file(i, w, h, seed):
    kinds = list(contents(w, h, seed).values()) + [O.synth_frame(0x5EED0004, seed % 97, w, h)]
    f = kinds[i % len(kinds)]
    s, extra = MIX[i % len(MIX)]
    q = (1, 50, 95, 100)[(i // len(MIX)) % 4]
    if s == "grey":
        return imencode(cv2.cvtColor(f, cv2.COLOR_BGR2GRAY), q, None, extra)
    return imencode(f, q, s, extra)


def _want(files):
    return np.stack([cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR) for b in files])


def _check(got, files):
    want = _want(files)
    assert got.shape == want.shape
    bad = [i for i in range(len(files)) if not (got[i] == want[i]).all()]
    assert not bad, "frames %s of %d differ from cv2.imdecode" % (bad[:10], len(files))


@pytest.mark.parametrize("n", [1, 3, 149])
def test_mixed_batch_equals_cv2(ctx, n):
    files = [_file(i, 53, 37, 100 + i) for i in range(n)]
    _check(ctx.jpeg_decode(files), files)
    assert not ctx.last_frame_flags(n).any()


def test_every_size(ctx):
    for (w, h) in SIZES + [(4, 3), (5, 4)]:
        files = [_file(i, w, h, 7 * w + h + i) for i in range(2 * len(MIX))]
        _check(ctx.jpeg_decode(files), files)


@pytest.mark.parametrize("q", [50, 95, 100])
def test_synthetic_4k(ctx, q):
    frames = [O.synth_frame(0x5EED0004, i, 3840, 2160) for i in range(3)]
    files = [imencode(f, q, "420") for f in frames]
    _check(ctx.jpeg_decode(files), files)


def test_golden_frame(ctx):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    files = [imencode(img, 95, "420"), imencode(img, 75, "444"), imencode(img, 90, "422", [cv2.IMWRITE_JPEG_RST_INTERVAL, 5])]
    _check(ctx.jpeg_decode(files), files)


def test_sync_stress(ctx):
    """Constant frames (every block a DC and an EOB: the shortest codewords) and quality-100 noise (the longest)."""
    rng = np.random.default_rng(5)
    w, h = 1280, 720
    frames = [np.full((h, w, 3), v, np.uint8) for v in (0, 128, 255)] + [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(3)]
    files = [imencode(f, 100 if i >= 3 else 95, s) for i, f in enumerate(frames) for s in ("420", "444")]
    _check(ctx.jpeg_decode(files), files)
    st = ctx.jpeg_decode_stats(len(files))
    assert (st >= 0).all()


def test_batch_split_independence(ctx):
    files = [_file(i, 97, 45, 3 + i) for i in range(11)]
    whole = ctx.jpeg_decode(files)
    parts = np.concatenate([ctx.jpeg_decode(files[:4]), ctx.jpeg_decode(files[4:5]), ctx.jpeg_decode(files[5:])])
    singles = np.stack([ctx.jpeg_decode(b) for b in files])
    assert (whole == parts).all() and (whole == singles).all()
    _check(whole, files)


def test_truncated_file_in_a_batch(ctx):
    frames = [O.synth_frame(0x5EED0004, i, 160, 96) for i in range(5)]
    files = [imencode(f, 95, "420") for f in frames]
    cut = files[2][:len(files[2]) * 2 // 3]
    batch = files[:2] + [cut] + files[3:]
    got = ctx.jpeg_decode(batch)
    flags = ctx.last_frame_flags(5)
    assert flags.tolist() == [0, 0, 4, 0, 0]
    assert not got[2].any()
    keep = [0, 1, 3, 4]
    _check(got[keep], [batch[i] for i in keep])


def test_refusals(ctx):
    import ctypes as C

    import torch

    from uwimageproc_b200 import UwipError

    f = O.synth_frame(0x5EED0004, 0, 40, 24)
    base = imencode(f, 90, "420")
    ok, prog = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    with pytest.raises(UwipError) as e:
        ctx.jpeg_decode([base, bytes(prog)])
    assert e.value.status == -3
    s411 = imencode(f, 90, None, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])
    with pytest.raises(UwipError) as e:
        ctx.jpeg_decode([s411])
    assert e.value.status == -3
    other = imencode(O.synth_frame(0x5EED0004, 0, 41, 24), 90, "420")
    with pytest.raises(UwipError) as e:
        ctx.jpeg_decode([base, other])   # one size per call
    assert e.value.status == -1
    lib = ctx.lib
    buf = np.frombuffer(base, np.uint8)
    d = torch.empty((1, 24, 40, 3), dtype=torch.uint8, device="cuda")
    ptrs, lens = (C.c_void_p * 1)(buf.ctypes.data), (C.c_size_t * 1)(buf.size)
    assert lib.uwip_jpeg_decode_bgr8_batch(ctx.h, ptrs, lens, 0, d.data_ptr(), 40, 24) == -1
    assert lib.uwip_jpeg_decode_bgr8_batch(ctx.h, ptrs, lens, 1, None, 40, 24) == -1
    assert lib.uwip_jpeg_decode_bgr8_batch(ctx.h, ptrs, lens, 1, d.data_ptr(), 40, 25) == -1
    assert lib.uwip_jpeg_decode_bgr8_batch(ctx.h, None, lens, 1, d.data_ptr(), 40, 24) == -1
    assert lib.uwip_jpeg_decode_bgr8_batch(ctx.h, ptrs, lens, 1, d.data_ptr(), 40, 24) == 0
    ctx.synchronize()
    assert (d[0].cpu().numpy() == cv2.imdecode(buf, cv2.IMREAD_COLOR)).all()


def _cv2_route(ctx, src_bytes, auto, q=95):
    img = cv2.imdecode(np.frombuffer(src_bytes, np.uint8), cv2.IMREAD_COLOR)
    out = ctx.chain_auto(img)[0] if auto else ctx.chain(img)
    ok, b = cv2.imencode(".jpg", out, [cv2.IMWRITE_JPEG_QUALITY, q])
    return bytes(b)


@pytest.mark.parametrize("auto", [False, True])
def test_cli_exact_decoder_and_encoder(ctx, tmp_path, auto):
    """`chain in.jpg out.jpg -decoder=exact -encoder=exact` writes cv2.imencode(chain(cv2.imdecode(in)))."""
    from uwimageproc_b200.cli import chain

    src, dst = tmp_path / "in.jpg", tmp_path / "out.jpg"
    src.write_bytes(imencode(O.synth_frame(0x5EED0004, 5, 320, 180), 95, "420"))
    args = [str(src), str(dst), "-decoder=exact", "-encoder=exact"] + (["-aclahe=auto"] if auto else [])
    assert chain.main(args) == 0
    assert dst.read_bytes() == _cv2_route(ctx, src.read_bytes(), auto)
    assert chain.main([str(src), str(dst), "-decoder=libjpeg"]) == -1


def test_cli_default_flags_unchanged(ctx, tmp_path):
    """Without -decoder the file is what uwip_chain_jpeg (nvJPEG in and out) writes, as before."""
    from uwimageproc_b200.cli import chain

    src, dst = tmp_path / "in.jpg", tmp_path / "out.jpg"
    src.write_bytes(imencode(O.synth_frame(0x5EED0004, 6, 320, 180), 95, "420"))
    assert chain.main([str(src), str(dst)]) == 0
    assert dst.read_bytes() == ctx.chain_jpeg(src.read_bytes(), quality=95)
    assert chain.main([str(src), str(dst), "-decoder=nvjpeg"]) == 0
    assert dst.read_bytes() == ctx.chain_jpeg(src.read_bytes(), quality=95)


@pytest.mark.parametrize("opts", [["-decoder=exact", "-encoder=exact"], ["-decoder=exact", "-encoder=exact", "-aclahe=auto"], []])
def test_cli_directory_equals_per_file_runs(ctx, tmp_path, opts):
    from uwimageproc_b200.cli import chain

    src, dst, one = tmp_path / "src", tmp_path / "dst", tmp_path / "one"
    for d in (src, dst, one):
        d.mkdir()
    sizes = [(160, 96), (160, 96), (97, 45), (160, 96), (97, 45)]
    for i, (w, h) in enumerate(sizes):
        (src / ("f%d.jpg" % i)).write_bytes(imencode(O.synth_frame(0x5EED0004, 20 + i, w, h), 90, ("420", "444")[i % 2]))
    (src / "notes.txt").write_text("not an image")
    assert chain.main([str(src), str(dst), "-batch=2"] + opts) == 0
    assert sorted(os.listdir(dst)) == ["f%d.jpg" % i for i in range(len(sizes))]
    for i in range(len(sizes)):
        name = "f%d.jpg" % i
        assert chain.main([str(src / name), str(one / name)] + opts) == 0
        assert (dst / name).read_bytes() == (one / name).read_bytes(), name
        if opts:
            assert (dst / name).read_bytes() == _cv2_route(ctx, (src / name).read_bytes(), "-aclahe=auto" in opts, 95)
