"""The batched device JPEG encoder (uwip_jpeg_encode_bgr8_batch_dev, csrc/jpegenc.cu): every file byte-identical to
cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q]) across batch sizes, odd sizes, qualities, 4K synthetic frames and the
chain's own output; a frame's bytes independent of its batch; refusals; and `chain -encoder=exact`."""
import os

import cv2
import numpy as np
import pytest

from oracle import uwip_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
QUALITIES = [1, 10, 50, 75, 90, 95, 100]
SIZES = [(1, 1), (1, 29), (23, 1), (7, 9), (8, 8), (15, 17), (16, 16), (17, 16), (53, 37), (481, 270)]   # (w, h)


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _cv2(f, q):
    ok, b = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return bytes(b)


def _frame(kind, w, h, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == 0:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        return np.stack([xx * 255 // max(w - 1, 1), yy * 255 // max(h - 1, 1), ((xx + yy) * 7) % 256], -1).astype(np.uint8)
    if kind == 2:
        return np.full((h, w, 3), (0, 128, 255)[seed % 3], np.uint8)
    if kind == 3:
        cols = np.array([[0, 0, 255], [0, 255, 0], [255, 0, 0], [255, 255, 255], [0, 0, 0]], np.uint8)
        return cols[((xx // 3) + (yy // 5) + seed) % len(cols)]
    return O.synth_frame(0x5EED0004, seed, w, h)


def _mixed(n, w, h, seed=0):
    return np.stack([_frame(i % 5, w, h, seed + i) for i in range(n)])


def _check(got, frames, q):
    assert len(got) == len(frames)
    bad = [i for i, (g, f) in enumerate(zip(got, frames)) if g != _cv2(f, q)]
    assert not bad, "q=%d: frames %s of %d differ from cv2.imencode" % (q, bad[:10], len(frames))


@pytest.mark.parametrize("n", [1, 3, 149])
@pytest.mark.parametrize("q", [75, 95])
def test_mixed_batch_equals_cv2(ctx, n, q):
    frames = _mixed(n, 53, 37, seed=n)
    _check(ctx.jpeg_encode(frames, q), frames, q)


@pytest.mark.parametrize("q", QUALITIES)
def test_sizes_and_qualities(ctx, q):
    for (w, h) in SIZES:
        frames = _mixed(5, w, h, seed=w * 131 + h)
        _check(ctx.jpeg_encode(frames, q), frames, q)


def test_full_hd_golden_frame(ctx):
    img = np.load(os.path.join(GOLD, "k3_pis_full.npz"))["PIS_T1A_259/full"]
    for q in (75, 95):
        assert ctx.jpeg_encode(img, q) == _cv2(img, q)


@pytest.mark.parametrize("q", [50, 95, 100])
def test_synthetic_4k(ctx, q):
    import torch

    n, w, h = 3, 3840, 2160
    d = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d, 0x5EED0004, 7, n, w, h)
    ctx.synchronize()
    _check(ctx.jpeg_encode_batch_dev(d, q), d.cpu().numpy(), q)


@pytest.mark.parametrize("auto", [False, True])
def test_chain_output_encodes_like_cv2(ctx, auto):
    import torch

    n, w, h = 4, 640, 360
    d_in = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    d_out = torch.empty_like(d_in)
    ctx.synth_dev(d_in, 0x5EED0004, 0, n, w, h)
    if auto:
        ctx.chain_auto_dev(d_in, d_out, n, w, h)
    else:
        ctx.chain_dev(d_in, d_out, n, w, h)
    got = ctx.jpeg_encode_batch_dev(d_out, 95)
    ctx.synchronize()
    _check(got, d_out.cpu().numpy(), 95)


def test_batch_split_independence(ctx):
    import torch

    frames = _mixed(11, 97, 45, seed=3)
    d = torch.from_numpy(frames).to("cuda")
    whole = ctx.jpeg_encode_batch_dev(d, 90)
    parts = ctx.jpeg_encode_batch_dev(d[:4], 90) + ctx.jpeg_encode_batch_dev(d[4:5], 90) + ctx.jpeg_encode_batch_dev(d[5:], 90)
    singles = [ctx.jpeg_encode_batch_dev(d[i], 90)[0] for i in range(len(frames))]
    assert whole == parts == singles
    _check(whole, frames, 90)


def test_refusals(ctx):
    import torch

    from uwimageproc_b200 import UwipError

    w, h = 33, 20
    bound = ctx.jpeg_encode_bound(w, h)
    assert bound > 0
    assert ctx.jpeg_encode_bound(0, 5) == 0 and ctx.jpeg_encode_bound(5, 65536) == 0 and ctx.jpeg_encode_bound(65535, 1) > 0
    d = torch.zeros((2, h, w, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((2, bound), dtype=torch.uint8, device="cuda")
    lens = torch.zeros(2, dtype=torch.int64, device="cuda")
    lib = ctx.lib

    def call(width=w, height=h, q=95, stride=bound, n=2):
        return lib.uwip_jpeg_encode_bgr8_batch_dev(ctx.h, d.data_ptr(), n, width, height, q, out.data_ptr(), stride, lens.data_ptr())

    assert call(stride=bound - 1) == -1
    assert call(q=0) == -1 and call(q=101) == -1
    assert call(width=0) == -1 and call(height=0) == -1 and call(width=65536) == -1 and call(height=70000) == -1
    assert call(n=0) == -1
    assert lib.uwip_jpeg_encode_bgr8_batch_dev(ctx.h, d.data_ptr(), 2, w, h, 95, None, bound, lens.data_ptr()) == -1
    assert call() == 0
    ctx.synchronize()
    assert lens.cpu().tolist() == [len(_cv2(np.zeros((h, w, 3), np.uint8), 95))] * 2
    with pytest.raises(UwipError):
        ctx.jpeg_encode(np.zeros((h, w, 3), np.uint8), 0)


@pytest.mark.parametrize("auto", [False, True])
def test_cli_exact_encoder(ctx, tmp_path, auto):
    """`chain in.jpg out.jpg -encoder=exact` writes cv2.imencode of the chain's output on the pixels nvJPEG decoded."""
    from uwimageproc_b200.cli import chain

    fr = O.synth_frame(0x5EED0004, 5, 320, 180)
    src, dst = tmp_path / "in.jpg", tmp_path / "out.jpg"
    src.write_bytes(_cv2(fr, 95))
    args = [str(src), str(dst), "-encoder=exact"] + (["-aclahe=auto"] if auto else [])
    assert chain.main(args) == 0
    dec = ctx.jpeg_decode_dev(src.read_bytes()).cpu().numpy()
    want = ctx.chain_auto(dec)[0] if auto else ctx.chain(dec)
    assert dst.read_bytes() == _cv2(want, 95)
    # other formats go through cv2.imwrite whatever the encoder
    png_a, png_b = tmp_path / "a.png", tmp_path / "b.png"
    assert chain.main([str(src), str(png_a), "-encoder=exact"]) == 0
    assert chain.main([str(src), str(png_b)]) == 0
    assert png_a.read_bytes() == png_b.read_bytes()
    assert chain.main([str(src), str(dst), "-encoder=libjpeg"]) == -1
