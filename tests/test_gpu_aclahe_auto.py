"""Automatic CLAHE parameters on the device (uwip_aclahe_params_u8_dev, uwip_aclahe_bgr8_auto_dev, uwip_chain_bgr8_auto_dev)
against the oracle's ParametrosACLAHE (scipy knee search) and against the fixed-parameter entry points called per frame
with the reported (BS, CL)."""
import os
import warnings

import numpy as np
import pytest

from oracle import uwip_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
H, W = 180, 320
NOFIT = 2


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def _oracle_params(plane):
    """(BS, CL) of the oracle, (-1, -1) where its curve fit raises."""
    try:
        bs, cl, _ = O.parametros_aclahe(plane)
        return bs, cl
    except RuntimeError:
        return -1, -1


def _grey_noise_frame(seed):
    g = np.random.default_rng(seed).integers(0, 256, (H, W), dtype=np.uint8)
    return np.stack([g, g, g], -1)   # V stays uniform noise through histretch: the fit fails (maxfev)


def _planes():
    rng = np.random.default_rng(3)
    crowd = np.load(os.path.join(GOLD, "crowd_full.npz"))["img"][200:200 + H, 300:300 + W]
    yy, xx = np.mgrid[0:H, 0:W]
    grad = ((xx * 255) // (W - 1) * 0.7 + (yy * 255) // (H - 1) * 0.3).astype(np.uint8)
    noise6 = np.clip(rng.normal(120, 6, (H, W)).round(), 0, 255).astype(np.uint8)
    uni = rng.integers(0, 256, (H, W), dtype=np.uint8)
    synth = O.bgr2hsv(O.synth_frame(0x5EED0004, 6, W, H))[..., 2].copy()
    return np.stack([crowd, grad, noise6, uni, synth])


def _params_dev(ctx, planes, loop="repaired"):
    import torch

    d = torch.from_numpy(np.ascontiguousarray(planes)).cuda()
    torch.cuda.synchronize()
    bs, cl = ctx.aclahe_params_dev(d, d.shape[0], d.shape[2], d.shape[1], loop)
    ctx.synchronize()
    return bs.cpu().numpy(), cl.cpu().numpy()


def test_crowd_golden(ctx):
    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    img = z["img"][None]
    bs, cl = _params_dev(ctx, img, "repaired")
    assert (bs[0], cl[0]) == tuple(z["repaired"]) == (4, 7)
    bs, cl = _params_dev(ctx, img, "as_committed")
    assert (bs[0], cl[0]) == tuple(z["as_committed"]) == (8, 0)
    assert ctx.last_frame_flags(1)[0] == 0


def test_mixed_batch_matches_oracle_and_single_planes(ctx):
    planes = _planes()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = [_oracle_params(p) for p in planes]
    assert (-1, -1) in want and len(set(want)) >= 3, want
    bs, cl = _params_dev(ctx, planes)
    flags = ctx.last_frame_flags(len(planes))
    assert list(zip(bs.tolist(), cl.tolist())) == want
    assert [int(f) for f in flags] == [NOFIT if w[1] < 0 else 0 for w in want]
    for i, p in enumerate(planes):
        b1, c1 = _params_dev(ctx, p[None])
        assert (b1[0], c1[0]) == (bs[i], cl[i]), i
    # the module-level convenience returns the same
    from uwimageproc_b200.modules.aclahe import parametros_aclahe_batch

    b2, c2 = parametros_aclahe_batch(planes)
    assert (b2 == bs).all() and (c2 == cl).all()


def test_too_small_is_refused(ctx):
    import uwimageproc_b200 as u
    import torch

    d = torch.zeros((1, 10, 10), dtype=torch.uint8, device="cuda")   # reflect-101 cannot pad 10 pixels to 32 tiles
    with pytest.raises(u.UwipError):
        ctx.aclahe_params_dev(d, 1, 10, 10)


def test_auto_frame_entry(ctx):
    import torch

    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in (3, 6)] + [_grey_noise_frame(1)])
    n = len(frames)
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    d_bs = torch.empty(n, dtype=torch.int32, device="cuda")
    d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.aclahe_auto_dev(d_in, d_out, n, W, H, clip=3.0, tiles=(4, 6), d_bs=d_bs, d_cl=d_cl)
    ctx.synchronize()
    got, bs, cl = d_out.cpu().numpy(), d_bs.cpu().numpy(), d_cl.cpu().numpy()
    flags = ctx.last_frame_flags(n)
    assert cl[2] == -1 and bs[2] == -1 and flags[2] == NOFIT
    for i in range(n):
        v = O.bgr2hsv(frames[i])[..., 2]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            assert _oracle_params(v) == (bs[i], cl[i]), i
        clip, tiles = (float(cl[i]), (int(bs[i]),) * 2) if cl[i] >= 0 else (3.0, (4, 6))
        one = torch.empty_like(d_in[i:i + 1])
        ctx.aclahe_dev(d_in[i:i + 1], one, 1, W, H, clip, tiles)
        ctx.synchronize()
        assert (one.cpu().numpy()[0] == got[i]).all(), i
        assert (O.aclahe_frame(frames[i], clip, tiles[0], tiles[1]) == got[i]).all(), i


@pytest.mark.parametrize("channels", ["V", "VS"])
def test_auto_chain(ctx, channels):
    import torch

    # synth frame 5 carries the D9 NaN pattern of the fixed chain; the grey noise frame fails the fit
    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in (3, 5, 6)] + [_grey_noise_frame(2)])
    n = len(frames)
    p = ctx.chain_params(channels=channels, clip=2.5, tiles=(8, 4))
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    d_bs = torch.empty(n, dtype=torch.int32, device="cuda")
    d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.chain_auto_dev(d_in, d_out, n, W, H, p, "repaired", d_bs, d_cl)
    flags = ctx.last_frame_flags(n)
    got, bs, cl = d_out.cpu().numpy(), d_bs.cpu().numpy(), d_cl.cpu().numpy()
    assert cl[3] == -1 and flags[3] & NOFIT
    for i in range(n):
        v = O.bgr2hsv(O.histretch_frame(frames[i], channels, 1, 99))[..., 2]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            assert _oracle_params(v) == (bs[i], cl[i]), i
        clip, tiles = (float(cl[i]), (int(bs[i]),) * 2) if cl[i] >= 0 else (2.5, (8, 4))
        q = ctx.chain_params(channels=channels, clip=clip, tiles=tiles)
        one = torch.empty_like(d_in[i:i + 1])
        ctx.chain_dev(d_in[i:i + 1], one, 1, W, H, q)
        f1 = ctx.last_frame_flags(1)
        assert (one.cpu().numpy()[0] == got[i]).all(), i
        assert (flags[i] & 1) == (f1[0] & 1), i          # D9 flag as the fixed chain with the same parameters
        assert bool(flags[i] & NOFIT) == (cl[i] < 0), i
    # a frame's bytes do not depend on the batch it is in
    d_out2 = torch.empty_like(d_in)
    ctx.chain_auto_dev(d_in[1:], d_out2[1:], n - 1, W, H, p)
    ctx.synchronize()
    assert (d_out2[1:].cpu().numpy() == got[1:]).all()
    # host-array convenience
    out, bs2, cl2 = ctx.chain_auto(frames, p)
    assert (out == got).all() and (bs2 == bs).all() and (cl2 == cl).all()


def test_auto_chain_d9_flag_kept(ctx):
    """The NaN frame of the fixed chain test stays flagged when it is the frame the automatic chain finds NaN."""
    frames = np.stack([O.synth_frame(0x5EED0004, i, W, H) for i in range(3, 8)])
    out, bs, cl = ctx.chain_auto(frames)
    flags = ctx.last_frame_flags(len(frames))
    for i, fr in enumerate(frames):
        b = O.aclahe_frame(O.histretch_frame(fr, "V", 1, 99), float(cl[i]), int(bs[i]), int(bs[i]))
        ref, ref8 = O.bgdehaze_frame(b, 15)
        assert bool(flags[i] & 1) == bool(np.isnan(ref).any()), i
        assert np.abs(out[i].astype(int) - ref8.astype(int)).max() <= 1


def test_params_4k_against_scipy_on_sweep_tables(ctx):
    """At 3840 x 2160 the oracle's sweep is too slow: the knee and float16 pick are computed with scipy from the existing
    clahe_entropy_sweep_dev tables of the same blurred V planes."""
    import torch

    Hk, Wk = 2160, 3840
    n = 2
    d = torch.empty((n, Hk, Wk, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d, 0x5EED0004, 40, n, Wk, Hk)
    ctx.synchronize()
    v = d.max(dim=3).values.contiguous()
    torch.cuda.synchronize()
    bs, cl = _params_dev(ctx, v.cpu().numpy())
    vb = torch.from_numpy(np.stack([ctx.gaussian_blur3(p) for p in v.cpu().numpy()])).cuda()
    torch.cuda.synchronize()
    grids = [2, 4, 8, 16, 32]
    clips = np.arange(0, 25, 0.5)
    ent = ctx.clahe_entropy_sweep_dev(vb, n, Wk, Hk, grids, clips, "py")
    xs = clips.astype(np.float32)[1:50]
    for i in range(n):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want_cl = max(O._aclahe_knee(xs, ent[i, g, 1:50]) for g in range(5))
        assert cl[i] == want_cl, i
        pick = np.array([ctx.clahe_entropy_sweep_dev(vb[i:i + 1], 1, Wk, Hk, [k], [float(want_cl)], "py")[0, 0, 0] for k in grids],
                        np.float16)
        assert bs[i] == grids[int(np.flatnonzero(pick == pick.max())[-1])], i
