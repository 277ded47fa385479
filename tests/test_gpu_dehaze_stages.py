"""bgdehaze (csrc/dehaze.cu, gfmarch.cuh) stage by stage against the fp64 oracle: the window pass with its three load paths
and the generic window, the background-light arg-min and its ties, the red-channel tables, each stage of the exposure
branch against its own device inputs (uwip_exposure_stages_bgr8), and mixed batches of degenerate frames at unaligned
device offsets.  The constructed frames are checked on the CPU by test_dehaze_stage_cases_host.py."""
import numpy as np
import pytest

from oracle import uwip_oracle as O
from test_dehaze_stage_cases_host import (GENERIC_SHAPES, GENERIC_WINDOWS, PAD_CASES, TIE_TILES_IDX, WINDOW15_SHAPES, frame_of_range,
                                          mixed_batch, pad_case, random_frame, rc_negative_avg, rc_red_at_kmin, rc_red_constant,
                                          tie_plateaus, tie_tiles)

pytestmark = pytest.mark.gpu

PSCALE = 2.0 ** 28   # the S plane holds rint(S 2^28) (GP_PSCALE)


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


def rel_err(got, want):
    """The bar of the float stages: |got - want| / max(|want|, 1e-3)."""
    return float((np.abs(got - want) / np.maximum(np.abs(want), 1e-3)).max())


def check_window(ctx, fr, tag, window=15):
    """B within 1e-15 and the arg-min indices equal; with the 15x15 window also t_raw within 1e-14.
    Where B_c = 0 the reference's t_raw is 0/0 and the whole output NaN: the frame must come out flagged (all zeros), and
    t_raw of that channel is not compared - the device divides the window minimum of the bytes, so at border pixels it has
    0/0 where the reference's zero padding gives min(0, k/0) = 0."""
    normI = O.normalize_frame(fr)
    B, idx = ctx.background_light(fr, window)
    with np.errstate(invalid="ignore", divide="ignore"):
        Bo, idxo = O.background_light(normI, window, True)
    assert idx == idxo, (tag, window, idx, idxo)
    assert np.abs(B - Bo).max() < 1e-15, (tag, window)
    if window == 15:
        tb, tg = ctx.transmission(fr)
        with np.errstate(invalid="ignore", divide="ignore"):
            t = O.transmission_map(normI, 15, Bo)
        for c, got in enumerate((tb, tg)):
            if Bo[c] == 0:
                assert ctx.bgdehaze(fr).max() == 0, (tag, "B_c = 0 frame not flagged")
                continue
            assert np.abs(got - t[..., c]).max() < 1e-14, (tag, c)
    return idx


def check_bytes(ctx, fr, tag, window=15, radius=40):
    with np.errstate(invalid="ignore", divide="ignore"):
        ref, ref8 = O.bgdehaze_frame(fr, window, r=radius)
    got = ctx.bgdehaze(fr, ctx.dehaze_params(window=window, radius=radius))
    if np.isnan(ref).any():
        assert got.max() == 0, tag
    else:
        assert np.abs(got.astype(int) - ref8.astype(int)).max() <= 1, tag


# ---- a. window pass, background light, transmission --------------------------------------------------------------------
@pytest.mark.parametrize("W,H", WINDOW15_SHAPES)
def test_window15_shapes(ctx, W, H):
    check_window(ctx, O.synth_frame(0x5EED0003, 1, W, H), "synth")
    check_window(ctx, random_frame(W * 1000 + H, W, H), "random")


@pytest.mark.parametrize("W,H", GENERIC_SHAPES)
def test_generic_windows(ctx, W, H):
    fr = O.synth_frame(0x5EED0003, 2, W, H)
    for w in GENERIC_WINDOWS:
        check_window(ctx, fr, (W, H), w)
        check_window(ctx, random_frame(w, W, H), (W, H, "random"), w)


@pytest.mark.parametrize("window", [2, 33])
def test_generic_window_bytes(ctx, window):
    """dehazed_BG's J takes the generic window's B, the transmission the 15x15 window's Bt (BGDehaze.py:51-52)."""
    check_bytes(ctx, O.synth_frame(0x5EED0003, 5, 131, 77), window, window)


@pytest.mark.parametrize("rng", [255, 7])
def test_argmin_plateaus(ctx, rng):
    """The fp64 minimum among the pixels of the smallest integer difference is not the first of them."""
    check_window(ctx, tie_plateaus(rng), rng)


def test_argmin_equal_minima_across_tiles(ctx):
    assert check_window(ctx, tie_tiles(), "tiles") == (TIE_TILES_IDX, TIE_TILES_IDX)


@pytest.mark.parametrize("lo,rng", [(0, 1), (37, 1), (100, 2), (7, 3), (60, 8), (3, 200)])
def test_window_low_ranges(ctx, lo, rng):
    """kmin > 0, kmax < 255 and ranges 1..3: the k' = k - kmin bias and the 1/range table of the window pass."""
    fr = frame_of_range(197, 70, lo, rng)
    check_window(ctx, fr, (lo, rng))
    check_window(ctx, fr, (lo, rng), 4)


def test_host_pitch_wider_than_the_row(ctx):
    """Host frames that are views of a wider array: the staging copy honours the pitch."""
    W, H = 131, 57
    fr = O.synth_frame(0x5EED0003, 6, W, H)
    wide = np.zeros((H, W + 13, 3), np.uint8)
    wide[:, 5:5 + W] = fr
    view = wide[:, 5:5 + W]
    assert view.strides[0] == (W + 13) * 3 and not view.flags.c_contiguous
    assert check_window(ctx, view, "view") == check_window(ctx, fr, "contiguous")
    assert (ctx.bgdehaze(view) == ctx.bgdehaze(fr)).all()
    assert (ctx.rc_correction(view) == ctx.rc_correction(fr)).all()


# ---- b. red-channel correction ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [rc_negative_avg, rc_red_at_kmin, rc_red_constant])
def test_red_channel_tables(ctx, case):
    fr = case()
    with np.errstate(invalid="ignore", divide="ignore"):
        want = O.rc_correction(O.normalize_frame(fr))
        ref, _ = O.bgdehaze_frame(fr, 15)
    got = ctx.rc_correction(fr)
    assert (np.isnan(got) == np.isnan(want)).all(), case.__name__
    ok = ~np.isnan(want)
    assert np.abs(got[ok] - want[ok]).max() < 1e-5, case.__name__
    xs = ctx.exposure_stages(fr)
    assert bool(xs["nan_flag"]) == bool(np.isnan(ref).any()), case.__name__
    check_bytes(ctx, fr, case.__name__)


# ---- c. the exposure branch, each stage against its own device inputs ----------------------------------------------------
def check_exposure(ctx, fr, tag, r=40, eps=1e-3):
    xs = ctx.exposure_stages(fr, ctx.dehaze_params(radius=r, eps=eps))
    normI = O.normalize_frame(fr)
    with np.errstate(invalid="ignore", divide="ignore"):
        ref, _ = O.bgdehaze_frame(fr, 15, r=r, eps=eps)
        want_rest = O.rc_correction(normI, 15, r=r, eps=eps)
    flagged = bool(np.isnan(ref).any())
    assert bool(xs["nan_flag"]) == flagged, (tag, "D9 flag", xs["nan_flag"])
    rest = xs["restored"]
    assert (np.isnan(rest) == np.isnan(want_rest)).all(), tag
    ok = ~np.isnan(want_rest)
    assert np.abs(rest[ok] - want_rest[ok]).max() < 1e-5, (tag, "restored")
    # I8, R8 and their YCrCb (BGDehaze.py:75-78): bytes, exact
    ycc = xs["ycc"].astype(np.int64)
    with np.errstate(invalid="ignore"):
        I8 = (normI * 255).astype(np.uint8)
        R8 = (rest * 255).astype(np.uint8)
    Yi, Yj = O.bgr2ycrcb(I8).astype(np.int64), O.bgr2ycrcb(R8).astype(np.int64)
    for c, name in enumerate(("Yi", "Cri", "Cbi")):
        bad = np.argwhere(ycc[..., c] != Yi[..., c])
        assert not len(bad), (tag, name, bad[:4])
    bad = np.argwhere(ycc[..., 3] != Yj[..., 0])
    assert not len(bad), (tag, "Yj", bad[:4])
    assert (xs["yi_min"], xs["yi_max"]) == (Yi.min(), Yi.max()), (tag, "yi range")
    assert (xs["yj_min"], xs["yj_max"]) == (Yj.min(), Yj.max()), (tag, "yj range")
    if flagged:
        assert np.isnan(xs["out"]).all(), tag
        return xs
    # S (BGDehaze.py:83) in fp64 on the device's bytes and ranges, held as rint(S 2^28) (both round half to even).  The
    # device fuses 0.3 yi^2 into the two sums; that moves S by an ulp and rint(S 2^28) only within 2^-24 of a half, which
    # none of the (Yi', Yj') pairs of these frames is
    yi = (ycc[..., 0] - xs["yi_min"]) / float(xs["yi_max"] - xs["yi_min"])
    yj = (ycc[..., 3] - xs["yj_min"]) / float(xs["yj_max"] - xs["yj_min"])
    S = (yj * yi + 0.3 * yi ** 2) / (yj ** 2 + 0.3 * yi ** 2)
    assert np.isfinite(S).all(), tag
    want_sp = np.rint(np.minimum(S, 1.6) * PSCALE).astype(np.uint32)
    bad = np.argwhere(xs["splane"] != want_sp)
    assert not len(bad), (tag, "S plane", bad[:4], xs["splane"][tuple(bad[0])] if len(bad) else None)
    # refined S (BGDehaze.py:85): the guided filter of the device's S plane guided by its YCrCb bytes
    nYi = (ycc[..., :3] - xs["yi_min"]) / float(xs["yi_max"] - xs["yi_min"])
    q = O.guided_filter(nYi, xs["splane"] / PSCALE, r, eps)
    err = rel_err(xs["refined_s"].astype(np.float64), q)
    assert err < 1e-5, (tag, "refined S", err)
    # final min-max normalisation (BGDehaze.py:86-89) of the device's restored x refined S
    o = rest * xs["refined_s"].astype(np.float64)[..., None]
    want_out = (o - o.min()) / (o.max() - o.min())
    assert np.abs(xs["out"] - want_out).max() < 1e-12, (tag, "final map")
    # bytes: sat(rint(255 x that)), except within 1e-9 of a .5 boundary
    got8 = ctx.bgdehaze(fr, ctx.dehaze_params(radius=r, eps=eps)).astype(np.int64)
    v = want_out * 255.0
    sure = np.abs(v - np.floor(v) - 0.5) > 1e-9
    want8 = np.clip(np.rint(v), 0, 255).astype(np.int64)
    bad = np.argwhere((got8 != want8) & sure)
    assert not len(bad), (tag, "bytes", bad[:4])
    return xs


@pytest.mark.parametrize("W,H", [(160, 90), (161, 91), (162, 67), (163, 75)])
def test_exposure_stages_synth(ctx, W, H):
    check_exposure(ctx, O.synth_frame(0x5EED0003, 7, W, H), (W, H))


def test_exposure_stages_golden_frames(ctx):
    import os

    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "dehaze_literal.npz"))
    for name in sorted({k.split("/")[0] for k in z.files}):
        check_exposure(ctx, z[name + "/frame"], name)


@pytest.mark.parametrize("rng", [2, 3, 5, 8])
def test_exposure_stages_low_contrast(ctx, rng):
    """Ranges 2 and 3 make reference outputs that are NaN (S = 0/0): the flag, the bytes and YCrCb planes are checked."""
    check_exposure(ctx, frame_of_range(141, 63, 40, rng, seed=rng), rng)


@pytest.mark.parametrize("r", [7, 40])
def test_exposure_stages_radii(ctx, r):
    check_exposure(ctx, O.synth_frame(0x5EED0003, 8, 203, 119), r, r=r)


@pytest.mark.parametrize("W,H,f,r", PAD_CASES)
def test_exposure_pad_columns_do_not_flag(ctx, W, H, f, r):
    """W % 4 != 0 and both joint YCrCb minima 0: the pad entries of the packed planes look like (Yi', Yj') = (0, 0), where
    S is 0/0.  The reference is finite, so the frame must not be flagged."""
    xs = check_exposure(ctx, pad_case(W, H, f), (W, H, f), r=r)
    assert xs["yi_min"] == 0 and xs["yj_min"] == 0


# ---- d. degenerate and mixed batches through bgdehaze_dev ---------------------------------------------------------------
def _run_dev(ctx, frames, offset=0):
    """The frames as one batch at `offset` bytes into device buffers -> (bytes, flags)."""
    import torch

    n, H, W = frames.shape[:3]
    nb = frames.nbytes
    d_src = torch.zeros(nb + 16, dtype=torch.uint8, device="cuda")
    d_dst = torch.full((nb + 16,), 77, dtype=torch.uint8, device="cuda")
    d_src[offset:offset + nb] = torch.from_numpy(frames.reshape(-1)).cuda()
    torch.cuda.synchronize()
    ctx.bgdehaze_dev(d_src.data_ptr() + offset, d_dst.data_ptr() + offset, n, W, H)
    ctx.synchronize()
    flags = ctx.last_frame_flags(n)
    out = d_dst.cpu().numpy()
    assert (out[:offset] == 77).all() and (out[offset + nb:] == 77).all(), "write outside the frames"
    return out[offset:offset + nb].reshape(frames.shape), flags


def test_mixed_batch(ctx):
    cases = mixed_batch()
    frames = np.stack([fr for _, fr, _ in cases])
    got, flags = _run_dev(ctx, frames)
    for i, (name, fr, nan) in enumerate(cases):
        with np.errstate(invalid="ignore", divide="ignore"):
            ref, ref8 = O.bgdehaze_frame(fr, 15)
        assert bool(np.isnan(ref).any()) == nan, name
        assert bool(flags[i] & 1) == nan, (name, flags[i])
        if nan:
            assert got[i].max() == 0, name
        else:
            assert np.abs(got[i].astype(int) - ref8.astype(int)).max() <= 1, name
        one, f1 = _run_dev(ctx, frames[i:i + 1])
        assert (one[0] == got[i]).all() and f1[0] == flags[i], name
    for off in (1, 3, 4, 8):
        g, f = _run_dev(ctx, frames, off)
        assert (g == got).all() and (f == flags).all(), off


def test_aligned_width_batch_offsets(ctx):
    """W % 8 == 0: minmax_kernel's 16-byte loads, window15_kernel's cp.async and word paths and final_kernel's word stores
    depend on the alignment of each frame; every offset gives the same bytes."""
    W, H = 200, 70
    frames = np.stack([O.synth_frame(0x5EED0003, f, W, H) for f in (9, 10, 11)])
    got, flags = _run_dev(ctx, frames)
    for i in range(len(frames)):
        ref, ref8 = O.bgdehaze_frame(frames[i], 15)
        assert bool(flags[i] & 1) == bool(np.isnan(ref).any()), i
        assert np.abs(got[i].astype(int) - ref8.astype(int)).max() <= 1, i
    for off in (1, 3, 4, 8):
        g, f = _run_dev(ctx, frames, off)
        assert (g == got).all() and (f == flags).all(), off
