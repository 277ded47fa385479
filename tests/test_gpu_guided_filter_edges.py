"""The guided-filter marches (csrc/gfpipe.cuh, gfmarch.cuh, dehaze_gf1a.cu) against the fp64 oracle at the edges of their
geometry and arithmetic: strip seams and a narrower last strip in both layouts, partial last quads (W % 4 != 0), vertical
segments down to a 1-row last one, frames smaller than the window, radii from 1 to 128, eps from 1e-6 to 1e-1, guide
ranges from 1 to 255, and the per-frame flags across batch splits and device sub-batches."""
import numpy as np
import pytest

from oracle import uwip_oracle as O

pytestmark = pytest.mark.gpu

OUT_TOL = 1.0 / 255.0   # final float map: 1 LSB of the 8-bit output (see test_gpu_parity.OUT_TOL)
NTR = {"wide": 152, "narrow": 128}   # quads of a strip that hold data: GP_NTR of dehaze.cu / dehaze_gf1a.cu (GP_NARROW)
MAXSW = 512                          # GP_MAXSW: output columns of a strip


def _cdiv(a, b):
    return -(-a // b)


def geometry(W, H, r, sms, n=1):
    """gf_geometry and gp_launch's choice of vertical segments (gfmarch.cuh), per layout: the wide one runs GF1b, GF2a, GF2b
    and GFq, the narrow one GF1a."""
    HL = (r + 3) & ~3
    out = {}
    for lay, ntr in NTR.items():
        strips = _cdiv(W, min(4 * (ntr - 1) - 2 * HL, MAXSW))
        SW = (_cdiv(W, strips) + 3) & ~3
        strips = _cdiv(W, SW)
        tasks, best, best_eff = strips * n, 1, 0.0
        for s in range(1, min(max(1, H // (4 * r + 2)), 64) + 1):
            sh = _cdiv(H, s)
            sc = _cdiv(H, sh)
            eff = (tasks * sc / (_cdiv(tasks * sc, sms) * sms)) * (sh / (sh + 2 * r))
            if eff > best_eff * 1.02:
                best_eff, best = eff, s
        seg_h = _cdiv(H, best)
        segs = _cdiv(H, seg_h)
        out[lay] = dict(strips=strips, SW=SW, last_strip=W - (strips - 1) * SW, segs=segs, last_seg=H - (segs - 1) * seg_h)
    return out


# (W, H, r): shapes chosen with geometry() on a 148-SM device (n = 1)
GEOMETRY_CASES = [
    (1283, 507, 5),    # 3 strips in both layouts, last one narrower; 23 segments of 23 rows, the last one 1 row
    (300, 211, 3),     # 15 segments, the last one 1 row
    (1029, 200, 1),    # W % 4 = 1, 3 strips, 29 segments
    (1030, 160, 2),    # W % 4 = 2
    (642, 250, 7),     # W % 4 = 2, 2 strips, 8 segments
    (641, 479, 40),    # the reference's radius: 2 strips in both layouts
    (530, 300, 63),
    (530, 260, 64),    # r >= 64, quad path
    (1001, 1100, 65),  # 3 strips, 4 segments
    (997, 651, 100),   # 3 wide / 4 narrow strips
    (777, 333, 128),   # the largest radius: 3 wide / 4 narrow strips
    (3, 2, 40),        # W <= 4, W < r, H < 2r + 1
    (90, 7, 40),       # H < 2r + 1
    (7, 90, 64),       # W < r
]


def regimes(W, H, r, sms):
    g = geometry(W, H, r, sms)
    got = set()
    for lay in NTR:
        if g[lay]["strips"] >= 2:
            got.add("2+ strips " + lay)
        if g[lay]["last_strip"] < g[lay]["SW"]:
            got.add("narrower last strip")
        if g[lay]["segs"] >= 2:
            got.add("2+ segments")
        if g[lay]["segs"] >= 2 and g[lay]["last_seg"] == 1:
            got.add("1-row last segment")
    got.add("W %% 4 = %d" % (W % 4))
    got.add("r % 4 = 0" if r % 4 == 0 else "r % 4 != 0")
    if r >= 64:
        got.add("r >= 64")
    if r == 128:
        got.add("r = 128")
    if W < r:
        got.add("W < r")
    if H < 2 * r + 1:
        got.add("H < 2r + 1")
    if W <= 4:
        got.add("W <= 4")
    return got


REGIMES = ["2+ strips wide", "2+ strips narrow", "narrower last strip", "W % 4 = 1", "W % 4 = 2", "W % 4 = 3", "r % 4 = 0",
           "r % 4 != 0", "r >= 64", "r = 128", "2+ segments", "1-row last segment", "W < r", "H < 2r + 1", "W <= 4"]


@pytest.fixture(scope="module")
def ctx():
    import uwimageproc_b200 as u

    c = u.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def rel_err(got, want):
    """The bar of the float stages: |got - want| / max(|want|, 1e-3)."""
    return float((np.abs(got - want) / np.maximum(np.abs(want), 1e-3)).max())


def guide_of_range(W, H, rng, seed=1):
    """A synthetic underwater frame requantised to bytes 0..rng (every level present on frames of a few hundred pixels)."""
    fr = O.synth_frame(0x5EED0007, seed, W, H).astype(np.int64)
    lo, hi = fr.min(), fr.max()
    return ((fr - lo) * rng // max(hi - lo, 1)).astype(np.uint8)


def signal(kind, W, H, seed=2):
    """p of the guided filter: the marches hold it on a 2^-28 grid in [0, 1.6]."""
    if kind == "zero":
        return np.zeros((H, W))
    if kind == "max":
        return np.full((H, W), 1.6)
    if kind == "step":
        p = np.zeros((H, W))
        p[:, W // 3:] = 1.6
        p[H // 2:, : W // 5] = 0.7
        return p
    return np.random.default_rng(seed).random((H, W)) * 1.6


def test_geometry_cases_reach_every_regime(sms):
    """The shapes of this file reach every strip and segment regime of the marches on this device."""
    seen = set()
    for W, H, r in GEOMETRY_CASES:
        seen |= regimes(W, H, r, sms)
    missed = [x for x in REGIMES if x not in seen]
    assert not missed, "regimes not reached on %d SMs: %s" % (sms, missed)


# ---- GF2a + GFq: uwip_guided_filter_u8 ---------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H,r", GEOMETRY_CASES)
def test_guided_filter_geometry(ctx, W, H, r):
    g = guide_of_range(W, H, 255)
    I = g / 255.0
    for kind in ("noise", "step"):
        p = signal(kind, W, H)
        err = rel_err(ctx.guided_filter_u8(g, 255, p, r, 1e-3), O.guided_filter(I, p, r, 1e-3))
        assert err < 1e-5, (kind, err)


@pytest.mark.parametrize("rng", [1, 2, 3, 17, 255])
@pytest.mark.parametrize("eps", [1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1])
def test_guided_filter_eps_and_guide_range(ctx, rng, eps):
    """coef_scale sets the fixed-point exponents of the stored a, b from eps and the guide range: small eps and
    low-contrast guides make the largest coefficients.  Two strips, ragged width, the scalar and the quad window paths.
    Below eps = 1e-3 the step of the stored b is too coarse for outputs near zero (a step edge of p): refused."""
    import uwimageproc_b200 as u

    W, H = 601, 203
    g = guide_of_range(W, H, rng)
    I = g / float(rng)
    for r, kind in ((5, "noise"), (8, "step")):
        p = signal(kind, W, H)
        if eps < 1e-3:
            with pytest.raises(u.UwipError) as e:
                ctx.guided_filter_u8(g, rng, p, r, eps)
            assert e.value.status == -1
            continue
        err = rel_err(ctx.guided_filter_u8(g, rng, p, r, eps), O.guided_filter(I, p, r, eps))
        assert err < 1e-5, (r, kind, err)
    if eps < 1e-3:
        with pytest.raises(u.UwipError) as e:
            ctx.bgdehaze(g, ctx.dehaze_params(radius=5, eps=eps))
        assert e.value.status == -1


@pytest.mark.parametrize("kind", ["zero", "max", "step", "noise"])
def test_guided_filter_signals(ctx, kind):
    """Constant p at both ends of the range (a = 0, b = p everywhere), a step edge and noise, across strip seams."""
    for W, H, r, rng in ((1283, 507, 5, 255), (997, 651, 100, 17), (90, 7, 40, 3)):
        g = guide_of_range(W, H, rng)
        p = signal(kind, W, H)
        err = rel_err(ctx.guided_filter_u8(g, rng, p, r, 1e-3), O.guided_filter(g / float(rng), p, r, 1e-3))
        assert err < 1e-5, (W, H, r, err)


def bright_guide(W, H, lo=245, seed=3):
    """k in lo..255 with a few black pixels: the moment sums of full windows come close to 2^32 at r = 128."""
    rs = np.random.default_rng(seed)
    g = rs.integers(lo, 256, (H, W, 3), dtype=np.uint8)
    g[rs.integers(0, H, 6), rs.integers(0, W, 6)] = 0
    return g


@pytest.mark.parametrize("r", [127, 128])
def test_guided_filter_bright_guide_largest_radius(ctx, r):
    W, H = 400, 400
    g = bright_guide(W, H)
    p = signal("noise", W, H)
    err = rel_err(ctx.guided_filter_u8(g, 255, p, r, 1e-3), O.guided_filter(g / 255.0, p, r, 1e-3))
    assert err < 1e-5, err


# ---- GF1a + GF1b: refined transmission ----------------------------------------------------------------------------------
def _refined_case(ctx, fr, r, eps, tmin):
    rb, rg = ctx.refined_transmission(fr, ctx.dehaze_params(radius=r, eps=eps, tmin=tmin))
    tb, tg = O.refined_t(O.normalize_frame(fr), 15, tmin, r, eps)
    return max(rel_err(rb, tb), rel_err(rg, tg))


@pytest.mark.parametrize("W,H,r", GEOMETRY_CASES)
def test_refined_transmission_geometry(ctx, W, H, r):
    fr = O.synth_frame(0x5EED0003, 2, W, H)
    for eps, tmin in ((1e-3, 0.2), (1e-3, 0.0)):
        err = _refined_case(ctx, fr, r, eps, tmin)
        assert err < 1e-5, (eps, tmin, err)


@pytest.mark.parametrize("tmin", [0.0, 0.2, 0.9])
def test_refined_transmission_tmin(ctx, tmin):
    """tmin = 0 lets t go below 0 where the frame is brighter than B throughout the window; 0.9 clips most of it."""
    fr = O.synth_frame(0x5EED0003, 6, 1283, 507)
    err = _refined_case(ctx, fr, 5, 1e-3, tmin)
    assert err < 1e-5, err


@pytest.mark.parametrize("rng", [2, 3, 5, 8])
def test_refined_transmission_low_contrast(ctx, rng):
    """A hazy frame: a synthetic frame requantised to a few levels (the transmission filters' guide range).  (At two
    levels the background light is 0 in every channel and the reference's transmission is 0/0 everywhere.)"""
    fr = guide_of_range(642, 250, rng, seed=4)
    err = _refined_case(ctx, fr, 7, 1e-3, 0.2)
    assert err < 1e-5, err


def test_refined_transmission_bright_frame_largest_radius(ctx):
    fr = bright_guide(400, 400)
    err = _refined_case(ctx, fr, 128, 1e-3, 0.2)
    assert err < 1e-5, err


# ---- all four marches: bgdehaze at other radius, eps and tmin --------------------------------------------------------
DEHAZE_CASES = [(1283, 507, 5, 1e-1, 0.1), (1001, 1100, 65, 1e-2, 0.3), (642, 250, 7, 1e-3, 0.0), (777, 333, 128, 1e-3, 0.2)]


@pytest.mark.parametrize("W,H,r,eps,tmin", DEHAZE_CASES)
def test_bgdehaze_other_parameters(ctx, W, H, r, eps, tmin):
    fr = O.synth_frame(0x5EED0003, 3, W, H)
    out, out8 = O.bgdehaze_frame(fr, 15, None, r, eps, tmin)
    got8, gotf = ctx.bgdehaze(fr, ctx.dehaze_params(radius=r, eps=eps, tmin=tmin), return_float=True)
    assert np.isnan(gotf).any() == np.isnan(out).any()
    if not np.isnan(out).any():
        assert np.abs(gotf - out).max() < OUT_TOL
    assert np.abs(got8.astype(int) - out8.astype(int)).max() <= 1


def test_bgdehaze_nan_flags_other_parameters(ctx):
    """D9 (S = 0/0 where Yi' = Yj' = 0 turns the frame NaN): the flags of a batch at r = 7 are exactly the oracle's NaN frames."""
    import torch

    W, H = 320, 180
    frames = np.stack([O.aclahe_frame(O.histretch_frame(O.synth_frame(0x5EED0004, i, W, H), "V", 1, 99), 2.0, 8, 8)
                       for i in range(3, 8)])   # frame 5 is a NaN frame at the default parameters
    p = ctx.dehaze_params(radius=7, eps=1e-2, tmin=0.1)
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    ctx.bgdehaze_dev(d_in, d_out, len(frames), W, H, p)
    ctx.synchronize()
    flags = ctx.last_frame_flags(len(frames))
    got = d_out.cpu().numpy()
    for i, fr in enumerate(frames):
        out, out8 = O.bgdehaze_frame(fr, 15, None, 7, 1e-2, 0.1)
        assert bool(flags[i] & 1) == bool(np.isnan(out).any()), i
        assert np.abs(got[i].astype(int) - out8.astype(int)).max() <= 1, i


# ---- a frame's bytes do not depend on the batch it is in ----------------------------------------------------------------
@pytest.mark.parametrize("W,H,r,n", [(300, 211, 3, 64), (1283, 507, 5, 64), (1001, 1100, 65, 16), (401, 1600, 128, 64)])
def test_split_independence_other_radii(ctx, sms, W, H, r, n):
    """Alone a frame is cut into more vertical segments than inside the batch: bytes and flags must not change."""
    import torch

    alone, batch = geometry(W, H, r, sms, 1), geometry(W, H, r, sms, n)
    assert any(alone[lay]["segs"] != batch[lay]["segs"] for lay in NTR), (alone, batch)
    p = ctx.dehaze_params(radius=r)
    d_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d_in, 0x5EED0008, 0, n, W, H)
    d_out = torch.empty_like(d_in)
    ctx.bgdehaze_dev(d_in, d_out, n, W, H, p)
    ctx.synchronize()
    whole = d_out.cpu().numpy()
    flags = np.asarray(ctx.last_frame_flags(n)).copy()
    for i in (0, n // 2, n - 1):
        one = torch.empty_like(d_in[i:i + 1])
        ctx.bgdehaze_dev(d_in[i:i + 1].contiguous(), one, 1, W, H, p)
        ctx.synchronize()
        assert (one.cpu().numpy()[0] == whole[i]).all(), i
        assert ctx.last_frame_flags(1)[0] == flags[i], i


def test_device_sub_batches(ctx, monkeypatch):
    """UWIP_WORKSPACE_GB=1 cuts 20 device-resident 1080p frames into sub-batches of at most 8 (60 B per pixel and frame):
    the bytes and the per-frame flags are those of the uncut batch."""
    import torch

    W, H, n = 1920, 1080, 20
    assert int(1e9 // (W * H * 60 + (512 << 10))) < n
    d_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d_in, 0x5EED0004, 0, n, W, H)
    res = {}
    for gb in (None, "1"):
        if gb is None:
            monkeypatch.delenv("UWIP_WORKSPACE_GB", raising=False)
        else:
            monkeypatch.setenv("UWIP_WORKSPACE_GB", gb)
        d_out = torch.empty_like(d_in)
        ctx.chain_dev(d_in, d_out, n, W, H)
        ctx.synchronize()
        res[gb] = (d_out.cpu().numpy(), np.asarray(ctx.last_frame_flags(n)).copy())
    monkeypatch.delenv("UWIP_WORKSPACE_GB", raising=False)
    assert (res[None][0] == res["1"][0]).all()
    assert (res[None][1] == res["1"][1]).all()
    assert res[None][1].any(), "no flagged frame among the 20: the flags' alignment is not tested"
