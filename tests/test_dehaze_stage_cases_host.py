"""The constructed frames of tests/test_gpu_dehaze_stages.py, checked on the CPU with the oracle: each one must have the
property its GPU test relies on (a load path of the window pass, a tie of the background-light arg-min, a negative red
coefficient, a NaN or finite reference output), so that the GPU tests cannot pass vacuously.  CPU only."""
import numpy as np
import pytest

from oracle import uwip_oracle as O


def _cdiv(a, b):
    return -(-a // b)


# ---- window pass (window15_kernel, csrc/dehaze.cu) ---------------------------------------------------------------------
WF_TX, WF_TY, WF_R, WF_VR = 64, 32, 7, 8   # tile, half window, output rows per vertical run


def window15_regimes(W, H, align=0):
    """window15_kernel's choices for a W x H frame whose first byte sits `align` bytes past a 16-byte boundary: the load
    path of each tile (8-byte cp.async copies of rows that need no column clamp, aligned 32-bit words, single bytes) and
    whether a run of WF_VR output rows takes the FAST variant of wf_emit_rows (inside the frame, no window at a border)."""
    Wp = (W + 3) & ~3
    words = W % 4 == 0 and align % 4 == 0
    dwords = W % 8 == 0 and align % 8 == 0
    got = set()
    for bx in range(_cdiv(Wp, WF_TX)):
        x0 = bx * WF_TX
        if dwords and x0 >= 8 and x0 - 8 + 80 <= W:
            got.add("8-byte cp.async")
        elif words:
            got.add("32-bit words")
        else:
            got.add("bytes")
        for gx in range(x0, min(x0 + WF_TX, Wp)):
            xt = gx < WF_R or gx + WF_R >= W
            for gy0 in range(0, H, WF_VR):
                fast = not xt and gy0 >= WF_R and gy0 + WF_VR - 1 + WF_R < H
                got.add("FAST" if fast else "!FAST")
    for k, name in ((-1, "64k-1"), (0, "64k"), (1, "64k+1")):
        if W > WF_TX and (W - k) % WF_TX == 0:
            got.add("W = " + name)
    for k, name in ((-1, "32k-1"), (0, "32k"), (1, "32k+1")):
        if H > WF_TY and (H - k) % WF_TY == 0:
            got.add("H = " + name)
    if W < 15 or H < 15:
        got.add("frame smaller than the window")
    if W < WF_TX and H < WF_TY:
        got.add("frame smaller than a tile")
    return got


# (W, H) of the 15x15 window tests
WINDOW15_SHAPES = [
    (192, 96),    # W % 8 = 0: cp.async for the interior tile, words for the edge tiles; 64k x 32k
    (136, 63),    # W % 8 = 0, one interior tile ending on the last column; 32k-1
    (200, 130),   # W % 8 = 0, two interior tiles
    (260, 65),    # W % 8 = 4: words everywhere; 32k+1
    (191, 95),    # bytes; 64k-1 x 32k-1
    (193, 97),    # bytes; 64k+1 x 32k+1
    (1, 1), (1, 37), (45, 1), (7, 7), (8, 15), (14, 16), (15, 15), (16, 14),
]
WINDOW15_REGIMES = ["8-byte cp.async", "32-bit words", "bytes", "FAST", "!FAST", "W = 64k-1", "W = 64k", "W = 64k+1",
                    "H = 32k-1", "H = 32k", "H = 32k+1", "frame smaller than the window", "frame smaller than a tile"]

# generic window_kernel (-w other than 15): windows and ragged shapes, some smaller than the window
GENERIC_WINDOWS = [1, 2, 3, 4, 14, 16, 32, 33]
GENERIC_SHAPES = [(67, 45), (131, 33), (10, 6), (1, 5), (33, 34)]


def random_frame(seed, W, H):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def frame_of_range(W, H, lo, rng, seed=1):
    """A synthetic underwater frame requantised to the bytes lo..lo+rng (kmin = lo > 0 and kmax < 255 unless lo = 0)."""
    fr = O.synth_frame(0x5EED0007, seed, W, H).astype(np.int64)
    a, b = fr.min(), fr.max()
    return (lo + (fr - a) * rng // max(b - a, 1)).astype(np.uint8)


# ---- background-light arg-min ties ---------------------------------------------------------------------------------------
def _blocks(W, H, fill, blocks):
    """Frame of colour `fill` with constant blocks (y0, y1, x0, x1, (b, g, r)) whose channels are all at least fill's; the
    blocks lie more than a window apart, so every pixel within 7 of a block has the block's window maxima."""
    fr = np.empty((H, W, 3), np.uint8)
    fr[:] = fill
    for y0, y1, x0, x1, bgr in blocks:
        fr[y0:y1, x0:x1] = bgr
    return fr


def tie_plateaus(rng):
    """Blocks of one integer difference max_R - max_B (= max_R - max_G - 1) in four tiles of a 200 x 100 frame of range
    `rng` (255 or 7).  a/rng - b/rng with equal a - b differs in the last bits: the fp64 minimum is in the third block (the
    fourth has the same value), not in the first block in flat order.  The fill's difference is larger and its blue and
    green are not 0, so B (the fill at the selected pixels) is not 0 either."""
    if rng == 255:
        d, r, fill = 50, (15, 205, 131, 130), (10, 9, 0)   # r = 130, 131: the smallest r/255 - (r + 50)/255; 205: kmax 255
    else:
        d, r, fill = 2, (0, 5, 3, 3), (1, 1, 0)            # r = 3: the smallest r/7 - (r + 2)/7; r = 5 makes kmax 7
    at = ((5, 15, 10, 20), (5, 15, 150, 160), (40, 50, 130, 140), (70, 80, 20, 30))   # tiles (0,0), (2,0), (2,1), (0,2)
    return _blocks(200, 100, fill, [(y0, y1, x0, x1, (rr + d, rr + d - 1, rr)) for (y0, y1, x0, x1), rr in zip(at, r)])


def tie_tiles():
    """Equal fp64 minima in tiles (0,0), (1,0) and (0,1) of a 150 x 70 frame: the window maxima of one block reach rows
    1.. in tile (1,0), rows 11.. in tile (0,0) (an earlier tile, later rows) and rows 37.. in tile (0,1).  The first flat
    index, row 1 column 73, must win."""
    bgr = (180, 179, 130)
    fr = _blocks(150, 70, (10, 9, 0), [(8, 13, 80, 111, bgr), (18, 25, 10, 21, bgr), (44, 57, 10, 41, bgr)])
    fr[66, 145] = 255
    return fr


TIE_TILES_IDX = 1 * 150 + 73


def integer_candidates(fr):
    """Flat indices of the pixels whose integer window difference max_R - max_B (and max_R - max_G) is the frame's
    smallest: the first step of window15_kernel's arg-min."""
    mx = [O._window_reduce(fr[..., c].astype(np.int64), 15, np.maximum, 0) for c in range(3)]
    out = []
    for c in (0, 1):
        d = (mx[2] - mx[c]).ravel()
        out.append(np.flatnonzero(d == d.min()))
    return out


# ---- red channel and degenerate frames (147 x 83: W % 4 = 3) --------------------------------------------------------------
RC_W, RC_H = 147, 83


def rc_negative_avg(W=RC_W, H=RC_H):
    """Blue and green bright almost everywhere: mean(restored blue) + mean(restored green) > 1.5, so avgRr and the red
    coefficient are negative and build_red_tables swaps the ends of the red range."""
    fr = np.empty((H, W, 3), np.uint8)
    fr[..., 0], fr[..., 1] = 200, 210
    fr[..., 2] = (np.arange(W)[None, :] * 3 % 90 + 20).astype(np.uint8)
    fr[40:46, 70:76, :2] = 5
    return fr


def rc_red_at_kmin(W=RC_W, H=RC_H):
    """Red at the frame's minimum everywhere: mean_r = 0, the coefficient is infinite and restored red 0 * inf = NaN."""
    fr = O.synth_frame(0x5EED0004, 3, W, H).copy()
    fr[..., 2] = fr.min()
    return fr


def rc_red_constant(W=RC_W, H=RC_H):
    """Red constant above the minimum: rmax == rmin, restored red is 0/0."""
    fr = O.synth_frame(0x5EED0004, 3, W, H).copy()
    fr[..., 2] = fr.min() + 40
    return fr


def pad_case(W, H, f):
    """A synthetic frame with three pixels set to its minimum: the joint YCrCb minima of I8 and R8 are both 0 while no
    pixel has both lumas at 0 (R8 reaches 0 on Cr only), so the exposure ratio S is finite everywhere."""
    fr = O.synth_frame(0x5EED0004, f, W, H).copy()
    rng = np.random.default_rng(f)
    ys, xs = rng.integers(0, H, 3), rng.integers(0, W, 3)
    fr[ys, xs] = fr.min()
    return fr


# (W, H, frame, radius): W % 4 != 0, so the packed planes have pad columns
PAD_CASES = [(147, 83, 18, 40), (101, 61, 14, 7)]


def d9_frame(W=RC_W, H=RC_H):
    """A black block in a synthetic frame: S = 0/0 where both lumas are at their minimum (SURVEY 8a-D9)."""
    fr = O.synth_frame(0x5EED0004, 0, W, H).copy()
    fr[30:50, 60:80] = 0
    return fr


def two_level(W=RC_W, H=RC_H):
    fr = np.full((H, W, 3), 93, np.uint8)
    fr[:, 60:] = (30, 200, 120)
    return fr


def mixed_batch():
    """(name, frame, the reference output has a NaN) of one W % 4 != 0 batch."""
    return [
        ("normal", O.synth_frame(0x5EED0004, 1, RC_W, RC_H), False),
        ("constant", np.full((RC_H, RC_W, 3), 93, np.uint8), True),
        ("d9", d9_frame(), True),
        ("avgRr<0", rc_negative_avg(), False),
        ("red at kmin", rc_red_at_kmin(), True),
        ("red constant", rc_red_constant(), True),
        ("pad", pad_case(RC_W, RC_H, 18), False),
        ("two-level", two_level(), False),
    ]


def exposure_bytes(fr, r=40):
    """(reference output, YCrCb of I8, YCrCb of R8, stages) of adaptiveExp_map (BGDehaze.py:75-78)."""
    st = {}
    with np.errstate(invalid="ignore", divide="ignore"):
        out, _ = O.bgdehaze_frame(fr, 15, st, r=r)
        R8 = (st["restored"] * 255).astype(np.uint8)
    I8 = (O.normalize_frame(fr) * 255).astype(np.uint8)
    return out, O.bgr2ycrcb(I8), O.bgr2ycrcb(R8), st


# ---- the premises ------------------------------------------------------------------------------------------------------------
def test_window15_shapes_reach_every_path():
    seen = set()
    for W, H in WINDOW15_SHAPES:
        seen |= window15_regimes(W, H)
    missed = [x for x in WINDOW15_REGIMES if x not in seen]
    assert not missed, missed


def test_window15_regimes_follow_the_alignment():
    """A frame of a batch starts f * W * H * 3 bytes into the buffer: a W % 8 == 0 frame at an odd offset takes the byte
    path, at an offset of 4 the word path."""
    assert window15_regimes(192, 96, 1) & {"8-byte cp.async", "32-bit words"} == set()
    assert "32-bit words" in window15_regimes(192, 96, 4) and "8-byte cp.async" not in window15_regimes(192, 96, 4)


def test_generic_shapes_include_frames_smaller_than_the_window():
    assert any(W < max(GENERIC_WINDOWS) and H < max(GENERIC_WINDOWS) for W, H in GENERIC_SHAPES)
    assert any(W % 4 != 0 for W, H in GENERIC_SHAPES) and any(w % 2 == 0 for w in GENERIC_WINDOWS)


@pytest.mark.parametrize("rng", [255, 7])
def test_tie_plateaus_are_ties(rng):
    fr = tie_plateaus(rng)
    assert fr.min() == 0 and fr.max() == rng
    B, idx = O.background_light(O.normalize_frame(fr), 15, True)
    assert B[0] > 0 and B[1] > 0
    for c, cand in enumerate(integer_candidates(fr)):
        tiles = {(int(i) % 200 // 64, int(i) // 200 // 32) for i in cand}
        assert len(tiles) >= 3, tiles
        assert idx[c] in cand, (c, idx[c])
    # max_R - max_B: the winner is the first pixel of the third block's window (row 33, column 123), not the first
    # integer-minimum pixel
    assert idx[0] == 33 * 200 + 123 != integer_candidates(fr)[0][0]


def test_tie_tiles_first_flat_index():
    fr = tie_tiles()
    normI = O.normalize_frame(fr)
    B, idx = O.background_light(normI, 15, True)
    assert idx == (TIE_TILES_IDX, TIE_TILES_IDX) and B[0] > 0 and B[1] > 0
    mx = [O._window_reduce(normI[..., c], 15, np.maximum, 0.0) for c in range(3)]
    d = mx[2] - mx[0]
    at = np.argwhere(d == d.min())
    tiles = {(int(x) // 64, int(y) // 32) for y, x in at}
    assert {(0, 0), (1, 0), (0, 1)} <= tiles and (at[:, 0] * 150 + at[:, 1]).min() == TIE_TILES_IDX


def test_low_range_frames():
    for lo, rng in ((0, 1), (37, 1), (100, 2), (7, 3), (0, 5), (60, 8)):
        fr = frame_of_range(93, 41, lo, rng)
        assert fr.min() == lo and fr.max() == lo + rng


def test_negative_red_coefficient():
    fr = rc_negative_avg()
    st = {}
    out, _ = O.bgdehaze_frame(fr, 15, st)
    nb, ng = st["restored"][..., 0], st["restored"][..., 1]
    assert 1.5 - nb.mean() - ng.mean() < 0
    assert np.isfinite(out).all()


@pytest.mark.parametrize("W,H,f,r", PAD_CASES)
def test_pad_reproducers(W, H, f, r):
    assert W % 4 != 0
    out, Yi, Yj, _ = exposure_bytes(pad_case(W, H, f), r)
    assert Yi.min() == 0 and Yj.min() == 0
    assert not ((Yi[..., 0] == 0) & (Yj[..., 0] == 0)).any()
    assert Yj[..., 0].min() > 0     # Yj reaches 0 on Cr only
    assert np.isfinite(out).all()
    # the same frame cropped to a multiple of 4 columns is finite too: nothing but the pad columns could flag it
    crop = pad_case(W, H, f)[:, : W & ~3]
    assert np.isfinite(exposure_bytes(crop, r)[0]).all()


def test_mixed_batch_expectations():
    for name, fr, nan in mixed_batch():
        assert fr.shape == (RC_H, RC_W, 3) and RC_W % 4 != 0
        with np.errstate(invalid="ignore", divide="ignore"):
            out, _ = O.bgdehaze_frame(fr, 15)
        assert bool(np.isnan(out).any()) == nan, name
