"""The knee search of ParametrosACLAHE in csrc/aclahe_knee.h (the code the GPU runs per frame and block size), compiled
with g++ for the host: same knee index as the oracle's scipy calls (curve_fit + splrep / splev + curvature argmax), same
success or failure of the fit, fitted parameters close to scipy's popt."""
import os
import shutil
import subprocess
import warnings

import numpy as np
import pytest

from oracle import uwip_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

KNEE_MAIN_SRC = r"""
#include <cstdio>
#include "aclahe_knee.h"
// stdin: lines of 49 floats (an entropy curve); stdout per line: knee nfev_y info_y p0 p1 p2 p3
int main() {
  double x1[knee::NE], x2[knee::NE], px[4];
  int nfx = 0;
  if (!knee::curve_derivs([] { static double x[knee::M]; for (int i = 0; i < knee::M; i++) x[i] = 0.5 * (i + 1); return x; }(),
                          x1, x2, px, &nfx)) { printf("xfit failed\n"); return 1; }
  printf("x %d %.17g %.17g %.17g %.17g\n", nfx, px[0], px[1], px[2], px[3]);
  float yf[knee::M];
  for (;;) {
    for (int i = 0; i < knee::M; i++) if (scanf("%f", &yf[i]) != 1) return 0;
    double y[knee::M], p[4];
    for (int i = 0; i < knee::M; i++) y[i] = yf[i];
    int nfev = 0;
    const int info = knee::fit(y, p, &nfev);
    printf("%d %d %d %.17g %.17g %.17g %.17g\n", knee::knee_of(yf, x1, x2), nfev, info, p[0], p[1], p[2], p[3]);
  }
}
"""


@pytest.fixture(scope="module")
def knee_exe(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("knee")
    src, exe = d / "knee.cpp", d / "knee"
    src.write_text(KNEE_MAIN_SRC)
    subprocess.run([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"),
                    str(src), "-o", str(exe)], check=True)
    return str(exe)


def _run(exe, curves):
    txt = "\n".join(" ".join("%.9g" % v for v in c) for c in curves) + "\n"
    out = subprocess.run([exe], input=txt, check=True, capture_output=True, text=True).stdout.split("\n")
    xline = out[0].split()
    rows = []
    for line in out[1:1 + len(curves)]:
        f = line.split()
        rows.append((int(f[0]), int(f[1]), int(f[2]), np.array([float(v) for v in f[3:7]])))
    return (int(xline[1]), np.array([float(v) for v in xline[2:6]])), rows


def _scipy(v):
    """curve_fit as the reference calls it: (knee or None, popt, nfev)."""
    from scipy.optimize import curve_fit

    def f(t, p0, p1, p2, p3):
        return p0 * np.exp(-p1 * t) + p2 * np.exp(-p3 * t)

    u = np.linspace(1, 49, 49)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            popt, _, info, _, _ = curve_fit(f, u, v, (7, 0.4, 0.9, 5), full_output=True)
        except RuntimeError:
            return False, None, None
    return True, popt, info["nfev"]


def _oracle_knee(row):
    """O._aclahe_knee on entries 1..49 of a 50-entry entropy row (None when scipy raises)."""
    cl = np.arange(0, 25, 0.5).astype(np.float32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return O._aclahe_knee(cl[1:50], row[1:50])
        except RuntimeError:
            return None


def _tables():
    """(name, [5][50] entropy table) of distinct planes: crowd.png (golden) and oracle sweeps of small planes."""
    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    out = [("crowd", z["entropies"], int(z["repaired"][1]))]
    rng = np.random.default_rng(7)
    crop = np.load(os.path.join(GOLD, "crowd_crop.npz"))["img"]
    yy, xx = np.mgrid[0:180, 0:320]
    grad = ((xx * 255) // 319 * 0.7 + (yy * 255) // 179 * 0.3).astype(np.uint8)
    noise6 = np.clip(rng.normal(120, 6, (180, 320)).round(), 0, 255).astype(np.uint8)
    uni = rng.integers(0, 256, (180, 320), dtype=np.uint8)
    for name, plane in (("crop", crop), ("gradient", grad), ("noise6", noise6)):
        bs, cl, ent = O.parametros_aclahe(plane)
        out.append((name, ent, cl))
    out.append(("uniform", _sweep_only(uni), None))   # scipy raises in the oracle
    return out


def _sweep_only(plane):
    blur = O.gaussian_blur3(plane)
    return np.array([[O.entropy_py(O.clahe_apply(blur, float(c), k, k)) for c in np.arange(0, 25, 0.5)]
                     for k in (2, 4, 8, 16, 32)], np.float32)


@pytest.fixture(scope="module")
def tables():
    return _tables()


def test_clip_curve_fit_matches_scipy(knee_exe):
    (nfev, p), _ = _run(knee_exe, [np.ones(49, np.float32)])
    ok, popt, nf = _scipy(np.arange(1, 50, dtype=np.float32) * np.float32(0.5))
    assert ok
    assert np.max(np.abs(p - popt) / np.abs(popt)) < 1e-6
    assert nfev == nf


def test_crowd_knees_golden(knee_exe):
    z = np.load(os.path.join(GOLD, "crowd_full.npz"))
    _, rows = _run(knee_exe, [r[1:50] for r in z["entropies"]])
    knees = [r[0] for r in rows]
    assert knees == [7, 7, 7, 5, 2] == list(z["knees"])
    assert max(knees) == 7


def test_knees_and_failures_match_the_oracle(knee_exe, tables):
    curves, names = [], []
    for name, t, _ in tables:
        for k in range(5):
            curves.append(t[k][1:50])
            names.append((name, k))
    _, rows = _run(knee_exe, curves)
    rel, nfev_diff = [], 0
    for (name, k), c, (kn, nfev, info, p) in zip(names, curves, rows):
        ok, popt, nf = _scipy(c)
        want = _oracle_knee(np.concatenate([[0], c]).astype(np.float32))
        assert (want is None) == (not ok)
        if ok:
            assert 1 <= info <= 4, (name, k, info)
            assert kn == want, (name, k, kn, want)
            rel.append(np.max(np.abs(p - popt) / np.abs(popt)))
            nfev_diff += nfev != nf
        else:
            assert kn == -1 and not 1 <= info <= 4, (name, k, info)
    assert any(kn == -1 for kn, *_ in rows), "the uniform-noise plane must fail the fit"
    # the fits stop at xtol = 1.49e-8 on ill-conditioned problems: exp rounded an ulp apart (numpy's SIMD exp, glibc's,
    # CUDA's) moves the weakest parameter by up to about 1e-3 relative without moving a knee
    print("popt max rel diff %.3g (median %.3g), nfev differs on %d of %d fits" % (max(rel), np.median(rel), nfev_diff, len(rel)))
    assert max(rel) < 1e-2, max(rel)
    assert nfev_diff <= len(rel) // 4


def test_clip_limits_of_distinct_planes(knee_exe, tables):
    """CL = max of the five knees equals the oracle's ParametrosACLAHE clip limit (crowd.png: 7); uniform noise fails."""
    assert [t[2] for t in tables][:2] == [7, 7]
    for name, t, want in tables:
        _, rows = _run(knee_exe, [r[1:50] for r in t])
        knees = [r[0] for r in rows]
        got = None if min(knees) < 0 else max(knees)
        assert got == want, (name, knees)


def test_knee_is_stable_under_perturbation(knee_exe, tables):
    """A few hundred copies of the tables with 1e-6 relative noise: the header and the oracle agree on every one."""
    rng = np.random.default_rng(11)
    curves = []
    for name, t, _ in tables:
        if name == "uniform":
            continue
        for k in range(5):
            for _ in range(12):
                curves.append((t[k][1:50] * (1 + 1e-6 * rng.standard_normal(49))).astype(np.float32))
    _, rows = _run(knee_exe, curves)
    for c, (kn, *_rest) in zip(curves, rows):
        assert kn == _oracle_knee(np.concatenate([[0], c]).astype(np.float32))
