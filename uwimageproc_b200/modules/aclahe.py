"""Mirror of modules/aclahe/python/{functions,ACLAHE,main}.py (reference function names kept).

Pixel work (GaussianBlur 3x3, CLAHE, entropy, the clip-limit sweep) runs in libuwip.so.  ParametrosACLAHE keeps the
reference's host-side knee search on the 49 entropy samples per block size (curve_fit + spline derivatives + curvature,
functions.py:49-93) with the same scipy calls; parametros_aclahe_batch runs the whole search for a batch on the device, and
main_batch the whole grey prototype (search and CLAHE).
"""
import warnings

import numpy as np

from ..api import default_context

BLOCK_SIZES = (2, 4, 8, 16, 32)  # ACLAHE.py:21


def Entropia(imagen):  # functions.py:14
    return default_context().entropy(imagen, "py")


def CLAHE(imagen, parametro, CL):  # functions.py:24
    return default_context().clahe(imagen, float(CL), (int(parametro), int(parametro)))


def _fit(u, Y):
    from scipy.optimize import curve_fit

    def f(x, p0, p1, p2, p3):
        return p0 * np.exp(-p1 * x) + p2 * np.exp(-p3 * x)

    popt, _ = curve_fit(f, u, Y, (7, 0.4, 0.9, 5))
    return f, popt


def DerivadaY(Y):  # functions.py:49
    from scipy.interpolate import splev, splrep

    f, popt = _fit(np.linspace(1, 49, 49), Y)
    x22 = np.linspace(1, 25, 25)
    tck = splrep(x22, f(x22, *popt))
    x222 = np.linspace(1, 25, 49)
    d1 = splev(x222, tck, der=1)
    return x22, x222, d1, splev(x222, tck, der=2), d1 ** 2


def DerivadaX(X, x22, x222):  # functions.py:66
    from scipy.interpolate import splev, splrep

    f, popt = _fit(np.linspace(1, 49, 49), X)
    tck = splrep(x22, f(x22, *popt))
    d1 = splev(x222, tck, der=1)
    return d1, d1 ** 2, splev(x222, tck, der=2)


def Curvatura(y220, y221, y222, y223, y224, y225):  # functions.py:81
    k = np.sqrt((y223 * y221 - y220 * y225) ** 2) / np.sqrt((y224 + y222) ** 3)
    return int(np.argmax(k))


def ParametrosACLAHE(imagen, loop="repaired"):
    """ACLAHE.py:9-129 -> (BS, CL).

    loop="repaired": the entropy-vs-clip-limit sweep the code intends (all 50 clip limits per block size).
    loop="as_committed": the file as it is in the reference, whose sweep body lost its indentation
    (ACLAHE.py:40-47): only column 1 of the table is ever written, the curves handed to the knee search
    are all zero and the clip limit degenerates to 0 (SURVEY 8a-A3, K4: crowd.png -> (8, 0)).
    """
    ctx = default_context()
    imgfilt = ctx.gaussian_blur3(imagen)  # ACLAHE.py:15
    cl = np.arange(0, 25, 0.5)
    if loop == "as_committed":
        d = 0
    elif loop == "repaired":
        ks = []
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # the reference's fit emits overflow / covariance warnings too
            for k in BLOCK_SIZES:
                row_x = np.zeros(51, np.float32)
                row_y = np.zeros(51, np.float32)
                row_x[1:51] = cl
                row_y[1:51] = ctx.clahe_entropy_sweep(imgfilt, k, cl, "py")  # ACLAHE.py:38-47, one pass per grid
                x, y = row_x[2:51], row_y[2:51]  # graficar, functions.py:32-38
                x22, x222, y220, y221, y222 = DerivadaY(y)
                y223, y224, y225 = DerivadaX(x, x22, x222)
                ks.append(Curvatura(y220, y221, y222, y223, y224, y225))
        d = max(ks)  # ACLAHE.py:92-96
    else:
        raise ValueError("loop must be 'repaired' or 'as_committed'")
    res = np.zeros((2, 5), np.float16)  # ACLAHE.py:102: entropies are compared in float16
    for m, k in enumerate(BLOCK_SIZES):
        res[0, m] = k
        res[1, m] = Entropia(CLAHE(imgfilt, k, d))
    w = int(np.flatnonzero(res[1] == res[1].max())[-1])  # last arg-max wins, ACLAHE.py:117-121
    return int(round(float(res[0, w]))), d


def parametros_aclahe_batch(planes, loop="repaired"):
    """ParametrosACLAHE of every plane of a batch, on the device: planes uint8 (N, H, W) host array or device tensor ->
    (BS int32[N], CL int32[N]); -1 where the reference's curve fit raises."""
    import torch

    ctx = default_context()
    t = planes if isinstance(planes, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(planes, dtype=np.uint8))
    if t.dtype != torch.uint8 or t.dim() != 3:
        raise ValueError("expected uint8 (N, H, W)")
    t = t.to("cuda:%d" % ctx.device).contiguous()
    torch.cuda.synchronize(ctx.device)
    bs, cl = ctx.aclahe_params_dev(t, t.shape[0], t.shape[2], t.shape[1], loop)
    ctx.synchronize()
    return bs.cpu().numpy(), cl.cpu().numpy()


def main(img):
    """aclahe/python/main.py:17-20 without the file I/O."""
    BS, CL = ParametrosACLAHE(img)
    return CLAHE(img, BS, CL)


def main_batch(planes, loop="repaired"):
    """main.py:18-20 for a batch, on the device: planes uint8 (N, H, W) host array or device tensor -> (out uint8 (N, H, W),
    BS int32[N], CL int32[N]) as host arrays; out[i] = createCLAHE(CL[i], (BS[i], BS[i])).apply(planes[i]).  Where the
    reference's curve fit raises, BS = CL = -1 and the plane gets the fixed 8 x 8 grid and clip 2 of the chain."""
    import torch

    ctx = default_context()
    t = planes if isinstance(planes, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(planes, dtype=np.uint8))
    if t.dtype != torch.uint8 or t.dim() != 3:
        raise ValueError("expected uint8 (N, H, W)")
    t = t.to("cuda:%d" % ctx.device).contiguous()
    torch.cuda.synchronize(ctx.device)
    n, h, w = t.shape
    out = torch.empty_like(t)
    bs = torch.empty(n, dtype=torch.int32, device=t.device)
    cl = torch.empty(n, dtype=torch.int32, device=t.device)
    ctx.aclahe_grey_auto_dev(t, out, n, w, h, loop, d_bs=bs, d_cl=cl)
    ctx.synchronize()
    return out.cpu().numpy(), bs.cpu().numpy(), cl.cpu().numpy()
