"""Cost of the automatic CLAHE parameters in the chain: chain_dev (fixed clip 2, 8 x 8) and chain_auto_dev timed alternately
in one process with CUDA events around whole 256-frame batches, at 4K and 1080p, plus the per-kernel device time of one
batch of each from uwip_profile.  Prints the result as JSON and, with --out, also writes it there.

    python scratch/bench_aclahe_auto.py [--frames 256] [--reps 3] [--out path]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KERNELS = ["clahe_tilehist", "clahe_lut", "clahe_sweep_hist", "clahe_apply", "entropy", "blur3", "aclahe_vplane", "aclahe_knee",
           "aclahe_pick", "aclahe_geom", "prelut2", "dz_"]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this path")
    a = ap.parse_args()
    import torch

    import uwimageproc_b200 as u

    ctx = u.Context(0)
    res = {"card": card(), "frames": a.frames, "sizes": {}}
    for (w, h) in ((3840, 2160), (1920, 1080)):
        n = a.frames
        d_in = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        ctx.synth_dev(d_in, 0x5EED0004, 0, n, w, h)
        d_out = torch.empty_like(d_in)
        d_bs = torch.empty(n, dtype=torch.int32, device="cuda")
        d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        runs = {"fixed": lambda: ctx.chain_dev(d_in, d_out, n, w, h),
                "auto": lambda: ctx.chain_auto_dev(d_in, d_out, n, w, h, None, "repaired", d_bs, d_cl)}
        for f in runs.values():   # warm-up: modules, workspace slots
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, f in runs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1))
        prof = {}
        for k, f in runs.items():
            ctx.profile(True)
            f()
            prof[k] = {t: round(ctx.profile_read(t)[0], 3) for t in KERNELS}
            ctx.profile(False)
        cl = d_cl.cpu().numpy()
        bs = d_bs.cpu().numpy()
        res["sizes"]["%dx%d" % (w, h)] = {
            "batch_ms": {k: [round(x, 2) for x in v] for k, v in times.items()},
            "frames_per_s": {k: round(n / (min(v) / 1e3), 1) for k, v in times.items()},
            "kernel_ms_one_batch": prof,
            "bs_hist": {int(b): int((bs == b).sum()) for b in np.unique(bs)},
            "cl_range": [int(cl.min()), int(cl.max())],
        }
        del d_in, d_out
        torch.cuda.empty_cache()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
