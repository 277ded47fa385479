"""Throughput of the batched exact JPEG encoder (uwip_jpeg_encode_bgr8_batch_dev) against the nvJPEG single-frame path
(uwip_jpeg_encode_bgr8_dev, one call per frame with its host round trips), on the same chain output frames at 4K and 1080p,
timed alternately in one process; the chain's own batch time for scale; per-pass device time of one batch from uwip_profile;
bytes per frame.  Prints one JSON line and, with --out, also writes it there.

    python scratch/bench_jpeg_encode.py [--frames 256] [--reps 3] [--quality 95] [--out path]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PASSES = ["jpeg_enc_setup", "jpeg_enc_blocks", "jpeg_enc_scan", "jpeg_enc_emit", "jpeg_enc_stuff"]


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
    ap.add_argument("--quality", type=int, default=95)
    ap.add_argument("--out", default=None, help="also write the JSON result to this path")
    a = ap.parse_args()
    import cv2
    import torch

    import uwimageproc_b200 as u

    ctx = u.Context(0)
    q, n = a.quality, a.frames
    res = {"card": card(), "frames": n, "quality": q, "input": "chain output of synthetic frames (seed 0x5EED0004)", "sizes": {}}
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    for (w, h) in ((3840, 2160), (1920, 1080)):
        d_in = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        ctx.synth_dev(d_in, 0x5EED0004, 0, n, w, h)
        d_fr = torch.empty_like(d_in)
        stride = ctx.jpeg_encode_bound(w, h)
        d_jpg = torch.empty((n, stride), dtype=torch.uint8, device="cuda")
        d_len = torch.empty(n, dtype=torch.int64, device="cuda")

        def chain():
            ctx.chain_dev(d_in, d_fr, n, w, h)

        def exact():
            ctx._ck(ctx.lib.uwip_jpeg_encode_bgr8_batch_dev(ctx.h, d_fr.data_ptr(), n, w, h, q, d_jpg.data_ptr(), stride, d_len.data_ptr()))

        def exact_to_host():   # the batch, then the lengths, then each file's bytes
            exact()
            lens = d_len.cpu().tolist()
            return [d_jpg[f, :lens[f]].cpu() for f in range(n)]

        def nvjpeg():
            return [ctx.jpeg_encode_dev(d_fr[f], w, h, q) for f in range(n)]

        runs = {"chain": chain, "exact": exact, "exact_to_host": exact_to_host, "nvjpeg_loop": nvjpeg}
        for f in runs.values():   # warm-up: modules, workspace slots, nvJPEG state
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, f in runs.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                f()
                e1.record()
                e1.synchronize()
                times[k].append(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
        ctx.profile(True)
        exact()
        prof = {t: round(ctx.profile_read(t)[0], 3) for t in PASSES}
        ctx.profile(False)
        lens = d_len.cpu().numpy()
        first = d_jpg[0, :int(lens[0])].cpu().numpy().tobytes()
        ok, ref = cv2.imencode(".jpg", d_fr[0].cpu().numpy(), [cv2.IMWRITE_JPEG_QUALITY, q])
        nv = nvjpeg()
        res["sizes"]["%dx%d" % (w, h)] = {
            "batch_ms": {k: [round(x, 2) for x in v] for k, v in times.items()},
            "frames_per_s": {k: round(n / (min(v) / 1e3), 1) for k, v in times.items()},
            "pass_ms_one_batch": prof,
            "bytes_per_frame": {"exact_mean": int(lens.mean()), "exact_max": int(lens.max()),
                                "nvjpeg_mean": int(np.mean([len(b) for b in nv])), "raw_bgr8": w * h * 3,
                                "bound": stride},
            "frame0_equals_cv2_imencode": bool(ok) and first == bytes(ref),
        }
        del d_in, d_fr, d_jpg
        torch.cuda.empty_cache()
    ctx.close()
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
