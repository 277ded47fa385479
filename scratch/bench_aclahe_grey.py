"""Cost of the grey prototype (modules/aclahe/python/main.py) on files: the device route - grey exact reader
(uwip_jpeg_decode_u8_batch) -> uwip_aclahe_u8_auto_dev -> grey writer (uwip_jpeg_encode_u8_batch_dev) -> bytes on the host -
against the host route of `aclahe -grey=1` - cv2.imdecode(.., IMREAD_GRAYSCALE) -> ParametrosACLAHE (scipy knee search, one
device sweep per grid) -> cv2 CLAHE -> cv2.imencode - timed alternately in one process.  Input: q95 grey JPEG files of the V
planes of synthetic frames (seed 0x5EED0004) at 4K and 1080p.  The host route takes seconds per frame, so it runs on the
first --host-frames files and is reported per frame.  Also the device time of each stage of one batch (uwip_profile: the
reader, the parameter search, the CLAHE passes as the call minus the search, the writer).  Prints one JSON line and, with
--out, also writes it there.

    python scratch/bench_aclahe_grey.py [--frames 256] [--host-frames 8] [--reps 2] [--out path]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
    ap.add_argument("--host-frames", type=int, default=8)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON result to this path")
    a = ap.parse_args()
    import cv2
    import torch

    import uwimageproc_b200 as u
    from uwimageproc_b200.modules import aclahe as A

    ctx = u.Context(0)
    n, q = a.frames, 95
    res = {"card": card(), "frames": n, "host_route_frames": a.host_frames, "quality": q,
           "input": "q95 grey JPEG of the V plane of synthetic frames (seed 0x5EED0004)", "sizes": {}}
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    for (w, h) in ((3840, 2160), (1920, 1080)):
        files = []
        d_fr = torch.empty((32, h, w, 3), dtype=torch.uint8, device="cuda")
        for b0 in range(0, n, 32):
            m = min(32, n - b0)
            ctx.synth_dev(d_fr, 0x5EED0004, b0, m, w, h)
            files += ctx.jpeg_encode_grey_batch_dev(d_fr[:m].amax(dim=3).contiguous(), q)
        del d_fr
        d_in = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
        d_out = torch.empty_like(d_in)
        d_bs = torch.empty(n, dtype=torch.int32, device="cuda")
        d_cl = torch.empty(n, dtype=torch.int32, device="cuda")

        def device():
            ctx.jpeg_decode_grey_batch_dev(files, d_in)
            ctx.aclahe_grey_auto_dev(d_in, d_out, n, w, h, "repaired", d_bs=d_bs, d_cl=d_cl)
            return ctx.jpeg_encode_grey_batch_dev(d_out, q)

        def host():
            out = []
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                for f in files[:a.host_frames]:
                    img = cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_GRAYSCALE)
                    try:
                        bs, cl = A.ParametrosACLAHE(img)
                    except RuntimeError:
                        bs, cl = 8, 2
                    res_img = cv2.createCLAHE(float(cl), (bs, bs)).apply(img)
                    out.append(bytes(cv2.imencode(".jpg", res_img, [cv2.IMWRITE_JPEG_QUALITY, q])[1]))
            return out

        runs = {"device": device, "host": host}
        for f in runs.values():
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, f in runs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                times[k].append((time.perf_counter() - t0) * 1e3)
        # device time of the stages of one batch
        ctx.profile(True)
        ctx.jpeg_decode_grey_batch_dev(files, d_in)
        dec = ctx.profile_read("")[0]   # every launch the profiled call made
        ctx.profile(False)
        ctx.profile(True)
        ctx.aclahe_grey_auto_dev(d_in, d_out, n, w, h, "repaired", d_bs=d_bs, d_cl=d_cl)
        ctx.synchronize()
        auto = ctx.profile_read("")[0]
        ctx.profile(False)
        ctx.profile(True)
        ctx.aclahe_params_dev(d_in, n, w, h, "repaired", d_bs, d_cl)
        ctx.synchronize()
        params = ctx.profile_read("")[0]
        ctx.profile(False)
        ctx.profile(True)
        got = ctx.jpeg_encode_grey_batch_dev(d_out, q)
        enc = ctx.profile_read("")[0]
        ctx.profile(False)
        bs, cl = d_bs.cpu().numpy(), d_cl.cpu().numpy()
        hd = host()
        res["sizes"]["%dx%d" % (w, h)] = {
            "device_route_batch_ms": [round(x, 1) for x in times["device"]],
            "device_route_frames_per_s": round(n / (min(times["device"]) / 1e3), 1),
            "host_route_ms_per_frame": [round(x / a.host_frames, 1) for x in times["host"]],
            "device_stage_ms_one_batch": {"decode": round(dec, 2), "params": round(params, 2), "clahe": round(auto - params, 2),
                                          "encode": round(enc, 2)},
            "device_files_equal_host_route": got[:a.host_frames] == hd,
            "bs_hist": {int(b): int((bs == b).sum()) for b in np.unique(bs)},
            "cl_range": [int(cl.min()), int(cl.max())],
            "file_bytes_mean": int(np.mean([len(f) for f in files])),
        }
        del d_in, d_out
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
