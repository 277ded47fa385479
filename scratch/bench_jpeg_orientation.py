"""Cost of applying the Exif orientation in the exact JPEG readers: the existing reader (uwip_jpeg_decode_bgr8_batch, stored
orientation, output pass jpeg_dec_color) against the oriented reader (uwip_jpeg_decode_bgr8_batch_oriented, output pass
jpeg_dec_color_oriented) on the same q95 4:2:0 files of chain-output frames at 4K and 1080p, each tagged with orientation 1
(nothing to do), 3 (a flip of both axes) and 6 (a transpose: the output is portrait).  All six arms are alternated in one
process.  Reports the whole call (host files to device frames, synchronised), the output pass's device time from
uwip_profile, and the card's name and power limit read in the same run.  Prints one JSON line and, with --out, also writes it
there.

    python scratch/bench_jpeg_orientation.py [--frames 256] [--reps 5] [--out profiles/jpeg_orientation_bench.json]
"""
import argparse
import json
import os
import struct
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ORIENTATIONS = (1, 3, 6)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def tag(data, o):
    """the file with a little-endian Exif APP1 holding orientation o spliced in after SOI"""
    t = b"Exif\0\0II" + struct.pack("<HIH", 42, 8, 1) + struct.pack("<HHIHH", 0x0112, 3, 1, o, 0) + struct.pack("<I", 0)
    return data[:2] + b"\xff\xe1" + struct.pack(">H", len(t) + 2) + t + data[2:]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result to this path")
    a = ap.parse_args()
    import cv2
    import numpy as np
    import torch

    import uwimageproc_b200 as u

    ctx = u.Context(0)
    n, q = a.frames, 95
    pool = ThreadPoolExecutor(max_workers=os.cpu_count() or 1)
    res = {"card": card(), "frames": n, "quality": q, "sampling": "4:2:0",
           "input": "cv2.imencode of the chain output of synthetic frames (seed 0x5EED0004), Exif orientation 1, 3 or 6 spliced in",
           "sizes": {}}
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    enc = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420]
    for (w, h) in ((3840, 2160), (1920, 1080)):
        plain = []
        d_in = torch.empty((32, h, w, 3), dtype=torch.uint8, device="cuda")
        d_fr = torch.empty_like(d_in)
        for b0 in range(0, n, 32):
            m = min(32, n - b0)
            ctx.synth_dev(d_in, 0x5EED0004, b0, m, w, h)
            ctx.chain_dev(d_in, d_fr, m, w, h)
            plain += list(pool.map(lambda f: bytes(cv2.imencode(".jpg", f, enc)[1]), d_fr[:m].cpu().numpy()))
        del d_in, d_fr
        files = {o: [tag(f, o) for f in plain] for o in ORIENTATIONS}
        d_out = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        arms = {}
        for o in ORIENTATIONS:
            for oriented in (False, True):
                name = "%s_o%d" % ("oriented" if oriented else "existing", o)
                shape = (n, w, h, 3) if oriented and o >= 5 else (n, h, w, 3)
                arms[name] = (files[o], d_out.view(shape), oriented, "jpeg_dec_color_oriented" if oriented else "jpeg_dec_color")

        def run(arm):
            fl, d, oriented, _ = arm
            ctx.jpeg_decode_batch_dev(fl, d, orientation=oriented)

        for arm in arms.values():
            run(arm)
        torch.cuda.synchronize()
        call_ms = {k: [] for k in arms}
        pass_ms = {k: [] for k in arms}
        for _ in range(a.reps):
            for k, arm in arms.items():   # whole calls, profiler off
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run(arm)
                torch.cuda.synchronize()
                call_ms[k].append(round((time.perf_counter() - t0) * 1e3, 2))
            for k, arm in arms.items():   # the output pass, from device events
                ctx.profile(True)
                run(arm)
                pass_ms[k].append(round(ctx.profile_read(arm[3])[0], 3))
                ctx.profile(False)
        checks = {}
        for k, (fl, d, oriented, _) in arms.items():
            run(arms[k])
            got = d.cpu().numpy()
            flags = cv2.IMREAD_COLOR | (0 if oriented else cv2.IMREAD_IGNORE_ORIENTATION)
            checks[k] = all((got[i] == cv2.imdecode(np.frombuffer(fl[i], np.uint8), flags)).all() for i in range(0, n, max(1, n // 8)))
        res["sizes"]["%dx%d" % (w, h)] = {
            "call_ms": call_ms,
            "call_ms_median": {k: float(np.median(v)) for k, v in call_ms.items()},
            "output_pass_ms": pass_ms,
            "output_pass_ms_median": {k: float(np.median(v)) for k, v in pass_ms.items()},
            "output_bytes_per_batch": n * w * h * 3,
            "sampled_frames_equal_cv2_imdecode": checks,
        }
        del d_out
        torch.cuda.empty_cache()
    ctx.close()
    pool.shutdown()
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
