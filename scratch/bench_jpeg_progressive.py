"""Cost of reading progressive JPEG files on the device: the progressive-capable reader (uwip_jpeg_decode_batch_ex) on
progressive files, the same reader and the existing reader (uwip_jpeg_decode_bgr8_batch) on baseline files of the same
frames, and cv2.imdecode of the progressive files on all host cores.  Inputs: chain-output frames of the synthetic generator
at 4K and 1080p, each written by cv2 at q95 4:2:0 as a progressive file (libjpeg-turbo's jpeg_simple_progression, 10 scans)
and as a baseline file.  Batches of 64 (the command lines' default) and 256 frames.  All arms alternated in one process;
medians reported.  Reports the whole call (host files to device frames, synchronised), the device time of each pass from
uwip_profile, and the card's name and power limit read in the same run.  Prints one JSON line and, with --out, also writes
it there.

    python scratch/bench_jpeg_progressive.py [--frames 256] [--reps 5] [--out profiles/jpeg_progressive_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PASSES = ("jpeg_dec_destuff", "jpeg_dec_sync", "jpeg_dec_fixup", "jpeg_dec_scan", "jpeg_dec_huff", "jpeg_dec_pdestuff", "jpeg_dec_prog",
          "jpeg_dec_idct", "jpeg_dec_color")


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
    res = {"card": card(), "frames": n, "quality": q, "sampling": "4:2:0", "host_threads": os.cpu_count(),
           "input": "cv2.imencode of the chain output of synthetic frames (seed 0x5EED0004), progressive and baseline",
           "sizes": {}}
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    enc = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420]
    for (w, h) in ((3840, 2160), (1920, 1080)):
        prog, base = [], []
        d_in = torch.empty((32, h, w, 3), dtype=torch.uint8, device="cuda")
        d_fr = torch.empty_like(d_in)
        for b0 in range(0, n, 32):
            m = min(32, n - b0)
            ctx.synth_dev(d_in, 0x5EED0004, b0, m, w, h)
            ctx.chain_dev(d_in, d_fr, m, w, h)
            fr = d_fr[:m].cpu().numpy()
            prog += list(pool.map(lambda f: bytes(cv2.imencode(".jpg", f, enc + [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1]), fr))
            base += list(pool.map(lambda f: bytes(cv2.imencode(".jpg", f, enc)[1]), fr))
        del d_in, d_fr
        d_out = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        size = {"mean_file_bytes": {"progressive": float(np.mean([len(b) for b in prog])), "baseline": float(np.mean([len(b) for b in base]))}}
        for batch in (64, 256):
            if batch > n:
                continue
            arms = {"ex_progressive": (prog[:batch], True), "ex_baseline": (base[:batch], True), "existing_baseline": (base[:batch], False)}
            d = d_out[:batch]

            def run(arm):
                fl, ex = arm
                ctx.jpeg_decode_batch_dev(fl, d, progressive=ex)

            def host(fl):
                return list(pool.map(lambda b: cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR), fl))

            for k, arm in arms.items():
                t0 = time.perf_counter()
                run(arm)
                torch.cuda.synchronize()
                print("%dx%d batch %d %s: first call %.1f ms" % (w, h, batch, k, (time.perf_counter() - t0) * 1e3), file=sys.stderr, flush=True)
            host(prog[:batch])
            torch.cuda.synchronize()
            call_ms = {k: [] for k in list(arms) + ["cv2_progressive_host"]}
            pass_ms = {k: {p: [] for p in PASSES} for k in arms}
            for _ in range(a.reps):
                for k, arm in arms.items():   # whole calls, profiler off
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    run(arm)
                    torch.cuda.synchronize()
                    call_ms[k].append(round((time.perf_counter() - t0) * 1e3, 2))
                t0 = time.perf_counter()
                host(prog[:batch])
                call_ms["cv2_progressive_host"].append(round((time.perf_counter() - t0) * 1e3, 2))
                for k, arm in arms.items():   # the passes, from device events
                    ctx.profile(True)
                    run(arm)
                    torch.cuda.synchronize()
                    for p in PASSES:
                        pass_ms[k][p].append(round(ctx.profile_read(p)[0], 3))
                    ctx.profile(False)
            checks = {}
            for k, arm in arms.items():
                run(arm)
                got = d.cpu().numpy()
                fl = arm[0]
                checks[k] = all((got[i] == cv2.imdecode(np.frombuffer(fl[i], np.uint8), cv2.IMREAD_COLOR)).all()
                                for i in range(0, batch, max(1, batch // 8)))
            size["batch_%d" % batch] = {
                "call_ms": call_ms,
                "call_ms_median": {k: float(np.median(v)) for k, v in call_ms.items()},
                "pass_ms_median": {k: {p: float(np.median(v)) for p, v in ps.items() if any(v)} for k, ps in pass_ms.items()},
                "sampled_frames_equal_cv2_imdecode": checks,
            }
        res["sizes"]["%dx%d" % (w, h)] = size
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
