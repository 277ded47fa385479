"""Throughput of the batched exact JPEG decoder (uwip_jpeg_decode_bgr8_batch) against the nvJPEG single-frame path
(uwip_jpeg_decode_bgr8_dev, one call per frame) and cv2.imdecode over all host cores, on q95 4:2:0 files of chain-output frames
at 4K and 1080p, timed alternately in one process; and files in -> files out: exact decode -> chain -> exact encode -> bytes on
the host against the cv2 route (imdecode -> uwip_chain_bgr8 -> imencode).  Also per-pass device time of one batch from
uwip_profile and the synchronisation statistics (re-decoded subsequences, fix-up steps).  Prints one JSON line and, with --out,
also writes it there.

    python scratch/bench_jpeg_decode.py [--frames 256] [--reps 3] [--out path]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PASSES = ["jpeg_dec_destuff", "jpeg_dec_sync", "jpeg_dec_fixup", "jpeg_dec_scan", "jpeg_dec_huff", "jpeg_dec_idct", "jpeg_dec_color"]


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
    import cv2
    import torch

    import uwimageproc_b200 as u

    ctx = u.Context(0)
    n, q = a.frames, 95
    cores = os.cpu_count() or 1
    pool = ThreadPoolExecutor(max_workers=cores)
    res = {"card": card(), "frames": n, "quality": q, "sampling": "4:2:0", "host_cores": cores,
           "input": "cv2.imencode of the chain output of synthetic frames (seed 0x5EED0004)", "sizes": {}}
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    enc = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420]
    for (w, h) in ((3840, 2160), (1920, 1080)):
        files = []
        d_in = torch.empty((32, h, w, 3), dtype=torch.uint8, device="cuda")
        d_fr = torch.empty_like(d_in)
        for b0 in range(0, n, 32):   # the input files: chain output of synthetic frames, encoded by cv2
            m = min(32, n - b0)
            ctx.synth_dev(d_in, 0x5EED0004, b0, m, w, h)
            ctx.chain_dev(d_in, d_fr, m, w, h)
            host = d_fr[:m].cpu().numpy()
            files += list(pool.map(lambda f: bytes(cv2.imencode(".jpg", f, enc)[1]), host))
        del d_in, d_fr
        d_out = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        d_enh = torch.empty_like(d_out)
        bufs = [np.frombuffer(f, np.uint8) for f in files]

        def exact():
            ctx.jpeg_decode_batch_dev(files, d_out)

        def nvjpeg():
            for f in range(n):
                ctx.jpeg_decode_dev(files[f], d_out[f])

        def cv2_pool():
            return list(pool.map(lambda b: cv2.imdecode(b, cv2.IMREAD_COLOR), bufs))

        def files_exact():   # files in -> exact decode -> chain -> exact encode -> files on the host
            ctx.jpeg_decode_batch_dev(files, d_out)
            ctx.chain_dev(d_out, d_enh, n, w, h)
            return ctx.jpeg_encode_batch_dev(d_enh, q)

        def files_cv2():     # imdecode -> uwip_chain_bgr8 (host buffers) -> imencode, cv2 over all cores
            fr = np.stack(cv2_pool())
            out = ctx.chain(fr)
            return list(pool.map(lambda f: bytes(cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])[1]), out))

        runs = {"exact": exact, "nvjpeg_loop": nvjpeg, "cv2_imdecode_all_cores": cv2_pool, "files_exact": files_exact,
                "files_cv2_route": files_cv2}
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
        # kernels only: the passes of one batch from device events
        ctx.profile(True)
        exact()
        prof = {t: round(ctx.profile_read(t)[0], 3) for t in PASSES}
        ctx.profile(False)
        kernels_ms = []
        for _ in range(a.reps):
            ctx.profile(True)
            exact()
            kernels_ms.append(round(ctx.profile_read("jpeg_dec_")[0], 2))
            ctx.profile(False)
        st = ctx.jpeg_decode_stats(n)
        got = d_out.cpu().numpy()
        same = all((got[i] == cv2.imdecode(bufs[i], cv2.IMREAD_COLOR)).all() for i in range(0, n, max(1, n // 8)))
        fe, fc = files_exact(), files_cv2()
        res["sizes"]["%dx%d" % (w, h)] = {
            "batch_ms": {k: [round(x, 2) for x in v] for k, v in times.items()},
            "frames_per_s": {k: round(n / (min(v) / 1e3), 1) for k, v in times.items()},
            "exact_kernels_only_ms": kernels_ms,
            "pass_ms_one_batch": prof,
            "sync_redecodes_per_frame": {"mean": round(float(st[:, 0].mean()), 2), "max": int(st[:, 0].max())},
            "fixup_steps_per_frame": {"mean": round(float(st[:, 1].mean()), 2), "max": int(st[:, 1].max())},
            "subsequences_per_frame_mean": round(float(np.mean([len(f) for f in files]) * 8 / 1024), 1),
            "file_bytes_mean": int(np.mean([len(f) for f in files])),
            "sampled_frames_equal_cv2_imdecode": bool(same),
            "files_exact_equal_cv2_route": fe == fc,
        }
        del d_out, d_enh
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
