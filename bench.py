#!/usr/bin/env python3
"""bench.py - frames/s of the fused histretch -> aclahe -> bgdehaze chain on synthetic 4K frames.

  python bench.py --gpus N --steps K --warmup W            (our arm: libuwip.so on N B200s)
  python bench.py --impl reference --gpus N --steps K ...   (CPU arm: the reference's algorithm on host cores)
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs, see dump_outputs)

A step = one pass of the chain over one batch of `--frames` (default 256) synthetic 3840x2160 bgr8
frames per GPU (BASELINE.json configs[3]); frames shard across ranks by batch with no collective on
the data path (weak scaling).  `value` = frames/s with inputs resident in HBM; `e2e` = the same
through the host-buffer C-ABI call (pinned host memory, H2D and D2H inside the timed region).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W4K, H4K = 3840, 2160
SEED = 0x5EED0004
# algorithmic bytes per pixel of each pass (SURVEY.md 8d accounting; DESIGN.md "Kernels")
# The canonical passes D-g (27) and D-h (30) both read the a,b planes of the third guided filter; here the filter is
# applied once, inside dz_gf2b, which therefore carries D-g plus the a,b half of D-h (27 + 11 = 38) while dz_final
# carries what is left of D-h (read refined S, J, I; write bgr8 = 19).  The chain total stays 188.
ALGO_BPP = {
    "hist_frame": 3, "clahe_tilehist": 3, "clahe_apply": 6, "dz_window": 3, "dz_gf1a": 35, "dz_gf1b": 43,
    "dz_exposure_minmax": 11, "dz_gf2a": 27, "dz_gf2b": 38, "dz_final": 19,
    # helper passes outside the canonical accounting (their bytes are extra traffic, counted as 0 algorithmic)
    "dz_splane": 0,
}
CHAIN_BPP = 188
assert sum(ALGO_BPP.values()) == CHAIN_BPP


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 9 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 9 and r[2].isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm / cpu_baseline: the oracle port (numpy; cv2 for the OpenCV calls the reference makes)
# ------------------------------------------------------------------------------------------------
def _cpu_chain_one(args):
    seed, f, w, h = args
    from oracle import uwip_oracle as O  # the one place bench.py executes oracle/ (timed CPU baseline)

    fr = O.synth_frame(seed, f, w, h)
    t0 = time.perf_counter()
    try:
        import cv2

        cv2.setNumThreads(1)
        hsv = cv2.cvtColor(fr, cv2.COLOR_BGR2HSV)
        v = np_ascontig(hsv[..., 2])
        hist = cv2.calcHist([v], [0], None, [256], [0, 256]).ravel()
        low, high = O.percentile_bins(hist, w, h, 1, 99)
        m = float(__import__("numpy").float32(255.0 / (high - low))) if high != low else float("inf")
        hsv[..., 2] = cv2.convertScaleAbs(cv2.add(v, -float(low)), alpha=m)
        a = cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)
        hsv = cv2.cvtColor(a, cv2.COLOR_BGR2HSV)
        hsv[..., 2] = cv2.createCLAHE(2.0, (8, 8)).apply(np_ascontig(hsv[..., 2]))
        b = cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)
    except ImportError:
        b = O.aclahe_frame(O.histretch_frame(fr, "V", 1, 99), 2.0, 8, 8)
    out = O.bgdehaze_frame(b, 15)[1]
    return time.perf_counter() - t0, int(out.sum())


def bind_to_gpu_numa_node(index):
    """Pin this process (and therefore the first-touch placement of its pinned host buffers) to the CPUs of the NUMA
    node the GPU hangs off.  Returns a description for the bench line; silently does nothing when the box does not
    expose the topology (single-node boxes report node -1 / 0 for every device)."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        if node < 0 or len(nodes) < 2:
            return {"node": node, "nodes": len(nodes), "bound": False}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "nodes": len(nodes), "bound": bool(cpus), "cpus": len(cpus)}
    except Exception as e:  # topology files missing in the container
        return {"bound": False, "why": str(e)[:80]}


def np_ascontig(a):
    import numpy as np

    return np.ascontiguousarray(a)


def cpu_chain_fps(procs, w, h, frames_per_proc=1, first=0):
    """Whole-box CPU frames/s of the chain at (w, h), frames farmed over `procs` processes."""
    import multiprocessing as mp

    jobs = [(SEED, first + i, w, h) for i in range(procs * frames_per_proc)]
    t0 = time.perf_counter()
    if procs == 1:
        for j in jobs:
            _cpu_chain_one(j)
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_cpu_chain_one, jobs, chunksize=1)
    dt = time.perf_counter() - t0
    return len(jobs) / dt, dt


DUMP_SAMPLE = 8 << 20   # output bytes written by --dump-outputs (32 MB as float32) when the batch holds more


def dump_outputs(path, d_out, flags):
    """What the last timed step returned to its caller, as float32 .npy files under `path`: `frames` = the output bytes
    (the whole (n, H, W, 3) batch, or when it holds more than DUMP_SAMPLE bytes, the bytes at the flat positions
    np.unique(default_rng(SEED).integers(0, batch size, DUMP_SAMPLE)) in that order) and `frame_flags` = the per-frame
    flags (1 = the reference's result is a NaN frame)."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    flat = d_out.reshape(-1)
    if flat.numel() <= DUMP_SAMPLE:
        frames = d_out.cpu().numpy()
    else:
        pos = np.unique(np.random.default_rng(SEED).integers(0, flat.numel(), DUMP_SAMPLE))
        frames = flat[torch.from_numpy(pos).to(flat.device)].cpu().numpy()
    np.save(os.path.join(path, "frames.npy"), frames.astype(np.float32))
    np.save(os.path.join(path, "frame_flags.npy"), np.asarray(flags, np.float32))


def chain_config(W, H, n):
    """`config` of the bench line: the same dictionary for the CUDA arm and for the reference arm."""
    fbytes = W * H * 3
    return {"workload": "fused histretch(V,1/99)->aclahe(8x8,clip2)->bgdehaze(w15,r40,eps1e-3) chain on %dx%d bgr8 frames, "
                        "batch of %d frames per GPU per step (BASELINE configs[3])" % (W, H, n),
            "frames_per_gpu_per_step": n, "l2": "inputs (%.2f GB per step) exceed the 126 MB L2" % (n * fbytes / 1e9),
            "sharding": "disjoint frame batches per rank, no collective on the data path"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 32))
    sw, sh = 960, 540  # bounded sample: 1/16 of the pixels of a 4K frame per sample frame
    scale = (sw * sh) / float(W4K * H4K)
    for _ in range(args.warmup):
        cpu_chain_fps(procs, sw, sh)
    t0 = time.perf_counter()
    n = 0
    for s in range(args.steps):
        cpu_chain_fps(procs, sw, sh, first=s * procs)
        n += procs
    dt = time.perf_counter() - t0
    fps4k = n / dt * scale
    line = {
        "impl": "reference", "metric": "chain_frames_per_s_4k", "value": fps4k, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": chain_config(args.width, args.height, args.frames),   # the arm's config (the driver compares the two arms' dictionaries) ...
        # ... and what a step of THIS arm actually ran: a bounded sample of that workload, scaled by pixel count
        "ran": "each step = %d synthetic %dx%d frames (1/16 of the pixels of a 4K frame each) through the CPU chain on %d processes; "
               "frames/s scaled by pixel count to 3840x2160" % (procs, sw, sh, procs),
        "cpu_baseline": {"value": fps4k, "unit": "frames/s", "cores": procs, "kind": "port",
                         "sample": "%d synthetic %dx%d frames per step on %d processes (cv2 for the OpenCV calls, numpy fp64 "
                                   "restatement for bgdehaze), scaled by pixel count to 3840x2160" % (procs, sw, sh, procs)},
        "e2e": {"value": fps4k, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# BASELINE configs[4]: a stream of frames, contiguous frame ranges per GPU, one pass
# ------------------------------------------------------------------------------------------------
def run_stream(ctx, stream, dist, rank, world, total, batch, W, H, params, barrier):
    """Each rank generates its frame range on the device in batches (the stream does not fit one GPU at once), runs the
    chain once over it and keeps one checksum per frame; the checksums are gathered in stream order and compared with
    a single-GPU recomputation of a sample of frames taken from every rank's range (rank 0)."""
    import hashlib

    import numpy as np
    import torch

    from uwimageproc_b200 import shard

    first, count = shard.frame_range(rank, world, total)
    sums = np.empty(count, np.uint64)
    nan = 0
    with torch.cuda.stream(stream):
        d_in = torch.empty((batch, H, W, 3), dtype=torch.uint8, device="cuda")
        d_out = torch.empty_like(d_in)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for f, nb in shard.batches(first, count, batch):
            ctx.synth_dev(d_in, SEED + 1, f, nb, W, H)      # configs[4] uses seed 0x5EED0005
            ctx.chain_dev(d_in, d_out, nb, W, H, params)
            sums[f - first:f - first + nb] = ctx.checksum_dev(d_out, nb, W, H)
            nan += int((np.asarray(ctx.last_frame_flags(nb)) != 0).sum())
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
    t = torch.tensor([ms, float(nan)], dtype=torch.float64, device="cuda")
    if dist:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms_max, nan_all = float(tmax[0].item()), int(t[1].item())
    else:
        ms_max, nan_all = ms, nan
    allsums = shard.gather_checksums(sums, rank, world, total, dist, device="cuda")
    res = None
    if rank == 0:
        # single-GPU recomputation of sampled frames (every rank's range contributes) on this rank
        sample = sorted(set(int(v) for v in np.linspace(0, total - 1, num=min(total, 64)).round()))
        ok = True
        with torch.cuda.stream(stream):
            for f in sample:
                ctx.synth_dev(d_in, SEED + 1, f, 1, W, H)
                ctx.chain_dev(d_in, d_out, 1, W, H, params)
                ok = ok and (int(ctx.checksum_dev(d_out, 1, W, H)[0]) == int(allsums[f]))
        res = {"frames": total, "stream_fps": total / (ms_max / 1000.0), "ms": ms_max, "includes": "on-device generation of the frames and "
               "the per-frame checksum kernel", "frames_per_rank": count, "batch": batch, "nan_frames": nan_all,
               "crc_equal": bool(ok), "crc_sampled_frames": len(sample),
               "crc_digest": hashlib.sha1(np.ascontiguousarray(allsums).tobytes()).hexdigest()[:16],
               "crc_digest_note": "sha1 over the per-frame checksums in stream order: equal digests at every GPU count = equal frames"}
    return res


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="uwip", choices=["uwip", "reference"])
    ap.add_argument("--frames", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--width", type=int, default=W4K)
    ap.add_argument("--height", type=int, default=H4K)
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the host-buffer call (default: --steps)")
    ap.add_argument("--stream", type=int, default=0, help="BASELINE configs[4]: one pass over a stream of this many frames, "
                                                           "contiguous frame ranges per rank, per-frame checksums gathered")
    ap.add_argument("--copy-ceiling", action="store_true", help="also time the bare H2D + D2H copies of the e2e step (no kernels)")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy; "
                                                          "CUDA arm only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA arm; the reference arm keeps none")
    if args.e2e_steps is None:
        args.e2e_steps = args.steps
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    import numpy as np
    import torch

    import uwimageproc_b200 as u

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libuwip has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa = None if args.no_numa_bind else bind_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        # the contract is ONE JSON line on stdout: keep NCCL's version banner (NCCL_DEBUG=VERSION) off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        import torch.distributed as dist

        # ... and whatever the environment (nccl.conf, a pod-level NCCL_DEBUG) still makes NCCL print while the
        # communicator comes up goes to stderr: file descriptor 1 points at stderr until the first collective is done
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    ctx = u.Context(local)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    n, W, H = args.frames, args.width, args.height
    fbytes = W * H * 3
    params = ctx.chain_params()

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        d_in = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
        d_out = torch.empty_like(d_in)
        # disjoint frame ranges per rank (frame-batch sharding, SURVEY 8e)
        ctx.synth_dev(d_in, SEED, rank * n, n, W, H)
        for _ in range(args.warmup):
            ctx.chain_dev(d_in, d_out, n, W, H, params)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ctx.profile(True)
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            ctx.chain_dev(d_in, d_out, n, W, H, params)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ctx.launch_count() - l0
        clocks = sampler.stop() if rank == 0 else None
        prof = {k: ctx.profile_read(k) for k in ALGO_BPP}
        ctx.profile(False)
        sums = ctx.checksum_dev(d_out, min(n, 4), W, H)
        # frames whose result is the reference's NaN frame (S = 0/0 somewhere, SURVEY D9): the chain writes zeros for them
        flags = np.asarray(ctx.last_frame_flags(n))
        nan_frames = int((flags != 0).sum())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, d_out, flags)

    stream_res = None
    if args.stream > 0:
        stream_res = run_stream(ctx, stream, dist, rank, world, args.stream, n, W, H, params, barrier)

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    fps = world * n * args.steps / (ms_max / 1000.0)

    # ---- end to end through the host-buffer C ABI (pinned host memory, copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        h_in = torch.empty((n, H, W, 3), dtype=torch.uint8).pin_memory()
        h_out = torch.empty((n, H, W, 3), dtype=torch.uint8).pin_memory()
        h_in.copy_(d_in)
        ctx.chain_host_ptr(h_in.data_ptr(), h_out.data_ptr(), n, W, H, params)  # warm-up (allocates staging)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            ctx.chain_host_ptr(h_in.data_ptr(), h_out.data_ptr(), n, W, H, params)  # returns after D2H completed
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        te = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        same = bool((h_out[: min(n, 4)].numpy() == d_out[: min(n, 4)].cpu().numpy()).all())
        e2e = {"value": world * n * args.e2e_steps / float(te.item()), "unit": "frames/s", "h2d_bytes_per_step": n * fbytes,
               "d2h_bytes_per_step": n * fbytes, "steps": args.e2e_steps, "matches_device_path": same, "numa": numa}
        if args.copy_ceiling:
            # the same bytes with no kernel in between: what the host side of the box can move with `world` ranks copying at once
            s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()   # both directions at once, like the pipelined e2e call
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                with torch.cuda.stream(s_up):
                    d_in.copy_(h_in, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    h_out.copy_(d_out, non_blocking=True)
            torch.cuda.synchronize()
            dtc = time.perf_counter() - t0
            tc = torch.tensor([dtc], dtype=torch.float64, device="cuda")
            if dist:
                dist.all_reduce(tc, op=dist.ReduceOp.MAX)
            ceil_fps = world * n * args.e2e_steps / float(tc.item())
            e2e["copy_ceiling"] = {"frames_per_s": ceil_fps, "GBps_per_rank_each_way": n * fbytes * args.e2e_steps / float(tc.item()) / 1e9,
                                   "e2e_frac_of_ceiling": e2e["value"] / ceil_fps,
                                   "what": "H2D of the step's inputs and D2H of its outputs on two streams (full duplex), all ranks at once, no kernels"}

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return 0

    peak, peak_kind = measured_peak()
    px_per_launch = float(n) * W * H  # every pass covers the whole batch (sub-batched inside the call)
    kern = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    tj = json.load(open(tp)) if os.path.exists(tp) else {}
    for k, (kms, cnt) in prof.items():
        if cnt:
            per_step_ms = kms / args.steps
            kern[k] = {"ms_per_step": per_step_ms, "launches_per_step": cnt / args.steps,
                       "algo_GBps": ALGO_BPP[k] * px_per_launch / (per_step_ms / 1000.0) / 1e9}
            if k in tj and (W, H) == (W4K, H4K):  # DRAM bytes per pixel of the committed ncu capture (profiles/)
                kern[k]["dram_GBps"] = tj[k]["dram_bytes_per_px"] * px_per_launch / (per_step_ms / 1000.0) / 1e9
    top = max(kern, key=lambda k: kern[k]["ms_per_step"]) if kern else None
    traffic = None
    if top and top in tj and "dram_bytes_per_px" in tj[top]:
        traffic = tj[top]["dram_bytes_per_px"] * px_per_launch / kern[top]["launches_per_step"]
    roofline = None
    if top:
        lps = kern[top]["launches_per_step"]
        achieved = ALGO_BPP[top] * px_per_launch / (kern[top]["ms_per_step"] / 1000.0) / 1e9
        roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "peak_kind": peak_kind + " (sustained copy)",
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                    "algo_bytes_per_launch": ALGO_BPP[top] * px_per_launch / lps, "avg_launch_ms": kern[top]["ms_per_step"] / lps,
                    "share_of_step": kern[top]["ms_per_step"] / (ms_max / args.steps)}
    chain_gbs = CHAIN_BPP * W * H * (fps / world) / 1e9

    cpu = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        procs = max(1, min(cores, 32))
        sw, sh = 960, 540
        cfps, cdt = cpu_chain_fps(procs, sw, sh)
        cpu = {"value": cfps * (sw * sh) / float(W * H), "unit": "frames/s", "cores": procs, "kind": "port",
               "sample": "%d synthetic %dx%d frames on %d processes in %.1f s (cv2 for the OpenCV calls the reference makes, numpy "
                         "fp64 restatement for bgdehaze), scaled by pixel count to %dx%d" % (procs, sw, sh, procs, cdt, W, H)}

    line = {
        "metric": "chain_frames_per_s_4k" if (W, H) == (W4K, H4K) else "chain_frames_per_s",
        "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (histretch, aclahe) / int32+f64 (bgdehaze)", "data": "synthetic",
        "config": dict(chain_config(W, H, n), nan_frames_per_step=nan_frames,
                       nan_frames="frames of the batch whose reference result is all-NaN (S = 0/0 where Yi = Yj = 0, SURVEY 8a-D9): "
                                  "flagged and written as zeros; they run the same kernels as every other frame"),
        "gpu_launches": launches,
        "chain_hbm": {"algo_bytes_per_frame": CHAIN_BPP * W * H, "achieved_GBps_per_gpu": chain_gbs, "frac_of_peak": chain_gbs / peak,
                      "roofline_fps_per_gpu": peak * 1e9 / (CHAIN_BPP * W * H)},
        "roofline": roofline, "kernels": kern, "e2e": e2e, "cpu_baseline": cpu, "clocks": clocks,
        "checksums": [int(s) for s in sums],
    }
    if stream_res is not None:
        line["stream"] = stream_res
    print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
