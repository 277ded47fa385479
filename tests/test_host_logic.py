"""CPU tests of the host side: the C ABI surface (library loads, exports every declared symbol, fails
loudly without a device - no compute calls), and the N>1 frame-batch sharding under gloo, world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "uwip.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(uwip_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from uwimageproc_b200 import _lib

    names = _declared_symbols()
    assert len(names) >= 40
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "libuwip.so does not export %s" % n
    # the ctypes binding covers the whole header, one to one
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.load().uwip_version() == 100


def test_letter_maps_match_reference():
    """numChannel / numSpace (preprocessing.cpp:147-161) are pure host logic."""
    from uwimageproc_b200 import _lib

    lib = _lib.load()
    chan = {"R": 0, "G": 1, "B": 2, "H": 0, "S": 1, "V": 2, "h": 0, "s": 1, "l": 2, "L": 0, "a": 1, "b": 2, "Y": 0, "C": 1, "X": 2, "r": -1, "?": -1}
    space = {"R": 0, "G": 0, "B": 0, "H": 1, "S": 1, "V": 1, "h": 2, "s": 2, "l": 2, "L": 3, "a": 3, "b": 3, "Y": 4, "C": 4, "X": 4, "r": -1}
    for c, v in chan.items():
        assert lib.uwip_num_channel(c.encode()) == v, c
    for c, v in space.items():
        assert lib.uwip_num_space(c.encode()) == v, c


def test_no_cpu_fallback():
    """Without an sm_100 device every operation must fail loudly (status -2), never compute on the host."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    import uwimageproc_b200 as u

    with pytest.raises(u.UwipError) as e:
        u.Context(0)
    assert e.value.status == -2 and "no CPU fallback" in str(e.value)
    # the reference-named Python modules are thin wrappers over the same context: same failure
    from uwimageproc_b200.modules import bgdehaze

    with pytest.raises(u.UwipError):
        bgdehaze.Background_light(np.zeros((8, 8, 3), np.uint8) + np.arange(8, dtype=np.uint8)[None, :, None] * 30)


def test_product_does_not_import_the_oracle():
    """oracle/ is test infrastructure: nothing under uwimageproc_b200/ may import or execute it."""
    pkg = os.path.join(ROOT, "uwimageproc_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(d, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(d, f)


def test_frame_ranges_partition_the_stream():
    from uwimageproc_b200.shard import batches, frame_range

    for total in [0, 1, 7, 256, 10000]:
        for world in [1, 2, 4, 8]:
            got = []
            for r in range(world):
                f, c = frame_range(r, world, total)
                got += list(range(f, f + c))
            assert got == list(range(total))
            sizes = [frame_range(r, world, total)[1] for r in range(world)]
            assert max(sizes) - min(sizes) <= 1
    assert batches(10, 7, 3) == [(10, 3), (13, 3), (16, 1)]
    with pytest.raises(ValueError):
        frame_range(2, 2, 10)


_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import torch.distributed as dist
from uwimageproc_b200.shard import frame_range, gather_checksums
from uwimageproc_b200.api import host_checksum
from oracle import uwip_oracle as O   # test infrastructure: frames for the checksums

rank, world, total = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(sys.argv[2])
dist.init_process_group("gloo", rank=rank, world_size=world)
first, count = frame_range(rank, world, total)
frames = np.stack([O.synth_frame(0x5EED0005, first + i, 64, 36) for i in range(count)]) if count else np.zeros((0, 36, 64, 3), np.uint8)
sums = host_checksum(frames) if count else np.zeros(0, np.uint64)
allsums = gather_checksums(sums, rank, world, total, dist)
ref = host_checksum(np.stack([O.synth_frame(0x5EED0005, i, 64, 36) for i in range(total)]))
assert (allsums == ref).all(), (rank, allsums, ref)
dist.barrier()
dist.destroy_process_group()
print("rank %d ok %d frames" % (rank, count))
"""


def test_two_rank_sharding_gloo(tmp_path):
    """world_size 2 over gloo on the CPU: disjoint contiguous ranges, per-frame checksums gathered in stream
    order equal the single-process checksums (the frames themselves never cross ranks)."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29500 + os.getpid() % 500), WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, "7"], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, p in enumerate(procs):
        assert p.returncode == 0, outs[r]
    assert "rank 0 ok 4 frames" in outs[0] and "rank 1 ok 3 frames" in outs[1]


def test_lab_tables_match_the_oracle():
    """The committed lab_tables.inc (product side, built by csrc/gen_lab_tables.py) holds the oracle's tables."""
    import re

    from oracle import uwip_oracle as O

    txt = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "uwimageproc_b200", "csrc", "lab_tables.inc")).read()

    def arr(name):
        m = re.search(name + r"\[\d+\] = \{(.*?)\};", txt, re.S)
        return np.array([int(v) for v in m.group(1).replace("\n", " ").split(",")], np.int64)

    gamma, cbrt, fwd, yf, invgamma, inv = O.lab_tables()
    assert (arr("kLabGamma") == gamma).all()
    assert (arr("kLabCbrt") == cbrt[:2048]).all()
    assert (arr("kLabYF") == yf).all()
    assert (arr("kLabInvGamma") == invgamma).all()
    assert [int(v) for v in re.search(r"LAB_FWD_COEFFS \{(.*?)\}", txt).group(1).split(",")] == list(fwd)
    assert [int(v) for v in re.search(r"LAB_INV_COEFFS \{(.*?)\}", txt).group(1).split(",")] == list(inv)


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the CUDA arm): ONE JSON line on stdout with the
    contract's keys, the same `config` dictionary as the CUDA arm, no GPU needed."""
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "chain_frames_per_s_4k" and d["unit"] == "frames/s" and d["higher_is_better"]
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    sys.path.insert(0, root)
    import bench

    assert d["config"] == bench.chain_config(3840, 2160, 256)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs DIR`: float32 .npy files of what the timed call returned, the whole batch when it is small,
    otherwise the same seeded sample of positions on every run; at most 64 MB for the default 256-frame 4K batch."""
    import torch

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench

    assert 4 * bench.DUMP_SAMPLE + 4 * 256 <= 64 << 20
    out = np.random.default_rng(2).integers(0, 256, (3, 20, 30, 3), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path / "a"), torch.from_numpy(out), np.array([0, 1, 0], np.int32))
    frames, flags = np.load(tmp_path / "a" / "frames.npy"), np.load(tmp_path / "a" / "frame_flags.npy")
    assert frames.dtype == flags.dtype == np.float32
    assert (frames == out).all() and flags.tolist() == [0, 1, 0]
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), torch.from_numpy(out), np.zeros(3, np.int32))
    b, c = np.load(tmp_path / "b" / "frames.npy"), np.load(tmp_path / "c" / "frames.npy")
    assert b.dtype == np.float32 and 900 < b.size <= 1000 and (b == c).all()
    pos = np.unique(np.random.default_rng(bench.SEED).integers(0, out.size, 1000))
    assert (b == out.reshape(-1)[pos]).all()
    # the reference arm keeps no outputs: asking it for them is an error, not a silent no-op
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "r")],
                       capture_output=True, text=True, timeout=60, cwd=root)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "r").exists()


def test_cli_argument_conventions():
    """The CLI shims keep cv::CommandLineParser's `-key=value` convention and the reference's defaults (histretch.cpp:68-74)."""
    from uwimageproc_b200.cli._args import parse

    keys = {"c": ("r", str), "cuda": (1, int), "time": (0, int), "help": (False, bool)}
    pos, opt, err = parse(["in.jpg", "out.jpg", "-c=HV", "-cuda=0", "--time=1", "-unknown=3"], keys)
    assert pos == ["in.jpg", "out.jpg"] and opt["c"] == "HV" and opt["cuda"] == 0 and opt["time"] == 1 and not err
    pos, opt, err = parse(["a", "b"], keys)
    assert opt["c"] == "r" and opt["time"] == 0          # the reference's default letter is the unrecognised lowercase r
    assert parse(["-h"], keys)[1]["help"] is True
    assert parse(["a", "b", "-time=x"], keys)[2]
    from uwimageproc_b200.cli import aclahe, bgdehaze_main, histretch

    assert histretch.main([]) == 0 and aclahe.main([]) == 0   # help paths need no GPU
    assert bgdehaze_main.get_filenames("/nonexistent") == []


def test_e2e_schedule_header(tmp_path):
    """The sub-batch schedule of uwip_chain_bgr8 (csrc/e2e_schedule.h, plain C++): every schedule adds up to the batch, stays
    inside the workspace cap, and the 4K / 148-SM / 256-frame one is the measured ramp."""
    import shutil

    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    src = tmp_path / "sched.cpp"
    src.write_text(
        '#include <cstdio>\n#include <cstdlib>\n#include "e2e_schedule.h"\n'
        "int main(int argc, char** argv) {\n"
        "  auto v = e2e_schedule(atoi(argv[1]), atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]));\n"
        '  for (int x : v) printf("%d ", x);\n  printf("\\n");\n  return 0;\n}\n')
    exe = tmp_path / "sched"
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "uwimageproc_b200", "csrc"), str(src), "-o", str(exe)], check=True)

    def sched(n, nb, sms=148, sw=8, sn=9):
        out = subprocess.run([str(exe)] + [str(a) for a in (n, nb, sms, sw, sn)], check=True, capture_output=True, text=True).stdout
        return [int(t) for t in out.split()]

    assert sched(256, 148) == [4, 8, 16, 24, 37, 55, 55, 32, 16, 6, 3]
    for n in list(range(1, 70)) + [100, 127, 200, 255, 256, 257, 1000, 1024]:
        for nb in (1, 3, 20, 55, 148):
            for (sms, sw, sn) in ((148, 8, 9), (148, 1, 1), (132, 4, 5), (148, 40, 44)):
                v = sched(n, nb, sms, sw, sn)
                assert sum(v) == n and min(v) >= 1 and max(v) <= nb, (n, nb, sms, sw, sn, v)
                if n > 1:
                    assert len(v) >= 2, (n, nb, v)   # at least two sub-batches: a copy overlaps a compute
