"""In-tree build of libuwip.so (hand-written sm_100a CUDA behind the C ABI of include/uwip.h).

nvcc cross-compiles without a GPU; the resulting .so stays next to this file so that it travels to
the GPU box with the repository snapshot.  Objects are rebuilt only when a source or header changed.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libuwip.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["cabi.cu", "histretch.cu", "clahe.cu", "dehaze.cu", "dehaze_gf1a.cu", "synth.cu", "blurmetric.cu", "jpegio.cu", "aclahe_knee.cu", "jpegenc.cu", "jpegdec.cu"]
# the knee search restates scipy's double-precision fit: no contraction into FMA
SOURCE_FLAGS = {"aclahe_knee.cu": ["--fmad=false"]}
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256((" ".join(NVCC_FLAGS) + repr(sorted(SOURCE_FLAGS.items()))).encode())
    paths = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(ROOT, "include", "uwip.h")]
    for p in paths:
        with open(p, "rb") as f:
            h.update(p.encode() + b"\0" + f.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every CUDA translation unit for sm_100a and link libuwip.so.  Returns the path."""
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    nvcc = _nvcc()

    def cc(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + SOURCE_FLAGS.get(src, []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(cc, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-lnvjpeg_static", "-lculibos", "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
