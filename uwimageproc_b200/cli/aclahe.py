"""aclahe <input> <output>      (modules/aclahe/src/aclahe.cpp:64-226, modules/aclahe/python/main.py:17-22)

The reference binary converts to HSV, sweeps CLAHE over 5 block sizes x 51 clip limits on the V channel, prints the
entropy table and stops at its TODO list (find the knee, pick the block size, apply, convert back, save:
aclahe.cpp:209-218).  This shim prints the same table (one pixel pass per grid on the GPU) and then carries the TODO list
out with the procedure of the Python prototype (ACLAHE.py:69-129): knee of the entropy curve -> clip limit, float16
arg-max -> block size, CLAHE on V, HSV -> BGR, imwrite.  `-grey=1` is the Python main.py: grey image in, CLAHE image out.

aclahe <input> <output> -grey=1 -device=1 [-q=95] [-loop=repaired|as_committed] [-orientation=ignore|exif]
aclahe <input dir> <output dir> -grey=1 -device=1 [-q=95] [-loop=..] [-batch=64] [-orientation=..]
      main.py with the whole procedure on the device (uwip_aclahe_u8_auto_dev): a JPEG input is read by the project's grey
      reader (the pixels of cv2.imread(input, 0)), any other format by cv2.imread(input, 0); a .jpg output is written by the
      project's grey writer (the bytes of cv2.imwrite), any other format by cv2.imwrite.  When the curve fit fails (the
      reference raises), the fixed 8x8 grid and clip 2 are used and a note is printed.  When both arguments are directories,
      every *.jpg / *.jpeg of the input directory is processed into the output directory under the same name, grouped by
      size and in batches of -batch planes; each file's name, BS, CL and notes are printed.
      -orientation=exif: a JPEG input is turned by its Exif orientation as cv2.imread(input, 0) does (the project's oriented
      grey reader), so the output is that of the host route for every file, and directory mode groups files by their size
      after orientation.  The default, ignore, keeps a JPEG file's stored orientation; the two agree on files without an
      Exif orientation tag.
"""
import os
import sys


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    from ._args import parse

    pos, opt, err = parse(argv, {"grey": (0, int), "loop": ("repaired", str), "device": (0, int), "q": (95, int), "batch": (64, int),
                                 "orientation": ("ignore", str), "help": (False, bool)})
    if opt["device"] and not opt["grey"]:
        err.append("-device=1 needs -grey=1")
    if opt["orientation"] not in ("ignore", "exif"):
        err.append("-orientation must be ignore or exif")
    elif opt["orientation"] == "exif" and not opt["device"]:
        err.append("-orientation=exif needs -grey=1 -device=1")
    if opt["device"] and opt["loop"] not in ("repaired", "as_committed"):
        err.append("-loop must be repaired or as_committed")
    if opt["batch"] < 1:
        err.append("-batch must be at least 1")
    print("ACLAHE: Automatic Contrast Limited Adaptive Histogram Equalization (B200 build)")
    if len(pos) < 2 or opt.get("help"):
        print("\n\tExample:\n\t$ aclahe input.jpg output.jpg")
        print("\tThis will apply ACLAHE to gray levels of 'input.jpg' image file, and save it into 'output.jpg'\n")
        return 0
    if err:
        for e in err:
            print(e)
        return -1
    import cv2
    import numpy as np

    from ..api import default_context
    from ..modules import aclahe as A

    print("***************************************")
    print("Input:", pos[0])
    print("Output:", pos[1])
    ctx = default_context()
    if opt["device"]:
        src, dst = pos[0], pos[1]
        if os.path.isdir(src) and os.path.isdir(dst):
            names = sorted(f for f in os.listdir(src) if f.lower().endswith((".jpg", ".jpeg")) and os.path.isfile(os.path.join(src, f)))
            return _grey_device(ctx, [(os.path.join(src, f), os.path.join(dst, f)) for f in names], opt, True)
        return _grey_device(ctx, [(src, dst)], opt, False)
    if opt["grey"]:
        img = cv2.imread(pos[0], 0)
        if img is None:
            print("Failed to read input image, exiting...")
            return -1
        BS, CL = A.ParametrosACLAHE(img, loop=opt["loop"])
        print("BS = %d, CL = %g" % (BS, CL))
        cv2.imwrite(pos[1], A.CLAHE(img, BS, CL))
        return 0
    src = cv2.imread(pos[0], cv2.IMREAD_COLOR)
    if src is None:
        print("Failed to read input image, exiting...")
        return -1
    print("Input image loaded...")
    hsv = cv2.cvtColor(src, cv2.COLOR_BGR2HSV)   # file-level glue only; the frame wrapper below converts on the GPU
    v = np.ascontiguousarray(hsv[..., 2])
    clips = np.arange(0.0, 25.0 + 1e-9, 0.5)     # aclahe.cpp:160-163: 0 ... 25 inclusive, 51 values
    for bs in A.BLOCK_SIZES:                      # the table the reference prints (aclahe.cpp:199-206), C++ entropy flavour
        print(" ".join("%g" % e for e in ctx.clahe_entropy_sweep(v, bs, clips, "cpp")))
    BS, CL = A.ParametrosACLAHE(v, loop=opt["loop"])
    print("BS = %d, CL = %g" % (BS, CL))
    cv2.imwrite(pos[1], ctx.aclahe(src, float(CL), (BS, BS)))
    return 0


def _grey_device(ctx, jobs, opt, named):
    """jobs: (input path, output path) pairs, grouped by size and run in batches of opt['batch'] planes through the grey
    reader (JPEG) or cv2.imread(.., 0), uwip_aclahe_u8_auto_dev, and the grey writer (.jpg) or cv2.imwrite.  named: each
    file's report starts with its name (directory mode)."""
    import cv2
    import torch

    from .chain import _notes

    exif = opt["orientation"] == "exif"
    groups = {}
    for src, dst in jobs:
        if src.lower().endswith((".jpg", ".jpeg")):
            with open(src, "rb") as f:
                data = f.read()
            item = (dst, data, None)
            size = ctx.jpeg_size(data) if exif else ctx.jpeg_info(data)
        else:
            img = cv2.imread(src, 0)
            if img is None:
                print("Failed to read input image, exiting...")
                return -1
            item = (dst, None, img)
            size = (img.shape[1], img.shape[0])
        groups.setdefault(size, []).append(item)
    dev = "cuda:%d" % ctx.device
    for (w, h), items in groups.items():
        for b0 in range(0, len(items), opt["batch"]):
            part = items[b0:b0 + opt["batch"]]
            n = len(part)
            if part[0][1] is not None:   # one JPEG job per batch unless in directory mode, which reads only JPEG files
                d_in = ctx.jpeg_decode_grey_batch_dev([data for _, data, _ in part], orientation=exif)
                dflags = ctx.last_frame_flags(n)   # read now: the CLAHE call resets the flags
            else:
                d_in = torch.from_numpy(part[0][2]).to(dev)[None]
                dflags = [0]
            d_out = torch.empty_like(d_in)
            d_bs = torch.empty(n, dtype=torch.int32, device=dev)
            d_cl = torch.empty(n, dtype=torch.int32, device=dev)
            ctx.aclahe_grey_auto_dev(d_in, d_out, n, w, h, loop=opt["loop"], d_bs=d_bs, d_cl=d_cl)
            flags = ctx.last_frame_flags(n)   # waits for the context's stream, which writes BS and CL
            bs, cl = d_bs.cpu().tolist(), d_cl.cpu().tolist()
            jpeg_out = [i for i, (dst, _, _) in enumerate(part) if dst.lower().endswith((".jpg", ".jpeg"))]
            files = dict(zip(jpeg_out, ctx.jpeg_encode_grey_batch_dev(d_out[jpeg_out], opt["q"]))) if jpeg_out else {}
            for i, (dst, _, _) in enumerate(part):
                if i in files:
                    with open(dst, "wb") as f:
                        f.write(files[i])
                else:
                    cv2.imwrite(dst, d_out[i].cpu().numpy(), [cv2.IMWRITE_JPEG_QUALITY, opt["q"]])
                print(*([os.path.basename(dst) + ":"] if named else []), "BS = %d, CL = %g" % (bs[i], cl[i]))
                _notes(int(dflags[i]) | int(flags[i]))
                if named:
                    print("saved", dst)
    return 0


if __name__ == "__main__":
    sys.exit(main())
