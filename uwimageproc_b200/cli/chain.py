"""chain <input.jpg> <output.jpg> [-q=95] [-aclahe=auto [-loop=repaired|as_committed]] [-encoder=nvjpeg|exact] [-decoder=nvjpeg|exact]
      [-orientation=ignore|exif]
chain <input dir> <output dir> [options above] [-batch=64]
      the whole path on one file: histretch(V, 1/99) -> aclahe(8x8, clip 2) -> bgdehaze

-aclahe=auto: the CLAHE clip limit and block size of the frame are chosen on the device (ParametrosACLAHE, ACLAHE.py:9-129) on
the V plane of the histretch output and printed as BS and CL; when the curve fit fails the fixed 8x8 / clip 2 are used.

JPEG files are read as bytes, decoded (nvJPEG by default), enhanced and encoded (nvJPEG by default) on the GPU, and written as
bytes - the pixels never exist on the host (SURVEY 8f row N3).  Other formats take the cv2 route of the per-module CLIs
(imread -> uwip_chain_bgr8 -> imwrite).

-encoder=exact: the output JPEG is written by the project's own encoder (uwip_jpeg_encode_bgr8_batch_dev), whose file is byte
for byte what cv2.imwrite(output, <chain output>) writes at -q, as the reference's command lines do.  The default, nvjpeg,
writes nvJPEG's bytes (its own DCT, quantisation and entropy coding).

-decoder=exact: the input JPEG is read by the project's own batched decoder (uwip_jpeg_decode_bgr8_batch), whose pixels are
those cv2.imread(input) returns, as the reference's command lines read them.  The default, nvjpeg, gives nvJPEG's pixels (a
few levels away, mostly in the 4:2:0 chroma upsampling), so the two decoders give different outputs, not the same output at
different speeds.  With -decoder=exact -encoder=exact the file written is cv2.imwrite(output, chain(cv2.imread(input))), with
-aclahe=auto too, and the pixels never exist on the host: for every file with -orientation=exif, and for files without an
Exif orientation tag with the default.

-orientation=exif (needs -decoder=exact; nvJPEG does not read Exif): each file is turned by its Exif orientation as
cv2.imread does (uwip_jpeg_decode_bgr8_batch_oriented), so a photograph taken with the camera on its side comes out upright,
with width and height swapped for orientations 5 to 8.  The default, ignore, keeps the stored orientation
(cv2.IMREAD_IGNORE_ORIENTATION).

When both arguments are directories, every *.jpg / *.jpeg of the input directory is enhanced into the output directory under
the same name (what bgdehaze/main.py does over img/*.jpg -> result/): the files are grouped by size (after orientation with
-orientation=exif) and run in batches of -batch frames through the same decoder, chain and encoder; BS, CL and the notes are printed per file.  One JPEG file takes
the same route as a batch of one.
"""
import os
import sys

NOTES = (
    (4, "note: the file's entropy-coded data is bad; the frame was decoded as zeros"),
    (2, "note: the entropy curve fit failed for this frame (the reference raises); the fixed 8x8 grid and clip 2 were used"),
    (1, "note: the reference's exposure map is NaN for this frame (S = 0/0); the output is all zeros, as imwrite would store it"),
)


def _notes(flags):
    for bit, text in NOTES:
        if flags & bit:
            print(text)


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _run_jpegs(ctx, jobs, opt, named):
    """jobs: (output path, JPEG file bytes) pairs, grouped by size and run in batches of opt['batch'] frames through the
    decoder, chain and encoder that opt names.  named: each file's report starts with its name (directory mode)."""
    import torch

    exif = opt["orientation"] == "exif"
    groups = {}
    for path, data in jobs:
        groups.setdefault(ctx.jpeg_size(data) if exif else ctx.jpeg_info(data), []).append((path, data))
    auto, q = opt["aclahe"] == "auto", opt["q"]
    for (w, h), files in groups.items():
        for b0 in range(0, len(files), opt["batch"]):
            part = files[b0:b0 + opt["batch"]]
            n = len(part)
            if opt["decoder"] == "exact":
                d_in = ctx.jpeg_decode_batch_dev([d for _, d in part], orientation=exif)
                dflags = ctx.last_frame_flags(n)   # read now: the chain's call resets the flags
            else:
                d_in = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda:%d" % ctx.device)
                for i, (_, data) in enumerate(part):
                    ctx.jpeg_decode_dev(data, d_in[i])
                dflags = [0] * n
            d_out = torch.empty_like(d_in)
            if auto:
                d_bs = torch.empty(n, dtype=torch.int32, device=d_in.device)
                d_cl = torch.empty(n, dtype=torch.int32, device=d_in.device)
                ctx.chain_auto_dev(d_in, d_out, n, w, h, loop=opt["loop"], d_bs=d_bs, d_cl=d_cl)
            else:
                ctx.chain_dev(d_in, d_out, n, w, h)
            flags = ctx.last_frame_flags(n)   # waits for the context's stream, which writes BS and CL: read them after it
            if auto:
                bs, cl = d_bs.cpu().tolist(), d_cl.cpu().tolist()
            if opt["encoder"] == "exact":
                outs = ctx.jpeg_encode_batch_dev(d_out, q)
            else:
                outs = [ctx.jpeg_encode_dev(d_out[i], w, h, q) for i in range(n)]
            for i, (path, _) in enumerate(part):
                with open(path, "wb") as f:
                    f.write(outs[i])
                head = [os.path.basename(path) + ":"] if named else []
                if named or auto:
                    print(*head, *(("BS =", bs[i], "CL =", cl[i]) if auto else ()))
                _notes(int(dflags[i]) | int(flags[i]))
                print("saved", path)
    return 0


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    from ._args import parse

    pos, opt, err = parse(argv, {"q": (95, int), "aclahe": ("fixed", str), "loop": ("repaired", str), "encoder": ("nvjpeg", str),
                                "decoder": ("nvjpeg", str), "orientation": ("ignore", str), "batch": (64, int), "help": (False, bool)})
    if opt["aclahe"] not in ("fixed", "auto") or opt["loop"] not in ("repaired", "as_committed"):
        err.append("-aclahe must be fixed or auto, -loop repaired or as_committed")
    if opt["encoder"] not in ("nvjpeg", "exact"):
        err.append("-encoder must be nvjpeg or exact")
    if opt["decoder"] not in ("nvjpeg", "exact"):
        err.append("-decoder must be nvjpeg or exact")
    if opt["orientation"] not in ("ignore", "exif"):
        err.append("-orientation must be ignore or exif")
    elif opt["orientation"] == "exif" and opt["decoder"] != "exact":
        err.append("-orientation=exif needs -decoder=exact (nvJPEG does not read Exif)")
    if opt["batch"] < 1:
        err.append("-batch must be at least 1")
    if len(pos) < 2 or opt.get("help") or err:
        print(__doc__)
        return 0 if not err else -1
    from ..api import default_context

    ctx = default_context()
    src, dst = pos[0], pos[1]
    if os.path.isdir(src) and os.path.isdir(dst):
        names = sorted(f for f in os.listdir(src) if f.lower().endswith((".jpg", ".jpeg")) and os.path.isfile(os.path.join(src, f)))
        return _run_jpegs(ctx, [(os.path.join(dst, name), _read(os.path.join(src, name))) for name in names], opt, True)
    if src.lower().endswith((".jpg", ".jpeg")) and dst.lower().endswith((".jpg", ".jpeg")):
        return _run_jpegs(ctx, [(dst, _read(src))], opt, False)
    import cv2

    img = cv2.imread(src, cv2.IMREAD_COLOR)
    if img is None:
        print("Failed to read input image, exiting...")
        return -1
    if opt["aclahe"] == "auto":
        out, bs, cl = ctx.chain_auto(img, loop=opt["loop"])
        print("BS =", int(bs[0]), "CL =", int(cl[0]))
    else:
        out = ctx.chain(img)
    cv2.imwrite(dst, out)
    _notes(int(ctx.last_frame_flags(1)[0]))
    print("saved", dst)
    return 0


if __name__ == "__main__":
    sys.exit(main())
