"""chain <input.jpg> <output.jpg> [-q=95] [-aclahe=auto [-loop=repaired|as_committed]] [-encoder=nvjpeg|exact]
      the whole path on one file: histretch(V, 1/99) -> aclahe(8x8, clip 2) -> bgdehaze

-aclahe=auto: the CLAHE clip limit and block size of the frame are chosen on the device (ParametrosACLAHE, ACLAHE.py:9-129) on
the V plane of the histretch output and printed as BS and CL; when the curve fit fails the fixed 8x8 / clip 2 are used.

JPEG files go through nvJPEG on the device (uwip_chain_jpeg): the file is read as bytes, decoded, enhanced and encoded on the
GPU, and written as bytes - the pixels never exist on the host (SURVEY 8f row N3).  Other formats take the cv2 route of the
per-module CLIs (imread -> uwip_chain_bgr8 -> imwrite).

-encoder=exact: the output JPEG is written by the project's own encoder (uwip_jpeg_encode_bgr8_batch_dev), whose file is byte
for byte what cv2.imwrite(output, <chain output>) writes at -q, as the reference's command lines do.  The default, nvjpeg,
writes nvJPEG's bytes (its own DCT, quantisation and entropy coding).
"""
import sys


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    from ._args import parse

    pos, opt, err = parse(argv, {"q": (95, int), "aclahe": ("fixed", str), "loop": ("repaired", str), "encoder": ("nvjpeg", str),
                                "help": (False, bool)})
    if opt["aclahe"] not in ("fixed", "auto") or opt["loop"] not in ("repaired", "as_committed"):
        err.append("-aclahe must be fixed or auto, -loop repaired or as_committed")
    if opt["encoder"] not in ("nvjpeg", "exact"):
        err.append("-encoder must be nvjpeg or exact")
    if len(pos) < 2 or opt.get("help") or err:
        print(__doc__)
        return 0 if not err else -1
    from ..api import default_context

    ctx = default_context()
    src, dst = pos[0], pos[1]
    auto = opt["aclahe"] == "auto"
    exact = opt["encoder"] == "exact"
    jpeg = src.lower().endswith((".jpg", ".jpeg")) and dst.lower().endswith((".jpg", ".jpeg"))
    if auto and jpeg:
        import torch

        with open(src, "rb") as f:
            data = f.read()
        d_in = ctx.jpeg_decode_dev(data)
        h, w = d_in.shape[:2]
        d_out = torch.empty_like(d_in)
        d_bs = torch.empty(1, dtype=torch.int32, device=d_in.device)
        d_cl = torch.empty(1, dtype=torch.int32, device=d_in.device)
        ctx.chain_auto_dev(d_in, d_out, 1, w, h, loop=opt["loop"], d_bs=d_bs, d_cl=d_cl)
        out = ctx.jpeg_encode_batch_dev(d_out, opt["q"])[0] if exact else ctx.jpeg_encode_dev(d_out, w, h, opt["q"])
        with open(dst, "wb") as f:
            f.write(out)
        print("BS =", int(d_bs.cpu()[0]), "CL =", int(d_cl.cpu()[0]))
    elif jpeg and exact:
        import torch

        with open(src, "rb") as f:
            data = f.read()
        d_in = ctx.jpeg_decode_dev(data)
        h, w = d_in.shape[:2]
        d_out = torch.empty_like(d_in)
        ctx.chain_dev(d_in, d_out, 1, w, h)
        out = ctx.jpeg_encode_batch_dev(d_out, opt["q"])[0]
        with open(dst, "wb") as f:
            f.write(out)
    elif jpeg:
        with open(src, "rb") as f:
            data = f.read()
        out = ctx.chain_jpeg(data, quality=opt["q"])
        with open(dst, "wb") as f:
            f.write(out)
    else:
        import cv2

        img = cv2.imread(src, cv2.IMREAD_COLOR)
        if img is None:
            print("Failed to read input image, exiting...")
            return -1
        if auto:
            out, bs, cl = ctx.chain_auto(img, loop=opt["loop"])
            print("BS =", int(bs[0]), "CL =", int(cl[0]))
        else:
            out = ctx.chain(img)
        cv2.imwrite(dst, out)
    flags = ctx.last_frame_flags(1)
    if flags[0] & 2:
        print("note: the entropy curve fit failed for this frame (the reference raises); the fixed 8x8 grid and clip 2 were used")
    if flags[0] & 1:
        print("note: the reference's exposure map is NaN for this frame (S = 0/0); the output is all zeros, as imwrite would store it")
    print("saved", dst)
    return 0


if __name__ == "__main__":
    sys.exit(main())
