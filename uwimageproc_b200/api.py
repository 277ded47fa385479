"""Thin numpy-level wrapper over the C ABI.  Plumbing only: argument checking, pointer passing."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import ChainParams, DehazeParams, UwipError

HSV_ROUND = {"cv2": 0, "trunc": 1, "rint": 2}
ACLAHE_LOOP = {"repaired": 0, "as_committed": 1}
JPEG_GREY, JPEG_ORIENT = 1, 2   # the flags of uwip_jpeg_decode_batch_ex
ORDER = {"intended": 0, "literal": 1}


def _ptr(a):
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or device)
        return a.data_ptr()
    return int(a)


def _plane(a):
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError("expected an 8-bit single-channel image (H, W)")
    if a.strides[1] != 1:
        a = np.ascontiguousarray(a)
    return a


def _frame(a):
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("expected an 8-bit BGR image (H, W, 3)")
    if a.strides[2] != 1 or a.strides[1] != 3:
        a = np.ascontiguousarray(a)
    return a


def _frames(a):
    """uint8 (N, H, W, 3) or (H, W, 3) host frames -> (contiguous (N, H, W, 3) array, whether one frame was given)."""
    a = np.asarray(a)
    single = a.ndim == 3
    if single:
        a = a[None]
    if a.dtype != np.uint8 or a.ndim != 4 or a.shape[3] != 3:
        raise ValueError("expected uint8 (N, H, W, 3)")
    return np.ascontiguousarray(a), single


class Context:
    """One context per (host thread, device); all work is ordered on its stream."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.uwip_create(int(device), C.byref(h))
        if rc != 0:
            raise UwipError(rc, (self.lib.uwip_last_error(None) or b"").decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.uwip_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise UwipError(rc, (self.lib.uwip_last_error(self.h) or b"").decode())

    # ---- bookkeeping -------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self.lib.uwip_set_stream(self.h, C.c_void_p(int(cuda_stream_ptr))))

    def synchronize(self):
        self._ck(self.lib.uwip_synchronize(self.h))

    def launch_count(self):
        return int(self.lib.uwip_launch_count(self.h))

    def profile(self, enable):
        self._ck(self.lib.uwip_profile(self.h, 1 if enable else 0))

    def profile_read(self, tag):
        ms, n = C.c_double(), C.c_int64()
        self._ck(self.lib.uwip_profile_read(self.h, tag.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # ---- preprocessing.cpp ---------------------------------------------------------------------
    def histogram(self, plane):
        p = _plane(plane)
        out = np.empty(256, np.float32)
        self._ck(self.lib.uwip_histogram_u8(self.h, _ptr(p), p.shape[1], p.shape[0], p.strides[0], _ptr(out)))
        return out

    def channel_stretch(self, plane, lo=0, hi=100, out=None, return_bins=False):
        p = _plane(plane)
        if out is None:
            out = np.empty(p.shape, np.uint8)
        low, high = C.c_int(), C.c_int()
        self._ck(self.lib.uwip_channel_stretch_u8(self.h, _ptr(p), p.strides[0], _ptr(out), out.strides[0],
                                                  p.shape[1], p.shape[0], lo, hi, C.byref(low), C.byref(high)))
        return (out, low.value, high.value) if return_bins else out

    def histretch(self, frame, channels="V", lo=2, hi=98, order="intended", hsv_round="cv2"):
        f = _frame(frame)
        out = np.empty(f.shape, np.uint8)
        self._ck(self.lib.uwip_histretch_bgr8(self.h, _ptr(f), f.strides[0], _ptr(out), out.strides[0], f.shape[1],
                                              f.shape[0], channels.encode(), lo, hi, ORDER[order], HSV_ROUND[hsv_round]))
        return out

    # ---- aclahe ----------------------------------------------------------------------------------
    def clahe(self, plane, clip=40.0, tiles=(8, 8)):
        p = _plane(plane)
        out = np.empty(p.shape, np.uint8)
        self._ck(self.lib.uwip_clahe_u8(self.h, _ptr(p), p.strides[0], _ptr(out), out.strides[0], p.shape[1], p.shape[0],
                                        float(clip), int(tiles[0]), int(tiles[1])))
        return out

    def entropy(self, plane, flavour="cpp"):
        p = _plane(plane)
        e = C.c_float()
        self._ck(self.lib.uwip_entropy_u8(self.h, _ptr(p), p.shape[1], p.shape[0], p.strides[0],
                                          0 if flavour == "cpp" else 1, C.byref(e)))
        return np.float32(e.value)

    def gaussian_blur3(self, plane):
        p = _plane(plane)
        out = np.empty(p.shape, np.uint8)
        self._ck(self.lib.uwip_gaussian_blur3_u8(self.h, _ptr(p), p.strides[0], _ptr(out), out.strides[0], p.shape[1], p.shape[0]))
        return out

    def clahe_entropy_sweep(self, plane, tiles, clips, flavour="py"):
        p = _plane(plane)
        clips = np.ascontiguousarray(clips, dtype=np.float64)
        out = np.empty(len(clips), np.float32)
        self._ck(self.lib.uwip_clahe_entropy_sweep_u8(
            self.h, _ptr(p), p.shape[1], p.shape[0], p.strides[0], int(tiles),
            clips.ctypes.data_as(C.POINTER(C.c_double)), len(clips), 0 if flavour == "cpp" else 1,
            out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def clahe_entropy_sweep_dev(self, d_planes, n, width, height, grids, clips, flavour="py"):
        """n device planes x grids x clips -> float32 [n][len(grids)][len(clips)] (one pixel pass per grid)."""
        grids = np.ascontiguousarray(grids, dtype=np.int32)
        clips = np.ascontiguousarray(clips, dtype=np.float64)
        out = np.empty((n, len(grids), len(clips)), np.float32)
        self._ck(self.lib.uwip_clahe_entropy_sweep_u8_dev(
            self.h, _ptr(d_planes), n, width, height, grids.ctypes.data_as(C.POINTER(C.c_int)), len(grids),
            clips.ctypes.data_as(C.POINTER(C.c_double)), len(clips), 0 if flavour == "cpp" else 1,
            out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def aclahe(self, frame, clip=2.0, tiles=(8, 8), hsv_round="cv2"):
        f = _frame(frame)
        out = np.empty(f.shape, np.uint8)
        self._ck(self.lib.uwip_aclahe_bgr8(self.h, _ptr(f), f.strides[0], _ptr(out), out.strides[0], f.shape[1], f.shape[0],
                                           float(clip), int(tiles[0]), int(tiles[1]), HSV_ROUND[hsv_round]))
        return out

    # ---- bgdehaze ----------------------------------------------------------------------------------
    def dehaze_params(self, window=15, radius=40, eps=1e-3, tmin=0.2):
        return DehazeParams(int(window), int(radius), float(eps), float(tmin))

    def background_light(self, frame, window=15):
        f = _frame(frame)
        B = (C.c_double * 3)()
        idx = (C.c_int64 * 2)()
        self._ck(self.lib.uwip_background_light_bgr8(self.h, _ptr(f), f.strides[0], f.shape[1], f.shape[0], int(window), B, idx))
        return np.array(B[:]), (int(idx[0]), int(idx[1]))

    def transmission(self, frame, window=15):
        f = _frame(frame)
        tb = np.empty(f.shape[:2], np.float64)
        tg = np.empty(f.shape[:2], np.float64)
        self._ck(self.lib.uwip_transmission_bgr8(self.h, _ptr(f), f.strides[0], f.shape[1], f.shape[0], int(window), _ptr(tb), _ptr(tg)))
        return tb, tg

    def boxfilter(self, plane, r):
        a = np.ascontiguousarray(plane, dtype=np.float64)
        if a.ndim != 2:
            raise ValueError("expected an H x W float64 plane")
        out = np.empty(a.shape, np.float64)
        self._ck(self.lib.uwip_boxfilter_f64(self.h, _ptr(a), a.shape[1], a.shape[0], int(r), _ptr(out)))
        return out

    def guided_filter_u8(self, guide8, rng, p, r=40, eps=1e-3):
        g = _frame(guide8)
        pp = np.ascontiguousarray(p, dtype=np.float64)
        if pp.shape != g.shape[:2]:
            raise ValueError("p must be H x W")
        out = np.empty(pp.shape, np.float64)
        self._ck(self.lib.uwip_guided_filter_u8(self.h, _ptr(g), g.strides[0], g.shape[1], g.shape[0], int(rng), _ptr(pp), int(r),
                                                float(eps), _ptr(out)))
        return out

    def refined_transmission(self, frame, params=None):
        f = _frame(frame)
        tb = np.empty(f.shape[:2], np.float64)
        tg = np.empty(f.shape[:2], np.float64)
        p = params or self.dehaze_params()
        self._ck(self.lib.uwip_refined_transmission_bgr8(self.h, _ptr(f), f.strides[0], f.shape[1], f.shape[0], C.byref(p), _ptr(tb), _ptr(tg)))
        return tb, tg

    def rc_correction(self, frame, params=None):
        f = _frame(frame)
        out = np.empty(f.shape, np.float64)
        p = params or self.dehaze_params()
        self._ck(self.lib.uwip_rc_correction_bgr8(self.h, _ptr(f), f.strides[0], f.shape[1], f.shape[0], C.byref(p), _ptr(out)))
        return out

    def exposure_stages(self, frame, params=None):
        """adaptiveExp_map's intermediates from one full bgdehaze run of the frame (uwip_exposure_stages_bgr8): dict of
        numpy arrays ycc (H, W, 4) uint8 (Yi, Cri, Cbi, Yj), splane (H, W) uint32 (rint(S 2^28)), refined_s (H, W)
        float32, restored and out (H, W, 3) float64, and the scalars yi_min, yi_max, yj_min, yj_max, nan_flag."""
        f = _frame(frame)
        h, w = f.shape[:2]
        ycc = np.empty((h, w), np.uint32)
        splane = np.empty((h, w), np.uint32)
        refs = np.empty((h, w), np.float32)
        restored = np.empty(f.shape, np.float64)
        out = np.empty(f.shape, np.float64)
        stats = np.empty(5, np.uint32)
        p = params or self.dehaze_params()
        self._ck(self.lib.uwip_exposure_stages_bgr8(self.h, _ptr(f), f.strides[0], w, h, C.byref(p), _ptr(ycc), _ptr(splane),
                                                    _ptr(refs), _ptr(restored), _ptr(out), _ptr(stats)))
        d = dict(ycc=ycc.view(np.uint8).reshape(h, w, 4), splane=splane, refined_s=refs, restored=restored, out=out)
        d.update(zip(("yi_min", "yi_max", "yj_min", "yj_max", "nan_flag"), (int(v) for v in stats)))
        return d

    def bgdehaze(self, frame, params=None, return_float=False):
        f = _frame(frame)
        out8 = np.empty(f.shape, np.uint8)
        outf = np.empty(f.shape, np.float64) if return_float else None
        p = params or self.dehaze_params()
        self._ck(self.lib.uwip_bgdehaze_bgr8(self.h, _ptr(f), f.strides[0], _ptr(out8), out8.strides[0], f.shape[1], f.shape[0],
                                             C.byref(p), _ptr(outf) if return_float else None))
        return (out8, outf) if return_float else out8

    # ---- chain ------------------------------------------------------------------------------------------
    def chain_params(self, channels="V", lo=1, hi=99, order="intended", hsv_round="cv2", clip=2.0, tiles=(8, 8),
                     window=15, radius=40, eps=1e-3, tmin=0.2):
        p = ChainParams()
        self.lib.uwip_chain_defaults(C.byref(p))
        p.channels = channels.encode()
        p.lo, p.hi, p.order, p.hsv_round = lo, hi, ORDER[order], HSV_ROUND[hsv_round]
        p.clip, p.tiles_x, p.tiles_y = float(clip), int(tiles[0]), int(tiles[1])
        p.dehaze = DehazeParams(int(window), int(radius), float(eps), float(tmin))
        return p

    def chain(self, frames, params=None):
        """frames: uint8 (N, H, W, 3) or (H, W, 3) host array -> same shape."""
        a, single = _frames(frames)
        out = np.empty_like(a)
        p = params or self.chain_params()
        self._ck(self.lib.uwip_chain_bgr8(self.h, _ptr(a), _ptr(out), a.shape[0], a.shape[2], a.shape[1], C.byref(p)))
        return out[0] if single else out

    def chain_auto(self, frames, params=None, loop="repaired"):
        """The chain with automatic CLAHE parameters on a host array: frames uint8 (N, H, W, 3) or (H, W, 3) ->
        (out of the same shape, BS int32[N], CL int32[N]); BS = CL = -1 where the fit failed (those frames used
        params' fixed clip and tiles)."""
        import torch

        a, single = _frames(frames)
        n, h, w = a.shape[:3]
        with torch.cuda.device(self.device):
            d_src = torch.from_numpy(a).to("cuda")
            d_dst = torch.empty_like(d_src)
            d_bs = torch.empty(n, dtype=torch.int32, device="cuda")
            d_cl = torch.empty(n, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            self.chain_auto_dev(d_src, d_dst, n, w, h, params, loop, d_bs, d_cl)
            self.synchronize()
            out, bs, cl = d_dst.cpu().numpy(), d_bs.cpu().numpy(), d_cl.cpu().numpy()
        return (out[0] if single else out), bs, cl

    def chain_host_ptr(self, src_ptr, dst_ptr, n, width, height, params=None):
        p = params or self.chain_params()
        self._ck(self.lib.uwip_chain_bgr8(self.h, int(src_ptr), int(dst_ptr), n, width, height, C.byref(p)))

    # ---- device-pointer variants (pointers as ints, e.g. torch tensor.data_ptr()) ----------------------
    def chain_dev(self, d_src, d_dst, n, width, height, params=None):
        p = params or self.chain_params()
        self._ck(self.lib.uwip_chain_bgr8_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, C.byref(p)))

    def chain_auto_dev(self, d_src, d_dst, n, width, height, params=None, loop="repaired", d_bs=None, d_cl=None):
        """The chain with the CLAHE clip limit and grid of every frame found on the device (ParametrosACLAHE on the V plane
        of the histretch output); d_bs, d_cl: optional device int32[n] outputs."""
        p = params or self.chain_params()
        self._ck(self.lib.uwip_chain_bgr8_auto_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, C.byref(p), ACLAHE_LOOP[loop],
                                                   _ptr(d_bs) if d_bs is not None else None, _ptr(d_cl) if d_cl is not None else None))

    # ---- JPEG files to and from the device (nvJPEG) ------------------------------------------------
    def jpeg_info(self, data):
        buf = np.frombuffer(bytes(data), np.uint8)
        w, h = C.c_int(), C.c_int()
        self._ck(self.lib.uwip_jpeg_info(self.h, _ptr(buf), buf.size, C.byref(w), C.byref(h)))
        return w.value, h.value

    def jpeg_decode_dev(self, data, d_bgr=None):
        """JPEG bytes -> bgr8 frame on the device (torch uint8 tensor H x W x 3 unless one is passed in)."""
        buf = np.frombuffer(bytes(data), np.uint8)
        w, h = self.jpeg_info(data)
        if d_bgr is None:
            import torch

            d_bgr = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
        self._ck(self.lib.uwip_jpeg_decode_bgr8_dev(self.h, _ptr(buf), buf.size, _ptr(d_bgr), w, h))
        self.synchronize()
        return d_bgr

    def jpeg_encode_dev(self, d_bgr, width, height, quality=95):
        n = C.c_size_t()
        cap = width * height * 3 + 65536
        out = np.empty(cap, np.uint8)
        self._ck(self.lib.uwip_jpeg_encode_bgr8_dev(self.h, _ptr(d_bgr), width, height, int(quality), _ptr(out), cap, C.byref(n)))
        return out[: n.value].tobytes()

    def chain_jpeg(self, data, params=None, quality=95):
        """JPEG bytes in -> chain on the device -> JPEG bytes out."""
        buf = np.frombuffer(bytes(data), np.uint8)
        w, h = self.jpeg_info(data)
        p = params or self.chain_params()
        n = C.c_size_t()
        cap = w * h * 3 + 65536
        out = np.empty(cap, np.uint8)
        self._ck(self.lib.uwip_chain_jpeg(self.h, _ptr(buf), buf.size, C.byref(p), int(quality), _ptr(out), cap, C.byref(n)))
        return out[: n.value].tobytes()

    # ---- JPEG files byte-identical to cv2.imwrite (csrc/jpegenc.cu) ---------------------------------------------
    def jpeg_encode_bound(self, width, height):
        """Largest file uwip_jpeg_encode_bgr8_batch_dev can write for one width x height frame (0 outside 1..65535)."""
        return int(self.lib.uwip_jpeg_encode_bound(int(width), int(height)))

    def jpeg_encode_batch_dev(self, d_frames, quality=95):
        """Device bgr8 frames (torch uint8 tensor (N, H, W, 3) or (H, W, 3)) -> list of N files, each the bytes of
        cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, quality]).  The batch is encoded in one device call; then the
        lengths are read and only each file's bytes are copied to the host."""
        import torch

        d = d_frames.unsqueeze(0) if d_frames.dim() == 3 else d_frames
        if d.dtype != torch.uint8 or d.dim() != 4 or d.shape[3] != 3 or not d.is_cuda:
            raise ValueError("expected a uint8 CUDA tensor (N, H, W, 3)")
        return self._jpeg_encode_batch(d, quality, self.jpeg_encode_bound(d.shape[2], d.shape[1]), self.lib.uwip_jpeg_encode_bgr8_batch_dev)

    def _jpeg_encode_batch(self, d, quality, stride, encode):
        import torch

        n, h, w = d.shape[:3]
        with torch.cuda.device(d.device):
            d = d.contiguous()
            d_out = torch.empty((n, max(stride, 1)), dtype=torch.uint8, device=d.device)
            d_len = torch.empty(n, dtype=torch.int64, device=d.device)
            torch.cuda.current_stream().synchronize()   # the frames are complete before the context's stream reads them
            self._ck(encode(self.h, _ptr(d), n, w, h, int(quality), _ptr(d_out), stride, _ptr(d_len)))
            self.synchronize()
            lens = d_len.cpu().tolist()
            return [d_out[f, :lens[f]].cpu().numpy().tobytes() for f in range(n)]

    def jpeg_encode(self, frames, quality=95):
        """Host bgr8 frames (N, H, W, 3) -> list of N files; one frame (H, W, 3) -> its file.  The bytes are those of
        cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, quality]), encoded on the device."""
        import torch

        a, single = _frames(frames)
        with torch.cuda.device(self.device):
            out = self.jpeg_encode_batch_dev(torch.from_numpy(a).to("cuda"), quality)
        return out[0] if single else out

    def jpeg_encode_grey_bound(self, width, height):
        """Largest file uwip_jpeg_encode_u8_batch_dev can write for one width x height plane (0 outside 1..65535)."""
        return int(self.lib.uwip_jpeg_encode_u8_bound(int(width), int(height)))

    def jpeg_encode_grey_batch_dev(self, d_planes, quality=95):
        """Device grey planes (torch uint8 tensor (N, H, W) or (H, W)) -> list of N files, each the bytes of
        cv2.imencode(".jpg", plane, [cv2.IMWRITE_JPEG_QUALITY, quality]) (one-component JPEG), encoded in one device call."""
        import torch

        d = d_planes.unsqueeze(0) if d_planes.dim() == 2 else d_planes
        if d.dtype != torch.uint8 or d.dim() != 3 or not d.is_cuda:
            raise ValueError("expected a uint8 CUDA tensor (N, H, W)")
        return self._jpeg_encode_batch(d, quality, self.jpeg_encode_grey_bound(d.shape[2], d.shape[1]), self.lib.uwip_jpeg_encode_u8_batch_dev)

    def jpeg_encode_grey(self, planes, quality=95):
        """Host grey planes (N, H, W) -> list of N files; one plane (H, W) -> its file: cv2.imencode's bytes, encoded on the
        device."""
        import torch

        a = np.asarray(planes)
        single = a.ndim == 2
        if a.dtype != np.uint8 or a.ndim not in (2, 3):
            raise ValueError("expected uint8 (N, H, W) or (H, W)")
        with torch.cuda.device(self.device):
            out = self.jpeg_encode_grey_batch_dev(torch.from_numpy(np.ascontiguousarray(a)).to("cuda"), quality)
        return out[0] if single else out

    # ---- JPEG files decoded as cv2.imdecode does (csrc/jpegdec.cu) ---------------------------------------------------
    def jpeg_decode_batch_dev(self, files, d_out=None, orientation=False, progressive=False):
        """JPEG files of one size (a list of bytes, or one bytes object) -> torch uint8 CUDA tensor (N, H, W, 3) holding
        cv2.imdecode(file, cv2.IMREAD_COLOR | cv2.IMREAD_IGNORE_ORIENTATION) of each, decoded in one device call; with
        orientation=True, cv2.imdecode(file, cv2.IMREAD_COLOR): each file's Exif orientation applied, and "one size" is the
        size after it (jpeg_size).  A file with bad entropy-coded data decodes to zeros and sets bit 4 of
        last_frame_flags(N).  progressive=True: progressive files are read too, in the same batch as sequential ones
        (uwip_jpeg_decode_batch_ex); a progression incomplete at EOI is refused."""
        if progressive:
            return self._jpeg_decode_batch(files, d_out, 3, self._decode_ex(orientation, False), orientation, True)
        decode = self.lib.uwip_jpeg_decode_bgr8_batch_oriented if orientation else self.lib.uwip_jpeg_decode_bgr8_batch
        return self._jpeg_decode_batch(files, d_out, 3, decode, orientation)

    def jpeg_decode_grey_batch_dev(self, files, d_out=None, orientation=False, progressive=False):
        """JPEG files of one size -> torch uint8 CUDA tensor (N, H, W) holding cv2.imdecode(file, cv2.IMREAD_GRAYSCALE |
        cv2.IMREAD_IGNORE_ORIENTATION) of each (for a colour file its Y component), decoded in one device call; with
        orientation=True, cv2.imdecode(file, cv2.IMREAD_GRAYSCALE), the Exif orientation applied.  Bad entropy-coded data:
        zeros and bit 4 of last_frame_flags(N).  progressive=True: progressive files are read too."""
        if progressive:
            return self._jpeg_decode_batch(files, d_out, 1, self._decode_ex(orientation, True), orientation, True)
        decode = self.lib.uwip_jpeg_decode_u8_batch_oriented if orientation else self.lib.uwip_jpeg_decode_u8_batch
        return self._jpeg_decode_batch(files, d_out, 1, decode, orientation)

    def _decode_ex(self, orientation, grey):
        """uwip_jpeg_decode_batch_ex with the flags of one reader, in the argument order of the other readers"""
        flags = (JPEG_GREY if grey else 0) | (JPEG_ORIENT if orientation else 0)
        return lambda h, ptrs, lens, n, out, w, hh: self.lib.uwip_jpeg_decode_batch_ex(h, ptrs, lens, n, out, w, hh, flags)

    def jpeg_probe(self, data):
        """(width, height, orientation, progressive) of JPEG file `data` from the host marker reader of the progressive-capable
        reader, without the device: the size is that of the image cv2.imdecode returns (after the Exif orientation)."""
        buf = np.frombuffer(bytes(data), np.uint8)
        w, h, o, p = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        rc = self.lib.uwip_jpeg_probe(_ptr(buf), buf.size, C.byref(w), C.byref(h), C.byref(o), C.byref(p))
        if rc != 0:
            raise UwipError(rc, "uwip_jpeg_probe: the JPEG header is malformed, its coding is not supported or its progression is "
                                "incomplete")
        return w.value, h.value, o.value, bool(p.value)

    def jpeg_orientation(self, data):
        """The Exif orientation (1..8) cv2.imdecode applies to JPEG file `data`; 1 when it has none (host marker reader)."""
        buf = np.frombuffer(bytes(data), np.uint8)
        o = C.c_int()
        rc = self.lib.uwip_jpeg_orientation(_ptr(buf), buf.size, C.byref(o))
        if rc != 0:
            raise UwipError(rc, "uwip_jpeg_orientation: the JPEG header is malformed or its coding is not supported")
        return o.value

    def jpeg_size(self, data, orientation=True):
        """(width, height) of the image cv2.imdecode returns for JPEG file `data`: the stored size, transposed for Exif
        orientations 5 to 8 unless orientation=False."""
        w, h = self.jpeg_info(data)
        return (h, w) if orientation and self.jpeg_orientation(data) >= 5 else (w, h)

    def _jpeg_decode_batch(self, files, d_out, channels, decode, orientation, progressive=False):
        import torch

        if isinstance(files, (bytes, bytearray, memoryview)):
            files = [files]
        bufs = [np.frombuffer(bytes(f), np.uint8) for f in files]
        n = len(bufs)
        if n == 0:
            raise ValueError("no files")
        if progressive:   # the progressive-capable reader: its own marker reader gives the size
            w, h, o, _ = self.jpeg_probe(bufs[0])
            if not orientation and o >= 5:
                w, h = h, w
        else:
            w, h = self.jpeg_size(bufs[0], orientation)
        shape = (n, h, w, 3) if channels == 3 else (n, h, w)
        if d_out is None:
            d_out = torch.empty(shape, dtype=torch.uint8, device="cuda:%d" % self.device)
        elif d_out.dtype != torch.uint8 or not d_out.is_cuda or not d_out.is_contiguous() or d_out.numel() != n * h * w * channels:
            raise ValueError("d_out must be a contiguous uint8 CUDA tensor of %s elements" % " x ".join(("N", "H", "W", "3")[:len(shape)]))
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
        lens = (C.c_size_t * n)(*[b.size for b in bufs])
        self._ck(decode(self.h, ptrs, lens, n, _ptr(d_out), w, h))
        self.synchronize()
        return d_out

    def jpeg_decode_grey(self, files, orientation=False, progressive=False):
        """JPEG files of one size -> numpy uint8 (N, H, W) equal to cv2.imdecode(file, cv2.IMREAD_GRAYSCALE) of files without
        an Exif orientation, and of every file with orientation=True; one bytes object -> (H, W).  Decoded on the device;
        progressive=True reads progressive files too."""
        single = isinstance(files, (bytes, bytearray, memoryview))
        out = self.jpeg_decode_grey_batch_dev(files, orientation=orientation, progressive=progressive).cpu().numpy()
        return out[0] if single else out

    def jpeg_decode(self, files, orientation=False, progressive=False):
        """JPEG files of one size -> numpy uint8 (N, H, W, 3) equal to cv2.imdecode(file, cv2.IMREAD_COLOR) of files without
        an Exif orientation, and of every file with orientation=True; one bytes object -> (H, W, 3).  Decoded on the device;
        progressive=True reads progressive files too."""
        single = isinstance(files, (bytes, bytearray, memoryview))
        out = self.jpeg_decode_batch_dev(files, orientation=orientation, progressive=progressive).cpu().numpy()
        return out[0] if single else out

    def jpeg_decode_stats(self, n):
        """(N, 2) int32 of the last jpeg_decode_batch_dev call: subsequence decodes repeated by the in-CTA synchronisation,
        subsequences re-decoded by the cross-CTA fix-up."""
        out = np.empty((n, 2), np.int32)
        self._ck(self.lib.uwip_jpeg_decode_stats(self.h, int(n), _ptr(out)))
        return out

    def last_frame_flags(self, n):
        """Per-frame status bits of the last batched chain / bgdehaze / automatic-aclahe / exact JPEG decode (bgr8 or grey) call: 1 = the
        reference output is NaN (D9), 2 = the automatic CLAHE fit failed (BS = CL = -1, fixed parameters used), 4 = the JPEG
        file's entropy-coded data is bad (the frame is zeros)."""
        out = np.empty(n, np.int32)
        self._ck(self.lib.uwip_last_frame_flags(self.h, int(n), _ptr(out)))
        return out

    def histretch_dev(self, d_src, d_dst, n, width, height, channels="V", lo=2, hi=98, order="intended", hsv_round="cv2"):
        self._ck(self.lib.uwip_histretch_bgr8_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, channels.encode(), lo, hi,
                                                  ORDER[order], HSV_ROUND[hsv_round]))

    def aclahe_dev(self, d_src, d_dst, n, width, height, clip=2.0, tiles=(8, 8), hsv_round="cv2"):
        self._ck(self.lib.uwip_aclahe_bgr8_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, float(clip), tiles[0], tiles[1],
                                               HSV_ROUND[hsv_round]))

    def aclahe_params_dev(self, d_planes, n, width, height, loop="repaired", d_bs=None, d_cl=None):
        """ParametrosACLAHE on n device planes -> (BS, CL) in device int32[n] arrays (torch tensors unless given).  Stream
        ordered: synchronise (or read the tensors on the context's stream) before using them."""
        if d_bs is None or d_cl is None:
            import torch

            d_bs = torch.empty(n, dtype=torch.int32, device="cuda:%d" % self.device) if d_bs is None else d_bs
            d_cl = torch.empty(n, dtype=torch.int32, device="cuda:%d" % self.device) if d_cl is None else d_cl
        self._ck(self.lib.uwip_aclahe_params_u8_dev(self.h, _ptr(d_planes), n, width, height, ACLAHE_LOOP[loop], _ptr(d_bs), _ptr(d_cl)))
        return d_bs, d_cl

    def aclahe_auto_dev(self, d_src, d_dst, n, width, height, loop="repaired", hsv_round="cv2", clip=2.0, tiles=(8, 8), d_bs=None,
                        d_cl=None):
        """aclahe with each frame's own automatic (BS, CL); clip and tiles apply to frames whose fit failed."""
        self._ck(self.lib.uwip_aclahe_bgr8_auto_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, ACLAHE_LOOP[loop],
                                                    HSV_ROUND[hsv_round], float(clip), int(tiles[0]), int(tiles[1]),
                                                    _ptr(d_bs) if d_bs is not None else None,
                                                    _ptr(d_cl) if d_cl is not None else None))

    def aclahe_grey_auto_dev(self, d_src, d_dst, n, width, height, loop="repaired", clip=2.0, tiles=(8, 8), d_bs=None, d_cl=None):
        """main.py:18-20 on n device grey planes: each plane's automatic (BS, CL), then CLAHE of the plane with them; clip and
        tiles apply to planes whose fit failed (BS = CL = -1, bit 2 of last_frame_flags).  Stream ordered."""
        self._ck(self.lib.uwip_aclahe_u8_auto_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, ACLAHE_LOOP[loop], float(clip),
                                                  int(tiles[0]), int(tiles[1]), _ptr(d_bs) if d_bs is not None else None,
                                                  _ptr(d_cl) if d_cl is not None else None))

    def clahe_dev(self, d_src, d_dst, n, width, height, clip=40.0, tiles=(8, 8)):
        self._ck(self.lib.uwip_clahe_u8_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, float(clip), int(tiles[0]), int(tiles[1])))

    def bgdehaze_dev(self, d_src, d_dst, n, width, height, params=None):
        p = params or self.dehaze_params()
        self._ck(self.lib.uwip_bgdehaze_bgr8_dev(self.h, _ptr(d_src), _ptr(d_dst), n, width, height, C.byref(p)))

    # ---- videostrip calcBlur (videostrip.cpp:170-184) ------------------------------------------------
    def calc_blur(self, frame, return_all=False, aperture=3):
        """float32 stdev of the 8-bit aperture-3 Laplacian of the grey frame; return_all: (stdev, (mean, stdev) f64, laplacian u8)."""
        f = _frame(frame)
        sd = C.c_float()
        ms = (C.c_double * 2)()
        lap = np.empty(f.shape[:2], np.uint8) if return_all else None
        self._ck(self.lib.uwip_calc_blur_bgr8(self.h, _ptr(f), f.strides[0], f.shape[1], f.shape[0], int(aperture), C.byref(sd), ms,
                                              _ptr(lap) if return_all else None, lap.strides[0] if return_all else 0))
        return (np.float32(sd.value), (ms[0], ms[1]), lap) if return_all else np.float32(sd.value)

    def calc_blur_dev(self, d_src, n, width, height, d_mean_std, aperture=3):
        self._ck(self.lib.uwip_calc_blur_bgr8_dev(self.h, _ptr(d_src), n, width, height, int(aperture), _ptr(d_mean_std)))

    def synth_dev(self, d_dst, seed, first_frame, n, width, height):
        self._ck(self.lib.uwip_synth_bgr8_dev(self.h, _ptr(d_dst), seed & 0xFFFFFFFF, first_frame, n, width, height))

    def checksum_dev(self, d_src, n, width, height):
        out = np.empty(n, np.uint64)
        self._ck(self.lib.uwip_checksum_bgr8_dev(self.h, _ptr(d_src), n, width, height, _ptr(out)))
        return out

    # raw device memory for callers without torch
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.lib.uwip_device_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr):
        self._ck(self.lib.uwip_device_free(self.h, C.c_void_p(ptr)))

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.lib.uwip_host_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def host_free(self, ptr):
        self._ck(self.lib.uwip_host_free(self.h, C.c_void_p(ptr)))

    def copy_h2d(self, dptr, hptr, nbytes):
        self._ck(self.lib.uwip_copy_h2d(self.h, C.c_void_p(_ptr(dptr)), C.c_void_p(_ptr(hptr)), nbytes))

    def copy_d2h(self, hptr, dptr, nbytes):
        self._ck(self.lib.uwip_copy_d2h(self.h, C.c_void_p(_ptr(hptr)), C.c_void_p(_ptr(dptr)), nbytes))


def host_checksum(frames):
    """numpy twin of uwip_checksum_bgr8_dev."""
    a = np.ascontiguousarray(frames, dtype=np.uint8)
    if a.ndim == 3:
        a = a[None]
    n = a.shape[0]
    flat = a.reshape(n, -1).astype(np.uint64)
    i = np.arange(flat.shape[1], dtype=np.uint64)
    w = ((i * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)) | np.uint64(1)
    with np.errstate(over="ignore"):
        return ((flat + np.uint64(1)) * w[None, :]).sum(axis=1, dtype=np.uint64)


_default = {}


def default_context(device=0):
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]
