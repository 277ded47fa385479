"""ctypes binding of libuwip.so (include/uwip.h).  There is no fallback: if the library is missing
or no sm_100 device is usable, importing works but every operation raises UwipError."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libuwip.so")

UWIP_OK = 0


class UwipError(RuntimeError):
    def __init__(self, status, text):
        super().__init__("uwip status %d: %s" % (status, text))
        self.status = status


class DehazeParams(C.Structure):
    _fields_ = [("window", C.c_int), ("radius", C.c_int), ("eps", C.c_double), ("tmin", C.c_double)]


class ChainParams(C.Structure):
    _fields_ = [
        ("channels", C.c_char * 16),
        ("lo", C.c_int), ("hi", C.c_int), ("order", C.c_int), ("hsv_round", C.c_int),
        ("clip", C.c_double), ("tiles_x", C.c_int), ("tiles_y", C.c_int),
        ("dehaze", DehazeParams),
    ]


_P = C.c_void_p
_u8p = C.c_void_p
_sz = C.c_size_t
_i = C.c_int
_d = C.c_double

# name -> (restype, argtypes); mirrors include/uwip.h one to one
SIGNATURES = {
    "uwip_version": (_i, []),
    "uwip_create": (_i, [_i, C.POINTER(_P)]),
    "uwip_destroy": (None, [_P]),
    "uwip_last_error": (C.c_char_p, [_P]),
    "uwip_set_stream": (_i, [_P, _P]),
    "uwip_synchronize": (_i, [_P]),
    "uwip_launch_count": (C.c_int64, [_P]),
    "uwip_profile": (_i, [_P, _i]),
    "uwip_profile_read": (_i, [_P, C.c_char_p, C.POINTER(_d), C.POINTER(C.c_int64)]),
    "uwip_device_alloc": (_i, [_P, _sz, C.POINTER(_P)]),
    "uwip_device_free": (_i, [_P, _P]),
    "uwip_host_alloc": (_i, [_P, _sz, C.POINTER(_P)]),
    "uwip_host_free": (_i, [_P, _P]),
    "uwip_copy_h2d": (_i, [_P, _P, _P, _sz]),
    "uwip_copy_d2h": (_i, [_P, _P, _P, _sz]),
    "uwip_num_channel": (_i, [C.c_char]),
    "uwip_num_space": (_i, [C.c_char]),
    "uwip_histogram_u8": (_i, [_P, _u8p, _i, _i, _sz, _P]),
    "uwip_histogram_u8_dev": (_i, [_P, _u8p, _i, _i, _P]),
    "uwip_channel_stretch_u8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "uwip_channel_stretch_u8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, _i]),
    "uwip_channel_stretch_u8_dev_pitched": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, _i, _i]),
    "uwip_histretch_bgr8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, C.c_char_p, _i, _i, _i, _i]),
    "uwip_histretch_bgr8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, C.c_char_p, _i, _i, _i, _i]),
    "uwip_clahe_u8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, _d, _i, _i]),
    "uwip_clahe_u8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, _d, _i, _i]),
    "uwip_entropy_u8": (_i, [_P, _u8p, _i, _i, _sz, _i, C.POINTER(C.c_float)]),
    "uwip_gaussian_blur3_u8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i]),
    "uwip_clahe_entropy_sweep_u8": (_i, [_P, _u8p, _i, _i, _sz, _i, C.POINTER(_d), _i, _i, C.POINTER(C.c_float)]),
    "uwip_clahe_entropy_sweep_u8_dev": (_i, [_P, _u8p, _i, _i, _i, C.POINTER(_i), _i, C.POINTER(_d), _i, _i, C.POINTER(C.c_float)]),
    "uwip_aclahe_bgr8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, _d, _i, _i, _i]),
    "uwip_aclahe_bgr8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, _d, _i, _i, _i]),
    "uwip_aclahe_params_u8_dev": (_i, [_P, _u8p, _i, _i, _i, _i, _P, _P]),
    "uwip_aclahe_bgr8_auto_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, _i, _i, _d, _i, _i, _P, _P]),
    "uwip_aclahe_u8_auto_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, _i, _d, _i, _i, _P, _P]),
    "uwip_dehaze_defaults": (None, [C.POINTER(DehazeParams)]),
    "uwip_chain_defaults": (None, [C.POINTER(ChainParams)]),
    "uwip_boxfilter_f64": (_i, [_P, _P, _i, _i, _i, _P]),
    "uwip_guided_filter_u8": (_i, [_P, _u8p, _sz, _i, _i, _i, _P, _i, _d, _P]),
    "uwip_background_light_bgr8": (_i, [_P, _u8p, _sz, _i, _i, _i, C.POINTER(_d), C.POINTER(C.c_int64)]),
    "uwip_transmission_bgr8": (_i, [_P, _u8p, _sz, _i, _i, _i, _P, _P]),
    "uwip_refined_transmission_bgr8": (_i, [_P, _u8p, _sz, _i, _i, C.POINTER(DehazeParams), _P, _P]),
    "uwip_rc_correction_bgr8": (_i, [_P, _u8p, _sz, _i, _i, C.POINTER(DehazeParams), _P]),
    "uwip_exposure_stages_bgr8": (_i, [_P, _u8p, _sz, _i, _i, C.POINTER(DehazeParams), _P, _P, _P, _P, _P, _P]),
    "uwip_bgdehaze_bgr8": (_i, [_P, _u8p, _sz, _u8p, _sz, _i, _i, C.POINTER(DehazeParams), _P]),
    "uwip_bgdehaze_bgr8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, C.POINTER(DehazeParams)]),
    "uwip_chain_bgr8_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, C.POINTER(ChainParams)]),
    "uwip_chain_bgr8_auto_dev": (_i, [_P, _u8p, _u8p, _i, _i, _i, C.POINTER(ChainParams), _i, _P, _P]),
    "uwip_chain_bgr8": (_i, [_P, _u8p, _u8p, _i, _i, _i, C.POINTER(ChainParams)]),
    "uwip_last_frame_flags": (_i, [_P, _i, _P]),
    "uwip_jpeg_info": (_i, [_P, _u8p, _sz, C.POINTER(_i), C.POINTER(_i)]),
    "uwip_jpeg_decode_bgr8_dev": (_i, [_P, _u8p, _sz, _u8p, _i, _i]),
    "uwip_jpeg_encode_bgr8_dev": (_i, [_P, _u8p, _i, _i, _i, _u8p, _sz, C.POINTER(_sz)]),
    "uwip_chain_jpeg": (_i, [_P, _u8p, _sz, C.POINTER(ChainParams), _i, _u8p, _sz, C.POINTER(_sz)]),
    "uwip_jpeg_encode_bound": (_sz, [_i, _i]),
    "uwip_jpeg_encode_bgr8_batch_dev": (_i, [_P, _u8p, _i, _i, _i, _i, _u8p, _sz, _P]),
    "uwip_jpeg_encode_u8_bound": (_sz, [_i, _i]),
    "uwip_jpeg_encode_u8_batch_dev": (_i, [_P, _u8p, _i, _i, _i, _i, _u8p, _sz, _P]),
    "uwip_jpeg_decode_bgr8_batch": (_i, [_P, _P, _P, _i, _u8p, _i, _i]),
    "uwip_jpeg_decode_u8_batch": (_i, [_P, _P, _P, _i, _u8p, _i, _i]),
    "uwip_jpeg_decode_bgr8_batch_oriented": (_i, [_P, _P, _P, _i, _u8p, _i, _i]),
    "uwip_jpeg_decode_u8_batch_oriented": (_i, [_P, _P, _P, _i, _u8p, _i, _i]),
    "uwip_jpeg_orientation": (_i, [_u8p, _sz, C.POINTER(_i)]),
    "uwip_jpeg_decode_batch_ex": (_i, [_P, _P, _P, _i, _u8p, _i, _i, _i]),
    "uwip_jpeg_probe": (_i, [_u8p, _sz, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "uwip_jpeg_decode_stats": (_i, [_P, _i, _P]),
    "uwip_calc_blur_bgr8": (_i, [_P, _u8p, _sz, _i, _i, _i, C.POINTER(C.c_float), C.POINTER(_d), _u8p, _sz]),
    "uwip_calc_blur_bgr8_dev": (_i, [_P, _u8p, _i, _i, _i, _i, _P]),
    "uwip_synth_bgr8_dev": (_i, [_P, _u8p, C.c_uint32, _i, _i, _i, _i]),
    "uwip_checksum_bgr8_dev": (_i, [_P, _u8p, _i, _i, _i, _P]),
}

_lib = None


def load():
    """Load libuwip.so (raises with build instructions if it is not there)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UwipError(-2, "libuwip.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
