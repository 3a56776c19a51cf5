"""ctypes binding of libb200jpeg.so (include/b200jpeg.h).  No torch types cross this boundary.

The library is built in-tree by ``pim_jpeg_decoder_b200/csrc/Makefile`` (see ``__graft_entry__.build``).  There
is no CPU decode path: if the shared object is missing, loading raises; if no CUDA device is present,
``bj_create`` returns BJ_ERR_CUDA and ``Context()`` raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200JPEG_LIB") or os.path.join(HERE, "libb200jpeg.so")   # (the override is for A/B measurements)

BJ_OK = 0
BJ_ERR_ARG = -1
BJ_ERR_CUDA = -2
BJ_ERR_NOMEM = -3
BJ_ERR_INVALID_JPEG = -4
BJ_ERR_UNSUPPORTED = -5
BJ_ERR_CORRUPT_SCAN = -6

BJ_OUT_RGB8 = 0
BJ_OUT_BMP = 1
BJ_OUT_REF_MCUS = 2
BJ_SCAN_RAW = 0
BJ_SCAN_UNSTUFFED = 1


class ImageDesc(C.Structure):
    """bj_image_desc"""
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32),
        ("mcu_w", C.c_uint32), ("mcu_h", C.c_uint32),
        ("mcu_w_real", C.c_uint32), ("mcu_h_real", C.c_uint32),
        ("restart_interval", C.c_uint32),
        ("ncomp", C.c_uint8), ("hs", C.c_uint8), ("vs", C.c_uint8), ("frame_type", C.c_uint8),
        ("comp_h", C.c_uint8 * 3), ("comp_v", C.c_uint8 * 3),
        ("qt_id", C.c_uint8 * 3), ("dc_id", C.c_uint8 * 3), ("ac_id", C.c_uint8 * 3),
        ("qt_set", C.c_uint8 * 4), ("dc_set", C.c_uint8 * 4), ("ac_set", C.c_uint8 * 4),
        ("scan_ncomp", C.c_uint8),
        ("qt_zz", (C.c_uint16 * 64) * 4),
        ("dc_offsets", (C.c_uint8 * 17) * 4), ("dc_symbols", (C.c_uint8 * 162) * 4),
        ("ac_offsets", (C.c_uint8 * 17) * 4), ("ac_symbols", (C.c_uint8 * 162) * 4),
        ("scan_off", C.c_uint64), ("scan_len", C.c_uint64),
    ]


class Roi(C.Structure):
    """bj_roi: pixels [y, y+h) x [x, x+w) of the image, top-left origin; all zero = the whole image"""
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32), ("w", C.c_uint32), ("h", C.c_uint32)]


class Size(C.Structure):
    """bj_size: a target size w x h in pixels; {0, 0} = no resize"""
    _fields_ = [("w", C.c_uint32), ("h", C.c_uint32)]


class BatchInfo(C.Structure):
    """bj_batch_info"""
    _fields_ = [
        ("pixels", C.c_uint64), ("scan_bytes", C.c_uint64), ("data_units", C.c_uint64), ("out_bytes", C.c_uint64),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("subsequences", C.c_uint32), ("sync_rounds", C.c_uint32), ("launches", C.c_uint32),
        ("ms_entropy", C.c_float), ("ms_idct", C.c_float),
        ("ms_unstuff", C.c_float), ("ms_sync", C.c_float), ("ms_write", C.c_float),
        ("clean_bytes", C.c_uint64),
    ]


SYMBOLS = {
    # name: (restype, argtypes)
    "bj_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "bj_create_multi": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int]),
    "bj_device_count": (C.c_int, [C.c_void_p]),
    "bj_destroy": (None, [C.c_void_p]),
    "bj_status_string": (C.c_char_p, [C.c_int]),
    "bj_last_error": (C.c_char_p, [C.c_void_p]),
    "bj_device_sm_count": (C.c_int, [C.c_void_p]),
    "bj_host_alloc": (C.c_void_p, [C.c_size_t]),
    "bj_host_free": (None, [C.c_void_p]),
    "bj_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "bj_host_unregister": (C.c_int, [C.c_void_p]),
    "bj_exec_mcus": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "bj_exec_mcus_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bj_parse_header": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(ImageDesc)]),
    "bj_peek_header": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(ImageDesc)]),
    "bj_output_size": (C.c_size_t, [C.POINTER(ImageDesc), C.c_int]),
    "bj_roi_output_size": (C.c_size_t, [C.POINTER(ImageDesc), C.POINTER(Roi), C.c_int]),
    "bj_scaled_output_size": (C.c_size_t, [C.POINTER(ImageDesc), C.POINTER(Roi), C.c_int, C.c_int]),
    "bj_resized_output_size": (C.c_size_t, [C.POINTER(ImageDesc), C.POINTER(Roi), C.c_int, C.POINTER(Size), C.c_int]),
    "bj_ref_mcus_size": (C.c_size_t, [C.POINTER(ImageDesc), C.c_int, C.POINTER(C.c_int)]),
    "bj_decode_batch_desc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bj_decode_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bj_decode_batch_roi": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bj_decode_batch_scaled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bj_decode_batch_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p]),
    "bj_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "bj_submit_roi": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "bj_submit_scaled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.POINTER(C.c_void_p)]),
    "bj_submit_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.POINTER(C.c_void_p)]),
    "bj_wait": (C.c_int, [C.c_void_p]),
    "bj_batch_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "bj_batch_create_roi": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "bj_batch_create_scaled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "bj_batch_create_resized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                          C.POINTER(C.c_void_p)]),
    "bj_batch_upload": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bj_batch_decode": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bj_batch_sync": (C.c_int, [C.c_void_p]),
    "bj_batch_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bj_batch_status": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bj_batch_destroy": (None, [C.c_void_p]),
    "bj_batch_get_info": (C.c_int, [C.c_void_p, C.POINTER(BatchInfo)]),
    "bj_batch_output_offset": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "bj_batch_device_output": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "bj_batch_device_coefficients": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_void_p)]),
    "bj_stage_idct_color": (C.c_int, [C.c_void_p, C.POINTER(ImageDesc), C.c_void_p, C.c_int, C.c_void_p]),
    "bj_stage_entropy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "bj_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_long]),
    "bj_get_stat": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double)]),
    "bj_build_info": (C.c_char_p, []),
}

_lib = None


def lib():
    """The loaded library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libb200jpeg.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C pim_jpeg_decoder_b200/csrc`); this package has no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(l, name)  # AttributeError if the header and the library disagree
            f.restype = res
            f.argtypes = args
        _lib = l
    return _lib


class BjError(RuntimeError):
    def __init__(self, status, what="", detail=""):
        self.status = status
        msg = lib().bj_status_string(status).decode()
        super().__init__(f"{what}: {msg} ({status}){' - ' + detail if detail else ''}")


def check(status, what="b200jpeg", ctx=None):
    if status != BJ_OK:
        detail = lib().bj_last_error(ctx).decode() if ctx and status == BJ_ERR_CUDA else ""
        raise BjError(status, what, detail)
