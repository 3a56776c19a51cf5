"""ctypes access to the oracle (TEST INFRASTRUCTURE ONLY - see oracle/restate.h).

``restate``  : oracle/librestate.so  - our C restatement, always buildable (gcc only).
``ref``      : oracle/_ref/libref.so - the real reference sources compiled verbatim against the fake UPMEM
               runtime; built in the dev container, travels to the GPU box prebuilt.  May be absent.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")
M = 100  # MAX_MCU_PER_DPU the reference is built with (Makefile:2)
CHUNK = 64 * M * 3


class RsHuff(C.Structure):
    _fields_ = [("offsets", C.c_uint8 * 17), ("symbols", C.c_uint8 * 162), ("set", C.c_uint8)]


class RsHeader(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("ncomp", C.c_uint32), ("hs", C.c_uint32), ("vs", C.c_uint32),
        ("mcu_w", C.c_uint32), ("mcu_h", C.c_uint32), ("mcu_w_real", C.c_uint32), ("mcu_h_real", C.c_uint32),
        ("restart_interval", C.c_uint32),
        ("qt_id", C.c_uint8 * 3), ("dc_id", C.c_uint8 * 3), ("ac_id", C.c_uint8 * 3), ("comp_h", C.c_uint8 * 3), ("comp_v", C.c_uint8 * 3),
        ("qt_zz", (C.c_uint16 * 64) * 4), ("qt_set", C.c_uint8 * 4),
        ("dc", RsHuff * 4), ("ac", RsHuff * 4),
        ("scan_off", C.c_size_t), ("scan_len", C.c_size_t), ("frame_type", C.c_int), ("valid", C.c_int),
    ]


class RefInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in (
        "width", "height", "ncomp", "h_samp", "v_samp", "mcu_w", "mcu_h", "mcu_w_real", "mcu_h_real",
        "restart_interval", "nchunks", "valid", "huffman_ok", "scan_bytes")]


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE, "all"], check=True, stdout=subprocess.DEVNULL)


_restate = None
_ref = None


def restate():
    global _restate
    if _restate is None:
        path = os.path.join(ORACLE, "librestate.so")
        if not os.path.exists(path):
            build_oracle()
        lib = C.CDLL(path)
        lib.rs_parse.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(RsHeader)]
        lib.rs_unstuff.restype = C.c_long
        lib.rs_unstuff.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        for f in ("rs_num_mcus", "rs_blocks_per_mcu"):
            getattr(lib, f).restype = C.c_uint32
            getattr(lib, f).argtypes = [C.POINTER(RsHeader)]
        lib.rs_num_chunks.restype = C.c_uint32
        lib.rs_num_chunks.argtypes = [C.POINTER(RsHeader), C.c_int]
        lib.rs_huffman_zz.argtypes = [C.POINTER(RsHeader), C.c_void_p, C.c_void_p, C.c_int]
        lib.rs_coef_to_ref_mcus.argtypes = [C.POINTER(RsHeader), C.c_void_p, C.c_void_p, C.c_int]
        lib.rs_metadata.argtypes = [C.POINTER(RsHeader), C.c_void_p, C.c_int]
        lib.rs_exec_mcus.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        lib.rs_bmp_size.restype = C.c_size_t
        lib.rs_bmp_size.argtypes = [C.c_uint32, C.c_uint32]
        lib.rs_mcus_to_bmp.restype = C.c_size_t
        lib.rs_mcus_to_bmp.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rs_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]
        lib.rs_idct8.argtypes = [C.c_void_p, C.c_void_p]
        _restate = lib
    return _restate


def ref_available():
    return os.path.exists(os.path.join(ORACLE, "_ref", "libref.so"))


REFERENCE_VECTORS = os.path.join(ROOT, "tests", "golden", "reference_vectors.json")


def reference_vectors():
    """What the reference computed on the seeded inputs of the exec and damaged-header tests (make_reference_vectors.py)."""
    import json
    with open(REFERENCE_VECTORS) as f:
        return json.load(f)


def sha256(*arrays):
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def ref():
    global _ref
    if _ref is None:
        lib = C.CDLL(os.path.join(ORACLE, "_ref", "libref.so"))
        lib.ref_probe.argtypes = [C.c_char_p, C.POINTER(RefInfo)]
        lib.ref_decode_file.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.POINTER(RefInfo)]
        lib.ref_exec_mcus.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        if hasattr(lib, "ref_write_bmp"):
            lib.ref_write_bmp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_char_p]
        _ref = lib
    return _ref


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------- restatement helpers

class Restated:
    """All stages of the restatement for one in-memory JPEG."""

    def __init__(self, data, restart_mode=0):
        lib = restate()
        self.data = np.frombuffer(data, dtype=np.uint8)
        self.h = RsHeader()
        self.rc = lib.rs_parse(_ptr(self.data), len(data), C.byref(self.h))
        self.valid = self.rc == 0 and self.h.frame_type == 0xC0
        if not self.valid:
            return
        h = self.h
        self.nmcu = lib.rs_num_mcus(C.byref(h))
        self.bpm = lib.rs_blocks_per_mcu(C.byref(h))
        self.nchunk = lib.rs_num_chunks(C.byref(h), M)
        self.coef_zz = np.zeros((self.nmcu * self.bpm, 64), dtype=np.int16)
        self.huff_rc = lib.rs_huffman_zz(C.byref(h), _ptr(self.data), _ptr(self.coef_zz), restart_mode)
        self.metadata = np.zeros((self.nchunk, 276), dtype=np.uint32)
        lib.rs_metadata(C.byref(h), _ptr(self.metadata), M)
        self.metadata[1:] = self.metadata[0]
        self.mcus_pre = np.zeros((self.nchunk, CHUNK), dtype=np.int16)
        lib.rs_coef_to_ref_mcus(C.byref(h), _ptr(self.coef_zz), _ptr(self.mcus_pre), M)
        self.mcus_post = self.mcus_pre.copy()
        lib.rs_exec_mcus(_ptr(self.metadata), _ptr(self.mcus_post), self.nchunk)
        self.bmp = np.zeros(lib.rs_bmp_size(h.width, h.height), dtype=np.uint8)
        lib.rs_mcus_to_bmp(_ptr(self.metadata), _ptr(self.mcus_post), _ptr(self.bmp))

    @property
    def rgb(self):
        """Top-down packed RGB8 [H, W, 3] recovered from the BMP bytes."""
        w, h = self.h.width, self.h.height
        stride = w * 3 + w % 4
        rows = self.bmp[26:].reshape(h, stride)[::-1, : w * 3].reshape(h, w, 3)
        return np.ascontiguousarray(rows[:, :, ::-1])


def restate_exec_mcus(metadata, mcus):
    out = np.ascontiguousarray(mcus).copy()
    md = np.ascontiguousarray(metadata, dtype=np.uint32)
    restate().rs_exec_mcus(_ptr(md), _ptr(out), md.shape[0])
    return out


# ---------------------------------------------------------------- real-reference helpers

class RefDecoded:
    """All stages of the REAL reference code for one JPEG file on disk."""

    def __init__(self, path, bmp_path=None):
        lib = ref()
        info = RefInfo()
        n = lib.ref_probe(path.encode(), C.byref(info))
        self.valid = n > 0
        if not self.valid:
            return
        self.nchunk = n
        self.metadata = np.zeros(276, dtype=np.uint32)
        self.mcus_pre = np.zeros((n, CHUNK), dtype=np.int16)
        self.mcus_post = np.zeros((n, CHUNK), dtype=np.int16)
        self.info = RefInfo()
        rc = lib.ref_decode_file(path.encode(), _ptr(self.metadata), _ptr(self.mcus_pre), _ptr(self.mcus_post),
                                 bmp_path.encode() if bmp_path else None, C.byref(self.info))
        assert rc == n


def ref_exec_mcus(metadata, mcus):
    out = np.ascontiguousarray(mcus).copy()
    md = np.ascontiguousarray(metadata, dtype=np.uint32)
    ref().ref_exec_mcus(_ptr(md), _ptr(out), md.shape[0])
    return out


def ref_write_bmp(metadata276, mcus, path):
    """The reference's real write_BMP on post-exec chunks [nchunk][64*M*3]."""
    md = np.ascontiguousarray(metadata276, dtype=np.uint32).reshape(-1)[:276]
    m = np.ascontiguousarray(mcus, dtype=np.int16)
    ref().ref_write_bmp(_ptr(md), _ptr(m), int(m.size // CHUNK), path.encode())


def unstuffed_scan(data):
    """Header::huffman_data as read_JPEG leaves it (un-stuffed, RSTn removed), from the restatement's scan filter."""
    h = RsHeader()
    buf = np.frombuffer(data, dtype=np.uint8)
    assert restate().rs_parse(_ptr(buf), len(data), C.byref(h)) == 0
    scan = np.ascontiguousarray(buf[h.scan_off:h.scan_off + h.scan_len])
    out = np.zeros(h.scan_len + 1, dtype=np.uint8)
    n = restate().rs_unstuff(_ptr(scan), h.scan_len, _ptr(out), None, 0, None)
    assert n >= 0
    return bytes(out[:n]), bytes(scan)
