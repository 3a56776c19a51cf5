"""CPU tests of the drop-in boundary itself (no GPU needed): the C-ABI library loads, exports every entry point
``include/b200jpeg.h`` declares, refuses to compute without a CUDA device (there is no CPU fallback), and its one
host-only entry, ``bj_parse_header`` (the in-memory restatement of the reference's ``read_JPEG``,
src/jpeg_scanner.cpp:345-436), accepts and rejects exactly the files the reference does."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _declared():
    text = open(os.path.join(ROOT, "include", "b200jpeg.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bj_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import pim_jpeg_decoder_b200 as bj
    from pim_jpeg_decoder_b200 import _lib
    names = _declared()
    assert len(names) >= 30
    raw = C.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} is declared in include/b200jpeg.h but not exported by libb200jpeg.so"
    assert sorted(_lib.SYMBOLS) == names, "the ctypes prototypes and the header disagree"
    assert b"sm_100a" in bj.lib().bj_build_info()


_NO_DEVICE_CHECKS = """
import ctypes as C
import pytest
import pim_jpeg_decoder_b200 as bj
ctx = C.c_void_p()
assert bj.lib().bj_create(C.byref(ctx), 0) == bj.BJ_ERR_CUDA and not ctx.value
assert bj.lib().bj_create_multi(C.byref(ctx), None, 0) == bj.BJ_ERR_CUDA and not ctx.value
with pytest.raises(bj.BjError):
    bj.Decoder(0)
assert bj.lib().bj_decode_batch(None, None, None, 0, 0, None, None) == -1      # BJ_ERR_ARG, not a crash
print("no device: refused")
"""


def test_no_cpu_fallback_without_a_device():
    """Without a CUDA device the context cannot be created - every compute entry needs one - and the package raises.
    Checked in a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so on a GPU machine as well."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECKS], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "no device: refused", r.stdout[-2000:] + r.stderr[-2000:]


def _desc_matches(d, h):
    return (d.width == h.width and d.height == h.height and d.ncomp == h.ncomp and d.hs == h.hs and d.vs == h.vs and
            d.mcu_w_real == h.mcu_w_real and d.mcu_h_real == h.mcu_h_real and d.restart_interval == h.restart_interval and
            d.scan_off == h.scan_off and d.scan_len == h.scan_len)


def _mutations(rng, base, scan_off, n):
    """Damaged variants of a valid file, most of the damage inside the headers."""
    markers = [0xC0, 0xC2, 0xC4, 0xDB, 0xDA, 0xDD, 0xE0, 0xFE, 0xD8, 0xD9, 0x01, 0xFF, 0x00, 0xC1, 0xD0]
    seg = [i for i in range(2, scan_off - 1) if base[i] == 0xFF and base[i + 1] not in (0x00, 0xFF)]
    for k in range(n):
        b = bytearray(base)
        kind = k % 8
        if kind == 0:                                   # flip a few header bytes
            for _ in range(int(rng.integers(1, 4))):
                b[int(rng.integers(2, scan_off))] = int(rng.integers(0, 256))
        elif kind == 1:                                 # truncate
            b = b[: int(rng.integers(1, len(b)))]
        elif kind == 2 and seg:                         # change a segment's length field
            i = seg[int(rng.integers(0, len(seg)))]
            b[i + 3] = (b[i + 3] + int(rng.integers(-3, 4))) & 0xFF
        elif kind == 3 and seg:                         # replace a marker code
            i = seg[int(rng.integers(0, len(seg)))]
            b[i + 1] = markers[int(rng.integers(0, len(markers)))]
        elif kind == 4:                                 # damage the scan: stray markers / FF runs
            i = int(rng.integers(scan_off, len(b) - 2))
            b[i:i + 2] = bytes([0xFF, markers[int(rng.integers(0, len(markers)))]])
        elif kind == 5 and seg:                         # duplicate a segment
            i = seg[int(rng.integers(0, len(seg)))]
            ln = (b[i + 2] << 8) | b[i + 3]
            b = b[:i] + b[i:i + 2 + ln] + b[i:]
        elif kind == 6:                                 # sampling / component fields of the frame header
            i = bytes(b).find(b"\xFF\xC0")
            if i > 0:
                b[i + int(rng.integers(4, 19))] = int(rng.integers(0, 256))
        else:                                           # cut off the end marker / append garbage
            b = b[:-2] + bytes(int(x) for x in rng.integers(0, 256, int(rng.integers(0, 6))))
        yield bytes(b)


def damaged_files():
    """The 640 seeded damaged variants the header test runs on (baseline files of every sampling)."""
    rng = np.random.default_rng(77)
    bases = [js.synth_jpeg(48, 40, seed=1, subsampling=2), js.synth_jpeg(33, 17, seed=2, subsampling=0, restart_blocks=2),
             js.synth_jpeg(40, 24, seed=3, gray=True), js.synth_jpeg(64, 32, seed=4, subsampling=1, optimize=True)]
    for base in bases:
        yield from _mutations(rng, base, ol.Restated(base, 0).h.scan_off, 160)


@pytest.mark.timeout(600)
def test_parse_header_validity_matches_the_reference_on_damaged_files(tmp_path):
    """bj_parse_header says BJ_ERR_INVALID_JPEG exactly where the reference's read_JPEG sets valid = false - on more
    than 500 damaged variants of baseline files of every sampling (checked against the restatement, against the
    reference's verdicts and sizes stored in tests/golden/reference_vectors.json, and against the live reference
    itself where oracle/_ref/libref.so is present)."""
    import pim_jpeg_decoder_b200 as bj
    files = list(damaged_files())
    want = ol.reference_vectors()["parse_header_damaged"]
    assert ol.sha256(*[np.frombuffer(f, dtype=np.uint8) for f in files]) == want["inputs_sha256"], \
        "the seeded inputs are not the ones the reference was run on"
    use_ref = ol.ref_available()
    n_invalid = 0
    path = str(tmp_path / "m.jpg")
    for n, (data, ref_result) in enumerate(zip(files, want["results"])):
        st, d = bj.parse_header(data)
        r = ol.Restated(data, 0)
        ours_valid = st in (bj.BJ_OK, bj.BJ_ERR_UNSUPPORTED)
        assert ours_valid == (r.rc == 0), (n, st, r.rc)
        ours = (d.width, d.height, d.ncomp, d.hs, d.vs, d.restart_interval)
        if st == bj.BJ_OK:
            assert _desc_matches(d, r.h), n
        assert ours_valid == bool(ref_result[0]), (n, st)       # [valid, width, height, ncomp, hs, vs, restart interval]
        if st == bj.BJ_OK:
            assert ours == tuple(ref_result[1:]), n
        if use_ref:
            with open(path, "wb") as f:
                f.write(data)
            info = ol.RefInfo()
            ref_valid = ol.ref().ref_probe(path.encode(), C.byref(info)) > 0
            assert ours_valid == ref_valid, (n, st)
            if st == bj.BJ_OK:
                assert ours == (info.width, info.height, info.ncomp, info.h_samp, info.v_samp, info.restart_interval)
        n_invalid += not ours_valid
    assert len(files) == len(want["results"]) >= 600 and 100 < n_invalid < len(files) - 100, (len(files), n_invalid)


def test_descriptor_layout_matches_the_header():
    """sizeof(bj_image_desc) as the C compiler sees it == the ctypes mirror (a silent mismatch would corrupt memory)."""
    import subprocess
    import sys
    import tempfile
    from pim_jpeg_decoder_b200 import _lib
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "b200jpeg.h"\nint main(void){printf("%zu %zu %zu %zu\\n", sizeof(bj_image_desc), offsetof(bj_image_desc, qt_zz), offsetof(bj_image_desc, scan_off), sizeof(bj_batch_info));return 0;}\n'
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "t")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, c], check=True)
        a, b, c2, d = (int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert a == C.sizeof(_lib.ImageDesc) and b == _lib.ImageDesc.qt_zz.offset and c2 == _lib.ImageDesc.scan_off.offset
    assert d == C.sizeof(_lib.BatchInfo)
    assert sys.byteorder == "little"
