"""CPU tests of progressive (SOF2) decode: the product's multi-scan walk (parse.h: parse_progressive) and work-item
decode (prog_core.h), driven by a sequential host emulation of the kernels (tests/emu/prog_emu.cpp), against the
oracle's coefficients of each file's baseline twin (same frame, same quantised coefficients, one baseline scan).

The test encoder (prog_synth.py) is pinned first: Pillow must decode its files to exactly the pixels of their twins.
"""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol
import prog_synth as ps

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, "emu", "libprogemu.so")
BJ_OK, BJ_ERR_INVALID_JPEG, BJ_ERR_UNSUPPORTED = 0, -4, -5

Y420 = [(2, 2, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)]
Y422 = [(2, 1, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)]
Y440 = [(1, 2, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)]
Y444 = [(1, 1, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)]
GRAY = [(1, 1, 0, 0, 0)]
SAMPLINGS = {"420": Y420, "422": Y422, "440": Y440, "444": Y444, "gray": GRAY}


def emu():
    src = os.path.join(HERE, "emu", "prog_emu.cpp")
    csrc = os.path.join(ol.ROOT, "pim_jpeg_decoder_b200", "csrc")
    deps = [src, os.path.join(csrc, "prog_core.h"), os.path.join(csrc, "parse.h")]
    if not os.path.exists(EMU) or os.path.getmtime(EMU) < max(os.path.getmtime(p) for p in deps):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", EMU, src], check=True)
    lib = C.CDLL(EMU)
    lib.emu_prog_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    return lib


def emu_decode(data, units):
    buf = np.frombuffer(data, dtype=np.uint8)
    coef = np.full((units, 64), 0x5A5A, dtype=np.int16)
    info = np.zeros(4, dtype=np.uint32)
    rc = emu().emu_prog_decode(ol._ptr(buf), len(data), ol._ptr(coef), units, ol._ptr(info))
    return rc, coef, info


def emu_status(data):
    return emu_decode(data, 1 << 16)[0]


# ---------------------------------------------------------------------------------------------- scan scripts
def _ac_full(n):
    return [((j,), 1, 63, 0, 0) for j in range(n)]


def scripts(n):
    dc_all = tuple(range(n))
    s = {
        "simple": ps.SCRIPT_YCC if n == 3 else ps.SCRIPT_GRAY,
        "dc_per_component": [((j,), 0, 0, 0, 0) for j in range(n)] + _ac_full(n),
        "dc_bit_by_bit": [(dc_all, 0, 0, 0, 7)] + [(dc_all, 0, 0, a + 1, a) for a in range(6, -1, -1)] + _ac_full(n),
        "spectral_only": [(dc_all, 0, 0, 0, 0)] + [((j,), lo, hi, 0, 0) for j in range(n) for lo, hi in ((1, 2), (3, 20), (21, 63))],
        "ac_bit_by_bit": [(dc_all, 0, 0, 0, 0)] + [((j,), 1, 63, 0, 4) for j in range(n)]
                         + [((j,), 1, 63, a + 1, a) for a in range(3, -1, -1) for j in range(n)],
    }
    if n == 1:
        s["single_coefficient_bands"] = [((0,), 0, 0, 0, 0)] + [((0,), k, k, 0, 0) for k in range(1, 64)]
    return s


def quirk_coefs(comps, w, h):
    """the zig-zag 48/52 aliasing and ZRL landings of the golden set (tests/golden/make_golden.py)"""
    co = js.random_coefs(comps, w, h, 11, density=0.0)
    pats = [{48: 5}, {52: -7}, {48: 5, 52: -7}, {36: 3, 52: 9}, {20: 2, 48: -4, 63: 1}, {32: 1, 48: 6}, {1: 300, 2: -300, 52: 1023, 48: -1023}]
    k = 0
    for a in co:
        for by in range(a.shape[0]):
            for bx in range(a.shape[1]):
                for z, v in pats[k % len(pats)].items():
                    a[by, bx, z] = v
                k += 1
    return co


def coef_sets(comps):
    return {
        "random": (45, 30, js.random_coefs(comps, 45, 30, 21)),
        "zz48_52": (40, 24, quirk_coefs(comps, 40, 24)),
        "extreme": (32, 32, js.random_coefs(comps, 32, 32, 13, density=0.5, amp=1023, dc_amp=1000)),
        "eobrun": (256, 200, js.random_coefs(comps, 256, 200, 5, density=0.002)),   # runs of hundreds of empty bands
    }


def encoder_cases():
    out = []
    for sname, comps in SAMPLINGS.items():
        for cname in ("random", "zz48_52", "extreme", "eobrun"):
            for scr in scripts(len(comps)):
                if cname == "eobrun" and scr not in ("simple", "ac_bit_by_bit"):
                    continue
                for ri in (0, 3) if cname == "random" else (0,):
                    out.append((sname, cname, scr, ri))
    return out


_CACHE = {}


def encoder_twins(sname, cname, scr, ri):
    key = (sname, cname, scr, ri)
    if key not in _CACHE:
        comps = SAMPLINGS[sname]
        w, h, co = coef_sets(comps)[cname]
        prog, twin = ps.prog_twins(w, h, comps, co, scripts(len(comps))[scr], ri)
        _CACHE[key] = (prog, twin, ps.within_grids(w, h, comps))
    return _CACHE[key]


def _pil(data):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


# ---------------------------------------------------------------------------------------------- the encoder itself
@pytest.mark.parametrize("sname,cname,scr,ri", [c for c in encoder_cases() if c[1] != "eobrun" or c[0] in ("420", "gray")])
def test_encoder_is_a_twin_for_pillow(sname, cname, scr, ri):
    prog, twin, _ = encoder_twins(sname, cname, scr, ri)
    if sname == "440":
        pytest.skip("Pillow decodes h1v2 files with its own upsampling")  # (checked against the oracle below)
    assert np.array_equal(_pil(prog), _pil(twin))


# ---------------------------------------------------------------------------------------------- emulated decode
@pytest.mark.parametrize("sname,cname,scr,ri", encoder_cases())
def test_emulated_decode_of_encoder_files(sname, cname, scr, ri):
    prog, twin, inside = encoder_twins(sname, cname, scr, ri)
    r = ol.Restated(twin, 0)
    assert r.valid and r.huff_rc == 0
    rc, coef, info = emu_decode(prog, r.coef_zz.shape[0])
    assert rc == BJ_OK and info[3] == 0
    assert np.array_equal(coef[inside], r.coef_zz[inside])


def pil_twins_or_skip(arr, sub, ri, gray):
    try:
        return ps.pil_twins(arr, 90, sub, ri, gray=gray)
    except OSError:                                     # Pillow 12 fails to write some large progressive files with
        pytest.skip("Pillow cannot write this progressive file")   # a restart marker after every MCU row


PIL_CASES = [(s, w, h, ri) for s in ("420", "422", "444", "gray") for (w, h) in ((1, 1), (17, 17), (45, 30), (500, 375)) for ri in (0, 1, 5, 64)]


@pytest.mark.parametrize("samp,w,h,ri", PIL_CASES)
def test_emulated_decode_of_pillow_files(samp, w, h, ri):
    arr = js.synth_rgb(w, h, w * 7 + h)
    sub = {"420": 2, "422": 1, "444": 0, "gray": 0}[samp]
    prog, twin = pil_twins_or_skip(arr, sub, ri, samp == "gray")
    r = ol.Restated(twin, 0)
    assert r.valid and r.huff_rc == 0
    comps = GRAY if samp == "gray" else {"420": Y420, "422": Y422, "444": Y444}[samp]
    rc, coef, info = emu_decode(prog, r.coef_zz.shape[0])
    assert rc == BJ_OK and info[3] == 0
    assert info[1] == 3                                 # libjpeg's script: three levels
    inside = ps.within_grids(w, h, comps)
    assert np.array_equal(coef[inside], r.coef_zz[inside])


# ---------------------------------------------------------------------------------------------- the walk's refusals
def _base():
    return encoder_twins("420", "random", "simple", 0)[0]


def _sos_positions(data):
    out, i = [], 2
    while i < len(data) - 1:
        if data[i] == 0xFF and data[i + 1] == 0xDA:
            out.append(i)
        i += 1
    return out


def _patch_sos(data, k, ss=None, se=None, ahal=None):
    p = _sos_positions(data)[k]
    ns = data[p + 4]
    b = bytearray(data)
    o = p + 5 + 2 * ns
    if ss is not None:
        b[o] = ss
    if se is not None:
        b[o + 1] = se
    if ahal is not None:
        b[o + 2] = ahal
    return bytes(b)


def test_walk_accepts_the_base_file():
    assert emu_status(_base()) == BJ_OK


@pytest.mark.parametrize("what", ["no_eoi", "bad_marker", "ss_gt_se", "se_gt_63", "dc_band", "ac_two_components",
                                  "ah_al", "ac_before_dc", "refine_without_first", "undefined_table", "first_pass_twice"])
def test_walk_refuses_structural_errors(what):
    d = _base()
    if what == "no_eoi":
        d = d[:-2]
    elif what == "bad_marker":
        p = _sos_positions(d)[1]
        d = d[:p] + b"\xFF\xC0\x00\x02" + d[p:]
    elif what == "ss_gt_se":
        d = _patch_sos(d, 1, ss=6, se=5)
    elif what == "se_gt_63":
        d = _patch_sos(d, 1, se=64)
    elif what == "dc_band":
        d = _patch_sos(d, 0, se=1)
    elif what == "ac_two_components":
        d = _patch_sos(d, 0, ss=1, se=5)
    elif what == "ah_al":
        d = _patch_sos(d, 5, ahal=0x20)
    elif what == "ac_before_dc":
        comps = SAMPLINGS["420"]
        w, h, co = coef_sets(comps)["random"]
        d = ps.encode_progressive(w, h, comps, co, [((0,), 1, 63, 0, 0), ((0, 1, 2), 0, 0, 0, 0)])
    elif what == "refine_without_first":
        d = _patch_sos(d, 5, ahal=0x32)                 # Ah 3 where the band's last Al is 2
    elif what == "undefined_table":
        p = _sos_positions(d)[0]
        b = bytearray(d)
        b[p + 6] = 0x30                                 # DC table 3, never defined
        d = bytes(b)
    elif what == "first_pass_twice":
        comps = SAMPLINGS["420"]
        w, h, co = coef_sets(comps)["random"]
        d = ps.encode_progressive(w, h, comps, co, [((0, 1, 2), 0, 0, 0, 0), ((0,), 1, 63, 0, 0), ((0,), 5, 10, 0, 0)])
    assert emu_status(d) == BJ_ERR_INVALID_JPEG


def test_walk_refuses_more_than_64_scans():
    comps = GRAY
    w, h, co = coef_sets(comps)["random"]
    ok = scripts(1)["single_coefficient_bands"]            # 64 scans
    assert emu_status(ps.encode_progressive(w, h, comps, co, ok)) == BJ_OK
    many = [((0,), 0, 0, 0, 1)] + [((0,), k, k, 0, 0) for k in range(1, 64)] + [((0,), 0, 0, 1, 0)]
    assert emu_status(ps.encode_progressive(w, h, comps, co, many)) == BJ_ERR_UNSUPPORTED


def test_walk_refuses_a_redefined_quantisation_table():
    d = _base()
    p = _sos_positions(d)[3]
    dqt = b"\xFF\xDB\x00\x43\x00" + bytes(range(1, 65))
    assert emu_status(d[:p] + dqt + d[p:]) == BJ_ERR_UNSUPPORTED
    # the same table again changes nothing
    i = d.index(b"\xFF\xDB")
    ln = (d[i + 2] << 8) | d[i + 3]
    assert emu_status(d[:p] + d[i:i + 2 + ln] + d[p:]) == BJ_OK


def test_levels_of_libjpeg_script():
    _, _, info = emu_decode(_base(), 1 << 16)
    assert info[0] == 10 and info[1] == 3


def test_damaged_scan_is_reported_and_bounded():
    d = bytearray(encoder_twins("420", "random", "simple", 3)[0])
    p = _sos_positions(bytes(d))[5]
    for k in range(40, 60):
        if d[p + k] not in (0xFF, 0x00) and d[p + k - 1] != 0xFF:
            d[p + k] ^= 0x5A
            if d[p + k] == 0xFF:
                d[p + k] ^= 0x01
    rc, _, info = emu_decode(bytes(d), 1 << 16)
    assert rc == BJ_OK and info[3] == 1
