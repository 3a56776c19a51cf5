"""GPU tests of progressive (SOF2) decode (context option "progressive"): every output must equal the output of the
file's baseline twin (same frame, same quantised coefficients, one interleaved baseline scan) - the GPU's decode of the
twin and the oracle's - byte for byte, in every entry and composed with ROIs, scales and sizes."""
import ctypes as C

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol
import prog_synth as ps
from test_progressive_emu import encoder_cases, encoder_twins, pil_twins_or_skip

pytestmark = pytest.mark.gpu

FMTS = (0, 1)     # BJ_OUT_RGB8, BJ_OUT_BMP


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    d.set_option("progressive", 1)
    yield d
    d.close()


def oracle_bytes(twin, fmt):
    r = ol.Restated(twin, 0)
    return r.rgb.reshape(-1) if fmt == 0 else r.bmp


def pillow_pairs(samp, sizes, ris):
    sub = {"420": 2, "422": 1, "444": 0, "gray": 0}[samp]
    out = []
    for (w, h) in sizes:
        for ri in ris:
            try:
                out.append(ps.pil_twins(js.synth_rgb(w, h, w + 3 * h + ri), 90, sub, ri, gray=samp == "gray"))
            except OSError:
                pass                                    # (Pillow cannot write a few large progressive files with restarts)
    return out


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("samp", ["420", "422", "444", "gray"])
def test_pillow_twins(dec, samp, fmt):
    pairs = pillow_pairs(samp, [(1, 1), (17, 17), (45, 30), (500, 375)], (0, 1, 5, 64))
    if samp == "420":
        pairs += pillow_pairs(samp, [(3840, 2160)], (0, 64))
    files = [p for p, _ in pairs] + [t for _, t in pairs]
    outs, st = dec.decode(files, fmt)
    assert st == [0] * len(files)
    n = len(pairs)
    for i, (_, twin) in enumerate(pairs):
        want = oracle_bytes(twin, fmt)
        assert np.array_equal(outs[n + i], want), f"twin {i} differs from the oracle"
        assert np.array_equal(outs[i], want), f"progressive file {i} differs from its twin"


@pytest.mark.parametrize("fmt", FMTS)
def test_encoder_twins(dec, fmt):
    cases = encoder_cases()
    files = [encoder_twins(*c)[0] for c in cases]
    outs, st = dec.decode(files, fmt)
    assert st == [0] * len(files)
    for c, o in zip(cases, outs):
        assert np.array_equal(o, oracle_bytes(encoder_twins(*c)[1], fmt)), c


# ------------------------------------------------------------------------------------------------ composition
def _mixed():
    """progressive, baseline, invalid, refused (65 scans), progressive with restarts - and the same with twins."""
    p1, t1 = ps.pil_twins(js.synth_rgb(500, 375, 1), 90, 2)
    p2, t2 = ps.pil_twins(js.synth_rgb(45, 30, 2), 90, 1, 5)
    base = js.synth_jpeg(64, 48, 3)
    comps = [(1, 1, 0, 0, 0)]
    co = js.random_coefs(comps, 16, 16, 4)
    many = ps.encode_progressive(16, 16, comps, co, [((0,), 0, 0, 0, 1)] + [((0,), k, k, 0, 0) for k in range(1, 64)] + [((0,), 0, 0, 1, 0)])
    prog = [p1, base, b"\xFF\xD8\xFF\xD9junk", many, p2]
    twin = [t1, base, b"\xFF\xD8\xFF\xD9junk", many, t2]
    return prog, twin


REQ = dict(rois=[(10, 20, 100, 50), (0, 0, 0, 0), (0, 0, 0, 0), (0, 0, 0, 0), (3, 2, 9, 7)],
           scales=[2, 4, 1, 1, 1], sizes=[(224, 224), (0, 0), (0, 0), (0, 0), (17, 9)])


def _submit(dec, files, fmt, rois, scales, sizes):
    import pim_jpeg_decoder_b200 as bj
    from pim_jpeg_decoder_b200 import decoder as D
    n = len(files)
    keep, ptrs, lens = D._file_arrays(files)
    ra, rp = D._roi_table(rois, n)
    sa, sp = D._scale_table(scales, n)
    za, zp = D._size_table(sizes, n)
    outs = []
    for i, f in enumerate(files):
        st, d = D._sizing_header(f)
        outs.append(np.zeros(bj.resized_output_size(d, rois[i], scales[i], sizes[i], fmt) if st == 0 else 0, dtype=np.uint8))
    optrs = (C.c_void_p * n)(*[o.ctypes.data if o.size else None for o in outs])
    status = (C.c_int * n)()
    job = C.c_void_p()
    assert bj.lib().bj_submit_resized(dec.ctx, ptrs, lens, rp, sp, zp, n, fmt, optrs, status, C.byref(job)) == 0
    assert bj.lib().bj_wait(job) == 0
    return outs, list(status)


def _batch(dec, files, fmt, rois, scales, sizes):
    import pim_jpeg_decoder_b200 as bj
    b = bj.Batch(dec, files, fmt, rois=rois, scales=scales, sizes=sizes)
    b.upload(); b.decode(); b.sync()
    outs = b.download()
    st = b.status()
    b.destroy()
    return outs, st


@pytest.mark.parametrize("entry", ["call", "submit", "batch", "multi"])
@pytest.mark.parametrize("fmt", FMTS)
def test_composition_in_mixed_batches(dec, entry, fmt):
    import pim_jpeg_decoder_b200 as bj
    prog, twin = _mixed()
    d = dec
    if entry == "multi":
        d = bj.Decoder(devices=[0, 0])
        d.set_option("progressive", 1)
        d.set_option("sub_batch_bytes", 1 << 16)
    run = {"call": lambda d, f: d.decode(f, fmt, **REQ), "multi": lambda d, f: d.decode(f, fmt, **REQ),
           "submit": lambda d, f: _submit(d, f, fmt, **REQ), "batch": lambda d, f: _batch(d, f, fmt, **REQ)}[entry]
    try:
        po, pst = run(d, prog)
        to, tst = run(d, twin)
    finally:
        if d is not dec:
            d.close()
    assert pst == [0, 0, -4, -5, 0] and tst == [0, 0, -4, -5, 0]
    for i in (0, 1, 4):
        assert np.array_equal(po[i], to[i]), i


def test_option_off(dec):
    import pim_jpeg_decoder_b200 as bj
    p, t = ps.pil_twins(js.synth_rgb(45, 30, 9), 90, 2)
    base = [js.synth_jpeg(64, 48, 3), js.synth_jpeg(33, 17, 4, 0)]
    off = bj.Decoder(0)
    try:
        outs, st = off.decode([base[0], p, base[1], p], 0)
        ref, rst = off.decode(base, 0)
    finally:
        off.close()
    assert st == [0, -5, 0, -5] and rst == [0, 0]
    assert np.array_equal(outs[0], ref[0]) and np.array_equal(outs[2], ref[1])


# ------------------------------------------------------------------------------------------------ refusals and damage
def test_refusals(dec):
    import pim_jpeg_decoder_b200 as bj
    p, t = ps.pil_twins(js.synth_rgb(45, 30, 5), 90, 2)
    base = js.synth_jpeg(64, 48, 3)
    # BJ_OUT_REF_MCUS: the progressive image alone is refused
    outs, st = dec.decode([base, p], bj.BJ_OUT_REF_MCUS)
    assert st == [0, -5]
    assert np.array_equal(outs[0], dec.decode([base], bj.BJ_OUT_REF_MCUS)[0][0])
    # a redefined quantisation table in use
    i = p.index(b"\xFF\xDA", p.index(b"\xFF\xDA") + 2)
    dqt = b"\xFF\xDB\x00\x43\x00" + bytes(range(1, 65))
    _, st = dec.decode([p[:i] + dqt + p[i:], p[:-2], base], 0)
    assert st == [-5, -4, 0]
    # the stage-level entries keep taking one scan
    assert bj.lib().bj_parse_header(p, len(p), C.byref(bj.ImageDesc())) == -4


def _flip(data):
    """flip bytes inside the third scan without making or breaking a marker"""
    d = bytearray(data)
    s = 0
    for _ in range(3):
        s = data.index(b"\xFF\xDA", s + 2)
    start = s + 2 + ((d[s + 2] << 8) | d[s + 3])
    for k in range(start + 20, start + 60, 7):
        if d[k] != 0xFF and d[k - 1] != 0xFF and d[k] ^ 0x5A != 0xFF:
            d[k] ^= 0x5A
    return bytes(d)


def test_damaged_scans_are_deterministic(dec):
    p, t = ps.pil_twins(js.synth_rgb(500, 375, 6), 90, 2, 5)
    base = js.synth_jpeg(64, 48, 3)
    bad = _flip(p)
    outs = []
    for poison in (0, 1):
        dec.set_option("debug_poison", poison)
        try:
            o, st = dec.decode([base, bad, p], 0)
        finally:
            dec.set_option("debug_poison", 0)
        assert st == [0, -6, 0]
        outs.append(o)
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    assert np.array_equal(outs[0][0], oracle_bytes(base, 0))
    assert np.array_equal(outs[0][2], oracle_bytes(t, 0))


def test_counters(dec):
    p, t = ps.pil_twins(js.synth_rgb(500, 375, 7), 90, 2)
    base = js.synth_jpeg(64, 48, 3)
    dec.decode([base], 0)
    l0 = dec.stat("decode_batch_launches")
    assert dec.stat("decode_batch_ms_progressive") == 0
    t0 = dec.stat("total_ms_progressive")
    _, st = dec.decode([base, p], 0)
    assert st == [0, 0]
    assert dec.stat("decode_batch_ms_progressive") > 0
    assert dec.stat("total_ms_progressive") > t0
    assert dec.stat("decode_batch_launches") == l0 + 1 + 3    # the DC clear and one launch per level
