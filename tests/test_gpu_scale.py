"""GPU tests of reduced-size decode (pytest -m gpu): the output of an image at 1/s of its size, cropped to a ROI of the
scaled image, is, byte for byte, what the same format holds for that crop of box_scale(full decode, s) - the full decode
being the oracle's (oracle_lib.Restated(data).rgb, pinned to the reference's hashes by test_oracle.py) - for RGB8 and
BMP, on every output path of the C ABI."""
import ctypes as C

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol
from test_gpu_roi import _DeviceBytes, _expected_rgb, _golden_names, _load, _pack, _peek, crop_bytes, rois_for

pytestmark = pytest.mark.gpu

SCALES = (1, 2, 4, 8)


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    yield d
    d.close()


def box_scale(rgb, s):
    """The scaled image: per channel, the rounded mean of each s x s box of the full decode rgb [H, W, 3], boxes cut
    short at the right and bottom edges."""
    H, W = rgb.shape[:2]
    Ho, Wo = -(-H // s), -(-W // s)
    acc = np.zeros((Ho * s, Wo * s, 3), np.uint32)
    acc[:H, :W] = rgb
    cnt = np.zeros((Ho * s, Wo * s), np.uint32)
    cnt[:H, :W] = 1
    S = acc.reshape(Ho, s, Wo, s, 3).sum((1, 3))
    N = cnt.reshape(Ho, s, Wo, s).sum((1, 3))[..., None]
    return ((S + N // 2) // N).astype(np.uint8)


def scaled_bytes(rgb, s, roi, fmt):
    return crop_bytes(box_scale(rgb, s), roi, fmt)


def test_box_scale_by_hand():
    """The expectation itself on a 3 x 5 image: interior boxes divide by s*s, edge boxes by what is left of them."""
    rgb = np.arange(45, dtype=np.uint8).reshape(3, 5, 3)
    assert np.array_equal(box_scale(rgb, 1), rgb)
    b2 = box_scale(rgb, 2)
    assert b2.shape == (2, 3, 3)
    assert b2[0, 0, 0] == (0 + 3 + 15 + 18 + 2) // 4
    assert b2[0, 2, 1] == (13 + 28 + 1) // 2           # the last column: 1 pixel wide
    assert b2[1, 2, 2] == 44                            # the corner: 1 pixel
    b8 = box_scale(rgb, 8)
    assert b8.shape == (1, 1, 3) and b8[0, 0, 0] == (int(rgb[..., 0].sum()) + 7) // 15


@pytest.mark.parametrize("fmt", [0, 1])
def test_golden_set_times_scales_and_rois(dec, fmt, golden, golden_dir):
    """Every golden image (4:2:0, 4:2:2, 4:4:0, 4:4:4, gray, odd sizes down to 1x1 and 17x17) at every scale under every
    ROI of rois_for on the scaled image - whole, 1x1 at each corner, crops ending in the partial edge box - in one batch."""
    files, rois, scales, wants = [], [], [], []
    for n in _golden_names(golden):
        data = _load(golden, golden_dir, n)
        rgb = _expected_rgb(golden, golden_dir, n)
        for s in SCALES:
            small = box_scale(rgb, s)
            for r in rois_for(small.shape[1], small.shape[0]):
                files.append(data)
                rois.append(r)
                scales.append(s)
                wants.append((n, s, r, crop_bytes(small, r, fmt)))
    outs, status = dec.decode(files, fmt, rois=np.array(rois, dtype=np.uint32), scales=np.array(scales, dtype=np.uint8))
    for (n, s, r, want), o, st in zip(wants, outs, status):
        assert st == 0 and o is not None and o.size == want.size and np.array_equal(o, want), (n, s, r)


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("sub,gray", [(2, False), (0, False), (0, True)])
def test_large_images_across_tiles(dec, w, h, sub, gray):
    """4:2:0, 4:4:4 and gray at 1920x1080 and 3840x2160 at every scale: a K2/K3 tile is 512 / 512 / 1536 pixels wide, so
    512 / s and 1536 / s output columns, and the crops straddle tile boundaries."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(w, h, seed=w + h + sub + 7 * gray + 3, subsampling=sub, gray=gray)
    rgb = ol.Restated(data, 0).rgb
    rng = np.random.default_rng(w + 3 * sub + gray)
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        files, rois, scales, wants = [], [], [], []
        for s in SCALES[1:]:
            small = box_scale(rgb, s)
            Hs, Ws = small.shape[:2]
            rs = [(0, 0, 0, 0), (512 // s - 3, 5, 40, 30), (1536 // s - 1, 0, 3, Hs), (Ws - 1, Hs - 1, 1, 1), (0, Hs - 1, Ws, 1),
                  (512 // s - 1, Hs // 2, 1024 // s + 2, Hs - Hs // 2)]
            for _ in range(4):
                rw, rh = int(rng.integers(1, Ws)), int(rng.integers(1, Hs))
                rs.append((int(rng.integers(0, Ws - rw + 1)), int(rng.integers(0, Hs - rh + 1)), rw, rh))
            for r in rs:
                files.append(data)
                rois.append(r)
                scales.append(s)
                wants.append((s, r, crop_bytes(small, r, fmt)))
        outs, status = dec.decode(files, fmt, rois=rois, scales=scales)
        for (s, r, want), o, st in zip(wants, outs, status):
            assert st == 0 and np.array_equal(o, want), (fmt, s, r)


def test_restart_images_scale_of_the_twin(dec):
    """A subsampled image with restart markers gives the scaled crop of its restart-free twin (restart-parity rule)."""
    import pim_jpeg_decoder_b200 as bj
    rgb0 = js.synth_rgb(961, 543, 5)
    with_ri = js.pil_jpeg(rgb0, 90, 2, restart_blocks=8)
    twin_rgb = ol.Restated(js.pil_jpeg(rgb0, 90, 2), 0).rgb
    cases = [(2, (0, 0, 0, 0)), (2, (17, 33, 400, 200)), (4, (0, 0, 0, 0)), (4, (239, 134, 2, 2)), (8, (0, 0, 0, 0)), (8, (100, 0, 21, 68)),
             (1, (5, 6, 7, 8))]
    outs, status = dec.decode([with_ri] * len(cases), bj.BJ_OUT_BMP, rois=[r for _, r in cases], scales=[s for s, _ in cases])
    for (s, r), o, st in zip(cases, outs, status):
        assert st == 0 and np.array_equal(o, scaled_bytes(twin_rgb, s, r, bj.BJ_OUT_BMP)), (s, r)


def test_damaged_and_truncated_scans_scale_of_the_partial_image(dec):
    """A damaged or truncated scan gives the scaled crop of the partial image the reference writes (BJ_ERR_CORRUPT_SCAN)."""
    import pim_jpeg_decoder_b200 as bj
    from test_huff_emu import _corrupt_scan
    data = js.synth_jpeg(320, 240, seed=19, subsampling=2)
    truncated = data[: len(data) - 2 - 3000] + b"\xFF\xD9"
    rng = np.random.default_rng(67)
    bads = [truncated] + [_corrupt_scan(js.synth_jpeg(200, 152, seed=50 + k, subsampling=k % 3), rng, 3)[0] for k in range(6)]
    scales = [2, 4, 8, 2, 4, 8, 2]
    rois = [(3, 100, 150, 20), (0, 0, 0, 0), (3, 1, 22, 18), (50, 30, 50, 46), (1, 1, 48, 37), (0, 0, 25, 19), (0, 75, 100, 1)]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(bads, fmt, rois=rois, scales=scales)
        failed = 0
        for b, s, r, o, st in zip(bads, scales, rois, outs, status):
            ro = ol.Restated(b, 0)
            failed += ro.huff_rc != 0
            assert st == (bj.BJ_ERR_CORRUPT_SCAN if ro.huff_rc != 0 else 0)
            assert np.array_equal(o, scaled_bytes(ro.rgb, s, r, fmt)), (s, r)
        assert failed >= 1


def _decode_roi_entry(bj, dec, files, rois, fmt, sizes):
    """bj_decode_batch_roi called directly, into buffers of `sizes` bytes pre-filled with 0x5A."""
    _, ptrs, lens = bj.decoder._file_arrays(files)
    outs = [np.full(s, 0x5A, dtype=np.uint8) if s else None for s in sizes]
    optrs = (C.c_void_p * len(files))(*[o.ctypes.data if o is not None else None for o in outs])
    ra = np.ascontiguousarray(rois, dtype=np.uint32)
    st = (C.c_int * len(files))()
    assert bj.lib().bj_decode_batch_roi(dec.ctx, ptrs, lens, ra.ctypes.data_as(C.c_void_p), len(files), fmt, optrs, st) == 0
    return outs, list(st)


def test_mixed_batch_and_refusals(dec, golden, golden_dir):
    """Scaled, s = 1 and whole-image entries, an invalid file, a scale the library does not have and a ROI that fits the
    full image but not the scaled one, in one batch: the refused images get BJ_ERR_ARG, the others are exact.  The s = 1
    entries are byte-identical to bj_decode_batch_roi, and so is scales=None; BJ_OUT_REF_MCUS with scales is refused."""
    import pim_jpeg_decoder_b200 as bj
    good = _load(golden, golden_dir, "p420_320x240")
    other = _load(golden, golden_dir, "p444_33x17")
    bad = _load(golden, golden_dir, "bad_not_jpeg")
    rgb, rgb2 = ol.Restated(good, 0).rgb, ol.Restated(other, 0).rgb
    files = [good, bad, good, other, good, other, good, other, good, good]
    rois = [(10, 20, 30, 40), (0, 0, 1, 1), (10, 20, 30, 40), (0, 0, 0, 0), (0, 0, 0, 0), (0, 0, 18, 9), (0, 0, 0, 0), (1, 1, 32, 16),
            (0, 0, 0, 0), (0x7FFFFFFF, 0, 0x80000002, 1)]
    scales = [2, 2, 1, 4, 3, 2, 8, 1, 16, 2]
    want_st = [0, bj.BJ_ERR_INVALID_JPEG, 0, 0, bj.BJ_ERR_ARG, bj.BJ_ERR_ARG, 0, 0, bj.BJ_ERR_ARG, bj.BJ_ERR_ARG]
    full = {id(good): rgb, id(other): rgb2}
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(files, fmt, rois=rois, scales=scales)
        assert status == want_st
        for i, (f, r, s, st) in enumerate(zip(files, rois, scales, status)):
            if st == 0:
                assert np.array_equal(outs[i], scaled_bytes(full[id(f)], s, r, fmt)), i
            else:
                assert outs[i] is None, i
        # the s = 1 entries: byte for byte what bj_decode_batch_roi writes for them
        ref, ref_st = _decode_roi_entry(bj, dec, files, rois, fmt, [o.size if (o is not None and s == 1) else 0 for o, s in zip(outs, scales)])
        for i, s in enumerate(scales):
            if s == 1:
                assert ref_st[i] == status[i] and np.array_equal(ref[i], outs[i]), i
        # scales=None through the _scaled entry == bj_decode_batch_roi, byte for byte and status for status
        roi_only = [(10, 20, 30, 40), (0, 0, 1, 1), (0, 0, 0, 0), (1, 1, 32, 16), (300, 0, 21, 1)]
        files5 = [good, bad, other, other, good]
        plain, st_plain = dec.decode(files5, fmt, rois=roi_only, scales=None)
        ref, ref_st = _decode_roi_entry(bj, dec, files5, roi_only, fmt, [o.size if o is not None else 0 for o in plain])
        assert st_plain == ref_st == [0, bj.BJ_ERR_INVALID_JPEG, 0, 0, bj.BJ_ERR_ARG]
        for a, b in zip(plain, ref):
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
    # BJ_OUT_REF_MCUS has no scale
    _, ptrs, lens = bj.decoder._file_arrays([good])
    sc = (C.c_uint8 * 1)(1)
    buf = np.zeros(1 << 20, dtype=np.uint8)
    optrs = (C.c_void_p * 1)(buf.ctypes.data)
    st = (C.c_int * 1)()
    assert bj.lib().bj_decode_batch_scaled(dec.ctx, ptrs, lens, None, sc, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == bj.BJ_ERR_ARG
    h = C.c_void_p()
    assert bj.lib().bj_batch_create_scaled(dec.ctx, ptrs, lens, None, sc, 1, bj.BJ_OUT_REF_MCUS, C.byref(h)) == bj.BJ_ERR_ARG and not h.value
    assert bj.lib().bj_submit_scaled(dec.ctx, ptrs, lens, None, sc, 1, bj.BJ_OUT_REF_MCUS, optrs, st, C.byref(h)) == bj.BJ_ERR_ARG
    assert bj.lib().bj_decode_batch_scaled(dec.ctx, ptrs, lens, None, None, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == 0 and st[0] == 0


def test_poisoned_buffers(dec, golden, golden_dir):
    """debug_poison = 1: every byte returned for a scaled crop was written by the decode."""
    import pim_jpeg_decoder_b200 as bj
    files, rois, scales, wants = [], [], [], []
    for k, n in enumerate(_golden_names(golden)):
        rgb = _expected_rgb(golden, golden_dir, n)
        for j, s in enumerate(SCALES):
            small = box_scale(rgb, s)
            rs = rois_for(small.shape[1], small.shape[0])
            files.append(_load(golden, golden_dir, n))
            rois.append(rs[(3 * k + j) % len(rs)])
            scales.append(s)
            wants.append(small)
    dec.set_option("debug_poison", 1)
    try:
        for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
            outs, status = dec.decode(files, fmt, rois=rois, scales=scales)
            for r, s, small, o, st in zip(rois, scales, wants, outs, status):
                assert st == 0 and np.array_equal(o, crop_bytes(small, r, fmt)), (s, r)
    finally:
        dec.set_option("debug_poison", 0)


def test_sub_batches_are_cut_by_scaled_bytes(dec):
    """The one-call path cuts sub-batches by the bytes of the scaled output: 12 images of 320x240 are 80x60 at 1/4
    (14400 B), four to a sub-batch of 64 KiB, and 40x30 at 1/8 (3600 B), all in one; whole, they take one each."""
    import pim_jpeg_decoder_b200 as bj
    uniq = [js.synth_jpeg(320, 240, seed=80 + k, subsampling=k % 3) for k in range(4)]
    files = [uniq[i % 4] for i in range(12)]
    rgbs = [ol.Restated(f, 0).rgb for f in uniq]
    dec.set_option("sub_batch_out_bytes", 1 << 16)
    try:
        for s, subs, nbytes in ((4, 3, 14400), (8, 1, 3600)):
            outs, status = dec.decode(files, bj.BJ_OUT_RGB8, scales=s)
            assert dec.stat("decode_batch_sub_batches") == subs
            assert dec.stat("decode_batch_d2h_bytes") == 12 * nbytes
            for i, (o, st) in enumerate(zip(outs, status)):
                assert st == 0 and np.array_equal(o, scaled_bytes(rgbs[i % 4], s, (0, 0, 0, 0), bj.BJ_OUT_RGB8)), (s, i)
        outs, status = dec.decode(files, bj.BJ_OUT_BMP, scales=4)
        assert dec.stat("decode_batch_sub_batches") == 3
        for i, (o, st) in enumerate(zip(outs, status)):
            assert st == 0 and np.array_equal(o, scaled_bytes(rgbs[i % 4], 4, (0, 0, 0, 0), bj.BJ_OUT_BMP)), i
        dec.decode(files, bj.BJ_OUT_RGB8)
        assert dec.stat("decode_batch_sub_batches") == 12
    finally:
        dec.set_option("sub_batch_out_bytes", 1 << 30)


def _mixed_case(golden, golden_dir):
    """Golden files three times over, each at a scale and with a ROI of its scaled image (invalid files: a 1x1 ROI)."""
    names = sorted(golden)
    files, rois, scales, wants = [], [], [], []
    for k, n in enumerate(names * 3):
        data = _load(golden, golden_dir, n)
        files.append(data)
        s = SCALES[k % 4]
        scales.append(s)
        if golden[n].get("invalid"):
            rois.append((0, 0, 1, 1))
            wants.append(None)
            continue
        small = box_scale(_expected_rgb(golden, golden_dir, n), s)
        rs = rois_for(small.shape[1], small.shape[0])
        rois.append(rs[(5 * k) % len(rs)])
        wants.append(small)
    return files, np.array(rois, dtype=np.uint32), np.array(scales, dtype=np.uint8), wants


def _layout(bj, files, rois, scales, fmt):
    sizes = []
    for f, r, s in zip(files, rois, scales):
        st, d = bj.parse_header(f)
        sizes.append(bj.scaled_output_size(d, r, s, fmt) if st == 0 else 0)
    offs = np.concatenate([[0], np.cumsum([(s + 15) // 16 * 16 for s in sizes])]).astype(np.int64)
    return sizes, offs[:-1], int(offs[-1]) + 16


def test_packed_outputs(dec, golden, golden_dir):
    """decode_packed with per-image scales and ROIs, outputs laid out by bj_scaled_output_size in one pinned buffer,
    copied out in runs (packed_outputs = 1), over many small sub-batches."""
    import pim_jpeg_decoder_b200 as bj
    files, rois, scales, wants = _mixed_case(golden, golden_dir)
    src, off, ln = _pack(bj, files)
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        sizes, dst_off, total = _layout(bj, files, rois, scales, fmt)
        dst = bj.PinnedBuffer(total)
        dec.set_option("packed_outputs", 1)
        dec.set_option("sub_batch_bytes", 1 << 16)
        try:
            status = dec.decode_packed(src.array, off, ln, dst.array, dst_off, fmt, rois=rois, scales=scales)
            assert dec.stat("decode_batch_sub_batches") > 3
            assert dec.stat("decode_batch_d2h_copies") < sum(1 for w in wants if w is not None)
        finally:
            dec.set_option("packed_outputs", 0)
            dec.set_option("sub_batch_bytes", 24 << 20)
        for i, (w, s, o, n) in enumerate(zip(wants, status, dst_off, sizes)):
            if w is None:
                assert s == bj.BJ_ERR_INVALID_JPEG
            else:
                assert s == 0 and np.array_equal(dst.array[o:o + n], crop_bytes(w, rois[i], fmt)), i
        dst.free()
    src.free()


def test_staged_batch_offsets_device_output_and_info(dec, golden, golden_dir):
    """Batch(..., rois=, scales=): offsets and sizes are the scaled crops', device_output reports their bytes, info()
    counts the scaled output bytes and the full images' pixels, and the download is exact."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    files, rois, scales, wants = _mixed_case(golden, golden_dir)
    peeked = [_peek(bj, f) for f in files]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        b = bj.Batch(dec, files, fmt, rois=rois, scales=scales)
        try:
            parsed = [st == 0 for st in b.parse_status]
            assert parsed == [d is not None for d in peeked]
            assert b.sizes == [bj.scaled_output_size(d, r, s, fmt) if d is not None else 0 for d, r, s in zip(peeked, rois, scales)]
            b.upload()
            b.decode()
            b.sync()
            assert [s == 0 for s in b.status()] == [w is not None for w in wants]
            views = b.download()
            info = b.info()
            assert info.out_bytes == sum((s + 15) // 16 * 16 for s, v in zip(b.sizes, parsed) if v)
            assert info.d2h_bytes == sum(s for s, v in zip(b.sizes, parsed) if v)
            assert info.pixels == sum(d.width * d.height for d in peeked if d is not None)
            for i, w in enumerate(wants):
                if w is None:
                    continue
                want = crop_bytes(w, rois[i], fmt)
                assert b.sizes[i] == want.size and np.array_equal(views[i], want), i
                p, nb = b.device_output(i)
                assert nb == want.size
                on_device = torch.as_tensor(_DeviceBytes(p, nb), device="cuda")
                assert np.array_equal(on_device.cpu().numpy(), want), i
        finally:
            b.destroy()


def test_submit_scaled_on_a_multi_device_context(golden, golden_dir):
    """bj_submit_scaled / bj_decode_batch_scaled on a context of three devices (the one GPU three times on a one-GPU
    box): sub-batches dealt over the devices, jobs in the background, outputs exact."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    ngpu = torch.cuda.device_count()
    devices = list(range(ngpu)) if ngpu > 1 else [0, 0, 0]
    md = bj.Decoder(devices=devices)
    try:
        files, rois, scales, wants = _mixed_case(golden, golden_dir)
        files, wants = files * 2, wants * 2
        rois, scales = np.concatenate([rois, rois]), np.concatenate([scales, scales])
        src, off, ln = _pack(bj, files)
        sizes, dst_off, total = _layout(bj, files, rois, scales, bj.BJ_OUT_BMP)
        md.set_option("sub_batch_bytes", 1 << 16)
        md.set_option("packed_outputs", 1)
        dsts = [bj.PinnedBuffer(total) for _ in range(3)]
        status = md.decode_packed(src.array, off, ln, dsts[0].array, dst_off, bj.BJ_OUT_BMP, rois=rois, scales=scales)
        assert md.stat("decode_batch_sub_batches") > 8
        jobs = [md.submit_packed(src.array, off, ln, d.array, dst_off, bj.BJ_OUT_BMP, rois=rois, scales=scales) for d in dsts[1:]]
        sts = [status] + [j.wait() for j in jobs]
        for st, d in zip(sts, dsts):
            for i, (w, s, o, n) in enumerate(zip(wants, st, dst_off, sizes)):
                if w is None:
                    assert s == bj.BJ_ERR_INVALID_JPEG
                else:
                    assert s == 0 and np.array_equal(d.array[o:o + n], crop_bytes(w, rois[i], bj.BJ_OUT_BMP)), i
        for d in dsts:
            d.free()
        src.free()
    finally:
        md.close()


def test_decode_without_outs_sizes_whole_images_in_every_format(dec, golden, golden_dir):
    """Decoder.decode without `outs`, `rois` and `scales` sizes each output with bj_output_size, in every format:
    BJ_OUT_REF_MCUS - which has no crop and no scale - included.  Its buffers are the reference's `mcus` tiles after the
    DPU program, whole."""
    import pim_jpeg_decoder_b200 as bj
    names = _golden_names(golden)
    files = [_load(golden, golden_dir, n) for n in names]
    rs = [ol.Restated(f, 0) for f in files]
    outs, status = dec.decode(files, bj.BJ_OUT_REF_MCUS)
    assert status == [0] * len(files)
    for n, f, o, r in zip(names, files, outs, rs):
        st, d = bj.parse_header(f)
        assert o is not None and o.size == bj.lib().bj_output_size(C.byref(d), bj.BJ_OUT_REF_MCUS) == r.mcus_post.nbytes, n
        assert np.array_equal(o.view(np.int16).reshape(r.mcus_post.shape), r.mcus_post), n
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(files, fmt)
        for n, o, st in zip(names, outs, status):
            assert st == 0 and np.array_equal(o, scaled_bytes(_expected_rgb(golden, golden_dir, n), 1, (0, 0, 0, 0), fmt)), (fmt, n)
