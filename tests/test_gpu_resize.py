"""GPU tests of fixed-size output (pytest -m gpu): the output of an image resized to w x h is, byte for byte, what the
same format holds for bilinear(crop(box_scale(full decode, s), roi), w, h) - the full decode being the oracle's
(oracle_lib.Restated(data).rgb, pinned to the reference's hashes by test_oracle.py) - for RGB8 and BMP, on every output
path of the C ABI."""
import ctypes as C

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol
from resize_ref import bilinear, crop
from test_gpu_roi import _DeviceBytes, _expected_rgb, _golden_names, _load, _pack, _peek, crop_bytes, rois_for
from test_gpu_scale import SCALES, box_scale

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    yield d
    d.close()


def resized(rgb, s, roi, size):
    """The expected w x h image (size None or (0, 0): the scaled crop itself)."""
    src = crop(box_scale(rgb, s), roi)
    if size is None or tuple(int(v) for v in size) == (0, 0):
        return src
    return bilinear(src, int(size[0]), int(size[1]))


def resized_bytes(rgb, s, roi, size, fmt):
    return crop_bytes(resized(rgb, s, roi, size), (0, 0, 0, 0), fmt)


def sizes_for(cw, ch):
    """The target sizes every crop is resized to: 1 x 1, its own size, an exact half, 224 x 224, 13 x 300 and an upscale
    by about 3.7x."""
    return [(1, 1), (cw, ch), (max(1, cw // 2), max(1, ch // 2)), (224, 224), (13, 300),
            (min(65535, -(-cw * 37 // 10)), min(65535, -(-ch * 37 // 10)))]


@pytest.mark.parametrize("fmt", [0, 1])
def test_golden_set_times_scales_rois_and_sizes(dec, fmt, golden, golden_dir):
    """Every golden image at every scale, under three ROIs of the scaled image, at every size of sizes_for, in one
    batch.  The decode's ms_resize counter sees the new kernel."""
    files, rois, scales, sizes, wants = [], [], [], [], []
    for k, n in enumerate(_golden_names(golden)):
        data = _load(golden, golden_dir, n)
        rgb = _expected_rgb(golden, golden_dir, n)
        for s in SCALES:
            small = box_scale(rgb, s)
            rs = rois_for(small.shape[1], small.shape[0])
            for r in {rs[0], rs[(k + s) % len(rs)], rs[-1]}:
                c = crop(small, r)
                for z in sizes_for(c.shape[1], c.shape[0]):
                    files.append(data)
                    rois.append(r)
                    scales.append(s)
                    sizes.append(z)
                    wants.append((n, s, r, z, crop_bytes(bilinear(c, *z), (0, 0, 0, 0), fmt)))
    outs, status = dec.decode(files, fmt, rois=rois, scales=scales, sizes=sizes)
    for (n, s, r, z, want), o, st in zip(wants, outs, status):
        assert st == 0 and o is not None and o.size == want.size and np.array_equal(o, want), (n, s, r, z)
    assert dec.stat("decode_batch_ms_resize") > 0


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("sub,gray", [(2, False), (0, False), (0, True)])
def test_large_images_across_tiles(dec, w, h, sub, gray):
    """4:2:0, 4:4:4 and gray at 1920x1080 and 3840x2160: crops that straddle IDCT tiles (512 / 1536 pixels wide) and
    resize tiles (64 x 48 output pixels), resized to 224 x 224 and up to 1920 x 1080."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(w, h, seed=w + h + sub + 7 * gray + 5, subsampling=sub, gray=gray)
    rgb = ol.Restated(data, 0).rgb
    rng = np.random.default_rng(w + 5 * sub + gray)
    reqs = [(1, (0, 0, 0, 0), (224, 224)), (1, (0, 0, 0, 0), (1920, 1080)), (2, (0, 0, 0, 0), (224, 224)), (8, (0, 0, 0, 0), (1920, 1080)),
            (1, (509, 3, 1030, 700), (224, 224)), (1, (1533, 17, 7, 1000), (1919, 1079)), (2, (255, 100, 300, 211), (1000, 37)),
            (4, (127, 1, 129, 100), (65, 25)), (1, (w - 300, h - 200, 300, 200), (1920, 1080))]
    for _ in range(3):
        s = int(rng.choice(SCALES))
        Ws, Hs = -(-w // s), -(-h // s)
        rw, rh = int(rng.integers(1, Ws)), int(rng.integers(1, Hs))
        reqs.append((s, (int(rng.integers(0, Ws - rw + 1)), int(rng.integers(0, Hs - rh + 1)), rw, rh), (int(rng.integers(1, 1921)), int(rng.integers(1, 1081)))))
    smalls = {s: box_scale(rgb, s) for s in SCALES}
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode([data] * len(reqs), fmt, rois=[r for _, r, _ in reqs], scales=[s for s, _, _ in reqs], sizes=[z for _, _, z in reqs])
        for (s, r, z), o, st in zip(reqs, outs, status):
            want = crop_bytes(bilinear(crop(smalls[s], r), *z), (0, 0, 0, 0), fmt)
            assert st == 0 and np.array_equal(o, want), (fmt, s, r, z)


def test_restart_images_resize_of_the_twin(dec):
    """A subsampled image with restart markers gives the resized crop of its restart-free twin."""
    import pim_jpeg_decoder_b200 as bj
    rgb0 = js.synth_rgb(961, 543, 5)
    with_ri = js.pil_jpeg(rgb0, 90, 2, restart_blocks=8)
    twin_rgb = ol.Restated(js.pil_jpeg(rgb0, 90, 2), 0).rgb
    cases = [(1, (0, 0, 0, 0), (224, 224)), (2, (17, 33, 400, 200), (13, 300)), (4, (0, 0, 0, 0), (961, 543)), (8, (100, 0, 21, 68), (1, 1)),
             (1, (5, 6, 7, 8), (26, 30))]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode([with_ri] * len(cases), fmt, rois=[r for _, r, _ in cases], scales=[s for s, _, _ in cases],
                                  sizes=[z for _, _, z in cases])
        for (s, r, z), o, st in zip(cases, outs, status):
            assert st == 0 and np.array_equal(o, resized_bytes(twin_rgb, s, r, z, fmt)), (s, r, z)


def test_damaged_and_truncated_scans_resize_of_the_partial_image(dec):
    """A damaged or truncated scan gives the resized crop of the partial image the reference writes (BJ_ERR_CORRUPT_SCAN)."""
    import pim_jpeg_decoder_b200 as bj
    from test_huff_emu import _corrupt_scan
    data = js.synth_jpeg(320, 240, seed=23, subsampling=2)
    truncated = data[: len(data) - 2 - 3000] + b"\xFF\xD9"
    rng = np.random.default_rng(71)
    bads = [truncated] + [_corrupt_scan(js.synth_jpeg(200, 152, seed=60 + k, subsampling=k % 3), rng, 3)[0] for k in range(6)]
    scales = [1, 2, 4, 8, 1, 2, 1]
    rois = [(3, 100, 150, 120), (0, 0, 0, 0), (3, 1, 22, 18), (0, 0, 0, 0), (1, 1, 48, 37), (0, 0, 25, 19), (0, 75, 100, 1)]
    sizes = [(224, 224), (50, 38), (1, 1), (100, 76), (13, 300), (0, 0), (64, 3)]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(bads, fmt, rois=rois, scales=scales, sizes=sizes)
        failed = 0
        for b, s, r, z, o, st in zip(bads, scales, rois, sizes, outs, status):
            ro = ol.Restated(b, 0)
            failed += ro.huff_rc != 0
            assert st == (bj.BJ_ERR_CORRUPT_SCAN if ro.huff_rc != 0 else 0)
            assert np.array_equal(o, resized_bytes(ro.rgb, s, r, z, fmt)), (s, r, z)
        assert failed >= 1


def _decode_scaled_entry(bj, dec, files, rois, scales, fmt, sizes):
    """bj_decode_batch_scaled called directly, into buffers of `sizes` bytes pre-filled with 0x5A."""
    _, ptrs, lens = bj.decoder._file_arrays(files)
    outs = [np.full(s, 0x5A, dtype=np.uint8) if s else None for s in sizes]
    optrs = (C.c_void_p * len(files))(*[o.ctypes.data if o is not None else None for o in outs])
    ra = np.ascontiguousarray(rois, dtype=np.uint32)
    sa = np.ascontiguousarray(scales, dtype=np.uint8)
    st = (C.c_int * len(files))()
    assert bj.lib().bj_decode_batch_scaled(dec.ctx, ptrs, lens, ra.ctypes.data_as(C.c_void_p), sa.ctypes.data_as(C.c_void_p), len(files), fmt,
                                           optrs, st) == 0
    return outs, list(st)


def test_mixed_batch_and_refusals(dec, golden, golden_dir):
    """Resized, unresized ({0,0}), scaled-only and refused entries in one batch: refused sizes (one side 0, a side above
    65535) and bad scales or ROIs get BJ_ERR_ARG, a size above max_image_pixels BJ_ERR_UNSUPPORTED, the others are
    exact.  The unresized entries are byte-identical to bj_decode_batch_scaled, and so is sizes=None; BJ_OUT_REF_MCUS
    with sizes is refused for the whole call."""
    import pim_jpeg_decoder_b200 as bj
    good = _load(golden, golden_dir, "p420_320x240")
    other = _load(golden, golden_dir, "p444_33x17")
    bad = _load(golden, golden_dir, "bad_not_jpeg")
    full = {id(good): ol.Restated(good, 0).rgb, id(other): ol.Restated(other, 0).rgb}
    E, U, I = bj.BJ_ERR_ARG, bj.BJ_ERR_UNSUPPORTED, bj.BJ_ERR_INVALID_JPEG
    cases = [  # file, roi, scale, size, status
        (good, (10, 20, 30, 40), 2, (224, 224), 0), (bad, (0, 0, 1, 1), 1, (5, 5), I), (good, (10, 20, 30, 40), 1, (0, 0), 0),
        (other, (0, 0, 0, 0), 4, (7, 3), 0), (good, (0, 0, 0, 0), 2, (1, 0), E), (other, (0, 0, 0, 0), 1, (0, 9), E),
        (good, (0, 0, 0, 0), 8, (0, 0), 0), (other, (1, 1, 32, 16), 1, (65536, 2), E), (good, (0, 0, 0, 0), 3, (10, 10), E),
        (good, (0, 0, 161, 1), 2, (10, 10), E), (good, (0, 0, 0, 0), 1, (4096, 513), U), (other, (2, 3, 5, 7), 1, (33, 17), 0),
        (good, (0, 0, 0, 0), 1, (320, 240), 0)]
    files = [c[0] for c in cases]
    rois = np.array([c[1] for c in cases], dtype=np.uint32)
    scales = np.array([c[2] for c in cases], dtype=np.uint8)
    sizes = np.array([c[3] for c in cases], dtype=np.uint32)          # (a side above 65535 is refused by the Python layer, the rest by the library)
    dec.set_option("max_image_pixels", 1 << 21)
    try:
        for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
            outs, status = dec.decode(files, fmt, rois=rois, scales=scales, sizes=sizes)
            assert status == [c[4] for c in cases]
            for i, (f, r, s, z, st) in enumerate(cases):
                if st == 0:
                    assert np.array_equal(outs[i], resized_bytes(full[id(f)], s, r, z, fmt)), i
                else:
                    assert outs[i] is None, i
            # the unresized entries: byte for byte what bj_decode_batch_scaled writes for them
            ref, ref_st = _decode_scaled_entry(bj, dec, files, rois, scales, fmt,
                                               [o.size if (o is not None and tuple(z) == (0, 0)) else 0 for o, z in zip(outs, sizes)])
            for i, z in enumerate(sizes):
                if tuple(z) == (0, 0):
                    assert ref_st[i] == status[i] and np.array_equal(ref[i], outs[i]), i
            # sizes=None through the _resized entry == bj_decode_batch_scaled, byte for byte and status for status
            plain, st_plain = dec.decode(files, fmt, rois=rois, scales=scales, sizes=None)
            ref, ref_st = _decode_scaled_entry(bj, dec, files, rois, scales, fmt, [o.size if o is not None else 0 for o in plain])
            assert st_plain == ref_st
            for a, b in zip(plain, ref):
                assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
    finally:
        dec.set_option("max_image_pixels", 1 << 28)
    _, ptrs, lens = bj.decoder._file_arrays([good])
    z = (bj.Size * 1)(bj.Size(0, 0))
    buf = np.zeros(1 << 20, dtype=np.uint8)
    optrs = (C.c_void_p * 1)(buf.ctypes.data)
    st = (C.c_int * 1)()
    assert bj.lib().bj_decode_batch_resized(dec.ctx, ptrs, lens, None, None, z, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == bj.BJ_ERR_ARG
    h = C.c_void_p()
    assert bj.lib().bj_batch_create_resized(dec.ctx, ptrs, lens, None, None, z, 1, bj.BJ_OUT_REF_MCUS, C.byref(h)) == bj.BJ_ERR_ARG and not h.value
    assert bj.lib().bj_submit_resized(dec.ctx, ptrs, lens, None, None, z, 1, bj.BJ_OUT_REF_MCUS, optrs, st, C.byref(h)) == bj.BJ_ERR_ARG
    assert bj.lib().bj_decode_batch_resized(dec.ctx, ptrs, lens, None, None, None, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == 0 and st[0] == 0


def test_poisoned_buffers(dec, golden, golden_dir):
    """debug_poison = 1 (which covers the intermediate region too): every byte returned was written by the decode."""
    import pim_jpeg_decoder_b200 as bj
    files, rois, scales, sizes, wants = [], [], [], [], []
    for k, n in enumerate(_golden_names(golden)):
        rgb = _expected_rgb(golden, golden_dir, n)
        for j, s in enumerate(SCALES):
            small = box_scale(rgb, s)
            rs = rois_for(small.shape[1], small.shape[0])
            r = rs[(3 * k + j) % len(rs)]
            c = crop(small, r)
            z = sizes_for(c.shape[1], c.shape[0])[(k + j) % 6]
            files.append(_load(golden, golden_dir, n))
            rois.append(r)
            scales.append(s)
            sizes.append(z)
            wants.append(bilinear(c, *z))
    dec.set_option("debug_poison", 1)
    try:
        for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
            outs, status = dec.decode(files, fmt, rois=rois, scales=scales, sizes=sizes)
            for r, s, z, want, o, st in zip(rois, scales, sizes, wants, outs, status):
                assert st == 0 and np.array_equal(o, crop_bytes(want, (0, 0, 0, 0), fmt)), (s, r, z)
    finally:
        dec.set_option("debug_poison", 0)


def test_sub_batches_are_cut_by_final_and_intermediate_bytes(dec):
    """The one-call path cuts sub-batches by the final bytes plus the scaled crop the resize reads: 12 images of 320x240
    to 64 x 48 (9216 B) at s = 1 hold 230400 B of source each, one to a sub-batch of 64 KiB; at s = 4 the source is
    14400 B, two to a sub-batch.  Only the final bytes are copied out."""
    import pim_jpeg_decoder_b200 as bj
    uniq = [js.synth_jpeg(320, 240, seed=90 + k, subsampling=k % 3) for k in range(4)]
    files = [uniq[i % 4] for i in range(12)]
    rgbs = [ol.Restated(f, 0).rgb for f in uniq]
    dec.set_option("sub_batch_out_bytes", 1 << 16)
    try:
        for s, subs in ((1, 12), (4, 6)):
            for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
                outs, status = dec.decode(files, fmt, scales=s, sizes=(64, 48))
                assert dec.stat("decode_batch_sub_batches") == subs
                assert dec.stat("decode_batch_d2h_bytes") == 12 * (9216 if fmt == bj.BJ_OUT_RGB8 else 26 + 9216)
                for i, (o, st) in enumerate(zip(outs, status)):
                    assert st == 0 and np.array_equal(o, resized_bytes(rgbs[i % 4], s, (0, 0, 0, 0), (64, 48), fmt)), (s, i)
    finally:
        dec.set_option("sub_batch_out_bytes", 1 << 30)


def _plan_case(bj, golden, golden_dir, tw, th):
    """Golden files three times over with a random box each, turned into a request by resize_plan (invalid files: a
    1x1 ROI at scale 1)."""
    rng = np.random.default_rng(tw * 7 + th)
    files, rois, scales, wants = [], [], [], []
    for n in sorted(golden) * 3:
        data = _load(golden, golden_dir, n)
        files.append(data)
        if golden[n].get("invalid"):
            rois.append((0, 0, 1, 1))
            scales.append(1)
            wants.append(None)
            continue
        rgb = _expected_rgb(golden, golden_dir, n)
        H, W = rgb.shape[:2]
        w, h = int(rng.integers(1, W + 1)), int(rng.integers(1, H + 1))
        box = (int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1)), w, h)
        s, r = bj.resize_plan(W, H, box, (tw, th))
        rois.append(r)
        scales.append(s)
        wants.append(resized(rgb, s, r, (tw, th)))
    return files, np.array(rois, dtype=np.uint32), np.array(scales, dtype=np.uint8), wants


def test_packed_into_one_array(dec, golden, golden_dir):
    """decode_packed and submit_packed with one size for every image write one [n, th, tw, 3] pinned array, copied out
    in runs (packed_outputs = 1) over many small sub-batches."""
    import pim_jpeg_decoder_b200 as bj
    tw, th = 48, 40
    files, rois, scales, wants = _plan_case(bj, golden, golden_dir, tw, th)
    n = len(files)
    src, off, ln = _pack(bj, files)
    dsts = [bj.PinnedBuffer(n * th * tw * 3) for _ in range(2)]
    dst_off = np.arange(n, dtype=np.int64) * (th * tw * 3)
    dec.set_option("packed_outputs", 1)
    dec.set_option("sub_batch_bytes", 1 << 16)
    try:
        status = dec.decode_packed(src.array, off, ln, dsts[0].array, dst_off, bj.BJ_OUT_RGB8, rois=rois, scales=scales, sizes=(tw, th))
        assert dec.stat("decode_batch_sub_batches") > 3
        assert dec.stat("decode_batch_d2h_copies") < sum(1 for w in wants if w is not None)
        status2 = dec.submit_packed(src.array, off, ln, dsts[1].array, dst_off, bj.BJ_OUT_RGB8, rois=rois, scales=scales, sizes=(tw, th)).wait()
    finally:
        dec.set_option("packed_outputs", 0)
        dec.set_option("sub_batch_bytes", 24 << 20)
    for st, d in zip((status, status2), dsts):
        arr = d.array.reshape(n, th, tw, 3)
        for i, (w, s) in enumerate(zip(wants, st)):
            if w is None:
                assert s == bj.BJ_ERR_INVALID_JPEG
            else:
                assert s == 0 and np.array_equal(arr[i], w), i
    for d in dsts:
        d.free()
    src.free()


def test_staged_batch_offsets_device_output_and_info(dec, golden, golden_dir):
    """Batch(..., sizes=): offsets and sizes are the final outputs', d2h_bytes is the sum of bj_resized_output_size,
    device_output holds the final bytes (read through torch), info() counts the full images' pixels."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    files, rois, scales, wants = _plan_case(bj, golden, golden_dir, 30, 20)
    sizes = np.array([(30, 20) if k % 3 else (0, 0) for k in range(len(files))], dtype=np.uint32)
    peeked = [_peek(bj, f) for f in files]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        b = bj.Batch(dec, files, fmt, rois=rois, scales=scales, sizes=sizes)
        try:
            parsed = [st == 0 for st in b.parse_status]
            want_sizes = [bj.resized_output_size(d, r, s, z, fmt) if d is not None else 0 for d, r, s, z in zip(peeked, rois, scales, sizes)]
            assert b.sizes == want_sizes
            b.upload()
            b.decode()
            b.sync()
            assert [s == 0 for s in b.status()] == [w is not None for w in wants]
            views = b.download()
            info = b.info()
            assert info.d2h_bytes == sum(s for s, v in zip(want_sizes, parsed) if v)
            assert info.out_bytes == sum((s + 15) // 16 * 16 for s, v in zip(want_sizes, parsed) if v)
            assert info.pixels == sum(d.width * d.height for d in peeked if d is not None)
            for i, w in enumerate(wants):
                if w is None:
                    continue
                img = w if tuple(sizes[i]) != (0, 0) else crop(box_scale(_expected_rgb(golden, golden_dir, sorted(golden)[i % len(golden)]), int(scales[i])), rois[i])
                want = crop_bytes(img, (0, 0, 0, 0), fmt)
                assert np.array_equal(views[i], want), i
                p, nb = b.device_output(i)
                assert nb == want.size
                assert np.array_equal(torch.as_tensor(_DeviceBytes(p, nb), device="cuda").cpu().numpy(), want), i
        finally:
            b.destroy()


def test_submit_resized_on_a_multi_device_context(golden, golden_dir):
    """bj_submit_resized / bj_decode_batch_resized on a context of three devices (the one GPU three times on a one-GPU
    box): sub-batches dealt over the devices, jobs in the background, outputs exact."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    ngpu = torch.cuda.device_count()
    md = bj.Decoder(devices=list(range(ngpu)) if ngpu > 1 else [0, 0, 0])
    try:
        tw, th = 24, 24
        files, rois, scales, wants = _plan_case(bj, golden, golden_dir, tw, th)
        files, wants = files * 2, wants * 2
        rois, scales = np.concatenate([rois, rois]), np.concatenate([scales, scales])
        n = len(files)
        src, off, ln = _pack(bj, files)
        one = 26 + th * (tw * 3 + tw % 4)
        dst_off = np.arange(n, dtype=np.int64) * ((one + 15) // 16 * 16)
        md.set_option("sub_batch_bytes", 1 << 16)
        md.set_option("packed_outputs", 1)
        dsts = [bj.PinnedBuffer(int(dst_off[-1]) + one + 16) for _ in range(3)]
        status = md.decode_packed(src.array, off, ln, dsts[0].array, dst_off, bj.BJ_OUT_BMP, rois=rois, scales=scales, sizes=(tw, th))
        assert md.stat("decode_batch_sub_batches") > 8
        jobs = [md.submit_packed(src.array, off, ln, d.array, dst_off, bj.BJ_OUT_BMP, rois=rois, scales=scales, sizes=(tw, th)) for d in dsts[1:]]
        sts = [status] + [j.wait() for j in jobs]
        for st, d in zip(sts, dsts):
            for i, (w, s, o) in enumerate(zip(wants, st, dst_off)):
                if w is None:
                    assert s == bj.BJ_ERR_INVALID_JPEG
                else:
                    assert s == 0 and np.array_equal(d.array[o:o + one], crop_bytes(w, (0, 0, 0, 0), bj.BJ_OUT_BMP)), i
        for d in dsts:
            d.free()
        src.free()
    finally:
        md.close()
