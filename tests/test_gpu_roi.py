"""GPU tests of region-of-interest decode (pytest -m gpu): the output of an image with a ROI is, byte for byte, what the
same format holds for the crop of the full decode - the oracle's (oracle_lib.Restated(data).rgb, pinned to the
reference's hashes by test_oracle.py) - for RGB8 and BMP, on every output path of the C ABI."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    yield d
    d.close()


def _golden_names(golden):
    return sorted(k for k, v in golden.items() if not v.get("invalid"))


def _load(golden, golden_dir, name):
    return open(os.path.join(golden_dir, golden[name]["file"]), "rb").read()


def crop_bytes(rgb, roi, fmt):
    """What the format holds for the crop roi = (x, y, w, h) of the top-down RGB image rgb [H, W, 3] (all zero: whole)."""
    import pim_jpeg_decoder_b200 as bj
    x, y, w, h = (int(v) for v in roi)
    if w == 0 and h == 0 and x == 0 and y == 0:
        h, w = rgb.shape[:2]
    c = rgb[y:y + h, x:x + w]
    if fmt == bj.BJ_OUT_RGB8:
        return np.ascontiguousarray(c).reshape(-1)
    pad = w % 4
    hdr = np.zeros(26, dtype=np.uint8)
    hdr[0:2] = (ord("B"), ord("M"))
    hdr[2:6] = np.frombuffer(np.uint32(26 + h * (w * 3 + pad)).tobytes(), dtype=np.uint8)
    hdr[10], hdr[14], hdr[22], hdr[24] = 0x1A, 12, 1, 24
    hdr[18:20] = (w & 0xFF, w >> 8)
    hdr[20:22] = (h & 0xFF, h >> 8)
    rows = np.zeros((h, w * 3 + pad), dtype=np.uint8)
    rows[:, :w * 3] = c[::-1, :, ::-1].reshape(h, w * 3)
    return np.concatenate([hdr, rows.reshape(-1)])


def rois_for(W, H):
    """The ROIs every image is cropped to: whole (explicit and {0,0,0,0}), 1x1 at each corner, offsets that are not
    multiples of 8 or 16, one inside a single MCU, one ending in the partial edge MCU, widths of each w % 4."""
    cands = [(0, 0, W, H), (0, 0, 0, 0), (0, 0, 1, 1), (W - 1, 0, 1, 1), (0, H - 1, 1, 1), (W - 1, H - 1, 1, 1),
             (3, 5, W - 3, H - 5), (13, 9, min(W - 13, 21), min(H - 9, 11)), (9, 10, 3, 2), (17, 18, 5, 4),
             (W - 11, H - 7, 11, 7), (W // 2, H // 3, W - W // 2, H - H // 3)]
    cands += [(1, 2, w, 3) for w in (4, 5, 6, 7)] + [(7, 1, w, H - 1) for w in (8, 9, 10, 11)]
    out = []
    for r in cands:
        x, y, w, h = r
        if r == (0, 0, 0, 0) or (x >= 0 and y >= 0 and w > 0 and h > 0 and x + w <= W and y + h <= H):
            if r not in out:
                out.append(r)
    return out


def _expected_rgb(golden, golden_dir, name):
    """The full image the crop is taken from: for a subsampled file with restart markers its restart-free twin
    (DESIGN.md section 4), which golden.json names in `expect`."""
    return ol.Restated(_load(golden, golden_dir, golden[name]["expect"]), 0).rgb


def test_crop_of_whole_image_is_the_reference_bmp(golden, golden_dir):
    """The expectation itself: the BMP bytes crop_bytes builds for the whole image are the golden BMP."""
    import pim_jpeg_decoder_b200 as bj
    for n in _golden_names(golden):
        r = ol.Restated(_load(golden, golden_dir, golden[n]["expect"]), 0)
        assert hashlib.sha256(crop_bytes(r.rgb, (0, 0, 0, 0), bj.BJ_OUT_BMP).tobytes()).hexdigest() == golden[golden[n]["expect"]]["bmp_sha256"], n


@pytest.mark.parametrize("fmt", [0, 1])
def test_golden_set_times_rois(dec, fmt, golden, golden_dir):
    """Every golden image under every ROI of rois_for, all in one batch."""
    import pim_jpeg_decoder_b200 as bj
    files, rois, wants = [], [], []
    for n in _golden_names(golden):
        data = _load(golden, golden_dir, n)
        rgb = _expected_rgb(golden, golden_dir, n)
        for r in rois_for(rgb.shape[1], rgb.shape[0]):
            files.append(data)
            rois.append(r)
            wants.append((n, r, crop_bytes(rgb, r, fmt)))
    outs, status = dec.decode(files, fmt, rois=np.array(rois, dtype=np.uint32))
    for (n, r, want), o, st in zip(wants, outs, status):
        assert st == 0 and o is not None and o.size == want.size and np.array_equal(o, want), (n, r)


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("sub,gray", [(2, False), (0, False), (0, True)])
def test_large_images_rois_across_tiles(dec, w, h, sub, gray):
    """4:2:0, 4:4:4 and gray at 1920x1080 and 3840x2160: pixel rows span several K2/K3 tiles (512 / 512 / 1536 px per
    tile), and the ROIs straddle tile boundaries."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(w, h, seed=w + h + sub + 7 * gray, subsampling=sub, gray=gray)
    rgb = ol.Restated(data, 0).rgb
    rng = np.random.default_rng(w + sub + gray)
    rois = [(0, 0, 0, 0), (500, 17, 30, 40), (1000, 300, 600, 21), (1530, 1, 13, h - 2), (511, 0, 2, h), (w - 1025, h - 33, 1025, 33),
            (1535, 700, 1, 1), (0, 0, w, 1)]
    for _ in range(6):
        rw, rh = int(rng.integers(1, w)), int(rng.integers(1, h))
        rois.append((int(rng.integers(0, w - rw + 1)), int(rng.integers(0, h - rh + 1)), rw, rh))
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode([data] * len(rois), fmt, rois=rois)
        for r, o, st in zip(rois, outs, status):
            assert st == 0 and np.array_equal(o, crop_bytes(rgb, r, fmt)), (fmt, r)


def test_restart_images_crop_of_the_twin(dec):
    """A subsampled image with restart markers gives the crop of its restart-free twin (restart-parity rule)."""
    import pim_jpeg_decoder_b200 as bj
    rgb0 = js.synth_rgb(960, 544, 3)
    with_ri = js.pil_jpeg(rgb0, 90, 2, restart_blocks=8)
    twin_rgb = ol.Restated(js.pil_jpeg(rgb0, 90, 2), 0).rgb
    rois = [(0, 0, 0, 0), (17, 33, 400, 300), (959, 543, 1, 1), (100, 0, 513, 544)]
    outs, status = dec.decode([with_ri] * len(rois), bj.BJ_OUT_BMP, rois=rois)
    for r, o, st in zip(rois, outs, status):
        assert st == 0 and np.array_equal(o, crop_bytes(twin_rgb, r, bj.BJ_OUT_BMP)), r


def test_damaged_and_truncated_scans_crop_of_the_partial_image(dec):
    """A damaged or truncated scan gives the crop of the partial image the reference writes (and BJ_ERR_CORRUPT_SCAN)."""
    import pim_jpeg_decoder_b200 as bj
    from test_huff_emu import _corrupt_scan
    data = js.synth_jpeg(320, 240, seed=9, subsampling=2)
    truncated = data[: len(data) - 2 - 3000] + b"\xFF\xD9"
    rng = np.random.default_rng(61)
    bads = [truncated] + [_corrupt_scan(js.synth_jpeg(200, 152, seed=40 + k, subsampling=k % 3), rng, 3)[0] for k in range(6)]
    rois = [(5, 200, 300, 40), (0, 0, 0, 0), (33, 7, 101, 99), (150, 100, 50, 52), (1, 1, 198, 150), (64, 64, 17, 3), (0, 151, 200, 1)]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(bads, fmt, rois=rois)
        failed = 0
        for b, r, o, st in zip(bads, rois, outs, status):
            ro = ol.Restated(b, 0)
            failed += ro.huff_rc != 0
            assert st == (bj.BJ_ERR_CORRUPT_SCAN if ro.huff_rc != 0 else 0)
            assert np.array_equal(o, crop_bytes(ro.rgb, r, fmt)), r
        assert failed >= 1


def test_mixed_batch_and_refusals(dec, golden, golden_dir):
    """ROI and whole-image entries, an invalid file and a ROI that does not fit (per-image BJ_ERR_ARG) in one batch: the
    others are exact.  rois=None is byte-identical to bj_decode_batch; BJ_OUT_REF_MCUS with rois is refused."""
    import pim_jpeg_decoder_b200 as bj
    good = _load(golden, golden_dir, "p420_320x240")
    other = _load(golden, golden_dir, "p444_33x17")
    bad = _load(golden, golden_dir, "bad_not_jpeg")
    rgb, rgb2 = ol.Restated(good, 0).rgb, ol.Restated(other, 0).rgb
    files = [good, bad, good, other, good, other, good]
    rois = [(10, 20, 30, 40), (0, 0, 5, 5), (0, 0, 0, 0), (0, 0, 34, 17), (300, 0, 21, 1), (1, 1, 32, 16), (0x7FFFFFFF, 0, 0x80000002, 1)]
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        outs, status = dec.decode(files, fmt, rois=rois)
        assert status == [0, bj.BJ_ERR_INVALID_JPEG, 0, bj.BJ_ERR_ARG, bj.BJ_ERR_ARG, 0, bj.BJ_ERR_ARG]
        for i in (0, 2):
            assert np.array_equal(outs[i], crop_bytes(rgb, rois[i], fmt)), i
        assert np.array_equal(outs[5], crop_bytes(rgb2, rois[5], fmt))
        assert outs[1] is None and outs[3] is None and outs[4] is None and outs[6] is None
        # rois=None through the _roi entry == bj_decode_batch, byte for byte and status for status
        whole, st_whole = dec.decode(files, fmt)
        _, ptrs, lens = bj.decoder._file_arrays(files)
        ref = [np.full(o.size, 0x5A, dtype=np.uint8) if o is not None else None for o in whole]
        optrs = (C.c_void_p * len(files))(*[o.ctypes.data if o is not None else None for o in ref])
        st = (C.c_int * len(files))()
        assert bj.lib().bj_decode_batch(dec.ctx, ptrs, lens, len(files), fmt, optrs, st) == 0
        assert list(st) == st_whole
        for a, b in zip(whole, ref):
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
    # BJ_OUT_REF_MCUS has no crop
    _, ptrs, lens = bj.decoder._file_arrays([good])
    roi = (bj.Roi * 1)(bj.Roi(0, 0, 0, 0))
    buf = np.zeros(1 << 20, dtype=np.uint8)
    optrs = (C.c_void_p * 1)(buf.ctypes.data)
    st = (C.c_int * 1)()
    assert bj.lib().bj_decode_batch_roi(dec.ctx, ptrs, lens, roi, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == bj.BJ_ERR_ARG
    h = C.c_void_p()
    assert bj.lib().bj_batch_create_roi(dec.ctx, ptrs, lens, roi, 1, bj.BJ_OUT_REF_MCUS, C.byref(h)) == bj.BJ_ERR_ARG and not h.value
    assert bj.lib().bj_submit_roi(dec.ctx, ptrs, lens, roi, 1, bj.BJ_OUT_REF_MCUS, optrs, st, C.byref(h)) == bj.BJ_ERR_ARG
    assert bj.lib().bj_decode_batch_roi(dec.ctx, ptrs, lens, None, 1, bj.BJ_OUT_REF_MCUS, optrs, st) == 0 and st[0] == 0


def test_poisoned_buffers(dec, golden, golden_dir):
    """debug_poison = 1: every byte returned for a ROI was written by the decode."""
    import pim_jpeg_decoder_b200 as bj
    names = _golden_names(golden)
    files, rois, wants = [], [], []
    for k, n in enumerate(names):
        rgb = _expected_rgb(golden, golden_dir, n)
        rs = rois_for(rgb.shape[1], rgb.shape[0])
        for r in (rs[k % len(rs)], rs[(3 * k + 1) % len(rs)]):
            files.append(_load(golden, golden_dir, n))
            rois.append(r)
            wants.append(rgb)
    dec.set_option("debug_poison", 1)
    try:
        for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
            outs, status = dec.decode(files, fmt, rois=rois)
            for r, rgb, o, st in zip(rois, wants, outs, status):
                assert st == 0 and np.array_equal(o, crop_bytes(rgb, r, fmt)), r
    finally:
        dec.set_option("debug_poison", 0)


def test_sub_batches_are_cut_by_cropped_bytes(dec):
    """The one-call path cuts sub-batches by the bytes of the crops: 12 images of 320x240 whose 100x100 RGB crops
    (30000 B) go two to a sub-batch of 64 KiB, where the whole images (230400 B) would take one each."""
    import pim_jpeg_decoder_b200 as bj
    uniq = [js.synth_jpeg(320, 240, seed=70 + k, subsampling=k % 3) for k in range(4)]
    files = [uniq[i % 4] for i in range(12)]
    rgbs = [ol.Restated(f, 0).rgb for f in uniq]
    rois = [(7 * i, 3 * i, 100, 100) for i in range(12)]
    dec.set_option("sub_batch_out_bytes", 1 << 16)
    try:
        outs, status = dec.decode(files, bj.BJ_OUT_RGB8, rois=rois)
        assert dec.stat("decode_batch_sub_batches") == 6
        assert dec.stat("decode_batch_d2h_bytes") == 12 * 30000
        for i, (o, st) in enumerate(zip(outs, status)):
            assert st == 0 and np.array_equal(o, crop_bytes(rgbs[i % 4], rois[i], bj.BJ_OUT_RGB8)), i
        outs, status = dec.decode(files, bj.BJ_OUT_BMP, rois=rois)
        assert dec.stat("decode_batch_sub_batches") == 6
        for i, (o, st) in enumerate(zip(outs, status)):
            assert st == 0 and np.array_equal(o, crop_bytes(rgbs[i % 4], rois[i], bj.BJ_OUT_BMP)), i
        dec.decode(files, bj.BJ_OUT_RGB8)
        assert dec.stat("decode_batch_sub_batches") == 12
    finally:
        dec.set_option("sub_batch_out_bytes", 1 << 30)


def _pack(bj, files):
    src = bj.PinnedBuffer(sum(len(f) for f in files) + 16)
    off, o = [], 0
    for f in files:
        src.array[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        off.append(o)
        o += len(f)
    return src, np.array(off, dtype=np.int64), [len(f) for f in files]


def _roi_layout(bj, files, rois, fmt):
    sizes = []
    for f, r in zip(files, rois):
        st, d = bj.parse_header(f)
        sizes.append(bj.roi_output_size(d, r, fmt) if st == 0 else 0)
    offs = np.concatenate([[0], np.cumsum([(s + 15) // 16 * 16 for s in sizes])]).astype(np.int64)
    return sizes, offs[:-1], int(offs[-1]) + 16


def _mixed_case(golden, golden_dir):
    names = sorted(golden)
    files, rois, wants = [], [], []
    for k, n in enumerate(names * 3):
        data = _load(golden, golden_dir, n)
        files.append(data)
        if golden[n].get("invalid"):
            rois.append((0, 0, 1, 1))
            wants.append(None)
            continue
        rgb = _expected_rgb(golden, golden_dir, n)
        rs = rois_for(rgb.shape[1], rgb.shape[0])
        rois.append(rs[(5 * k) % len(rs)])
        wants.append(rgb)
    return files, np.array(rois, dtype=np.uint32), wants


def test_packed_outputs(dec, golden, golden_dir):
    """decode_packed with an (n, 4) ROI array, outputs laid out by bj_roi_output_size in one pinned buffer, copied out
    in runs (packed_outputs = 1), over many small sub-batches."""
    import pim_jpeg_decoder_b200 as bj
    files, rois, wants = _mixed_case(golden, golden_dir)
    src, off, ln = _pack(bj, files)
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        sizes, dst_off, total = _roi_layout(bj, files, rois, fmt)
        dst = bj.PinnedBuffer(total)
        dec.set_option("packed_outputs", 1)
        dec.set_option("sub_batch_bytes", 1 << 16)
        try:
            status = dec.decode_packed(src.array, off, ln, dst.array, dst_off, fmt, rois=rois)
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


def _peek(bj, data):
    d = bj.ImageDesc()
    buf = np.frombuffer(data, dtype=np.uint8)
    return d if bj.lib().bj_peek_header(buf.ctypes.data_as(C.c_void_p), len(data), C.byref(d)) == 0 else None


class _DeviceBytes:
    """A device pointer the library returned, as an array torch can read (CUDA array interface)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def test_staged_batch_offsets_device_output_and_info(dec, golden, golden_dir):
    """Batch(..., rois=): offsets and sizes are the crops', device_output reports the cropped bytes, info() counts the
    cropped output bytes and the full images' pixels, and the download is exact."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    files, rois, wants = _mixed_case(golden, golden_dir)
    peeked = [_peek(bj, f) for f in files]                # what the batch sees: headers only (a scan's end is found on the device)
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        b = bj.Batch(dec, files, fmt, rois=rois)
        try:
            parsed = [st == 0 for st in b.parse_status]
            assert parsed == [d is not None for d in peeked]
            assert b.sizes == [bj.roi_output_size(d, r, fmt) if d is not None else 0 for d, r in zip(peeked, rois)]
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


def test_submit_roi_on_a_multi_device_context(golden, golden_dir):
    """bj_submit_roi / bj_decode_batch_roi on a context of three devices (the one GPU three times on a one-GPU box):
    sub-batches dealt over the devices, jobs in the background, outputs exact."""
    import pim_jpeg_decoder_b200 as bj
    import torch
    ngpu = torch.cuda.device_count()
    devices = list(range(ngpu)) if ngpu > 1 else [0, 0, 0]
    md = bj.Decoder(devices=devices)
    try:
        files, rois, wants = _mixed_case(golden, golden_dir)
        files, wants = files * 2, wants * 2
        rois = np.concatenate([rois, rois])
        src, off, ln = _pack(bj, files)
        sizes, dst_off, total = _roi_layout(bj, files, rois, bj.BJ_OUT_BMP)
        md.set_option("sub_batch_bytes", 1 << 16)
        md.set_option("packed_outputs", 1)
        dsts = [bj.PinnedBuffer(total) for _ in range(3)]
        status = md.decode_packed(src.array, off, ln, dsts[0].array, dst_off, bj.BJ_OUT_BMP, rois=rois)
        assert md.stat("decode_batch_sub_batches") > 8
        jobs = [md.submit_packed(src.array, off, ln, d.array, dst_off, bj.BJ_OUT_BMP, rois=rois) for d in dsts[1:]]
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
