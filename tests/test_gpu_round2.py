"""GPU parity tests, second set (pytest -m gpu): full-size shapes against the oracle, "every byte written exactly
once" under buffer poisoning, the device-side scan-end detection, the re-launch path of the Huffman fix-up, zero-copy
uploads, the multi-GPU context and the asynchronous pair.  Every comparison is BIT-EXACT; all calls go through the
C ABI (libb200jpeg.so)."""
import hashlib
import os

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    yield d
    d.close()


def _names(include_invalid=False):
    import json
    with open(os.path.join(HERE, "golden", "golden.json")) as f:
        g = json.load(f)
    return sorted(k for k, v in g.items() if include_invalid or not v.get("invalid"))


def _load(golden, golden_dir, name):
    return open(os.path.join(golden_dir, golden[name]["file"]), "rb").read()


def _pack(bj, files):
    """files -> (pinned source buffer, offsets, lengths)"""
    src = bj.PinnedBuffer(sum(len(f) for f in files) + 16)
    off, o = [], 0
    for f in files:
        src.array[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        off.append(o)
        o += len(f)
    return src, off, [len(f) for f in files]


def _out_layout(bj, files, fmt):
    sizes = []
    for f in files:
        st, d = bj.parse_header(f)
        sizes.append(bj.lib().bj_output_size(d, fmt) if st == 0 else 0)
    offs = np.concatenate([[0], np.cumsum([(s + 15) // 16 * 16 for s in sizes])]).astype(np.int64)
    return sizes, offs[:-1], int(offs[-1]) + 16


# ------------------------------------------------------------------ full-size shapes against the oracle (VERDICT r1, parity holes)

def test_config3_full_size_restart_parity_rule(dec):
    """BASELINE config 3 as stated: ONE 3840x2160 4:2:0 image with a restart interval of 8 MCUs.  Restart-parity rule
    (DESIGN.md section 4): the output equals the reference's decode of the restart-free twin; the reference's own decode
    of the DRI file differs."""
    import pim_jpeg_decoder_b200 as bj
    rgb = js.synth_rgb(3840, 2160, 0)
    with_ri = js.pil_jpeg(rgb, 90, 2, restart_blocks=8)
    twin = js.pil_jpeg(rgb, 90, 2)
    want = ol.Restated(twin, 0).bmp
    o1, s1 = dec.decode([with_ri], bj.BJ_OUT_BMP)              # alone: the single-image layout
    assert s1 == [0] and np.array_equal(o1[0], want)
    o2, s2 = dec.decode([twin, with_ri, twin], bj.BJ_OUT_BMP)
    assert s2 == [0, 0, 0]
    for o in o2:
        assert np.array_equal(o, want)
    assert not np.array_equal(ol.Restated(with_ri, 1).bmp, want)


@pytest.mark.parametrize("w,h,sub,gray", [(3840, 2160, 2, True), (1920, 1080, 2, False), (3840, 2160, 2, False)])
def test_full_size_members_of_the_mix_vs_oracle(dec, w, h, sub, gray):
    """4K gray (config 4), and the 1920x1080 / 3840x2160 4:2:0 members of the config-5 mix: BMP bytes == oracle."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(w, h, seed=w + h + gray, subsampling=sub, gray=gray)
    outs, status = dec.decode([data], bj.BJ_OUT_BMP)
    assert status == [0]
    assert np.array_equal(outs[0], ol.Restated(data, 0).bmp)


def test_config2_batch_of_4096_sampled_against_oracle(dec):
    """BASELINE config 2 at its full size: 4096 images of 500x375 4:2:0 in one call (256 unique, cycled); 64 images
    spread over the batch are compared with the oracle, and every copy of an image must equal its first copy."""
    import pim_jpeg_decoder_b200 as bj
    uniq = [js.synth_jpeg(500, 375, seed=9000 + k, subsampling=2) for k in range(256)]
    files = [uniq[i % 256] for i in range(4096)]
    src, off, ln = _pack(bj, files)
    sizes, dst_off, total = _out_layout(bj, files[:1], bj.BJ_OUT_BMP)
    size = sizes[0]
    pitch = (size + 15) // 16 * 16
    dst = bj.PinnedBuffer(pitch * 4096 + 16)
    dst.array[:] = 0x5A
    dst_off = np.arange(4096, dtype=np.int64) * pitch
    dec.set_option("packed_outputs", 1)
    try:
        status = dec.decode_packed(src.array, off, ln, dst.array, dst_off, bj.BJ_OUT_BMP)
        assert dec.stat("decode_batch_direct_uploads") == dec.stat("decode_batch_sub_batches") > 4   # zero-copy: the source is bj_host_alloc memory
    finally:
        dec.set_option("packed_outputs", 0)
    assert not status.any()
    view = dst.array[: pitch * 4096].reshape(4096, pitch)[:, :size]
    for k in range(256):
        assert (view[k::256] == view[k]).all(), k
    for i in range(0, 4096, 64):
        assert np.array_equal(view[i], ol.Restated(files[i], 0).bmp), i
    src.free()
    dst.free()


# ------------------------------------------------------------------ every byte written exactly once

def test_poisoned_buffers_golden_set_and_mixed_batch(dec, golden, golden_dir):
    """Option "debug_poison": coefficient, DC, stream and output buffers are filled with 0xA5 before every decode, so a
    byte the kernels fail to write (and that an earlier decode of the same data would have left in place) shows."""
    import pim_jpeg_decoder_b200 as bj
    names = _names()
    files = [_load(golden, golden_dir, n) for n in names]
    mixed = files + [js.synth_jpeg(640, 480, seed=50 + k, subsampling=k % 3, restart_blocks=(0, 5, 0, 9)[k % 4], gray=(k % 5 == 4)) for k in range(10)]
    dec.set_option("debug_poison", 1)
    try:
        for rep in range(2):                              # the second pass re-uses every buffer
            for fmt in (bj.BJ_OUT_BMP, bj.BJ_OUT_RGB8):
                outs, status = dec.decode(mixed, fmt)
                assert all(s == 0 for s in status)
                for f, o in zip(mixed, outs):
                    r = ol.Restated(f, 0)
                    if fmt == bj.BJ_OUT_BMP:
                        assert np.array_equal(o, r.bmp)
                    else:
                        assert np.array_equal(o.reshape(r.rgb.shape), r.rgb)
            for f in files[:12]:
                coef, st = dec.stage_entropy(f)
                assert st == 0 and np.array_equal(coef, ol.Restated(f, 0).coef_zz)
        for n, f in zip(names, files):
            o, st = dec.decode([f], bj.BJ_OUT_BMP)
            assert st == [0] and sha(o[0]) == golden[golden[n]["expect"]]["bmp_sha256"], n
    finally:
        dec.set_option("debug_poison", 0)


# ------------------------------------------------------------------ the scan's end is found on the device

def test_scan_end_found_on_device(dec):
    """The host reads headers only; k_unstuff finds where each scan ends.  Garbage behind EOI is
    ignored; a scan that ends in another marker, or not at all, makes the file invalid exactly like read_JPEG
    (src/jpeg_scanner.cpp:405-433) - per image, inside a batch whose other images decode normally."""
    import pim_jpeg_decoder_b200 as bj
    good = js.synth_jpeg(320, 240, seed=1, subsampling=2)
    good2 = js.synth_jpeg(200, 120, seed=2, subsampling=0, restart_blocks=3)
    rng = np.random.default_rng(5)
    trailing = good[:-2] + b"\xFF\xD9" + bytes(int(x) for x in rng.integers(0, 256, 5000)) + b"\xFF\xD9\xFF\xD8"
    no_eoi = good[:-2]
    ends_ff = good[:-2] + b"\xFF"
    other_marker = good[:len(good) // 2] + b"\xFF\xC4" + good[len(good) // 2:]
    early_eoi = good[:len(good) - 4000] + b"\xFF\xD9" + good[len(good) - 4000:]        # the reference stops at the first EOI
    files = [good, trailing, no_eoi, good2, ends_ff, other_marker, early_eoi, good]
    want_valid = [ol.Restated(f, 0).rc == 0 for f in files]
    assert want_valid == [True, True, False, True, False, False, True, True]
    sizes, offs, total = _out_layout(bj, [good] * len(files), bj.BJ_OUT_BMP)
    sizes2 = [bj.lib().bj_output_size(bj.parse_header(good2)[1], bj.BJ_OUT_BMP)]
    outs = [np.full(max(sizes[0], sizes2[0]), 0x11, dtype=np.uint8) for _ in files]
    for direct in (0, 1):                                  # staged and straight from pinned memory
        if direct:
            src, off, ln = _pack(bj, files)
            big = bj.PinnedBuffer(len(files) * (max(sizes[0], sizes2[0]) + 16))
            pitch = (max(sizes[0], sizes2[0]) + 15) // 16 * 16
            status = dec.decode_packed(src.array, off, ln, big.array, np.arange(len(files)) * pitch, bj.BJ_OUT_BMP)
            assert dec.stat("decode_batch_direct_uploads") >= 1
            got = [big.array[i * pitch: i * pitch + len(ol.Restated(f, 0).bmp)] if v else None for i, (f, v) in enumerate(zip(files, want_valid))]
        else:
            res, status = dec.decode(files, bj.BJ_OUT_BMP, outs=outs)
            got = [o[: len(ol.Restated(f, 0).bmp)] if v else None for o, f, v in zip(outs, files, want_valid)]
        for i, (f, v) in enumerate(zip(files, want_valid)):
            if not v:
                assert status[i] == bj.BJ_ERR_INVALID_JPEG, i
                continue
            r = ol.Restated(f, 0)
            assert status[i] == (0 if r.huff_rc == 0 else bj.BJ_ERR_CORRUPT_SCAN), i
            assert np.array_equal(got[i], r.bmp), i


def test_hostile_header_is_refused_alone(dec):
    """A tiny file that declares 65535 x 65535 pixels is valid for the parser; it gets BJ_ERR_UNSUPPORTED (the
    reference prints "Too high resolution", src/decoder_host.cpp:146-149) and the rest of the batch decodes."""
    import pim_jpeg_decoder_b200 as bj
    good = js.synth_jpeg(64, 48, seed=3, subsampling=2)
    i = good.find(b"\xFF\xC0")
    hostile = bytearray(good)
    hostile[i + 5:i + 9] = b"\xFF\xFF\xFF\xFF"
    hostile = bytes(hostile)
    assert bj.parse_header(hostile)[0] == 0
    outs, status = dec.decode([good, hostile, good], bj.BJ_OUT_RGB8,
                              outs=[np.zeros(64 * 48 * 3, np.uint8), np.zeros(16, np.uint8), np.zeros(64 * 48 * 3, np.uint8)])
    assert status == [0, bj.BJ_ERR_UNSUPPORTED, 0]
    r = ol.Restated(good, 0)
    assert np.array_equal(outs[0].reshape(r.rgb.shape), r.rgb) and np.array_equal(outs[2].reshape(r.rgb.shape), r.rgb)
    # decoded bytes cut sub-batches too
    many = [js.synth_jpeg(640, 480, seed=k, subsampling=2) for k in range(12)]
    dec.set_option("sub_batch_out_bytes", 2 << 20)
    try:
        outs, status = dec.decode(many, bj.BJ_OUT_BMP)
        assert dec.stat("decode_batch_sub_batches") >= 6
    finally:
        dec.set_option("sub_batch_out_bytes", 1 << 30)
    for f, o in zip(many, outs):
        assert np.array_equal(o, ol.Restated(f, 0).bmp)


# ------------------------------------------------------------------ the fix-up's re-launch path

def _flat_image(w, h):
    """Every data unit identical (one small pattern, constant DC): a periodic bit stream on which a decoder that starts
    at the wrong bit never falls into step - the speculative decode does not self-synchronise, the true state has to be
    handed down the whole chain."""
    comps = [(1, 1, 0, 0, 0)]
    a = np.zeros(((h + 7) // 8, (w + 7) // 8, 64), dtype=np.int64)
    a[..., 0] = 5
    a[..., 10] = 3
    a[..., 12] = -2
    return js.encode_from_coefs(w, h, comps, [a])


@pytest.mark.parametrize("rounds", [2, 3, 0])
def test_unconverged_first_write_pass_is_redone_from_k0_state(dec, rounds):
    """ADVICE r1 (medium): with too few blind fix-up rounds the first write pass runs on entry states that have not
    settled (here: a stream that needs one round per CTA, 9 CTAs at 128-bit sub-sequences) and may flag spurious
    failures; the re-launch must start from the state K0 left, so the image comes out clean and exact."""
    import pim_jpeg_decoder_b200 as bj
    data = _flat_image(1024, 1024)
    r = ol.Restated(data, 0)
    assert r.huff_rc == 0 and len(data) > 8 * 256 * 16
    dec.set_option("subseq_bits", 128)
    dec.set_option("sync_rounds", rounds)
    try:
        coef, status = dec.stage_entropy(data)
        assert status == 0
        assert np.array_equal(coef, r.coef_zz)
        outs, st = dec.decode([data, js.synth_jpeg(100, 80, seed=1)], bj.BJ_OUT_BMP)
        assert st == [0, 0] and np.array_equal(outs[0], r.bmp)
    finally:
        dec.set_option("subseq_bits", 0)
        dec.set_option("sync_rounds", 0)
    outs, st = dec.decode([data], bj.BJ_OUT_BMP)           # default layout
    assert st == [0] and np.array_equal(outs[0], r.bmp)


# ------------------------------------------------------------------ zero-copy upload, multi-GPU context, asynchronous pair

def test_registered_caller_memory_is_uploaded_directly(dec, golden, golden_dir):
    """bj_host_register: the caller's own (numpy) buffer is page-locked in place; files inside it go up without a staging
    copy.  Files scattered over ordinary memory are staged.  Same pixels either way."""
    import ctypes as C
    import pim_jpeg_decoder_b200 as bj
    names = _names()
    files = [_load(golden, golden_dir, n) for n in names]
    blob = np.zeros(sum(len(f) for f in files) + 4096, dtype=np.uint8)
    off, o = [], 0
    for f in files:
        blob[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        off.append(o)
        o += len(f)
    sizes, dst_off, total = _out_layout(bj, files, bj.BJ_OUT_BMP)
    dst = np.zeros(total, dtype=np.uint8)
    status = dec.decode_packed(blob, off, [len(f) for f in files], dst, dst_off, bj.BJ_OUT_BMP)
    assert dec.stat("decode_batch_direct_uploads") == 0 and not status.any()
    first = dst.copy()
    assert bj.lib().bj_host_register(blob.ctypes.data_as(C.c_void_p), blob.nbytes) == 0
    try:
        dst[:] = 0
        status = dec.decode_packed(blob, off, [len(f) for f in files], dst, dst_off, bj.BJ_OUT_BMP)
        assert dec.stat("decode_batch_direct_uploads") >= 1 and not status.any()
    finally:
        assert bj.lib().bj_host_unregister(blob.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(first, dst)
    for n, o2, s in zip(names, dst_off, sizes):
        assert sha(dst[int(o2):int(o2) + s]) == golden[golden[n]["expect"]]["bmp_sha256"], n


def test_multi_device_context_and_async_jobs(golden, golden_dir):
    """bj_create_multi deals sub-batches to its devices from one shared cursor (here: three contexts on the one GPU of
    the test box, which exercises the same host code as three GPUs); bj_submit / bj_wait run batches in the background,
    in order.  Outputs are the golden ones."""
    import torch
    import pim_jpeg_decoder_b200 as bj
    ngpu = torch.cuda.device_count()
    devices = list(range(ngpu)) if ngpu > 1 else [0, 0, 0]
    md = bj.Decoder(devices=devices)
    try:
        assert md.device_count == len(devices)
        names = _names(include_invalid=True) * 6
        files = [_load(golden, golden_dir, n) for n in names]
        src, off, ln = _pack(bj, files)
        sizes, dst_off, total = _out_layout(bj, files, bj.BJ_OUT_BMP)
        md.set_option("sub_batch_bytes", 1 << 16)
        md.set_option("packed_outputs", 1)
        dsts = [bj.PinnedBuffer(total) for _ in range(3)]
        status = md.decode_packed(src.array, off, ln, dsts[0].array, dst_off, bj.BJ_OUT_BMP)
        assert md.stat("decode_batch_sub_batches") > 8 and md.stat("devices") == len(devices)
        jobs = [md.submit_packed(src.array, off, ln, d.array, dst_off, bj.BJ_OUT_BMP) for d in dsts[1:]]
        sts = [status] + [j.wait() for j in jobs]
        for st, d in zip(sts, dsts):
            for n, s, o, size in zip(names, st, dst_off, sizes):
                if golden[n].get("invalid"):
                    assert s == bj.BJ_ERR_INVALID_JPEG
                else:
                    assert s == 0 and sha(d.array[int(o):int(o) + size]) == golden[golden[n]["expect"]]["bmp_sha256"], n
        # the DPU program on a multi-GPU context: chunks split over the devices
        r = ol.Restated(_load(golden, golden_dir, "ilsvrc_444"), 1)
        assert np.array_equal(md.exec_mcus(r.metadata, r.mcus_pre), r.mcus_post)
        for d in dsts:
            d.free()
        src.free()
    finally:
        md.close()


# ------------------------------------------------------------------ behind the unchanged scanner, in front of the unchanged BMP writer

def _desc_from_oracle_header(bj, data):
    """What a host that keeps read_JPEG does: one bj_image_desc per `Header`, field for field (INTEGRATION.md).  Here the
    parsed header comes from bj_peek_header; scan_off / scan_len are not used by bj_decode_batch_desc."""
    import ctypes as C
    d = bj.ImageDesc()
    buf = np.frombuffer(data, dtype=np.uint8)
    assert bj.lib().bj_peek_header(buf.ctypes.data_as(C.c_void_p), len(data), C.byref(d)) == 0
    d.scan_off = 0
    d.scan_len = 0
    return d


def test_ref_mcus_output_and_descriptor_input(dec, golden, golden_dir, tmp_path):
    """BJ_OUT_REF_MCUS = the reference's `mcus` buffers after pim.exec(): the WHOLE buffer (every chunk, the 128 fill of
    unused tiles included) equals the reference's post-exec buffer - hash from golden.json, made by the real reference -
    and the reference's own, unchanged write_BMP (through oracle/_ref/libref.so) turns it into the golden BMP.  Input
    three ways: the file (bj_decode_batch), descriptor + Header::huffman_data (BJ_SCAN_UNSTUFFED, what read_JPEG leaves),
    descriptor + raw scan bytes (BJ_SCAN_RAW, needed for files with restart markers)."""
    import pim_jpeg_decoder_b200 as bj
    names = _names()
    files = [_load(golden, golden_dir, n) for n in names]
    rs = [ol.Restated(f, 0) for f in files]
    # (1) files in, mcus out - one batch
    sizes = [r.mcus_post.nbytes for r in rs]
    outs = [np.zeros(s, dtype=np.uint8) for s in sizes]
    res, status = dec.decode(files, bj.BJ_OUT_REF_MCUS, outs=outs)
    assert all(s == 0 for s in status)
    for n, o, r in zip(names, outs, rs):
        got = o.view(np.int16).reshape(r.mcus_post.shape)
        assert np.array_equal(got, r.mcus_post), n
        if golden[n]["expect"] == n:                                   # (not a restart-parity twin case)
            assert sha(got) == golden[n]["mcus_post_sha256"], n
    # (2) descriptor + scan, both kinds
    descs = [_desc_from_oracle_header(bj, f) for f in files]
    pairs = [ol.unstuffed_scan(f) for f in files]
    ri0 = [i for i, d in enumerate(descs) if d.restart_interval == 0]
    o_clean, st_clean = dec.decode_desc([descs[i] for i in ri0], [pairs[i][0] for i in ri0], [bj.BJ_SCAN_UNSTUFFED] * len(ri0))
    assert st_clean == [0] * len(ri0)
    for i, o in zip(ri0, o_clean):
        assert np.array_equal(o.reshape(rs[i].mcus_post.shape), rs[i].mcus_post), names[i]
    o_raw, st_raw = dec.decode_desc(descs, [p[1] for p in pairs], None)
    assert st_raw == [0] * len(files)
    for n, o, r in zip(names, o_raw, rs):
        assert np.array_equal(o.reshape(r.mcus_post.shape), r.mcus_post), n
    # un-stuffed data of a file WITH restart markers cannot be split into segments any more: refused, per image
    with_ri = [i for i, d in enumerate(descs) if d.restart_interval != 0][:2]
    _, st_bad = dec.decode_desc([descs[i] for i in with_ri], [pairs[i][0] for i in with_ri], [bj.BJ_SCAN_UNSTUFFED] * len(with_ri))
    assert st_bad == [bj.BJ_ERR_UNSUPPORTED] * len(with_ri)
    # BMP bytes straight from a descriptor, too
    o_bmp, st_bmp = dec.decode_desc(descs, [p[1] for p in pairs], None, fmt=bj.BJ_OUT_BMP)
    for n, o in zip(names, o_bmp):
        assert sha(o) == golden[golden[n]["expect"]]["bmp_sha256"], n
    # (3) the reference's own write_BMP on our buffers: its inputs - metadata and post-exec buffer - are the ones it
    # turned into the golden BMP (golden.json holds the reference's hashes of both; for a restart-parity twin, the
    # twin's); where oracle/_ref/libref.so is built, write_BMP itself runs on them too
    for n, o, r in zip(names, o_raw, rs):
        e = golden[golden[n]["expect"]]
        assert sha(o) == e["mcus_post_sha256"] and sha(r.metadata[0]) == e["metadata_sha256"], n
    if ol.ref_available() and hasattr(ol.ref(), "ref_write_bmp"):
        for n, o, r in list(zip(names, o_raw, rs))[::3]:
            path = str(tmp_path / (n + ".bmp"))
            ol.ref_write_bmp(r.metadata[0], o, path)
            assert sha(np.fromfile(path, dtype=np.uint8)) == golden[golden[n]["expect"]]["bmp_sha256"], n
    # another MAX_MCU_PER_DPU: the same linear buffer, cut into other chunks
    dec.set_option("ref_max_mcu_per_dpu", 400)
    try:
        import ctypes as C
        i = names.index("ilsvrc_444")
        m = C.c_int(0)
        nbytes = bj.lib().bj_ref_mcus_size(C.byref(descs[i]), 400, C.byref(m))
        out = np.zeros(nbytes, dtype=np.uint8)
        _, st = dec.decode([files[i]], bj.BJ_OUT_REF_MCUS, outs=[out])
        assert st == [0] and m.value == (rs[i].nchunk * 100 + 399) // 400
        flat = rs[i].mcus_post.reshape(-1)
        got = out.view(np.int16)
        assert np.array_equal(got[:flat.size], flat) and (got[flat.size:] == 128).all()
    finally:
        dec.set_option("ref_max_mcu_per_dpu", 100)


# ------------------------------------------------------------------ edges: empty, ragged, extreme shapes, caller-made descriptors

def test_empty_ragged_and_extreme_inputs(dec):
    """Empty batch; a batch of nothing but rejects; zero-length and tiny inputs between good files; the widest and
    tallest shapes the 16-bit frame header allows in one dimension (one MCU row / one MCU column), every sampling."""
    import pim_jpeg_decoder_b200 as bj
    outs, status = dec.decode([], bj.BJ_OUT_BMP)
    assert outs == [] and status == []
    junk = [b"", b"\xFF", b"\xFF\xD8", b"\xFF\xD8\xFF\xD9", b"not a jpeg at all" * 10]
    outs, status = dec.decode(junk, bj.BJ_OUT_RGB8)
    assert status == [bj.BJ_ERR_INVALID_JPEG] * len(junk) and all(o is None for o in outs)
    good = js.synth_jpeg(37, 21, seed=8, subsampling=1)
    outs, status = dec.decode([junk[0], good, junk[3], good, junk[1]], bj.BJ_OUT_BMP)
    assert status == [bj.BJ_ERR_INVALID_JPEG, 0, bj.BJ_ERR_INVALID_JPEG, 0, bj.BJ_ERR_INVALID_JPEG]
    want = ol.Restated(good, 0).bmp
    assert np.array_equal(outs[1], want) and np.array_equal(outs[3], want)
    # (libjpeg-turbo writes at most 65500 pixels per side; the full 65535 comes from the coefficient-level encoder)
    comps = [(2, 2, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)]
    widest = js.encode_from_coefs(65535, 16, comps, js.random_coefs(comps, 65535, 16, seed=3, density=0.05), restart_interval=100)
    tallest = js.encode_from_coefs(8, 65535, [(1, 1, 0, 0, 0)], js.random_coefs([(1, 1, 0, 0, 0)], 8, 65535, seed=4, density=0.05))
    cases = [(widest, "65535x16 4:2:0 ri100"), (tallest, "8x65535 gray")]
    for w, h, sub, gray, ri in [(65500, 9, 2, False, 0), (9, 65500, 2, False, 0), (65500, 8, 0, False, 64), (16, 65500, 1, False, 0),
                                (65500, 1, 2, True, 0), (1, 65500, 2, True, 7), (8, 8, 2, False, 0), (1, 1, 0, False, 0)]:
        cases.append((js.synth_jpeg(w, h, seed=w + 3 * h, subsampling=sub, gray=gray, restart_blocks=ri), (w, h, sub, gray, ri)))
    for data, what in cases:
        w = h = what
        r = ol.Restated(data, 0)
        assert r.valid and r.huff_rc == 0, what
        outs, status = dec.decode([data, good], bj.BJ_OUT_BMP)
        assert status == [0, 0], (w, h)
        assert np.array_equal(outs[0], r.bmp), what
        rgb, st = dec.decode([data], bj.BJ_OUT_RGB8)
        assert st == [0] and np.array_equal(rgb[0].reshape(r.rgb.shape), r.rgb), (w, h)


def test_caller_made_descriptors_are_checked(dec, golden, golden_dir):
    """bj_decode_batch_desc / bj_stage_idct_color take descriptors the library did not parse: nonsense in them (zero
    components, sampling factors the tile sizes do not cover, table ids out of range, tables never set, a size that does
    not match the MCU counts) must come back as a status, never reach a kernel."""
    import ctypes as C
    import pim_jpeg_decoder_b200 as bj
    data = _load(golden, golden_dir, "p420_320x240")
    clean, raw = ol.unstuffed_scan(data)

    def fresh():
        return _desc_from_oracle_header(bj, data)

    def broken(**kw):
        d = fresh()
        for k, v in kw.items():
            if isinstance(v, tuple):
                getattr(d, k)[v[0]] = v[1]
            else:
                setattr(d, k, v)
        return d

    bad = [broken(ncomp=0), broken(ncomp=4), broken(hs=3), broken(vs=0), broken(comp_h=(1, 2)), broken(qt_id=(0, 7)), broken(dc_id=(2, 9)),
           broken(width=0), broken(mcu_w=5), broken(qt_set=(0, 0)), broken(ac_set=(0, 0)), broken(frame_type=0xC2), broken(scan_ncomp=1)]
    descs = [fresh()] + bad + [fresh()]
    outs, status = dec.decode_desc(descs, [raw] * len(descs), None, fmt=bj.BJ_OUT_BMP)
    assert status[0] == 0 and status[-1] == 0
    assert all(s in (bj.BJ_ERR_INVALID_JPEG, bj.BJ_ERR_UNSUPPORTED) for s in status[1:-1]), status
    want = ol.Restated(data, 0)
    assert np.array_equal(outs[0], want.bmp) and np.array_equal(outs[-1], want.bmp)
    for d in bad[:9]:
        out = np.zeros(16, dtype=np.uint8)
        rc = bj.lib().bj_stage_idct_color(dec.ctx, C.byref(d), want.coef_zz.ctypes.data_as(C.c_void_p), bj.BJ_OUT_RGB8, out.ctypes.data_as(C.c_void_p))
        assert rc == -1                                           # BJ_ERR_ARG
