"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every comparison is BIT-EXACT (tolerance 0): the
reference's path is all-integer (SURVEY.md section 0).  All calls go through the C ABI (libb200jpeg.so)."""
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


# ------------------------------------------------------------------ compat entry = the DPU program (K2+K3, ref layout)

@pytest.mark.parametrize("name", _names())
def test_exec_mcus_matches_reference_buffers(dec, name, golden, golden_dir):
    """bj_exec_mcus on the reference's own metadata/mcus buffers == pim.exec(): memcmp of the whole buffer."""
    r = ol.Restated(_load(golden, golden_dir, name), restart_mode=1)
    got = dec.exec_mcus(r.metadata, r.mcus_pre)
    assert np.array_equal(got, r.mcus_post)
    assert sha(got) == golden[name]["mcus_post_sha256"]          # the hash the REAL reference produced


@pytest.mark.parametrize("vs,hs,ncomp", [(1, 1, 3), (2, 1, 3), (1, 2, 3), (2, 2, 3), (1, 1, 1), (2, 2, 1), (0, 0, 0), (3, 1, 3)])
@pytest.mark.parametrize("full_range", [False, True])
def test_exec_mcus_random_buffers(dec, vs, hs, ncomp, full_range):
    """Random coefficient buffers incl. values that wrap 16 and 32 bits; idle DPUs (all-zero metadata) untouched."""
    from test_oracle import _random_exec_case
    rng = np.random.default_rng(vs * 100 + hs * 10 + ncomp + (1000 if full_range else 0))
    md, mcus = _random_exec_case(rng, vs, hs, max(ncomp, 1), 37, full_range)
    if ncomp == 0:
        md[:] = 0
    md[5] = 0                                                   # one idle DPU in the middle of the batch
    got = dec.exec_mcus(md, mcus)
    assert np.array_equal(got, ol.restate_exec_mcus(md, mcus))


# ------------------------------------------------------------------ stage tests on the fast layout

@pytest.mark.parametrize("name", _names())
def test_stage_idct_color_from_oracle_coefficients(dec, name, golden, golden_dir):
    import pim_jpeg_decoder_b200 as bj
    data = _load(golden, golden_dir, name)
    r = ol.Restated(data, restart_mode=0)
    st, d = bj.parse_header(data)
    assert st == 0
    bmp = dec.stage_idct_color(d, r.coef_zz, bj.BJ_OUT_BMP)
    assert np.array_equal(bmp, r.bmp)
    rgb = dec.stage_idct_color(d, r.coef_zz, bj.BJ_OUT_RGB8)
    assert np.array_equal(rgb.reshape(r.rgb.shape), r.rgb)


@pytest.mark.parametrize("name", _names())
def test_stage_entropy_matches_oracle_coefficients(dec, name, golden, golden_dir):
    data = _load(golden, golden_dir, name)
    r = ol.Restated(data, restart_mode=0)
    coef, status = dec.stage_entropy(data)
    assert status == 0
    assert np.array_equal(coef, r.coef_zz)


@pytest.mark.parametrize("bits", [128, 256, 1024, 4096])
def test_stage_entropy_subsequence_sizes(dec, bits, golden, golden_dir):
    dec.set_option("subseq_bits", bits)
    try:
        for name in ("ilsvrc_444", "p420_320x240", "enc_444_100x60_ri1", "p420_q100_64x64", "gray_ri3_64x48"):
            data = _load(golden, golden_dir, name)
            coef, status = dec.stage_entropy(data)
            assert status == 0
            assert np.array_equal(coef, ol.Restated(data, 0).coef_zz), (name, bits)
    finally:
        dec.set_option("subseq_bits", 0)


@pytest.mark.parametrize("slices,bits", [(1, 128), (2, 256), (8, 512), (8, 160), (4, 4096), (1, 4096), (2, 0), (8, 0)])
def test_stage_entropy_slices(dec, slices, bits, golden, golden_dir):
    """The write pass works on `slices` pieces of every sub-sequence of the synchronisation pass (entry states
    recorded while synchronising); 160 bits = 20 bytes is not divisible by 8 (the slice count is lowered)."""
    dec.set_option("slices", slices)
    dec.set_option("subseq_bits", bits)
    try:
        for name in ("ilsvrc_444", "p420_320x240", "enc_444_100x60_ri1", "p420_q100_64x64", "gray_ri3_64x48", "enc_420_100x60_ri4"):
            data = _load(golden, golden_dir, name)
            coef, status = dec.stage_entropy(data)
            assert status == 0
            assert np.array_equal(coef, ol.Restated(data, 0).coef_zz), (name, slices, bits)
    finally:
        dec.set_option("slices", 0)
        dec.set_option("subseq_bits", 0)


@pytest.mark.parametrize("bits,slices,rounds", [(0, 0, 0), (128, 0, 0), (256, 2, 0), (1024, 0, 2), (4096, 4, 0), (512, 8, 0), (160, 0, 0), (0, 8, 0)])
def test_stage_entropy_sync_layouts(dec, bits, slices, rounds, golden, golden_dir):
    """Every golden file under a grid of sub-sequence sizes, slice counts and fix-up rounds: the synchronisation pass
    decodes quarter by quarter (eighth by eighth with 8 slices), re-decodes stop where they meet the previous decode's
    trajectory, and the write pass' slice table is derived from the quarter records.  Same coefficients."""
    dec.set_option("subseq_bits", bits)
    dec.set_option("slices", slices)
    dec.set_option("sync_rounds", rounds)
    try:
        for name in _names():
            data = _load(golden, golden_dir, name)
            coef, status = dec.stage_entropy(data)
            assert status == 0
            assert np.array_equal(coef, ol.Restated(data, 0).coef_zz), (name, bits, slices)
    finally:
        dec.set_option("subseq_bits", 0)
        dec.set_option("slices", 0)
        dec.set_option("sync_rounds", 0)


def test_removed_kernel_options_refused(dec):
    """The persistent TMA IDCT kernel, the synchronisation pass without early stop, its pre-roll and its iteration cap
    are gone: their options are refused, and "sync_phased" = 1 and "sync_preroll_bits" = 0 name the one
    synchronisation pass that is left."""
    import pim_jpeg_decoder_b200 as bj
    for name, value in (("idct_tma", 0), ("idct_tma", 1), ("sync_phased", 0), ("sync_preroll_bits", 512),
                        ("debug_sync_iters", 1)):
        with pytest.raises(bj.BjError) as e:
            dec.set_option(name, value)
        assert e.value.status == -1, (name, value)                   # BJ_ERR_ARG
    dec.set_option("sync_phased", 1)
    dec.set_option("sync_preroll_bits", 0)


@pytest.mark.parametrize("rounds,bits", [(1, 128), (2, 256), (7, 128), (12, 1024)])
def test_stage_entropy_few_blind_rounds(dec, rounds, bits, golden, golden_dir):
    """Too few blind fix-up rounds for the chain to settle: the host's convergence check must add rounds (which walk
    along unsettled chains without a limit) until the result is the fixed point - same coefficients."""
    dec.set_option("sync_rounds", rounds)
    dec.set_option("subseq_bits", bits)
    try:
        for name in ("ilsvrc_444", "p420_320x240", "p420_q100_64x64", "gray_ri3_64x48", "enc_420_100x60_ri4"):
            data = _load(golden, golden_dir, name)
            coef, status = dec.stage_entropy(data)
            assert status == 0
            assert np.array_equal(coef, ol.Restated(data, 0).coef_zz), (name, rounds, bits)
    finally:
        dec.set_option("sync_rounds", 0)
        dec.set_option("subseq_bits", 0)


# ------------------------------------------------------------------ full path against the reference's BMPs

@pytest.mark.parametrize("name", _names())
def test_full_path_bmp_matches_reference_hash(dec, name, golden, golden_dir):
    """Compressed bytes -> BMP bytes; the SHA-256 must be the one the REAL reference produced (golden.json).
    For subsampled files with restart markers the restart-parity rule applies: `expect` names the restart-free twin."""
    import pim_jpeg_decoder_b200 as bj
    data = _load(golden, golden_dir, name)
    outs, status = dec.decode([data], bj.BJ_OUT_BMP)
    assert status == [0]
    assert sha(outs[0]) == golden[golden[name]["expect"]]["bmp_sha256"]


def test_full_path_batch_mixed(dec, golden, golden_dir):
    """All fixtures in ONE batch (mixed sizes, samplings, restart intervals, invalid files in between)."""
    import pim_jpeg_decoder_b200 as bj
    names = _names(include_invalid=True)
    files = [_load(golden, golden_dir, n) for n in names]
    for fmt in (bj.BJ_OUT_BMP, bj.BJ_OUT_RGB8):
        outs, status = dec.decode(files, fmt)
        for n, o, st, data in zip(names, outs, status, files):
            if golden[n].get("invalid"):
                assert st == bj.BJ_ERR_INVALID_JPEG and o is None
                continue
            assert st == 0, n
            r = ol.Restated(data, 0)
            if fmt == bj.BJ_OUT_BMP:
                assert sha(o) == golden[golden[n]["expect"]]["bmp_sha256"], n
            else:
                assert np.array_equal(o.reshape(r.rgb.shape), r.rgb), n


def test_full_path_sub_batching(dec, golden, golden_dir):
    """Force many sub-batches through the double-buffered one-call path."""
    import pim_jpeg_decoder_b200 as bj
    names = [n for n in _names()] * 3
    files = [_load(golden, golden_dir, n) for n in names]
    dec.set_option("sub_batch_bytes", 1 << 16)
    try:
        outs, status = dec.decode(files, bj.BJ_OUT_BMP)
        assert dec.stat("decode_batch_sub_batches") > 4
    finally:
        dec.set_option("sub_batch_bytes", 24 << 20)
    for n, o, st in zip(names, outs, status):
        assert st == 0 and sha(o) == golden[golden[n]["expect"]]["bmp_sha256"], n


@pytest.mark.parametrize("threads,direct", [(1, 0), (5, 0), (3, 1)])
def test_decode_packed_host_threads(dec, threads, direct, golden, golden_dir):
    """The batch-pipeline form of the one-call path (all files in one pinned buffer, outputs in another), with the
    host parse/pack work on 1 and on 5 worker threads, over 3 slots of small sub-batches."""
    import pim_jpeg_decoder_b200 as bj
    names = _names(include_invalid=True) * 4
    files = [_load(golden, golden_dir, n) for n in names]
    src = bj.PinnedBuffer(sum(len(f) for f in files))
    src_off, o = [], 0
    for f in files:
        src.array[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        src_off.append(o)
        o += len(f)
    sizes = []
    for f in files:
        st, d = bj.parse_header(f)
        sizes.append(bj.lib().bj_output_size(d, bj.BJ_OUT_BMP) if st == 0 else 0)
    dst_off = np.concatenate([[0], np.cumsum([(s + 15) // 16 * 16 for s in sizes])])[:-1]
    dst = bj.PinnedBuffer(int(dst_off[-1]) + sizes[-1] + 16)
    dst.array[:] = 0x5A
    dec.set_option("host_threads", threads)
    dec.set_option("sub_batch_bytes", 1 << 16)
    dec.set_option("packed_outputs", 1)
    dec.set_option("packed_inputs", direct)           # upload straight from the pinned source buffer
    try:
        status = dec.decode_packed(src.array, src_off, [len(f) for f in files], dst.array, dst_off, bj.BJ_OUT_BMP)
        assert dec.stat("host_threads") == threads and dec.stat("decode_batch_sub_batches") > 6
    finally:
        dec.set_option("sub_batch_bytes", 24 << 20)
        dec.set_option("packed_outputs", 0)
        dec.set_option("packed_inputs", 0)
        dec.set_option("host_threads", 4)
    for n, st, off, size in zip(names, status, dst_off, sizes):
        if golden[n].get("invalid"):
            assert st == bj.BJ_ERR_INVALID_JPEG
        else:
            assert st == 0 and sha(dst.array[int(off):int(off) + size]) == golden[golden[n]["expect"]]["bmp_sha256"], n
    src.free()
    dst.free()


@pytest.mark.parametrize("w,h,sub,gray,ri", [(500, 375, 2, False, 0), (375, 500, 2, False, 0), (640, 480, 0, False, 0),
                                             (640, 480, 1, False, 0), (224, 224, 2, True, 0), (1024, 768, 2, False, 0),
                                             (512, 384, 0, False, 8), (400, 300, 2, True, 5)])
def test_full_path_synthetic_vs_oracle(dec, w, h, sub, gray, ri):
    """The generator of SURVEY.md 8d; the oracle (restatement pinned to the reference) decodes the same bytes."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(w, h, seed=w * 7 + h, subsampling=sub, gray=gray, restart_blocks=ri)
    r = ol.Restated(data, 0)
    outs, status = dec.decode([data], bj.BJ_OUT_BMP)
    assert status == [0]
    assert np.array_equal(outs[0], r.bmp)


def test_large_mixed_batch_matches_single_image_decodes(dec):
    """A batch big enough for the throughput layout (long sub-sequences, several CTAs per image, 4 slices for the
    images with restart markers, 1 for the others - chosen per image): every image must come out exactly as when it
    is decoded alone (small-batch layout), and a sample is checked against the oracle."""
    import pim_jpeg_decoder_b200 as bj
    uniq = []
    for k in range(12):
        uniq.append(js.synth_jpeg(500, 375, seed=100 + k, subsampling=2))
        uniq.append(js.synth_jpeg(512, 384, seed=200 + k, subsampling=0, restart_blocks=4 + k))
        uniq.append(js.synth_jpeg(1280, 720, seed=300 + k, subsampling=1 if k % 2 else 0, gray=(k % 3 == 0)))
    files = (uniq * 5)[:170]
    assert sum(len(f) for f in files) > (16 << 20)
    dec.set_option("sub_batch_bytes", 64 << 20)          # one sub-batch
    try:
        outs, status = dec.decode(files, bj.BJ_OUT_BMP)
    finally:
        dec.set_option("sub_batch_bytes", 24 << 20)
    assert all(st == 0 for st in status)
    singles = {}
    for i, f in enumerate(files):
        key = i % len(uniq)
        if key not in singles:
            o, st = dec.decode([f], bj.BJ_OUT_BMP)
            assert st == [0]
            singles[key] = o[0]
        assert np.array_equal(outs[i], singles[key]), i
    for key in (0, 1, 2, 4, 17):
        assert np.array_equal(singles[key], ol.Restated(uniq[key], 0).bmp), key


def test_config3_restart_parity_rule(dec):
    """Config 3 shape (4:2:0 + restart interval 8), reduced size: GPU output == reference decode of the
    restart-free twin (SURVEY.md 8c); the reference's own decode of the DRI file differs (its restart test is
    wrong for subsampled files)."""
    import pim_jpeg_decoder_b200 as bj
    rgb = js.synth_rgb(960, 544, 0)
    with_ri = js.pil_jpeg(rgb, 90, 2, restart_blocks=8)
    twin = js.pil_jpeg(rgb, 90, 2)
    outs, status = dec.decode([with_ri, twin], bj.BJ_OUT_BMP)
    assert status == [0, 0]
    want = ol.Restated(twin, 0).bmp
    assert np.array_equal(outs[0], want) and np.array_equal(outs[1], want)
    assert not np.array_equal(ol.Restated(with_ri, 1).bmp, want)


def test_truncated_scan_matches_reference_partial_image(dec):
    """The reference ignores the Huffman failure and writes the partial image (src/decoder_host.cpp:181);
    undecoded units stay zero -> grey.  Same pixels here, plus a per-image status."""
    import pim_jpeg_decoder_b200 as bj
    data = js.synth_jpeg(320, 240, seed=9, subsampling=2)
    bad = data[: len(data) - 2 - 3000] + b"\xFF\xD9"
    r = ol.Restated(bad, 0)
    assert r.huff_rc != 0
    outs, status = dec.decode([bad, data], bj.BJ_OUT_BMP)
    assert status == [bj.BJ_ERR_CORRUPT_SCAN, 0]
    assert np.array_equal(outs[0], r.bmp)
    assert np.array_equal(outs[1], ol.Restated(data, 0).bmp)


@pytest.mark.parametrize("sub,bits,slices", [(2, 0, 0), (0, 256, 2), (1, 1024, 0), (2, 128, 8), (0, 4096, 4)])
def test_damaged_scans_stop_where_the_reference_stops(dec, sub, bits, slices):
    """Bits flipped inside the Huffman data (no restart markers): refused codes, over-long runs, bits running out.  The
    write pass decodes such a unit to its end and then again, exactly (huff_core.h: WriteCursor::redo_unit); the
    coefficients - which unit is the last one with values, and what the failing unit keeps - must be the reference's."""
    import pim_jpeg_decoder_b200 as bj
    from test_huff_emu import _corrupt_scan
    rng = np.random.default_rng(500 + 10 * sub + slices)
    base = js.synth_jpeg(200, 152, seed=40 + sub, subsampling=sub)
    dec.set_option("subseq_bits", bits)
    dec.set_option("slices", slices)
    failed = 0
    try:
        for trial in range(24):
            bad, _ = _corrupt_scan(base, rng, 1 + trial % 8)
            r = ol.Restated(bad, 0)
            coef, status = dec.stage_entropy(bad)
            failed += r.huff_rc != 0
            assert (status != 0) == (r.huff_rc != 0), trial
            assert np.array_equal(coef, r.coef_zz), trial
        bads = [_corrupt_scan(base, rng, 3)[0] for _ in range(8)]
        outs, status = dec.decode(bads + [base], bj.BJ_OUT_BMP)
        for b, o in zip(bads + [base], outs):
            assert np.array_equal(o, ol.Restated(b, 0).bmp)
    finally:
        dec.set_option("subseq_bits", 0)
        dec.set_option("slices", 0)
    assert failed >= 2


def test_random_images_sizes_and_damage(dec):
    """Random geometry / sampling / quality / restart interval / sub-sequence length / slice count, and for the files
    without restart markers a damaged twin: coefficients against the oracle, bit for bit."""
    from test_huff_emu import _corrupt_scan
    rng = np.random.default_rng(2024)
    try:
        for trial in range(48):
            w, h = int(rng.integers(8, 400)), int(rng.integers(8, 300))
            sub, gray = int(rng.integers(0, 3)), bool(rng.integers(0, 5) == 0)
            ri = int(rng.choice([0, 0, 0, 1, 3, 8]))
            dec.set_option("subseq_bits", int(rng.choice([0, 128, 160, 256, 1024, 4096])))
            dec.set_option("slices", int(rng.choice([0, 1, 2, 4, 8])))
            data = js.synth_jpeg(w, h, seed=trial, subsampling=sub, gray=gray, restart_blocks=ri)
            coef, status = dec.stage_entropy(data)
            assert status == 0 and np.array_equal(coef, ol.Restated(data, 0).coef_zz), trial
            if ri == 0:
                bad, _ = _corrupt_scan(data, rng, int(rng.integers(1, 6)))
                r = ol.Restated(bad, 0)
                if r.valid:
                    coef, status = dec.stage_entropy(bad)
                    assert (status != 0) == (r.huff_rc != 0), trial
                    assert np.array_equal(coef, r.coef_zz), trial
    finally:
        dec.set_option("subseq_bits", 0)
        dec.set_option("slices", 0)


def test_large_image_properties(dec):
    """Full-size config-4 shapes (3840x2160 4:4:4 and gray, no restart markers): checked through size-independent
    properties - the image decodes identically alone, inside a batch, and at another sub-sequence size - plus an
    oracle comparison on the 4:4:4 one (the C oracle takes ~1 s for it)."""
    import pim_jpeg_decoder_b200 as bj
    a = js.synth_jpeg(3840, 2160, seed=1, subsampling=0)
    g = js.synth_jpeg(3840, 2160, seed=2, gray=True)
    small = js.synth_jpeg(100, 80, seed=3)
    o1, s1 = dec.decode([a], bj.BJ_OUT_RGB8)
    o2, s2 = dec.decode([small, g, a, small], bj.BJ_OUT_RGB8)
    assert s1 == [0] and s2 == [0, 0, 0, 0]
    assert np.array_equal(o1[0], o2[2]) and np.array_equal(o2[0], o2[3])
    dec.set_option("subseq_bits", 2048)
    try:
        o3, s3 = dec.decode([g, a], bj.BJ_OUT_RGB8)
    finally:
        dec.set_option("subseq_bits", 0)
    assert np.array_equal(o3[0], o2[1]) and np.array_equal(o3[1], o1[0])
    r = ol.Restated(a, 0)
    assert np.array_equal(o1[0].reshape(r.rgb.shape), r.rgb)


def test_decode_files_cli_behaviour(dec, tmp_path, golden, golden_dir):
    """`./bin/decoder a.jpg b.jpg` writes a.bmp / b.bmp beside the inputs (src/decoder_host.cpp:328-330)."""
    import shutil
    import pim_jpeg_decoder_b200 as bj
    names = ["ilsvrc_444", "p420_50x37", "bad_not_jpeg"]
    paths = []
    for n in names:
        p = str(tmp_path / golden[n]["file"])
        shutil.copy(os.path.join(golden_dir, golden[n]["file"]), p)
        paths.append(p)
    res = bj.decode_files(paths, decoder=dec)
    assert res[paths[2]] == bj.BJ_ERR_INVALID_JPEG and not os.path.exists(paths[2][:-4] + ".bmp")
    for n, p in zip(names[:2], paths[:2]):
        assert sha(np.fromfile(p[:-4] + ".bmp", dtype=np.uint8)) == golden[n]["bmp_sha256"]
