"""The synchronisation pass at both of its CTA widths (option "sync_threads" = 128 or 256 sub-sequences per CTA),
against the oracle, bit for bit.  The automatic choice (0) is what every other test runs; here each width is pinned
for the golden set, the sub-sequence / slice / round grid, a config-2-shaped batch, restart images with 8 slices,
damaged and truncated scans and poisoned buffers."""
import hashlib

import numpy as np
import pytest

import jpeg_synth as js
import oracle_lib as ol
from test_gpu_parity import _load, _names

pytestmark = pytest.mark.gpu

WIDTHS = [128, 256]


@pytest.fixture(scope="module")
def dec():
    import pim_jpeg_decoder_b200 as bj
    d = bj.Decoder(0)
    yield d
    d.close()


@pytest.fixture
def width(dec, request):
    """Pins the CTA width for one test and puts every option it or the test sets back to automatic afterwards."""
    dec.set_option("sync_threads", request.param)
    yield request.param
    for name in ("sync_threads", "subseq_bits", "slices", "sync_rounds", "debug_poison"):
        dec.set_option(name, 0)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("width", WIDTHS, indirect=True)
def test_golden_set(dec, width, golden, golden_dir):
    import pim_jpeg_decoder_b200 as bj
    names = _names()
    files = [_load(golden, golden_dir, n) for n in names]
    for n, f in zip(names, files):
        coef, st = dec.stage_entropy(f)
        assert st == 0 and np.array_equal(coef, ol.Restated(f, 0).coef_zz), n
    outs, status = dec.decode(files, bj.BJ_OUT_BMP)
    for n, o, st in zip(names, outs, status):
        assert st == 0 and sha(o) == golden[golden[n]["expect"]]["bmp_sha256"], n


@pytest.mark.parametrize("width", WIDTHS, indirect=True)
@pytest.mark.parametrize("bits,slices,rounds", [(0, 0, 0), (128, 0, 0), (256, 2, 0), (1024, 0, 2), (4096, 4, 0), (512, 8, 0), (160, 0, 0), (0, 8, 0)])
def test_sync_layouts(dec, width, bits, slices, rounds, golden, golden_dir):
    """The grid of sub-sequence sizes, slice counts and fix-up rounds at each width (with width 128 a sub-sequence has
    at least 2 slices whatever "slices" says)."""
    dec.set_option("subseq_bits", bits)
    dec.set_option("slices", slices)
    dec.set_option("sync_rounds", rounds)
    for name in _names():
        data = _load(golden, golden_dir, name)
        coef, status = dec.stage_entropy(data)
        assert status == 0
        assert np.array_equal(coef, ol.Restated(data, 0).coef_zz), (name, bits, slices)


def _sampled_batch(dec, files, sample):
    """Decode `files` as one device-resident batch: its sub-sequence count and the outputs of the images in `sample`."""
    import pim_jpeg_decoder_b200 as bj
    b = bj.Batch(dec, files, bj.BJ_OUT_BMP)
    try:
        b.upload()
        b.decode()
        b.sync()
        assert all(s == 0 for s in b.status())
        outs = b.download(only=sample)
        return b.info().subsequences, [outs[i].copy() for i in sample]
    finally:
        b.destroy()


def test_config2_batch_both_widths(dec):
    """The bench's config-2 batch: 4096 images of 500x375 4:2:0 (64 distinct, cycled).  The automatic layout picks
    width 128 (one 128-wide CTA per image instead of one 256-wide one), and either width decodes the batch to the
    oracle's pixels."""
    unique = [js.synth_jpeg(500, 375, seed=i, subsampling=2) for i in range(64)]
    files = [unique[i % 64] for i in range(4096)]
    sample = list(range(0, 4096, 331)) + [4095]
    want = [ol.Restated(files[i], 0).bmp for i in sample]
    subs = {}
    try:
        for w in (0, 128, 256):
            dec.set_option("sync_threads", w)
            subs[w], outs = _sampled_batch(dec, files, sample)
            for i, o, r in zip(sample, outs, want):
                assert np.array_equal(o, r), (w, i)
    finally:
        dec.set_option("sync_threads", 0)
    assert subs[0] == subs[128] < subs[256]


def test_single_large_image_keeps_width_256(dec):
    """A single image larger than a CTA of sub-sequences (config 3 / 4 at batch 1) keeps the 256-wide layout."""
    for data in (js.synth_jpeg(3840, 2160, seed=1, subsampling=2, restart_blocks=8), js.synth_jpeg(3840, 2160, seed=2, subsampling=2, gray=True)):
        try:
            auto, _ = _sampled_batch(dec, [data], [])
            dec.set_option("sync_threads", 256)
            assert _sampled_batch(dec, [data], [])[0] == auto
        finally:
            dec.set_option("sync_threads", 0)


@pytest.mark.parametrize("width", WIDTHS, indirect=True)
def test_restart_images_with_8_slices(dec, width, golden, golden_dir):
    dec.set_option("slices", 8)
    files = [_load(golden, golden_dir, n) for n in _names() if "_ri" in n]
    files += [js.synth_jpeg(w, h, seed=w + ri, subsampling=sub, restart_blocks=ri) for w, h, sub, ri in ((640, 480, 2, 5), (333, 111, 0, 1), (512, 512, 1, 9))]
    assert len(files) >= 8
    for f in files:
        coef, st = dec.stage_entropy(f)
        assert st == 0 and np.array_equal(coef, ol.Restated(f, 0).coef_zz)


@pytest.mark.parametrize("width", WIDTHS, indirect=True)
@pytest.mark.parametrize("sub,bits,slices", [(2, 0, 0), (0, 256, 2), (2, 128, 8)])
def test_damaged_and_truncated_scans(dec, width, sub, bits, slices):
    import pim_jpeg_decoder_b200 as bj
    from test_huff_emu import _corrupt_scan
    rng = np.random.default_rng(900 + 10 * sub + slices + width)
    base = js.synth_jpeg(200, 152, seed=40 + sub, subsampling=sub)
    dec.set_option("subseq_bits", bits)
    dec.set_option("slices", slices)
    failed = 0
    for trial in range(16):
        bad, _ = _corrupt_scan(base, rng, 1 + trial % 8)
        r = ol.Restated(bad, 0)
        coef, status = dec.stage_entropy(bad)
        failed += r.huff_rc != 0
        assert (status != 0) == (r.huff_rc != 0), trial
        assert np.array_equal(coef, r.coef_zz), trial
    assert failed >= 2
    cut = base[: len(base) - 2 - 700] + b"\xFF\xD9"
    bads = [_corrupt_scan(base, rng, 3)[0] for _ in range(6)] + [cut]
    outs, status = dec.decode(bads + [base], bj.BJ_OUT_BMP)
    assert status[-2] == bj.BJ_ERR_CORRUPT_SCAN and status[-1] == 0
    for b, o in zip(bads + [base], outs):
        assert np.array_equal(o, ol.Restated(b, 0).bmp)


@pytest.mark.parametrize("width", WIDTHS, indirect=True)
def test_poisoned_buffers(dec, width, golden, golden_dir):
    import pim_jpeg_decoder_b200 as bj
    files = [_load(golden, golden_dir, n) for n in _names()]
    files += [js.synth_jpeg(640, 480, seed=70 + k, subsampling=k % 3, restart_blocks=(0, 5, 0, 9)[k % 4], gray=(k % 5 == 4)) for k in range(6)]
    dec.set_option("debug_poison", 1)
    for rep in range(2):
        outs, status = dec.decode(files, bj.BJ_OUT_BMP)
        assert all(s == 0 for s in status)
        for f, o in zip(files, outs):
            assert np.array_equal(o, ol.Restated(f, 0).bmp)


def test_other_widths_refused(dec):
    import pim_jpeg_decoder_b200 as bj
    for value in (64, 512, 1, -1, 192):
        with pytest.raises(bj.BjError) as e:
            dec.set_option("sync_threads", value)
        assert e.value.status == -1, value                       # BJ_ERR_ARG
    for value in (128, 256, 0):
        dec.set_option("sync_threads", value)
