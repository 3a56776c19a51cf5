"""CPU tests of fixed-size output (no GPU needed): bj_resized_output_size, the numpy expectation bilinear() worked out by
hand, resize_plan, and the Python validation of sizes=."""
import ctypes as C

import numpy as np
import pytest

from resize_ref import bilinear, taps
from test_gpu_scale import box_scale
from test_scale_abi import _golden_descs, _rois, _want


def _rsize(d, roi, s, size, fmt):
    import pim_jpeg_decoder_b200 as bj
    r = bj.Roi(*roi) if roi is not None else None
    z = bj.Size(*size) if size is not None else None
    return bj.lib().bj_resized_output_size(C.byref(d), C.byref(r) if r is not None else None, s, C.byref(z) if z is not None else None, fmt)


def _ssize(d, roi, s, fmt):
    import pim_jpeg_decoder_b200 as bj
    r = bj.Roi(*roi) if roi is not None else None
    return bj.lib().bj_scaled_output_size(C.byref(d), C.byref(r) if r is not None else None, s, fmt)


SIZES = [(1, 1), (224, 224), (13, 300), (300, 13), (5, 7), (65535, 1), (1, 65535), (16384, 16384)]
REFUSED = [(1, 0), (0, 1), (65536, 1), (1, 65536), (0, 65536), (0xFFFFFFFF, 0xFFFFFFFF), (65535, 65535), (16385, 16384)]


@pytest.mark.parametrize("fmt", [0, 1])
def test_resized_output_size_golden(fmt):
    """No size ({0,0} or NULL) is bj_scaled_output_size; a size gives the bytes of a w x h output whatever the crop; a
    refused size (one of w, h zero, either above 65535, w*h above the default max_image_pixels), a refused scale or ROI,
    and BJ_OUT_REF_MCUS give 0."""
    import pim_jpeg_decoder_b200 as bj
    for name, d in _golden_descs():
        for s in (1, 2, 4, 8):
            Ws, Hs = -(-d.width // s), -(-d.height // s)
            for roi in [None, (0, 0, 0, 0)] + _rois(Ws, Hs):
                want = _ssize(d, roi, s, fmt)
                assert want > 0
                assert _rsize(d, roi, s, None, fmt) == _rsize(d, roi, s, (0, 0), fmt) == want, (name, s, roi)
                assert bj.resized_output_size(d, roi, s, None, fmt) == bj.resized_output_size(d, roi, s, (0, 0), fmt) == want
                for z in SIZES + [(roi[2], roi[3]) if roi and roi[2] else (Ws, Hs)]:
                    assert _rsize(d, roi, s, z, fmt) == _want(z[0], z[1], fmt), (name, s, roi, z)
                    assert bj.resized_output_size(d, roi, s, z, fmt) == _want(z[0], z[1], fmt)
                for z in REFUSED:
                    assert _rsize(d, roi, s, z, fmt) == 0, (name, s, roi, z)
                    assert _rsize(d, roi, s, z, bj.BJ_OUT_REF_MCUS) == 0
            for roi in [(0, 0, Ws + 1, 1), (Ws, 0, 1, 1), (0, 0xFFFFFFFF, 1, 2)]:      # does not fit the scaled image
                for z in (None, (0, 0), (224, 224)):
                    assert _rsize(d, roi, s, z, fmt) == 0, (name, s, roi, z)
        for s in (0, 3, 16, -1):
            for z in (None, (0, 0), (1, 1)):
                assert _rsize(d, None, s, z, fmt) == 0
        for z in (None, (0, 0), (1, 1), (224, 224)):
            assert _rsize(d, None, 1, z, bj.BJ_OUT_REF_MCUS) == 0
            assert _rsize(d, None, 1, z, 7) == 0
    assert bj.lib().bj_resized_output_size(None, None, 1, None, bj.BJ_OUT_RGB8) == 0
    assert bj.lib().bj_resized_output_size(None, None, 1, C.byref(bj.Size(2, 2)), bj.BJ_OUT_RGB8) == 0


def test_bilinear_identity_half_and_centre():
    """At the source's own size the resize is the source; an exact 2x reduction of an even-sized source is its 2x2 box
    average; a 1 x 1 output is the centre sample (the mean of the two middle samples, rounded, where the size is even)."""
    rng = np.random.default_rng(5)
    for h, w in ((1, 1), (3, 5), (17, 9), (64, 48), (2, 30)):
        src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(bilinear(src, w, h), src)
    for h, w in ((2, 2), (4, 6), (30, 18), (224, 448)):
        src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(bilinear(src, w // 2, h // 2), box_scale(src, 2)), (h, w)
    odd = rng.integers(0, 256, (7, 5, 3), dtype=np.uint8)
    assert np.array_equal(bilinear(odd, 1, 1)[0, 0], odd[3, 2])
    even = rng.integers(0, 256, (1, 4, 3), dtype=np.uint8)
    assert np.array_equal(bilinear(even, 1, 1)[0, 0], (even[0, 1].astype(int) + even[0, 2] + 1) // 2)


def test_bilinear_by_hand():
    """A 3-row x 5-column source, S[y][x] = 10 y + 20 x in every channel, resized to 3 columns x 5 rows."""
    src = np.repeat((10 * np.arange(3)[:, None] + 20 * np.arange(5)[None, :]).astype(np.uint8)[..., None], 3, axis=2)
    # columns 5 -> 3: num = (2X + 1) 5 - 3 = 2, 12, 22 over den = 6
    assert [v.tolist() for v in taps(5, 3)] == [[0, 2, 3], [1, 3, 4], [85, 0, 170]]
    # rows 3 -> 5: num = max((2Y + 1) 3 - 5, 0) = 0, 4, 10, 16, 22 over den = 10; the last row's i1 is clamped to 2
    assert [v.tolist() for v in taps(3, 5)] == [[0, 0, 1, 1, 2], [1, 1, 2, 2, 2], [0, 102, 0, 153, 51]]
    out = bilinear(src, 3, 5)
    assert out.shape == (5, 3, 3)
    # (X, Y) = (0, 1): top = 171 * 0 + 85 * 20 = 1700, bot = 171 * 10 + 85 * 30 = 4260,
    # (154 * 1700 + 102 * 4260 + 32768) >> 16 = 729088 >> 16 = 11
    assert out[1, 0, 0] == 11
    # (1, 0): x0 = 2 with weight 256, y0 = 0 with weight 256: S[0][2] = 40
    assert out[0, 1, 0] == 40
    # (2, 4): x 3/4 at 170, y 2/2: top = 86 * 80 + 170 * 100 = 23880, (205 * 23880 + 51 * 23880 + 32768) >> 16 = 93
    assert out[4, 2, 0] == 93
    assert np.array_equal(out[..., 0], out[..., 1]) and np.array_equal(out[..., 0], out[..., 2])


def test_resize_plan():
    """The scale is the largest of 8, 4, 2, 1 that leaves the box at least as large as the target; the ROI is the box
    rounded outward onto the scaled image, so it covers the box and always fits - boxes at the right and bottom edges
    included - and the bilinear stage reduces by less than 2x below s = 8."""
    import pim_jpeg_decoder_b200 as bj
    assert bj.resize_plan(500, 375, None, (224, 224)) == (1, (0, 0, 500, 375))
    assert bj.resize_plan(500, 375, None, (100, 50)) == (4, (0, 0, 125, 94))
    assert bj.resize_plan(500, 375, None, (200, 50)) == (2, (0, 0, 250, 188))
    assert bj.resize_plan(4000, 3000, None, (224, 224)) == (8, (0, 0, 500, 375))
    assert bj.resize_plan(999, 999, (1, 3, 997, 995), (124, 124)) == (8, (0, 0, 125, 125))
    assert bj.resize_plan(500, 375, (10, 20, 30, 40), (224, 224)) == (1, (10, 20, 30, 40))
    rng = np.random.default_rng(11)
    for _ in range(3000):
        W, H = int(rng.integers(1, 5000)), int(rng.integers(1, 5000))
        w, h = int(rng.integers(1, W + 1)), int(rng.integers(1, H + 1))
        x, y = (W - w, H - h) if rng.random() < 0.3 else (int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1)))
        tw, th = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        s, (rx, ry, rw, rh) = bj.resize_plan(W, H, (x, y, w, h), (tw, th))
        assert s in (1, 2, 4, 8)
        assert (w >= s * tw and h >= s * th) or s == 1
        if s < 8:
            assert not (w >= 2 * s * tw and h >= 2 * s * th)
        assert rw >= 1 and rh >= 1 and rx + rw <= -(-W // s) and ry + rh <= -(-H // s)
        assert rx * s <= x and (rx + rw) * s >= x + w and ry * s <= y and (ry + rh) * s >= y + h
        assert (rx + rw - 1) * s < x + w and (ry + rh - 1) * s < y + h
    for bad in ((0, 0, 501, 1), (-1, 0, 5, 5), (0, 0, 0, 5)):
        with pytest.raises(ValueError):
            bj.resize_plan(500, 375, bad, (10, 10))
    with pytest.raises(ValueError):
        bj.resize_plan(500, 375, None, (0, 10))


def test_python_size_table_refuses_what_is_not_a_size():
    """sizes= reaches the library as one uint32 pair per image.  A pair that is not two whole numbers in 1..65535, nor
    (0, 0), must not wrap or truncate to a size the caller did not ask for: it goes as (1, 0), which the library refuses
    per image.  One pair stands for every image."""
    from pim_jpeg_decoder_b200.decoder import _size_table
    assert _size_table(None, 3) == (None, None)
    rows = [(224, 224), (0, 0), (1, 0), (0, 7), (65536, 2), (-1, 5), (2 ** 32 + 5, 5), (65535, 65535), (1, 1)]
    want = [[224, 224], [0, 0], [1, 0], [1, 0], [1, 0], [1, 0], [1, 0], [65535, 65535], [1, 1]]
    for kind in (list, np.array):
        a, p = _size_table(kind(rows), len(rows))
        assert a.dtype == np.uint32 and a.shape == (len(rows), 2) and a.tolist() == want and p is not None
    a, _ = _size_table(np.array([[2.0, 3.0], [2.5, 3.0], [1e9, 1.0]]), 3)
    assert a.tolist() == [[2, 3], [1, 0], [1, 0]]
    assert _size_table((224, 160), 3)[0].tolist() == [[224, 160]] * 3
    assert _size_table([7, 9], 2)[0].tolist() == [[7, 9]] * 2
    with pytest.raises(TypeError):
        _size_table([["2", "3"]], 1)
    with pytest.raises(TypeError):
        _size_table(np.array([[True, True]]), 1)
    with pytest.raises(ValueError):
        _size_table([(1, 2), (3, 4), (5, 6)], 2)
