"""CPU tests of the reduced-size sizing (no GPU needed): bj_scaled_output_size gives the bytes of the RGB8 / BMP output of a
w x h crop of the image scaled by 1/s (ceil(W / s) x ceil(H / s)), all of the scaled image for {0,0,0,0} or no ROI, and 0
for a scale other than 1, 2, 4 and 8, for a ROI that does not fit the scaled image (sums taken in 64 bits) and for
BJ_OUT_REF_MCUS.  At s = 1 it is bj_roi_output_size."""
import ctypes as C
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden_descs():
    import json
    import pim_jpeg_decoder_b200 as bj
    golden = json.load(open(os.path.join(HERE, "golden", "golden.json")))
    out = []
    for name in sorted(golden):
        if golden[name].get("invalid"):
            continue
        st, d = bj.parse_header(open(os.path.join(HERE, "golden", golden[name]["file"]), "rb").read())
        assert st == bj.BJ_OK, name
        out.append((name, d))
    return out


def _size(d, roi, s, fmt):
    import pim_jpeg_decoder_b200 as bj
    r = bj.Roi(*roi) if roi is not None else None
    return bj.lib().bj_scaled_output_size(C.byref(d), C.byref(r) if r is not None else None, s, fmt)


def _roi_size(d, roi, fmt):
    import pim_jpeg_decoder_b200 as bj
    r = bj.Roi(*roi) if roi is not None else None
    return bj.lib().bj_roi_output_size(C.byref(d), C.byref(r) if r is not None else None, fmt)


def _want(w, h, fmt):
    import pim_jpeg_decoder_b200 as bj
    return w * h * 3 if fmt == bj.BJ_OUT_RGB8 else 26 + h * (w * 3 + w % 4)


def _rois(W, H):
    """ROIs of a W x H (scaled) image that fit: all of it, 1x1 at each corner, every w % 4 at both edges, a middle one."""
    out = [(0, 0, W, H), (0, 0, 1, 1), (W - 1, 0, 1, 1), (0, H - 1, 1, 1), (W - 1, H - 1, 1, 1), (W // 3, H // 3, W - W // 3, H - H // 3)]
    for w in range(1, min(W, 8) + 1):
        out += [(0, 0, w, H), (W - w, H - 1, w, 1)]
    return out


@pytest.mark.parametrize("fmt", [0, 1])
def test_scaled_output_size_golden(fmt):
    import pim_jpeg_decoder_b200 as bj
    for name, d in _golden_descs():
        W, H = d.width, d.height
        for s in (1, 2, 4, 8):
            Ws, Hs = -(-W // s), -(-H // s)
            whole = _want(Ws, Hs, fmt)
            assert _size(d, None, s, fmt) == _size(d, (0, 0, 0, 0), s, fmt) == _size(d, (0, 0, Ws, Hs), s, fmt) == whole, (name, s)
            assert bj.scaled_output_size(d, None, s, fmt) == bj.scaled_output_size(d, (0, 0, 0, 0), s, fmt) == whole
            for roi in _rois(Ws, Hs):
                want = _want(roi[2], roi[3], fmt)
                assert _size(d, roi, s, fmt) == want, (name, s, roi)
                assert bj.scaled_output_size(d, roi, s, fmt) == want
            # fits the full image but not the scaled one (from s = 2 on, where the scaled image is smaller)
            beyond = [(0, 0, Ws + 1, 1), (0, 0, 1, Hs + 1), (Ws, 0, 1, 1), (0, Hs, 1, 1), (1, 0, Ws, 1), (0, 1, 1, Hs)]
            for roi in beyond:
                assert _size(d, roi, s, fmt) == 0, (name, s, roi)
                if s > 1 and roi[0] + roi[2] <= W and roi[1] + roi[3] <= H:
                    assert _size(d, roi, 1, fmt) == _want(roi[2], roi[3], fmt)
            # empty, and x + w / y + h that wrap in 32 bits to a value that would fit
            refused = [(0, 0, 0, 1), (0, 0, 1, 0), (1, 0, 0, 0), (0xFFFFFFFF, 0, 2, 1), (0, 0xFFFFFFFF, 1, 2), (1, 0, 0xFFFFFFFF, 1),
                       (0, 1, 1, 0xFFFFFFFF), (0x80000000, 0x80000000, 0x80000000, 0x80000000)]
            for roi in refused:
                assert _size(d, roi, s, fmt) == 0, (name, s, roi)
        # scales the library does not have
        for s in (0, 3, 16, 255, -1, -2, 5, 6, 7):
            for roi in (None, (0, 0, 0, 0), (0, 0, 1, 1)):
                assert _size(d, roi, s, fmt) == 0, (name, s, roi)
                assert bj.scaled_output_size(d, roi, s, fmt) == 0


def test_scaled_output_size_is_roi_output_size_at_scale_1():
    import pim_jpeg_decoder_b200 as bj
    for name, d in _golden_descs():
        W, H = d.width, d.height
        for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP, bj.BJ_OUT_REF_MCUS, 7):
            for roi in [None, (0, 0, 0, 0), (0, 0, W + 1, 1), (0xFFFFFFFF, 0, 2, 1)] + _rois(W, H):
                assert _size(d, roi, 1, fmt) == _roi_size(d, roi, fmt), (name, fmt, roi)


def test_ref_mcus_and_bad_arguments():
    import pim_jpeg_decoder_b200 as bj
    for name, d in _golden_descs():
        for s in (1, 2, 4, 8):
            for roi in (None, (0, 0, 0, 0), (0, 0, 1, 1)):   # the reference's tile buffers have no crop and no scale
                assert _size(d, roi, s, bj.BJ_OUT_REF_MCUS) == 0, (name, s, roi)
            assert _size(d, None, s, 7) == 0
    assert bj.lib().bj_scaled_output_size(None, None, 2, bj.BJ_OUT_RGB8) == 0


def test_scale_edges_by_hand():
    """The scaled size is ceil(W / s) x ceil(H / s): 1x1 stays 1x1 at every scale, 17x17 is 9, 5 and 3 pixels square."""
    import pim_jpeg_decoder_b200 as bj
    descs = dict(_golden_descs())
    one, seventeen = descs["p420_1x1"], descs["p420_17x17"]
    for s in (1, 2, 4, 8):
        assert _size(one, None, s, bj.BJ_OUT_RGB8) == 3
        assert _size(one, None, s, bj.BJ_OUT_BMP) == 26 + 3 + 1
    for s, n in ((1, 17), (2, 9), (4, 5), (8, 3)):
        assert _size(seventeen, None, s, bj.BJ_OUT_RGB8) == n * n * 3
        assert _size(seventeen, (n - 1, n - 1, 1, 1), s, bj.BJ_OUT_RGB8) == 3
        assert _size(seventeen, (n, 0, 1, 1), s, bj.BJ_OUT_RGB8) == 0


def test_python_scale_table_refuses_what_is_not_a_scale():
    """Decoder's scales= argument reaches the library as one uint8 per image.  A value that is not a whole number in 1..8
    (258, -1, 2.7, ...) must not wrap or truncate to a scale the caller did not ask for: it goes as 0, which the library
    refuses per image.  Lists and arrays behave the same; one number stands for every image."""
    import numpy as np
    from pim_jpeg_decoder_b200.decoder import _scale_table
    assert _scale_table(None, 3) == (None, None)
    want = [0, 2, 4, 8, 3, 0, 0, 0, 1]
    for kind in (list, np.array):
        a, p = _scale_table(kind([258, 2, 4, 8, 3, 0, -1, 16, 1]), 9)
        assert a.dtype == np.uint8 and list(a) == want and p is not None
    a, _ = _scale_table(np.array([2.0, 2.7, 8.0, 1e9]), 4)
    assert list(a) == [2, 0, 8, 0]
    assert list(_scale_table(4, 3)[0]) == [4, 4, 4]
    assert list(_scale_table(2.5, 2)[0]) == [0, 0]
    assert list(_scale_table(np.array([1, 2], dtype=np.uint8), 2)[0]) == [1, 2]
    with pytest.raises(TypeError):
        _scale_table(["2"], 1)
    with pytest.raises(TypeError):
        _scale_table(np.array([True]), 1)
