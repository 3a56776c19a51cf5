"""CPU tests of the region-of-interest sizing (no GPU needed): bj_roi_output_size gives the bytes of the RGB8 / BMP output
of a w x h crop, the whole image for {0,0,0,0} or no ROI, and 0 for a ROI that does not fit the image (sums taken in 64
bits) and for BJ_OUT_REF_MCUS, which has no crop."""
import ctypes as C
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _desc(name):
    import pim_jpeg_decoder_b200 as bj
    st, d = bj.parse_header(open(os.path.join(HERE, "golden", name), "rb").read())
    assert st == bj.BJ_OK
    return d


def _size(d, roi, fmt):
    import pim_jpeg_decoder_b200 as bj
    r = bj.Roi(*roi) if roi is not None else None
    return bj.lib().bj_roi_output_size(C.byref(d), C.byref(r) if r is not None else None, fmt)


def _want(w, h, fmt):
    import pim_jpeg_decoder_b200 as bj
    return w * h * 3 if fmt == bj.BJ_OUT_RGB8 else 26 + h * (w * 3 + w % 4)


@pytest.mark.parametrize("name", ["p420_50x37.jpg", "p444_33x17.jpg", "gray_40x24.jpg", "p420_1x1.jpg"])
def test_roi_output_size(name):
    import pim_jpeg_decoder_b200 as bj
    d = _desc(name)
    W, H = d.width, d.height
    for fmt in (bj.BJ_OUT_RGB8, bj.BJ_OUT_BMP):
        whole = bj.lib().bj_output_size(C.byref(d), fmt)
        assert _size(d, (0, 0, 0, 0), fmt) == _size(d, None, fmt) == _size(d, (0, 0, W, H), fmt) == whole == _want(W, H, fmt)
        assert bj.roi_output_size(d, None, fmt) == bj.roi_output_size(d, (0, 0, 0, 0), fmt) == whole
        for w in range(1, min(W, 8) + 1):                      # every w % 4, where the image is that wide
            for x in (0, W - w):
                for (y, h) in ((0, 1), (H - 1, 1), (0, H)):
                    assert _size(d, (x, y, w, h), fmt) == _want(w, h, fmt), (x, y, w, h)
                    assert bj.roi_output_size(d, (x, y, w, h), fmt) == _want(w, h, fmt)
        refused = [(0, 0, 0, 1), (0, 0, 1, 0), (1, 0, 0, 0), (0, 0, W + 1, 1), (0, 0, 1, H + 1), (W, 0, 1, 1), (0, H, 1, 1),
                   (1, 0, W, 1), (0, 1, 1, H),
                   # x + w and y + h wrap in 32 bits to a value that would fit
                   (0xFFFFFFFF, 0, 2, 1), (0, 0xFFFFFFFF, 1, 2), (1, 0, 0xFFFFFFFF, 1), (0, 1, 1, 0xFFFFFFFF),
                   (0x80000000, 0x80000000, 0x80000000, 0x80000000)]
        for roi in refused:
            assert _size(d, roi, fmt) == 0, roi
            assert bj.roi_output_size(d, roi, fmt) == 0, roi
    for roi in (None, (0, 0, 0, 0), (0, 0, 1, 1)):              # the reference's tile buffers have no crop
        assert _size(d, roi, bj.BJ_OUT_REF_MCUS) == 0
    assert bj.lib().bj_roi_output_size(None, None, bj.BJ_OUT_RGB8) == 0
    assert _size(d, (0, 0, 1, 1), 7) == 0


def test_roi_structure_layout():
    """sizeof(bj_roi) and its field offsets as the C compiler sees them == the ctypes mirror."""
    import subprocess
    import tempfile
    from pim_jpeg_decoder_b200 import _lib
    root = os.path.dirname(HERE)
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "b200jpeg.h"\n'
           'int main(void){printf("%zu %zu %zu\\n", sizeof(bj_roi), offsetof(bj_roi, w), offsetof(bj_roi, h));return 0;}\n')
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "t")
        subprocess.run(["gcc", "-I", os.path.join(root, "include"), "-o", exe, c], check=True)
        size, ow, oh = (int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert (size, ow, oh) == (C.sizeof(_lib.Roi), _lib.Roi.w.offset, _lib.Roi.h.offset) == (16, 8, 12)
