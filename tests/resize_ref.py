"""The expectation of fixed-size output (include/b200jpeg.h, bj_decode_batch_resized): the integer bilinear sample with
half-pixel centres of the scaled crop, which is itself a box average of the oracle's full decode (test_gpu_scale)."""
import numpy as np


def taps(n_src, n_dst):
    """(i0, i1, f) for every output index 0..n_dst-1, in 64-bit integers: the source indices and the weight of i1."""
    X = np.arange(n_dst, dtype=np.int64)
    num = np.maximum((2 * X + 1) * n_src - n_dst, 0)
    den = 2 * n_dst
    i0 = num // den
    return i0, np.minimum(i0 + 1, n_src - 1), ((num % den) * 256) // den


def bilinear(src, w, h):
    """src [ch, cw, 3] uint8 -> [h, w, 3] uint8: the library's bilinear resize, in numpy."""
    ch, cw = src.shape[:2]
    x0, x1, fx = taps(cw, w)
    y0, y1, fy = taps(ch, h)
    S = src.astype(np.int64)
    fx = fx[None, :, None]
    top = (256 - fx) * S[y0][:, x0] + fx * S[y0][:, x1]
    bot = (256 - fx) * S[y1][:, x0] + fx * S[y1][:, x1]
    fy = fy[:, None, None]
    return (((256 - fy) * top + fy * bot + 32768) >> 16).astype(np.uint8)


def crop(rgb, roi):
    """The crop (x, y, w, h) of rgb [H, W, 3]; all zero: all of it."""
    x, y, w, h = (int(v) for v in roi)
    if (x, y, w, h) == (0, 0, 0, 0):
        return rgb
    return rgb[y:y + h, x:x + w]
