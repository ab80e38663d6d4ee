"""Reference for the RGB24 encoder input (hcj_encode_rgb_batch / hcj_rgb_to_yuv): a literal int64 restatement of the stated
forward conversion (not in the reference model; include/hcjpeg.h, DESIGN.md 5), composed with the oracle's
Planar_444.convert_to_420 / _422 (subsample_hv2 / subsample_h2)."""
import numpy as np


def rgb24_to_ycbcr_exact(rgb):
    """The formula's values, before any cast, of an (..., 3) uint8 array: int64 (Y, Cb, Cr).  JFIF full range, libjpeg's
    jccolor.c in 16-bit fixed point, arithmetic shifts."""
    rgb = np.asarray(rgb, np.uint8)
    assert rgb.shape[-1] == 3
    r, g, b = (rgb[..., k].astype(np.int64) for k in range(3))
    y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16
    cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16
    cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16
    return y, cb, cr


def rgb24_to_ycbcr(rgb):
    """(Y, Cb, Cr) uint8 planes of the leading shape.  Every value of the formula lies in [0, 255]
    (test_forward_formula_over_the_cube), so the cast is exact."""
    return tuple(p.astype(np.uint8) for p in rgb24_to_ycbcr_exact(rgb))


def rgb24_to_frame(orc, rgb, width, height, chroma=420):
    """The planar frame (bytes, Frame.input layout) that hcj_encode_rgb_batch encodes for RGB24 `rgb` (bytes or an
    (height, width, 3) uint8 array): the forward conversion, then the oracle's Planar_444.convert_to_420 / _422 of the
    rounded chroma planes (an odd last column / row dropped); 444 keeps the planes, 400 keeps Y only."""
    a = np.frombuffer(rgb, np.uint8) if isinstance(rgb, (bytes, bytearray)) else np.asarray(rgb, np.uint8)
    y, cb, cr = rgb24_to_ycbcr(a.reshape(height, width, 3))
    if chroma == 400:
        return y.tobytes()
    if chroma == 420:
        cb, cr = orc.subsample_hv2(cb), orc.subsample_hv2(cr)
    elif chroma == 422:
        cb, cr = orc.subsample_h2(cb), orc.subsample_h2(cr)
    return y.tobytes() + cb.tobytes() + cr.tobytes()
