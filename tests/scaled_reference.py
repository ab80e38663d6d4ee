"""TEST INFRASTRUCTURE: the scaled decode (HCJ_FLAG_SCALE_*, include/hcjpeg.h) restated independently of the library.

libjpeg's reduced inverse DCTs (jidctred.c: jpeg_idct_4x4 / _2x2 / _1x1) in exact int64 arithmetic on the oracle's
dequantised blocks, placed in decode_seq order into scaled padded planes and cropped by the geometry rule of the
header.  RGB24 / YUV444 compose the result with the oracle's own up-sampling and colour conversion, as
rgb_reference.py composes its formula with the oracle."""
import numpy as np

CB, P1 = 13, 2  # CONST_BITS, PASS1_BITS
SCALES = (2, 4, 8)
FLAG = {1: 0, 2: 0x10, 4: 0x20, 8: 0x30}  # HCJ_FLAG_SCALE_1_2 / _1_4 / _1_8


def _ds(x, n):  # DESCALE: round, arithmetic shift
    return (x + (1 << (n - 1))) >> n


def _out(x):
    return np.clip(x + 128, 0, 255).astype(np.uint8)


def idct_4x4(b):
    """s = 2.  b: [N, 8, 8] natural-order dequantised blocks [block, row, col] -> [N, 4, 4]."""
    def p(c0, c1, c2, c3, c5, c6, c7, sh):
        t0 = c0 << (CB + 1)
        t2 = c2 * 15137 - c6 * 6270
        t10, t12 = t0 + t2, t0 - t2
        o0 = -c7 * 1730 + c5 * 11893 - c3 * 17799 + c1 * 8697
        o2 = -c7 * 4176 - c5 * 4926 + c3 * 7373 + c1 * 20995
        return [_ds(t10 + o2, sh), _ds(t12 + o0, sh), _ds(t12 - o0, sh), _ds(t10 - o2, sh)]

    b = np.asarray(b).astype(np.int64)
    ws = np.stack(p(*(b[:, r, :] for r in (0, 1, 2, 3, 5, 6, 7)), CB - P1 + 1), 1)  # columns first: [N, 4, 8]
    return _out(np.stack(p(*(ws[:, :, c] for c in (0, 1, 2, 3, 5, 6, 7)), CB + P1 + 3 + 1), 2))


def idct_2x2(b):
    """s = 4 -> [N, 2, 2]."""
    def p(c0, c1, c3, c5, c7, sh):
        t10 = c0 << (CB + 2)
        t0 = -c7 * 5906 + c5 * 6967 - c3 * 10426 + c1 * 29692
        return [_ds(t10 + t0, sh), _ds(t10 - t0, sh)]

    b = np.asarray(b).astype(np.int64)
    ws = np.stack(p(*(b[:, r, :] for r in (0, 1, 3, 5, 7)), CB - P1 + 2), 1)  # [N, 2, 8]
    return _out(np.stack(p(*(ws[:, :, c] for c in (0, 1, 3, 5, 7)), CB + P1 + 3 + 2), 2))


def idct_1x1(b):
    """s = 8 -> [N, 1, 1]."""
    b = np.asarray(b)
    return _out(_ds(b[:, 0, 0].astype(np.int64), 3)).reshape(-1, 1, 1)


def reduced(dequant, s):
    """[N, 64] natural-order dequantised blocks -> [N, k, k] samples, k = 8 / s."""
    b = np.asarray(dequant).reshape(-1, 8, 8)
    return {2: idct_4x4, 4: idct_2x2, 8: idct_1x1}[s](b)


ZIGZAG_INVERSE = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                           21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                           60, 61, 54, 47, 55, 62, 63])


def dequantise(coefs_zz, qt_zz):
    """int16 zig-zag blocks (DC absolute) x a zig-zag quant table -> [N, 64] natural-order int64."""
    c = np.asarray(coefs_zz, np.int64).reshape(-1, 64)
    d = np.zeros_like(c)
    d[:, ZIGZAG_INVERSE] = c * np.asarray(qt_zz, np.int64)
    return d


def geometry(width, height, hs, vs, decoded_size, s):
    """The frame_info fields the scale changes: (W', H', decoded [(w, h)], actual [(w, h)], chroma)."""
    mh, mv = max(hs), max(vs)
    W, H = -(-width // s), -(-height // s)
    decoded = [(w // s, h // s) for w, h in decoded_size]
    actual = [(W * a // mh, H * b // mv) for a, b in zip(hs, vs)]
    chroma = 0
    if len(hs) >= 3 and actual[1] == actual[2]:
        (yw, yh), (uw, uh) = actual[0], actual[1]
        chroma = 420 if (yw // 2, yh // 2) == (uw, uh) else 422 if (yw // 2, yh) == (uw, uh) else 444 if (yw, yh) == (uw, uh) else 0
    return W, H, decoded, actual, chroma


class ScaledDecode:
    """The scaled decode of one file (s = 1: the oracle's decode): planes (padded), cropped, width, height, chroma."""

    def __init__(self, orc, jpeg, s, **kw):
        dec = orc.decode(jpeg, want_blocks=s > 1, **kw)
        self.orc, self.s = orc, s
        k = 8 // s
        self.width, self.height, dsz, asz, self.chroma = geometry(dec.width, dec.height, dec.hs, dec.vs, dec.decoded_size, s)
        if s == 1:  # the oracle's own decode
            self.planes = [p.copy() for p in dec.planes]
        else:
            self.planes = [np.zeros((h, w), np.uint8) for w, h in dsz]
            pix = reduced(dec.dequant, s)
            bi = 0
            for my in range(dec.mcus_high):  # decode_seq: MCU raster -> component -> v x h
                for mx in range(dec.mcus_wide):
                    for c in range(dec.ncomp):
                        for by in range(dec.vs[c]):
                            for bx in range(dec.hs[c]):
                                y, x = (my * dec.vs[c] + by) * k, (mx * dec.hs[c] + bx) * k
                                self.planes[c][y:y + k, x:x + k] = pix[bi]
                                bi += 1
            assert bi == dec.nblocks
        self.cropped = [p[:h, :w] for p, (w, h) in zip(self.planes, asz)]

    def yuv(self):
        assert self.chroma
        return b"".join(np.ascontiguousarray(p).tobytes() for p in self.cropped[:3])

    def planes_bytes(self):
        return b"".join(p.tobytes() for p in self.planes)

    def yuv444(self):
        """Planar_444 of the cropped frame into a fresh (zero) 4:4:4 frame (HCJ_OUT_YUV444)."""
        y, u, v = self.orc.upsample_to_444([np.ascontiguousarray(p) for p in self.cropped[:3]], self.chroma)
        h, w = y.shape
        out = np.zeros((3, h, w), np.uint8)
        for i, p in enumerate((y, u, v)):
            out[i, : min(h, p.shape[0]), : min(w, p.shape[1])] = p[:h, :w]
        return out

    def rgb(self):
        y, u, v = self.yuv444()
        return self.orc.ycbcr_to_rgb24(y, u, v)

    def output(self, mode):
        """Bytes of HCJ_OUT_YUV (0) / PLANES (1) / RGB24 (2) / YUV444 (3)."""
        return {0: self.yuv, 1: self.planes_bytes, 2: lambda: self.rgb().tobytes(), 3: lambda: self.yuv444().tobytes()}[mode]()
