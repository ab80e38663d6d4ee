"""TEST INFRASTRUCTURE: the libjpeg reconstruction (HCJ_FLAG_LIBJPEG, include/hcjpeg.h) restated independently of the library.

libjpeg-turbo's jidctint.c jpeg_idct_islow in int64 numpy on the oracle's dequantised blocks (with the C code's int
workspace and range-limit wrap), placed in decode_seq order like scaled_reference.ScaledDecode; jdsample.c's up-sampling
of every component's real plane; the colour conversion is the oracle's (jdcolor.c's formula)."""
import numpy as np

FLAG = 0x40  # HCJ_FLAG_LIBJPEG


def _islow_pass(c, sh):
    """One pass over c[0..7] (int64 arrays), descaled by `sh`: jidctint.c's even and odd parts."""
    c0, c1, c2, c3, c4, c5, c6, c7 = c
    z1 = (c2 + c6) * 4433
    t2, t3 = z1 - c6 * 15137, z1 + c2 * 6270
    t0, t1 = (c0 + c4) << 13, (c0 - c4) << 13
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    z5 = (c7 + c3 + c5 + c1) * 9633
    za, zb = (c7 + c1) * -7373, (c5 + c3) * -20995
    zc, zd = (c7 + c3) * -16069 + z5, (c5 + c1) * -3196 + z5
    p0, p1 = c7 * 2446 + za + zc, c5 * 16819 + zb + zd
    p2, p3 = c3 * 25172 + zb + zc, c1 * 12299 + za + zd
    o = [t10 + p3, t11 + p2, t12 + p1, t13 + p0, t13 - p0, t12 - p1, t11 - p2, t10 - p3]
    return [(v + (1 << (sh - 1))) >> sh for v in o]


def islow(dequant):
    """[N, 64] natural-order dequantised blocks -> [N, 8, 8] samples."""
    b = np.asarray(dequant, np.int64).reshape(-1, 8, 8)
    ws = np.stack(_islow_pass([b[:, r, :] for r in range(8)], 11), 1)  # columns: [N, row, col]
    ws = ws.astype(np.int32).astype(np.int64)  # the C int workspace: truncated to 32 bits
    v = np.stack(_islow_pass([ws[:, :, k] for k in range(8)], 18), 2)
    return np.clip(((v + 512) & 1023) - 512 + 128, 0, 255).astype(np.uint8)  # range_limit[v & RANGE_MASK]


def upsample(plane, rw, rh, hr, vr, W, H):
    """jdsample.c (do_fancy_upsampling) of the real rw x rh samples of `plane` by (hr, vr) = (h_max / h_c, v_max / v_c),
    cropped to W x H."""
    R = np.asarray(plane)[:rh, :rw].astype(np.int64)
    up = R[np.maximum(np.arange(rh) - 1, 0)]
    dn = R[np.minimum(np.arange(rh) + 1, rh - 1)]

    def horiz(x, bias_even, bias_odd, sh):  # out[2j] from the left neighbour, out[2j + 1] from the right one
        left = x[:, np.maximum(np.arange(rw) - 1, 0)]
        right = x[:, np.minimum(np.arange(rw) + 1, rw - 1)]
        out = np.empty((x.shape[0], 2 * rw), np.int64)
        out[:, 0::2] = (3 * x + left + bias_even) >> sh
        out[:, 1::2] = (3 * x + right + bias_odd) >> sh
        return out

    if (hr, vr) == (1, 1):
        out = R
    elif (hr, vr) == (2, 1) and rw > 2:  # h2v1_fancy_upsample
        out = horiz(R, 1, 2, 2)
    elif (hr, vr) == (2, 2) and rw > 2:  # h2v2_fancy_upsample
        out = np.empty((2 * rh, 2 * rw), np.int64)
        out[0::2] = horiz(3 * R + up, 8, 7, 4)
        out[1::2] = horiz(3 * R + dn, 8, 7, 4)
    elif (hr, vr) == (1, 2):  # h1v2_fancy_upsample
        out = np.empty((2 * rh, rw), np.int64)
        out[0::2] = (3 * R + up + 1) >> 2
        out[1::2] = (3 * R + dn + 2) >> 2
    else:  # h2v1 / h2v2_upsample of narrow planes, int_upsample
        out = np.repeat(np.repeat(R, vr, 0), hr, 1)
    assert out.shape[0] >= H and out.shape[1] >= W
    return out[:H, :W].astype(np.uint8)


class LibjpegDecode:
    """The HCJ_FLAG_LIBJPEG decode of one file: planes (padded), cropped (the model's crop rule), up-sampled components."""

    def __init__(self, orc, jpeg, **kw):
        dec = orc.decode(jpeg, want_blocks=True, **kw)
        self.orc, self.width, self.height, self.chroma, self.ncomp = orc, dec.width, dec.height, dec.chroma, dec.ncomp
        self.hs, self.vs = dec.hs, dec.vs
        self.planes = [np.zeros((h, w), np.uint8) for w, h in dec.decoded_size]
        pix = islow(dec.dequant)
        bi = 0
        for my in range(dec.mcus_high):  # decode_seq: MCU raster -> component -> v x h
            for mx in range(dec.mcus_wide):
                for c in range(dec.ncomp):
                    for by in range(dec.vs[c]):
                        for bx in range(dec.hs[c]):
                            y, x = (my * dec.vs[c] + by) * 8, (mx * dec.hs[c] + bx) * 8
                            self.planes[c][y:y + 8, x:x + 8] = pix[bi]
                            bi += 1
        assert bi == dec.nblocks
        self.cropped = [p[:h, :w] for p, (w, h) in zip(self.planes, dec.actual_size)]

    def ratios(self):
        mh, mv = max(self.hs), max(self.vs)
        return [(mh // h if mh % h == 0 else 0, mv // v if mv % v == 0 else 0) for h, v in zip(self.hs, self.vs)]

    def yuv444(self):
        """[3, H, W]: every component up-sampled from its real plane (HCJ_OUT_YUV444, Image.draft("YCbCr", size))."""
        W, H = self.width, self.height
        out = []
        for c, (hr, vr) in enumerate(self.ratios()[:3]):
            assert hr and vr, "non-integral sampling ratio"
            out.append(upsample(self.planes[c], -(-W // hr), -(-H // vr), hr, vr, W, H))
        return np.stack(out)

    def rgb(self):
        y, u, v = self.yuv444()
        return self.orc.ycbcr_to_rgb24(y, u, v)

    def yuv(self):
        assert self.chroma
        return b"".join(np.ascontiguousarray(p).tobytes() for p in self.cropped[:3])

    def planes_bytes(self):
        return b"".join(p.tobytes() for p in self.planes)

    def output(self, mode):
        """Bytes of HCJ_OUT_YUV (0) / PLANES (1) / RGB24 (2) / YUV444 (3)."""
        return {0: self.yuv, 1: self.planes_bytes, 2: lambda: self.rgb().tobytes(), 3: lambda: self.yuv444().tobytes()}[mode]()
