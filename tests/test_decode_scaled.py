"""Scaled decode (HCJ_FLAG_SCALE_1_2 / _1_4 / _1_8): libjpeg's reduced IDCTs on the device, for every decode entry point.

The semantics are pinned twice: the int64 restatement in scaled_reference.py equals Pillow's Image.draft (libjpeg-turbo)
exactly, and the device equals that restatement byte for byte in every output mode."""
import ctypes as C
import hashlib
import io
import os
import subprocess

import numpy as np
import pytest

import scaled_reference as sr
import synth

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "video-coding_b200", "csrc")
_EMUL_OUT = os.path.join(_HERE, "_build", "libemul_scaled.so")
_emul = None

# (chroma, quality, w, h, restart_interval): the geometries of test_gpu_decode.CASES
CASES = [
    (420, 75, 256, 192, 0), (420, 75, 256, 192, 8), (422, 50, 200, 120, 0), (444, 95, 160, 96, 0),
    (420, 10, 333, 77, 0), (420, 95, 52, 44, 0), (444, 75, 17, 9, 0), (420, 75, 16, 16, 1),
    (422, 75, 130, 70, 3), (444, 100, 64, 64, 2), (420, 1, 96, 80, 0), (420, 75, 8, 8, 0),
]
MODES = {"yuv": 0, "planes": 1, "rgb": 2, "yuv444": 3}


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def emul():
    """tests/emul/scaled.cpp built with g++ (rebuilt when a source is newer)."""
    global _emul
    if _emul is None:
        srcs = [os.path.join(_HERE, "emul", "scaled.cpp")] + [os.path.join(_CSRC, f) for f in ("hcj_device.cuh", "hcj_common.h")]
        if not (os.path.exists(_EMUL_OUT) and all(os.path.getmtime(_EMUL_OUT) >= os.path.getmtime(s) for s in srcs)):
            os.makedirs(os.path.dirname(_EMUL_OUT), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I", _CSRC, "-x", "c++",
                                   srcs[0], "-o", _EMUL_OUT])
        L = C.CDLL(_EMUL_OUT)
        L.emu_reconstruct_scaled.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _emul = L
    return _emul


def emul_scaled(coefs, qt, s, wide=-1):
    c = np.ascontiguousarray(coefs, np.int16).reshape(-1, 64)
    q = np.ascontiguousarray(qt, np.uint16)
    k = 8 // s
    out = np.zeros((c.shape[0], k, k), np.uint8)
    emul().emu_reconstruct_scaled(c.ctypes.data, c.shape[0], q.ctypes.data, k, wide, out.ctypes.data)
    return out


def _rgb_image(seed, w, h, saturated=False):
    rng = np.random.default_rng(seed)
    if saturated:
        return (rng.random((h, w, 3)) < 0.5).astype(np.uint8) * 255
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) * 3) % 256], -1)
    return np.clip(base + rng.normal(0, 25, (h, w, 3)), 0, 255).astype(np.uint8)


def _pil_jpeg(img, **kw):
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(img).save(buf, "JPEG", **kw)
    return buf.getvalue()


def _draft(jpg, mode, s):
    from PIL import Image

    im = Image.open(io.BytesIO(jpg))
    w, h = im.size
    im.draft(mode, (max(1, w // s), max(1, h // s)))
    assert im.size == (-(-w // s), -(-h // s))  # libjpeg's output size is the geometry rule's W' x H'
    return np.asarray(im)


def _pillow_cases():
    """(name, jpeg, channels pinned): 4:4:4 and grayscale whole, luma of 4:2:0 / 4:2:2; Pillow's and the oracle's encoder."""
    from oracle import pyoracle as orc

    out = []
    for (w, h) in ((203, 117), (131, 97)):
        for q in (50, 75, 95, 100):
            img = _rgb_image(w * q, w, h)
            out.append(("pil444 %dx%d q%d" % (w, h, q), _pil_jpeg(img, quality=q, subsampling=0), "ycc"))
            out.append(("pilL %dx%d q%d" % (w, h, q), _pil_jpeg(img[:, :, 1], quality=q), "L"))
            out.append(("pil420 %dx%d q%d" % (w, h, q), _pil_jpeg(img, quality=q, subsampling=2), "Y"))
            out.append(("pil422 %dx%d q%d" % (w, h, q), _pil_jpeg(img, quality=q, subsampling=1), "Y"))
        sat = _rgb_image(7 + w, w, h, saturated=True)
        out.append(("pil444 saturated %dx%d q100" % (w, h), _pil_jpeg(sat, quality=100, subsampling=0), "ycc"))
        out.append(("pilL saturated %dx%d q100" % (w, h), _pil_jpeg(sat[:, :, 0], quality=100), "L"))
    for (w, h) in ((203, 117), (333, 77)):  # (the model's encoder rejects some odd 4:2:0 sizes, 131 x 97 among them)
        for c in (444, 420):
            for q in (75, 100):
                out.append(("oracle %d %dx%d q%d" % (c, w, h, q), orc.encode(synth.frame(q + c + w, w, h, c), w, h, c, q), "ycc" if c == 444 else "Y"))
    return out


# ---- CPU tier ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", sr.SCALES)
def test_reference_equals_pillow_draft(orc, s):
    """The int64 restatement is libjpeg's scaled decode: Pillow (libjpeg-turbo) Image.draft, exactly."""
    pytest.importorskip("PIL.Image")
    for name, jpg, what in _pillow_cases():
        ref = sr.ScaledDecode(orc, jpg, s, t81_tables=True)
        if what == "L":
            got = _draft(jpg, "L", s)
            assert np.array_equal(got, ref.cropped[0]), name
        else:
            got = _draft(jpg, "YCbCr", s)
            assert np.array_equal(got[:, :, 0], ref.cropped[0]), name
            if what == "ycc":
                assert np.array_equal(got[:, :, 1], ref.cropped[1]) and np.array_equal(got[:, :, 2], ref.cropped[2]), name


def _info_dict(f):
    return {k: (list(v) if not isinstance(v, int) else v) for k, v in ((n, getattr(f, n)) for n, _ in f._fields_)}


def _geometry_files(orc):
    """The CASES geometries (the oracle's encoder) plus 1 x 1, 8 x 8, 17 x 9 and 3 x 3 (Pillow's: the model's encoder
    rejects some of these sizes) in 4:2:0, 4:2:2 and 4:4:4."""
    out = [((c, q, w, h, ri), orc.encode(synth.frame(400 + i, w, h, c), w, h, c, q, restart_interval=ri)) for i, (c, q, w, h, ri) in enumerate(CASES)]
    for w, h in ((1, 1), (8, 8), (17, 9), (3, 3)):
        for sub, c in ((2, 420), (1, 422), (0, 444)):
            out.append(((c, 75, w, h, 0), _pil_jpeg(_rgb_image(w * h, w, h), quality=75, subsampling=sub)))
    return out


def test_frame_info_geometry_rule(orc):
    import hcjpeg as hcj

    t81 = hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES
    for case, jpg in _geometry_files(orc):
        base = hcj.frame_info(jpg, t81)
        dec = orc.decode(jpg, t81_tables=True)
        b = _info_dict(base)
        n = base.ncomp
        # s = 1 is today's geometry: the oracle's Decoder.init, field for field
        assert (base.width, base.height) == (dec.width, dec.height), case
        assert [(b["decoded_width"][i], b["decoded_height"][i]) for i in range(n)] == dec.decoded_size, case
        assert [(b["actual_width"][i], b["actual_height"][i]) for i in range(n)] == dec.actual_size, case
        assert (base.mcus_wide, base.mcus_high, base.nblocks) == (dec.mcus_wide, dec.mcus_high, dec.nblocks), case
        for s in sr.SCALES:
            f = hcj.frame_info(jpg, t81 | sr.FLAG[s])
            d = _info_dict(f)
            W, H, dsz, asz, chroma = sr.geometry(base.width, base.height, b["hs"][:n], b["vs"][:n],
                                                 list(zip(b["decoded_width"][:n], b["decoded_height"][:n])), s)
            assert (f.width, f.height, f.chroma) == (W, H, chroma), (case, s)
            assert [(d["decoded_width"][i], d["decoded_height"][i]) for i in range(n)] == dsz, (case, s)
            assert [(d["actual_width"][i], d["actual_height"][i]) for i in range(n)] == asz, (case, s)
            for i in range(n):  # the padded plane covers the cropped one
                assert dsz[i][0] >= asz[i][0] and dsz[i][1] >= asz[i][1]
            for k in ("ncomp", "hs", "vs", "mcus_wide", "mcus_high", "blocks_per_mcu", "nblocks", "restart_interval"):
                assert d[k] == b[k], (case, s, k)
            assert f.planes_bytes == sum(w * h for w, h in dsz)
            assert f.yuv_bytes == (sum(w * h for w, h in asz[:3]) if chroma else 0)
            assert f.rgb_bytes == (W * H * 3 if chroma else 0)
    # the header decoder ignores the scale bits
    jpg = _geometry_files(orc)[0][1]
    a, z = hcj.header_decode(jpg, hcj.FLAG_T81_TABLES), hcj.header_decode(jpg, hcj.FLAG_T81_TABLES | hcj.FLAG_SCALE_1_8)
    assert bytes(a) == bytes(z)
    assert (hcj.FLAG_SCALE_1_2, hcj.FLAG_SCALE_1_4, hcj.FLAG_SCALE_1_8, hcj.FLAG_SCALE_MASK) == (0x10, 0x20, 0x30, 0x30)


def _check_emul(coefs, qt, s, modes=(-1, 1)):
    want = sr.reduced(sr.dequantise(coefs, qt), s)
    for w in modes:
        got = emul_scaled(coefs, qt, s, w)
        bad = np.nonzero((got != want).reshape(len(want), -1).any(1))[0]
        assert bad.size == 0, (s, w, bad[:5])


@pytest.mark.parametrize("s", sr.SCALES)
def test_emul_reduced_transforms(orc, s):
    """The device-side transforms (run on the CPU) against the reference: random blocks, extreme blocks, and blocks
    just below / above the wide-block guard (the 32-bit column pass is exact below it)."""
    rng = np.random.default_rng(40 + s)
    limit = emul().emu_scaled_l1_limit()
    qt = orc.quant_scale(False, 50).astype(np.uint16)
    c = np.where(rng.random((4000, 64)) < 0.2, rng.integers(-300, 300, (4000, 64)), 0).astype(np.int16)
    c[:, 0] = rng.integers(-1024, 1024, 4000)
    small = np.where(rng.random((4000, 64)) < 0.2, rng.integers(-40, 40, (4000, 64)), 0).astype(np.int16)
    small[:, 0] = c[:, 0]
    under = small[(np.abs(small.astype(np.int64)) * qt).sum(1) < limit]
    assert len(under) > 1000
    _check_emul(under, qt, s, (-1, 0, 1))
    _check_emul(c, qt, s)
    # extreme: int16 limits with 8-bit (255) and 16-bit (65535) quant entries, every sign pattern at random
    for qv in (255, 65535):
        q = np.full(64, qv, np.uint16)
        ext = np.where(rng.random((500, 64)) < 0.5, -32768, 32767).astype(np.int16)
        ext[:4] = [np.full(64, -32768), np.full(64, 32767), np.zeros(64), np.arange(64) * 511 - 16000]
        _check_emul(ext, q, s)
        q2 = rng.integers(1, qv + 1, 64).astype(np.uint16)
        _check_emul(rng.integers(-32768, 32768, (500, 64)).astype(np.int16), q2, s)
    # at the guard: blocks whose sum(|dequantised coefficient|) is limit - 1 and limit (+ a little), the mass on one
    # coefficient or spread over a column with the signs of the largest weights
    q1 = np.ones(64, np.uint16)
    q2 = np.full(64, 2, np.uint16)
    edge = []
    for target in (limit - 1, limit, limit + 37):
        for pos in range(64):
            b = np.zeros(64, np.int64)
            b[pos] = target // 2
            edge.append((b, q2, target // 2 * 2))
        for sign in (1, -1):
            for col in range(8):
                b = np.zeros(64, np.int64)
                rows = [0, 1, 2, 3, 5, 6, 7]
                wts = np.array([1, 1, 1, 1, -1, -1, -1])
                share = target // len(rows)
                for r, w in zip(rows, wts):
                    b[sr.ZIGZAG_INVERSE.tolist().index(r * 8 + col)] = sign * w * share
                b[0] += sign * (target - share * len(rows))
                edge.append((b, q1, None))
        for trial in range(200):
            b = rng.normal(0, 1, 64) * (rng.random(64) < 0.4)
            b = np.round(b / max(np.abs(b).sum(), 1e-9) * (target // 2)).astype(np.int64)
            edge.append((b, q2, None))
    below = [(b, q) for b, q, _ in edge if (np.abs(b) * q.astype(np.int64)).sum() < limit]
    above = [(b, q) for b, q, _ in edge if (np.abs(b) * q.astype(np.int64)).sum() >= limit]
    assert len(below) > 100 and len(above) > 100
    for group, modes in ((below, (-1, 0, 1)), (above, (-1, 1))):
        for q in (q1, q2):
            blocks = np.array([b for b, qq in group if qq is q], np.int64)
            if len(blocks):
                _check_emul(blocks.astype(np.int16), q, s, modes)


# ---- GPU tier ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hcj():
    import hcjpeg

    assert hcjpeg.lib() is not None
    return hcjpeg


@pytest.fixture(scope="module")
def ctx(hcj):
    c = hcj.Context(0)
    yield c
    c.close()


def _case_files(orc):
    return [orc.encode(synth.frame(100 + i, w, h, c), w, h, c, q, restart_interval=ri) for i, (c, q, w, h, ri) in enumerate(CASES)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode_name", list(MODES))
@pytest.mark.parametrize("s", sr.SCALES)
def test_scaled_batch_matches_reference(hcj, ctx, orc, mode_name, s):
    """One mixed batch (restart and speculative entropy routes, odd sizes, 8 x 8) in every output mode."""
    mode = MODES[mode_name]
    jpgs = _case_files(orc)
    outs, st = ctx.decode_batch(jpgs, mode, hcj.FLAG_DEFAULT | sr.FLAG[s])
    assert st == [0] * len(jpgs)
    for jpg, out, case in zip(jpgs, outs, CASES):
        assert bytes(out) == sr.ScaledDecode(orc, jpg, s).output(mode), (case, s)


@pytest.mark.gpu
@pytest.mark.parametrize("s", sr.SCALES)
def test_scaled_device_equals_pillow_draft(hcj, ctx, orc, s):
    """The device's 4:4:4 and grayscale output against libjpeg-turbo's scaled decode directly."""
    pytest.importorskip("PIL.Image")
    cases = [c for c in _pillow_cases() if c[2] in ("ycc", "L")]
    jpgs = [j for _, j, _ in cases]
    flags = hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES | sr.FLAG[s]
    outs, st = ctx.decode_batch(jpgs, hcj.OUT_PLANES, flags)
    assert st == [0] * len(jpgs)
    for (name, jpg, what), out in zip(cases, outs):
        f = hcj.frame_info(jpg, flags)
        planes, off = [], 0
        for i in range(f.ncomp):
            dw, dh = f.decoded_width[i], f.decoded_height[i]
            planes.append(out[off:off + dw * dh].reshape(dh, dw)[: f.actual_height[i], : f.actual_width[i]])
            off += dw * dh
        if what == "L":
            assert np.array_equal(planes[0], _draft(jpg, "L", s)), name
        else:
            assert np.array_equal(np.stack(planes, -1), _draft(jpg, "YCbCr", s)), name


def _b16(jpg):
    """Every DQT rewritten as a 16-bit table (Pq = 1) of large entries (as test_gpu_decode.test_wide_idct_path)."""
    out, i, src = bytearray(), 0, bytearray(jpg)
    while i < len(src):
        if src[i] == 0xFF and src[i + 1] == 0xDB:
            tq = src[i + 4] & 15
            out += bytes([0xFF, 0xDB, 0x00, 0x83, 0x10 | tq]) + b"".join(bytes([1 + (k % 3), 0x2C]) for k in range(64))
            i += 69
        else:
            out.append(src[i])
            i += 1
    return bytes(out)


@pytest.mark.gpu
@pytest.mark.parametrize("s", sr.SCALES)
def test_scaled_wide_path(hcj, ctx, orc, data, s):
    """Quant tables patched to 255 and 16-bit tables: flagged blocks and wide images come out exact at every scale."""
    from test_emul_device_logic import _patch_dqt

    base = orc.encode(data("mini64x64.444"), 64, 64, 444, 100)
    jr = _patch_dqt(orc.encode(synth.frame(77, 96, 64, 420), 96, 64, 420, 90, restart_interval=2), 200)
    batch = [base, _patch_dqt(base, 255), _b16(base), data("Mouse480.jpg"), jr]
    for mode in (hcj.OUT_YUV, hcj.OUT_PLANES):
        outs, st = ctx.decode_batch(batch, mode, hcj.FLAG_DEFAULT | sr.FLAG[s])
        assert st == [0] * len(batch)
        for i, (jpg, out) in enumerate(zip(batch, outs)):
            assert bytes(out) == sr.ScaledDecode(orc, jpg, s).output(mode), (i, mode, s)


@pytest.mark.gpu
@pytest.mark.parametrize("s", sr.SCALES)
def test_scaled_other_entry_points(hcj, ctx, orc, data, s):
    from test_abi import mjpeg_stream

    flags = hcj.FLAG_DEFAULT | sr.FLAG[s]
    jpgs = _case_files(orc)[:6] + [data("Mouse480.jpg")]
    refs = [sr.ScaledDecode(orc, j, s) for j in jpgs]
    # decode_a_frame
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        assert bytes(ctx.decode_a_frame(jpgs[-1], mode, flags)) == refs[-1].output(mode)
    # decode_batch_multi with one context
    outs, st = hcj.decode_batch_multi([ctx], jpgs, hcj.OUT_YUV444, flags)
    assert st == [0] * len(jpgs) and all(bytes(o) == r.output(hcj.OUT_YUV444) for o, r in zip(outs, refs))
    # decode_stream on a Motion-JPEG stream
    js, stream, _ = mjpeg_stream(orc, data)
    for mode in (hcj.OUT_YUV, hcj.OUT_PLANES):
        frames, st = ctx.decode_stream(stream, mode, flags | hcj.FLAG_T81_TABLES)
        assert st == [0] * len(js)
        for j, f in zip(js, frames):
            assert bytes(f) == sr.ScaledDecode(orc, j, s, t81_tables=True).output(mode)
    # the three-step batch: device output sizes, on-device compare, coefficient taps unscaled
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        with hcj.Batch(ctx, jpgs, mode, flags) as b, hcj.Batch(ctx, jpgs, mode) as full:
            assert b.host_status == [0] * len(jpgs)
            b.decode()
            full.decode()
            for i, j in enumerate(jpgs):
                assert b.device_output(i)[1] == hcj.out_size(hcj.frame_info(j, flags), mode) == len(refs[i].output(mode))
            ms = b.compare([r.output(mode) for r in refs])
            for m in ms:
                assert m.status == 0 and list(m.max_difference) == [0] * 4 and list(m.square_error) == [0] * 4
            for i in range(len(jpgs)):
                assert np.array_equal(b.coefficients(i), full.coefficients(i))
            outs, st = b.fetch()
            assert st == [0] * len(jpgs) and all(bytes(o) == r.output(mode) for o, r in zip(outs, refs))


@pytest.mark.gpu
@pytest.mark.parametrize("ri", [0, 8])
def test_scaled_1080p_420_full_size(hcj, ctx, orc, ri):
    """48 x 1080p 4:2:0 (3 distinct images) at every scale against the reference."""
    w, h = 1920, 1080
    uniq = [orc.encode(synth.frame(2000 + i, w, h, 420), w, h, 420, 75, restart_interval=ri) for i in range(3)]
    batch = [uniq[i % 3] for i in range(48)]
    for s in sr.SCALES:
        want = [sha(sr.ScaledDecode(orc, j, s).yuv()) for j in uniq]
        outs, st = ctx.decode_batch(batch, hcj.OUT_YUV, hcj.FLAG_DEFAULT | sr.FLAG[s])
        assert st == [0] * 48
        assert [sha(o) for o in outs] == [want[i % 3] for i in range(48)], s


@pytest.mark.gpu
def test_gray_411_440_planes(hcj, ctx, orc):
    """Grayscale and OpenCV 4:1:1 / 4:4:0 files through HCJ_OUT_PLANES, unscaled (against the oracle) and at every scale
    (against the reference): geometries K5's thread mapping serves for both."""
    cv2 = pytest.importorskip("cv2")
    jpgs = []
    for i, (w, h) in enumerate(((203, 117), (96, 64), (331, 250))):
        img = _rgb_image(900 + i, w, h)
        for sf in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440):
            ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
            assert ok
            jpgs.append(enc.tobytes())
        ok, enc = cv2.imencode(".jpg", img[:, :, 0], [cv2.IMWRITE_JPEG_QUALITY, 85])
        assert ok
        jpgs.append(enc.tobytes())
    hs = [tuple(hcj.frame_info(j, hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES).hs[:3]) for j in jpgs]
    assert (4, 1, 1) in hs and (1, 0, 0) in hs
    flags = hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES
    outs, st = ctx.decode_batch(jpgs, hcj.OUT_PLANES, flags)
    assert st == [0] * len(jpgs)
    for j, o in zip(jpgs, outs):
        assert bytes(o) == b"".join(p.tobytes() for p in orc.decode(j, t81_tables=True).planes)
    for s in sr.SCALES:
        outs, st = ctx.decode_batch(jpgs, hcj.OUT_PLANES, flags | sr.FLAG[s])
        assert st == [0] * len(jpgs)
        for j, o in zip(jpgs, outs):
            assert bytes(o) == sr.ScaledDecode(orc, j, s, t81_tables=True).planes_bytes(), s
