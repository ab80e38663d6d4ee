"""libjpeg reconstruction (HCJ_FLAG_LIBJPEG): libjpeg-turbo's islow IDCT and fancy chroma up-sampling on the device.

The semantics are pinned twice: the int64 restatement in libjpeg_reference.py equals Pillow (libjpeg-turbo) exactly, and
the device equals that restatement byte for byte in every output mode (and Pillow directly)."""
import ctypes as C
import hashlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import libjpeg_reference as lr
import scaled_reference as sr
import synth

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "video-coding_b200", "csrc")
_EMUL_OUT = os.path.join(_HERE, "_build", "libemul_libjpeg.so")
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
    """tests/emul/libjpeg.cpp built with g++ (rebuilt when a source is newer)."""
    global _emul
    if _emul is None:
        srcs = [os.path.join(_HERE, "emul", "libjpeg.cpp")] + [os.path.join(_CSRC, f) for f in ("hcj_device.cuh", "hcj_common.h")]
        if not (os.path.exists(_EMUL_OUT) and all(os.path.getmtime(_EMUL_OUT) >= os.path.getmtime(s) for s in srcs)):
            os.makedirs(os.path.dirname(_EMUL_OUT), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I", _CSRC, "-x", "c++",
                                   srcs[0], "-o", _EMUL_OUT])
        L = C.CDLL(_EMUL_OUT)
        L.emu_islow.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]
        L.emu_upsample.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _emul = L
    return _emul


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


def _cv2_jpeg(img, sf, q=90):
    import cv2

    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
    assert ok
    return enc.tobytes()


def _pillow(jpg):
    """What Pillow gives: (RGB or None, draft("YCbCr") or None, draft("L") / the L image)."""
    from PIL import Image

    im = Image.open(io.BytesIO(jpg))
    if im.mode == "L":
        return None, None, np.asarray(im)
    rgb = np.asarray(im.convert("RGB"))
    im = Image.open(io.BytesIO(jpg))
    im.draft("YCbCr", im.size)
    ycc = np.asarray(im)
    im = Image.open(io.BytesIO(jpg))
    im.draft("L", im.size)
    return rgb, ycc, np.asarray(im)


def _corpus(orc):
    """(name, jpeg): Pillow 4:4:4 / 4:2:2 / 4:2:0 / grayscale at odd and tiny sizes (chroma planes of width <= 2 among
    them), q50-100 and saturated noise; OpenCV 4:1:1 / 4:4:0; the oracle's encoder with and without restart intervals."""
    out = []
    for (w, h) in ((203, 117), (131, 97), (64, 48), (4, 4), (3, 5), (2, 7), (1, 1)):
        for q in (50, 75, 95, 100):
            img = _rgb_image(w * 7 + q, w, h)
            for sub, c in ((0, 444), (1, 422), (2, 420)):
                out.append(("pil%d %dx%d q%d" % (c, w, h, q), _pil_jpeg(img, quality=q, subsampling=sub)))
            out.append(("pilL %dx%d q%d" % (w, h, q), _pil_jpeg(img[:, :, 1], quality=q)))
    for (w, h) in ((203, 117), (131, 97)):
        sat = _rgb_image(7 + w, w, h, saturated=True)
        for sub, c in ((0, 444), (1, 422), (2, 420)):
            out.append(("pil%d saturated %dx%d q100" % (c, w, h), _pil_jpeg(sat, quality=100, subsampling=sub)))
    try:
        import cv2

        for (w, h) in ((203, 117), (37, 29), (331, 250)):
            img = _rgb_image(900 + w, w, h)
            out.append(("cv411 %dx%d" % (w, h), _cv2_jpeg(img, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)))
            out.append(("cv440 %dx%d" % (w, h), _cv2_jpeg(img, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440)))
            out.append(("cv420 %dx%d" % (w, h), _cv2_jpeg(img, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420)))
    except ImportError:
        pass
    for i, (c, q, w, h, ri) in enumerate(CASES):
        out.append(("oracle %s" % (CASES[i],), orc.encode(synth.frame(100 + i, w, h, c), w, h, c, q, restart_interval=ri)))
    # the model's entropy decoder reads past the end of a few tiny scans (1 x 1 grayscale): outside its domain
    return [(n, j) for n, j in out if orc.decode_status(j, t81_tables=True) == 0]


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


def _wide_files(orc, data):
    """Blocks the entropy decoders flag (quant tables patched to 255 / 200) and 16-bit tables."""
    from test_emul_device_logic import _patch_dqt

    base = orc.encode(data("mini64x64.444"), 64, 64, 444, 100)
    jr = _patch_dqt(orc.encode(synth.frame(77, 96, 64, 420), 96, 64, 420, 90, restart_interval=2), 200)
    return [_patch_dqt(base, 255), _b16(base), jr]


def _pillow_c_semantics(jpgs):
    """Pillow's RGB in a subprocess with libjpeg-turbo's SIMD off (JSIMD_FORCENONE=1): its C code paths."""
    code = ("import io, sys, json, numpy as np\nfrom PIL import Image\n"
            "out = []\nfor h in json.loads(sys.stdin.read()):\n"
            "    out.append(np.asarray(Image.open(io.BytesIO(bytes.fromhex(h))).convert('RGB')).tobytes().hex())\n"
            "print(json.dumps(out))\n")
    env = dict(os.environ, JSIMD_FORCENONE="1")
    r = subprocess.run([sys.executable, "-c", code], input=json.dumps([j.hex() for j in jpgs]), capture_output=True, text=True,
                       env=env, check=True)
    return [bytes.fromhex(h) for h in json.loads(r.stdout)]


# ---- CPU tier ---------------------------------------------------------------------------------------------------------
def test_reference_equals_pillow(orc):
    """The int64 restatement is libjpeg-turbo's default decompression: Pillow's RGB, draft("YCbCr") and draft("L"),
    exactly; and OpenCV's imdecode gives the same RGB."""
    pytest.importorskip("PIL.Image")
    try:
        import cv2
    except ImportError:
        cv2 = None
    for name, jpg in _corpus(orc):
        ref = lr.LibjpegDecode(orc, jpg, t81_tables=True)
        rgb, ycc, lum = _pillow(jpg)
        H, W = ref.height, ref.width
        assert np.array_equal(lum, ref.planes[0][:H, :W]), name
        if rgb is None:
            continue
        assert np.array_equal(np.moveaxis(ref.yuv444(), 0, -1), ycc), name
        assert np.array_equal(ref.rgb(), rgb), name
        if cv2 is not None:
            bgr = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR)
            assert np.array_equal(bgr[:, :, ::-1], rgb), name


def test_reference_wide_files_equal_pillow_c(orc, data):
    """Files whose dequantised coefficients do not fit 16 bits: the reference equals libjpeg-turbo's C code (SIMD off).
    Whether Pillow with its SIMD IDCT differs there is recorded, not asserted."""
    pytest.importorskip("PIL.Image")
    jpgs = _wide_files(orc, data)
    want = _pillow_c_semantics(jpgs)
    for i, (jpg, w) in enumerate(zip(jpgs, want)):
        assert lr.LibjpegDecode(orc, jpg, t81_tables=True).rgb().tobytes() == w, i
        simd, _, _ = _pillow(jpg)
        print("wide file %d: default Pillow %s the C semantics" % (i, "equals" if simd.tobytes() == w else "differs from"))


def _check_emul(coefs, qt, modes=(-1, 1)):
    want = lr.islow(_dequant(coefs, qt)).reshape(-1, 64)
    c = np.ascontiguousarray(coefs, np.int16).reshape(-1, 64)
    q = np.ascontiguousarray(qt, np.uint16)
    for w in modes:
        got = np.zeros((c.shape[0], 64), np.uint8)
        emul().emu_islow(c.ctypes.data, c.shape[0], q.ctypes.data, w, got.ctypes.data)
        bad = np.nonzero((got != want).any(1))[0]
        assert bad.size == 0, (w, bad[:5])


def _dequant(coefs_zz, qt_zz):
    return sr.dequantise(coefs_zz, qt_zz)


def test_emul_islow(orc):
    """The device transform (run on the CPU) against the reference: random blocks, int16 extremes with 255 and 65535
    quant entries (the 32-bit workspace truncation), both sides of the wide-block guard, and the range-limit wrap."""
    rng = np.random.default_rng(41)
    limit = emul().emu_islow_l1_limit()
    qt = orc.quant_scale(False, 50).astype(np.uint16)
    c = np.where(rng.random((4000, 64)) < 0.2, rng.integers(-300, 300, (4000, 64)), 0).astype(np.int16)
    c[:, 0] = rng.integers(-1024, 1024, 4000)
    small = np.where(rng.random((4000, 64)) < 0.2, rng.integers(-40, 40, (4000, 64)), 0).astype(np.int16)
    small[:, 0] = c[:, 0]
    under = small[(np.abs(small.astype(np.int64)) * qt).sum(1) < limit]
    assert len(under) > 1000
    _check_emul(under, qt, (-1, 0, 1))
    _check_emul(c, qt)
    wraps = 0
    for qv in (255, 65535):
        q = np.full(64, qv, np.uint16)
        ext = np.where(rng.random((500, 64)) < 0.5, -32768, 32767).astype(np.int16)
        ext[:4] = [np.full(64, -32768), np.full(64, 32767), np.zeros(64), np.arange(64) * 511 - 16000]
        _check_emul(ext, q)
        q2 = rng.integers(1, qv + 1, 64).astype(np.uint16)
        r = rng.integers(-32768, 32768, (500, 64)).astype(np.int16)
        _check_emul(r, q2)
        # samples from the wrapped part of the range-limit table: neither saturated 0 / 255 nor what a clamp would give
        b = np.asarray(_dequant(r, q2), np.int64).reshape(-1, 8, 8)
        wraps += int(((lr.islow(b) > 0) & (lr.islow(b) < 255)).sum())
    assert wraps > 1000
    # DC-only blocks around the wrap points (v = 640 .. 1400 after the descale)
    dc = np.zeros((400, 64), np.int16)
    dc[:, 0] = np.arange(400) * 20 + 2000
    _check_emul(dc, np.full(64, 10, np.uint16), (-1, 0, 1))
    _check_emul(-dc, np.full(64, 10, np.uint16), (-1, 0, 1))
    # at the guard: sum(|dequantised coefficient|) just below and above it, the mass on one coefficient or spread
    q2 = np.full(64, 2, np.uint16)
    below, above = [], []
    for target in (limit - 1, limit, limit + 37):
        for pos in range(64):
            blk = np.zeros(64, np.int64)
            blk[pos] = target // 2
            (below if target // 2 * 2 < limit else above).append(blk)
        for trial in range(200):
            blk = rng.normal(0, 1, 64) * (rng.random(64) < 0.4)
            blk = np.round(blk / max(np.abs(blk).sum(), 1e-9) * (target // 2)).astype(np.int64)
            (below if (np.abs(blk) * 2).sum() < limit else above).append(blk)
    assert len(below) > 100 and len(above) > 100
    _check_emul(np.array(below).astype(np.int16), q2, (-1, 0, 1))
    _check_emul(np.array(above).astype(np.int16), q2, (-1, 1))


def test_emul_upsample():
    """libjpeg_upsample (run on the CPU) against the reference for every ratio, including narrow and one-row planes."""
    rng = np.random.default_rng(5)
    for hr, vr in ((1, 1), (2, 1), (2, 2), (1, 2), (4, 1), (1, 4), (4, 2), (2, 4), (3, 1), (4, 4)):
        for W, H in ((1, 1), (2, 2), (3, 5), (4, 4), (5, 3), (6, 2), (17, 9), (64, 48), (203, 117)):
            rw, rh = -(-W // hr), -(-H // vr)
            pitch = (rw + 7) // 8 * 8 + 8
            plane = rng.integers(0, 256, (rh + 3, pitch), dtype=np.uint8)  # rows and columns past the real plane are noise
            want = lr.upsample(plane, rw, rh, hr, vr, W, H)
            got = np.zeros((H, W), np.uint8)
            p = np.ascontiguousarray(plane)
            emul().emu_upsample(p.ctypes.data, pitch, rw, rh, hr, vr, W, H, got.ctypes.data)
            assert np.array_equal(got, want), (hr, vr, W, H)


def test_frame_info_and_flag_rules(orc):
    """Geometry under the flag: unchanged but for rgb_bytes of 4:4:0 / 4:1:1; the flag with a scale is an invalid
    argument; the header decoder ignores the flag."""
    import hcjpeg as hcj

    assert hcj.FLAG_LIBJPEG == 0x40
    t81 = hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES
    for name, jpg in _corpus(orc):
        a, b = hcj.frame_info(jpg, t81), hcj.frame_info(jpg, t81 | hcj.FLAG_LIBJPEG)
        for k, _ in a._fields_:
            va, vb = getattr(a, k), getattr(b, k)
            va, vb = (list(va), list(vb)) if not isinstance(va, int) else (va, vb)
            if k == "rgb_bytes" and a.ncomp == 3 and a.chroma == 0:
                assert vb == a.width * a.height * 3, name
            else:
                assert va == vb, (name, k)
        for s in (0x10, 0x20, 0x30):
            with pytest.raises(Exception):
                hcj.frame_info(jpg, t81 | hcj.FLAG_LIBJPEG | s)
    jpg = _corpus(orc)[0][1]
    assert bytes(hcj.header_decode(jpg, hcj.FLAG_T81_TABLES)) == bytes(hcj.header_decode(jpg, hcj.FLAG_T81_TABLES | hcj.FLAG_LIBJPEG))


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


FLAGS = 1 | 2 | lr.FLAG  # FLAG_DEFAULT | FLAG_T81_TABLES | FLAG_LIBJPEG


@pytest.mark.gpu
@pytest.mark.parametrize("mode_name", list(MODES))
def test_libjpeg_batch_matches_reference(hcj, ctx, orc, mode_name):
    """The whole corpus (CASES geometries, Pillow and OpenCV files, 4:4:0 / 4:1:1 / grayscale) in one batch per mode."""
    mode = MODES[mode_name]
    cases = _corpus(orc)
    jpgs = [j for _, j in cases]
    outs, st = ctx.decode_batch(jpgs, mode, FLAGS)
    for (name, jpg), out, s in zip(cases, outs, st):
        f = hcj.frame_info(jpg, FLAGS)
        if f.ncomp < 3 and mode != hcj.OUT_PLANES:
            assert s == -12, name  # HCJ_ERR_NEED_3_COMPONENTS
            continue
        if mode == hcj.OUT_YUV and f.chroma == 0:
            assert s == -11, name  # HCJ_ERR_FRAME_INFER: YUV keeps the model's rules
            continue
        assert s == 0, (name, s)
        assert bytes(out) == lr.LibjpegDecode(orc, jpg, t81_tables=True).output(mode), (name, mode_name)


@pytest.mark.gpu
def test_libjpeg_device_equals_pillow(hcj, ctx, orc):
    """RGB24, YUV444 and the Y plane from the device against Pillow directly."""
    pytest.importorskip("PIL.Image")
    cases = _corpus(orc)
    jpgs = [j for _, j in cases]
    color = [i for i, j in enumerate(jpgs) if hcj.frame_info(j, FLAGS).ncomp == 3]
    rgb, st = ctx.decode_batch([jpgs[i] for i in color], hcj.OUT_RGB24, FLAGS)
    assert st == [0] * len(color)
    ycc, st = ctx.decode_batch([jpgs[i] for i in color], hcj.OUT_YUV444, FLAGS)
    assert st == [0] * len(color)
    planes, st = ctx.decode_batch(jpgs, hcj.OUT_PLANES, FLAGS)
    assert st == [0] * len(jpgs)
    for k, i in enumerate(color):
        want_rgb, want_ycc, _ = _pillow(jpgs[i])
        assert np.array_equal(rgb[k].reshape(want_rgb.shape), want_rgb), cases[i][0]
        assert np.array_equal(np.moveaxis(ycc[k].reshape(3, *want_ycc.shape[:2]), 0, -1), want_ycc), cases[i][0]
    for (name, jpg), out in zip(cases, planes):
        f = hcj.frame_info(jpg, FLAGS)
        lum = out[: f.decoded_width[0] * f.decoded_height[0]].reshape(f.decoded_height[0], f.decoded_width[0])
        assert np.array_equal(lum[: f.height, : f.width], _pillow(jpg)[2]), name


@pytest.mark.gpu
def test_libjpeg_wide_path(hcj, ctx, orc, data):
    """Flagged blocks and 16-bit tables: every mode equals the reference, RGB24 equals Pillow's C code (SIMD off)."""
    jpgs = _wide_files(orc, data)
    for mode in MODES.values():
        outs, st = ctx.decode_batch(jpgs, mode, FLAGS)
        assert st == [0] * len(jpgs)
        for i, (jpg, out) in enumerate(zip(jpgs, outs)):
            assert bytes(out) == lr.LibjpegDecode(orc, jpg, t81_tables=True).output(mode), (i, mode)
    if pytest.importorskip("PIL.Image"):
        outs, _ = ctx.decode_batch(jpgs, hcj.OUT_RGB24, FLAGS)
        assert [bytes(o) for o in outs] == _pillow_c_semantics(jpgs)


@pytest.mark.gpu
def test_libjpeg_mixed_odd_widths(hcj, ctx, orc):
    """4:2:0 and 4:4:4 images of odd widths in one batch: RGB24 rows that start at any byte alignment."""
    pytest.importorskip("PIL.Image")
    jpgs = []
    for i, w in enumerate((97, 131, 203, 65, 33, 18, 255, 1001)):
        img = _rgb_image(3000 + i, w, 23 + i)
        jpgs.append(_pil_jpeg(img, quality=85, subsampling=2 if i % 2 == 0 else 0))
    outs, st = ctx.decode_batch(jpgs, hcj.OUT_RGB24, FLAGS)
    assert st == [0] * len(jpgs)
    for jpg, out in zip(jpgs, outs):
        want = _pillow(jpg)[0]
        assert np.array_equal(out.reshape(want.shape), want)


@pytest.mark.gpu
def test_libjpeg_other_entry_points(hcj, ctx, orc, data):
    from test_abi import mjpeg_stream

    jpgs = [j for _, j in _corpus(orc)[-12:]] + [data("Mouse480.jpg")]
    refs = [lr.LibjpegDecode(orc, j, t81_tables=True) for j in jpgs]
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        assert bytes(ctx.decode_a_frame(jpgs[-1], mode, FLAGS)) == refs[-1].output(mode)
    outs, st = hcj.decode_batch_multi([ctx], jpgs, hcj.OUT_YUV444, FLAGS)
    assert st == [0] * len(jpgs) and all(bytes(o) == r.output(hcj.OUT_YUV444) for o, r in zip(outs, refs))
    js, stream, _ = mjpeg_stream(orc, data)
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        frames, st = ctx.decode_stream(stream, mode, FLAGS)
        assert st == [0] * len(js)
        for j, f in zip(js, frames):
            assert bytes(f) == lr.LibjpegDecode(orc, j, t81_tables=True).output(mode)
    # the three-step batch: device output sizes, on-device compare, the coefficient tap unaffected
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        with hcj.Batch(ctx, jpgs, mode, FLAGS) as b, hcj.Batch(ctx, jpgs, mode, FLAGS & ~lr.FLAG) as plain:
            assert b.host_status == [0] * len(jpgs)
            b.decode()
            plain.decode()
            for i, j in enumerate(jpgs):
                assert b.device_output(i)[1] == hcj.out_size(hcj.frame_info(j, FLAGS), mode) == len(refs[i].output(mode))
            ms = b.compare([r.output(mode) for r in refs])
            for m in ms:
                assert m.status == 0 and list(m.max_difference) == [0] * 4 and list(m.square_error) == [0] * 4
            for i in range(len(jpgs)):
                assert np.array_equal(b.coefficients(i), plain.coefficients(i))
            outs, st = b.fetch()
            assert st == [0] * len(jpgs) and all(bytes(o) == r.output(mode) for o, r in zip(outs, refs))
    # kernels actually launched: k_rgb for the 4:4:4 image, and k_rgb_libjpeg once there is a 4:2:0 image too
    j444, j420 = jpgs[3], jpgs[0]  # CASES 3 and 0: no restart intervals
    with hcj.Batch(ctx, [j444], hcj.OUT_RGB24, FLAGS) as one, hcj.Batch(ctx, [j444, j420], hcj.OUT_RGB24, FLAGS) as two:
        assert two.kernels() == one.kernels() + 1


@pytest.mark.gpu
@pytest.mark.parametrize("ri", [0, 8])
def test_libjpeg_1080p_420(hcj, ctx, orc, ri):
    """48 x 1080p 4:2:0 (3 distinct images) in YUV and RGB24 against the reference."""
    w, h = 1920, 1080
    uniq = [orc.encode(synth.frame(2000 + i, w, h, 420), w, h, 420, 75, restart_interval=ri) for i in range(3)]
    batch = [uniq[i % 3] for i in range(48)]
    refs = [lr.LibjpegDecode(orc, j) for j in uniq]
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        want = [sha(r.output(mode)) for r in refs]
        outs, st = ctx.decode_batch(batch, mode, hcj.FLAG_DEFAULT | hcj.FLAG_LIBJPEG)
        assert st == [0] * 48
        assert [sha(o) for o in outs] == [want[i % 3] for i in range(48)], mode


def _sof_factors(jpg, factors):
    """The file with the SOF0 sampling factors of its components replaced by `factors` [(h, v), ...]."""
    b = bytearray(jpg)
    i = b.index(b"\xff\xc0")
    for k, (h, v) in enumerate(factors):
        b[i + 11 + 3 * k] = h << 4 | v
    return bytes(b)


@pytest.mark.gpu
def test_libjpeg_statuses_and_plain_decode(hcj, ctx, orc):
    """Flag + scale is an invalid argument, 4-component and non-integral-ratio frames are unsupported in RGB24 / YUV444,
    and a decode without the flag in the same process is still the oracle's."""
    from PIL import Image

    good = orc.encode(synth.frame(5, 64, 48, 420), 64, 48, 420, 75)
    for sc in (0x10, 0x20, 0x30):
        with pytest.raises(hcj.HcjError):
            ctx.decode_batch([good], hcj.OUT_RGB24, FLAGS | sc)
    buf = io.BytesIO()
    Image.fromarray(_rgb_image(1, 40, 24)).convert("CMYK").save(buf, "JPEG", quality=90)
    cmyk = buf.getvalue()
    odd = _sof_factors(orc.encode(synth.frame(6, 48, 32, 444), 48, 32, 444, 75), [(3, 1), (2, 1), (2, 1)])  # ratio 3 / 2
    assert hcj.frame_info(cmyk, FLAGS).ncomp == 4
    for mode in (hcj.OUT_RGB24, hcj.OUT_YUV444):
        st = ctx.decode_batch([cmyk, odd, good], mode, FLAGS)[1]
        assert st[:2] == [-22, -22] and st[2] == 0, (mode, st)  # HCJ_ERR_UNSUPPORTED_GEOMETRY
    outs, st = ctx.decode_batch([cmyk], hcj.OUT_PLANES, FLAGS)
    assert st == [0] and bytes(outs[0]) == lr.LibjpegDecode(orc, cmyk, t81_tables=True).planes_bytes()
    # no flag: the model's decode, in the same process as the flagged batches above
    jpgs = [orc.encode(synth.frame(100 + i, w, h, c), w, h, c, q, restart_interval=ri) for i, (c, q, w, h, ri) in enumerate(CASES)]
    for mode in (hcj.OUT_YUV, hcj.OUT_RGB24):
        outs, st = ctx.decode_batch(jpgs, mode)
        assert st == [0] * len(jpgs)
        for j, o in zip(jpgs, outs):
            assert bytes(o) == sr.ScaledDecode(orc, j, 1).output(mode)  # s = 1: the oracle's decode
