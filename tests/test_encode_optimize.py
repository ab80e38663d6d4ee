"""HCJ_ENC_OPTIMIZE_HUFFMAN: every frame encoded with its own optimal Huffman tables (k_symbol_counts, k_huff_tables).

The expected file of a frame is optimized_file(orc.encode(frame, ...)) (optimal_huffman_reference): the oracle's
coefficients, counted and given libjpeg's K.2 tables by a literal restatement, and re-written through huffman_writer.
The CPU tier pins the restatement against Pillow and OpenCV optimized files, the device procedures (through their g++
build in tests/emul/huffopt.cpp) against the restatement, and the reference files' pixels against the default files';
the GPU tier checks the device files byte for byte."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest

import huffman_writer as hw
import synth
from optimal_huffman_reference import gen_optimal_table, optimized_file, table_counts
from rgb_reference import rgb24_to_frame

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "video-coding_b200", "csrc")
_EMUL_OUT = os.path.join(_HERE, "_build", "libhuffopt.so")
_emul = None


def emul():
    """tests/emul/huffopt.cpp built with g++ (rebuilt when a source is newer)."""
    global _emul
    if _emul is None:
        srcs = [os.path.join(_HERE, "emul", "huffopt.cpp")] + [os.path.join(_CSRC, f) for f in ("hcj_device.cuh", "hcj_common.h")]
        if not (os.path.exists(_EMUL_OUT) and all(os.path.getmtime(_EMUL_OUT) >= os.path.getmtime(s) for s in srcs)):
            os.makedirs(os.path.dirname(_EMUL_OUT), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I", _CSRC, "-x", "c++",
                                   srcs[0], "-o", _EMUL_OUT])
        L = C.CDLL(_EMUL_OUT)
        for f in (L.emu_gen_optimal_table, L.emu_k2_single_lane):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
            f.restype = C.c_int
        L.emu_block_symbols.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.emu_block_symbols.restype = C.c_int64
        _emul = L
    return _emul


def emul_table(fn, freq):
    f = np.zeros(256, np.uint32)
    for s, c in (freq.items() if isinstance(freq, dict) else enumerate(freq)):
        f[s] = c
    bits = np.zeros(16, np.uint8)
    vals = np.zeros(256, np.uint8)
    n = fn(f.ctypes.data, bits.ctypes.data, vals.ctypes.data)
    return bits.tolist(), vals[:n].tolist()


def file_tables(jpg):
    """[(class, id, bits, values)] of a file's DHT segments, and the counts of its scan per (class, id)."""
    from oracle import pyoracle as orc

    frame, dhts, ri, _ = hw.read_file(jpg)
    return dhts, table_counts(orc.decode(jpg, want_blocks=True).coefs_abs_dc(), frame, ri)


def check_tables(jpg, info=None):
    dhts, counts = file_tables(jpg)
    mx = 0
    for tc, th, lengths, values in dhts:
        i = {}
        assert gen_optimal_table(counts[(tc, th)], i) == (lengths, values), (tc, th)
        mx = max(mx, i["max_codesize"])
    return mx


def pil_file(img, **kw):
    from PIL import Image

    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", optimize=True, **kw)
    return b.getvalue()


def rgb_image(seed, w, h):
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.stack([synth.plane(rng, w, h) for _ in range(3)], axis=-1))


# ---- CPU tier: the restatement against libjpeg's optimized files ------------------------------------------------

@pytest.mark.parametrize("subsampling", [0, 1, 2, "L"])
@pytest.mark.parametrize("size", [(160, 120), (77, 53), (33, 17)])
def test_restatement_equals_pillow_tables(orc, subsampling, size):
    """Pillow optimize=True (libjpeg-turbo) at 4:4:4, 4:2:2, 4:2:0 and grayscale, odd sizes, q 50..100, with and without
    restart markers: the counts of the file's scan give back every DHT segment, lengths and values."""
    pytest.importorskip("PIL")
    w, h = size
    img = rgb_image(w * 7 + h, w, h)
    for q, rmb in ((50, 0), (75, 3), (90, 0), (100, 1)):
        if subsampling == "L":
            jpg = pil_file(np.ascontiguousarray(img[:, :, 0]), quality=q, restart_marker_blocks=rmb)
        else:
            jpg = pil_file(img, quality=q, subsampling=subsampling, restart_marker_blocks=rmb)
        assert (hw.read_file(jpg)[2] != 0) == (rmb != 0)
        check_tables(jpg)


def test_restatement_equals_pillow_on_noise_with_long_codes(orc):
    """The 640 x 480 q90 noise image: AC code sizes above 16 before the limit, where ordering HUFFVAL by the final length
    (huffman_writer.optimal_lengths) gives other values.  The restatement matches Pillow byte for byte."""
    pytest.importorskip("PIL")
    img = np.random.default_rng(12).integers(0, 256, (480, 640, 3), dtype=np.uint8)
    jpg = pil_file(img, quality=90)
    assert check_tables(jpg) > 16
    dhts, counts = file_tables(jpg)
    assert any(hw.optimal_lengths(counts[(tc, th)])[1] != v for tc, th, _, v in dhts)


@pytest.mark.parametrize("ri", [0, 4])
def test_restatement_equals_opencv_tables(orc, ri):
    cv2 = pytest.importorskip("cv2")
    for i, (w, h, q) in enumerate(((320, 200, 90), (77, 53, 100), (161, 99, 60))):
        a = rgb_image(40 + i, w, h)
        for img in (a, a[:, :, 0]):
            ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(img), [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1,
                                                                       cv2.IMWRITE_JPEG_RST_INTERVAL, ri])
            assert ok
            check_tables(buf.tobytes())


@pytest.mark.parametrize("chroma", [420, 422, 444, 400])
def test_reference_files_decode_to_the_default_pixels(orc, chroma):
    """optimized_file decodes, in the oracle and in Pillow, to exactly the planes / pixels of the default-table file, and
    is smaller."""
    Image = pytest.importorskip("PIL.Image")
    for w, h, q, ri in ((96, 64, 75, 0), (77, 53, 50, 7), (40, 24, 100, 1)):
        src = synth.frame(w + 3 * h + chroma, w, h, 420 if chroma == 400 else chroma)
        base = orc.encode(src, w, h, chroma, q, ri)
        opt = optimized_file(base)
        assert len(opt) < len(base)
        d0, d1 = orc.decode(base), orc.decode(opt)
        assert len(d1.planes) == len(d0.planes) and all(np.array_equal(a, b) for a, b in zip(d0.planes, d1.planes))
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(opt))), np.asarray(Image.open(io.BytesIO(base))))


# ---- CPU tier: the device procedures (g++ build) against the restatement -----------------------------------------

def _freq_sets():
    rng = np.random.default_rng(3)
    sets = []
    for k in range(40):  # random sets, sparse and dense, small and large counts
        n = int(rng.integers(1, 257))
        syms = rng.choice(256, n, replace=False)
        hi = int(rng.choice([4, 100, 10000, 1 << 22]))
        sets.append({int(s): int(rng.integers(1, hi)) for s in syms})
    sets.append({7: 5})  # a single symbol
    sets.append({0: 1})
    sets.append({s: 1 for s in range(256)})  # all 256 symbols, all tied
    sets.append({s: 3 for s in range(0, 256, 3)})  # ties
    sets.append({s: 1 + (s % 4) for s in range(100)})
    sets.append({s: int(c) for s, c in enumerate(rng.integers(1, 1000, 256))})  # all 256 symbols
    fib = [1, 1]
    while len(fib) < 45:
        fib.append(fib[-1] + fib[-2])
    sets.append({s: fib[s] for s in range(24)})  # code sizes past 16
    sets.append({s: fib[s] for s in range(45)})  # past 32 (the sum stays below 2^32)
    sets.append({255 - s: fib[s] for s in range(40)})
    return sets


def test_device_k2_matches_restatement():
    """gen_optimal_table (serial) and k2_optimal_table (the warp procedure, one lane) equal the restatement on random
    sets, ties, a single symbol, all 256 symbols and Fibonacci counts that push code sizes past 16 and past 32."""
    L = emul()
    seen = 0
    for freq in _freq_sets():
        info = {}
        want = gen_optimal_table(freq, info)
        seen = max(seen, info["max_codesize"])
        assert emul_table(L.emu_gen_optimal_table, freq) == want, freq
        assert emul_table(L.emu_k2_single_lane, freq) == want, freq
        assert sum(want[0]) == len(freq) and hw.kraft_ok(want[0]) and max(i for i, b in enumerate(want[0]) if b) < 16
    assert seen > 32


def _blocks():
    rng = np.random.default_rng(9)
    out = []
    for k in range(400):
        b = np.zeros(64, np.int16)
        nnz = int(rng.integers(0, 64))
        pos = rng.choice(np.arange(1, 64), nnz, replace=False)
        b[pos] = rng.integers(-1023, 1024, nnz) * rng.choice([1, 0], nnz, p=[0.9, 0.1])
        out.append((b, int(rng.integers(-2047, 2048))))
    for v in (1023, -1023, 1, -1):  # saturated: every coefficient non-zero
        out.append((np.full(64, v, np.int16), 2047 if v > 0 else -2047))
    z = np.zeros(64, np.int16)
    z[63] = 5
    out += [(np.zeros(64, np.int16), 0), (z, -1)]
    z2 = np.zeros(64, np.int16)
    z2[40] = -3
    out.append((z2, 0))  # runs of 16 and more: ZRL
    return out


def test_block_symbols_match_encoded_fields():
    """block_symbols_sparse visits exactly the symbols whose codes encode_block_fields_sparse emits, in order, and the
    symbols huffman_writer.block_symbols lists."""
    L = emul()
    for blk, diff in _blocks():
        vis = np.zeros(200, np.uint32)
        emi = np.zeros(200, np.uint32)
        r = L.emu_block_symbols(blk.ctypes.data, diff, vis.ctypes.data, emi.ctypes.data)
        assert r >= 0
        nv, ne = r & 0xFFFF, r >> 16
        assert nv == ne and np.array_equal(vis[:nv], emi[:ne])
        b = blk.astype(np.int64)
        want = [(256 if a else 0) | s for a, s, _, _ in hw.block_symbols(b, diff)]
        assert vis[:nv].tolist() == want


def test_flags_rejected_before_any_work(hcj):
    """hcj_encode_batch_ex with flag bits other than HCJ_ENC_OPTIMIZE_HUFFMAN returns HCJ_ERR_INVALID_ARG before it
    looks at the context or the frames: nothing is written."""
    dummy = (C.c_uint8 * 4096)()
    frame = np.zeros(32 * 16 * 3 // 2, np.uint8)
    out = np.full(4096, 0xA5, np.uint8)
    fp = (C.c_void_p * 1)(frame.ctypes.data)
    op = (C.c_void_p * 1)(out.ctypes.data)
    caps = (C.c_size_t * 1)(4096)
    for flags in (1, 2, 1 << 31, hcj.ENC_OPTIMIZE_HUFFMAN | 1):
        lens = (C.c_size_t * 1)(12345)
        status = (C.c_int * 1)(77)
        rc = hcj.lib().hcj_encode_batch_ex(C.cast(dummy, C.c_void_p), fp, 1, 32, 16, 420, 75, 0, flags, op, caps, lens, status)
        assert rc == -31
        assert (out == 0xA5).all() and lens[0] == 12345 and status[0] == 77
        ctxs = (C.c_void_p * 1)(C.cast(dummy, C.c_void_p).value)
        rc = hcj.lib().hcj_encode_batch_multi_ex(ctxs, 1, fp, 1, 32, 16, 420, 75, 0, flags, op, caps, lens, status)
        assert rc == -31
        assert (out == 0xA5).all() and lens[0] == 12345 and status[0] == 77


@pytest.fixture(scope="module")
def hcj():
    import hcjpeg

    assert hcjpeg.lib() is not None
    return hcjpeg


# ---- GPU tier ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx(hcj):
    c = hcj.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def torch():
    t = pytest.importorskip("torch")
    if not t.cuda.is_available():
        pytest.skip("torch has no CUDA device")
    return t


def expected(orc, src, w, h, chroma, q, ri):
    jpg, quant, _ = orc.encode(src, w, h, chroma, q, ri, want_blocks=True)
    return optimized_file(jpg, coefs=quant)


def src_frame(seed, w, h, chroma):
    return synth.frame(seed, w, h, 420 if chroma == 400 else chroma)


@pytest.mark.gpu
@pytest.mark.parametrize("chroma", [420, 422, 444, 400])
@pytest.mark.parametrize("size", [(1, 1), (17, 9), (77, 53), (640, 480)])
def test_device_files_equal_reference(hcj, ctx, orc, chroma, size):
    """Planar host frames at every chroma and size: the device file equals the reference byte for byte; where the
    default path refuses the geometry, the flag gives the same error."""
    w, h = size
    frames = [src_frame(100 * w + h + i, w, h, chroma) for i in range(2)]
    for ri in (0, 7):
        try:
            base, st0 = ctx.encode_batch(frames, w, h, chroma, 75, ri)
        except hcj.HcjError as e:
            with pytest.raises(hcj.HcjError) as e2:
                ctx.encode_batch(frames, w, h, chroma, 75, ri, optimize=True)
            assert e2.value.status == e.status
            continue
        got, st = ctx.encode_batch(frames, w, h, chroma, 75, ri, optimize=True)
        assert st == st0
        for i, f in enumerate(frames):
            if st[i] == 0:
                assert got[i] == expected(orc, f, w, h, chroma, 75, ri), (i, ri)


@pytest.mark.gpu
@pytest.mark.parametrize("q", [1, 50, 75, 95, 100])
def test_device_files_equal_reference_quality_and_restart(ctx, orc, q):
    w, h = 77, 53
    for chroma in (420, 444):
        frames = [src_frame(q * 13 + ri, w, h, chroma) for ri in (0, 1, 7, 8)]
        for ri in (0, 1, 7, 8):
            got, st = ctx.encode_batch(frames, w, h, chroma, q, ri, optimize=True)
            _, st0 = ctx.encode_batch(frames, w, h, chroma, q, ri)
            assert st == st0
            for i, f in enumerate(frames):
                if st[i] == 0:
                    assert got[i] == expected(orc, f, w, h, chroma, q, ri), (chroma, ri, i)


@pytest.mark.gpu
def test_device_files_equal_reference_1080p(ctx, orc):
    w, h = 1920, 1080
    for chroma, q, ri in ((420, 75, 0), (422, 90, 8)):
        f = src_frame(5 + chroma, w, h, chroma)
        got, st = ctx.encode_batch([f], w, h, chroma, q, ri, optimize=True)
        assert st == [0] and got[0] == expected(orc, f, w, h, chroma, q, ri)


@pytest.mark.gpu
def test_rgb_sources_equal_reference(hcj, ctx, orc, torch):
    """RGB24 frames from host memory and from torch device tensors: the reference of the converted planar frame."""
    for chroma, (w, h), ri in ((420, (77, 53), 0), (422, (130, 70), 8), (444, (64, 48), 1), (400, (33, 17), 7)):
        imgs = [rgb_image(w + i, w, h) for i in range(3)]
        want = [expected(orc, rgb24_to_frame(orc, im, w, h, chroma), w, h, chroma, 75, ri) for im in imgs]
        got, st = ctx.encode_rgb_batch(imgs, w, h, chroma, 75, ri, optimize=True)
        assert st == [0] * 3 and got == want
        dev = [torch.from_numpy(im).to("cuda:%d" % ctx.device) for im in imgs]
        torch.cuda.synchronize()
        got, st = ctx.encode_rgb_batch(dev, w, h, chroma, 75, ri, optimize=True)
        assert st == [0] * 3 and got == want


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", ["1", "3", None])
def test_chunks_keep_tables_per_frame(ctx, orc, chunk):
    """130 different frames in chunks of 1, 3 and the default 64: every file equals its own reference, and neighbouring
    frames carry different tables (nothing leaks from one frame or chunk to the next)."""
    w, h = 48, 32
    frames = [synth.frame(700 + i, w, h, 420) if i % 2 else synth.frame(700 + i, w, h, 420)[::-1] for i in range(130)]
    old = os.environ.get("HCJ_ENC_CHUNK")
    try:
        if chunk is None:
            os.environ.pop("HCJ_ENC_CHUNK", None)
        else:
            os.environ["HCJ_ENC_CHUNK"] = chunk
        got, st = ctx.encode_batch(frames, w, h, 420, 75, 2 if chunk == "3" else 0, optimize=True)
    finally:
        if old is None:
            os.environ.pop("HCJ_ENC_CHUNK", None)
        else:
            os.environ["HCJ_ENC_CHUNK"] = old
    assert st == [0] * 130
    ri = 2 if chunk == "3" else 0
    for i, f in enumerate(frames):
        assert got[i] == expected(orc, f, w, h, 420, 75, ri), i
    dhts = [hw.read_file(j)[1] for j in got]
    assert all(dhts[i] != dhts[i + 1] for i in range(129))


@pytest.mark.gpu
def test_several_contexts(hcj, orc):
    if hcj.device_count() < 2:
        pytest.skip("one GPU")
    ctxs = [hcj.Context(d) for d in range(min(hcj.device_count(), 4))]
    try:
        w, h = 96, 64
        frames = [synth.frame(40 + i, w, h, 420) for i in range(9)]
        got, st = hcj.encode_batch_multi(ctxs, frames, w, h, 420, 75, 3, optimize=True)
        assert st == [0] * 9
        assert got == [expected(orc, f, w, h, 420, 75, 3) for f in frames]
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.gpu
def test_saturated_noise_takes_long_block_path(ctx, orc):
    """Noise at q100: blocks longer than their 512-bit slot (k_pack) coded with the frame's tables."""
    w, h = 128, 96
    rng = np.random.default_rng(77)
    f = rng.integers(0, 256, w * h * 3, dtype=np.uint8).tobytes()
    got, st = ctx.encode_batch([f], w, h, 444, 100, 0, optimize=True)
    assert st == [0] and got[0] == expected(orc, f, w, h, 444, 100, 0)
    assert len(got[0]) * 8 > (w * h * 3 // 64) * 512  # the average block exceeds the slot


@pytest.mark.gpu
def test_status_and_buffer_retry_as_default(hcj, ctx, orc):
    """HCJ_ERR_PLANE_BOUNDS as without the flag; HCJ_ERR_BUFFER_TOO_SMALL reports the optimized file's length (never
    above hcj_encode_bound), and the automatic retry at that length gives the file."""
    with pytest.raises(hcj.HcjError) as e0:
        ctx.encode_batch([synth.frame(1, 17, 16, 420)], 17, 16, 420, 75)
    with pytest.raises(hcj.HcjError) as e1:
        ctx.encode_batch([synth.frame(1, 17, 16, 420)], 17, 16, 420, 75, optimize=True)
    assert e0.value.status == e1.value.status == -10
    w, h = 64, 48
    frames = [np.random.default_rng(i).integers(0, 256, w * h * 3, dtype=np.uint8).tobytes() for i in range(3)]
    want = [expected(orc, f, w, h, 444, 100, 0) for f in frames]
    got, st = ctx.encode_batch(frames, w, h, 444, 100, 0, capacity=200, optimize=True)
    assert st == [-30] * 3
    n = 3
    outs = [np.zeros(200, np.uint8) for _ in range(n)]
    fp = (C.c_void_p * n)(*[np.frombuffer(f, np.uint8).ctypes.data for f in frames])
    keep = [np.frombuffer(f, np.uint8) for f in frames]
    fp = (C.c_void_p * n)(*[k.ctypes.data for k in keep])
    op = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
    caps = (C.c_size_t * n)(*([200] * n))
    lens = (C.c_size_t * n)()
    status = (C.c_int * n)()
    assert hcj.lib().hcj_encode_batch_ex(ctx._h, fp, n, w, h, 444, 100, 0, hcj.ENC_OPTIMIZE_HUFFMAN, op, caps, lens, status) == 0
    assert list(status) == [-30] * n and list(lens) == [len(x) for x in want]
    assert max(lens) <= hcj.lib().hcj_encode_bound(w, h, 444)
    got, st = ctx.encode_batch(frames, w, h, 444, 100, 0, capacity=None, optimize=True)
    assert st == [0] * n and got == want
    assert ctx.encode_batch(frames[:1], w, h, 444, 100, 0, capacity=len(want[0]) - 1, optimize=True)[1] == [-30]


@pytest.mark.gpu
def test_flags_rejected_with_a_context(hcj, ctx):
    w, h = 32, 16
    frame = np.zeros(w * h * 3 // 2, np.uint8)
    out = np.full(4096, 0xA5, np.uint8)
    fp = (C.c_void_p * 1)(frame.ctypes.data)
    op = (C.c_void_p * 1)(out.ctypes.data)
    caps = (C.c_size_t * 1)(4096)
    for flags in (1, 2, 1 << 31):
        lens = (C.c_size_t * 1)(12345)
        status = (C.c_int * 1)(77)
        assert hcj.lib().hcj_encode_batch_ex(ctx._h, fp, 1, w, h, 420, 75, 0, flags, op, caps, lens, status) == -31
        assert (out == 0xA5).all() and lens[0] == 12345 and status[0] == 77
    lens = (C.c_size_t * 1)(12345)
    status = (C.c_int * 1)(77)
    assert hcj.lib().hcj_encode_batch_ex(ctx._h, fp, 1, w, h, 420, 75, 0, hcj.ENC_OPTIMIZE_HUFFMAN, op, caps, lens, status) == 0
    assert status[0] == 0 and out[:2].tobytes() == b"\xff\xd8"


@pytest.mark.gpu
def test_decoded_pixels_equal_default_files(hcj, ctx):
    """hcj_decode_batch of the optimized files equals the decode of the default files, planar and RGB24, through the
    restart-interval decoder (DRI) and the speculative one (no DRI); the optimized files are smaller in total."""
    total0 = total1 = 0
    for chroma, (w, h), ri in ((420, (640, 480), 0), (420, (640, 480), 8), (422, (320, 240), 1), (444, (256, 160), 0), (400, (160, 96), 4)):
        frames = [src_frame(900 + i + chroma, w, h, chroma) for i in range(4)]
        base, st0 = ctx.encode_batch(frames, w, h, chroma, 75, ri)
        opt, st1 = ctx.encode_batch(frames, w, h, chroma, 75, ri, optimize=True)
        assert st0 == st1 == [0] * 4
        total0 += sum(map(len, base))
        total1 += sum(map(len, opt))
        for mode in (hcj.OUT_YUV, hcj.OUT_RGB24, hcj.OUT_PLANES):
            a, sa = ctx.decode_batch(base, mode)
            b, sb = ctx.decode_batch(opt, mode)
            assert sa == sb and (sa == [0] * 4 or (chroma == 400 and mode != hcj.OUT_PLANES))  # (400 has planes only)
            assert all(np.array_equal(x, y) for x, y, s in zip(a, b, sa) if s == 0)
    assert total1 < total0
