"""hcj_encode_rgb_batch / hcj_rgb_to_yuv: RGB24 frames encoded through the device-side forward conversion (K10).

The expected value of every file is a composition of pinned pieces: the stated forward formula (rgb_reference, a literal
int64 restatement), Planar_444.convert_to_420 / _422 (the oracle's subsample_hv2 / _h2) and the encoder (orc.encode,
hcj_encode_batch).  The CPU tier pins the formula against two independent libraries and the whole chain against an
independent decoder; the GPU tier checks the kernel and the three source paths byte for byte."""
import ctypes as C
import io

import numpy as np
import pytest

import synth
from rgb_reference import rgb24_to_frame, rgb24_to_ycbcr, rgb24_to_ycbcr_exact


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


def rgb_frame(seed, w, h):
    """Seeded RGB24 content: three synth planes interleaved, (h, w, 3) uint8."""
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.stack([synth.plane(rng, w, h) for _ in range(3)], axis=-1))


def all_triples():
    """Every (R, G, B) once: a 4096 x 4096 image."""
    i = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(i >> 16) & 255, (i >> 8) & 255, i & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)


# ---- CPU tier -------------------------------------------------------------------------------------------------

def test_forward_formula_over_the_cube(orc):
    """The formula's Y / Cb / Cr for all 2^24 triples: the unclamped values lie in [0, 255] (so the uint8 planes are the
    formula), and each channel is within 1 of OpenCV's COLOR_RGB2YCrCb and of Pillow's convert("YCbCr")."""
    cv2 = pytest.importorskip("cv2")
    Image = pytest.importorskip("PIL.Image")
    img = all_triples()
    exact = rgb24_to_ycbcr_exact(img)
    for want in exact:
        assert want.min() >= 0 and want.max() <= 255
    y, cb, cr = (p.astype(np.uint8) for p in exact)
    del exact
    ocv = cv2.cvtColor(img, cv2.COLOR_RGB2YCrCb)
    pil = np.asarray(Image.fromarray(img, "RGB").convert("YCbCr"))
    for got, k_cv, k_pil in ((y, 0, 0), (cb, 2, 1), (cr, 1, 2)):
        assert np.abs(got.astype(np.int16) - ocv[..., k_cv]).max() <= 1
        assert np.abs(got.astype(np.int16) - pil[..., k_pil]).max() <= 1


def _psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 10 * np.log10(255.0 ** 2 / mse)


@pytest.mark.parametrize("size", [(256, 192), (130, 70)])
def test_standard_jfif_colour_end_to_end(orc, size):
    """An independent decoder (Pillow) reads the chain's files as the input colours: >= 30 dB against the input RGB at q75,
    < 20 dB against the R<->B swapped input (which catches swapped channels or swapped Cb / Cr that the oracle and the
    kernel could share); at 400 the file is a greyscale JPEG."""
    Image = pytest.importorskip("PIL.Image")
    w, h = size
    rgb = rgb_frame(11, w, h)
    for chroma in (444, 422, 420):
        jpg = orc.encode(rgb24_to_frame(orc, rgb, w, h, chroma), w, h, chroma, 75)
        dec = Image.open(io.BytesIO(jpg))
        assert dec.mode == "RGB" and dec.size == (w, h)
        out = np.asarray(dec)
        assert _psnr(out, rgb) >= 30.0, chroma
        assert _psnr(out, rgb[..., ::-1]) < 20.0, chroma
    mono = Image.open(io.BytesIO(orc.encode(rgb24_to_frame(orc, rgb, w, h, 400), w, h, 400, 75)))
    assert mono.mode == "L"


def test_front_end_rejects_malformed_frames(hcj):
    """Shape, dtype, contiguity and mixed kinds are refused before the library is called (no device needed)."""
    w, h = 16, 8
    good = np.zeros((h, w, 3), np.uint8)

    class Dev:
        def __init__(self, shape, typestr="|u1", strides=None):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (0, False), "version": 3, "strides": strides}

    bad = [
        [np.zeros((h, w, 4), np.uint8)],
        [np.zeros((h, w, 3), np.uint16)],
        [np.zeros((h, 2 * w, 3), np.uint8)[:, ::2]],
        [bytes(w * h * 3 - 1)],
        [good, Dev((h, w, 3))],
        [Dev((h, w, 4))],
        [Dev((h, w, 3), "<u2")],
        [Dev((h, w, 3), strides=(w * 6, 3, 1))],
        ["not a frame"],
    ]
    for frames in bad:
        with pytest.raises(ValueError):
            hcj._rgb_frames(frames, w, h)
    ptrs, flags = hcj._rgb_frames([good, bytes(w * h * 3)], w, h)
    assert flags == 0 and len(ptrs) == 2
    ptrs, flags = hcj._rgb_frames([Dev((h, w, 3)), Dev((h, w, 3), strides=(w * 3, 3, 1))], w, h)
    assert flags == hcj.ENC_SRC_DEVICE


# ---- GPU tier -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_conversion_tap_all_triples_444(ctx, orc):
    img = all_triples()
    y, cb, cr = rgb24_to_ycbcr(img)
    assert ctx.rgb_to_yuv(img, 4096, 4096, 444) == y.tobytes() + cb.tobytes() + cr.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("chroma", [420, 422, 400, 444])
@pytest.mark.parametrize("size", [(17, 9), (131, 71), (1366, 768), (1920, 1080), (16, 1), (33, 2), (5, 3)])
def test_conversion_tap_matches_oracle(ctx, orc, chroma, size):
    w, h = size
    rgb = rgb_frame(w * 7 + h, w, h)
    assert ctx.rgb_to_yuv(rgb, w, h, chroma) == rgb24_to_frame(orc, rgb, w, h, chroma)


RGB_CASES = [
    # (chroma, quality, w, h, restart_interval)
    (420, 75, 16, 16, 0), (420, 1, 52, 44, 1), (420, 100, 130, 70, 3), (420, 50, 1366, 768, 8),
    (422, 10, 16, 16, 8), (422, 95, 52, 44, 0), (422, 75, 130, 70, 1), (422, 100, 1366, 768, 3),
    (444, 50, 16, 16, 3), (444, 75, 52, 44, 8), (444, 1, 17, 9, 0), (444, 10, 130, 70, 0), (444, 95, 1366, 768, 1),
    (400, 100, 16, 16, 1), (400, 75, 17, 9, 3), (400, 95, 52, 44, 8), (400, 1, 130, 70, 0), (400, 10, 1366, 768, 0),
    (420, 10, 130, 71, 0), (422, 50, 131, 71, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", RGB_CASES)
def test_encode_rgb_matches_oracle_and_yuv_path(ctx, orc, case):
    """encode_rgb_batch(rgb) == orc.encode(rgb24_to_frame(rgb)) == encode_batch([that frame]), byte for byte."""
    chroma, q, w, h, ri = case
    rgbs = [rgb_frame(700 + i, w, h) for i in range(2)]
    outs, st = ctx.encode_rgb_batch(rgbs, w, h, chroma, q, ri)
    assert st == [0, 0]
    for rgb, o in zip(rgbs, outs):
        planar = rgb24_to_frame(orc, rgb, w, h, chroma)
        want = orc.encode(planar, w, h, chroma, q, restart_interval=ri)
        assert o == want
        yuv, st2 = ctx.encode_batch([planar], w, h, chroma, q, ri)
        assert st2 == [0] and yuv[0] == want


@pytest.fixture(scope="module")
def torch():
    t = pytest.importorskip("torch")
    if not t.cuda.is_available():
        pytest.skip("torch has no CUDA device")
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("size,offset", [((130, 70), 1), ((1366, 768), 0), ((1366, 768), 5), ((64, 48), 3)])
def test_device_source_matches_host(ctx, torch, size, offset):
    """Torch CUDA tensors, including a slice at an odd byte offset of a larger allocation and rows that are not 16-byte
    aligned (1366 * 3 = 4098-byte rows), give the same files as the host path."""
    w, h = size
    rgbs = [rgb_frame(900 + i, w, h) for i in range(3)]
    big = torch.zeros(3 * (w * h * 3 + offset) + 64, dtype=torch.uint8, device="cuda:%d" % ctx.device)
    tens = []
    for i, r in enumerate(rgbs):
        lo = offset + i * (w * h * 3 + offset)
        t = big[lo:lo + w * h * 3].view(h, w, 3)
        t.copy_(torch.from_numpy(r))
        tens.append(t)
    torch.cuda.synchronize()
    for chroma in (420, 444):
        want, st = ctx.encode_rgb_batch(rgbs, w, h, chroma, 75, 0)
        got, st2 = ctx.encode_rgb_batch(tens, w, h, chroma, 75, 0)
        assert st == st2 == [0] * 3 and got == want


def _raw_encode_rgb(hcj, ctx, ptrs, w, h, flags, n_out=None, cap=1 << 16):
    n = len(ptrs)
    outs = [np.full(cap, 0xA5, np.uint8) for _ in range(n_out or n)]
    fp = (C.c_void_p * n)(*ptrs)
    op = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
    caps = (C.c_size_t * n)(*([cap] * n))
    lens = (C.c_size_t * n)(*([12345] * n))
    status = (C.c_int * n)(*([77] * n))
    rc = hcj.lib().hcj_encode_rgb_batch(ctx._h, fp, n, w, h, 420, 75, 0, flags, op, caps, lens, status)
    return rc, outs, list(lens), list(status)


@pytest.mark.gpu
def test_device_flag_rejects_host_pointer_and_unknown_flags(hcj, ctx, torch):
    """A host pointer under HCJ_ENC_SRC_DEVICE, or an unknown flag bit, is HCJ_ERR_INVALID_ARG for the whole call with
    nothing written."""
    w, h = 32, 16
    host = rgb_frame(1, w, h)
    dev = torch.from_numpy(host).to("cuda:%d" % ctx.device)
    torch.cuda.synchronize()
    for ptrs, flags in (([host.ctypes.data], hcj.ENC_SRC_DEVICE), ([dev.data_ptr(), host.ctypes.data], hcj.ENC_SRC_DEVICE),
                        ([host.ctypes.data], 2), ([host.ctypes.data], 1 << 31), ([dev.data_ptr()], hcj.ENC_SRC_DEVICE | 4)):
        rc, outs, lens, status = _raw_encode_rgb(hcj, ctx, ptrs, w, h, flags)
        assert rc == -31  # HCJ_ERR_INVALID_ARG
        assert all((o == 0xA5).all() for o in outs) and lens == [12345] * len(ptrs) and status == [77] * len(ptrs)
    rc, outs, lens, status = _raw_encode_rgb(hcj, ctx, [dev.data_ptr()], w, h, hcj.ENC_SRC_DEVICE)
    assert rc == 0 and status == [0]


@pytest.mark.gpu
def test_device_frame_on_another_gpu_rejected(hcj, ctx, torch):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    w, h = 32, 16
    other = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:%d" % (1 - ctx.device if ctx.device < 2 else 0))
    with pytest.raises(hcj.HcjError) as e:
        ctx.encode_rgb_batch([other], w, h, 420)
    assert e.value.status == -31


@pytest.mark.gpu
def test_every_slot_across_chunks(ctx, orc, torch):
    """130 frames: two full chunks of 64 and a partial one, from host and from device; every file equals the planar
    path's file for the same converted frame."""
    w, h, n = 72, 40, 130
    rgbs = [rgb_frame(2000 + i, w, h) for i in range(n)]
    planar = [rgb24_to_frame(orc, r, w, h, 420) for r in rgbs]
    want, st = ctx.encode_batch(planar, w, h, 420, 75, 2)
    assert st == [0] * n
    host, st = ctx.encode_rgb_batch(rgbs, w, h, 420, 75, 2)
    assert st == [0] * n
    assert [i for i in range(n) if host[i] != want[i]] == []
    # back to back in one pinned-size host buffer (merged uploads)
    block = np.stack(rgbs)
    host2, st = ctx.encode_rgb_batch(list(block), w, h, 420, 75, 2)
    assert st == [0] * n and [i for i in range(n) if host2[i] != want[i]] == []
    dev = torch.from_numpy(block).to("cuda:%d" % ctx.device)
    torch.cuda.synchronize()
    got, st = ctx.encode_rgb_batch([dev[i] for i in range(n)], w, h, 420, 75, 2)
    assert st == [0] * n and [i for i in range(n) if got[i] != want[i]] == []


class _DeviceFrame:
    """Minimal __cuda_array_interface__ over a device address (an RGB24 output of a resident decode batch)."""

    def __init__(self, ptr, w, h):
        self.__cuda_array_interface__ = {"shape": (h, w, 3), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None}


@pytest.mark.gpu
def test_on_device_transcode(hcj, ctx, orc):
    """Decode to RGB24 resident, encode the decoder's device outputs: the same files as encoding the fetched RGB from host."""
    w, h = 200, 120
    jpgs = [orc.encode(synth.frame(3000 + i, w, h, 420), w, h, 420, 90) for i in range(4)]
    with ctx.batch(jpgs, hcj.OUT_RGB24) as b:
        b.decode()
        frames = [_DeviceFrame(b.device_output(i)[0], w, h) for i in range(len(jpgs))]
        for chroma in (420, 444):
            got, st = ctx.encode_rgb_batch(frames, w, h, chroma, 75, 4)
            fetched, st2 = b.fetch()
            assert st2 == [0] * 4
            want, st3 = ctx.encode_rgb_batch([bytes(f) for f in fetched], w, h, chroma, 75, 4)
            assert st == st3 == [0] * 4 and got == want


@pytest.mark.gpu
def test_dense_rgb_exceeds_default_capacity(hcj, ctx, orc):
    """Saturated RGB noise at 4:4:4 q100 needs more than the front-end's default capacity: retried at the reported length."""
    w, h = 245, 137
    rng = np.random.default_rng(30)
    noise = rng.choice([0, 255], (h, w, 3)).astype(np.uint8)
    want = orc.encode(rgb24_to_frame(orc, noise, w, h, 444), w, h, 444, 100)
    assert len(want) > w * h * 3 + (1 << 16)
    assert len(want) <= hcj.lib().hcj_encode_bound(w, h, 444)
    outs, st = ctx.encode_rgb_batch([noise], w, h, 444, 100)
    assert st == [0] and outs == [want]
    outs, st = ctx.encode_rgb_batch([noise], w, h, 444, 100, capacity=len(want) - 1)
    assert st == [-30] and outs == [None]


@pytest.mark.gpu
def test_plane_bounds_status(hcj, ctx, orc):
    """W = 17 at 4:2:0 raises HCJ_ERR_PLANE_BOUNDS, as orc.encode does on the converted frame."""
    rgb = rgb_frame(5, 17, 16)
    with pytest.raises(orc.OracleError) as e:
        orc.encode(rgb24_to_frame(orc, rgb, 17, 16, 420), 17, 16, 420, 75)
    with pytest.raises(hcj.HcjError) as g:
        ctx.encode_rgb_batch([rgb], 17, 16, 420, 75)
    assert g.value.status == e.value.status == -10
