"""hcjpeg — Python host side of the B200 JPEG path (ctypes over the C ABI in include/hcjpeg.h).

The reference's host language is OCaml, which this image does not have; the OCaml stubs live in
``video-coding_b200/ocaml`` (see INTEGRATION.md).  This package is the tested front-end: it mirrors the
reference's ``Decoder`` / ``Encoder`` / ``Frame`` / ``Plane`` interface (same names, argument meaning
and error behaviour; jpeg/model/src/decoder.mli, encoder.mli, common/src/frame.mli) on top of
``libhcjpeg.so``.  There is no CPU fallback: without the CUDA library every call raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.path.join(_ROOT, "lib", "libhcjpeg.so")
if os.environ.get("HCJ_LIB_PATH"):  # A/B measurements of a variant build (make -C csrc OUT=../lib_x EXTRA=-D...)
    LIB_PATH = os.path.abspath(os.environ["HCJ_LIB_PATH"])

OUT_YUV, OUT_PLANES, OUT_RGB24, OUT_YUV444 = 0, 1, 2, 3
FLAG_RESTART_EXT = 1
FLAG_T81_TABLES = 2
FLAG_DEFAULT = FLAG_RESTART_EXT
# Scaled decode (stated extension, include/hcjpeg.h): OR one of these into the decode flags to decode at 1/2, 1/4 or 1/8
# size with libjpeg's reduced IDCTs (what Pillow's Image.draft gives); frame_info(jpeg, flags) reports the scaled frame.
FLAG_SCALE_1_2 = 0x10
FLAG_SCALE_1_4 = 0x20
FLAG_SCALE_1_8 = 0x30
FLAG_SCALE_MASK = 0x30
# libjpeg-turbo's default reconstruction (stated extension, include/hcjpeg.h): islow IDCT and fancy chroma up-sampling, so
# RGB24 equals Pillow / OpenCV.  Not combinable with FLAG_SCALE_*.
FLAG_LIBJPEG = 0x40
ENC_SRC_DEVICE = 1  # hcj_encode_rgb_batch: the frames are device pointers on the context's device

MAX_COMPONENTS = 4
MAX_TABLE_SEGMENTS = 64

STATUS = {
    0: "HCJ_OK",
    -1: "HCJ_ERR_UNSUPPORTED_MARKER",
    -2: "HCJ_ERR_NO_DC_CODE",
    -3: "HCJ_ERR_NO_AC_CODE",
    -4: "HCJ_ERR_COEF_INDEX",
    -5: "HCJ_ERR_NO_COMPONENT",
    -6: "HCJ_ERR_NO_QUANT_TABLE",
    -7: "HCJ_ERR_NO_HUFFMAN_TABLE",
    -8: "HCJ_ERR_NO_FRAME_OR_SCAN",
    -9: "HCJ_ERR_BITS_OUT_OF_BOUNDS",
    -10: "HCJ_ERR_PLANE_BOUNDS",
    -11: "HCJ_ERR_FRAME_INFER",
    -12: "HCJ_ERR_NEED_3_COMPONENTS",
    -13: "HCJ_ERR_ENCODER_PARAMS",
    -20: "HCJ_ERR_NO_TERMINATOR",
    -21: "HCJ_ERR_RESTART_COUNT",
    -22: "HCJ_ERR_UNSUPPORTED_GEOMETRY",
    -23: "HCJ_ERR_DC_RANGE",
    -24: "HCJ_ERR_TRUNCATED",
    -25: "HCJ_ERR_BAD_HUFFMAN_TABLE",
    -30: "HCJ_ERR_BUFFER_TOO_SMALL",
    -31: "HCJ_ERR_INVALID_ARG",
    -32: "HCJ_ERR_OUT_OF_MEMORY",
}


class HcjError(RuntimeError):
    """Raised where the model raises (raise_s / failwith) or CUDA fails; ``status`` is the hcj_status."""

    def __init__(self, status, where=""):
        msg = lib().hcj_strerror(status).decode() if _lib is not None else str(status)
        super().__init__("%s%s (%s, %d)" % (where + ": " if where else "", msg, STATUS.get(status, "CUDA"), status))
        self.status = status


class Component(C.Structure):
    _fields_ = [
        ("identifier", C.c_int),
        ("horizontal_sampling_factor", C.c_int),
        ("vertical_sampling_factor", C.c_int),
        ("quantization_table_identifier", C.c_int),
    ]


class ScanComponent(C.Structure):
    _fields_ = [("selector", C.c_int), ("dc_coef_selector", C.c_int), ("ac_coef_selector", C.c_int)]


class Dqt(C.Structure):
    _fields_ = [("length", C.c_int), ("element_precision", C.c_int), ("table_identifier", C.c_int), ("elements", C.c_int * 64)]


class Dht(C.Structure):
    _fields_ = [
        ("length", C.c_int),
        ("table_class", C.c_int),
        ("destination_identifier", C.c_int),
        ("lengths", C.c_int * 16),
        ("nvalues", C.c_int),
        ("values", C.c_uint8 * 256),
    ]


class Header(C.Structure):
    """Decoder.Header.t (decoder.ml:6-13)."""

    _fields_ = [
        ("has_frame", C.c_int),
        ("sof_length", C.c_int),
        ("sample_precision", C.c_int),
        ("width", C.c_int),
        ("height", C.c_int),
        ("number_of_components", C.c_int),
        ("components", Component * MAX_COMPONENTS),
        ("has_scan", C.c_int),
        ("sos_length", C.c_int),
        ("number_of_image_components", C.c_int),
        ("scan_components", ScanComponent * MAX_COMPONENTS),
        ("start_of_predictor_selection", C.c_int),
        ("end_of_predictor_selection", C.c_int),
        ("successive_approximation_bit_high", C.c_int),
        ("successive_approximation_bit_low", C.c_int),
        ("has_restart_interval", C.c_int),
        ("dri_length", C.c_int),
        ("restart_interval", C.c_int),
        ("n_quant_tables", C.c_int),
        ("quant_tables", Dqt * MAX_TABLE_SEGMENTS),
        ("n_huffman_tables", C.c_int),
        ("huffman_tables", Dht * MAX_TABLE_SEGMENTS),
        ("scan_byte_pos", C.c_int64),
    ]


class FrameInfo(C.Structure):
    _fields_ = [
        ("width", C.c_int),
        ("height", C.c_int),
        ("ncomp", C.c_int),
        ("chroma", C.c_int),
        ("hs", C.c_int * MAX_COMPONENTS),
        ("vs", C.c_int * MAX_COMPONENTS),
        ("decoded_width", C.c_int * MAX_COMPONENTS),
        ("decoded_height", C.c_int * MAX_COMPONENTS),
        ("actual_width", C.c_int * MAX_COMPONENTS),
        ("actual_height", C.c_int * MAX_COMPONENTS),
        ("mcus_wide", C.c_int),
        ("mcus_high", C.c_int),
        ("blocks_per_mcu", C.c_int),
        ("nblocks", C.c_int64),
        ("restart_interval", C.c_int),
        ("yuv_bytes", C.c_size_t),
        ("planes_bytes", C.c_size_t),
        ("rgb_bytes", C.c_size_t),
    ]


# Every entry point include/hcjpeg.h declares: name -> (restype, argtypes)
_P = C.POINTER
_SIGS = {
    "hcj_strerror": (C.c_char_p, [C.c_int]),
    "hcj_version": (C.c_int, []),
    "hcj_header_decode": (C.c_int, [C.c_char_p, C.c_size_t, _P(Header)]),
    "hcj_frame_info_get": (C.c_int, [C.c_char_p, C.c_size_t, _P(FrameInfo)]),
    "hcj_header_decode_ex": (C.c_int, [C.c_char_p, C.c_size_t, C.c_uint, _P(Header)]),
    "hcj_frame_info_get_ex": (C.c_int, [C.c_char_p, C.c_size_t, C.c_uint, _P(FrameInfo)]),
    "hcj_ctx_create": (C.c_int, [C.c_int, C.c_void_p, _P(C.c_void_p)]),
    "hcj_ctx_destroy": (None, [C.c_void_p]),
    "hcj_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "hcj_host_alloc": (C.c_void_p, [C.c_size_t]),
    "hcj_host_free": (None, [C.c_void_p]),
    "hcj_decode_batch": (C.c_int, [C.c_void_p, _P(C.c_void_p), _P(C.c_size_t), C.c_int, C.c_int, C.c_uint, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_decode_batch_multi": (C.c_int, [_P(C.c_void_p), C.c_int, _P(C.c_void_p), _P(C.c_size_t), C.c_int, C.c_int, C.c_uint, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_encode_batch_multi": (C.c_int, [_P(C.c_void_p), C.c_int, _P(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_shard_range": (None, [C.c_int, C.c_int, C.c_int, _P(C.c_int), _P(C.c_int)]),
    "hcj_device_count": (C.c_int, []),
    "hcj_encode_block_log": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p]),
    "hcj_batch_create": (C.c_int, [C.c_void_p, _P(C.c_void_p), _P(C.c_size_t), C.c_int, C.c_int, C.c_uint, _P(C.c_int), _P(C.c_void_p)]),
    "hcj_batch_decode": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hcj_batch_fetch": (C.c_int, [C.c_void_p, C.c_void_p, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_batch_device_output": (C.c_int, [C.c_void_p, C.c_int, _P(C.c_void_p), _P(C.c_size_t)]),
    "hcj_batch_count_kernels": (C.c_int, [C.c_void_p]),
    "hcj_batch_destroy": (None, [C.c_void_p, C.c_void_p]),
    "hcj_batch_fetch_coefficients": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "hcj_batch_fetch_entropy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "hcj_idct_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "hcj_encode_batch": (C.c_int, [C.c_void_p, _P(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_encode_rgb_batch": (C.c_int, [C.c_void_p, _P(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_size_t), _P(C.c_int)]),
    "hcj_rgb_to_yuv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hcj_encode_bound": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "hcj_encode_count_kernels": (C.c_int, []),
    "hcj_write_headers": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "hcj_encode_quantized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hcj_compare_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, _P(C.c_int64), _P(C.c_int)]),
    "hcj_compare_planes_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, _P(C.c_int64), _P(C.c_int), _P(C.c_int64)]),
    "hcj_quant_scale": (C.c_int, [C.c_int, C.c_int, C.c_void_p]),
    "hcj_encoder_code": (C.c_int, [C.c_int, C.c_int, C.c_int, _P(C.c_int), _P(C.c_int)]),
    "hcj_mag": (C.c_int, [C.c_int, C.c_int]),
    "hcj_size": (C.c_int, [C.c_int]),
    "hcj_magnitude": (C.c_int, [C.c_int, C.c_int]),
    "hcj_batch_fetch_block_log": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p]),
    "hcj_decode_a_frame": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.c_int, C.c_uint, C.c_void_p, C.c_size_t]),
    "hcj_mjpeg_split": (C.c_int, [C.c_char_p, C.c_size_t, _P(C.c_size_t), _P(C.c_size_t), C.c_int, _P(C.c_int)]),
    "hcj_decode_stream": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.c_int, C.c_uint, C.c_void_p, C.c_size_t, _P(C.c_size_t), _P(C.c_int), C.c_int, _P(C.c_int)]),
    "hcj_yuv_convert": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t]),
    "hcj_batch_compare": (C.c_int, [C.c_void_p, C.c_void_p, _P(C.c_void_p), _P(C.c_size_t), C.c_void_p]),
    "hcj_batch_decode_stages": (C.c_int, [C.c_void_p, C.c_void_p, _P(C.c_float), C.c_int, _P(C.c_int)]),
    "hcj_decode_stage_name": (C.c_char_p, [C.c_int]),
    "hcj_encode_last_device_ms": (C.c_int, [C.c_void_p, _P(C.c_float)]),
    "hcj_timer_start": (C.c_int, [C.c_void_p]),
    "hcj_timer_stop": (C.c_int, [C.c_void_p, _P(C.c_float)]),
}

BLOCK_LOG_DTYPE = np.dtype([("x", np.int32), ("y", np.int32), ("dc_pred", np.int32), ("component", np.int32),
                            ("coefs", np.int16, 64), ("dequant", np.int32, 64), ("idct", np.int32, 64), ("recon", np.uint8, 64)])


ENCODER_BLOCK_DTYPE = np.dtype([("x_pos", np.int32), ("y_pos", np.int32), ("dc_pred", np.int32), ("component", np.int32),
                                ("nrle", np.int32), ("input_pixels", np.uint8, 64), ("fdct", np.int32, 64), ("quant", np.int16, 64),
                                ("rle_run", np.int16, 64), ("rle_value", np.int16, 64), ("dequant", np.int32, 64),
                                ("idct", np.int32, 64), ("recon", np.uint8, 64), ("error", np.uint8, 64)])


class PlaneMetrics(C.Structure):
    """hcj_plane_metrics: Ocompare results per plane of one image (tools/src/ocompare.ml:8-56)."""
    _fields_ = [("status", C.c_int), ("max_difference", C.c_int * 4), ("square_error", C.c_int64 * 4),
                ("total_difference", C.c_int64 * 4), ("samples", C.c_int64 * 4)]

    def mean_square_error(self, k):
        return self.square_error[k] / self.samples[k]

    def mean_difference(self, k):
        return self.total_difference[k] / self.samples[k]

    def psnr(self, k, r=255.0):
        """Ocompare.psnr (ocompare.ml:54-56): 10 log10(r^2 / mse); inf for identical planes, like the model's float division."""
        import math

        mse = self.mean_square_error(k)
        return math.inf if mse == 0 else 10.0 * math.log10(r * r / mse)


_lib = None


def _source_digest():
    import hashlib

    csrc = os.path.join(_ROOT, "csrc")
    h = hashlib.sha256()
    for f in sorted(os.listdir(csrc)) + [os.path.join(os.path.dirname(_ROOT), "include", "hcjpeg.h")]:
        path = f if os.path.isabs(f) else os.path.join(csrc, f)
        h.update(os.path.basename(path).encode())
        with open(path, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force=False):
    """Compile libhcjpeg.so for sm_100a with the committed Makefile (nvcc cross-compiles without a GPU).
    The library is rebuilt when the sources differ from the ones it was built from (a content stamp next to
    it: file times do not survive being copied to another machine)."""
    if os.environ.get("HCJ_LIB_PATH"):
        return LIB_PATH  # a variant build made by hand
    csrc = os.path.join(_ROOT, "csrc")
    stamp = LIB_PATH + ".stamp"
    digest = _source_digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB_PATH
    subprocess.check_call(["make", "-s", "-C", csrc, "-B"] if os.path.exists(LIB_PATH) else ["make", "-s", "-C", csrc])
    with open(stamp, "w") as f:
        f.write(digest + "\n")
    return LIB_PATH


def lib():
    """The loaded C-ABI library; fails loudly if it has not been built (there is nothing to fall back to)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libhcjpeg.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'`" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _check(status, where=""):
    if status != 0:
        raise HcjError(status, where)


def _ptr_array(bufs):
    arr = (C.c_void_p * max(len(bufs), 1))()
    keep = []
    for i, b in enumerate(bufs):
        if isinstance(b, np.ndarray):
            arr[i] = b.ctypes.data
            keep.append(b)
        elif isinstance(b, int):
            arr[i] = b
        else:
            cb = (C.c_char * len(b)).from_buffer_copy(b) if len(b) else (C.c_char * 1)()
            arr[i] = C.addressof(cb)
            keep.append(cb)
    return arr, keep


def _rgb_frames(frames, width, height, allow_device=True):
    """Checks RGB24 frames before the library sees them: ([uint8 array, or device address as int], flags).  Host frames:
    bytes of width*height*3, or C-contiguous uint8 arrays of shape (height, width, 3); device frames: objects with
    __cuda_array_interface__ of that shape, dtype and (C-contiguous) layout.  All frames of one call are of one kind."""
    dev = [hasattr(f, "__cuda_array_interface__") for f in frames]
    if any(dev) and not all(dev):
        raise ValueError("RGB frames: all host frames or all device frames in one call")
    if any(dev) and not allow_device:
        raise ValueError("RGB frames: a host frame is required here")
    shape = (height, width, 3)
    out = []
    for f in frames:
        if dev and dev[0]:
            cai = f.__cuda_array_interface__
            strides = cai.get("strides")
            if tuple(cai["shape"]) != shape or np.dtype(cai["typestr"]) != np.uint8:
                raise ValueError("RGB frame: need uint8 of shape %s, got %s %s" % (shape, cai["typestr"], tuple(cai["shape"])))
            if strides is not None and tuple(strides) != (width * 3, 3, 1):
                raise ValueError("RGB frame: not C-contiguous (strides %s)" % (tuple(strides),))
            out.append(int(cai["data"][0]))
        elif isinstance(f, np.ndarray):
            if f.dtype != np.uint8 or f.shape != shape or not f.flags["C_CONTIGUOUS"]:
                raise ValueError("RGB frame: need a C-contiguous uint8 array of shape %s, got %s %s" % (shape, f.dtype, f.shape))
            out.append(f)
        elif isinstance(f, (bytes, bytearray)):
            if len(f) != width * height * 3:
                raise ValueError("RGB frame: need %d bytes, got %d" % (width * height * 3, len(f)))
            out.append(np.frombuffer(f, np.uint8))
        else:
            raise ValueError("RGB frame: bytes, a uint8 array or an object with __cuda_array_interface__, got %s" % type(f).__name__)
    return out, (ENC_SRC_DEVICE if dev and dev[0] else 0)


def header_decode(jpeg, flags=0):
    """Decoder.Header.decode (decoder.ml:37-70); flags=FLAG_T81_TABLES reads every table of a DQT / DHT segment."""
    h = Header()
    _check(lib().hcj_header_decode_ex(jpeg, len(jpeg), flags, C.byref(h)), "Header.decode")
    return h


def frame_info(jpeg, flags=FLAG_DEFAULT):
    """Geometry fixed by Decoder.init (decoder.ml:304-345).  With FLAG_SCALE_* in ``flags``: the scaled frame (width,
    height, planes and output sizes of the 1/s decode; the block geometry stays that of the file)."""
    f = FrameInfo()
    _check(lib().hcj_frame_info_get_ex(jpeg, len(jpeg), flags, C.byref(f)), "Decoder.init")
    return f


def mjpeg_split(stream):
    """Frame boundaries [(offset, length)] of a Motion-JPEG stream (whole JPEG files back to back)."""
    n = C.c_int()
    _check(lib().hcj_mjpeg_split(stream, len(stream), None, None, 0, C.byref(n)), "hcj_mjpeg_split")
    off, ln = (C.c_size_t * max(n.value, 1))(), (C.c_size_t * max(n.value, 1))()
    _check(lib().hcj_mjpeg_split(stream, len(stream), off, ln, n.value, C.byref(n)), "hcj_mjpeg_split")
    return [(off[i], ln[i]) for i in range(n.value)]


def out_size(info, mode):
    return {OUT_YUV: info.yuv_bytes, OUT_PLANES: info.planes_bytes, OUT_RGB24: info.rgb_bytes, OUT_YUV444: info.rgb_bytes}[mode]


class Context:
    """One per GPU.  ``stream`` may be a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""

    def __init__(self, device=0, stream=None):
        self._h = C.c_void_p()
        _check(lib().hcj_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self._h)), "hcj_ctx_create")
        self.device = device

    def close(self):
        if self._h:
            lib().hcj_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        _check(lib().hcj_ctx_synchronize(self._h))

    def timer_start(self):
        _check(lib().hcj_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float()
        _check(lib().hcj_timer_stop(self._h, C.byref(ms)))
        return ms.value

    # ---- decode -----------------------------------------------------------------------------
    def decode_batch(self, jpegs, mode=OUT_YUV, flags=FLAG_DEFAULT, raise_on_error=False):
        """Decoder.decode_a_frame for every element of ``jpegs`` (bytes).  Returns (outputs, status):
        outputs[i] is a uint8 array (None where status[i] != 0).  Outputs are sized by frame_info(jpeg, flags), so a
        FLAG_SCALE_* in ``flags`` (here and in every decode entry point) gives the scaled frames."""
        n = len(jpegs)
        infos, caps, outs = [], [], []
        for j in jpegs:
            f = FrameInfo()
            st = lib().hcj_frame_info_get_ex(j, len(j), flags, C.byref(f))
            size = out_size(f, mode) if st == 0 else 0
            infos.append(f if st == 0 else None)
            caps.append(size)
            outs.append(np.zeros(max(size, 1), np.uint8))
        jp, keep = _ptr_array(jpegs)
        lens = (C.c_size_t * max(n, 1))(*[len(j) for j in jpegs])
        op, keep2 = _ptr_array(outs)
        capa = (C.c_size_t * max(n, 1))(*caps)
        status = (C.c_int * max(n, 1))()
        _check(lib().hcj_decode_batch(self._h, jp, lens, n, mode, flags, op, capa, status), "hcj_decode_batch")
        st = [status[i] for i in range(n)]
        if raise_on_error:
            for s in st:
                _check(s, "Decoder.decode_a_frame")
        return [outs[i][: caps[i]] if st[i] == 0 else None for i in range(n)], st

    def decode_a_frame(self, jpeg, mode=OUT_YUV, flags=FLAG_DEFAULT):
        """Decoder.decode_a_frame (decoder.ml:422-427): the frame as a uint8 array; raises HcjError like the model raises."""
        f = frame_info(jpeg, flags)
        out = np.zeros(max(out_size(f, mode), 1), np.uint8)
        _check(lib().hcj_decode_a_frame(self._h, jpeg, len(jpeg), mode, flags, out.ctypes.data, out.size), "Decoder.decode_a_frame")
        return out[: out_size(f, mode)]

    def decode_stream(self, stream, mode=OUT_YUV, flags=FLAG_DEFAULT):
        """Every frame of a Motion-JPEG stream: (frames, status), frames[i] a uint8 array (None where status[i] != 0)."""
        frames = mjpeg_split(stream)
        n = len(frames)
        total = 0
        for o, l in frames:
            f = FrameInfo()
            if lib().hcj_frame_info_get_ex(stream[o:o + l], l, flags, C.byref(f)) == 0:
                total += (out_size(f, mode) + 255) & ~255
        out = np.zeros(max(total, 1), np.uint8)
        offs, status, nf = (C.c_size_t * (n + 1))(), (C.c_int * max(n, 1))(), C.c_int()
        _check(lib().hcj_decode_stream(self._h, stream, len(stream), mode, flags, out.ctypes.data, out.size, offs, status, n, C.byref(nf)), "hcj_decode_stream")
        assert nf.value == n
        res = []
        for i, (o, l) in enumerate(frames):
            f = FrameInfo()
            ok = status[i] == 0 and lib().hcj_frame_info_get_ex(stream[o:o + l], l, flags, C.byref(f)) == 0
            res.append(out[offs[i]: offs[i] + out_size(f, mode)] if ok else None)
        return res, [status[i] for i in range(n)]

    def batch(self, jpegs, mode=OUT_YUV, flags=FLAG_DEFAULT):
        return Batch(self, jpegs, mode, flags)

    def idct_blocks(self, coefs, quant_table):
        """Component.recon for caller-provided zig-zag blocks (DC absolute)."""
        coefs = np.ascontiguousarray(coefs, np.int16).reshape(-1, 64)
        qt = np.ascontiguousarray(quant_table, np.uint16).reshape(64)
        out = np.zeros((coefs.shape[0], 64), np.uint8)
        _check(lib().hcj_idct_blocks(self._h, coefs.ctypes.data, coefs.shape[0], qt.ctypes.data, out.ctypes.data), "hcj_idct_blocks")
        return out

    # ---- encode -----------------------------------------------------------------------------
    def encode_batch(self, frames, width, height, chroma=420, quality=75, restart_interval=0, capacity=None):
        """Encoder.encode_420/422/444 for every raw planar frame (bytes / uint8 arrays) in ``frames``."""
        return self._encode(frames, None, width, height, chroma, quality, restart_interval, capacity)

    def encode_rgb_batch(self, frames, width, height, chroma=420, quality=75, restart_interval=0, capacity=None):
        """hcj_encode_rgb_batch: every RGB24 frame converted and sub-sampled to ``chroma`` on the device (the stated forward
        formula, include/hcjpeg.h) and encoded as encode_batch encodes that planar frame.  ``frames``: all host frames
        (bytes of width*height*3, or C-contiguous uint8 arrays of shape (height, width, 3)) or all device frames (objects
        with ``__cuda_array_interface__`` of that shape, e.g. torch CUDA tensors, read on the context's stream).
        Returns (files, status) like encode_batch."""
        ptrs, flags = _rgb_frames(frames, width, height)
        return self._encode(ptrs, flags, width, height, chroma, quality, restart_interval, capacity)

    def _encode(self, frames, rgb_flags, width, height, chroma, quality, restart_interval, capacity):
        """hcj_encode_batch (rgb_flags None) or hcj_encode_rgb_batch with those flags."""
        n = len(frames)
        auto = capacity is None
        if auto:
            capacity = width * height * 3 + (1 << 16)  # above any natural frame; hcj_encode_bound is the hard bound
        outs = [np.zeros(capacity, np.uint8) for _ in range(n)]
        fp, keep = _ptr_array(frames)
        op, keep2 = _ptr_array(outs)
        caps = (C.c_size_t * max(n, 1))(*([capacity] * n))
        lens = (C.c_size_t * max(n, 1))()
        status = (C.c_int * max(n, 1))()
        if rgb_flags is None:
            _check(
                lib().hcj_encode_batch(self._h, fp, n, width, height, chroma, quality, restart_interval, op, caps, lens, status),
                "hcj_encode_batch",
            )
        else:
            _check(
                lib().hcj_encode_rgb_batch(self._h, fp, n, width, height, chroma, quality, restart_interval, rgb_flags, op, caps,
                                           lens, status),
                "hcj_encode_rgb_batch",
            )
        st = [status[i] for i in range(n)]
        res = [outs[i][: lens[i]].tobytes() if st[i] == 0 else None for i in range(n)]
        # The default capacity is a guess (dense 4:4:4 content at quality 100 exceeds 3 bytes per pixel); the library
        # reports the length a frame needs with HCJ_ERR_BUFFER_TOO_SMALL, so those frames go through once more at that size.
        redo = [i for i in range(n) if st[i] == -30] if auto else []
        if redo:
            again, st2 = self._encode(
                [frames[i] for i in redo], rgb_flags, width, height, chroma, quality, restart_interval, max(lens[i] for i in redo)
            )
            for i, o, s2 in zip(redo, again, st2):
                res[i], st[i] = o, s2
        return res, st

    def rgb_to_yuv(self, frame, width, height, chroma=420):
        """hcj_rgb_to_yuv: the planar frame (bytes) that encode_rgb_batch encodes for one host RGB24 frame."""
        (p,), _ = _rgb_frames([frame], width, height, allow_device=False)
        cw = width if chroma == 444 else width // 2
        ch = height // 2 if chroma == 420 else height
        out = np.zeros(width * height + (0 if chroma == 400 else 2 * cw * ch), np.uint8)
        _check(lib().hcj_rgb_to_yuv(self._h, p if isinstance(p, int) else p.ctypes.data, width, height, chroma, out.ctypes.data, out.size),
               "hcj_rgb_to_yuv")
        return out.tobytes()

    def encode_quantized(self, frame, width, height, chroma=420, quality=75):
        """Block.quant of every block in encode_seq order (encoder.ml:56-66)."""
        f = FrameInfo()
        hdr = write_headers(width, height, chroma, quality) + b"\xff\xd9"
        _check(lib().hcj_frame_info_get(hdr, len(hdr), C.byref(f)))
        out = np.zeros((f.nblocks, 64), np.int16)
        buf = np.frombuffer(frame, np.uint8)
        _check(lib().hcj_encode_quantized(self._h, buf.ctypes.data, width, height, chroma, quality, out.ctypes.data, f.nblocks), "hcj_encode_quantized")
        return out

    def encode_block_log(self, frame, width, height, chroma=420, quality=75, restart_interval=0, first=0, count=None):
        """`model encode log -verbose`: Encoder.Block.t of blocks [first, first + count) in encode_seq order as a structured
        array (x_pos, y_pos, dc_pred, component, nrle, input_pixels, fdct, quant, rle_run, rle_value, dequant, idct, recon, error)."""
        if count is None:
            f = FrameInfo()
            hdr = write_headers(width, height, chroma, quality) + b"\xff\xd9"
            _check(lib().hcj_frame_info_get(hdr, len(hdr), C.byref(f)))
            count = f.nblocks - first
        out = np.zeros(max(count, 1), ENCODER_BLOCK_DTYPE)
        buf = np.frombuffer(frame, np.uint8)
        _check(lib().hcj_encode_block_log(self._h, buf.ctypes.data, width, height, chroma, quality, restart_interval, first, count,
                                          out.ctypes.data), "hcj_encode_block_log")
        return out[:count]

    def yuv_convert(self, frame, width, height, chroma, dst_width=None, dst_height=None, dst_chroma=444, x_off=0, y_off=0):
        """`oyuv convert`: planar frame -> 4:4:4 -> crop with edge clamp -> dst_chroma, on the device."""
        dw, dh = dst_width or width, dst_height or height
        cw, ch = (dw if dst_chroma == 444 else dw // 2), (dh // 2 if dst_chroma == 420 else dh)
        out = np.zeros(dw * dh + 2 * cw * ch, np.uint8)
        src = np.frombuffer(frame, np.uint8)
        _check(lib().hcj_yuv_convert(self._h, src.ctypes.data, width, height, chroma, x_off, y_off, out.ctypes.data, dw, dh, dst_chroma, out.size), "hcj_yuv_convert")
        return out

    def compare_planes(self, a, b):
        """Ocompare.square_error / max_difference (tools/src/ocompare.ml:8-52) on the device."""
        a = np.ascontiguousarray(a, np.uint8).ravel()
        b = np.ascontiguousarray(b, np.uint8).ravel()
        assert a.size == b.size
        sse, mx = C.c_int64(), C.c_int()
        _check(lib().hcj_compare_planes(self._h, a.ctypes.data, b.ctypes.data, a.size, C.byref(sse), C.byref(mx)))
        return sse.value, mx.value

    def compare_planes_ex(self, a, b):
        """(square_error, max_difference, total_difference) of two planes (tools/src/ocompare.ml:8-52) on the device."""
        a = np.ascontiguousarray(a, np.uint8).ravel()
        b = np.ascontiguousarray(b, np.uint8).ravel()
        assert a.size == b.size
        sse, mx, tot = C.c_int64(), C.c_int(), C.c_int64()
        _check(lib().hcj_compare_planes_ex(self._h, a.ctypes.data, b.ctypes.data, a.size, C.byref(sse), C.byref(mx), C.byref(tot)))
        return sse.value, mx.value, tot.value


def device_count():
    """CUDA devices visible to the process."""
    return lib().hcj_device_count()


def shard_range(n, part, nparts):
    """Batch indices [lo, hi) that part `part` of `nparts` handles (hcj_shard_range)."""
    lo, hi = C.c_int(), C.c_int()
    lib().hcj_shard_range(n, part, nparts, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def decode_batch_multi(ctxs, jpegs, mode=OUT_YUV, flags=FLAG_DEFAULT):
    """hcj_decode_batch_multi: one process, one Context per GPU, images sharded by batch index over them (a host thread
    per context inside the library).  Returns (outputs, status) like Context.decode_batch."""
    n = len(jpegs)
    caps, outs = [], []
    for j in jpegs:
        f = FrameInfo()
        st = lib().hcj_frame_info_get_ex(j, len(j), flags, C.byref(f))
        caps.append(out_size(f, mode) if st == 0 else 0)
        outs.append(np.zeros(max(caps[-1], 1), np.uint8))
    jp, keep = _ptr_array(jpegs)
    lens = (C.c_size_t * max(n, 1))(*[len(j) for j in jpegs])
    op, keep2 = _ptr_array(outs)
    capa = (C.c_size_t * max(n, 1))(*caps)
    status = (C.c_int * max(n, 1))()
    hs = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    _check(lib().hcj_decode_batch_multi(hs, len(ctxs), jp, lens, n, mode, flags, op, capa, status), "hcj_decode_batch_multi")
    st = [status[i] for i in range(n)]
    return [outs[i][: caps[i]] if st[i] == 0 else None for i in range(n)], st


def encode_batch_multi(ctxs, frames, width, height, chroma=420, quality=75, restart_interval=0):
    """hcj_encode_batch_multi: frames sharded by index over one Context per GPU."""
    n = len(frames)
    capacity = lib().hcj_encode_bound(width, height, chroma) if n <= 64 else width * height * 3 + (1 << 16)
    outs = [np.zeros(capacity, np.uint8) for _ in range(n)]
    fp, keep = _ptr_array(frames)
    op, keep2 = _ptr_array(outs)
    caps = (C.c_size_t * max(n, 1))(*([capacity] * n))
    lens = (C.c_size_t * max(n, 1))()
    status = (C.c_int * max(n, 1))()
    hs = (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
    _check(lib().hcj_encode_batch_multi(hs, len(ctxs), fp, n, width, height, chroma, quality, restart_interval, op, caps, lens, status),
           "hcj_encode_batch_multi")
    st = [status[i] for i in range(n)]
    return [outs[i][: lens[i]].tobytes() if st[i] == 0 else None for i in range(n)], st


class Batch:
    """Device-resident decode batch: create (parse + H2D) / decode (kernels) / fetch (D2H)."""

    def __init__(self, ctx, jpegs, mode=OUT_YUV, flags=FLAG_DEFAULT):
        self.ctx, self.mode, self.n = ctx, mode, len(jpegs)
        self._jp, self._keep = _ptr_array(jpegs)
        lens = (C.c_size_t * max(self.n, 1))(*[len(j) for j in jpegs])
        self._status = (C.c_int * max(self.n, 1))()
        self._h = C.c_void_p()
        _check(lib().hcj_batch_create(ctx._h, self._jp, lens, self.n, mode, flags, self._status, C.byref(self._h)), "hcj_batch_create")
        self.host_status = [self._status[i] for i in range(self.n)]
        self.infos = []
        for j in jpegs:
            f = FrameInfo()
            self.infos.append(f if lib().hcj_frame_info_get_ex(j, len(j), flags, C.byref(f)) == 0 else None)

    def decode(self):
        _check(lib().hcj_batch_decode(self.ctx._h, self._h), "hcj_batch_decode")

    def kernels(self):
        return lib().hcj_batch_count_kernels(self._h)

    def decode_stages(self):
        """One decode pass timed stage by stage with CUDA events: {stage name: ms}."""
        ms = (C.c_float * 8)()
        n = C.c_int()
        _check(lib().hcj_batch_decode_stages(self.ctx._h, self._h, ms, 8, C.byref(n)), "hcj_batch_decode_stages")
        return {lib().hcj_decode_stage_name(i).decode(): ms[i] for i in range(n.value)}

    def fetch(self, outs=None):
        caps = [out_size(f, self.mode) if f is not None else 0 for f in self.infos]
        if outs is None:
            outs = [np.zeros(max(c, 1), np.uint8) for c in caps]
        op, keep = _ptr_array(outs)
        capa = (C.c_size_t * max(self.n, 1))(*caps)
        status = (C.c_int * max(self.n, 1))()
        _check(lib().hcj_batch_fetch(self.ctx._h, self._h, op, capa, status), "hcj_batch_fetch")
        st = [status[i] for i in range(self.n)]
        return [outs[i][: caps[i]] if st[i] == 0 else None for i in range(self.n)], st

    def compare(self, refs):
        """`oyuv compare` of every decoded image (resident in HBM) with refs[i] (bytes in the batch's output layout):
        a PlaneMetrics per image."""
        assert len(refs) == self.n
        bufs = [np.frombuffer(r, np.uint8) if r is not None else np.zeros(1, np.uint8) for r in refs]
        rp, keep = _ptr_array(bufs)
        lens = (C.c_size_t * max(self.n, 1))(*[len(r) if r is not None else 0 for r in refs])
        out = (PlaneMetrics * max(self.n, 1))()
        _check(lib().hcj_batch_compare(self.ctx._h, self._h, rp, lens, out), "hcj_batch_compare")
        return [out[i] for i in range(self.n)]

    def coefficients(self, i):
        """Component.coefs of image i (int16 zig-zag, DC resolved), decode_seq order."""
        nb = self.infos[i].nblocks
        out = np.zeros((nb, 64), np.int16)
        _check(lib().hcj_batch_fetch_coefficients(self.ctx._h, self._h, i, out.ctypes.data, nb), "coefficients")
        return out

    def block_log(self, i, first=0, count=None):
        """`model decode log`: Decoder.Component.Summary of blocks [first, first + count) of image i as a structured array
        (fields x, y, dc_pred, component, coefs, dequant, idct, recon)."""
        count = self.infos[i].nblocks - first if count is None else count
        out = np.zeros(max(count, 1), BLOCK_LOG_DTYPE)
        _check(lib().hcj_batch_fetch_block_log(self.ctx._h, self._h, i, first, count, out.ctypes.data), "block_log")
        return out[:count]

    def entropy(self, i):
        """For_testing.extract_entropy_coded_bits of image i."""
        cap = 1 << 26
        out = np.zeros(cap, np.uint8)
        n = C.c_size_t()
        _check(lib().hcj_batch_fetch_entropy(self.ctx._h, self._h, i, out.ctypes.data, cap, C.byref(n)), "entropy")
        return out[: n.value].tobytes()

    def device_output(self, i):
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib().hcj_batch_device_output(self._h, i, C.byref(p), C.byref(n)))
        return p.value, n.value

    def close(self):
        if self._h:
            lib().hcj_batch_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def write_headers(width, height, chroma=420, quality=75, restart_interval=0):
    """Encoder.write_headers (encoder.ml:371-418)."""
    buf = np.zeros(2048, np.uint8)
    n = C.c_size_t()
    _check(lib().hcj_write_headers(width, height, chroma, quality, restart_interval, buf.ctypes.data, buf.size, C.byref(n)), "write_headers")
    return buf[: n.value].tobytes()
