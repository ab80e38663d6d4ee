"""Measures hcj_encode_rgb_batch against hcj_encode_batch on 512 x 1080p 4:2:0 q75 (BASELINE's encode geometry) and
prints one JSON line (also written to --out FILE when given).  Needs a CUDA device; fails without one.

  device_ms    hcj_encode_last_device_ms of the RGB call (device frames) and of the planar call on the converted frames,
               the whole batch as one chunk (HCJ_ENC_CHUNK=512, like bench.py's encode value leg), 3 warm-ups + 10 runs
               each, alternating; medians
  k_rgb_to_ycc its kernel time from torch.profiler (CUDA activities) in a separate run, and its rate by algorithmic bytes:
               3 W H read + the planar frame written, per frame
  e2e_ms       wall clock of the call with default chunking from pinned host RGB (hcj_host_alloc), from torch CUDA
               tensors, and of the planar call from pinned host frames
  parity       every one of the 512 files of both RGB paths equals the planar path's file for the same converted frame
               (checked outside the timed regions)
The frames are 16 seeded RGB images (three synth planes each) repeated over 512 distinct buffers."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "video-coding_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import hcjpeg  # noqa: E402
import synth  # noqa: E402
from rgb_reference import rgb24_to_frame  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402

HBM_COPY_PEAK_GBPS = 6549.0  # measured device-to-device copy rate quoted in DESIGN.md


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    line = subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).splitlines()[0]
    return dict(zip(q.split(","), [s.strip() for s in line.split(",")]))


class Calls:
    """Raw C-ABI calls over fixed pointer arrays (no per-call Python allocation inside the timed regions)."""

    def __init__(self, ctx, n, w, h, cap):
        self.ctx, self.n, self.w, self.h = ctx, n, w, h
        self.out = np.zeros((n, cap), np.uint8)
        self.op = (C.c_void_p * n)(*[self.out[i].ctypes.data for i in range(n)])
        self.caps = (C.c_size_t * n)(*([cap] * n))
        self.lens = (C.c_size_t * n)()
        self.status = (C.c_int * n)()

    def rgb(self, ptrs, flags):
        rc = hcjpeg.lib().hcj_encode_rgb_batch(self.ctx._h, ptrs, self.n, self.w, self.h, 420, 75, 0, flags, self.op, self.caps,
                                               self.lens, self.status)
        assert rc == 0 and all(self.status[i] == 0 for i in range(self.n)), (rc, self.status[0])

    def yuv(self, ptrs):
        rc = hcjpeg.lib().hcj_encode_batch(self.ctx._h, ptrs, self.n, self.w, self.h, 420, 75, 0, self.op, self.caps, self.lens,
                                           self.status)
        assert rc == 0 and all(self.status[i] == 0 for i in range(self.n)), (rc, self.status[0])

    def device_ms(self):
        ms = C.c_float()
        assert hcjpeg.lib().hcj_encode_last_device_ms(self.ctx._h, C.byref(ms)) == 0
        return ms.value

    def files(self):
        return [self.out[i, : self.lens[i]].tobytes() for i in range(self.n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "needs a CUDA device"
    w, h, n = 1920, 1080, a.frames
    fb_rgb, fb_yuv = w * h * 3, w * h * 3 // 2
    res = {"gpu": gpu_info(), "workload": "%d x %dx%d RGB24 -> 4:2:0 q75, restart 0" % (n, w, h)}
    L = hcjpeg.lib()
    rgb_host = L.hcj_host_alloc(n * fb_rgb)
    yuv_host = L.hcj_host_alloc(n * fb_yuv)
    assert rgb_host and yuv_host
    rgb_np = np.ctypeslib.as_array((C.c_uint8 * (n * fb_rgb)).from_address(rgb_host)).reshape(n, h, w, 3)
    yuv_np = np.ctypeslib.as_array((C.c_uint8 * (n * fb_yuv)).from_address(yuv_host)).reshape(n, fb_yuv)
    for k in range(a.distinct):
        rng = np.random.default_rng(7000 + k)
        img = np.stack([synth.plane(rng, w, h) for _ in range(3)], axis=-1)
        planar = np.frombuffer(rgb24_to_frame(orc, img, w, h, 420), np.uint8)
        rgb_np[k::a.distinct] = img
        yuv_np[k::a.distinct] = planar
    dev = torch.from_numpy(rgb_np).to("cuda:0")
    torch.cuda.synchronize()
    p_rgb_host = (C.c_void_p * n)(*[rgb_host + i * fb_rgb for i in range(n)])
    p_yuv_host = (C.c_void_p * n)(*[yuv_host + i * fb_yuv for i in range(n)])
    p_dev = (C.c_void_p * n)(*[dev[i].data_ptr() for i in range(n)])

    with hcjpeg.Context(0) as ctx:
        calls = Calls(ctx, n, w, h, w * h)
        # parity (untimed): planar path is the reference
        calls.yuv(p_yuv_host)
        want = calls.files()
        calls.rgb(p_rgb_host, 0)
        host_ok = calls.files() == want
        calls.rgb(p_dev, hcjpeg.ENC_SRC_DEVICE)
        dev_ok = calls.files() == want
        res["parity"] = {"files": n, "rgb_host_identical": host_ok, "rgb_device_identical": dev_ok,
                         "file_bytes_mean": sum(map(len, want)) / n}

        # device time, one chunk, alternating
        os.environ["HCJ_ENC_CHUNK"] = str(n)
        d_rgb, d_yuv = [], []
        for it in range(13):
            calls.rgb(p_dev, hcjpeg.ENC_SRC_DEVICE)
            r = calls.device_ms()
            calls.yuv(p_yuv_host)
            y = calls.device_ms()
            if it >= 3:
                d_rgb.append(r)
                d_yuv.append(y)
        res["device_ms"] = {"rgb": statistics.median(d_rgb), "yuv": statistics.median(d_yuv),
                            "rgb_runs": d_rgb, "yuv_runs": d_yuv}
        del os.environ["HCJ_ENC_CHUNK"]

        # end to end, default chunking
        def wall(fn, reps=5):
            fn()
            t = []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                t.append((time.perf_counter() - t0) * 1e3)
            return statistics.median(t)

        res["e2e_ms"] = {
            "rgb_host_pinned": wall(lambda: calls.rgb(p_rgb_host, 0)),
            "rgb_device_torch": wall(lambda: calls.rgb(p_dev, hcjpeg.ENC_SRC_DEVICE)),
            "yuv_host_pinned": wall(lambda: calls.yuv(p_yuv_host)),
        }

        # kernel time (separate, profiled run)
        from torch.profiler import ProfilerActivity, profile

        os.environ["HCJ_ENC_CHUNK"] = str(n)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                calls.rgb(p_dev, hcjpeg.ENC_SRC_DEVICE)
        del os.environ["HCJ_ENC_CHUNK"]
        ks = [e for e in prof.events() if "k_rgb_to_ycc" in e.name]
        kms = statistics.median([e.time_range.elapsed_us() for e in ks]) / 1e3
        algo_bytes = n * (fb_rgb + fb_yuv)
        gbps = algo_bytes / (kms * 1e-3) / 1e9
        res["k_rgb_to_ycc"] = {"launches": len(ks), "ms": kms, "algorithmic_GB": algo_bytes / 1e9, "GBps": gbps,
                               "share_of_hbm_copy_peak": gbps / HBM_COPY_PEAK_GBPS, "hbm_copy_peak_GBps": HBM_COPY_PEAK_GBPS}
    del dev
    L.hcj_host_free(C.c_void_p(rgb_host))
    L.hcj_host_free(C.c_void_p(yuv_host))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
