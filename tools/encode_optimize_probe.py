"""Measures HCJ_ENC_OPTIMIZE_HUFFMAN against the default tables on 512 x 1080p 4:2:0 q75 (bench.py's encode frames,
bench.make_frames) and prints one JSON line (also written to --out FILE when given).  Needs a CUDA device; fails without
one.

  gpu          card name, power limit and maximum SM clock (read-only nvidia-smi query)
  device_ms    hcj_encode_last_device_ms of the planar call with and without the flag, the whole batch as one chunk
               (HCJ_ENC_CHUNK=512, like bench.py's encode value leg), 3 warm-ups + 10 runs each, alternating; medians
  e2e_ms       wall clock of the call with default chunking from pinned host frames (hcj_host_alloc), with and without
               the flag, alternating, medians of 10
  kernels_ms   per-kernel time from torch.profiler (CUDA activities) in a separate run, median over the launches
  bytes        total file bytes with and without the flag, and their ratio
  rgb          the same device_ms / e2e_ms / bytes for RGB24 frames from torch device tensors (hcj_encode_rgb_batch)
  parity       the first --check files of the flag equal the reference (tests/optimal_huffman_reference.py)"""
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

import bench  # noqa: E402
import hcjpeg  # noqa: E402
import synth  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402
from optimal_huffman_reference import optimized_file  # noqa: E402
from rgb_reference import rgb24_to_frame  # noqa: E402


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

    def yuv(self, ptrs, flags):
        rc = hcjpeg.lib().hcj_encode_batch_ex(self.ctx._h, ptrs, self.n, self.w, self.h, 420, 75, 0, flags, self.op, self.caps,
                                              self.lens, self.status)
        assert rc == 0 and all(self.status[i] == 0 for i in range(self.n)), (rc, self.status[0])

    def rgb(self, ptrs, flags):
        rc = hcjpeg.lib().hcj_encode_rgb_batch(self.ctx._h, ptrs, self.n, self.w, self.h, 420, 75, 0, flags, self.op, self.caps,
                                               self.lens, self.status)
        assert rc == 0 and all(self.status[i] == 0 for i in range(self.n)), (rc, self.status[0])

    def device_ms(self):
        ms = C.c_float()
        assert hcjpeg.lib().hcj_encode_last_device_ms(self.ctx._h, C.byref(ms)) == 0
        return ms.value

    def files(self):
        return [self.out[i, : self.lens[i]].tobytes() for i in range(self.n)]

    def total(self):
        return sum(self.lens[i] for i in range(self.n))


def alternate(a, b, measure, runs=10, warm=3):
    """Medians of measure() after a() and after b(), alternating."""
    ra, rb = [], []
    for it in range(warm + runs):
        a()
        x = measure()
        b()
        y = measure()
        if it >= warm:
            ra.append(x)
            rb.append(y)
    return statistics.median(ra), statistics.median(rb), ra, rb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--check", type=int, default=8)
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "needs a CUDA device"
    w, h, n = 1920, 1080, a.frames
    fb = w * h * 3 // 2
    frames = bench.make_frames(n, w, h, 420, 0)
    res = {"gpu": gpu_info(), "workload": "%d x %dx%d 4:2:0 q75, restart 0 (bench.make_frames)" % (n, w, h)}
    L = hcjpeg.lib()
    host = L.hcj_host_alloc(n * fb)
    assert host
    host_np = np.ctypeslib.as_array((C.c_uint8 * (n * fb)).from_address(host)).reshape(n, fb)
    for i, f in enumerate(frames):
        host_np[i] = np.frombuffer(f, np.uint8)
    ptrs = (C.c_void_p * n)(*[host + i * fb for i in range(n)])
    OPT = hcjpeg.ENC_OPTIMIZE_HUFFMAN
    with hcjpeg.Context(0) as ctx:
        calls = Calls(ctx, n, w, h, w * h * 2)
        calls.yuv(ptrs, OPT)
        got = calls.files()[: a.check]
        parity = [got[i] == optimized_file(orc.encode(frames[i], w, h, 420, 75, 0)) for i in range(a.check)]

        # the timed legs: the two kinds of call alternate, device time and wall time in separate loops
        res["planar"] = leg(calls, calls.yuv, ptrs, 0)

        from torch.profiler import ProfilerActivity, profile

        os.environ["HCJ_ENC_CHUNK"] = str(n)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                calls.yuv(ptrs, OPT)
        del os.environ["HCJ_ENC_CHUNK"]
        per = {}
        for e in prof.events():
            if e.name.startswith("void hcjk::k_") or "hcjk::k_" in e.name:
                k = e.name.split("hcjk::")[1].split("(")[0].split("<")[0]
                per.setdefault(k, []).append(e.time_range.elapsed_us() / 1e3)
        res["kernels_ms"] = {k: statistics.median(v) for k, v in sorted(per.items())}

        # RGB24 from device tensors: the first 16 frames' RGB images, repeated
        rgb = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
        imgs = []
        for k in range(16):
            rng = np.random.default_rng(7000 + k)
            imgs.append(np.stack([synth.plane(rng, w, h) for _ in range(3)], axis=-1))
        for i in range(n):
            rgb[i].copy_(torch.from_numpy(imgs[i % 16]))
        torch.cuda.synchronize()
        p_dev = (C.c_void_p * n)(*[rgb[i].data_ptr() for i in range(n)])
        calls.rgb(p_dev, hcjpeg.ENC_SRC_DEVICE | OPT)
        got = calls.files()
        parity += [got[i] == optimized_file(orc.encode(rgb24_to_frame(orc, imgs[i], w, h, 420), w, h, 420, 75, 0))
                   for i in range(2)]
        res["rgb_device"] = leg(calls, calls.rgb, p_dev, hcjpeg.ENC_SRC_DEVICE)
        res["parity"] = {"files_checked": len(parity), "identical": all(parity)}
        del rgb
    L.hcj_host_free(C.c_void_p(host))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


def leg(calls, call, ptrs, flags):
    """device_ms (one chunk), e2e_ms (default chunking) and total bytes of one source, default vs optimize, alternating."""
    OPT = hcjpeg.ENC_OPTIMIZE_HUFFMAN
    out = {}
    os.environ["HCJ_ENC_CHUNK"] = str(calls.n)
    dd, do, rd, ro = alternate(lambda: call(ptrs, flags), lambda: call(ptrs, flags | OPT), calls.device_ms)
    del os.environ["HCJ_ENC_CHUNK"]
    out["device_ms"] = {"default": dd, "optimize": do, "default_runs": rd, "optimize_runs": ro}
    walls = {"a": [], "b": []}
    for it in range(13):
        for key, f in (("a", flags), ("b", flags | OPT)):
            t0 = time.perf_counter()
            call(ptrs, f)
            if it >= 3:
                walls[key].append((time.perf_counter() - t0) * 1e3)
    out["e2e_ms"] = {"default": statistics.median(walls["a"]), "optimize": statistics.median(walls["b"])}
    call(ptrs, flags)
    b0 = calls.total()
    call(ptrs, flags | OPT)
    b1 = calls.total()
    out["bytes"] = {"default": int(b0), "optimize": int(b1), "ratio": b1 / b0}
    return out


if __name__ == "__main__":
    main()
