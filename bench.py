#!/usr/bin/env python3
"""bench.py — decoded megapixels/sec of the B200 JPEG path (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--only]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the reference's CPU algorithm (oracle port) on the host cores
    python bench.py --dump-outputs DIR        # also write a seeded sample of every workload's outputs to DIR/<name>.npy

A step = one pass of the hot path over one batch of synthetic images.  The headline workload (`--workload`,
default restart8 = BASELINE configs[1]) fills the top-level keys of the JSON line:
  value   whole-job MP/s with the compressed batch already resident in HBM (kernels only), CUDA events on the
          library's stream, max over ranks;
  e2e     the same metric through hcj_decode_batch with pinned HOST buffers: header parse, H2D of the files,
          kernels, D2H of the frames, all inside the timed region (wall clock around the call);
  roofline  algorithmic bytes of the dominant kernel / its CUDA-event duration vs MEASURED_PEAKS.json;
  cpu_baseline  the CPU oracle (a port of the OCaml model) on the host cores, one process per core, on a bounded
          sample of the same images.
Unless --only is given the other BASELINE configs are timed in the same run (3 warm-ups, <= 10 steps each) and
reported under "workloads": norestart (configs[2]: 8192 images over the ranks when N > 1), 4k444rgb (configs[3]),
encode (configs[4]), plus restart8rgb and restart120 (one MCU row per restart interval: the no-cliff check).
Every workload is checked against the oracle outside its timed region ("parity_checked": images compared bit for bit).
Images are sharded by batch index (weak scaling: a fixed batch per GPU), no collective on the data path.
The inputs are seeded, so the same arguments give the same images on every run and `--dump-outputs` files of two builds
can be compared value for value.
The synthetic JPEGs are produced by the product's own GPU encoder (byte-identical to the model's encoder,
tests/test_gpu_encode.py); oracle/ is executed only as the checker and for cpu_baseline / --impl reference.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "video-coding_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (width, height, chroma, quality, restart_interval, out mode name, default batch per GPU)
    "restart8": (1920, 1080, 420, 75, 8, "yuv", 1024),     # BASELINE configs[1]
    "norestart": (1920, 1080, 420, 75, 0, "yuv", 1024),    # BASELINE configs[2] (8192 / N per GPU for N >= 2)
    "4k444rgb": (3840, 2160, 444, 95, 0, "rgb", 128),      # BASELINE configs[3]
    "restart8rgb": (1920, 1080, 420, 75, 8, "rgb", 1024),  # configs[1] with RGB24 output (Planar_444 up-sampling + colour)
    "restart120": (1920, 1080, 420, 75, 120, "yuv", 1024), # one MCU row per restart interval (camera style)
    "encode": (1920, 1080, 420, 75, 0, "jpeg", 512),       # BASELINE configs[4]
}
EXTRAS = ["norestart", "4k444rgb", "encode", "restart8rgb", "restart120"]
PARITY_IMAGES = 4
DUMP_VALUES = 1 << 21  # values per workload that --dump-outputs keeps: 8 MB of float32, all six workloads under 64 MB


def _synth_one(args):
    import synth

    seed, w, h, chroma = args
    return synth.frame(seed, w, h, chroma)


def make_frames(n, w, h, chroma, seed0):
    """`n` distinct seeded frames (SURVEY 8d recipe), generated on the host cores before CUDA starts."""
    import multiprocessing as mp

    jobs = [(seed0 + i, w, h, chroma) for i in range(n)]
    with mp.get_context("fork").Pool(min(len(jobs), os.cpu_count() or 1)) as pool:
        return pool.map(_synth_one, jobs)


def _cpu_decode_worker(args):
    sys.path.insert(0, ROOT)
    from oracle import pyoracle as orc

    jpgs, reps = args
    orc.lib()
    return orc.time_decode(jpgs, True, reps)


def _cpu_encode_worker(args):
    sys.path.insert(0, ROOT)
    from oracle import pyoracle as orc

    frames, w, h, chroma, q, ri = args
    orc.lib()
    return sum(orc.time_encode(f, w, h, chroma, q, ri, 1) for f in frames)


def _oracle_encode_worker(args):
    sys.path.insert(0, ROOT)
    from oracle import pyoracle as orc

    f, w, h, chroma, q, ri = args
    return orc.encode(f, w, h, chroma, q, restart_interval=ri)


def _oracle_decode_sha(args):
    sys.path.insert(0, ROOT)
    from oracle import pyoracle as orc

    jpg, rgb, chroma = args
    d = orc.decode(jpg)
    if not rgb:
        return hashlib.sha256(d.yuv()).hexdigest()
    y, u, v = orc.upsample_to_444(d.cropped, chroma)
    return hashlib.sha256(orc.ycbcr_to_rgb24(y, u, v).tobytes()).hexdigest()


def _noop(_):
    return 0


def cpu_arm(kind, items, w, h, chroma, q, ri, target_s=12.0):
    """Time the oracle (port of the model's algorithm) with one process per host core on a bounded sample."""
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    per_image = 0.07 * (w * h) / (1920 * 1080) * (3.0 if chroma == 444 else 1.0)
    per_core = max(1, min(64, int(target_s / per_image / 1.0)))
    ctx = mp.get_context("spawn")
    chunks = [[items[(c * per_core + i) % len(items)] for i in range(per_core)] for c in range(cores)]
    with ctx.Pool(cores) as pool:
        pool.map(_noop, range(cores))  # start the workers (imports) outside the timed region
        t0 = time.perf_counter()
        if kind == "decode":
            pool.map(_cpu_decode_worker, [(ch, 1) for ch in chunks])
        else:
            pool.map(_cpu_encode_worker, [(ch, w, h, chroma, q, ri) for ch in chunks])
        wall = time.perf_counter() - t0
    n = per_core * cores
    return {
        "value": n * w * h / 1e6 / wall,
        "unit": "MP/s",
        "cores": cores,
        "kind": "port",
        "sample": "%d images (%d per core, one process per core, oracle/hcj_oracle.c -O2), %.1f s wall" % (n, per_core, wall),
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index, self.first = [], None, index, 0

    def mark(self):
        """Samples before this point (input generation, warm-up of nvidia-smi itself) are ignored."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def snapshot(self):
        rows = self.rows[self.first:]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


def measured_traffic(kernel, n_images):
    """dram__bytes_read + dram__bytes_write of `kernel` for one launch over n_images images, from the committed
    ncu --set full capture (profiles/*_traffic.json, the newest round first: per-image bytes on the same synthetic
    1080p images).  None for kernels / workloads that were not captured."""
    for name in ("r02_traffic.json", "r01s3_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                per_image = json.load(f)["dram_bytes_per_image"].get(kernel)
            if per_image is not None:
                return per_image * n_images, "profiles/%s (ncu --set full, dram read + write per image x batch)" % name
        except Exception:
            pass
    return None, None


def bind_to_gpu_numa_node(index):
    """Pin this process (and so its pinned host buffers, first-touch) to the CPUs of the NUMA node the GPU hangs
    off: with one process per GPU the PCIe copies of the end-to-end leg then stay on the GPU's own socket.
    Best effort: returns the node or None."""
    try:
        bdf = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                      text=True).strip().lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(dirname, name, arrays):
    """DIR/<name>.npy: float32 of shape (images, k), row i holding k values of arrays[i] (what the caller received for image
    i) at seeded relative positions.  The positions depend only on the array lengths, so two builds with the same outputs
    write the same file."""
    k = max(1, DUMP_VALUES // len(arrays))
    u = np.random.default_rng(0).random((len(arrays), k))
    rows = [np.asarray(a)[(u[i] * len(a)).astype(np.int64)] for i, a in enumerate(arrays)]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), np.asarray(rows, np.float32))


def workload_config(name, batch_n, unique):
    w, h, chroma, quality, ri, out_name, _ = WORKLOADS[name]
    return {"workload": "%s: %d x %dx%d %d q%d %s per GPU -> %s" % (
        name, batch_n, w, h, chroma, quality, "DRI=%d MCUs" % ri if ri else "no restart markers", out_name),
        "batch_per_gpu": batch_n, "unique_images": unique, "sharding": "batch index, no collective",
        "l2": "per-step working set (compressed batch + coefficient buffer) exceeds the 126 MB L2"}


def batch_for(name, world, override=0):
    if override:
        return override
    if name == "norestart" and world >= 2:
        return 8192 // world  # BASELINE configs[2]: 8192 images sharded over 2 / 4 / 8 GPUs
    return WORKLOADS[name][6]


class Env:
    """What every workload needs: the context, the barrier / reduction helpers, the per-stage byte counts."""

    def __init__(self, ctx, world, barrier, max_over_ranks, sampler):
        self.ctx, self.world, self.barrier, self.max_over_ranks, self.sampler = ctx, world, barrier, max_over_ranks, sampler


def run_decode(env, name, frames, batch_n, steps, warmup, e2e_steps, parity=PARITY_IMAGES, dump_dir=None):
    """One decode workload: resident (`value`), per-stage roofline, end to end, oracle check of `parity` images; with
    `dump_dir`, a sample of the frames the last timed step decoded goes to dump_dir/<name>.npy."""
    import hcjpeg

    ctx = env.ctx
    w, h, chroma, quality, ri, out_name, _ = WORKLOADS[name]
    mode = {"yuv": hcjpeg.OUT_YUV, "rgb": hcjpeg.OUT_RGB24}[out_name]
    unique = len(frames)
    mp_per_step = batch_n * w * h / 1e6
    # compressed inputs from the GPU encoder (byte-identical to the model's encoder)
    jpgs, st = [], []
    for i in range(0, unique, 16):
        o, s = ctx.encode_batch(frames[i:i + 16], w, h, chroma, quality, ri)
        jpgs += o
        st += s
    assert all(s == 0 for s in st), st
    batch_jpgs = [jpgs[i % unique] for i in range(batch_n)]
    comp_bytes = sum(len(j) for j in batch_jpgs)

    # ---- value: resident inputs, kernels only
    b = ctx.batch(batch_jpgs, mode)
    assert all(s == 0 for s in b.host_status)
    env.sampler.mark()
    for _ in range(max(warmup, 3)):
        b.decode()
    ctx.synchronize()
    env.barrier()
    ctx.timer_start()
    for _ in range(steps):
        b.decode()
    ms = ctx.timer_stop()
    env.barrier()
    ms_per_step = env.max_over_ranks(ms) / steps
    outs, st = b.fetch()  # the frames of the last timed step
    assert all(s == 0 for s in st), [s for s in st if s][:4]
    if dump_dir:
        dump_outputs(dump_dir, name, outs)
    # per-stage timing for the roofline of the dominant kernel (separate passes, same stream, CUDA events)
    stages = {}
    for _ in range(steps):
        for k, v in b.decode_stages().items():
            stages[k] = stages.get(k, 0.0) + v / steps
    clocks = env.sampler.snapshot()
    nblocks = sum(f.nblocks for f in b.infos)
    out_bytes = sum(hcjpeg.out_size(f, mode) for f in b.infos)
    launches = b.kernels() * steps
    fused_rgb = "rgb" not in {k for k, v in stages.items() if v > 0.02}
    b.close()
    # ---- parity: a few of the benched images against the oracle, outside the timed region
    import multiprocessing as mp

    npar = min(parity, unique)
    with mp.get_context("spawn").Pool(min(npar, os.cpu_count() or 1)) as pool:
        want = pool.map(_oracle_decode_sha, [(jpgs[i], mode == hcjpeg.OUT_RGB24, chroma) for i in range(npar)])
    for i in range(npar):
        assert hashlib.sha256(outs[i].tobytes()).hexdigest() == want[i], "%s: image %d differs from the oracle" % (name, i)
    alg = {  # algorithmic bytes per launch (SURVEY 8d / DESIGN.md)
        "destuff": 2 * comp_bytes,
        "huffman_restart": comp_bytes + 128 * nblocks,
        "huffman_speculative": comp_bytes + 128 * nblocks,
        # planar output: coefficient blocks in, frames out; RGB: fused = coefficient blocks in, RGB out; two kernels = planes in between
        "idct": 128 * nblocks + (out_bytes if (mode != hcjpeg.OUT_RGB24 or fused_rgb) else nblocks * 64),
        "rgb": nblocks * 64 + out_bytes,
        "clear_flags": nblocks // 8,
    }
    stages = {k: v for k, v in stages.items() if v > 0.02}  # stages that did not launch read as ~0.003 ms
    kernels_only = {k: v for k, v in stages.items() if k != "clear_flags"}
    dom = max(kernels_only, key=kernels_only.get)
    peak, peak_src = peaks()
    achieved = alg[dom] / (stages[dom] * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic(dom, batch_n) if (w, h, chroma, quality, ri) == (1920, 1080, 420, 75, 8) else (None, None)
    roofline = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes": alg[dom],
                "traffic_source": traffic_src, "peak_source": peak_src,
                "stages": {k: {"ms": v, "algorithmic_GBps": alg[k] / (v * 1e-3) / 1e9, "frac": alg[k] / (v * 1e-3) / 1e9 / peak}
                           for k, v in stages.items()}}
    if mode == hcjpeg.OUT_RGB24:  # the pixel stage as a whole (north_star: dequant + IDCT + up-sampling + colour), one kernel or two
        pix_ms = stages.get("idct", 0.0) + stages.get("rgb", 0.0)
        pix_bytes = 128 * nblocks + out_bytes
        roofline["pixel_stage"] = {"ms": pix_ms, "kernels": 1 if fused_rgb else 2, "algorithmic_bytes": pix_bytes,
                                   "frac": pix_bytes / (pix_ms * 1e-3) / 1e9 / peak}
    res = {"metric": "decoded megapixels/sec (%dx%d %d baseline)" % (w, h, chroma), "ms_per_step": ms_per_step,
           "value": env.world * mp_per_step / (ms_per_step * 1e-3), "unit": "MP/s", "steps": steps, "roofline": roofline,
           "gpu_launches": launches, "clocks": clocks, "parity_checked": npar, "config": workload_config(name, batch_n, unique)}

    # ---- e2e: host buffers in and out through hcj_decode_batch (calls of at most 1024 images reuse the pinned buffers)
    if e2e_steps > 0:
        L = hcjpeg.lib()
        call_n = min(batch_n, 1024)
        in_bytes = sum((len(j) + 31) // 16 * 16 for j in batch_jpgs[:call_n])
        sizes = [hcjpeg.out_size(hcjpeg.frame_info(j), mode) for j in jpgs]
        out_cap = sum((sizes[i % unique] + 255) // 256 * 256 for i in range(call_n))
        pin_in = L.hcj_host_alloc(in_bytes + 64)
        pin_out = L.hcj_host_alloc(out_cap + 256)
        assert pin_in and pin_out
        jp = (C.c_void_p * call_n)()
        lens = (C.c_size_t * call_n)()
        op = (C.c_void_p * call_n)()
        caps = (C.c_size_t * call_n)()
        status = (C.c_int * call_n)()
        off_i = off_o = 0
        for i in range(call_n):
            j = batch_jpgs[i]
            C.memmove(pin_in + off_i, j, len(j))
            jp[i], lens[i] = pin_in + off_i, len(j)
            off_i += (len(j) + 31) // 16 * 16
            op[i], caps[i] = pin_out + off_o, sizes[i % unique]
            off_o += (sizes[i % unique] + 255) // 256 * 256
        ncalls = (batch_n + call_n - 1) // call_n

        def one_step():
            for _ in range(ncalls):
                hcjpeg._check(L.hcj_decode_batch(ctx._h, jp, lens, call_n, mode, hcjpeg.FLAG_DEFAULT, op, caps, status))

        one_step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            one_step()
        ctx.synchronize()
        env.barrier()
        dt = env.max_over_ranks(time.perf_counter() - t0) / e2e_steps
        assert all(status[i] == 0 for i in range(call_n))
        for i in range(npar):  # the e2e leg's own outputs against the oracle too
            got = np.ctypeslib.as_array(C.cast(op[i], C.POINTER(C.c_uint8)), shape=(caps[i],))
            assert hashlib.sha256(got.tobytes()).hexdigest() == want[i], "%s: e2e image %d differs from the oracle" % (name, i)
        res["e2e"] = {"value": env.world * (ncalls * call_n * w * h / 1e6) / dt, "unit": "MP/s",
                      "h2d_bytes_per_step": comp_bytes * ncalls * call_n // batch_n,
                      "d2h_bytes_per_step": (out_bytes + 4 * batch_n) * ncalls * call_n // batch_n, "ms_per_step": dt * 1e3,
                      "steps": e2e_steps, "images_per_call": call_n}
        L.hcj_host_free(pin_in)
        L.hcj_host_free(pin_out)
    return res, jpgs


def run_encode(env, name, frames, batch_n, steps, warmup, parity=PARITY_IMAGES, dump_dir=None):
    """Encode workload: frames in pinned host memory -> files in pinned host memory through hcj_encode_batch.  With
    `dump_dir`, the file lengths of the last timed step go to dump_dir/<name>_lengths.npy and a sample of the files'
    bytes to dump_dir/<name>.npy."""
    import hcjpeg

    ctx = env.ctx
    w, h, chroma, quality, ri, _, _ = WORKLOADS[name]
    L = hcjpeg.lib()
    unique = len(frames)
    mp_per_step = batch_n * w * h / 1e6
    frame_bytes = len(frames[0])
    cap = 1 << 20
    pin_in = L.hcj_host_alloc(frame_bytes * batch_n)
    pin_out = L.hcj_host_alloc(cap * batch_n)
    assert pin_in and pin_out
    fp = (C.c_void_p * batch_n)()
    op = (C.c_void_p * batch_n)()
    caps = (C.c_size_t * batch_n)(*([cap] * batch_n))
    lens = (C.c_size_t * batch_n)()
    status = (C.c_int * batch_n)()
    for i in range(batch_n):
        C.memmove(pin_in + i * frame_bytes, frames[i % unique], frame_bytes)
        fp[i], op[i] = pin_in + i * frame_bytes, pin_out + i * cap

    def run():
        hcjpeg._check(L.hcj_encode_batch(ctx._h, fp, batch_n, w, h, chroma, quality, ri, op, caps, lens, status))
        ms = C.c_float()
        hcjpeg._check(L.hcj_encode_last_device_ms(ctx._h, C.byref(ms)))
        return ms.value

    # `value` leg: kernel time with the whole batch on the device at once (HCJ_ENC_CHUNK = batch: one chunk, the
    # frames are resident in HBM before the first kernel starts; CUDA events around the kernels inside the library)
    os.environ["HCJ_ENC_CHUNK"] = str(batch_n)
    for _ in range(max(warmup, 3)):
        run()
    env.barrier()
    env.sampler.mark()
    dev_ms = [run() for _ in range(steps)]
    ctx.synchronize()
    clocks = env.sampler.snapshot()
    # `e2e` leg: the call as a user makes it (chunks of 64 frames: upload, kernels and download overlap), wall clock
    del os.environ["HCJ_ENC_CHUNK"]
    for _ in range(3):
        run()
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    ctx.synchronize()
    env.barrier()
    dt = env.max_over_ranks(time.perf_counter() - t0) / steps
    assert all(status[i] == 0 for i in range(batch_n))
    if dump_dir:
        dump_outputs(dump_dir, name, [np.ctypeslib.as_array(C.cast(op[i], C.POINTER(C.c_uint8)), shape=(lens[i],)) for i in range(batch_n)])
        np.save(os.path.join(dump_dir, name + "_lengths.npy"), np.array(lens[:batch_n], np.float64))
    # ---- parity: byte-identical files versus the oracle encoder
    import multiprocessing as mp

    npar = min(parity, unique)
    with mp.get_context("spawn").Pool(min(npar, os.cpu_count() or 1)) as pool:
        want = pool.map(_oracle_encode_worker, [(frames[i], w, h, chroma, quality, ri) for i in range(npar)])
    for i in range(npar):
        got = bytes(np.ctypeslib.as_array(C.cast(op[i], C.POINTER(C.c_uint8)), shape=(lens[i],)))
        assert got == want[i], "encode: frame %d differs from the oracle encoder" % i
    kms = env.max_over_ranks(float(np.mean(dev_ms)))
    out_total = sum(lens[i] for i in range(batch_n))
    nblocks = hcjpeg.frame_info(want[0]).nblocks * batch_n
    # SURVEY 8d: K6 = frames in + 128 Nb out; K7/K8 = 128 Nb in + C out  ->  in + 256 Nb + C for the pipeline
    alg = frame_bytes * batch_n + 2 * 128 * nblocks + out_total
    peak, peak_src = peaks()
    res = {"metric": "encoded megapixels/sec (%dx%d %d baseline)" % (w, h, chroma), "ms_per_step": kms,
           "value": env.world * mp_per_step / (kms * 1e-3), "unit": "MP/s", "steps": steps,
           "gpu_launches": L.hcj_encode_count_kernels() * steps, "clocks": clocks, "parity_checked": npar,
           "config": workload_config(name, batch_n, unique),
           "roofline": {"kernel": "encode pipeline (fdct_quant + bit lengths + pack + stuff)", "bound": "hbm",
                        "achieved": alg / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (kms * 1e-3) / 1e9 / peak,
                        "traffic": None, "algorithmic_bytes": alg, "peak_source": peak_src,
                        "note": "algorithmic bytes (SURVEY 8d): frames in + coefficient blocks written and read once + files out"},
           "e2e": {"value": env.world * mp_per_step / dt, "unit": "MP/s", "h2d_bytes_per_step": frame_bytes * batch_n,
                   "d2h_bytes_per_step": out_total, "ms_per_step": dt * 1e3, "steps": steps}}
    L.hcj_host_free(pin_in)
    L.hcj_host_free(pin_out)
    return res


def main():
    # Libraries print to stdout on their own (NCCL announces its version there at communicator creation): everything
    # but the JSON line goes to stderr.
    global _REAL_STDOUT
    sys.dont_write_bytecode = True  # the run leaves the tree as it found it (no __pycache__ of the modules imported from it)
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="restart8", choices=sorted(WORKLOADS))
    ap.add_argument("--only", action="store_true", help="time the headline workload only (no `workloads` section)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU of the headline workload (default: per workload)")
    ap.add_argument("--unique", type=int, default=64, help="distinct images cycled to fill the batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write a seeded sample of what each timed workload computed in its last step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    w, h, chroma, quality, ri, out_name, _ = WORKLOADS[args.workload]
    batch_n = batch_for(args.workload, world, args.batch)
    unique = max(1, min(args.unique, batch_n))
    config = workload_config(args.workload, batch_n, unique)

    if args.impl == "reference" and rank != 0:
        return 0

    # ---- synthetic inputs (host cores, before CUDA is touched); both arms use the same `unique` images
    frames = make_frames(unique, w, h, chroma, 1000 * (1 + rank))

    import hcjpeg

    hcjpeg.build()
    if args.impl == "reference":
        # The reference's own CPU implementation cannot run here (OCaml, no toolchain): the oracle port of its
        # algorithm is timed on all host cores, on inputs from the oracle encoder.
        import multiprocessing as mp

        kind = "encode" if args.workload == "encode" else "decode"
        if kind == "decode":
            with mp.get_context("spawn").Pool(os.cpu_count() or 1) as pool:
                items = pool.map(_oracle_encode_worker, [(f, w, h, chroma, quality, ri) for f in frames])
        else:
            items = frames
        vals = []
        for step in range(args.warmup + args.steps):
            r = cpu_arm(kind, items, w, h, chroma, quality, ri, target_s=8.0)
            if step >= args.warmup:
                vals.append(r)
        v = float(np.mean([x["value"] for x in vals]))
        cb = dict(vals[-1], value=v)
        emit(({
            "impl": "reference", "metric": "%s megapixels/sec (%dx%d %d baseline)" % ("decoded" if kind == "decode" else "encoded", w, h, chroma),
            "value": v, "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.mean([float(x["sample"].split(",")[-1].split()[0]) for x in vals])),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": config, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    # extra workloads: their frames are generated before CUDA starts as well
    extras = [] if args.only else [x for x in EXTRAS if x != args.workload]
    extra_frames = {}
    for name in extras:
        ew, eh, ec = WORKLOADS[name][:3]
        key = (ew, eh, ec)
        if key == (w, h, chroma):
            extra_frames[key] = frames
        elif key not in extra_frames:
            extra_frames[key] = make_frames(min(unique, 16), ew, eh, ec, 7000 * (1 + rank))

    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    import torch

    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from hcjpeg import shard

    dist_mod = dist if world > 1 else None
    ctx = hcjpeg.Context(local)
    sampler = ClockSampler(local)
    sampler.start()
    env = Env(ctx, world, lambda: shard.barrier(dist_mod, torch.cuda.synchronize),
              lambda x: shard.max_over_ranks(x, dist_mod, "cuda"), sampler)

    e2e_steps = 0 if args.no_e2e else max(1, min(args.steps, 3))
    dump_dir = args.dump_outputs if rank == 0 else None
    if args.workload != "encode":
        result, jpgs = run_decode(env, args.workload, frames, batch_n, args.steps, args.warmup, e2e_steps, dump_dir=dump_dir)
        cpu_items, cpu_kind = jpgs, "decode"
    else:
        result = run_encode(env, args.workload, frames, batch_n, args.steps, args.warmup, dump_dir=dump_dir)
        cpu_items, cpu_kind = frames, "encode"

    workloads = {}
    for name in extras:
        ew, eh, ec = WORKLOADS[name][:3]
        bn = batch_for(name, world)
        fr = extra_frames[(ew, eh, ec)]
        steps = max(1, min(args.steps, 10))
        if name == "encode":
            r = run_encode(env, name, fr, bn, steps, 3, dump_dir=dump_dir)
        else:
            r, _ = run_decode(env, name, fr, bn, steps, 3, 0 if args.no_e2e else min(2, steps), dump_dir=dump_dir)
        workloads[name] = r

    sampler.stop()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_arm(cpu_kind, cpu_items, w, h, chroma, quality, ri)
    line = {
        "metric": result["metric"], "value": result["value"], "unit": "MP/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": result["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int16/int32 (integer, bit-exact)", "data": "synthetic", "config": config,
        "clocks": result["clocks"], "e2e": result.get("e2e"), "gpu_launches": result["gpu_launches"],
        "roofline": result["roofline"], "cpu_baseline": cpu, "parity_checked": result["parity_checked"], "numa_node": numa,
    }
    if workloads:
        line["workloads"] = workloads
    emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
