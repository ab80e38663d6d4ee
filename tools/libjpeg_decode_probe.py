"""Measures the libjpeg reconstruction (HCJ_FLAG_LIBJPEG: islow IDCT, fancy chroma up-sampling) against the default
decode and prints one JSON line (also written to --out FILE when given).  Needs a CUDA device; fails without one.

  workloads   "1080p420": --images x 1080p 4:2:0 q75 DRI 8 (bench.py's default workload), HCJ_OUT_YUV and HCJ_OUT_RGB24;
              "4k444": --images-4k x 3840x2160 4:4:4 q95, HCJ_OUT_RGB24 (the default decode fuses the colour conversion
              into the IDCT kernel there; the flag does not)
  stages_ms   hcj_batch_decode_stages (CUDA events between the stages) of a resident batch, with and without the flag
              alternating: 3 warm-up passes, then --reps passes; medians
  e2e_ms      wall clock of hcj_decode_batch from pinned host files to pinned host frames, alternating; medians
  parity      images 0 .. --distinct - 1 of every flagged output against libjpeg_reference, and of every unflagged one
              against the oracle, outside the timed regions
  pillow      Pillow (libjpeg-turbo) decoding the 1080p files to RGB on every host core (a process per core), as the CPU
              point of comparison
The files are --distinct seeded images (synth frames, the oracle's encoder) repeated over the batch."""
import argparse
import ctypes as C
import io
import json
import multiprocessing as mp
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
import libjpeg_reference as lr  # noqa: E402
import synth  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402

FLAGS = {"default": hcjpeg.FLAG_DEFAULT, "libjpeg": hcjpeg.FLAG_DEFAULT | hcjpeg.FLAG_LIBJPEG}
MODE_NAMES = {hcjpeg.OUT_YUV: "yuv", hcjpeg.OUT_RGB24: "rgb"}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    line = subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).splitlines()[0]
    return dict(zip(q.split(","), [s.strip() for s in line.split(",")]))


def oracle_output(jpg, mode):
    dec = orc.decode(jpg)
    if mode == hcjpeg.OUT_YUV:
        return dec.yuv()
    y, u, v = orc.upsample_to_444(dec.cropped, dec.chroma)
    return orc.ycbcr_to_rgb24(y, u, v).tobytes()


def measure(L, ctx, uniq, n, modes, reps):
    """stages, e2e and parity of one workload, both reconstructions, every mode."""
    jpgs = [uniq[i % len(uniq)] for i in range(n)]
    infos = {k: [hcjpeg.frame_info(j, f) for j in uniq] for k, f in FLAGS.items()}
    offs, acc = [], 0
    for j in jpgs:
        offs.append(acc)
        acc += (len(j) + 15) & ~15
    fin = L.hcj_host_alloc(acc)
    sizes = {(k, m): [hcjpeg.out_size(infos[k][i % len(uniq)], m) for i in range(n)] for k in FLAGS for m in modes}
    out_offs = {}
    for key, sz in sizes.items():
        o = [0]
        for b in sz:
            o.append(o[-1] + ((b + 255) & ~255))
        out_offs[key] = o
    fout = L.hcj_host_alloc(max(o[-1] for o in out_offs.values()))
    assert fin and fout
    fin_np = np.ctypeslib.as_array((C.c_uint8 * acc).from_address(fin))
    for o, j in zip(offs, jpgs):
        fin_np[o:o + len(j)] = np.frombuffer(j, np.uint8)
    p_in = (C.c_void_p * n)(*[fin + o for o in offs])
    lens = (C.c_size_t * n)(*[len(j) for j in jpgs])
    p_out = {k: (C.c_void_p * n)(*[fout + o[i] for i in range(n)]) for k, o in out_offs.items()}
    caps = {k: (C.c_size_t * n)(*[o[i + 1] - o[i] for i in range(n)]) for k, o in out_offs.items()}
    status = (C.c_int * n)()

    def decode(k, m):
        rc = L.hcj_decode_batch(ctx._h, p_in, lens, n, m, FLAGS[k], p_out[(k, m)], caps[(k, m)], status)
        assert rc == 0 and all(status[i] == 0 for i in range(n)), (rc, k, m)

    res = {"parity": {}, "stages_ms": {}, "e2e_ms": {}, "output_GB": {}}
    refs = {}
    for m in modes:
        for k in FLAGS:
            decode(k, m)
            ok = True
            for i in range(len(uniq)):
                got = np.ctypeslib.as_array((C.c_uint8 * sizes[(k, m)][i]).from_address(fout + out_offs[(k, m)][i])).tobytes()
                if (i, k, m) not in refs:
                    refs[(i, k, m)] = lr.LibjpegDecode(orc, uniq[i]).output(m) if k == "libjpeg" else oracle_output(uniq[i], m)
                ok = ok and got == refs[(i, k, m)]
            res["parity"]["%s_%s" % (MODE_NAMES[m], k)] = ok
            res["output_GB"]["%s_%s" % (MODE_NAMES[m], k)] = sum(sizes[(k, m)]) / 1e9
    for m in modes:
        batches = {k: hcjpeg.Batch(ctx, jpgs, m, f) for k, f in FLAGS.items()}
        runs = {k: [] for k in FLAGS}
        for it in range(3 + reps):
            for k in FLAGS:
                st = batches[k].decode_stages()
                if it >= 3:
                    runs[k].append(st)
        for k in FLAGS:
            med = {s: statistics.median(r[s] for r in runs[k]) for s in runs[k][0]}
            med["total"] = statistics.median(sum(r.values()) for r in runs[k])
            res["stages_ms"]["%s_%s" % (MODE_NAMES[m], k)] = {"median": med, "idct_runs": [r["idct"] for r in runs[k]],
                                                               "rgb_runs": [r["rgb"] for r in runs[k]], "kernels": batches[k].kernels()}
        for b in batches.values():
            b.close()
    for m in modes:
        t = {k: [] for k in FLAGS}
        for it in range(2 + reps // 2):
            for k in FLAGS:
                t0 = time.perf_counter()
                decode(k, m)
                dt = (time.perf_counter() - t0) * 1e3
                if it >= 2:
                    t[k].append(dt)
        for k in FLAGS:
            res["e2e_ms"]["%s_%s" % (MODE_NAMES[m], k)] = {"median": statistics.median(t[k]), "runs": t[k]}
    L.hcj_host_free(C.c_void_p(fin))
    L.hcj_host_free(C.c_void_p(fout))
    return res


def _pil_rgb(jpg):
    from PIL import Image

    return np.asarray(Image.open(io.BytesIO(jpg)).convert("RGB")).nbytes


def pillow_rate(jpgs, reps):
    procs = os.cpu_count() or 1
    with mp.Pool(procs) as pool:
        pool.map(_pil_rgb, jpgs[: procs * 2])  # warm-up
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            pool.map(_pil_rgb, jpgs, chunksize=max(1, len(jpgs) // (4 * procs)))
            t.append((time.perf_counter() - t0) * 1e3)
    return {"processes": procs, "median_ms": statistics.median(t), "runs_ms": t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--images-4k", type=int, default=128)
    ap.add_argument("--distinct", type=int, default=4)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    L = hcjpeg.lib()
    assert L.hcj_device_count() > 0, "needs a CUDA device"
    res = {"gpu": gpu_info()}
    w, h = 1920, 1080
    u1080 = [orc.encode(synth.frame(5000 + k, w, h, 420), w, h, 420, 75, restart_interval=8) for k in range(a.distinct)]
    u4k = [orc.encode(synth.frame(6000 + k, 3840, 2160, 444), 3840, 2160, 444, 95) for k in range(min(2, a.distinct))]
    with hcjpeg.Context(0) as ctx:
        r = measure(L, ctx, u1080, a.images, (hcjpeg.OUT_YUV, hcjpeg.OUT_RGB24), a.reps)
        r["workload"] = "%d x %dx%d 4:2:0 q75, restart 8 (%d distinct)" % (a.images, w, h, len(u1080))
        res["1080p420"] = r
        r = measure(L, ctx, u4k, a.images_4k, (hcjpeg.OUT_RGB24,), a.reps)
        r["workload"] = "%d x 3840x2160 4:4:4 q95 (%d distinct)" % (a.images_4k, len(u4k))
        res["4k444"] = r
    res["pillow_1080p420_rgb"] = pillow_rate([u1080[i % len(u1080)] for i in range(a.images)], 3)
    res["pillow_1080p420_rgb"]["workload"] = "the 1080p420 files, Image.open(f).convert('RGB')"
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
