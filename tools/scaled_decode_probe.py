"""Measures the scaled decode (HCJ_FLAG_SCALE_1_2 / _1_4 / _1_8) against the full-size decode on 1024 x 1080p 4:2:0 q75
DRI 8 (bench.py's default workload) and prints one JSON line (also written to --out FILE when given).  Needs a CUDA
device; fails without one.

  stages_ms   hcj_batch_decode_stages (CUDA events between the stages) of a resident batch per scale and output mode
              (HCJ_OUT_YUV, HCJ_OUT_RGB24): 3 warm-up passes, then --reps passes with the scales alternating; medians
  idct        the idct stage's rate by algorithmic bytes: 128 bytes of coefficients read per block + the planes written
              (the cropped frame for HCJ_OUT_YUV, the padded planes for HCJ_OUT_RGB24), against the measured HBM copy peak
  e2e_ms      wall clock of hcj_decode_batch from pinned host files to pinned host frames, scales alternating; medians
  parity      images 0 .. --distinct - 1 of every e2e output against scaled_reference (s = 1: the oracle), outside the
              timed regions
The files are --distinct seeded images (synth frames, the oracle's encoder) repeated over the batch."""
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
import scaled_reference as sr  # noqa: E402
import synth  # noqa: E402
from oracle import pyoracle as orc  # noqa: E402

HBM_COPY_PEAK_GBPS = 6549.0  # measured device-to-device copy rate quoted in DESIGN.md
SCALES = (1, 2, 4, 8)
MODES = {"yuv": hcjpeg.OUT_YUV, "rgb": hcjpeg.OUT_RGB24}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    line = subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).splitlines()[0]
    return dict(zip(q.split(","), [s.strip() for s in line.split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--distinct", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    L = hcjpeg.lib()
    assert L.hcj_device_count() > 0, "needs a CUDA device"
    w, h, n = 1920, 1080, a.images
    uniq = [orc.encode(synth.frame(5000 + k, w, h, 420), w, h, 420, 75, restart_interval=8) for k in range(a.distinct)]
    jpgs = [uniq[i % a.distinct] for i in range(n)]
    flags = {s: hcjpeg.FLAG_DEFAULT | sr.FLAG[s] for s in SCALES}
    infos = {s: [hcjpeg.frame_info(j, flags[s]) for j in uniq] for s in SCALES}
    nblocks = sum(infos[1][i % a.distinct].nblocks for i in range(n))
    res = {"gpu": gpu_info(), "workload": "%d x %dx%d 4:2:0 q75, restart 8 (%d distinct)" % (n, w, h, a.distinct),
           "blocks": nblocks, "coefficient_GB": nblocks * 128 / 1e9}

    # pinned host files, back to back at 16-byte boundaries, and pinned frames back to back at 256-byte boundaries (the
    # device buffer's layout, so that consecutive frames come down in one copy, as hcj_decode_stream lays them out)
    offs, acc = [], 0
    for j in jpgs:
        offs.append(acc)
        acc += (len(j) + 15) & ~15
    fin = L.hcj_host_alloc(acc)
    out_bytes = {(s, m): [hcjpeg.out_size(infos[s][i % a.distinct], mode) for i in range(n)] for s in SCALES for m, mode in MODES.items()}
    out_offs = {}
    for key, sizes in out_bytes.items():
        o = [0]
        for b in sizes:
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
    res["output_GB"] = {m: {str(s): sum(out_bytes[(s, m)]) / 1e9 for s in SCALES} for m in MODES}

    with hcjpeg.Context(0) as ctx:
        def decode(s, m):
            rc = L.hcj_decode_batch(ctx._h, p_in, lens, n, MODES[m], flags[s], p_out[(s, m)], caps[(s, m)], status)
            assert rc == 0 and all(status[i] == 0 for i in range(n)), (rc, s, m)

        # parity (untimed)
        parity, refs = {}, {}
        for m, mode in MODES.items():
            for s in SCALES:
                decode(s, m)
                ok = True
                for i in range(a.distinct):
                    got = np.ctypeslib.as_array((C.c_uint8 * out_bytes[(s, m)][i]).from_address(fout + out_offs[(s, m)][i])).tobytes()
                    if (i, s) not in refs:
                        refs[(i, s)] = sr.ScaledDecode(orc, uniq[i], s)
                    ok = ok and got == refs[(i, s)].output(mode)
                parity["%s_s%d" % (m, s)] = ok
        res["parity"] = {"images_checked_per_case": a.distinct, "identical": parity}

        # per-stage device times, batch resident
        stages = {}
        for m, mode in MODES.items():
            batches = {s: hcjpeg.Batch(ctx, jpgs, mode, flags[s]) for s in SCALES}
            runs = {s: [] for s in SCALES}
            for it in range(3 + a.reps):
                for s in SCALES:
                    st = batches[s].decode_stages()
                    if it >= 3:
                        runs[s].append(st)
            for s in SCALES:
                names = runs[s][0].keys()
                med = {k: statistics.median(r[k] for r in runs[s]) for k in names}
                med["total"] = statistics.median(sum(r.values()) for r in runs[s])
                planes = sum(out_bytes[(s, m)]) if mode == hcjpeg.OUT_YUV else sum(infos[s][i % a.distinct].planes_bytes for i in range(n))
                algo = nblocks * 128 + planes
                gbps = algo / (med["idct"] * 1e-3) / 1e9
                stages["%s_s%d" % (m, s)] = {"ms": med, "idct_runs": [r["idct"] for r in runs[s]],
                                             "idct": {"algorithmic_GB": algo / 1e9, "GBps": gbps, "share_of_hbm_copy_peak": gbps / HBM_COPY_PEAK_GBPS}}
            for b in batches.values():
                b.close()
        res["stages_ms"] = stages
        res["hbm_copy_peak_GBps"] = HBM_COPY_PEAK_GBPS

        # end to end from pinned host memory
        e2e = {}
        for m in MODES:
            t = {s: [] for s in SCALES}
            for it in range(2 + a.reps // 2):
                for s in SCALES:
                    t0 = time.perf_counter()
                    decode(s, m)
                    dt = (time.perf_counter() - t0) * 1e3
                    if it >= 2:
                        t[s].append(dt)
            for s in SCALES:
                e2e["%s_s%d" % (m, s)] = {"median": statistics.median(t[s]), "runs": t[s]}
        res["e2e_ms"] = e2e
    L.hcj_host_free(C.c_void_p(fin))
    L.hcj_host_free(C.c_void_p(fout))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
