"""The entropy decoders (K2 k_huff_restart, K3 k_spec_*) on Huffman tables and symbols the reference encoder never writes.

Files come from tests/huffman_writer.py: given coefficients, written with tables of every shape the decoders' lookup
paths distinguish (primary LUT, the 8 shared-memory sub-tables, the model's full table in global memory), every
max_bits 1..16, complete code spaces, fixed-length codes, 1-2 bit codes, OpenCV-optimized and Annex K tables; table
bindings of 1..4 pairs, ids 2 and 3, a table defined twice; (r, 0) runs, blocks without EOB, AC sizes 11-15 and DC
categories 12-15 with 16-bit quant tables, DC predictors at the int16 edge, and the defined failures.  The CPU tests
check the writer and run the corpus through the emulation of K2 / K3; the GPU tests decode it on every route.
"""
import functools
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import huffman_writer as hw
import synth

SAMPLING = {"420": [(2, 2), (1, 1), (1, 1)], "422": [(2, 1), (1, 1), (1, 1)], "444": [(1, 1)] * 3, "400": [(1, 1)],
            "4c": [(2, 1), (1, 1), (1, 1), (1, 1)]}
BINDING = {"annex": [(0, 0), (1, 1), (1, 1), (1, 1)], "shared": [(0, 0)] * 4, "three": [(0, 0), (0, 1), (1, 0)],
           "four": [(0, 0), (1, 1), (2, 2), (3, 3)]}


# ---- coefficients ---------------------------------------------------------------------------------------------------
def _dc_walk(rng, frame, ri, cats):
    """Absolute DC values whose differences (per component, predictors reset at each restart) have categories drawn
    from `cats`."""
    n = frame.nblocks
    out = np.zeros(n, np.int64)
    pred = [0] * len(frame.comps)
    for b in range(n):
        if ri and b % (ri * frame.bpm) == 0:
            pred = [0] * len(frame.comps)
        c = frame.block_comp[b % frame.bpm]
        cat = int(rng.choice(cats))
        d = 0 if cat == 0 else int(rng.integers(1 << (cat - 1), 1 << cat)) * (1 if rng.random() < 0.5 else -1)
        if not -2047 <= pred[c] + d <= 2047 and cat <= 11:
            d = -d  # keep 8-bit-legal DC values where the categories allow it
        if not -32767 <= pred[c] + d <= 32767:
            d = -d
        pred[c] += d
        out[b] = pred[c]
    return out


def content(kind, frame, ri, seed):
    rng = np.random.default_rng(seed)
    n = frame.nblocks
    c = np.zeros((n, 64), np.int64)
    k = np.arange(1, 64)
    if kind == "tiny":  # DC differences of category 0 / 1, AC: a run of +-1 from coefficient 1 (symbols EOB, (0, 1))
        c[:, 0] = _dc_walk(rng, frame, ri, [0, 0, 1])
        ln = np.minimum(rng.geometric(0.45, n) - 1, 63)
        ln[::17] = 63
        for b in range(n):
            c[b, 1:1 + ln[b]] = rng.choice([-1, 1], ln[b])
    elif kind == "small":  # AC: +-1 after runs of 0..3
        c[:, 0] = _dc_walk(rng, frame, ri, list(range(8)))
        for b in range(n):
            z = 1 + int(rng.integers(0, 4))
            while z < 64 and rng.random() < 0.8:
                c[b, z] = rng.choice([-1, 1])
                z += 1 + int(rng.integers(0, 4))
    elif kind in ("natural", "uniform_dc"):  # decaying sparse AC of sizes 1..10
        cats = list(range(11)) if kind == "uniform_dc" else [0, 0, 1, 1, 2, 2, 3, 3, 4, 5, 6, 7, 8, 9, 10]
        c[:, 0] = _dc_walk(rng, frame, ri, cats)
        mask = rng.random((n, 63)) < 0.55 * np.exp(-k / 9.0)
        mag = np.minimum(np.rint(rng.exponential(1 + 40 * np.exp(-k / 8.0), (n, 63))) + 1, 1023)
        c[:, 1:] = np.where(mask, mag * rng.choice([-1, 1], (n, 63)), 0)
        c[::5, 1:] = 0  # EOB right after the DC
        c[3::11, 63] = rng.choice([-1, 1, 700], len(range(3, n, 11)))  # blocks that end on coefficient 63
    elif kind == "wide":  # AC sizes 1..15, DC categories up to 15
        c[:, 0] = _dc_walk(rng, frame, ri, list(range(16)))
        mask = rng.random((n, 63)) < 0.12
        size = rng.integers(1, 16, (n, 63))
        val = rng.integers(0, 1 << 14, (n, 63)) % (1 << (size - 1)) + (1 << (size - 1))
        c[:, 1:] = np.where(mask, val * rng.choice([-1, 1], (n, 63)), 0)
        c[::7, 1:] = 0
    else:
        raise ValueError(kind)
    return c


def dc_edge(frame, beyond):
    """Luma DC walked to exactly 32767 and -32768 (and, with beyond = +1 / -1, one step past one of them)."""
    c = np.zeros((frame.nblocks, 64), np.int64)
    walk = [100, 32767, 32767, 0, -32767, -32768, -32768, -20000, 0, 5]
    if beyond > 0:
        walk[2:5] = [32768, 1, -32766]
    elif beyond < 0:
        walk[6] = -32769
    luma = [b for b in range(frame.nblocks) if frame.block_comp[b % frame.bpm] == 0]
    for i, b in enumerate(luma):
        c[b, 0] = walk[i] if i < len(walk) else 7 * (i % 5)
        c[b, 1 + i % 63] = 1 - 2 * (i & 1)
    return c


# ---- tables ---------------------------------------------------------------------------------------------------------
def shape_max(freq, m):
    """max_bits exactly m: K.2 limited to m bits (all-ones code free when the alphabet allows), then the last code
    lengthened to m."""
    n = len(freq)
    assert n <= 1 << m, (n, m)
    lengths, values = hw.optimal_lengths(freq, m, reserve=n + 1 <= 1 << m)
    mb = max(i + 1 for i in range(16) if lengths[i])
    if mb < m:
        lengths[mb - 1] -= 1
        lengths[m - 1] += 1
    return lengths, values


def shape_prefixes(freq, nprefix):
    """Exactly `nprefix` 10-bit prefixes with longer codes: the frequent symbols get K.2 codes of 2..10 bits (half the
    code space), 4 * nprefix - 2 entries get 12-bit codes (the rarest symbols, listed more than once if the alphabet is
    small)."""
    syms = sorted(freq, key=lambda s: (-freq[s], s))
    nlong = 4 * nprefix - 2
    nshort = len(syms) - nlong if len(syms) > nlong + 1 else max(1, len(syms) // 2)
    short, rare = syms[:nshort], syms[nshort:]
    sl, sv = hw.optimal_lengths({s: freq[s] for s in short}, 9)
    lengths = [0] + sl[:9] + [0] * 6
    longv = [rare[i % len(rare)] for i in range(nlong)]
    lengths[11] = nlong
    return lengths, sv + longv


def shape_long(freq):
    """Every code longer than 10 bits."""
    lengths, values = hw.optimal_lengths(freq, 16)
    sym_len = {}
    for l, _, v in hw.codes(lengths, values):
        sym_len[v] = max(11, l)
    return hw.table_from_lengths(sym_len, values)


def shape_fixed(tc):
    """Fixed-length codes over every symbol, complete code spaces: 16 DC categories of 4 bits; 254 AC symbols of 8 bits
    and (15, 14), (15, 15) of 9 (a DHT cannot list 256 codes of one length)."""
    return ([0, 0, 0, 16] + [0] * 12, list(range(16))) if tc == 0 else ([0] * 7 + [254, 2] + [0] * 7, list(range(256)))


def make_table(shape, tc, freq):
    if shape == "opt":
        return hw.optimal_lengths(freq)
    if shape == "complete":
        return hw.optimal_lengths(freq, reserve=False)
    if shape == "long":
        return shape_long(freq)
    if shape == "fixed":
        return shape_fixed(tc)
    if shape[0] == "max":
        return shape_max(freq, shape[1])
    if shape[0] == "prefixes":
        return shape_prefixes(freq, shape[1])
    raise ValueError(shape)


def quant_tables(ncomp, wide):
    rng = np.random.default_rng(ncomp)
    if wide:  # 16-bit tables: products up to 32767 x 65535
        return {0: [65535] + rng.integers(1, 65536, 63).tolist(), 1: rng.integers(1, 65536, 64).tolist()}
    return {0: (1 + (np.arange(64) * 3) % 40).tolist(), 1: (2 + (np.arange(64) * 5) % 60).tolist()}


# ---- the corpus -----------------------------------------------------------------------------------------------------
# name: (geometry, width, height, binding, content, dc shape, ac shape, restart intervals, options)
SPECS = {
    "m1": ("400", 23, 17, "annex", "tiny", ("max", 1), ("max", 1), (0, 1), {}),
    "m2": ("420", 37, 29, "annex", "tiny", ("max", 2), ("max", 2), (0, 2), {}),
    "m3": ("422", 45, 31, "annex", "tiny", ("max", 3), ("max", 3), (0,), {}),
    "m4": ("444", 19, 27, "annex", "small", ("max", 4), ("max", 4), (0, 3), {}),
    "m5": ("420", 50, 34, "annex", "small", ("max", 5), ("max", 5), (0,), {}),
    "m6": ("400", 61, 9, "annex", "small", ("max", 6), ("max", 6), (0, 4), {}),
    "m7": ("422", 33, 41, "annex", "small", ("max", 7), ("max", 7), (0,), {}),
    "m8": ("420", 71, 53, "annex", "natural", ("max", 8), ("max", 8), (0, 5), {}),
    "m9": ("444", 40, 39, "annex", "natural", ("max", 9), ("max", 9), (0,), {}),
    "m10": ("420", 63, 47, "annex", "natural", ("max", 10), ("max", 10), (0, 2), {}),
    "m11": ("422", 55, 37, "annex", "natural", ("max", 11), ("max", 11), (0,), {}),
    "m12": ("400", 81, 35, "annex", "natural", ("max", 12), ("max", 12), (0, 7), {}),
    "m13": ("420", 90, 66, "annex", "natural", ("max", 13), ("max", 13), (0,), {}),
    "m14": ("444", 47, 45, "annex", "natural", ("max", 14), ("max", 14), (0, 3), {}),
    "m15": ("420", 77, 59, "annex", "natural", ("max", 15), ("max", 15), (0,), {}),
    "m16": ("422", 99, 43, "annex", "natural", ("max", 16), ("max", 16), (0, 6), {}),
    "sub8": ("420", 203, 151, "annex", "uniform_dc", ("prefixes", 8), ("prefixes", 8), (0, 4, 30), {"rotate": True}),
    "full9": ("444", 129, 97, "annex", "uniform_dc", ("prefixes", 9), ("prefixes", 12), (0, 5, 50), {"rotate": True}),
    "long": ("422", 121, 83, "annex", "natural", "long", "long", (0, 3, 40), {}),
    "complete": ("420", 97, 75, "annex", "natural", "complete", "complete", (0, 2), {}),
    "fixed8": ("420", 240, 176, "annex", "natural", "fixed", "fixed", (0, 40), {}),
    "tiny_ri1": ("420", 57, 41, "annex", "tiny", ("max", 1), ("max", 1), (1,), {}),
    "tiny_ri2": ("420", 66, 50, "annex", "tiny", ("max", 2), ("max", 1), (2, 3), {}),
    "tiny_show": ("400", 40, 24, "annex", "tiny", ("max", 16), ("max", 2), (1,), {}),
    "shared": ("444", 67, 35, "shared", "natural", "opt", "opt", (0, 3), {}),
    "three": ("420", 85, 63, "three", "natural", "opt", ("max", 15), (0, 4), {}),
    "four": ("4c", 75, 41, "four", "natural", ("max", 12), "opt", (0, 2, 30), {}),
    "redefined": ("420", 59, 43, "annex", "natural", "opt", "opt", (0, 3), {"decoy": True}),
    "runs_r0": ("420", 87, 65, "annex", "natural", "opt", "opt", (0, 3), {"split_runs": True}),
    "no_eob": ("444", 53, 29, "annex", "natural", "opt", "opt", (0, 2), {"omit_eob63": True, "split_runs": True}),
    "wide": ("444", 45, 37, "annex", "wide", "opt", "opt", (0, 2), {"wide": True}),
    "wide_420": ("420", 48, 32, "three", "wide", ("max", 16), "long", (0, 1), {"wide": True}),
    "dc_edge": ("400", 88, 8, "annex", "dc_edge", "opt", "opt", (0,), {}),
    "dc_over": ("400", 88, 8, "annex", "dc_over", "opt", "opt", (0, 9), {}),
    "dc_under": ("420", 64, 16, "annex", "dc_under", "opt", "opt", (0, 3), {}),
    "bad_dc_code": ("420", 61, 45, "annex", "natural", "opt", "opt", (0, 2), {"inject": (40, "dc_code")}),
    "bad_ac_code": ("422", 61, 45, "annex", "natural", "opt", "opt", (0, 2), {"inject": (33, "ac_code")}),
    "overrun": ("444", 61, 45, "annex", "natural", "opt", "opt", (0, 2), {"inject": (27, "overrun")}),
    "dc_symbol_16": ("420", 30, 30, "annex", "natural", "opt", "opt", (0,), {"dc_value_16": True}),
    "oversubscribed": ("400", 30, 30, "annex", "natural", "opt", "opt", (0,), {"oversubscribed": True}),
}
INTENDED = {"tiny_show": -9, "dc_over": -23, "dc_under": -23, "bad_dc_code": -2, "bad_ac_code": -3, "overrun": -4, "dc_symbol_16": -22,
            "oversubscribed": -25}


class Case:
    def __init__(self, name, jpg, coefs, status, legal, tables=None, used=None, frame=None, ri=0):
        self.name, self.jpg, self.coefs, self.status, self.legal = name, jpg, coefs, status, legal
        self.tables, self.used, self.frame, self.ri = tables or {}, used or {}, frame, ri


def _build(name, ri, seed):
    geom, w, h, binding, kind, dc_shape, ac_shape, _, opt = SPECS[name]
    sampling = SAMPLING[geom]
    bind = BINDING[binding]
    comps = [(k + 1, sh, sv, min(k, 1), bind[k][0], bind[k][1]) for k, (sh, sv) in enumerate(sampling)]
    frame = hw.Frame(w, h, comps, quant_tables(len(comps), opt.get("wide", False)))
    if kind.startswith("dc_"):
        coefs = dc_edge(frame, {"dc_edge": 0, "dc_over": 1, "dc_under": -1}[kind])
    else:
        coefs = content(kind, frame, ri, seed)
    wopts = {k: opt[k] for k in ("split_runs", "omit_eob63") if k in opt}
    counts = hw.symbol_counts(coefs, frame, ri, **wopts)
    if "inject" in opt and opt["inject"][1] == "overrun":
        for ci in range(len(comps)):
            counts[(1, ci)][0xF0] = counts[(1, ci)].get(0xF0, 0) + 1
            counts[(1, ci)][0xF1] = counts[(1, ci)].get(0xF1, 0) + 1
    dhts, tables = [], {}
    for tc, shape in ((0, dc_shape), (1, ac_shape)):
        for tid in sorted({c[4 + tc] for c in comps}):
            freq = {}
            for ci, c in enumerate(comps):
                if c[4 + tc] == tid:
                    for s, n in counts.get((tc, ci), {}).items():
                        freq[s] = freq.get(s, 0) + n
            lengths, values = make_table(shape, tc, freq)
            if tc == 0 and opt.get("dc_value_16"):
                lengths, values = hw.optimal_lengths({**freq, 16: 1})
            assert len(values) == sum(lengths) and all(0 <= v < 256 for v in values)
            if opt.get("decoy") and (tc, tid) == (1, 0):
                dhts.append((1, 0, [0, 0, 0, 0, 0, 0, 0, 255, 0, 0, 0, 0, 0, 0, 0, 0], [(i * 37) & 255 for i in range(255)]))
            dhts.append((tc, tid, lengths, values))
            tables[(tc, tid)] = (lengths, values)
    used = {}
    scan = hw.write_scan(coefs, frame, dhts, ri, rotate=opt.get("rotate", False), inject=opt.get("inject"), used=used, **wopts)
    if opt.get("oversubscribed"):  # the DC table in the header gets three 1-bit codes
        dhts = [(tc, th, [3] + [0] * 15, v[:3]) if tc == 0 else (tc, th, l, v) for tc, th, l, v in dhts]
        tables = hw.bindings(frame, dhts)
    jpg = hw.write_headers(frame, dhts, ri) + scan + b"\xff\xd9"
    legal = (geom in ("420", "422", "444") and kind not in ("wide",) and not wopts and "inject" not in opt
             and name not in INTENDED and not opt.get("decoy")
             and all(_no_all_ones(l) and len(set(v)) == len(v) for l, v in tables.values()))
    return Case("%s_ri%d" % (name, ri), jpg, coefs, INTENDED.get(name, 0), legal, tables, used, frame, ri)


def _no_all_ones(lengths):
    cs = hw.codes(lengths, list(range(sum(lengths))))
    l, c, _ = cs[-1]
    return c != (1 << l) - 1


def _opencv_cases():
    cv2 = pytest.importorskip("cv2")
    out = []
    for i, (w, h, q, ri) in enumerate(((160, 120, 90, 0), (131, 97, 95, 4), (200, 150, 75, 40))):
        rng = np.random.default_rng(70 + i)
        a = np.stack([synth.plane(rng, w, h) for _ in range(3)], -1)
        ok, buf = cv2.imencode(".jpg", a, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1, cv2.IMWRITE_JPEG_RST_INTERVAL, ri])
        assert ok
        out.append(("opencv%d_ri%d" % (i, ri), buf.tobytes()))
    return out


def _annex_cases(orc):
    out = []
    for i, (w, h, chroma, ri) in enumerate(((98, 70, 420, 0), (64, 48, 400, 3), (75, 51, 422, 20))):
        out.append(("annexk%d_ri%d" % (i, ri), orc.encode(synth.frame(300 + i, w, h, 420 if chroma == 400 else chroma), w, h, chroma, 85, ri)))
    return out


CASE_NAMES = ["%s_ri%d" % (n, ri) for n, s in SPECS.items() for ri in s[7]]


@functools.lru_cache(maxsize=None)
def corpus():
    """Every case of SPECS (written here) plus OpenCV-optimized and Annex K files (re-read through the writer)."""
    from oracle import pyoracle as orc

    orc.build()
    cases = {}
    for i, (name, s) in enumerate(SPECS.items()):
        for ri in s[7]:
            c = _build(name, ri, 1000 + 17 * i + ri)
            cases[c.name] = c
    for name, jpg in _opencv_cases() + _annex_cases(orc):
        frame, dhts, ri, ent = hw.read_file(jpg)
        d = orc.decode(jpg, want_blocks=True)
        used = {}
        assert hw.write_scan(d.coefs_abs_dc(), frame, dhts, ri, used=used) == ent
        legal = len(frame.comps) == 3
        cases[name] = Case(name, jpg, d.coefs_abs_dc().astype(np.int64), 0, legal, hw.bindings(frame, dhts), used, frame, ri)
    return cases


def _max_dequant(c):
    """The largest |coefficient x quant entry| of a case."""
    q = np.array([c.frame.quant[c.frame.comps[k][3]] for k in c.frame.block_comp], np.int64)
    return int(np.abs(c.coefs.reshape(-1, c.frame.bpm, 64) * q[None]).max())


def expected_status(orc, jpg):
    """The oracle's status, with HCJ_ERR_DC_RANGE (-23) where the oracle's absolute DC leaves int16."""
    st = orc.decode_status(jpg)
    if st:
        return st
    dc = orc.decode(jpg, want_blocks=True).dc_abs
    return -23 if (dc < -32768).any() or (dc > 32767).any() else 0


# ---- CPU: the writer --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chroma", [420, 422, 444, 400])
@pytest.mark.parametrize("ri", [0, 3, 5])
def test_writer_reproduces_oracle_files(orc, chroma, ri):
    """The oracle's coefficients re-written with the Annex K tables behind orc.write_headers give its file byte for byte."""
    for w, h, q in ((61, 45, 80), (24, 16, 100), (130, 34, 75)):
        src = synth.frame(7 * w + h, w, h, 420 if chroma == 400 else chroma)
        jpg = orc.encode(src, w, h, chroma, q, ri)
        frame, dhts, ri2, ent = hw.read_file(jpg)
        assert ri2 == ri and [(tc, th) for tc, th, _, _ in dhts] == ([(0, 0), (1, 0)] if chroma == 400 else [(0, 0), (0, 1), (1, 0), (1, 1)])
        assert all(hw.ANNEX_K[(tc, th)] == (l, v) for tc, th, l, v in dhts)
        coefs = orc.decode(jpg, want_blocks=True).coefs_abs_dc()
        assert orc.write_headers(w, h, chroma, q, ri) + hw.write_scan(coefs, frame, dhts, ri) + b"\xff\xd9" == jpg


@pytest.mark.parametrize("ri", [0, 1, 4, 40])
def test_writer_reproduces_opencv_optimized_scans(orc, ri):
    """OpenCV IMWRITE_JPEG_OPTIMIZE files (K.2 tables): re-writing with the file's own DHTs gives its entropy-coded
    segment byte for byte, RSTn included."""
    cv2 = pytest.importorskip("cv2")
    for i, (w, h, q) in enumerate(((320, 200, 90), (77, 53, 100), (161, 99, 60))):
        rng = np.random.default_rng(40 + i)
        a = np.stack([synth.plane(rng, w, h) for _ in range(3)], -1)
        params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1, cv2.IMWRITE_JPEG_RST_INTERVAL, ri]
        for img in (a, a[:, :, 0]):
            ok, buf = cv2.imencode(".jpg", img, params)
            assert ok
            jpg = buf.tobytes()
            frame, dhts, ri2, ent = hw.read_file(jpg)
            assert ri2 == ri
            assert any(hw.classify(l, v)[0] > 10 for tc, _, l, v in dhts if tc == 1)  # not the Annex K tables
            coefs = orc.decode(jpg, want_blocks=True).coefs_abs_dc()
            assert hw.write_scan(coefs, frame, dhts, ri) == ent


def test_k2_procedure_matches_opencv_tables(orc):
    """optimal_lengths is libjpeg's K.2: counting the symbols of an OpenCV-optimized file gives back its DHTs' lengths."""
    cv2 = pytest.importorskip("cv2")
    a = np.stack([synth.plane(np.random.default_rng(5), 150, 100) for _ in range(3)], -1)
    ok, buf = cv2.imencode(".jpg", a, [cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_OPTIMIZE, 1])
    jpg = buf.tobytes()
    frame, dhts, ri, _ = hw.read_file(jpg)
    counts = hw.symbol_counts(orc.decode(jpg, want_blocks=True).coefs_abs_dc(), frame, ri)
    for tc, th, lengths, values in dhts:
        freq = {}
        for ci, c in enumerate(frame.comps):
            if c[4 + tc] == th:
                for s, n in counts[(tc, ci)].items():
                    freq[s] = freq.get(s, 0) + n
        assert hw.optimal_lengths(freq)[0] == lengths


@pytest.mark.parametrize("name", CASE_NAMES + ["opencv", "annexk"])
def test_corpus_file_decodes_to_its_coefficients(orc, name):
    """Every written file: the oracle gives back exactly the written coefficients, or the intended status."""
    cases = [c for n, c in corpus().items() if n == name or (name in ("opencv", "annexk") and n.startswith(name))]
    assert cases
    for c in cases:
        st = expected_status(orc, c.jpg)
        assert st == c.status, (c.name, st)
        if c.status in (0, -23):
            got = orc.decode(c.jpg, want_blocks=True).coefs_abs_dc()
            assert np.array_equal(got, c.coefs), c.name
        for key, (l, v) in c.tables.items():
            assert hw.kraft_ok(l) or c.status == -25, (c.name, key)


def test_writer_speed(orc):
    """A scan of a few hundred KB encodes in well under a second."""
    import time

    frame = hw.Frame(1600, 1200, [(1, 2, 2, 0, 0, 0), (2, 1, 1, 1, 1, 1), (3, 1, 1, 1, 1, 1)], quant_tables(3, False))
    coefs = content("natural", frame, 0, 3)
    counts = hw.symbol_counts(coefs, frame)
    dhts = []
    for tc in (0, 1):
        for tid in (0, 1):
            freq = {}
            for ci in ((0,) if tid == 0 else (1, 2)):
                for s, n in counts[(tc, ci)].items():
                    freq[s] = freq.get(s, 0) + n
            dhts.append((tc, tid) + hw.optimal_lengths(freq))
    t = time.perf_counter()
    jpg = hw.write_jpeg(coefs, frame, dhts, 0)
    dt = time.perf_counter() - t
    assert len(jpg) > 200_000 and dt < 0.8, (len(jpg), dt)


# ---- CPU: coverage that cannot drift ------------------------------------------------------------------------------------
def _paths(cases):
    """{(class, path)} and {(class, max_bits)} of the codes the corpus writes."""
    paths, maxbits = set(), set()
    for c in cases.values():
        if c.status in (-22, -25):
            continue
        for (tc, tid), codes in c.used.items():
            l, v = c.tables[(tc, tid)]
            mb, cls = hw.classify(l, v)
            for length, code in codes:
                if length == mb:
                    maxbits.add((tc, mb))
                paths.add((tc, hw.PRIMARY if length <= hw.LUT_BITS or mb <= hw.LUT_BITS else int(cls[code >> (length - hw.LUT_BITS)])))
    return paths, maxbits


def test_corpus_coverage():
    """Symbols that occur in the corpus's streams use the full-table path (DC and AC), the 8th sub-table (DC and AC),
    codes of every length 1..16 as their table's longest (DC and AC), complete code spaces and 3 / 4 table pairs."""
    cases = corpus()
    paths, maxbits = _paths(cases)
    for tc in (0, 1):
        assert (tc, hw.FULL) in paths, tc
        assert (tc, hw.LUT_NSUB - 1) in paths, tc
        assert (tc, hw.PRIMARY) in paths, tc
        assert {m for t, m in maxbits if t == tc} == set(range(1, 17)), tc
    # a table with exactly 8 unresolved prefixes, one with 9 or more, one with every code longer than 10 bits
    nunres = [(tc, int((hw.classify(l, v)[1] != hw.PRIMARY).sum()), min(i + 1 for i in range(16) if l[i]))
              for c in cases.values() if c.status == 0 for (tc, _), (l, v) in c.tables.items()]
    for tc in (0, 1):
        assert (tc, 8) in {(t, n) for t, n, _ in nunres}
        assert any(t == tc and n >= 9 for t, n, _ in nunres)
    assert any(t == 1 and shortest > 10 for t, _, shortest in nunres)
    complete = [c.name for c in cases.values() if c.status == 0 and any(not _no_all_ones(l) for l, _ in c.tables.values())]
    assert complete
    pairs = {len({(cc[4], cc[5]) for cc in c.frame.comps}) for c in cases.values() if c.frame is not None and c.status == 0}
    assert {1, 2, 3, 4} <= pairs


# ---- CPU: the corpus through the emulation of K2 and K3 -----------------------------------------------------------------
def _emul_check(orc, emul, c, S_T):
    start = orc.header_decode(c.jpg).scan_bit_pos // 8 if c.status not in (-22, -25) else 0
    nb = c.frame.nblocks
    want = c.coefs.astype(np.int16) if c.status == 0 else None
    if c.status in (-22, -25):  # the tables are refused before any entropy decoding
        st, _ = emul.decode_segments(c.jpg, nb, len(c.jpg), c.ri > 0)
        assert st == c.status, c.name
        return 0
    st, got = emul.decode_segments(c.jpg, nb, start, c.ri > 0)
    assert st == c.status, (c.name, "K2", st)
    if want is not None:
        assert np.array_equal(got, want), (c.name, "K2")
    worst = 0
    for S, T in S_T:
        st, got, rounds = emul.decode_units(c.jpg, nb, start, T=T, S=S)
        assert st == c.status, (c.name, "K3", S, T, st)
        if want is not None:
            assert np.array_equal(got, want), (c.name, "K3", S, T)
        worst = max(worst, rounds)
    return worst


S_T = [(128, 32), (256, 64), (1024, 32), (1024, 64)]


@pytest.mark.parametrize("name", CASE_NAMES)
def test_emulated_decoders_on_corpus(orc, name):
    """K2 (decode_segments: one thread per interval) and K3 (decode_units at S in {128, 256, 1024}, T in {32, 64}) give
    the written coefficients and the oracle's status."""
    import emul

    emul.build()
    _emul_check(orc, emul, corpus()[name], S_T)


def test_emulated_decoders_on_reference_tables(orc):
    import emul

    for name, c in corpus().items():
        if name.startswith(("opencv", "annexk")):
            _emul_check(orc, emul, c, S_T)


def test_emulated_fixed_length_tables_need_many_rounds(orc):
    """Fixed-length 8-bit AC codes: a misaligned decoder falls back into step only by accident, so k_spec_fix's
    fix-point iteration runs many rounds."""
    import emul

    assert _emul_check(orc, emul, corpus()["fixed8_ri0"], [(128, 64)]) > 2


# ---- GPU ----------------------------------------------------------------------------------------------------------------
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


ROUTES = {"default": {}, "long_ri_1": {"HCJ_LONG_RI_BLOCKS": "1"}, "sub8_guess64": {"HCJ_SUB_LOG2": "8", "HCJ_GUESS_BITS": "64"}}


def _decode(hcj, ctx, cases, mode, flags=None):
    b = ctx.batch([c.jpg for c in cases], mode, hcj.FLAG_DEFAULT if flags is None else flags)
    try:
        b.decode()
        outs, st = b.fetch()
        coefs = [b.coefficients(i) if s == 0 else None for i, s in enumerate(st)]
    finally:
        b.close()
    return outs, st, coefs


def _check_batch(hcj, ctx, orc, cases, what):
    outs, st, coefs = _decode(hcj, ctx, cases, hcj.OUT_PLANES)
    assert st == [c.status for c in cases], (what, [(c.name, s) for c, s in zip(cases, st) if s != c.status])
    for c, o, k in zip(cases, outs, coefs):
        if c.status == 0:
            assert np.array_equal(k, c.coefs.astype(np.int16)), (what, c.name)
            assert bytes(o) == b"".join(p.tobytes() for p in orc.decode(c.jpg).planes), (what, c.name)
    yuv_cases = [c for c in cases if c.frame.bpm != 5 and len(c.frame.comps) == 3]
    outs, st, _ = _decode(hcj, ctx, yuv_cases, hcj.OUT_YUV)
    for c, o, s in zip(yuv_cases, outs, st):
        if c.status == 0:
            assert s == 0 and bytes(o) == orc.decode(c.jpg).yuv(), (what, c.name)
        elif c.status not in (-22, -25):
            assert s == c.status, (what, c.name, s)


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
def test_gpu_corpus_every_route(hcj, ctx, orc, monkeypatch, route):
    """The whole corpus in one batch: intervals of fewer than 128 blocks take K2, scans without DRI one K3 unit, long
    intervals K3 units; HCJ_LONG_RI_BLOCKS=1 sends every interval to K3, HCJ_SUB_LOG2=8 / HCJ_GUESS_BITS=64 give small
    images many subsequences and short warm-ups.  Coefficients equal the written ones, planes and YUV the oracle's,
    statuses the oracle's image by image (-23 included)."""
    for k, v in ROUTES[route].items():
        monkeypatch.setenv(k, v)
    cases = list(corpus().values())
    for c in cases:
        c.status = expected_status(orc, c.jpg)
    ris = {(c.ri, c.frame.bpm) for c in cases}
    assert any(ri == 0 for ri, _ in ris) and any(0 < ri * bpm < 128 for ri, bpm in ris) and any(ri * bpm >= 128 for ri, bpm in ris)
    _check_batch(hcj, ctx, orc, cases, route)


def _pillow_rgb(jpgs, simd=True):
    """Pillow's RGB of each file, in a subprocess; simd=False runs libjpeg-turbo's C code paths (JSIMD_FORCENONE=1)."""
    code = ("import io, sys, json, numpy as np\nfrom PIL import Image\n"
            "print(json.dumps([np.asarray(Image.open(io.BytesIO(bytes.fromhex(h))).convert('RGB')).tobytes().hex()"
            " for h in json.loads(sys.stdin.read())]))\n")
    env = dict(os.environ)
    env.pop("JSIMD_FORCENONE", None)
    if not simd:
        env["JSIMD_FORCENONE"] = "1"
    r = subprocess.run([sys.executable, "-c", code], input=json.dumps([j.hex() for j in jpgs]), capture_output=True, text=True,
                       env=env, check=True)
    return [bytes.fromhex(h) for h in json.loads(r.stdout)]


@pytest.mark.gpu
def test_gpu_libjpeg_rgb_equals_pillow(hcj, ctx):
    """T.81-legal files with custom tables: FLAG_LIBJPEG RGB24 equals Pillow (libjpeg-turbo reading the same tables).
    Files whose dequantised coefficients stay in the 12-bit range of an 8-bit encoder are compared with Pillow as it
    runs; the others with Pillow on libjpeg-turbo's C code paths, which the flag reproduces (its 16-bit SIMD IDCT
    leaves them there)."""
    pytest.importorskip("PIL.Image")
    cases = [c for c in corpus().values() if c.legal and c.status == 0]
    narrow = [_max_dequant(c) <= 2047 for c in cases]
    assert len(cases) >= 15 and sum(narrow) >= 10 and not all(narrow)
    outs, st = ctx.decode_batch([c.jpg for c in cases], hcj.OUT_RGB24, hcj.FLAG_DEFAULT | hcj.FLAG_LIBJPEG)
    assert st == [0] * len(cases)
    simd = dict(zip([c.name for c, n in zip(cases, narrow) if n], _pillow_rgb([c.jpg for c, n in zip(cases, narrow) if n])))
    plain = dict(zip([c.name for c in cases], _pillow_rgb([c.jpg for c in cases], simd=False)))
    for c, o, n in zip(cases, outs, narrow):
        assert bytes(o) == plain[c.name], c.name
        if n:
            assert bytes(o) == simd[c.name], c.name


@pytest.mark.gpu
def test_gpu_interleaved_table_sets(hcj, ctx, orc):
    """One batch of 40+ images with 20+ distinct table sets, Annex K images between them (A B A C A ...) and repeats, so
    that same-as-previous, set_index reuse and fresh table builds all occur; results checked image by image."""
    cases = corpus()
    a, b = cases["annexk0_ri0"], cases["annexk2_ri20"]
    others = [c for n, c in cases.items() if c.status == 0 and not n.startswith("annexk")]
    order = []
    for i, c in enumerate(others):
        order += [a if i % 3 else b, c] + ([c] if i % 4 == 0 else [])
    order += others[:5]
    sets = {tuple(sorted((k, tuple(l), tuple(v)) for k, (l, v) in c.tables.items())) for c in order}
    assert len(order) >= 40 and len(sets) >= 20
    _check_batch(hcj, ctx, orc, order, "interleaved")


@pytest.mark.gpu
def test_gpu_fixed_length_tables_redo_rounds(hcj, ctx, monkeypatch, capfd):
    """Fixed-length 8-bit AC codes, many small subsequences: the speculative decoder's fix-point rounds run more than
    once on the device (HCJ_SPEC_STATS) and the result is still exact."""
    monkeypatch.setenv("HCJ_SPEC_STATS", "1")
    monkeypatch.setenv("HCJ_SUB_LOG2", "8")
    monkeypatch.setenv("HCJ_GUESS_BITS", "64")
    c = corpus()["fixed8_ri0"]
    capfd.readouterr()
    b = ctx.batch([c.jpg], hcj.OUT_PLANES)
    try:
        b.decode_stages()
        assert np.array_equal(b.coefficients(0), c.coefs.astype(np.int16))
    finally:
        b.close()
    err = capfd.readouterr().err
    m = re.search(r"\[spec\].*rounds total (\d+) max (\d+)", err)
    assert m, err
    assert int(m.group(2)) > 1, err
