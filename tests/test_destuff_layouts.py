"""The destuff kernel (K1: k_destuff, k_destuff_count / _scan / _write) and the restart-interval plumbing behind it on
scan layouts the reference encoder never writes.

Files come from tests/scan_layout.py: oracle and huffman_writer files re-emitted with the scan starting at every phase
mod 16, stuffed pairs, restart markers and terminators at every byte of a thread's 16 and at byte 4095 of a tile,
words with two dropped bytes, threads with eight, a tile of nothing but FF 00, empty intervals, RSTn numbered any way,
other terminators with data behind them, junk behind the last MCU of an interval or scan, and truncation.  The CPU
tests check the layout writer against its source files, the construction against the numpy reference and the oracle,
and that the corpus keeps covering these layouts; the GPU tests decode it on both destuff forms and both interval
routes, through both entry points, next to look-back neighbours of very different sizes and around the 65 535-tile
switch between the two forms.
"""
import ctypes as C
import functools

import numpy as np
import pytest

import huffman_writer as hw
import scan_layout as sl
import synth

# name: (chroma, width, height, restart interval, seed)
SOURCES = {"420_r0": (420, 64, 48, 0, 1), "420_r1": (420, 64, 48, 1, 2), "420_r3": (420, 80, 64, 3, 3),
           "422_r1": (422, 48, 32, 1, 4), "444_r3": (444, 40, 24, 3, 5), "400_r0": (400, 56, 40, 0, 6),
           "400_r1": (400, 56, 40, 1, 7), "420_r40": (420, 640, 368, 40, 8), "420_long_r0": (420, 640, 368, 0, 9)}


def _orc():
    from oracle import pyoracle

    pyoracle.build()
    return pyoracle


@functools.lru_cache(None)
def sources():
    """Oracle files, and one huffman_writer file with tables K.2-optimised for its content (not Annex K)."""
    orc = _orc()
    out = {n: orc.encode(synth.frame(s, w, h, c), w, h, c, 75, restart_interval=ri) for n, (c, w, h, ri, s) in SOURCES.items()}
    frame, _, _, _ = hw.read_file(out["420_r1"])
    coefs = orc.decode(out["420_r1"], want_blocks=True).coefs_abs_dc()
    counts = hw.symbol_counts(coefs, frame, 2)
    dhts = []
    for tc in (0, 1):
        for tid, comps in ((0, (0,)), (1, (1, 2))):
            freq = {}
            for ci in comps:
                for s, n in counts[(tc, ci)].items():
                    freq[s] = freq.get(s, 0) + n
            dhts.append((tc, tid) + hw.optimal_lengths(freq))
    out["hw_r2"] = hw.write_jpeg(coefs, frame, dhts, 2)
    return out


def _nparts(src):
    return len(sl.split(src)[1])


def _junk(seed, n, ff=0.2):
    """n random bytes, a fraction `ff` of them FF (written stuffed)."""
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, n, dtype=np.uint8)
    b[rng.random(n) < ff] = 0xFF
    return b.tobytes()


def _with_len_mod16(r, **kw):
    """emit(**kw) with raw bytes behind the terminator so that the file length is r mod 16."""
    lay = sl.emit(**kw)
    return sl.emit(after=kw.pop("after", b"") + b"\x5a" * ((r - len(lay.jpg)) % 16), **kw)


def _com_for_phase(src, ph):
    """COM payload length that makes the scan start at phase ph mod 16 (the segment adds 4 + length bytes)."""
    return (ph - 4 - sl.scan_start(src)) % 16


def _zero_scan(src, ph):
    """`src` cut right behind its SOS, the scan at phase ph."""
    com = _com_for_phase(src, ph)
    return sl.emit(src, com=com, trunc=sl.emit(src, com=com).scan_start)


@functools.lru_cache(None)
def corpus():
    """{name: (Layout, source name)}."""
    src = sources()
    c = {}
    # the scan at every phase; stuffed pairs everywhere, each marker at a chosen byte of its thread's 16, the
    # terminator at byte `ph` of its 16, every file length mod 16
    for ph in range(16):
        s = ["420_r1", "422_r1", "444_r3", "hw_r2"][ph % 4]
        n = _nparts(src[s])
        pads = {k: [_junk(100 * ph + k, 3 + (7 * k + ph) % 37, 0.3), ((ph + 3 * k) % 16, 16) if k + 1 < n else (ph, 16)]
                for k in range(n)}
        c["phase%02d" % ph] = (_with_len_mod16(ph, src=src[s], com=_com_for_phase(src[s], ph), pads=pads, seed=ph), s)
    # tile and word edges: a stuffed pair and a restart marker with their FF at byte 4095 of a tile, two-drop words
    # {0, 2}, {1, 3}, {0, 3}, a thread of eight FF 00, a tile of FF 00 only; then the terminator at byte 4095
    words = [(0, 16), b"\xff\xff", (1, 16), b"\xff\xff", (0, 16), b"\xff\x01\xff", (0, 16), b"\xff" * 8, (0, 4096),
             b"\xff" * 2048]
    for s, com in (("420_r1", None), ("400_r1", 5), ("hw_r2", 11)):
        n = _nparts(src[s])
        pads = {0: [(4095, 4096), b"\xff", b"\x12\x34"], 1: [(4095, 4096)], 2: words, n - 1: [(4094, 4096)]}
        c["edges_" + s] = (sl.emit(src[s], com=com, pads=pads, seed=7), s)
    for s, com in (("420_r0", None), ("400_r0", 2)):
        c["edges_" + s] = (sl.emit(src[s], com=com, pads={0: [(4095, 4096), b"\xff", b"\x12"] + words + [(4095, 4096)]}), s)
    # restart numbering, terminators, data behind them
    c["rst_const"] = (sl.emit(src["420_r3"], rst="const", pads={2: [b"\xff"]}), "420_r3")
    c["rst_random"] = (sl.emit(src["422_r1"], rst="random", seed=3, com=1), "422_r1")
    c["rst_random_hw"] = (sl.emit(src["hw_r2"], rst="random", seed=4, com=9), "hw_r2")
    c["fill_ff_before_eoi"] = (sl.emit(src["420_r3"], term=b"\xff\xff\xff\xff\xd9", pads={6: [(15, 16)]}), "420_r3")
    c["term_dht"] = (sl.emit(src["420_r1"], term=b"\xff\xc4\x00\x1f", after=_junk(5, 3000), com=3), "420_r1")
    marks = _junk(6, 2_000_000, 0.05).replace(b"\xff\x00", b"\xff\xd0").replace(b"\xff\x01", b"\xff\xd9")
    c["term_then_2mb_with_markers"] = (sl.emit(src["444_r3"], after=marks, com=4), "444_r3")
    c["term_then_1_5mb_r0"] = (sl.emit(src["420_r0"], after=marks[:1_500_001], com=13), "420_r0")
    c["rst_without_dri"] = (sl.emit(src["420_r0"], term=b"\xff\xd3", after=b"\x00\xff\xd0\x11\xff\xd9", com=6), "420_r0")
    c["junk_before_eoi_gray"] = (sl.emit(src["400_r0"], pads={0: [_junk(8, 9000, 0.5)]}, com=8), "400_r0")
    # broken on purpose: what the construction implies, -20 / -21 / -9
    n1 = _nparts(src["420_r1"])
    lay = sl.emit(src["420_r1"], pads={3: [_junk(9, 300)]})
    c["trunc_mid"] = (sl.emit(src["420_r1"], pads={3: [_junk(9, 300)]}, trunc=(lay.scan_start + lay.term) // 2), "420_r1")
    lay = sl.emit(src["420_r3"], pads={6: [b"\x01\xff\x02"]})
    c["trunc_after_stuffed_ff"] = (sl.emit(src["420_r3"], pads={6: [b"\x01\xff\x02"]}, trunc=lay.term - 2), "420_r3")
    c["trunc_inside_eoi"] = (sl.emit(src["422_r1"], trunc=-1, com=14), "422_r1")
    lay = sl.emit(src["420_r1"], pads={4: [(7, 16)]})
    c["trunc_inside_rst"] = (sl.emit(src["420_r1"], pads={4: [(7, 16)]}, trunc=_marker_pos(lay, 4) + 1), "420_r1")
    for ph in (0, 3, 10, 15):  # phase 0: no destuff tile at all; else one tile without a byte of the scan
        c["zero_scan_phase%02d" % ph] = (_zero_scan(src["420_r1"], ph), "420_r1")
    c["dropped_marker"] = (sl.emit(src["420_r1"], drop={2}), "420_r1")
    c["extra_marker"] = (sl.emit(src["422_r1"], dup={4}), "422_r1")
    c["marker_at_scan_start"] = (sl.emit(src["420_r3"], dup={-1}, com=12), "420_r3")
    c["empty_first_interval"] = (sl.emit(src["420_r1"], dup={-1}, drop={n1 - 2}, com=1), "420_r1")
    c["empty_middle_interval"] = (sl.emit(src["420_r1"], dup={3}, drop={n1 - 2}, com=2), "420_r1")
    c["empty_last_interval"] = (sl.emit(src["420_r1"], dup={n1 - 1}, drop={0}, com=15), "420_r1")
    return c


def _marker_pos(lay, m):
    """File offset of the FF of restart marker m (0-based) of a layout."""
    ref = sl.reference(lay.jpg, lay.scan_start, True)
    return int(ref.rst[m])


# ---- CPU: the writer, the construction, the reference, the oracle ---------------------------------------------------
@pytest.mark.parametrize("name", list(SOURCES) + ["hw_r2"])
def test_reemit_without_layout_is_identity(name):
    src = sources()[name]
    lay = sl.emit(src)
    assert lay.jpg == src and lay.status == 0
    assert sl.scan_start(src) == _orc().header_decode(src).scan_bit_pos // 8


@pytest.mark.parametrize("name", sorted(corpus()))
def test_construction_equals_reference_and_oracle(name):
    """The construction's destuffed bytes, interval starts and terminator equal the numpy reference's (and without DRI
    the oracle's extract_entropy_coded_bits); the oracle's status equals the construction's, status-0 files decode to
    the source's coefficients and planes."""
    orc = _orc()
    lay, s = corpus()[name]
    src = sources()[s]
    assert lay.scan_start == orc.header_decode(lay.jpg).scan_bit_pos // 8
    ref = sl.reference(lay.jpg, lay.scan_start, lay.restart)
    assert ref.term == lay.term
    if lay.term is not None:
        assert ref.destuffed == lay.destuffed
        assert ref.starts == lay.starts
        if not lay.restart:
            assert ref.destuffed == orc.extract_entropy_coded_bits(lay.jpg, lay.scan_start)
    assert orc.decode_status(lay.jpg) == lay.status, name
    if lay.status == 0:
        a, b = orc.decode(src, want_blocks=True), orc.decode(lay.jpg, want_blocks=True)
        assert np.array_equal(a.coefs_abs_dc(), b.coefs_abs_dc())
        assert all(np.array_equal(p, q) for p, q in zip(a.planes, b.planes))
        assert b.entropy_len == len(lay.destuffed)


def test_reference_matches_oracle_on_random_bytes():
    """The reference's byte rule against the oracle's on scans of random bytes with dense FF, markers and zeros."""
    orc = _orc()
    src = sources()["420_r0"]
    head = src[:sl.scan_start(src)]
    for seed in range(40):
        rng = np.random.default_rng(seed)
        body = rng.choice(np.array([0x00, 0xFF, 0xD0, 0xD7, 0xD9, 0x12, 0xFE], np.uint8), 4000).tobytes()
        jpg = head + body + b"\xff\xd9"
        ref = sl.reference(jpg, len(head), False)
        assert ref.destuffed == orc.extract_entropy_coded_bits(jpg, len(head))


# ---- CPU: coverage that cannot drift ------------------------------------------------------------------------------------
def test_corpus_coverage():
    """Placed by K1's tiling, the status-0 files hold: a stuffed pair and a restart marker with the FF at every byte of
    a thread's 16 and at byte 4095 of a tile; the two-drop words {0, 2}, {1, 3}, {0, 3}; a thread of eight dropped
    bytes and a tile of FF 00 only; scans at every phase and files of every length mod 16.  Over the whole corpus:
    terminators at every byte mod 16 and at 4095, empty first / middle / last intervals, zero-byte scans with 0 and 1
    tiles, megabytes behind an early terminator."""
    cases = corpus().values()
    ok = [lay for lay, _ in cases if lay.status == 0]
    refs = [(lay, sl.reference(lay.jpg, lay.scan_start, lay.restart)) for lay in ok]
    stuffed = set()
    rst = set()
    words, eight, full_tile = set(), False, False
    for lay, ref in refs:
        for pos, into in ((ref.stuffed, stuffed), (ref.rst, rst)):
            t, th, w, b = sl.place(pos, lay.scan_start)
            into.update((4 * w + b).tolist())
            if np.any(th * 16 + 4 * w + b == 4095):
                into.add("tile4095")
        d = sl.dropped_words(ref, lay.scan_start)
        words.update(d.tolist())
        pad = (-d.size) % 4
        per_thread = np.concatenate([d, np.zeros(pad, d.dtype)]).reshape(-1, 4)
        drops = sum(((per_thread >> i) & 1).sum(axis=1) for i in range(4))
        eight |= bool((drops == 8).any())
        pad = (-per_thread.shape[0]) % 256
        tiles = np.concatenate([drops, np.zeros(pad, drops.dtype)]).reshape(-1, 256)
        full_tile |= bool((tiles == 8).all(axis=1).any())
    for into in (stuffed, rst):
        assert set(range(16)) | {"tile4095"} <= into, into
    assert {0b0101, 0b1010, 0b1001} <= words
    assert eight and full_tile
    assert {(lay.term - (lay.scan_start & ~15)) % 16 for lay, _ in cases if lay.term is not None} == set(range(16))
    assert any((lay.term - (lay.scan_start & ~15)) % 4096 == 4095 for lay, _ in cases if lay.term is not None)
    assert {lay.scan_start % 16 for lay in ok} == set(range(16))
    assert {len(lay.jpg) % 16 for lay in ok} == set(range(16))
    # empty intervals (an interval with MCUs has at least one byte, so these files are -9 by construction)
    empties = set()
    for lay, _ in cases:
        lens = [b - a for a, b in zip(lay.starts, lay.starts[1:] + [len(lay.destuffed)])]
        if lay.restart and lay.term is not None:
            for i, n in enumerate(lens):
                if n == 0:
                    empties.add("first" if i == 0 else "last" if i + 1 == len(lens) else "middle")
    assert empties == {"first", "middle", "last"}
    assert {lay.status for lay, _ in cases} == {0, -9, -20, -21}
    # scans of zero bytes with 0 and with 1 destuff tile, data behind an early terminator spanning many tiles
    zero = [lay for lay, _ in cases if len(lay.jpg) == lay.scan_start]
    assert {lay.scan_start % 16 == 0 for lay in zero} == {True, False}
    assert any(lay.term is not None and (len(lay.jpg) - lay.term) > 100 * sl.TILE for lay, _ in cases)


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


def _entropy(hcj, b, i, cap):
    """Batch.entropy with room for `cap` bytes."""
    out = np.zeros(cap + 16, np.uint8)
    n = C.c_size_t()
    st = hcj.lib().hcj_batch_fetch_entropy(b.ctx._h, b._h, i, out.ctypes.data, out.size, C.byref(n))
    assert st == 0, st
    return out[: n.value].tobytes()


def _check(hcj, ctx, orc, items, what, yuv=True):
    """items: [(Layout or raw bytes, source bytes or None)].  Resident batch: statuses against the construction (or
    the oracle for raw files), coefficients of status-0 images against the source's, entropy against the reference.
    One-call form: statuses and YUV / planes against the oracle."""
    jpgs = [x.jpg if isinstance(x, sl.Layout) else x for x, _ in items]
    want = [x.status if isinstance(x, sl.Layout) else orc.decode_status(x) for x, _ in items]
    with ctx.batch(jpgs, hcj.OUT_PLANES) as b:
        b.decode()
        outs, st = b.fetch()
        assert st == want, (what, [(i, s, w) for i, (s, w) in enumerate(zip(st, want)) if s != w])
        for i, ((x, src), s) in enumerate(zip(items, st)):
            if not isinstance(x, sl.Layout) or b.host_status[i] != 0:
                continue
            if s != -20:
                assert _entropy(hcj, b, i, len(x.jpg)) == sl.reference(x.jpg, x.scan_start, x.restart).destuffed, (what, i)
            if s == 0:
                ref = orc.decode(src, want_blocks=True)
                assert np.array_equal(b.coefficients(i), ref.coefs_abs_dc().astype(np.int16)), (what, i)
                assert bytes(outs[i]) == b"".join(p.tobytes() for p in ref.planes), (what, i)
    if yuv:
        outs, st = ctx.decode_batch(jpgs, hcj.OUT_YUV)
        for i, (j, s, w) in enumerate(zip(jpgs, st, want)):
            d = None if w != 0 else orc.decode(j)
            if d is not None and d.yuv_status == 0:
                assert s == 0 and bytes(outs[i]) == d.yuv(), (what, i)
            elif d is None:
                assert s == w, (what, i, s, w)


DESTUFF = {"one_pass": {}, "three_pass": {"HCJ_DESTUFF_3PASS": "1"}}
ROUTE = {"default": {}, "long_ri_1": {"HCJ_LONG_RI_BLOCKS": "1"}}


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTE))
@pytest.mark.parametrize("form", list(DESTUFF))
def test_gpu_corpus(hcj, ctx, orc, monkeypatch, form, route):
    """The whole corpus (twice, 100+ images: the one-call form runs several chunks) in one batch."""
    for k, v in {**DESTUFF[form], **ROUTE[route]}.items():
        monkeypatch.setenv(k, v)
    src = sources()
    items = [(lay, src[s]) for lay, s in corpus().values()]
    items = items + items[::-1]
    assert len(items) > 40
    _check(hcj, ctx, orc, items, (form, route))


def _tiles(lay):
    return -(-(len(lay.jpg) - (lay.scan_start & ~15)) // sl.TILE)


def _padded(src, rel, interval=0, com=None):
    """`src` with filler behind interval `interval` so that its scan, from scan_start & ~15 to the end of the file, is
    `rel` bytes long (the filler holds no FF: the length is linear in the filler's end offset)."""
    x1 = 1 << 16
    lay = sl.emit(src, com=com, pads={interval: [x1]})
    tail = len(lay.jpg) - (lay.scan_start & ~15) - x1
    lay = sl.emit(src, com=com, pads={interval: [rel - tail]})
    assert len(lay.jpg) - (lay.scan_start & ~15) == rel
    return lay


@pytest.mark.gpu
@pytest.mark.parametrize("form", list(DESTUFF))
def test_gpu_lookback_neighbours(hcj, ctx, orc, monkeypatch, form):
    """Scans of 0, 1, 2, 33 and 1100 tiles side by side, with images that fail on the host and zero-byte scans at
    several phases between them: no tile is ever counted into another image's prefix."""
    for k, v in DESTUFF[form].items():
        monkeypatch.setenv(k, v)
    src = sources()
    zero = [_zero_scan(src["420_r1"], ph) for ph in (0, 1, 8, 15)]
    assert [_tiles(z) for z in zero] == [0, 1, 1, 1]
    sized = [(_padded(src[s], t * sl.TILE - 100, i, c), src[s]) for s, t, i, c in
             (("420_r1", 1, 0, None), ("420_r3", 2, 1, 3), ("422_r1", 33, 5, 7), ("420_r1", 1100, 10, 1), ("444_r3", 33, 4, None))]
    bad = b"\xff\xd8\xff\xdb\x00\x03\x00\xff\xd9"
    items = []
    for k in range(3):
        for j, x in enumerate(sized):
            items += [x, (zero[(j + k) % 4], None)]
            if (j + k) % 2:
                items.append((bad, None))
    assert sorted({_tiles(x) for x, _ in items if isinstance(x, sl.Layout)}) == [0, 1, 2, 33, 1100]
    _check(hcj, ctx, orc, items, form)


@functools.lru_cache(None)
def junk_files():
    """Long intervals (K3 units: 240 blocks each) with 0-20 KB of junk behind some of them, and a DRI-free scan with
    64 KB / 1 MB of junk in front of EOI."""
    src = sources()
    pads = {0: [_junk(11, 20_000)], 5: [b"\x01"], 7: [_junk(12, 5_000, 0.5)], 13: [_junk(13, 700, 0.9)], 22: [_junk(14, 12_000)]}
    out = [(sl.emit(src["420_r40"], pads=pads, com=3), "420_r40"),
           (sl.emit(src["420_r40"], pads={k: [_junk(20 + k, 16 * k + 1)] for k in range(23)}), "420_r40")]
    for n, com in ((64 << 10, None), (1 << 20, 5)):
        out.append((sl.emit(src["420_long_r0"], pads={0: [_junk(n, n)]}, com=com), "420_long_r0"))
    return out


def test_junk_files_construction():
    orc = _orc()
    for lay, s in junk_files():
        assert lay.status == 0 and orc.decode_status(lay.jpg) == 0
        assert np.array_equal(orc.decode(lay.jpg, want_blocks=True).coefs_abs_dc(),
                              orc.decode(sources()[s], want_blocks=True).coefs_abs_dc())


@pytest.mark.gpu
@pytest.mark.parametrize("sub", ["default", "sub_log2_8"])
def test_gpu_spec_decoder_ignores_junk(hcj, ctx, orc, monkeypatch, sub):
    """Junk behind the last MCU of a K3 unit is cut into subsequences and synchronised like real data, but none of it
    reaches the coefficients or the status (HCJ_SUB_LOG2=8: the junk spans many subsequences)."""
    if sub != "default":
        monkeypatch.setenv("HCJ_SUB_LOG2", "8")
    src = sources()
    _check(hcj, ctx, orc, [(lay, src[s]) for lay, s in junk_files()], sub)


@pytest.mark.gpu
def test_gpu_model_without_restart_extension(hcj, ctx, orc):
    """flags=0 (the model alone): the first RSTn ends the scan, so the entropy-coded segment is the first interval's
    payload (with its padding) and the frame decodes as the model decodes it; FF fill in front of EOI decodes alike with and without
    FLAG_T81_TABLES."""
    names = ["rst_const", "phase05", "edges_420_r1", "empty_first_interval"]
    lays = [corpus()[n][0] for n in names]
    want = [orc.decode_status(lay.jpg, restart_ext=False) for lay in lays]
    with ctx.batch([lay.jpg for lay in lays], hcj.OUT_PLANES, 0) as b:
        b.decode()
        outs, st = b.fetch()
        assert st == want
        for i, (lay, n) in enumerate(zip(lays, names)):
            assert _entropy(hcj, b, i, len(lay.jpg)) == lay.destuffed[:lay.starts[1]], n
            if st[i] == 0:
                assert bytes(outs[i]) == b"".join(p.tobytes() for p in orc.decode(lay.jpg, restart_ext=False).planes), n
    fill = corpus()["fill_ff_before_eoi"][0].jpg
    a, sa = ctx.decode_batch([fill], hcj.OUT_YUV, hcj.FLAG_DEFAULT)
    b, sb = ctx.decode_batch([fill], hcj.OUT_YUV, hcj.FLAG_DEFAULT | hcj.FLAG_T81_TABLES)
    assert sa == sb == [0] and bytes(a[0]) == bytes(b[0]) == orc.decode(fill).yuv()


@pytest.mark.gpu
@pytest.mark.parametrize("ntiles", [65535, 65536])
def test_gpu_scan_at_tile_limit(hcj, ctx, orc, ntiles):
    """A small DRI frame (intervals of 6 blocks: K2) whose second interval is padded so that the scan spans exactly
    65 535 tiles to the last byte (the one-pass kernel's largest grid) or 65 536, the last holding only the D9 of EOI (the
    three kernels, chosen automatically)."""
    s = sources()["420_r1"]
    lay = _padded(s, 65535 * sl.TILE + (ntiles - 65535), interval=1, com=2)
    assert lay.status == 0 and _tiles(lay) == ntiles
    with ctx.batch([lay.jpg], hcj.OUT_PLANES) as b:
        b.decode()
        _, st = b.fetch()
        assert st == [0]
        assert _entropy(hcj, b, 0, len(lay.jpg)) == lay.destuffed
        assert np.array_equal(b.coefficients(0), orc.decode(s, want_blocks=True).coefs_abs_dc().astype(np.int16))
