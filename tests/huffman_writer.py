"""TEST INFRASTRUCTURE: a baseline JPEG writer over given coefficients and arbitrary Huffman tables.

The oracle's encoder always writes the four Annex K tables.  This writer takes coefficient blocks in the layout of the
coefficient tap (int zig-zag, absolute DC, blocks in MCU order: what ``orc.decode(j, want_blocks=True).coefs_abs_dc()``
returns), a frame description and any DHT contents, and writes a complete file: 1-bit padding, FF 00 stuffing, RSTn.
It can also write symbol forms a T.81 encoder never emits: zero runs as (r, 0) symbols, blocks that end on coefficient
63 without an EOB, and an undefined code or an overlong run at a chosen block.  Plain Python + numpy.
"""
import numpy as np

# ITU-T T.81 Annex K.3 tables: (class, id) -> (lengths[16], values)
ANNEX_K = {
    (0, 0): ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12))),
    (0, 1): ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12))),
    (1, 0): ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D], bytes.fromhex(
        "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738"
        "393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5"
        "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa")),
    (1, 1): ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77], bytes.fromhex(
        "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a353637"
        "38393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3"
        "a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa")),
}
ANNEX_K = {k: (list(l), list(v)) for k, (l, v) in ANNEX_K.items()}

LUT_BITS, LUT_NSUB, LUT_SUB_BITS = 10, 8, 6  # hcj_common.h: HCJ_LUT_BITS, HCJ_LUT_NSUB, HCJ_LUT_SUB_BITS
FULL = LUT_NSUB  # prefix class: the model's full table in global memory
PRIMARY = -1  # prefix class: resolved by the primary table


def codes(lengths, values):
    """Specification.create_code_table: [(length, code, value)] in DHT order (canonical codes)."""
    out, code, pos = [], 0, 0
    for l in range(16):
        for i in range(lengths[l]):
            out.append((l + 1, code + i, values[pos + i]))
        code = (code + lengths[l]) << 1
        pos += lengths[l]
    return out


def full_table(lengths, values):
    """Tables.Lut over max_bits: int array of (length << 8 | value), 0 = no code; later codes overwrite earlier ones.
    None for an over-subscribed table (the model raises)."""
    cs = codes(lengths, values)
    mb = max(l for l, _, _ in cs)
    t = np.zeros(1 << mb, np.int32)
    for l, c, v in cs:
        lo = c << (mb - l)
        hi = lo + (1 << (mb - l))
        if hi > t.size:
            return None
        t[lo:hi] = (l << 8) | v
    return t


def classify(lengths, values):
    """What build_lut (hcj_host.cpp) makes of a table: (max_bits, cls) with cls[p] for every 10-bit prefix p:
    PRIMARY (resolved by the primary table, or no code at all), 0..7 (that shared-memory sub-table), FULL."""
    t = full_table(lengths, values)
    mb = int(np.log2(t.size))
    cls = np.full(1 << LUT_BITS, PRIMARY, np.int32)
    if mb <= LUT_BITS:
        return mb, cls
    sub = t.reshape(1 << LUT_BITS, -1)
    nsub = 0
    for p in range(1 << LUT_BITS):
        row = sub[p]
        if (row == row[0]).all() and (row[0] >> 8) <= LUT_BITS:
            continue
        if nsub < LUT_NSUB:
            cls[p] = nsub
            nsub += 1
        else:
            cls[p] = FULL
    return mb, cls


def optimal_lengths(freq, max_len=16, reserve=True):
    """T.81 K.2 as libjpeg's jpeg_gen_optimal_table does it (a reserved pseudo-symbol keeps the all-ones code free
    unless reserve=False), with the code-length limit `max_len` instead of 16.  freq: {symbol: count}.
    Returns (lengths[16], values)."""
    syms = [s for s in sorted(freq) if freq[s] > 0]
    if len(syms) == 1 and not reserve:
        return table_from_lengths({syms[0]: 1})
    f = [freq[s] for s in syms] + ([1] if reserve else [])
    n = len(f)
    codesize = [0] * n
    others = [-1] * n
    f = list(f)
    while True:
        c1 = c2 = -1
        v = None
        for i in range(n):
            if f[i] and (v is None or f[i] <= v):
                v, c1 = f[i], i
        v = None
        for i in range(n):
            if f[i] and i != c1 and (v is None or f[i] <= v):
                v, c2 = f[i], i
        if c2 < 0:
            break
        f[c1] += f[c2]
        f[c2] = 0
        codesize[c1] += 1
        while others[c1] >= 0:
            c1 = others[c1]
            codesize[c1] += 1
        others[c1] = c2
        codesize[c2] += 1
        while others[c2] >= 0:
            c2 = others[c2]
            codesize[c2] += 1
    bits = [0] * 64
    for c in codesize:
        if c:
            bits[c] += 1
    for i in range(63, max_len, -1):
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
    if reserve:
        i = max_len
        while bits[i] == 0:
            i -= 1
        bits[i] -= 1
    order = sorted(range(len(syms)), key=lambda k: (codesize[k], syms[k]))
    # lengths after the limit: hand them out again in order of the original code sizes
    lens = []
    for l in range(1, 17):
        lens += [l] * bits[l]
    sym_len = {syms[k]: lens[i] for i, k in enumerate(order)}
    return table_from_lengths(sym_len)


def table_from_lengths(sym_len, order=None):
    """{symbol: code length} -> (lengths[16], values) in order of (length, rank) where rank is the symbol's position
    in `order` (default: the symbol value)."""
    rank = {s: i for i, s in enumerate(order)} if order is not None else {}
    items = sorted(sym_len.items(), key=lambda kv: (kv[1], rank.get(kv[0], kv[0])))
    lengths = [0] * 16
    for _, l in items:
        lengths[l - 1] += 1
    return lengths, [s for s, _ in items]


def kraft_ok(lengths):
    return sum(n << (16 - (i + 1)) for i, n in enumerate(lengths)) <= 1 << 16


def size_of(v):
    v = abs(int(v))
    return v.bit_length()


def magnitude(v, size):
    return v if v >= 0 else v + (1 << size) - 1


class Frame:
    """A baseline frame: comps = [(component id, h, v, quant table id, dc table id, ac table id)], quant =
    {table id: 64 zig-zag entries}; a table with an entry above 255 (or listed in `wide_quant`) is written as 16-bit."""

    def __init__(self, width, height, comps, quant, wide_quant=()):
        self.width, self.height, self.comps, self.quant = width, height, list(comps), dict(quant)
        self.wide_quant = set(wide_quant) | {k for k, q in self.quant.items() if max(q) > 255}
        self.max_h = max(c[1] for c in self.comps)
        self.max_v = max(c[2] for c in self.comps)
        self.mcus_wide = -(-width // (8 * self.max_h))
        self.mcus_high = -(-height // (8 * self.max_v))
        self.block_comp = [k for k, c in enumerate(self.comps) for _ in range(c[1] * c[2])]
        self.bpm = len(self.block_comp)
        self.nblocks = self.mcus_wide * self.mcus_high * self.bpm


def bindings(frame, dhts):
    """(class, id) -> (lengths, values) as the model binds them: the DHT defined last wins."""
    out = {}
    for tc, th, lengths, values in dhts:
        out[(tc, th)] = (list(lengths), list(values))
    return out


class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, bits, n):
        self.acc = (self.acc << n) | bits
        self.n += n
        while self.n >= 8:
            self.n -= 8
            b = (self.acc >> self.n) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)
        self.acc &= (1 << self.n) - 1

    def flush_ones(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def _undefined_code(lengths, values):
    """A max_bits-bit pattern no code covers (the decoder's 'Can't find code')."""
    t = full_table(lengths, values)
    free = np.flatnonzero(t == 0)
    assert free.size, "the table has no unused code space"
    return int(free[-1]), int(np.log2(t.size))


def block_symbols(blk, diff, split_runs=False, omit_eob63=False):
    """The symbols of one block: [(is_ac, symbol, magnitude value, size)], DC first.  Standard run-length coding,
    or with split_runs zero runs of 2 or more written partly as (r, 0) symbols (skip r zeros, store a zero) instead of
    ZRL, and with omit_eob63 trailing zeros of 2 or more written as (r, 0) symbols up to coefficient 63 (no EOB)."""
    cat = size_of(diff)
    out = [(False, cat, diff, cat)]
    z = 1
    for pos in (np.flatnonzero(blk[1:]) + 1).tolist():
        run = pos - z
        v = int(blk[pos])
        if split_runs:
            while run >= 2:
                a = 2 + (run * 7 + z) % min(15, run - 1)
                out.append((True, (a - 1) << 4, 0, 0))
                run -= a
                z += a
        while run >= 16:
            out.append((True, 0xF0, 0, 0))
            run -= 16
        s = size_of(v)
        out.append((True, (run << 4) | s, v, s))
        z = pos + 1
    if z <= 63:
        t = 64 - z
        if omit_eob63 and t >= 2:
            while t > 0:
                a = t if t <= 16 else (16 if t - 16 != 1 else 15)
                out.append((True, (a - 1) << 4, 0, 0))
                t -= a
        else:
            out.append((True, 0x00, 0, 0))
    return out


def write_scan(coefs, frame, dhts, restart_interval=0, split_runs=False, omit_eob63=False, inject=None, rotate=False,
               used=None):
    """The entropy-coded segment (RSTn included, no EOI) of `coefs` (nblocks x 64, zig-zag, absolute DC).
    inject: (block, kind) with kind 'dc_code' (an undefined DC code instead of the block's DC symbol), 'ac_code' (an
    undefined AC code right after its DC symbol) or 'overrun' (after its DC: three ZRL and (15, 1), a run past
    coefficient 63).  rotate: a symbol with several codes (a value listed more than once) uses them in turn.
    used: a dict that receives {(class, id): {(length, code)}} of the codes written."""
    coefs = np.asarray(coefs)
    assert coefs.shape == (frame.nblocks, 64), (coefs.shape, frame.nblocks)
    tabs = bindings(frame, dhts)
    enc = {}
    for key, (l, v) in tabs.items():
        m = {}
        for length, code, val in codes(l, v):
            m.setdefault(val, []).append((code, length))
        enc[key] = m
    turn = {}
    w = _Bits()
    pred = [0] * len(frame.comps)
    nmcu = frame.mcus_wide * frame.mcus_high
    bpm = frame.bpm

    def put_symbol(key, sym):
        cl = enc[key].get(sym)
        if cl is None:
            raise KeyError("symbol 0x%02x is not in table %s" % (sym, key))
        k = 0
        if rotate and len(cl) > 1:
            k = turn.get((key, sym), 0)
            turn[(key, sym)] = (k + 1) % len(cl)
        code, length = cl[k]
        w.put(code, length)
        if used is not None:
            used.setdefault(key, set()).add((length, code))

    for mcu in range(nmcu):
        if restart_interval and mcu and mcu % restart_interval == 0:
            w.flush_ones()
            w.out += bytes([0xFF, 0xD0 + (mcu // restart_interval - 1) % 8])
            pred = [0] * len(frame.comps)
        for k in range(bpm):
            b = mcu * bpm + k
            c = frame.block_comp[b % bpm]
            cid, _, _, _, td, ta = frame.comps[c]
            blk = coefs[b]
            diff = int(blk[0]) - pred[c]
            pred[c] = int(blk[0])
            kind = inject[1] if inject is not None and inject[0] == b else None
            syms = block_symbols(blk, diff, split_runs, omit_eob63)
            if kind == "dc_code":
                code, nb = _undefined_code(*tabs[(0, td)])
                w.put(code, nb)
                syms = syms[1:]
            elif kind in ("ac_code", "overrun"):
                syms = syms[:1] + ([None] if kind == "ac_code" else [(True, 0xF0, 0, 0)] * 3 + [(True, 0xF1, 1, 1)]) + syms[1:]
            for s in syms:
                if s is None:
                    code, nb = _undefined_code(*tabs[(1, ta)])
                    w.put(code, nb)
                    continue
                is_ac, sym, val, size = s
                put_symbol((1, ta) if is_ac else (0, td), sym)
                if size:
                    w.put(magnitude(val, size), size)
    w.flush_ones()
    return bytes(w.out)


def write_headers(frame, dhts, restart_interval=0):
    """SOI, DQT (one table per segment), SOF0, DHT (one table per segment, in the given order), DRI, SOS."""
    def seg(code, payload):
        return bytes([0xFF, code]) + (len(payload) + 2).to_bytes(2, "big") + payload

    out = [b"\xff\xd8"]
    for tq, q in sorted(frame.quant.items()):
        wide = tq in frame.wide_quant
        out.append(seg(0xDB, bytes([(1 if wide else 0) << 4 | tq]) + b"".join(int(x).to_bytes(2 if wide else 1, "big") for x in q)))
    sof = bytes([8]) + frame.height.to_bytes(2, "big") + frame.width.to_bytes(2, "big") + bytes([len(frame.comps)])
    for cid, h, v, tq, _, _ in frame.comps:
        sof += bytes([cid, h << 4 | v, tq])
    out.append(seg(0xC0, sof))
    for tc, th, lengths, values in dhts:
        out.append(seg(0xC4, bytes([tc << 4 | th]) + bytes(lengths) + bytes(values)))
    if restart_interval:
        out.append(seg(0xDD, restart_interval.to_bytes(2, "big")))
    sos = bytes([len(frame.comps)]) + b"".join(bytes([cid, td << 4 | ta]) for cid, _, _, _, td, ta in frame.comps) + b"\x00\x3f\x00"
    out.append(seg(0xDA, sos))
    return b"".join(out)


def write_jpeg(coefs, frame, dhts, restart_interval=0, **opts):
    """A complete file: headers, the entropy-coded segment, EOI.  opts: see write_scan."""
    return write_headers(frame, dhts, restart_interval) + write_scan(coefs, frame, dhts, restart_interval, **opts) + b"\xff\xd9"


def read_file(jpg):
    """(frame, dhts, restart interval, entropy-coded segment up to the EOI) of a baseline file with one table per DHT
    segment or several."""
    p, quant, wide, dhts, ri, sof, sos = 2, {}, set(), [], 0, None, None
    while True:
        assert jpg[p] == 0xFF
        code = jpg[p + 1]
        n = int.from_bytes(jpg[p + 2:p + 4], "big")
        body = jpg[p + 4:p + 2 + n]
        p += 2 + n
        if code == 0xDB:
            i = 0
            while i < len(body):
                pq, tq = body[i] >> 4, body[i] & 15
                w = 2 if pq else 1
                quant[tq] = [int.from_bytes(body[i + 1 + w * k:i + 1 + w * k + w], "big") for k in range(64)]
                if pq:
                    wide.add(tq)
                i += 1 + 64 * w
        elif code == 0xC4:
            i = 0
            while i < len(body):
                lengths = list(body[i + 1:i + 17])
                dhts.append((body[i] >> 4, body[i] & 15, lengths, list(body[i + 17:i + 17 + sum(lengths)])))
                i += 17 + sum(lengths)
        elif code == 0xDD:
            ri = int.from_bytes(body[:2], "big")
        elif code == 0xC0:
            sof = body
        elif code == 0xDA:
            sos = body
            break
    comps = {}
    for k in range(sof[5]):
        cid, hv, tq = sof[6 + 3 * k:9 + 3 * k]
        comps[cid] = (cid, hv >> 4, hv & 15, tq)
    sc = [comps[sos[1 + 2 * k]] + (sos[2 + 2 * k] >> 4, sos[2 + 2 * k] & 15) for k in range(sos[0])]
    frame = Frame(int.from_bytes(sof[3:5], "big"), int.from_bytes(sof[1:3], "big"), sc, quant, wide)
    end = jpg.rindex(b"\xff\xd9")
    return frame, dhts, ri, jpg[p:end]


def symbol_counts(coefs, frame, restart_interval=0, split_runs=False, omit_eob63=False):
    """{(class, component index): {symbol: count}} of what write_scan writes (no injection)."""
    out = {}
    pred = [0] * len(frame.comps)
    for b in range(frame.nblocks):
        if restart_interval and b % (restart_interval * frame.bpm) == 0:
            pred = [0] * len(frame.comps)
        c = frame.block_comp[b % frame.bpm]
        blk = coefs[b]
        diff = int(blk[0]) - pred[c]
        pred[c] = int(blk[0])
        for is_ac, sym, _, _ in block_symbols(blk, diff, split_runs, omit_eob63):
            d = out.setdefault((int(is_ac), c), {})
            d[sym] = d.get(sym, 0) + 1
    return out
