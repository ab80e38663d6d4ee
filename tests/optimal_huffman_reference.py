"""TEST INFRASTRUCTURE: reference for HCJ_ENC_OPTIMIZE_HUFFMAN (include/hcjpeg.h, DESIGN.md 5).

gen_optimal_table is a literal restatement of libjpeg's jpeg_gen_optimal_table (jchuff.c, T.81 Annex K.2): HUFFVAL is
ordered by the code size BEFORE the 16-bit length limit, then by symbol (huffman_writer.optimal_lengths gets the lengths
right but orders the values by the final length).  optimized_file turns a default-table file of the encoder into the
file the flag writes: the same coefficients re-coded with per-frame tables."""
from oracle import pyoracle as orc

import huffman_writer as hw

MAX_CLEN = 64  # code sizes before the limit: counts below 2^32 keep them under 50


def gen_optimal_table(freq, info=None):
    """freq: {symbol: count} or a sequence of 256 counts; the reserved symbol 256 gets count 1.  Returns (bits[16],
    huffval).  info (a dict) receives "max_codesize", the longest code size before the limit."""
    f = [0] * 257
    items = freq.items() if isinstance(freq, dict) else enumerate(freq)
    for s, c in items:
        f[int(s)] = int(c)
    f[256] = 1
    codesize = [0] * 257
    others = [-1] * 257
    while True:
        c1, v = -1, None
        for i in range(257):
            if f[i] and (v is None or f[i] <= v):
                v, c1 = f[i], i
        c2, v = -1, None
        for i in range(257):
            if f[i] and (v is None or f[i] <= v) and i != c1:
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
    bits = [0] * MAX_CLEN
    for i in range(257):
        if codesize[i]:
            bits[codesize[i]] += 1
    i = MAX_CLEN - 1
    while i > 16:
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
        i -= 1
    while i > 0 and bits[i] == 0:
        i -= 1
    if i > 0:
        bits[i] -= 1
    huffval = [j for l in range(1, MAX_CLEN) for j in range(256) if codesize[j] == l]
    if info is not None:
        info["max_codesize"] = max(codesize)
    return bits[1:17], huffval


def table_counts(coefs, frame, restart_interval):
    """{(class, table id): {symbol: count}} of the scan the encoder writes for `coefs`: hw.symbol_counts merged over the
    components that share a table."""
    out = {}
    for (cls, c), d in hw.symbol_counts(coefs, frame, restart_interval).items():
        tid = frame.comps[c][5 if cls else 4]
        m = out.setdefault((cls, tid), {})
        for s, n in d.items():
            m[s] = m.get(s, 0) + n
    return out


def segments(jpg):
    """[(marker, offset, total length)] of the header segments up to and including SOS."""
    out, p = [], 2
    while True:
        code = jpg[p + 1]
        n = 2 + int.from_bytes(jpg[p + 2:p + 4], "big")
        out.append((code, p, n))
        p += n
        if code == 0xDA:
            return out


def optimized_file(default_jpg, info=None, coefs=None):
    """The file HCJ_ENC_OPTIMIZE_HUFFMAN writes for the frame whose default-table file is `default_jpg`: the default
    header with each DHT payload replaced in place by the frame's optimal table, the scan re-coded with those tables,
    EOI.  The coefficients are the oracle decoder's, or `coefs` (the encoder's Block.quant tap, orc.encode(...,
    want_blocks=True)) for files the model's decoder does not read back, such as some at quality 1.  info (a dict)
    receives "max_codesize" over the tables."""
    frame, dhts, ri, _ = hw.read_file(default_jpg)
    if coefs is None:
        coefs = orc.decode(default_jpg, want_blocks=True).coefs_abs_dc()
    counts = table_counts(coefs, frame, ri)
    new_dhts, tables, mx = [], {}, 0
    for tc, th, _, _ in dhts:
        i = {}
        tables[(tc, th)] = gen_optimal_table(counts.get((tc, th), {}), i)
        mx = max(mx, i["max_codesize"])
        new_dhts.append((tc, th) + tables[(tc, th)])
    if info is not None:
        info["max_codesize"] = mx
    head = bytearray(default_jpg[:2])
    for code, p, n in segments(default_jpg):
        if code == 0xC4:
            tc, th = default_jpg[p + 4] >> 4, default_jpg[p + 4] & 15
            bits, vals = tables[(tc, th)]
            payload = bytes([tc << 4 | th]) + bytes(bits) + bytes(vals)
            head += b"\xff\xc4" + (len(payload) + 2).to_bytes(2, "big") + payload
        else:
            head += default_jpg[p:p + n]
    return bytes(head) + hw.write_scan(coefs, frame, new_dhts, ri) + b"\xff\xd9"
