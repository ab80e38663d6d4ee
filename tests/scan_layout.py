"""TEST INFRASTRUCTURE: re-emit a baseline scan with a chosen byte layout, and a numpy reference destuffer.

Encoders write the entropy-coded segment as compactly as they can, so their files reach only a few of the byte layouts
the destuff kernel (K1) distinguishes.  ``split`` cuts a valid file into the destuffed payload of each restart
interval; ``emit`` writes it back with a COM segment of chosen length (the scan's start phase), padding after any
interval (explicit bytes, or filler up to a chosen offset from ``scan_start & ~15``), RSTn numbering, dropped or
duplicated markers, a chosen terminator with data behind it, and truncation.  It returns the destuffed bytes, the
interval starts and the terminator position the construction implies.  ``reference`` derives the same from the raw
bytes alone (vectorised numpy, the model's byte rule); ``place`` tells where special pairs fall in K1's tiles.
Plain Python + numpy.
"""
from dataclasses import dataclass, field

import numpy as np

TILE, CHUNK = 4096, 16  # K1: 4 KiB tiles of 256 threads x 16 bytes, starting at scan_start & ~15


def scan_start(jpg):
    """Offset of the first byte behind the SOS segment."""
    p = 2
    while True:
        assert jpg[p] == 0xFF, p
        code, n = jpg[p + 1], int.from_bytes(jpg[p + 2:p + 4], "big")
        p += 2 + n
        if code == 0xDA:
            return p


def restart_interval(jpg):
    p = 2
    while True:
        code, n = jpg[p + 1], int.from_bytes(jpg[p + 2:p + 4], "big")
        if code == 0xDD:
            return int.from_bytes(jpg[p + 4:p + 6], "big")
        if code == 0xDA:
            return 0
        p += 2 + n


def split(jpg):
    """(header up to the end of SOS, [destuffed payload of each interval], raw bytes from the terminator on).  RSTn ends
    an interval when the file has a DRI segment; any other FF xx (xx != 00) ends the scan."""
    start = scan_start(jpg)
    restart = restart_interval(jpg) > 0
    parts, cur, i = [], bytearray(), start
    while True:
        c = jpg[i]
        if c != 0xFF:
            cur.append(c)
            i += 1
            continue
        n = jpg[i + 1]
        if n == 0:
            cur.append(0xFF)
            i += 2
        elif restart and 0xD0 <= n <= 0xD7:
            parts.append(bytes(cur))
            cur = bytearray()
            i += 2
        else:
            parts.append(bytes(cur))
            return jpg[:start], parts, jpg[i:]


def stuff(b):
    return bytes(b).replace(b"\xff", b"\xff\x00")


@dataclass
class Layout:
    jpg: bytes
    scan_start: int
    restart: bool            # RSTn splits intervals (the file has a DRI segment)
    destuffed: bytes         # what the construction puts into the entropy-coded segment (up to the terminator)
    starts: list             # destuffed offset of every interval
    term: object             # file offset of the terminator's FF, None when the file ends before it
    status: int              # what the construction implies under the restart extension
    nseg_expected: int
    notes: dict = field(default_factory=dict)


def filler(rng, n):
    """n bytes that are never FF."""
    return (rng.integers(0, 255, n, dtype=np.uint8)).tobytes()


def emit(src, com=None, pads=None, rst="cyclic", drop=(), dup=(), term=b"\xff\xd9", after=b"", trunc=None, seed=0,
         nseg_expected=None):
    """Re-emit `src` (a valid file).  com: payload length of a COM segment placed behind SOI (None: no segment).
    pads: {interval: [piece, ...]} written behind the interval's payload; a piece is bytes (written with FF stuffed)
    or an int o (non-FF filler up to offset o from scan_start & ~15, which is then where the next byte lands) or a pair
    (r, m) (filler up to the next offset that is r modulo m).
    rst: 'cyclic' (D0..D7), 'const' (always D5), 'random' or a list of marker numbers.  drop: markers (index k = the
    one behind interval k) left out; dup: markers written twice, -1 = one right at the scan start, the last index =
    one right before the terminator.  term: the terminating marker; after: raw bytes behind it; trunc: cut the file
    to this many bytes (negative: from the end)."""
    header, parts, _ = split(src)
    restart = restart_interval(src) > 0
    pads = pads or {}
    rng = np.random.default_rng(seed)
    out = bytearray(header[:2])
    if com is not None:
        out += b"\xff\xfe" + (com + 2).to_bytes(2, "big") + bytes((7 * i + 1) % 255 for i in range(com))
    out += header[2:]
    start = len(out)
    base0 = start & ~15
    dest = bytearray()
    starts = [0]
    nmark = [0]

    def marker():
        m = nmark[0]
        nmark[0] += 1
        n = {"cyclic": m % 8, "const": 5, "random": int(rng.integers(0, 8))}[rst] if isinstance(rst, str) else rst[m]
        out.extend((0xFF, 0xD0 + n))
        starts.append(len(dest))

    if -1 in dup:
        marker()
    for k, p in enumerate(parts):
        out += stuff(p)
        dest += p
        for piece in pads.get(k, ()):
            if isinstance(piece, (int, tuple)):
                at = len(out) - base0
                n = piece - at if isinstance(piece, int) else (piece[0] - at) % piece[1]
                assert n >= 0, (k, piece, at)
                f = filler(rng, n)
            else:
                f = bytes(piece)
            out += stuff(f)
            dest += f
        last = k + 1 == len(parts)
        if not last and k not in drop:
            marker()
        if k in dup:
            marker()
    term_pos = len(out)
    out += term + after
    if trunc is not None:
        out = out[:trunc]
    jpg = bytes(out)
    if term_pos + 1 >= len(jpg):
        term_pos = None
    nseg = len(starts)
    if nseg_expected is None:
        nseg_expected = len(parts) if restart else 1
    lens = [b - a for a, b in zip(starts, starts[1:] + [len(dest)])]
    if term_pos is None:
        status = -20
    elif restart and nseg != nseg_expected:
        status = -21
    elif restart and 0 in lens:
        status = -9  # an interval without a byte still has MCUs to decode
    else:
        assert not drop and not dup, "dropped and duplicated markers that keep the count decode other intervals' data"
        status = 0
    return Layout(jpg, start, restart, bytes(dest), starts, term_pos, status, nseg_expected)


@dataclass
class Reference:
    destuffed: bytes
    starts: list
    term: object      # file offset of the terminator's FF, or None
    stuffed: np.ndarray  # file offsets of the FF of every FF 00 pair before the terminator
    rst: np.ndarray      # file offsets of the FF of every restart marker before the terminator
    keep: np.ndarray     # per byte of [start, end): the byte yields an output byte (bool)


def reference(jpg, start, restart):
    """The model's destuffing (extract_entropy_coded_bits, + RSTn splitting with restart=True) over jpg[start:], in
    uint8 / bool arrays: a byte's fate depends on itself and the raw byte in front of it, except that the byte at
    `start` sees no predecessor.  FF 00 yields FF; FF then RSTn (restart only) starts an interval; FF then anything
    else ends the scan.  An FF is never kept on its own."""
    b = np.frombuffer(jpg, np.uint8)[start:]
    pff = np.zeros(b.size, bool)
    pff[1:] = b[:-1] == 0xFF
    zero = b == 0
    rst = ((b & 0xF8) == 0xD0) if restart else np.zeros(b.size, bool)
    term = np.flatnonzero(pff & ~zero & ~rst)
    end = int(term[0]) if term.size else b.size
    keep = (pff & zero) | (~pff & (b != 0xFF))
    keep[end:] = False
    mark = np.flatnonzero(pff[:end] & rst[:end])
    stuffed = np.flatnonzero(pff[:end] & zero[:end])
    vals = b[:end][keep[:end]].copy()
    vals[pff[:end][keep[:end]]] = 0xFF
    if mark.size:
        kept_before = np.cumsum(keep[:end], dtype=np.uint32)[mark]
        starts = [0] + kept_before.astype(np.int64).tolist()
    else:
        starts = [0]
    return Reference(vals.tobytes(), starts, start + end - 1 if term.size else None, start + stuffed - 1, start + mark - 1, keep)


def place(pos, start):
    """(tile, thread in tile, word in thread, byte in word) of file offsets `pos` in K1's tiling of a scan that
    starts at `start`."""
    rel = np.asarray(pos, np.int64) - (start & ~15)
    return rel // TILE, (rel % TILE) // CHUNK, (rel % CHUNK) // 4, rel % 4


def dropped_words(ref, start):
    """Per 4-byte word of the scan (aligned to scan_start & ~15) up to the terminator: a bit mask of its bytes that yield
    no output byte (the FF of a stuffed pair, both bytes of a marker).  Bytes in front of `start` count as kept."""
    base0 = start & ~15
    n = ref.keep.size if ref.term is None else ref.term - start
    k = np.ones((start - base0) + n + 3 & ~3, bool)
    k[start - base0:start - base0 + n] = ref.keep[:n]
    d = (~k).reshape(-1, 4)
    return d[:, 0] * 1 + d[:, 1] * 2 + d[:, 2] * 4 + d[:, 3] * 8
