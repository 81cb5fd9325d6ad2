"""Plain restatement of the PNG files K3 writes (hmrm_render_png_async, hmrm_encode_png): the definition in
include/hmrm.h, in numpy and Python integers, byte for byte.  Nothing here is shared with the device or host code.

  filter     per row, the type (0 None, 1 Sub, 2 Up, 3 Average, 4 Paeth) with the smallest sum of min(r, 256 - r) over
             the row, r = residual & 255; the lowest type wins a tie.  The row above row 0 is zero, a and c are zero
             for i < C.
  stream     H rows of 1 + W*C bytes (type byte, residuals), cut into segments of SEG bytes; the last may be shorter.
  parse      greedy, per segment: at position o each candidate distance (1, C, then W*C + 1 while that is <= 32768)
             has a run, the number of bytes from o on that equal the byte that many positions back (never before byte
             0 of the stream, never past the segment's end), capped at 258.  The longest run of at least 3 is a match,
             the earlier distance winning a tie; otherwise one literal.
  coding     RFC 1951 fixed Huffman: header BFINAL 0 BTYPE 01, the tokens, EOB, an empty stored block (00 00 FF FF
             after byte alignment).  With `bits` the tokens' bits the segment stays coded when 3 + bits + 10 <= 8 (n + 1)
             (the tie included); otherwise it is one stored block 00 LEN NLEN bytes.
  framing    signature, IHDR, one IDAT per segment (the first starts with the zlib header 78 01), an IDAT holding 03 00
             and the Adler-32 of the stream, IEND."""
import struct
import zlib
from collections import namedtuple

import numpy as np

SEG = 4096
MAX_MATCH = 258
WINDOW = 32768
SIGNATURE = b"\x89PNG\r\n\x1a\n"

# RFC 1951 3.2.5: length codes 257..285 and distance codes 0..29, each with its base and number of extra bits
LENGTH_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
               227, 258]
LENGTH_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]

Segment = namedtuple("Segment", "data coded coded_bits n tokens")


# ---- filter ----
def paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(px: np.ndarray, y0: int, y1: int) -> np.ndarray:
    """Filtered bytes of rows y0 .. y1 - 1 ([y1 - y0, 1 + W*C] uint8: type byte, then the residuals)."""
    h, w, ch = px.shape
    rb = w * ch
    rows = px.reshape(h, rb).astype(np.int32)
    out = np.empty((y1 - y0, rb + 1), dtype=np.uint8)
    step = max(1, (1 << 20) // rb)
    for b0 in range(y0, y1, step):
        b1 = min(y1, b0 + step)
        x = rows[b0:b1]
        up = np.zeros_like(x)
        if b0 > 0:
            up[:] = rows[b0 - 1:b1 - 1]
        else:
            up[1:] = rows[b0:b1 - 1]
        a = np.zeros_like(x)
        a[:, ch:] = x[:, :-ch]
        c = np.zeros_like(x)
        c[:, ch:] = up[:, :-ch]
        res = np.stack([x, x - a, x - up, x - ((a + up) >> 1), x - paeth(a, up, c)]) & 255
        cost = np.minimum(res, 256 - res).sum(axis=2, dtype=np.int64)
        ft = np.argmin(cost, axis=0)                     # the first minimum: the lowest type wins a tie
        out[b0 - y0:b1 - y0, 0] = ft
        out[b0 - y0:b1 - y0, 1:] = res[ft, np.arange(b1 - b0)]
    return out


def filtered_stream(px: np.ndarray) -> np.ndarray:
    return filter_rows(px, 0, px.shape[0]).reshape(-1)


def distances(width: int, channels: int) -> list:
    d = [1, channels]
    if width * channels + 1 <= WINDOW:
        d.append(width * channels + 1)
    return d


# ---- parse ----
def run_lengths(eq: np.ndarray) -> np.ndarray:
    """run[i] = how many consecutive entries of eq from i on are True."""
    n = len(eq)
    pos = np.arange(n)
    first_false = np.minimum.accumulate(np.where(eq, n, pos)[::-1])[::-1]
    return first_false - pos


def parse(stream: np.ndarray, base: int, s0: int, s1: int, dists) -> list:
    """Greedy tokens of the segment [s0, s1) of the filtered stream; stream[i] is byte base + i of it.  A literal is an
    int, a match a (length, distance) tuple."""
    seg = stream[s0 - base:s1 - base]
    runs = []
    for d in dists:
        eq = np.zeros(s1 - s0, dtype=bool)
        k = max(s0, d)                                   # never before byte 0 of the stream
        if k < s1:
            assert k - d >= base, "the stream must reach back one candidate distance"
            eq[k - s0:] = stream[k - base:s1 - base] == stream[k - d - base:s1 - d - base]
        runs.append(np.minimum(run_lengths(eq), MAX_MATCH).tolist())
    lits = seg.tolist()
    tokens, o = [], 0
    while o < s1 - s0:
        best, best_d = 0, 0
        for d, r in zip(dists, runs):
            if r[o] > best:
                best, best_d = r[o], d
        if best >= 3:
            tokens.append((best, best_d))
            o += best
        else:
            tokens.append(lits[o])
            o += 1
    return tokens


# ---- coding ----
class Bits:
    def __init__(self):
        self.bits = []

    def put(self, value: int, n: int):             # extra bits and headers: least significant bit first
        self.bits.extend((value >> i) & 1 for i in range(n))

    def huff(self, code: int, n: int):             # Huffman codes: most significant bit first
        self.bits.extend((code >> (n - 1 - i)) & 1 for i in range(n))

    def bytes(self) -> bytes:
        return np.packbits(np.array(self.bits, dtype=np.uint8), bitorder="little").tobytes()


def code_of(base: list, value: int) -> int:
    return max(i for i, b in enumerate(base) if b <= value)


def put_symbol(out: Bits, sym: int):
    if sym < 144:
        out.huff(0x30 + sym, 8)
    elif sym < 256:
        out.huff(0x190 + sym - 144, 9)
    elif sym < 280:
        out.huff(sym - 256, 7)
    else:
        out.huff(0xC0 + sym - 280, 8)


def put_tokens(out: Bits, tokens):
    for t in tokens:
        if isinstance(t, tuple):
            length, dist = t
            i = code_of(LENGTH_BASE, length)
            put_symbol(out, 257 + i)
            out.put(length - LENGTH_BASE[i], LENGTH_EXTRA[i])
            j = code_of(DIST_BASE, dist)
            out.huff(j, 5)
            out.put(dist - DIST_BASE[j], DIST_EXTRA[j])
        else:
            put_symbol(out, t)


def fixed_block(tokens) -> Bits:
    """BFINAL 0, BTYPE 01, the tokens, EOB, then BFINAL 0 BTYPE 00 of the empty stored block (not yet aligned)."""
    out = Bits()
    out.put(0, 1)
    out.put(1, 2)
    put_tokens(out, tokens)
    put_symbol(out, 256)
    out.put(0, 3)
    return out


def deflate_segment(stream: np.ndarray, base: int, s0: int, s1: int, dists) -> Segment:
    """The deflate data of one segment: a fixed-Huffman block closed by an empty stored block, or one stored block."""
    n = s1 - s0
    tokens = parse(stream, base, s0, s1, dists)
    block = fixed_block(tokens)
    coded_bits = len(block.bits)                    # 3 + the tokens' bits + 10
    if coded_bits <= 8 * (n + 1):
        return Segment(block.bytes() + b"\x00\x00\xff\xff", True, coded_bits, n, tokens)
    raw = stream[s0 - base:s1 - base].tobytes()
    return Segment(bytes([0, n & 255, n >> 8, ~n & 255, (~n >> 8) & 255]) + raw, False, coded_bits, n, tokens)


# ---- framing ----
def chunk(typ: bytes, body: bytes) -> bytes:
    return struct.pack(">I", len(body)) + typ + body + struct.pack(">I", zlib.crc32(typ + body))


def head(width: int, height: int, channels: int) -> bytes:
    return SIGNATURE + chunk(b"IHDR", struct.pack(">IIBBBBB", width, height, 8, 6 if channels == 4 else 2, 0, 0, 0))


def tail(adler: int) -> bytes:
    return chunk(b"IDAT", b"\x03\x00" + struct.pack(">I", adler)) + chunk(b"IEND", b"")


def idat_chunk(stream: np.ndarray, base: int, k: int, total: int, width: int, channels: int) -> bytes:
    s0 = k * SEG
    seg = deflate_segment(stream, base, s0, min(total, s0 + SEG), distances(width, channels))
    return chunk(b"IDAT", (b"\x78\x01" if k == 0 else b"") + seg.data)


def segment_count(px: np.ndarray) -> int:
    h, w, ch = px.shape
    return -(-h * (w * ch + 1) // SEG)


def segment_chunk(px: np.ndarray, k: int) -> bytes:
    """Segment k's IDAT chunk, from only the rows its bytes and their candidate distances reach."""
    h, w, ch = px.shape
    rowlen = w * ch + 1
    total = h * rowlen
    s0, s1 = k * SEG, min(total, (k + 1) * SEG)
    y0 = max(0, s0 - max(distances(w, ch))) // rowlen
    y1 = (s1 - 1) // rowlen + 1
    part = filter_rows(px, y0, y1).reshape(-1)
    return idat_chunk(part, y0 * rowlen, k, total, w, ch)


def write(px: np.ndarray) -> bytes:
    """The whole PNG file of [H, W, 3 | 4] uint8 pixels."""
    h, w, ch = px.shape
    stream = filtered_stream(px)
    body = b"".join(idat_chunk(stream, 0, k, len(stream), w, ch) for k in range(segment_count(px)))
    return head(w, h, ch) + body + tail(zlib.adler32(stream.tobytes()))
