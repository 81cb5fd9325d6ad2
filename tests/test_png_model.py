"""CPU: the PNG model (tests/png_model.py), the definition the device PNG files (K3) are compared with byte for byte in
tests/test_gpu_png.py.  Nothing else writes these exact bytes, so the model is proven piece by piece: its files
decode (the checker of tests/test_png_encode.py, PIL, zlib); its filter choice equals a slow per-byte argmin; every
literal, length and producible distance code inflates to what it stands for; the coded / stored rule keeps a byte
tie coded; its files stay within hmrm_png_bound.  The content generators of the GPU edge cases live here too, with
the assertions that they produce the edge they are named for."""
import io
import zlib

import numpy as np
import pytest
from PIL import Image

import png_model as M
from test_png_encode import check_png, expected_bound, png_chunks


# ---- content ----
def gradient(h, w, ch):
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(xx + k * 30) % 256 if k % 2 == 0 else (yy * 3 + xx // 7) % 256 for k in range(ch)],
                    axis=2).astype(np.uint8)


def content(kind, h, w, ch, seed=0):
    """The content kinds of tests/test_gpu_png.py; "repeat" is noise in which every third row repeats the row above."""
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, size=(h, w, ch), dtype=np.uint8)
    if kind == "constant":
        return np.full((h, w, ch), 77, dtype=np.uint8)
    if kind == "rows":
        return np.broadcast_to(rng.integers(0, 256, size=(1, w, ch), dtype=np.uint8), (h, w, ch)).copy()
    if kind == "repeat":
        px = rng.integers(0, 256, size=(h, w, ch), dtype=np.uint8)
        px[1::3] = px[0:h - 1:3]
        return px
    return gradient(h, w, ch)


def sub_rows(residuals: np.ndarray, ch: int) -> np.ndarray:
    """Pixels [H, W, ch] whose Sub residuals are `residuals` [H, W * ch] (their running sums per channel, mod 256)."""
    h, n = residuals.shape
    return (np.cumsum(residuals.reshape(h, n // ch, ch).astype(np.int64), axis=1) % 256).astype(np.uint8)


def row_distance_pixels(w, ch, h=3, seed=0):
    """Rows whose Sub residuals are one small random walk's steps, the same in every row, while every row is the one
    above plus 50: Sub wins every row, so the filtered rows repeat exactly and the byte one row up is the best match
    (when the candidate is allowed), not distance 1 or C."""
    steps = np.random.default_rng(seed).integers(-3, 4, size=(1, w * ch)) % 256
    base = sub_rows(steps, ch).astype(np.int64)
    return ((base + 50 * np.arange(h)[:, None, None]) % 256).astype(np.uint8)


MATCH_LENGTHS = (258, 257, 11, 10, 3)


def match_length_pixels(ch, seed=0, rows=4):
    """Rows whose Sub residuals are small random bytes with runs of L + 1 equal bytes planted for each L of
    MATCH_LENGTHS and a run of 600: distance 1 matches of exactly those lengths, and 258 capping the long run."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(rows):
        parts = []
        for k, length in enumerate(MATCH_LENGTHS + (600,)):
            parts.append(rng.integers(1, 21, size=40))
            parts.append(np.full(length + 1, 30 + k))
        res = np.concatenate(parts + [rng.integers(1, 21, size=40)])
        res = np.concatenate([res, rng.integers(1, 21, size=-len(res) % ch)])
        out.append(res)
    return sub_rows(np.stack(out), ch)


def literal_edge_pixels(h, w, ch, seed=0):
    """A checkerboard of bytes 142..145 and 14..17: every predictor but None is off by about 128, so rows are stored
    with filter None and the literals sit on both sides of the 143 / 144 code boundary."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    hi = (((yy + xx) % 2) == 0)[:, :, None]
    return np.where(hi, 142, 14).astype(np.uint8) + rng.integers(0, 4, size=(h, w, ch), dtype=np.uint8)


TIE_SEED = 0


def tie_pixels(seed=TIE_SEED):
    """One RGB row of 300 pixels whose filtered stream (Sub) is 901 literals below 144 but for one match of length 3
    at distance 1: coded it takes 3 + 8 * 898 + 12 + 10 = 8 * 901 + 1 bits, one byte more than the stream, which is
    exactly the stored block's size.  The random steps (1..40) could repeat by chance and add matches; TIE_SEED is the
    first seed, searched from 0, for which none does (test_coded_stored_byte_tie_stays_coded asserts it)."""
    rng = np.random.default_rng(seed)
    res = rng.integers(1, 41, size=900)
    res[400:404] = 7
    res[399], res[404] = 8, 9
    return sub_rows(res[None, :], 3)


def slow_filter_costs(px, y):
    """The five sums of min(r, 256 - r) of row y, byte by byte."""
    h, w, ch = px.shape
    cur = [int(v) for v in px[y].reshape(-1)]
    up = [int(v) for v in px[y - 1].reshape(-1)] if y > 0 else [0] * len(cur)
    sums = [0] * 5
    for i, x in enumerate(cur):
        a = cur[i - ch] if i >= ch else 0
        b = up[i]
        c = up[i - ch] if i >= ch else 0
        p = a + b - c
        pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
        pr = a if pa <= pb and pa <= pc else b if pb <= pc else c
        for t, pred in enumerate((0, a, b, (a + b) // 2, pr)):
            r = (x - pred) % 256
            sums[t] += min(r, 256 - r)
    return sums


def slow_filter_types(px):
    types = []
    for y in range(px.shape[0]):
        s = slow_filter_costs(px, y)
        types.append(min(range(5), key=lambda t: (s[t], t)))
    return types


def filter_tie_pixels(ch):
    """Pairs of rows (above, row) of 3 pixels, bytes 0..5, searched from seed 0 until every pair of filter types has a
    row in which both share the smallest sum; stacked, each row still sits under its own row above."""
    rng = np.random.default_rng(ch)
    found = {}
    while len(found) < 10:
        pair = rng.integers(0, 6, size=(2, 3, ch), dtype=np.uint8)
        s = slow_filter_costs(pair, 1)
        best = [t for t in range(5) if s[t] == min(s)]
        for i in range(len(best)):
            for j in range(i + 1, len(best)):
                found.setdefault((best[i], best[j]), pair)
    return np.concatenate([found[k] for k in sorted(found)])


def idat_stream(data: bytes) -> bytes:
    d = zlib.decompressobj()
    out = d.decompress(b"".join(b for t, b in png_chunks(data) if t == b"IDAT")) + d.flush()
    assert d.eof and d.unused_data == b""
    return out


def inflate_raw(block: bytes) -> bytes:
    """A raw deflate stream of `block` (ending byte-aligned after a sync flush) closed by the final block 03 00."""
    d = zlib.decompressobj(-15)
    out = d.decompress(block + b"\x03\x00") + d.flush()
    assert d.eof and d.unused_data == b""
    return out


def model_segments(px):
    h, w, ch = px.shape
    stream = M.filtered_stream(px)
    return [M.deflate_segment(stream, 0, s0, min(len(stream), s0 + M.SEG), M.distances(w, ch))
            for s0 in range(0, len(stream), M.SEG)]


def matches(px):
    return [t for s in model_segments(px) for t in s.tokens if isinstance(t, tuple)]


# ---- the files decode ----
SHAPES = [(1, 1), (5, 1), (7, 2), (9, 3), (1, 5), (2, 2), (33, 17), (101, 77), (181, 243)]


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("h,w", SHAPES)
def test_model_files_decode_to_the_pixels(h, w, ch):
    for kind in ("noise", "constant", "rows", "gradient", "repeat"):
        px = content(kind, h, w, ch, seed=h * 1000 + w)
        data = M.write(px)
        got, ftypes = check_png(data)
        assert np.array_equal(got, px), kind
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(data))), px), kind
        assert idat_stream(data) == M.filtered_stream(px).tobytes(), kind
        assert ftypes == slow_filter_types(px), kind
        assert len(data) <= expected_bound(w, h, ch), kind


@pytest.mark.parametrize("make", ["match_lengths", "literal_edge", "filter_ties", "row_distance", "tie"])
@pytest.mark.parametrize("ch", [3, 4])
def test_model_files_of_the_edge_cases_decode(make, ch):
    px = {"match_lengths": lambda: match_length_pixels(ch), "literal_edge": lambda: literal_edge_pixels(9, 31, ch),
          "filter_ties": lambda: filter_tie_pixels(ch), "row_distance": lambda: row_distance_pixels(40, ch),
          "tie": lambda: tie_pixels()}[make]()
    data = M.write(px)
    assert np.array_equal(check_png(data)[0], px)
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(data))), px)
    assert idat_stream(data) == M.filtered_stream(px).tobytes()


def test_per_segment_chunks_equal_the_whole_file():
    """segment_chunk, from only the rows it needs, gives the chunks of write: at 3 and 4 channels, with and without the
    row-up candidate, across rows that repeat the one above."""
    for px in (content("repeat", 37, 300, 3, seed=1), content("repeat", 5, 8200, 4, seed=2),
               row_distance_pixels(8191, 4), row_distance_pixels(10923, 3)):
        chunks = png_chunks(M.write(px))
        idats = [t + b for t, b in chunks[1:-2]]
        assert len(idats) == M.segment_count(px)
        for k in range(len(idats)):
            assert M.segment_chunk(px, k)[4:-4] == idats[k], k


# ---- filter choice ----
@pytest.mark.parametrize("ch", [3, 4])
def test_filter_choice_equals_slow_argmin(ch):
    rng = np.random.default_rng(ch)
    small = rng.integers(0, 6, size=(40, 9, ch), dtype=np.uint8)
    images = [small, filter_tie_pixels(ch), literal_edge_pixels(6, 11, ch), match_length_pixels(ch, rows=2),
              tie_pixels(), content("constant", 4, 7, ch), content("rows", 4, 7, ch, seed=3),
              content("gradient", 30, 50, ch), content("noise", 20, 9, ch, seed=5)]
    for px in images:
        got = M.filtered_stream(px).reshape(px.shape[0], -1)[:, 0].tolist()
        assert got == slow_filter_types(px)


@pytest.mark.parametrize("ch", [3, 4])
def test_filter_tie_rows_cover_every_pair(ch):
    """Each pair of types ties for the smallest sum in some row, and the lower type is the one taken."""
    px = filter_tie_pixels(ch)
    types = M.filtered_stream(px).reshape(px.shape[0], -1)[:, 0]
    pairs = sorted({(i, j) for i in range(5) for j in range(i + 1, 5)})
    assert len(px) == 2 * len(pairs)
    for k, (i, j) in enumerate(pairs):
        s = slow_filter_costs(px, 2 * k + 1)
        assert s[i] == s[j] == min(s) and types[2 * k + 1] == min(t for t in range(5) if s[t] == min(s)), (i, j)


def test_row_zero_and_repeated_constant_rows_take_the_lower_type():
    """Row 0: Up ties None and Paeth ties Sub.  A constant row under an identical row: Up and Paeth both sum to 0, and
    Up is taken."""
    px = content("constant", 3, 20, 4)
    s = slow_filter_costs(px, 0)
    assert s[2] == s[0] and s[4] == s[1]
    s = slow_filter_costs(px, 1)
    assert s[2] == s[4] == 0
    assert M.filtered_stream(px).reshape(3, -1)[:, 0].tolist() == [1, 2, 2]


# ---- token coding ----
def test_every_literal_inflates():
    lits = list(range(256)) + list(range(255, -1, -1))
    block = M.fixed_block(lits)
    assert len(block.bits) == 3 + 2 * (144 * 8 + 112 * 9) + 7 + 3
    assert inflate_raw(block.bytes() + b"\x00\x00\xff\xff") == bytes(lits)


def test_every_match_length_inflates():
    for length in range(3, 259):
        tokens = [200, 7, (length, 1), 150, (length, 2)]
        want = bytes([200, 7] + [7] * length + [150] + ([7, 150] * length)[:length])
        assert inflate_raw(M.fixed_block(tokens).bytes() + b"\x00\x00\xff\xff") == want, length


def producible_distances():
    """Every distance K3 can use: 1, C = 3 | 4, and W * C + 1 <= 32768."""
    d = {1, 3, 4}
    for ch in (3, 4):
        d.update(w * ch + 1 for w in range(1, (M.WINDOW - 1) // ch + 1))
    return d


def test_distance_codes_at_every_producible_boundary():
    """For each distance code, the smallest and largest producible distance in its range (32767 = 3 * 10922 + 1 is the
    largest of all), coded after that many random literals and inflated."""
    prod = producible_distances()
    assert max(prod) == 32767
    rng = np.random.default_rng(1)
    checked = set()
    for code, base in enumerate(M.DIST_BASE):
        inside = [d for d in prod if base <= d < base + (1 << M.DIST_EXTRA[code])]
        for d in {min(inside), max(inside)} if inside else ():
            lits = rng.integers(0, 256, size=d).tolist()
            tokens = lits + [(3, d), (258, d)]
            want = bytes(lits)
            for length in (3, 258):
                for _ in range(length):
                    want += bytes([want[-d]])
            assert inflate_raw(M.fixed_block(tokens).bytes() + b"\x00\x00\xff\xff") == want, d
            checked.add(d)
    # every code but 1 (distance 2 alone) is reachable
    assert {1, 3, 4, 5, 32767} <= checked and {M.code_of(M.DIST_BASE, d) for d in checked} == set(range(30)) - {1}


@pytest.mark.parametrize("w,ch,used", [(8191, 4, True), (8192, 4, False), (10922, 3, True), (10923, 3, False)])
def test_row_distance_candidate_at_the_window_limit(w, ch, used):
    px = row_distance_pixels(w, ch)
    dists = {d for _, d in matches(px)}
    assert (w * ch + 1 in dists) == used
    assert M.distances(w, ch) == ([1, ch, w * ch + 1] if used else [1, ch])


@pytest.mark.parametrize("ch", [3, 4])
def test_match_length_content_hits_every_planned_length(ch):
    lengths = {n for n, d in matches(match_length_pixels(ch)) if d == 1}
    assert set(MATCH_LENGTHS) <= lengths and max(lengths) == 258


@pytest.mark.parametrize("ch", [3, 4])
def test_literal_edge_content_codes_both_sides_of_144(ch):
    px = literal_edge_pixels(9, 31, ch)
    lits = [t for s in model_segments(px) for t in s.tokens if not isinstance(t, tuple)]
    assert {142, 143, 144, 145} <= set(lits)
    assert set(M.filtered_stream(px).reshape(9, -1)[:, 0].tolist()) == {0}


# ---- coded or stored ----
def test_coded_stored_byte_tie_stays_coded():
    px = tie_pixels()
    (seg,) = model_segments(px)
    assert seg.n == 901 and [t for t in seg.tokens if isinstance(t, tuple)] == [(3, 1)]
    assert all(t < 144 for t in seg.tokens if not isinstance(t, tuple))
    assert seg.coded_bits == 8 * seg.n + 1                     # one bit over n + 1 bytes: both blocks take n + 5 bytes
    assert seg.coded and len(seg.data) == seg.n + 5
    assert inflate_raw(seg.data) == M.filtered_stream(px).tobytes()


def test_noise_segments_are_stored_and_constant_ones_coded():
    for seg in model_segments(content("noise", 20, 300, 4, seed=9)):
        assert not seg.coded and len(seg.data) == seg.n + 5
    for seg in model_segments(content("constant", 20, 300, 4)):
        assert seg.coded and len(seg.data) < 64


# ---- sizes ----
@pytest.mark.parametrize("w,h,ch", [(1, 1, 3), (1, 1, 4), (2, 3, 3), (9, 5, 4), (320, 180, 4), (1365, 3, 3),
                                    (341, 3, 4), (8200, 3, 4)])
def test_model_files_stay_within_the_bound(w, h, ch):
    for kind in ("noise", "constant", "rows", "gradient", "repeat"):
        assert len(M.write(content(kind, h, w, ch, seed=w))) <= expected_bound(w, h, ch), kind
