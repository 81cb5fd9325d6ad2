"""CPU: the independent PNG checker the device encoder is tested with (tests/test_gpu_png.py), proven here against files
PIL writes and against hand-built streams that use every filter type; hmrm_png_bound's formula; the PNG entry points
refuse a NULL context; the host has no CPU PNG encoder left.

The checker is pure Python + zlib + numpy: it walks the chunks and verifies every CRC with zlib.crc32, checks IHDR,
inflates the concatenated IDATs (zlib verifies the Adler-32; nothing may follow the stream) and undoes the five
filter types itself."""
import io
import math
import re
import struct
import zlib
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
SIGNATURE = b"\x89PNG\r\n\x1a\n"


def png_chunks(data: bytes):
    """[(type, body)] of a PNG file; every chunk's CRC-32 is verified."""
    assert data[:8] == SIGNATURE, "PNG signature"
    pos, out = 8, []
    while pos < len(data):
        assert pos + 12 <= len(data), "truncated chunk"
        n, typ = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        assert len(body) == n, "truncated chunk body"
        (crc,) = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(typ + body) == crc, f"CRC of the {typ!r} chunk at byte {pos}"
        out.append((typ, body))
        pos += 12 + n
    assert pos == len(data)
    return out


def _unfilter_row(ft: int, f: bytes, prev: list, bpp: int) -> list:
    cur = list(f)
    n = len(cur)
    if ft == 0:
        return cur
    if ft == 1:
        for i in range(bpp, n):
            cur[i] = (cur[i] + cur[i - bpp]) & 255
    elif ft == 2:
        cur = [(x + p) & 255 for x, p in zip(cur, prev)]
    elif ft == 3:
        for i in range(n):
            a = cur[i - bpp] if i >= bpp else 0
            cur[i] = (cur[i] + ((a + prev[i]) >> 1)) & 255
    elif ft == 4:
        for i in range(n):
            a = cur[i - bpp] if i >= bpp else 0
            b = prev[i]
            c = prev[i - bpp] if i >= bpp else 0
            p = a + b - c
            pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
            pr = a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)
            cur[i] = (cur[i] + pr) & 255
    else:
        raise AssertionError(f"filter type {ft}")
    return cur


def check_png(data: bytes, unfilter: bool = True):
    """-> (pixels [H, W, C] uint8 or None when unfilter is False, filter type of each row).  Asserts the structure:
    signature, CRCs, IHDR first (8 bit, colour type 2 or 6, no interlace), consecutive IDATs, IEND last, one complete
    zlib stream with nothing after it."""
    chunks = png_chunks(data)
    types = [t for t, _ in chunks]
    assert types[0] == b"IHDR" and types[-1] == b"IEND" and chunks[-1][1] == b""
    w, h, depth, ctype, comp, filt, inter = struct.unpack(">IIBBBBB", chunks[0][1])
    assert w >= 1 and h >= 1 and depth == 8 and ctype in (2, 6) and (comp, filt, inter) == (0, 0, 0)
    first = types.index(b"IDAT")
    last = len(types) - 1 - types[::-1].index(b"IDAT")
    assert all(t == b"IDAT" for t in types[first:last + 1]), "IDAT chunks must be consecutive"
    channels = 4 if ctype == 6 else 3
    d = zlib.decompressobj()
    raw = d.decompress(b"".join(b for t, b in chunks if t == b"IDAT")) + d.flush()
    assert d.eof and d.unused_data == b"", "one complete zlib stream"
    stride = w * channels
    assert len(raw) == h * (stride + 1)
    ftypes = [raw[y * (stride + 1)] for y in range(h)]
    assert max(ftypes) <= 4
    if not unfilter:
        return None, ftypes
    out = np.empty((h, stride), dtype=np.uint8)
    prev = [0] * stride
    for y in range(h):
        row = raw[y * (stride + 1) + 1:(y + 1) * (stride + 1)]
        prev = _unfilter_row(ftypes[y], row, prev, channels)
        out[y] = prev
    return out.reshape(h, w, channels), ftypes


# ---- a reference encoder for the checker's own tests: explicit filter type per row ----
def _filter_row(ft: int, cur: bytes, prev: bytes, bpp: int) -> bytes:
    out = bytearray(len(cur))
    for i, x in enumerate(cur):
        a = cur[i - bpp] if i >= bpp else 0
        b = prev[i]
        c = prev[i - bpp] if i >= bpp else 0
        if ft == 0:
            pr = 0
        elif ft == 1:
            pr = a
        elif ft == 2:
            pr = b
        elif ft == 3:
            pr = (a + b) >> 1
        else:
            p = a + b - c
            pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
            pr = a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)
        out[i] = (x - pr) & 255
    return bytes(out)


def _chunk(typ: bytes, body: bytes) -> bytes:
    return struct.pack(">I", len(body)) + typ + body + struct.pack(">I", zlib.crc32(typ + body))


def build_png(pixels: np.ndarray, filters, idat_pieces: int = 1) -> bytes:
    h, w, ch = pixels.shape
    stride = w * ch
    prev = bytes(stride)
    raw = bytearray()
    for y in range(h):
        cur = pixels[y].tobytes()
        ft = filters[y % len(filters)]
        raw += bytes([ft]) + _filter_row(ft, cur, prev, ch)
        prev = cur
    z = zlib.compress(bytes(raw), 6)
    cut = [len(z) * k // idat_pieces for k in range(idat_pieces + 1)]
    ihdr = struct.pack(">IIBBBBB", w, h, 8, 6 if ch == 4 else 2, 0, 0, 0)
    return (SIGNATURE + _chunk(b"IHDR", ihdr) + b"".join(_chunk(b"IDAT", z[cut[k]:cut[k + 1]]) for k in range(idat_pieces))
            + _chunk(b"IEND", b""))


def _sample(h, w, ch, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 7 + yy * 3 + k * 40) % 256 for k in range(ch)], axis=2)
    noise = rng.integers(0, 12, size=(h, w, ch))
    return ((base + noise) % 256).astype(np.uint8)


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("shape", [(1, 1), (7, 1), (1, 9), (13, 19), (40, 33)])
def test_checker_decodes_pil_files(ch, shape):
    from PIL import Image

    px = _sample(*shape, ch, seed=shape[0] * 100 + shape[1])
    buf = io.BytesIO()
    Image.fromarray(px, "RGBA" if ch == 4 else "RGB").save(buf, format="PNG")
    got, _ = check_png(buf.getvalue())
    assert np.array_equal(got, px)


@pytest.mark.parametrize("ch", [3, 4])
def test_checker_undoes_every_filter_type(ch):
    px = _sample(23, 17, ch, seed=ch)
    for filters in ([0], [1], [2], [3], [4], [0, 1, 2, 3, 4], [4, 3, 2, 1, 0, 2]):
        data = build_png(px, filters, idat_pieces=3)
        got, ftypes = check_png(data)
        assert np.array_equal(got, px), filters
        assert ftypes == [filters[y % len(filters)] for y in range(px.shape[0])]
    # and it agrees with PIL on the same hand-built file
    from PIL import Image

    assert np.array_equal(np.asarray(Image.open(io.BytesIO(build_png(px, [0, 1, 2, 3, 4])))), px)


def test_checker_rejects_damage():
    data = bytearray(build_png(_sample(8, 8, 4, seed=1), [0, 1, 2, 3, 4], idat_pieces=2))
    bad_crc = bytearray(data)
    bad_crc[40] ^= 1                             # inside IDAT data
    with pytest.raises(AssertionError):
        check_png(bytes(bad_crc))
    with pytest.raises(AssertionError):
        check_png(bytes(data[:-3]))              # truncated IEND
    with pytest.raises(AssertionError):
        check_png(b"\x89PNX" + bytes(data[4:]))  # signature


def expected_bound(w, h, ch):
    n = h * (w * ch + 1)
    return n + 17 * math.ceil(n / 4096) + 65


@pytest.mark.parametrize("w,h,ch", [(1, 1, 3), (1, 1, 4), (2, 3, 3), (9, 5, 4), (320, 180, 4), (3840, 2160, 4),
                                    (3840, 2160, 3), (8200, 8, 4), (7680, 4320, 4), (65536, 65536, 4)])
def test_png_bound_formula(hmrm, w, h, ch):
    assert hmrm.png_bound(w, h, ch) == expected_bound(w, h, ch)


@pytest.mark.parametrize("w,h,ch", [(0, 5, 4), (5, 0, 4), (-1, 5, 3), (5, 5, 2), (5, 5, 1), (65537, 2, 4), (2, 65537, 3)])
def test_png_bound_refuses_other_shapes(hmrm, w, h, ch):
    assert hmrm.png_bound(w, h, ch) == 0


def test_png_entry_points_refuse_null_context(hmrm):
    import ctypes as C

    lib = hmrm.load_library()
    f = hmrm.Frame()
    lib.hmrm_frame_defaults(C.byref(f))
    buf = (C.c_uint8 * 64)()
    size = C.c_uint64()
    assert lib.hmrm_render_png_async(None, C.byref(f), buf, 64, C.byref(size)) == 1          # HMRM_ERR_INVALID
    px = (C.c_uint8 * 12)()
    assert lib.hmrm_encode_png(None, px, 2, 2, 3, buf, 64, C.byref(size)) == 1


def test_host_has_no_cpu_png_encoder():
    """Every PNG hmap writes is encoded on the device: the zlib-on-one-thread writer is gone from the host sources."""
    host = ROOT / "heightmap-ray-marcher_b200" / "host"
    for path in sorted(host.glob("*.[ch]pp")):
        text = path.read_text()
        assert not re.search(r"\bwrite_png\b", text), path      # (stb's stbi_write_png is named in comments)
        for token in ("compress2", "compressBound", "deflateInit"):
            assert token not in text, (path, token)
