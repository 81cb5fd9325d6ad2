"""TEST INFRASTRUCTURE: the 16-bit height definition (include/hmrm.h, hmrm_set_maps16) as a numpy model and as the
C statement of tests/height16_ref.c (ctypes), plus a small 16-bit PNG / PGM writer for the ingest tests.

The C library is compiled on first use into a temporary directory keyed by the source's hash, so the test tree is
never written to.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import struct
import subprocess
import tempfile
import zlib
from pathlib import Path

import numpy as np

TESTS = Path(__file__).resolve().parent
SRC = TESTS / "height16_ref.c"
SYNTH_H = TESTS.parent / "heightmap-ray-marcher_b200" / "csrc" / "synth_fbm.h"

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        key = hashlib.sha256(SRC.read_bytes() + SYNTH_H.read_bytes()).hexdigest()[:16]
        out = Path(tempfile.gettempdir()) / f"hmrm_height16_{os.getuid()}_{key}.so"
        if not out.exists():
            tmp = out.with_suffix(f".{os.getpid()}.tmp")
            subprocess.run(["gcc", "-std=gnu99", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                            "-shared", "-Wall", "-Wextra", "-o", str(tmp), str(SRC)], check=True)
            os.replace(tmp, out)
        L = C.CDLL(str(out))
        L.h16_update_heightmap.restype = None
        L.h16_update_heightmap.argtypes = [C.c_void_p, C.c_int64] + [C.c_double] * 5 + [C.c_void_p]
        L.h16_synth_maps16.restype = None
        L.h16_synth_maps16.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def heights16(x: np.ndarray, lum=(0.299, 0.587, 0.114), min_height=0.0, max_height=10.0) -> np.ndarray:
    """numpy model: v = (lum_r*x + lum_g*x) + lum_b*x clamped to [0, 65535]; (v / 65535) * span + min_height."""
    s = np.asarray(x, dtype=np.uint16).astype(np.float64)
    v = (np.float64(lum[0]) * s + np.float64(lum[1]) * s) + np.float64(lum[2]) * s
    v = np.where(v < 0.0, 0.0, np.where(v > 65535.0, 65535.0, v))
    span = np.float64(max_height) - np.float64(min_height)
    return (v / 65535.0) * span + np.float64(min_height)


def c_heights16(x: np.ndarray, lum=(0.299, 0.587, 0.114), min_height=0.0, max_height=10.0) -> np.ndarray:
    """The C statement (tests/height16_ref.c)."""
    x = np.ascontiguousarray(x, dtype=np.uint16)
    out = np.empty(x.shape, dtype=np.float64)
    lib().h16_update_heightmap(x.ctypes.data, x.size, lum[0], lum[1], lum[2], min_height, max_height,
                               out.ctypes.data)
    return out


def synth_maps16(log2n: int, seed: int = 1234, want_color=True):
    """hmrm_synth_maps16 on the CPU: (height u16 [n,n], colormap RGBA8 [n,n,4] or None)."""
    n = 1 << log2n
    hm = np.empty((n, n), dtype=np.uint16)
    cm = np.empty((n, n, 4), dtype=np.uint8) if want_color else None
    lib().h16_synth_maps16(log2n, seed, hm.ctypes.data, cm.ctypes.data if want_color else None)
    return hm, cm


# ---- 16-bit image writers ------------------------------------------------------------------------------------------
def _chunk(tag: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def _filter_rows(raw: np.ndarray, bpp: int, filters) -> bytes:
    """raw: [rows][stride] uint8; row y gets filter filters[y % len(filters)] (0 none .. 4 Paeth)."""
    out = bytearray()
    prev = np.zeros(raw.shape[1], dtype=np.int32)
    for y in range(raw.shape[0]):
        cur = raw[y].astype(np.int32)
        left = np.concatenate([np.zeros(bpp, np.int32), cur[:-bpp]])
        upleft = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]])
        ft = filters[y % len(filters)]
        if ft == 0:
            res = cur
        elif ft == 1:
            res = cur - left
        elif ft == 2:
            res = cur - prev
        elif ft == 3:
            res = cur - (left + prev) // 2
        else:
            res = cur - _paeth(left, prev, upleft)
        out.append(ft)
        out += (res & 255).astype(np.uint8).tobytes()
        prev = cur
    return bytes(out)


ADAM7 = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]


def write_png16(path, samples: np.ndarray, filters=(0, 1, 2, 3, 4), interlace=False, trns=None) -> None:
    """16-bit PNG of samples [H,W] (grey, colour type 0) or [H,W,C] with C = 2 (grey+alpha), 3 (RGB), 4 (RGBA).
    trns: a colour key (one 16-bit value per channel, grey or RGB only) written as a tRNS chunk."""
    a = np.asarray(samples, dtype=np.uint16)
    if a.ndim == 2:
        a = a[:, :, None]
    h, w, ch = a.shape
    color = {1: 0, 2: 4, 3: 2, 4: 6}[ch]
    bpp = 2 * ch

    def encode(img):
        raw = img.astype(">u2").view(np.uint8).reshape(img.shape[0], img.shape[1] * bpp)
        return _filter_rows(raw, bpp, filters)

    if interlace:
        data = b""
        for xo, yo, xs, ys in ADAM7:
            sub = a[yo::ys, xo::xs]
            if sub.shape[0] and sub.shape[1]:
                data += encode(sub)
    else:
        data = encode(a)
    ihdr = struct.pack(">IIBBBBB", w, h, 16, color, 0, 0, 1 if interlace else 0)
    extra = _chunk(b"tRNS", b"".join(struct.pack(">H", v) for v in trns)) if trns is not None else b""
    Path(path).write_bytes(b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", ihdr) + extra + _chunk(b"IDAT", zlib.compress(data, 6)) +
                           _chunk(b"IEND", b""))


def write_pgm16(path, samples: np.ndarray, maxval=65535) -> None:
    """Binary PNM of 16-bit samples: [H,W] as P5 (PGM), [H,W,3] as P6 (PPM)."""
    a = np.asarray(samples, dtype=np.uint16)
    h, w = a.shape[:2]
    magic = b"P6" if a.ndim == 3 else b"P5"
    Path(path).write_bytes(magic + b"\n%d %d\n%d\n" % (w, h, maxval) + a.astype(">u2").tobytes())
