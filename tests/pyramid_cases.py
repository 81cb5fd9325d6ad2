"""Deterministic cases for tests/test_gpu_pyramid_fuzz.py: maps larger than 1024 cells, at every fixed-point resolution
k = fx_bits(w, h) from 20 down to 15, 8-bit RGB and 16-bit heights.

The max-mip pyramid that K1 builds (csrc/k1_prepass.cuh) is observed only through its consumer: a skip traversal that
trusts a block maximum that is too low jumps through terrain, and the frame, the per-pixel first-hit step index or the
step totals then differ from the brute kernel and from the CPU oracle.  The cases are chosen so that such an error
is visible:

* map shapes whose long side puts k at each value (SIZES), paired with short sides of 1 .. 130 cells, plus one 2-D
  map with both sides not powers of two per k <= 18 (MAP2D).  Widths 2^m + 1 have a width = 1 (mod 4) at every level
  down to 5 texels; maps of more than 2^20 cells make k1_range sample every row_stride-th row only;
* terrain: white noise (half of the cells grey), flat, ramp with steps, blocks, and for 16-bit narrow-band maps
  (samples within +-50 of a base, neighbours 1 apart, one far-off range pin: adjacent samples share a Zq16 value, so
  decisions near the surface fall to the FP64 plane);
* needle maps: a flat base, one range pin in row 0, and single-cell needles where K1 has edge cases (PLACEMENTS), each
  with a colour used nowhere else and a grazing camera outside the map that aims at it from far away, so that the
  march arrives at a high mip level;
* edge maps: a low first column and high cells beyond it, rays parallel to the x axis whose first sample after the
  entry lands less than one fixed-point unit (2^-k cells) below the edge of cell 1, and rays marching exactly along
  a cell edge: the cell-edge margin of k2_render_lin at the case's k, and its exact FP64 path.

Nothing here needs a GPU; tests/test_pyramid_cases.py checks that the cases keep reaching what they are meant to.
"""
from __future__ import annotations

import math

import numpy as np

K_VALUES = (20, 19, 18, 17, 16, 15)
SIZES = {20: (1024,), 19: (1025, 1201, 2048), 18: (2049, 3601), 17: (4097, 8192), 16: (8193, 16384),
         15: (16385, 32768)}
SHORT = (1, 2, 3, 5, 64, 130)
MAP2D = {18: (3001, 2999), 17: (5000, 4097), 16: (8193, 1503), 15: (16385, 1027)}      # (w, h)
NEEDLE_MAP = {20: (1017, 1024), 19: (1025, 1025), 18: (2049, 600), 17: (4097, 300), 16: (8193, 150),
              15: (16385, 130)}                                                        # (w, h)
KINDS8 = ("noise", "flat", "ramp", "blocks")
KINDS16 = KINDS8 + ("narrow",)
PLACEMENTS = ("last_col", "last_row", "block_seam", "region_seam", "zorder_seam", "level_last_col", "unsampled_row")
LUMS = ((0.299, 0.587, 0.114), (1.0, 0.0, 0.0), (0.2, -0.1, 0.9))
BG = (1, 2, 3)


def fx_bits(w: int, h: int) -> int:
    """Fixed-point resolution of the skip traversals: positions in units of 2^-k cells (csrc/hmrm_api.cu)."""
    clog = max(int(math.ceil(math.log2(max(w, h)))), 0)
    return min(30 - clog, 20)


def mip_shapes(w: int, h: int):
    """(w_l, h_l) of the max-mip levels: ceil halving down to one texel, at most 16 levels."""
    out = [(w, h)]
    while out[-1] != (1, 1) and len(out) < 16:
        lw, lh = out[-1]
        out.append(((lw + 1) // 2, (lh + 1) // 2))
    return out


def row_stride(w: int, h: int) -> int:
    """k1_range reads every row_stride-th row (row 0 always) to estimate the quantiser's range."""
    return max(1, -(-(w * h) // (1 << 20)))


def mip_regions(w: int, h: int) -> int:
    """CTAs (128 x 128 regions of plain level 2) of k1_mip_upper."""
    shapes = mip_shapes(w, h)
    if len(shapes) <= 3:
        return 0
    w2, h2 = shapes[2]
    return ((w2 + 127) // 128) * ((h2 + 127) // 128)


# ---- maps ------------------------------------------------------------------------------------------------------------
def _colormap(rng, h, w):
    """Random RGBA with 10 % transparent cells; red stays below 255 so that needle colours (255, g, 255) are unique."""
    cm = rng.randint(0, 256, size=(h, w, 4)).astype(np.uint8)
    np.minimum(cm[:, :, 0], 254, out=cm[:, :, 0])
    cm[rng.rand(h, w) < 0.1, 3] = 0
    return cm


def _terrain(rng, kind, w, h, depth):
    """[h, w, 3] uint8 (depth 8) or [h, w] uint16 (depth 16) samples of one terrain kind."""
    top = 255 if depth == 8 else 65535
    if kind == "noise":
        if depth == 16:
            return rng.randint(0, 65536, size=(h, w)).astype(np.uint16)
        hm = rng.randint(0, 256, size=(h, w, 3)).astype(np.uint8)
        grey = rng.rand(h, w) < 0.5
        hm[grey] = hm[grey][:, :1]          # R == G == B: K1's table path; the rest takes the arithmetic
        return hm
    if kind == "flat":
        v = np.full((h, w), int(rng.randint(0, top + 1)), dtype=np.int64)
    elif kind == "ramp":
        xx = np.arange(w, dtype=np.int64)[None, :]
        yy = np.arange(h, dtype=np.int64)[:, None]
        v = (xx * top // max(w - 1, 1) + (yy // 7) * (top // 8 + 1)) % (top + 1)
    elif kind == "blocks":
        b = int(rng.choice([3, 6, 16, 64]))
        base = rng.randint(0, top + 1, size=(h // b + 1, w // b + 1))
        v = np.repeat(np.repeat(base, b, axis=0), b, axis=1)[:h, :w]
    else:   # narrow band (16-bit): a triangle wave of amplitude 50 around a base, neighbours 1 apart, one far-off pin
        base = int(rng.randint(1000, 64000))
        t = (np.arange(w, dtype=np.int64)[None, :] + np.arange(h, dtype=np.int64)[:, None] + int(rng.randint(0, 100))) % 100
        v = base - 25 + np.minimum(t, 100 - t)
        v[0, int(rng.randint(0, w))] = 0 if base > 32768 else 65535
    if depth == 16:
        return v.astype(np.uint16)
    return np.repeat(v.astype(np.uint8)[:, :, None], 3, axis=2)


def heights_of(case, sample_value):
    """surf (height + min_height, the value the march compares against) of a grey sample value, as the reference
    computes it (main/hmap.cpp:171-191 with 65535 in place of 255 at depth 16)."""
    top = 255.0 if case["depth"] == 8 else 65535.0
    lum = case["lum"]
    s = float(sample_value)
    v = min(max((lum[0] * s + lum[1] * s) + lum[2] * s, 0.0), top)
    return (v / top) * (case["max_height"] - case["min_height"]) + case["min_height"] + case["min_height"]


# ---- cameras -----------------------------------------------------------------------------------------------------------
def _look(pos, target):
    d = np.array([target[0] - pos[0], target[1] - pos[1], target[2] - pos[2]], dtype=np.float64)
    return float(np.arctan2(d[1], d[0])), float(np.arccos(np.clip(d[2] / np.linalg.norm(d), -1.0, 1.0)))


def _random_camera(rng, w, h, gw, mn, mx):
    """The camera modes of test_gpu_fuzz.random_case: far away, hugging the box, below / beside, general; some
    axis-parallel and diagonal headings."""
    step_cells = float(rng.choice([0.05, 0.3, 1.0, 2.0, 5.0, 17.3, 400.0]))
    ext_x, ext_y = w * gw, h * gw
    scale = max(ext_x, ext_y, abs(mx), abs(mn), gw)
    mode = rng.randint(0, 4)
    if mode == 0:
        pos = (ext_x / 2 + rng.uniform(-1, 1) * 300 * scale, -ext_y / 2 + rng.uniform(-1, 1) * 300 * scale,
               rng.uniform(50, 400) * scale)
    elif mode == 1:
        pos = (rng.uniform(-0.1, 1.1) * ext_x, -rng.uniform(-0.1, 1.1) * ext_y, max(mn, mx) + rng.uniform(1e-6, 0.3) * scale)
    elif mode == 2:
        pos = (rng.uniform(-2, 3) * ext_x, -rng.uniform(-2, 3) * ext_y, rng.uniform(-2, 0.5) * scale)
    else:
        pos = (rng.uniform(-1.5, 2.5) * ext_x, -rng.uniform(-1.5, 2.5) * ext_y, max(mn, mx) + rng.uniform(0.05, 3) * scale)
    target = (rng.uniform(0.05, 0.95) * ext_x, -rng.uniform(0.05, 0.95) * ext_y, min(mn, mx) + rng.uniform(0, 1) * abs(mx - mn))
    hang, vang = _look(pos, target)
    hang += rng.uniform(-0.05, 0.05)
    vang = float(np.clip(vang + rng.uniform(-0.05, 0.05), 0.0, np.pi))
    if rng.rand() < 0.15:
        hang = float(rng.choice([0.0, np.pi / 2, -np.pi / 2, np.pi, np.pi / 4]))
    dist = math.dist(pos, target) + 1e-30
    fov = 2.0 * np.arctan2(0.7 * max(ext_x, ext_y), dist)
    return dict(projection=int(rng.randint(1, 4)), screen_width=int(rng.randint(2, 33)),
                screen_height=int(rng.randint(2, 21)), cam_pos=pos, hang=hang, vang=vang,
                hfov=float(np.clip(fov * rng.uniform(0.5, 2.0), 0.02, 3.0)),
                ortho_width=float(rng.uniform(0.3, 2.0) * max(ext_x, ext_y) / 50), grid_width=gw,
                step_dist=gw * step_cells, bg=tuple(int(v) for v in rng.randint(0, 256, size=3)))


def _strip_march(rng, w, h, gw, mn, mx):
    """A low camera beyond one end of the long axis, looking along it: rays cross thousands of cells."""
    lo, hi = min(mn, mx), max(mn, mx)
    z = lo + (hi - lo) * rng.uniform(0.3, 1.3) + 1e-3 * gw
    tz = lo + (hi - lo) * rng.uniform(0.0, 0.6)
    off = rng.uniform(2, 40) * gw
    if w >= h:
        y = -rng.uniform(0.2, 0.8) * h * gw
        pos, target = ((-off, y, z), (0.85 * w * gw, y, tz)) if rng.rand() < 0.5 else ((w * gw + off, y, z), (0.15 * w * gw, y, tz))
    else:
        x = rng.uniform(0.2, 0.8) * w * gw
        pos, target = ((x, off, z), (x, -0.85 * h * gw, tz)) if rng.rand() < 0.5 else ((x, -h * gw - off, z), (x, -0.15 * h * gw, tz))
    hang, vang = _look(pos, target)
    return dict(projection=int(rng.choice([1, 2, 3])), screen_width=int(rng.randint(8, 25)),
                screen_height=int(rng.randint(4, 13)), cam_pos=pos, hang=hang, vang=vang,
                hfov=float(rng.uniform(0.05, 0.6)), ortho_width=float(min(w, h) * gw / 16 + gw / 8), grid_width=gw,
                step_dist=gw * float(rng.choice([0.3, 0.7, 1.0, 2.0])), bg=BG)


# ---- needle maps ---------------------------------------------------------------------------------------------------------
def needle_sites(w: int, h: int, rng):
    """[(placement, x, y)] single-cell needles of a w x h map (w > 512), away from the range pin at (0, 0)."""
    stride = row_stride(w, h)
    ys = list(rng.permutation(np.arange(1, h - 1)))        # row 0 holds the pin, row h - 1 the last-row needle

    def row():          # a distinct row that k1_range samples
        while ys:
            y = int(ys.pop())
            if y % stride == 0:
                return y
        raise ValueError(f"{w}x{h}: too few rows for the needles")

    sites = [("last_col", w - 1, row()), ("last_row", int(rng.randint(w // 4, w // 2)), h - 1)]
    m = int(rng.randint(w // 16, w // 8)) * 4
    sites += [("block_seam", m - 1, row()), ("block_seam", m + 2 * 4 * 17, row())]
    region = 512 * int(rng.randint(1, max(2, w // 512)))
    sites += [("region_seam", region - 1, row()), ("region_seam", min(region + 1024, w - 2) if w > 1600 else region, row())]
    zl = max(1, min(9, int(math.log2(w // 2)) - 6))             # a z-order block of level zl is 64 * 2^zl cells wide
    zb = 64 << zl
    zx = zb * int(rng.randint(1, max(2, (w - 1) // zb)))
    sites += [("zorder_seam", zx - 1 if zx - 1 < w else w // 2, row()), ("zorder_seam", zx if zx < w else w // 2 + 1, row())]
    # the last texel column of the highest level whose width is 1 (mod 4): its first cell
    lvl = [(l, lw) for l, (lw, _) in enumerate(mip_shapes(w, h)) if l >= 1 and lw % 4 == 1 and lw >= 5]
    if lvl:
        l, lw = lvl[-1]
        sites.append(("level_last_col", min((lw - 1) << l, w - 1), row()))
    if stride > 1:      # a row that k1_range skips
        skipped = [y for y in ys if y % stride != 0]
        sites.append(("unsampled_row", int(rng.randint(w // 3, 2 * w // 3)), int(skipped[0])))
    return [(p, int(x), int(y)) for p, x, y in sites]


def _needle_case(rng, k, depth, w, h):
    base, needle, clamp = (40, 200, 255) if depth == 8 else (10000, 30000, 60000)
    gw = float(rng.choice([0.015625, 0.01, 0.2]))
    v = np.full((h, w), base, dtype=np.int64)
    v[0, 0] = needle                                             # range pin: row 0 is always sampled
    cm = _colormap(rng, h, w)
    cm[:, :, 3] = 255
    sites = needle_sites(w, h, rng)
    needles = []
    for i, (placement, x, y) in enumerate(sites):
        v[y, x] = clamp if placement == "unsampled_row" else needle
        rgba = (255, 16 + 8 * i, 255, 255)
        cm[y, x] = rgba
        needles.append(dict(placement=placement, x=x, y=y, rgba=rgba))
    hm = v.astype(np.uint16) if depth == 16 else np.repeat(v.astype(np.uint8)[:, :, None], 3, axis=2)
    case = dict(kind="needles", depth=depth, w=w, h=h, hm=hm, cm=cm, lum=LUMS[0], min_height=0.0,
                max_height=64.0 * gw, needles=needles)
    zb, zn = heights_of(case, base), heights_of(case, needle)
    frames = []
    for nd in needles:
        x, y = nd["x"], nd["y"]
        # from the side with more room; the last columns are approached from the left (moving +x)
        from_left = nd["placement"] in ("last_col", "level_last_col") or x >= w // 2
        off = float(rng.uniform(20, 200))
        d = (x + off) if from_left else (w - x + off)
        cx = -off * gw if from_left else (w + off) * gw
        cy = -(y + 0.5) * gw
        pos = (cx, cy, zb + 0.5 * (zn - zb))
        hang, vang = _look(pos, ((x + 0.5) * gw, cy, zb + 0.3 * (zn - zb)))
        frames.append(dict(projection=1, screen_width=16, screen_height=8, cam_pos=pos, hang=hang, vang=vang,
                           hfov=4.0 / d, ortho_width=gw, grid_width=gw,
                           step_dist=gw * float(rng.choice([0.37, 0.61, 0.83])) * min(1.0, d / 12000.0), bg=BG,
                           needle=nd["placement"]))
    case["frames"] = frames
    return case


# ---- edge maps -----------------------------------------------------------------------------------------------------------
def _edge_case(rng, k, depth, w, h):
    """Column 0 low, every other cell high.  Frame 1: rays along +x whose sample 1 lies 1/2 .. 1 unit (2^-k cells) below
    the edge of cell 1 while k2_render_lin's integer model rounds it onto the edge; frame 2: rays along -y exactly on the
    cell edges x = 0, 2 and 4 (power-of-two grid width), which only the exact FP64 path decides."""
    top = 255 if depth == 8 else 65535
    v = np.full((h, w), top, dtype=np.int64)
    v[:, 0] = 0
    hm = v.astype(np.uint16) if depth == 16 else np.repeat(v.astype(np.uint8)[:, :, None], 3, axis=2)
    cm = _colormap(rng, h, w)
    gw = float(rng.choice([1.0, 0.25, 0.0078125]))
    case = dict(kind="edge", depth=depth, w=w, h=h, hm=hm, cm=cm, lum=LUMS[0], min_height=0.0, max_height=8.0 * gw,
                needles=[])
    # frame 1: an orthographic camera left of the map looking along +x (dir = (1, 0, ~6e-17)): the entry point is
    # x = 0 exactly, sample 0 is at x0 = 0.01 gw (the reference's nudge), sample 1 at x0 + s.  The model puts sample 0 at
    # V0 = round(X0) units and sample 1 at V0 + round(Xs) with X = x 2^k / gw; Xs = E - V0 - 1/2 (E = 2^k: the edge of
    # cell 1) gives V1 = E while X1 = E + (X0 - V0) - 1/2 < E.
    x0 = gw * 0.01
    X0 = x0 * 2.0 ** k / gw
    V0 = math.floor(X0 + 0.5)
    step = ((1 << k) - V0 - 0.5) * gw / 2.0 ** k
    f1 = dict(projection=3, screen_width=8, screen_height=6, cam_pos=(-3.0 * gw, -(h / 2.0) * gw, 4.0 * gw), hang=0.0,
              vang=math.pi / 2, hfov=1.0, ortho_width=min(0.01 * gw, h * gw / 16), grid_width=gw, step_dist=step,
              bg=BG, needle=None)
    # frame 2: orthographic, looking along -y from above row 0; pixel columns at x = -2, 1 and 4 cells, rows at
    # z = 2 gw and 6 gw
    f2 = dict(projection=3, screen_width=3, screen_height=2, cam_pos=(1.0 * gw, 2.0 * gw, 4.0 * gw), hang=-math.pi / 2,
              vang=math.pi / 2, hfov=1.0, ortho_width=2.0 * gw, grid_width=gw, step_dist=gw * 0.5, bg=BG, needle=None)
    case["frames"] = [f1, f2]
    return case


# ---- all cases of one (k, depth, seed) -------------------------------------------------------------------------------------
def shapes(k: int, seed: int):
    """[(w, h)] of the terrain cases: each long side of SIZES[k] with one short side, wide or tall, plus MAP2D[k]."""
    out = []
    for i, n in enumerate(SIZES[k]):
        s = SHORT[(seed + 2 * i + k) % len(SHORT)]
        out.append((n, s) if (seed + i + k) % 2 == 0 else (s, n))
    if k in MAP2D:
        out.append(MAP2D[k])
    return out


def cases(fx: int, depth: int, seed: int):
    """Yields the cases of resolution k = fx at height depth 8 or 16, one at a time (each holds its own maps):
    dict(name, k, depth, seed, index, w, h, hm, cm, lum, min_height, max_height, upload ("host" | "device"),
    frames [frame kwargs + "needle": placement or None], needles, relum (lum, min, max) or None)."""
    assert fx in SIZES and depth in (8, 16)
    rng = np.random.RandomState(1_000_003 * fx + 7919 * depth + seed)
    kinds = KINDS8 if depth == 8 else KINDS16
    built = []
    for i, (w, h) in enumerate(shapes(fx, seed)):
        kind = kinds[(seed + i + fx) % len(kinds)]
        gw = float(rng.choice([0.01, 0.03125, 0.0078125, 1.0, 0.2]))
        mn, mx = [(0.0, 10.0), (0.0, 1.0), (-3.0, 2.0), (2.0, 0.5), (0.75, 2.5)][rng.randint(0, 5)]
        mx, mn = mx * max(w, h) * gw / 64, mn * max(w, h) * gw / 64
        built.append(lambda w=w, h=h, kind=kind, gw=gw, mn=mn, mx=mx: dict(
            kind=kind, depth=depth, w=w, h=h, hm=_terrain(rng, kind, w, h, depth), cm=_colormap(rng, h, w),
            lum=LUMS[rng.randint(0, 3)], min_height=mn, max_height=mx, needles=[],
            frames=[dict(_random_camera(rng, w, h, gw, mn, mx), needle=None),
                    dict(_strip_march(rng, w, h, gw, mn, mx), needle=None)]))
    built.append(lambda: _needle_case(rng, fx, depth, *NEEDLE_MAP[fx]))
    long_side = SIZES[fx][seed % len(SIZES[fx])]
    built.append(lambda: _edge_case(rng, fx, depth, long_side, 5))
    for index, make in enumerate(built):
        case = make()
        assert fx_bits(case["w"], case["h"]) == fx, (case["w"], case["h"], fx)
        case.update(name=f"k{fx}_d{depth}_s{seed}_c{index}_{case['kind']}", k=fx, seed=seed, index=index,
                    upload="device" if (index + seed) % 2 else "host")
        case["relum"] = None
        if index % 3 == 1:
            lo, hi = case["min_height"], case["max_height"]
            case["relum"] = (LUMS[(index + 1) % 3], hi, lo) if case["kind"] not in ("needles", "edge") else \
                (case["lum"], lo - 0.5 * (hi - lo), hi + 0.25 * (hi - lo))
        yield case
