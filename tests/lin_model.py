"""A plain restatement of k2_render_lin's per-sample arithmetic (csrc/k2_render_lin.cuh, DESIGN.md §4 "K2 lin", fact 4)
next to the reference's own per-sample expressions (main/hmap.cpp:998-1037, oracle/hmap_oracle.c render_core).

Only what is a pure function of the sample index is restated, not the traversal: the reference's samples P_n, the
integer model V_n of x, y and z, the height quantiser, the decision predicates with their margins as parameters, and
the FP64 "linear look" with its constants as parameters.  numpy for whole rays, `fractions` where a value must be exact
(the magic-number roundings, the fma of the look).

Why the margins are what they are.  Let X(P) = P 2^k / gw (x), -P 2^k / gw (y) and 16 Zr(P) = 16 (P zq_scale + zc) (z)
be the reference's sample in model units.  The header of k2_render_lin.cuh argues |V_n - X(P_n)| < 1.6 within a
65536-sample window (test_lin_model.py measures at most 1.47 over 10^8 pairs).  V is an integer, so a predicate
`V >= E + m` (or `V < E - m`) about a break point E that the reference compares against is right for every V that
satisfies it iff m + (the distance from the predicate's first V to E) > 1.6:

| predicate (kernel)                                   | first V it decides | wrong if           | smallest m | first wrong m |
|------------------------------------------------------|--------------------|--------------------|------------|---------------|
| cell test fx < m .. fx > mask - m (line 272)         | E + m (low side)   | m < 1.6            | 2          | 1             |
|                                                      | E - 1 - m (high)   | m + 1 < 1.6        | 1          | 0             |
| certainly outside, high: V >= grid + m (line 250)    | grid + m           | m < 1.6            | 2          | 1             |
| certainly outside, low: V < -2^k - m (line 250)      | -2^k - m - 1       | m + 1 < 1.6        | 1          | 0             |
| inside: m <= V < grid - m (line 245, lin_span_*)     | grid - m - 1 (high)| m + 1 < 1.6        | 1          | 0             |
|                                                      | m (low: still in the (-1, 0) strip, cell 0)  | never |  0  |   -           |
| above: V > 16 q + m (line 213)                       | 16 q + m + 1       | m + 1 - 1.6 < 8    | 9          | 8             |
| hit: V < 16 q - m (line 316)                         | 16 q - m - 1       | m + 1 - 1.6 < 8    | 9          | 8             |

(z: q = round(Zr(surf)) puts 16 Zr(surf) anywhere in [16 q - 8, 16 q + 8], so the break point E is 16 q +- 8.)  The
cell test's high side and the inside test's low side are never the binding ones.  Production uses 4 and 10.

The FP64 look (lines 334-371) estimates P_n as fma(n - a, s, P_a) from the exact anchor a.  The reference's n - a adds
round by at most 2^-53 |P| each and the fma once more, so |P_n - xe| <= (n - a + 1) 2^-53 max|P|; the kernel's bound
rel = (n - a + 2) 2.3e-16 is twice that plus 2.3e-16, which also covers the two divides by gw (2^-53 |q| each): the
`axq * 4.5e-16` term is a second cover of the same roundings, and no input makes the look decide wrong without it.
rel itself and the `ze +- bz` band are tight in the other sense: a path inside one binade drifts by the same rounding
at every add, so |P_n - xe| grows like n, and a sample placed between xe and a cell edge (or surf) is decided wrong by a
look with rel / 100 (or comparing ze without bz).
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

MAGIC = 6755399441055744.0          # 1.5 * 2^52 (k1_prepass.cuh)
PERIOD = 65536                      # HMRM_LIN_PERIOD: samples between exact re-anchors
FRAC = 16                           # HMRM_LIN_FRAC
MARGIN = 4                          # HMRM_LIN_MARGIN
ZMARGIN = 10                        # HMRM_LIN_ZMARGIN


# ---- frame constants (hmrm_api.cu frame_params / skip_params / hmrm_update_heightmap) -------------------------------
def fx_bits(w: int, h: int) -> int:
    dim, clog = max(w, h), 0
    while (1 << clog) < dim:
        clog += 1
    return min(30 - clog, 20)


def fx_scale(k: int, gw: float) -> float:
    return float(1 << k) / gw


def quantiser(min_surf: float, max_surf: float) -> tuple[float, float]:
    """(zq_scale, zq_offset) of a map whose surf values range over [min_surf, max_surf] (maps of at most 2^20 cells:
    every row is sampled, so these are the exact extremes)."""
    rng = max_surf - min_surf
    scale = 61000.0 / rng if (rng > 0.0 and math.isfinite(rng) and math.isfinite(61000.0 / rng)) else 1.0
    return scale, MAGIC + (2000.0 - min_surf * scale)


def rne(x: Fraction) -> int:
    return round(x)                 # Fraction.__round__: half to even


def zq16(surf: float, zq_scale: float, zq_offset: float) -> int:
    """The pyramid's level-0 value of a cell: clamp(round(surf * zq_scale + zq_offset) - MAGIC, 0, 65535)."""
    v = rne(Fraction(surf) * Fraction(zq_scale) + Fraction(zq_offset)) - int(MAGIC)
    return min(max(v, 0), 65535)


def zr16(z: float, zq_scale: float, zq_offset: float) -> Fraction:
    """16 Zr(z), exact: the height in the model's sixteenths of a Zq unit."""
    return 16 * (Fraction(z) * Fraction(zq_scale) + Fraction(zq_offset) - Fraction(MAGIC))


# ---- the reference's samples ---------------------------------------------------------------------------------------
def ray_start(e, d, gw: float, step_dist: float):
    """(P_0, s) per axis: P_0 = fl(e + fl(nudge d)), nudge = fl(gw 0.01) (main/hmap.cpp:998), s = fl(step d) (:1037)."""
    nudge = gw * 0.01
    return tuple(e[i] + nudge * d[i] for i in range(3)), tuple(step_dist * d[i] for i in range(3))


def ray_of(fk: dict, w: int, h: int, mn: float, mx: float):
    """(entered, e, d) of pixel (0, 0) of an orthographic frame `fk` over a w x h map: the ray and the box entry point
    from the oracle (pinned bit for bit to the reference and to the device)."""
    import oracle_lib as O

    of = O.make_frame(projection=3, width=fk["screen_width"], height=fk["screen_height"], pos=fk["cam_pos"],
                      hang=fk["hang"], vang=fk["vang"], ortho_width=fk["ortho_width"], grid_width=fk["grid_width"],
                      step_dist=fk["step_dist"], min_height=mn, max_height=mx)
    pos, d = O.get_ray(of, 0.0, 0.0)
    hit, e = O.intersection(pos, d, (0.0, 0.0, mn), (w * fk["grid_width"], -h * fk["grid_width"], mx))
    return hit, e, d


def march(fk: dict, w: int, h: int, mn: float, mx: float, nmax: int):
    """(P per axis, s per axis): the first nmax samples of pixel (0, 0), or None if its ray misses the box."""
    hit, e, d = ray_of(fk, w, h, mn, mx)
    if not hit:
        return None
    p0, s = ray_start(e, d, fk["grid_width"], fk["step_dist"])
    return [samples(p0[i], s[i], nmax) for i in range(3)], s


def samples(p0: float, s: float, n: int) -> np.ndarray:
    """P_0 .. P_{n-1} of one axis: sequential IEEE adds, as the reference's `x += sx`."""
    a = np.full(n, s, dtype=np.float64)
    a[0] = p0
    return np.add.accumulate(a)


def truth_cell(P, gw: float, axis: str):
    """The reference's cell index per sample: (int)(x / gw), (int)(-y / gw), truncation toward zero."""
    q = (P if axis == "x" else -P) / gw
    with np.errstate(invalid="ignore"):
        return np.trunc(q).astype(np.int64)


# ---- the integer model ---------------------------------------------------------------------------------------------
def slope(s_units: float) -> int | None:
    """D = rint(s_units 2^16) (lin_slope); None when the axis does not fit the model (|motion| >= 2^26 units, NaN)."""
    if not abs(s_units) < 67108864.0:
        return None
    return rne(Fraction(s_units * 65536.0))


class Axis:
    """One axis of the model: V_n = V_0(base) + ((n - base) D + 2^15) >> 16, base = 65536 floor(n / 65536), and V_0(base)
    = round(P_base * scale + off) exactly (magic_decode(fma(P, scale, MAGIC + off))).  The re-anchors are at the
    reference's own P_base, so V_n does not depend on the path the kernel took."""

    def __init__(self, P: np.ndarray, s: float, scale: float, off: Fraction = Fraction(0)):
        self.P, self.scale, self.off = P, scale, off
        self.D = slope(s * scale)

    def v0(self, base: int) -> int:
        return rne(Fraction(float(self.P[base])) * Fraction(self.scale) + self.off)

    def V(self, n0: int = 0, n1: int | None = None) -> np.ndarray:
        n1 = len(self.P) if n1 is None else n1
        out = np.empty(n1 - n0, dtype=np.int64)
        for base in range(n0 - n0 % PERIOD, n1, PERIOD):
            lo, hi = max(base, n0), min(base + PERIOD, n1)
            j = np.arange(lo - base, hi - base, dtype=np.int64)
            out[lo - n0:hi - n0] = self.v0(base) + ((j * self.D + (1 << (FRAC - 1))) >> FRAC)
        return out

    def at(self, n: int) -> int:
        base = n - n % PERIOD
        return self.v0(base) + (((n - base) * self.D + (1 << (FRAC - 1))) >> FRAC)


def axes(P3, s3, k: int, gw: float, zq_scale: float, zq_offset: float):
    """(x, y, z) Axis objects: x in units of 2^-k cells, y the same along -y, z in sixteenths of a Zq unit."""
    sc = fx_scale(k, gw)
    zc = Fraction(zq_offset) - Fraction(MAGIC)
    zs16 = zq_scale * 16.0
    return (Axis(P3[0], s3[0], sc), Axis(P3[1], s3[1], -sc), Axis(P3[2], s3[2], zs16, 16 * zc))


# ---- decision predicates: the kernel's, with the margin as a parameter, and the reference's truth ---------------------
def cell_decides(v: int, k: int, margin: int) -> int | None:
    """Level-0 cell test (line 272): the cell V >> k, or None when V is within the margin of a cell edge (sent on)."""
    mask = (1 << k) - 1
    f = v & mask
    if f < margin or f > mask - margin:
        return None
    return v >> k


def inside(v: int, grid: int, margin: int) -> bool:
    """Inside test (line 245 with lin_span = grid - 2 margin): certainly inside the grid along this axis."""
    return margin <= v < grid - margin


def outside_high(v: int, grid: int, margin: int) -> bool:
    return v >= grid + margin


def outside_low(v: int, k: int, margin: int) -> bool:
    """The low edge is at -1 cell: (int) truncates toward zero, so (-1, 0) cells still are cell 0."""
    return v < -(1 << k) - margin


def truth_inside(cell: int, n_cells: int) -> bool:
    return 0 <= cell < n_cells


def above(vz: int, q: int, zmargin: int) -> bool:
    """`above q` (line 213): certainly z > surf of every cell whose Zq16 is at most q."""
    return vz > (q << 4) + zmargin and q < 65535


def hit(vz: int, q: int, zmargin: int) -> bool:
    """Hit test (line 316): certainly z < surf of a cell whose Zq16 is q."""
    return vz < (q << 4) - zmargin and q > 0


# ---- the FP64 linear look (lines 328-372) ---------------------------------------------------------------------------
REL = 2.3e-16                       # per-add bound of the estimate
QREL = 4.5e-16                      # quotient term


def fma(a: float, b: float, c: float) -> float:
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def look(n: int, a: int, pa, s, gw: float, map_w: int, map_h: int, surf_of, rel_c: float = REL, qrel: float = QREL,
         use_bz: bool = True):
    """The look at sample n from the exact anchor a (positions pa, steps s per axis), in the kernel's FP64 operations:
    "hit", "miss" (the reference's bounds test), "above" (certainly not below the surface), or None: refused, the
    sample goes to advance_exact.  surf_of(gx, gy) is the cell's surf.  rel_c, qrel and use_bz are the constants."""
    mj = float(n - a)
    rel = (mj + 2.0) * rel_c
    xe, ye, ze = (fma(mj, s[i], pa[i]) for i in range(3))
    bx, by = rel * max(abs(pa[0]), abs(xe)), rel * max(abs(pa[1]), abs(ye))
    bz = rel * max(abs(pa[2]), abs(ze))
    qx, qy = xe / gw, -ye / gw
    inv_gw_up = (1.0 / gw) * 1.000001
    axq, ayq = abs(qx), abs(qy)
    ex_, ey_ = bx * inv_gw_up + axq * qrel, by * inv_gw_up + ayq * qrel
    fxq, fyq = axq - math.floor(axq), ayq - math.floor(ayq)
    near_x = 1.0 - axq if axq < 1.0 else min(fxq, 1.0 - fxq)
    near_y = 1.0 - ayq if ayq < 1.0 else min(fyq, 1.0 - fyq)
    if not (axq < 2.0e9 and ayq < 2.0e9 and near_x > ex_ and near_y > ey_):
        return None
    gx, gy = math.trunc(qx), math.trunc(qy)
    if gx < 0 or gy < 0 or gx >= map_w or gy >= map_h:
        return "miss"
    surf = surf_of(gx, gy)
    if (ze + bz if use_bz else ze) < surf:
        return "hit"
    if ze - bz > surf:
        return "above"
    return None


def truth(P3, n: int, gw: float, map_w: int, map_h: int, surf_of):
    """The reference's verdict on sample n: "hit", "miss" or "above" (main/hmap.cpp:1001-1016)."""
    gx, gy = int(truth_cell(P3[0][n:n + 1], gw, "x")[0]), int(truth_cell(P3[1][n:n + 1], gw, "y")[0])
    if gx < 0 or gy < 0 or gx >= map_w or gy >= map_h:
        return "miss"
    return "hit" if P3[2][n] < surf_of(gx, gy) else "above"

def undecided(P, s, k, gw, w, h, zs, zo, surf, n):
    """Samples 0 .. n-1 that the integer model cannot decide with the production margins (a superset of those
    k2_render_lin sends to the look: cell, grid and height edges, as if every sample were examined at level 0)."""
    axs = axes([p[:n] for p in P], s, k, gw, zs, zo)
    vx, vy, vz = (a.V() for a in axs)
    mask = (1 << k) - 1
    near = lambda v: ((v & mask) < MARGIN) | ((v & mask) > mask - MARGIN)
    ins = lambda v, g: (v >= MARGIN) & (v < g - MARGIN)
    flag = near(vx) | near(vy) | ~ins(vx, w << k) | ~ins(vy, h << k)
    qmap = np.vectorize(lambda v: zq16(float(v), zs, zo))(surf)
    cx, cy = np.clip(vx >> k, 0, w - 1), np.clip(vy >> k, 0, h - 1)
    q = qmap[cy, cx].astype(np.int64)
    dec_z = ((vz > 16 * q + ZMARGIN) & (q < 65535)) | ((vz < 16 * q - ZMARGIN) & (q > 0))
    return np.flatnonzero(flag | ~dec_z)


# ---- the maps of the committed cases -------------------------------------------------------------------------------
LUM = (0.299, 0.587, 0.114)


def case_maps(m: dict):
    """(height RGB8 [h, w, 3], colour RGBA8 [h, w, 4]) of a case's map description: `low` everywhere, `high` on the cells
    whose x (or y, `wall_axis`) index is in [wall_lo, wall_hi), and the single cells of `cells` ([x, y, value])."""
    w, h = m["w"], m["h"]
    v = np.full((h, w), m["low"], dtype=np.uint8)
    if m.get("wall_axis") is not None:
        sl = slice(m["wall_lo"], m["wall_hi"])
        if m["wall_axis"] == "x":
            v[:, sl] = m["high"]
        else:
            v[sl, :] = m["high"]
    for x, y, val in m.get("cells", []):
        v[y, x] = val
    hm = np.dstack([v, v, v])
    yy, xx = np.mgrid[0:h, 0:w]
    cm = np.dstack([(xx * 37 + yy * 11) % 251, (xx * 5 + yy * 53) % 241, (xx * 101 + yy * 7) % 239,
                    np.full((h, w), 255)]).astype(np.uint8)
    return hm, cm
