"""Seeded search for the cases of tests/golden/lin_margin_cases.json: small orthographic frames whose first pixel's ray
reaches one of k2_render_lin's decision margins at a sample n where the model error V_n - X(P_n) exceeds one unit in the
direction that a one-unit-smaller margin would misjudge, with a map built around that sample so that the decision at n
decides the frame (tests/lin_model.py restates the arithmetic).

    python tools/lin_margin_search.py [--check]      (--check: compare with the committed file instead of writing it)

Bands and the mutant each case must break:
  cell_x / cell_y    cell test margin 1        V_n = edge + 1 while the reference is still in the cell before the edge
  grid_high          certainly-outside 1       V_n = grid + 1 while the reference is still in the last cell
  grid_low           low-edge margin 0         V_n = -2^k - 1 while the reference is still above -1 cell (cell 0)
  inside_high        inside margin 0           V_n = grid - 1 while the reference is already outside
  z_above            ZMARGIN 8 in `above`      Z_n = 16 q + 9 at the first sample below a plateau's surf
  z_hit              ZMARGIN 8 in the hit test Z_n = 16 q - 9 while the sample is still on or above the surf
  fp64_x             the look's rel / 100      P_n just past a cell edge, the look's estimate fma(n, s, P_0) before it
  fp64_z             the look without bz       z_n just on or above surf, the estimate below it

The FP64 cases keep x (or z) inside one binade for the whole window, so the reference's adds all round the same way
and P_n - fma(n, s, P_0) grows linearly with n; the camera coordinate is then moved ulp-exactly (every P_j moves by the
same amount inside a binade) to put the sample between the estimate and the edge.  The production look refuses there
and advance_exact decides; the model checks that no earlier sample of the window needed advance_exact, so the look at
n is taken from the anchor a = 0.

The lateral cases use rays nearly parallel to the edge: the model crosses it over hundreds of samples, and the first
sample that a smaller margin misjudges is where the search looks.  Why sample n of a cell case is always examined at
level 0 by k2_render_lin: the wall's cells are tall (surf above the ray) and V_n lies in a wall cell or next to one, so
at every level the 3x3-dilated block maximum around V_n includes the wall and `above` fails; the descent ends at level
0.  No jump passes over n: a jump of m samples keeps V_{j..j+m} at least 5 units inside a cleared neighbourhood (room -
margin - 1), and a neighbourhood that contained V_n would contain the wall and not be cleared.  The same holds for
z_above / z_hit (n is below the block maximum of the plateau at every level, and a z-limited jump ends >= 11 sixteenths
above it) and for the grid cases whose rays sit high above flat terrain: there the inside mutant's sample is decided at
a level > 0, where no cell test can send it on.
"""
from __future__ import annotations

import argparse
import json
import math
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))

import lin_model as L  # noqa: E402
import oracle_lib as O  # noqa: E402

OUT = ROOT / "tests" / "golden" / "lin_margin_cases.json"
SEED = 14
GW = 0.01
WINDOWS = {1: (20000, 64000), 2: (65536 + 20000, 65536 + 64000)}


def hx(v: float) -> str:
    return float(v).hex()


def frame_kw(cam, hang, vang, step):
    return dict(projection=3, screen_width=2, screen_height=2, cam_pos=cam, hang=hang, vang=vang, hfov=0.5,
                ortho_width=2.0 ** -30, grid_width=GW, step_dist=step, bg=(4, 5, 6))


def first(mask):
    idx = np.flatnonzero(mask)
    return int(idx[0]) if len(idx) else None


def slope_err(s: float, scale: float) -> float:
    """(D - 2^16 X(s)): the model's per-step error in 2^-16 units; its sign is the sign of the error it accumulates."""
    D = L.slope(s * scale)
    return float(D - Fraction(s) * Fraction(scale) * 65536) if D is not None else 0.0


def tune(fk, ci, scale, off, base, sign_err, w, h, mn, mx):
    """Shift camera coordinate ci by less than one model unit so that V_0 at the window's base sample rounds by about
    0.45 units in the direction sign_err (the first of the three error terms that add up to more than one unit)."""
    for _ in range(3):
        hit, e, d = L.ray_of(fk, w, h, mn, mx)
        if not hit:
            return False
        p0, s = L.ray_start(e, d, fk["grid_width"], fk["step_dist"])
        pb = float(L.samples(p0[ci], s[ci], base + 1)[base])
        x = Fraction(pb) * Fraction(scale) + off
        err = float(L.rne(x) - x)
        if abs(err - 0.45 * sign_err) < 0.04:
            return True
        # want frac(X) = 0.55 (rounds up by 0.45) or 0.45 (rounds down by 0.45)
        frac = float(x - math.floor(x))
        delta = (0.55 if sign_err > 0 else 0.45) - frac
        cam = list(fk["cam_pos"])
        cam[ci] = cam[ci] + delta / scale
        fk["cam_pos"] = tuple(cam)
    return False


def lateral_trial(rng, k, w, h, band, axis, sign, window, z):
    """One random near-parallel ray.  `axis`: the model axis whose edge is crossed; `sign`: its direction of motion in
    model units (+1: x grows / y falls).  Returns a case or None."""
    n_lo, n_hi = WINDOWS[window]
    nmax = n_hi + 2000
    n_t = int(rng.randint(n_lo + 2000, n_hi - 2000))
    if band == "grid_low":
        # from inside the box (x or -y >= 0) to -1 cell within the window
        rate = (1 << k) / n_t * float(rng.uniform(1.02, 1.3))
    else:
        rate = float(rng.uniform(0.03, 0.7))                    # model units per sample across the edge
    unit = GW / (1 << k)
    ext = (h if axis == "x" else w) * GW                        # extent along the travel axis
    step = ext * float(rng.uniform(0.5, 0.8)) / nmax
    rho = rate * unit / step                                    # lateral / travel direction ratio
    n_edge = w if axis == "x" else h
    if band == "cell":
        c = int(rng.randint(n_edge // 4, 3 * n_edge // 4))
        edge = c * GW
    elif band in ("grid_high", "inside_high"):
        edge = n_edge * GW
    else:
        edge = -GW                                             # the low edge: -1 cell
    # world direction of the lateral drift: x grows with +x; the model's y runs along -y
    drift = sign if axis == "x" else -sign
    if axis == "x":
        travel = 1 if rng.randint(2) else -1                    # along +y or -y
        hang = travel * math.pi / 2 - travel * drift * rho
        y_cam = -h * GW - 1e-3 if travel > 0 else 1e-3
        lat0 = edge - drift * rate * unit * (n_t + 1e-3 / step)
        cam = (lat0, y_cam, z)
    else:
        travel = 1
        hang = drift * rho
        lat0 = -edge + (-drift) * rate * unit * (n_t + 1e-3 / step)   # world y: model y = -y
        cam = (-1e-3, lat0, z)
    fk = frame_kw(cam, hang, math.pi / 2, step)
    ai = 0 if axis == "x" else 1
    sc = L.fx_scale(k, GW) * (1 if axis == "x" else -1)
    sign_err = -1 if band in ("grid_low", "inside_high") else 1
    hit_, _, d = L.ray_of(fk, w, h, 0.0, 1.0)
    if not hit_ or slope_err(fk["step_dist"] * d[ai], sc) * sign_err < 0.3:
        return None
    if not tune(fk, ai, sc, Fraction(0), (n_t // L.PERIOD) * L.PERIOD, sign_err, w, h, 0.0, 1.0):
        return None
    r = L.march(fk, w, h, 0.0, 1.0, nmax)
    if r is None:
        return None
    P, s = r
    ax = L.axes(P, s, k, GW, 1.0, L.MAGIC)[ai]
    if ax.D is None or (ax.D > 0) != (sign > 0):
        return None
    V = ax.V()
    cells = L.truth_cell(P[ai], GW, axis)
    other = L.truth_cell(P[1 - ai], GW, "y" if axis == "x" else "x")
    n_other = h if axis == "x" else w
    grid = n_edge << k
    mask = (1 << k) - 1
    if band == "cell":
        f = V & mask
        dec = np.where((f >= 1) & (f <= mask - 1), V >> k, cells)
        n = first(dec != cells)
        mut = "cell_margin_1"
    elif band == "grid_high":
        n = first((V >= grid + 1) & (cells < n_edge))
        mut = "outside_margin_1"
    elif band == "grid_low":
        n = first((V < -(1 << k)) & (cells >= 0))
        mut = "low_edge_margin_0"
    else:
        n = first((V >= 0) & (V < grid) & (cells >= n_edge))
        mut = "inside_margin_0"
    if n is None or not n_lo <= n < n_hi:
        return None
    if not np.all((cells[:n] >= 0) & (cells[:n] < n_edge)):
        return None
    vn = int(V[n])
    # the model and the truth at n, every margin
    rec = dict(band=band if band != "cell" else f"cell_{axis}", mutant=mut, axis=axis, motion=("+" if sign > 0 else "-") + axis,
               k=k, n=n, window=window, v=vn, truth_cell=int(cells[n]))
    m = dict(w=w, h=h, low=0, high=255, wall_axis=None, cells=[])
    if band == "cell":
        T = int(cells[n])
        lo_hi = (T + 1, n_edge) if sign > 0 else (0, T + 1)
        m.update(wall_axis=axis, wall_lo=lo_hi[0], wall_hi=lo_hi[1])
        later = np.flatnonzero((cells >= lo_hi[0]) & (cells < lo_hi[1]))
        rec["expect_first_hit"] = int(later[0]) if len(later) else None
    else:
        # one tall cell for the quantiser's range, in the corner farthest from every cell the ray visits
        out_ = (cells < 0) | (cells >= n_edge)
        seen = first(out_)
        seen = nmax if seen is None else seen
        xs = cells[:seen] if axis == "x" else other[:seen]
        ys = other[:seen] if axis == "x" else cells[:seen]
        corners = [(0, 0), (w - 1, 0), (0, h - 1), (w - 1, h - 1)]
        dist = [int(np.min(np.maximum(np.abs(xs - cx), np.abs(ys - cy)))) for cx, cy in corners]
        cx, cy = corners[int(np.argmax(dist))]
        if max(dist) < 3:
            return None
        m["cells"] = [[cx, cy, 255]]
        rec["expect_steps"] = seen
    # the ray stays inside the other axis' range for every sample the oracle examines
    end = rec.get("expect_first_hit", rec.get("expect_steps"))
    if end is None or end >= nmax - 1 or not np.all((other[:end + 1] >= 0) & (other[:end + 1] < n_other)):
        return None
    fk["cam_pos"] = tuple(float(v) for v in fk["cam_pos"])
    return rec, m, fk


def z_trial(rng, kind, window, h0):
    """A slowly descending ray along +x over a plateau.  kind 'above': Z_t = 16 q + 9 at the first sample below the
    plateau's surf; 'hit': Z_n = 16 q - 9 at a sample still on or above it."""
    w, h, k = 256, 64, 20
    n_lo, n_hi = WINDOWS[window]
    nmax = n_hi + 2000
    vp = 128
    mn, mx = h0, h0 + 1.0
    hm = np.array([[[0, 0, 0], [255, 255, 255], [vp, vp, vp]]], dtype=np.uint8)
    ht = O.update_heightmap(hm, L.LUM, mn, mx)[0]
    surf = [float(v) + mn for v in ht]
    zs, zo = L.quantiser(min(surf), max(surf))
    sp = surf[2]
    q = L.zq16(sp, zs, zo)
    frac = L.zr16(sp, zs, zo) - 16 * q
    if kind == "above" and not 7.9 < frac < 7.995:
        return None
    if kind == "hit" and not -7.995 < frac < -7.9:
        return None
    n_t = int(rng.randint(n_lo + 2000, n_hi - 2000))
    step = 150 * GW / nmax
    rate = float(rng.uniform(0.03, 0.5)) / (16 * zs)           # height per sample
    eps = rate / step
    row = int(rng.randint(20, 44))
    cam = (-1e-3, -(row + float(rng.uniform(0.2, 0.8))) * GW, sp + rate * (n_t + 1e-3 / step))
    fk = frame_kw(cam, 0.0, math.pi / 2 + eps, step)
    sign_err = 1 if kind == "above" else -1
    zs16, off = zs * 16.0, 16 * (Fraction(zo) - Fraction(L.MAGIC))
    hit_, _, d = L.ray_of(fk, w, h, mn, mx)
    if not hit_ or slope_err(fk["step_dist"] * d[2], zs16) * sign_err < 0.3:
        return None
    if not tune(fk, 2, zs16, off, (n_t // L.PERIOD) * L.PERIOD, sign_err, w, h, mn, mx):
        return None
    r = L.march(fk, w, h, mn, mx, nmax)
    if r is None:
        return None
    P, s = r
    axs = L.axes(P, s, k, GW, zs, zo)
    if axs[2].D is None or axs[2].D >= 0:
        return None
    Vz = axs[2].V()
    below = P[2] < sp
    t = first(below)
    if t is None:
        return None
    if kind == "above":
        n, want = t, (q << 4) + 9
    else:
        n = first((Vz <= (q << 4) - 9) & ~below)
        want = (q << 4) - 9
    if n is None or not n_lo <= n < n_hi or int(Vz[n]) != want:
        return None
    # sample n is decided in x and y by the model (no cell edge within the margin), so the z predicate alone decides it
    for i in (0, 1):
        if L.cell_decides(axs[i].at(n), k, L.MARGIN) is None:
            return None
    m = dict(w=w, h=h, low=vp, high=vp, wall_axis=None, cells=[[0, 0, 0], [w - 1, h - 1, 255]])
    rec = dict(band=f"z_{kind}", mutant=f"zmargin_{kind}_8", axis="z", motion="-z", k=k, n=n, window=window,
               v=int(Vz[n]), q=q, expect_first_hit=t)
    fk["cam_pos"] = tuple(float(v) for v in fk["cam_pos"])
    return rec, m, fk, (mn, mx)


def fp64_check(P, s, n, gw, w, h, zs, zo, surf, mutant):
    """True if the look refuses sample n, decides it wrong with the mutant's constant, and decides every earlier
    undecided sample of the window (so no advance_exact moved the anchor before n)."""
    sof = lambda gx, gy: float(surf[gy, gx])
    p0 = [float(p[0]) for p in P]
    t = L.truth(P, n, gw, w, h, sof)
    if L.look(n, 0, p0, s, gw, w, h, sof) is not None:
        return False
    kw = dict(rel_c=L.REL / 100) if mutant == "look_rel_100" else dict(use_bz=False)
    got = L.look(n, 0, p0, s, gw, w, h, sof, **kw)
    if got is None or got == t:
        return False
    return all(L.look(int(j), 0, p0, s, gw, w, h, sof) is not None for j in L.undecided(P, s, 20, gw, w, h, zs, zo, surf, n))


def edge_double(c, gw):
    """The smallest double x with fl(x / gw) >= c."""
    x = c * gw
    while x / gw >= c:
        x = math.nextafter(x, -math.inf)
    while x / gw < c:
        x = math.nextafter(x, math.inf)
    return x


def place(fk, ci, target_of, w, h, mn, mx, n):
    """Move camera coordinate ci until sample n of axis ci lands where target_of(P_n) says (exact within a binade)."""
    for _ in range(6):
        r = L.march(fk, w, h, mn, mx, n + 2)
        if r is None:
            return None
        P, s = r
        lo, hi = target_of(P, s)
        pn = float(P[ci][n])
        if lo <= pn <= hi:
            return P, s
        cam = list(fk["cam_pos"])
        cam[ci] += (lo + hi) / 2 - pn
        fk["cam_pos"] = tuple(cam)
    return None


def tune_step(fk, ci, ulp, lo, hi, rng, w, h, mn, mx):
    """Nudge step_dist (by ~1e-9 relative) until fl(step d) / ulp has a fractional part in (lo, hi): the rounding
    every add of the reference makes inside the binade of ulp."""
    hit, _, d = L.ray_of(fk, w, h, mn, mx)
    if not hit:
        return False
    base = fk["step_dist"]
    for _ in range(200):
        st = base * (1.0 + float(rng.uniform(-1e-9, 1e-9)))
        sv = abs(st * d[ci]) / ulp
        if lo < sv - math.floor(sv) < hi:
            fk["step_dist"] = st
            return True
    return False


def fp64_x_trial(rng):
    """Along +x (and slowly +y) inside the binade [1, 2) of x; tall cells from the edge on."""
    w, h, k = 256, 64, 20
    n = int(rng.randint(20000, 40000))
    x0 = float(rng.uniform(1.30, 1.35))
    sx = (float(rng.uniform(1.6, 1.9)) - x0) / n
    th = math.atan(0.2 / (n * sx))
    fk = frame_kw((x0 - 1e-3 / math.tan(th), -h * GW - 1e-3, 0.5), th, math.pi / 2, sx / math.cos(th))
    # rounding up by 0.35 .. 0.45 ulp per add: P_n runs ahead of fma(n, s, P_0)
    if not tune_step(fk, 0, 2.0 ** -52, 0.55, 0.65, rng, w, h, 0.0, 1.0):
        return None
    r = L.march(fk, w, h, 0.0, 1.0, n + 2)
    if r is None:
        return None
    c = int(float(r[0][0][n]) / GW) + 1
    ex = edge_double(c, GW)

    def target(P, s):
        d = float(P[0][n]) - L.fma(float(n), s[0], float(P[0][0]))
        return ex + d / 8, ex + d / 3

    r = place(fk, 0, target, w, h, 0.0, 1.0, n)
    if r is None:
        return None
    P, s = r
    if not (1.0 <= P[0][0] and P[0][n + 1] < 2.0) or int(P[0][n - 1] / GW) != c - 1 or int(P[0][n] / GW) != c:
        return None
    m = dict(w=w, h=h, low=0, high=255, wall_axis="x", wall_lo=c, wall_hi=w, cells=[])
    hm, _ = L.case_maps(m)
    surf = O.update_heightmap(hm, L.LUM, 0.0, 1.0) + 0.0
    zs, zo = L.quantiser(float(surf.min()), float(surf.max()))
    if not fp64_check(P, s, n, GW, w, h, zs, zo, surf, "look_rel_100"):
        return None
    fk["cam_pos"] = tuple(float(v) for v in fk["cam_pos"])
    rec = dict(band="fp64_x", mutant="look_rel_100", axis="x", motion="+x", k=k, n=n, window=1, truth_cell=c,
               expect_first_hit=n)
    return rec, m, fk, (0.0, 1.0)


def fp64_z_trial(rng):
    """Along +x, descending ~1e-9 per sample inside the binade [0.5, 1) of z, over a plateau at surf ~0.65."""
    w, h, k = 256, 64, 20
    mn, mx = 0.2, 0.7
    n = int(rng.randint(20000, 40000))
    m = dict(w=w, h=h, low=128, high=128, wall_axis=None, cells=[[0, 0, 0], [w - 1, h - 1, 255]])
    hm, _ = L.case_maps(m)
    surf = O.update_heightmap(hm, L.LUM, mn, mx) + mn
    sp = float(surf[h // 2, w // 2])
    step = 5e-5
    eps = float(rng.uniform(1.5e-5, 2.5e-5))
    fk = frame_kw((-1e-3, -(h // 2 + float(rng.uniform(0.3, 0.7))) * GW, sp + eps * step * n + eps * 1e-3), 0.0,
                  math.pi / 2 + eps, step)
    # |s| rounded down by 0.35 .. 0.45 ulp per add: z_n stays above fma(n, s, z_0)
    if not tune_step(fk, 2, 2.0 ** -53, 0.35, 0.45, rng, w, h, mn, mx):
        return None

    def target(P, s):
        d = float(P[2][n]) - L.fma(float(n), s[2], float(P[2][0]))
        return sp + d / 8, sp + d / 3

    r = place(fk, 2, target, w, h, mn, mx, n)
    if r is None:
        return None
    P, s = r
    if not (P[2][n + 1] >= 0.5 and P[2][0] < 1.0 and P[2][n] >= sp > P[2][n + 1] and P[2][n - 1] > P[2][n]):
        return None
    zs, zo = L.quantiser(float(surf.min()), float(surf.max()))
    if not fp64_check(P, s, n, GW, w, h, zs, zo, surf, "look_no_bz"):
        return None
    fk["cam_pos"] = tuple(float(v) for v in fk["cam_pos"])
    rec = dict(band="fp64_z", mutant="look_no_bz", axis="z", motion="-z", k=k, n=n, window=1, expect_first_hit=n + 1)
    return rec, m, fk, (mn, mx)


PLAN = (
    # (band, k, axis, sign, window)
    ("cell", 20, "x", +1, 1), ("cell", 20, "x", -1, 2), ("cell", 20, "y", +1, 2), ("cell", 20, "y", -1, 1),
    ("cell", 15, "x", +1, 2), ("cell", 15, "x", -1, 1), ("cell", 15, "y", +1, 1), ("cell", 15, "y", -1, 2),
    ("grid_high", 20, "x", +1, 1), ("grid_high", 15, "y", +1, 2),
    ("grid_low", 15, "x", -1, 2), ("grid_low", 15, "y", -1, 1),
    ("inside_high", 20, "x", +1, 2), ("inside_high", 20, "y", +1, 1),
)
MAPS = {20: (256, 256), 15: (32768, 16)}


def search():
    rng = np.random.RandomState(SEED)
    out = []
    for band, k, axis, sign, window in PLAN:
        w, h = MAPS[k]
        for _ in range(20000):
            r = lateral_trial(rng, k, w, h, band, axis, sign, window, 0.5 if band == "cell" else 0.9)
            if r is not None:
                break
        else:
            raise RuntimeError(f"no case for {band} k {k} {axis} {sign} window {window}")
        rec, m, fk = r
        out.append(dict(rec, name=f"{rec['band']}_k{k}_{rec['motion']}_w{window}", map=m, min_height=hx(0.0),
                        max_height=hx(1.0), frame=enc_frame(fk)))
    for kind, window in (("above", 1), ("above", 2), ("hit", 1), ("hit", 2)):
        for _ in range(200000):
            r = z_trial(rng, kind, window, float(rng.uniform(0.05, 0.4)))
            if r is not None:
                break
        else:
            raise RuntimeError(f"no z case {kind} window {window}")
        rec, m, fk, (mn, mx) = r
        out.append(dict(rec, name=f"{rec['band']}_k20_w{window}", map=m, min_height=hx(mn), max_height=hx(mx),
                        frame=enc_frame(fk)))
    for trial in (fp64_x_trial, fp64_z_trial):
        for _ in range(2000):
            r = trial(rng)
            if r is not None:
                break
        else:
            raise RuntimeError(f"no case from {trial.__name__}")
        rec, m, fk, (mn, mx) = r
        out.append(dict(rec, name=f"{rec['band']}_k20_w1", map=m, min_height=hx(mn), max_height=hx(mx),
                        frame=enc_frame(fk)))
    return out


def enc_frame(fk):
    return dict(fk, cam_pos=[hx(v) for v in fk["cam_pos"]], hang=hx(fk["hang"]), vang=hx(fk["vang"]),
                hfov=hx(fk["hfov"]), ortho_width=hx(fk["ortho_width"]), grid_width=hx(fk["grid_width"]),
                step_dist=hx(fk["step_dist"]), bg=list(fk["bg"]))


def dumps(cases) -> str:
    return json.dumps({"seed": SEED, "cases": cases}, indent=1, sort_keys=True) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    a = ap.parse_args()
    text = dumps(search())
    if a.check:
        sys.exit(0 if OUT.read_text() == text else 1)
    OUT.write_text(text)
    print(f"wrote {OUT}")


if __name__ == "__main__":
    main()
