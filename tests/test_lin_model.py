"""CPU: k2_render_lin's integer ray model (tests/lin_model.py) against the reference's samples.

The error bound |V_n - X(P_n)| < 1.6 units that every margin of the march rests on is measured over 10^8 (ray, sample)
pairs, and each committed case of tests/golden/lin_margin_cases.json is checked to be where it claims to be: the
production margin decides its sample correctly or sends it on, the named one-unit-smaller margin decides it wrong, the
smallest correct margin decides it correctly or sends it on, and the oracle's frame depends on that decision.  The FP64
look's cases are checked the same way against its restatement: the production look refuses, the mutant's decides
wrong."""
import json
import math
import subprocess
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

import lin_model as L

ROOT = Path(__file__).resolve().parent.parent
CASES = json.loads((ROOT / "tests" / "golden" / "lin_margin_cases.json").read_text())["cases"]


def window_errors(rng, rays, k, axis):
    """max |V - X| over `rays` random rays of one 65536-sample window each, and the number of pairs."""
    n = L.PERIOD
    j = np.arange(n, dtype=np.int64)
    worst, pairs = 0.0, 0
    for _ in range(rays):
        if axis == "z":
            rng_z = float(rng.uniform(0.01, 100.0))
            zq_scale = 61000.0 / rng_z
            scale, off = zq_scale * 16.0, 16 * int(rng.randint(-40000, 40000))
            p0 = float(rng.uniform(-rng_z, rng_z)) * 2.0 ** float(rng.uniform(-30, 0))
            s = float(rng.choice([-1, 1])) * 2.0 ** float(rng.uniform(-12, 7)) / zq_scale
        else:
            gw = 2.0 ** float(rng.uniform(-10, 0)) * float(rng.uniform(1.0, 2.0))
            scale, off = L.fx_scale(k, gw) * (1 if axis == "x" else -1), 0
            cells = 1 << (30 - k)
            # start anywhere in the grid down to a few cells from 0, move towards 0: binades are crossed
            p0 = cells * gw * 2.0 ** float(rng.uniform(-(30 - k) - 3, 0))
            s = -gw * 2.0 ** float(rng.uniform(math.log2(1 / 4000), math.log2(100)))
            if axis == "y":
                p0, s = -p0, -s
        D = L.slope(s * scale)
        if D is None:               # more than 2^26 units per step: the kernel's per-step loop, not the model
            continue
        P = L.samples(p0, s, n)
        v0 = L.rne(Fraction(p0) * Fraction(scale) + off)
        V = v0 + ((j * D + (1 << 15)) >> 16)
        X = P * scale + off if axis == "z" else (P * float(1 << k)) / gw * (1 if axis == "x" else -1)
        ok = np.abs(X) < 2.0 ** 31
        e = np.abs(V[ok] - X[ok])
        if len(e):
            worst = max(worst, float(e.max()))
            pairs += int(ok.sum())
    return worst, pairs


def test_model_error_bound_measured():
    """10^8 pairs at k = 20 .. 15 (x, y) and in z: every error < 1.6 units, and the largest > 1 (the margin cases exist)."""
    rng = np.random.RandomState(2024)
    worst, pairs = {}, 0
    for axis in ("x", "y", "z"):
        for k in range(15, 21) if axis != "z" else (None,):
            w, p = window_errors(rng, 200 if axis != "z" else 400, k, axis)
            worst[axis] = max(worst.get(axis, 0.0), w)
            pairs += p
    assert pairs >= 10 ** 8, pairs
    for axis, w in worst.items():
        assert 1.0 < w < 1.6, (axis, w, worst)


def case_ray(c):
    f = c["frame"]
    fk = dict(f, cam_pos=[float.fromhex(v) for v in f["cam_pos"]],
              **{key: float.fromhex(f[key]) for key in ("hang", "vang", "hfov", "ortho_width", "grid_width", "step_dist")})
    mn, mx = float.fromhex(c["min_height"]), float.fromhex(c["max_height"])
    return fk, mn, mx


def case_model(c):
    """(axes of the model, samples, quantiser, surf of the case's cells) of a case's pixel (0, 0)."""
    fk, mn, mx = case_ray(c)
    m = c["map"]
    hm, _ = L.case_maps(m)
    import oracle_lib as O

    surf = O.update_heightmap(hm, L.LUM, mn, mx) + mn
    zs, zo = L.quantiser(float(surf.min()), float(surf.max()))
    P, s = L.march(fk, m["w"], m["h"], mn, mx, c["n"] + 1)
    return L.axes(P, s, c["k"], fk["grid_width"], zs, zo), P, (zs, zo), surf, fk, mn, mx


def check_look_case(c, P, fk, surf, zs, zo):
    """The FP64 look at sample n from the anchor a = 0: production refuses (advance_exact decides), the mutant's constant
    decides it against the reference, and every earlier sample the model leaves undecided is decided by the look, so
    no advance_exact moved the anchor before n."""
    n, gw, w, h = c["n"], fk["grid_width"], c["map"]["w"], c["map"]["h"]
    _, s = L.march(fk, w, h, float.fromhex(c["min_height"]), float.fromhex(c["max_height"]), 1)
    sof = lambda gx, gy: float(surf[gy, gx])
    p0 = [float(p[0]) for p in P]
    truth = L.truth(P, n, gw, w, h, sof)
    assert truth == ("hit" if c["band"] == "fp64_x" else "above"), c["name"]
    assert L.look(n, 0, p0, s, gw, w, h, sof) is None, f"{c['name']}: the production look decides sample {n}"
    mutant = dict(rel_c=L.REL / 100) if c["mutant"] == "look_rel_100" else dict(use_bz=False)
    got = L.look(n, 0, p0, s, gw, w, h, sof, **mutant)
    assert got is not None and got != truth, f"{c['name']}: {c['mutant']} decides sample {n} {got}, the reference {truth}"
    # the sample lies between the estimate fma(n, s, P_0) and the break point, inside the rigorous bound
    i = 0 if c["axis"] == "x" else 2
    xe = L.fma(float(n), s[i], p0[i])
    bound = (n + 1) * 2.0 ** -53 * max(abs(p0[i]), abs(float(P[i][n])))
    assert 0 < abs(float(P[i][n]) - xe) <= bound, c["name"]
    for j in L.undecided(P, s, c["k"], gw, w, h, zs, zo, surf, n):
        assert L.look(int(j), 0, p0, s, gw, w, h, sof) is not None, f"{c['name']}: sample {j} needs advance_exact"


# (production, mutant, smallest correct) margin of each band
MARGINS = {"cell": (L.MARGIN, 1, 2), "grid_high": (L.MARGIN, 1, 2), "grid_low": (L.MARGIN, 0, 1),
           "inside_high": (L.MARGIN, 0, 1), "z_above": (L.ZMARGIN, 8, 9), "z_hit": (L.ZMARGIN, 8, 9)}


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_case_is_where_it_claims(case, oracle):
    c = case
    axs, P, (zs, zo), surf, fk, mn, mx = case_model(c)
    n, k, gw = c["n"], c["k"], fk["grid_width"]
    band = c["band"][:4] if c["band"].startswith("cell") else c["band"]
    if band.startswith("fp64"):
        check_look_case(c, P, fk, surf, zs, zo)
        return
    prod, mut, smallest = MARGINS[band]
    w, h = c["map"]["w"], c["map"]["h"]
    if c["axis"] in ("x", "y"):
        ai = 0 if c["axis"] == "x" else 1
        v = axs[ai].at(n)
        assert v == c["v"]
        truth = int(L.truth_cell(P[ai][n:n + 1], gw, c["axis"])[0])
        assert truth == c["truth_cell"]
        n_cells = w if c["axis"] == "x" else h
        grid = n_cells << k
        if band == "cell":
            def right(m):
                d = L.cell_decides(v, k, m)
                return d is None or d == truth
        elif band == "grid_high":
            def right(m):
                return not L.outside_high(v, grid, m) or not L.truth_inside(truth, n_cells)
        elif band == "grid_low":
            def right(m):
                return not L.outside_low(v, k, m) or not L.truth_inside(truth, n_cells)
        else:
            def right(m):
                return not L.inside(v, grid, m) or L.truth_inside(truth, n_cells)
    else:
        v = axs[2].at(n)
        assert v == c["v"]
        gx, gy = (int(L.truth_cell(P[i][n:n + 1], gw, a)[0]) for i, a in ((0, "x"), (1, "y")))
        sp = float(surf[gy, gx])
        q = L.zq16(sp, zs, zo)
        assert q == c["q"]
        below = P[2][n] < sp
        # x and y are decided by the model at n, so only the z predicate decides the sample
        assert L.cell_decides(axs[0].at(n), k, L.MARGIN) == gx and L.cell_decides(axs[1].at(n), k, L.MARGIN) == gy
        if band == "z_above":
            def right(m):
                return not L.above(v, q, m) or not below
        else:
            def right(m):
                return not L.hit(v, q, m) or below
    assert right(prod), f"{c['name']}: the production margin decides sample {n} wrong"
    assert right(smallest), f"{c['name']}: margin {smallest} decides sample {n} wrong"
    assert not right(mut), f"{c['name']}: margin {mut} decides sample {n} right: the case does not reach the edge"

    # the oracle's frame turns on sample n: the reference hits or leaves there, or the mutant would have
    hm, cm = L.case_maps(c["map"])
    of = oracle.make_frame(projection=3, width=fk["screen_width"], height=fk["screen_height"], pos=fk["cam_pos"],
                           hang=fk["hang"], vang=fk["vang"], hfov=fk["hfov"], ortho_width=fk["ortho_width"],
                           grid_width=gw, step_dist=fk["step_dist"], min_height=mn, max_height=mx, bg=fk["bg"],
                           cycle=0, cycle_period=4)        # pixel (0, 0) alone
    _, si, st = oracle.render(of, oracle.update_heightmap(hm, L.LUM, mn, mx), cm)
    if "expect_first_hit" in c:
        assert si[0, 0] == c["expect_first_hit"] and st.steps == si[0, 0] + 1, (c["name"], si[0, 0])
        assert c["expect_first_hit"] in (n, n + 1, n + 2), c
        if c["band"] == "fp64_x":
            assert si[0, 0] == n
    else:
        assert si[0, 0] == -2 and st.steps == c["expect_steps"], (c["name"], si[0, 0], st.steps)
        assert c["expect_steps"] in (n, n + 1), c


def test_cases_cover_every_band_direction_and_window():
    seen = {(c["band"], c["k"], c["motion"]) for c in CASES}
    for band in ("cell_x", "cell_y"):
        for k in (20, 15):
            assert {m for b, kk, m in seen if b == band and kk == k} == {"+" + band[-1], "-" + band[-1]}, (band, k)
    for band in ("cell_x", "cell_y", "grid_high", "grid_low", "inside_high", "z_above", "z_hit"):
        assert {c["window"] for c in CASES if c["band"] == band} == {1, 2}, band
    assert {c["mutant"] for c in CASES if c["band"].startswith("fp64")} == {"look_rel_100", "look_no_bz"}


def test_search_regenerates_the_committed_cases():
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "lin_margin_search.py"), "--check"], cwd=ROOT)
    assert r.returncode == 0, "tools/lin_margin_search.py does not reproduce tests/golden/lin_margin_cases.json"
