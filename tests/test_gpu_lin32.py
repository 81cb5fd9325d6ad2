"""GPU: k2_render_lin evaluates its integer ray model in 32 bits (V_j = V_0 + j Di + ((j Df + 2^15) >> 16), DESIGN.md
§4).  These scenes put rays at the edges of the argument that this is exact: the height coordinate of an ascending
ray leaving the int range inside one model window, per-step motion close to the 2^26-unit limit of the model on a
2^30-unit grid, and slow rays that cross several 65536-sample re-anchors; each also with a far too narrow height
quantiser (HMRM_ZQ_RANGE_SHRINK), which multiplies the model's height units.  Frame, per-pixel step index and step
totals of the skip traversal must equal the brute traversal's and the oracle's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LUM = (0.299, 0.587, 0.114)


def noise_maps(seed, h, w, lo, hi):
    """An h x w map of grey noise between lo and hi (0..255) in blocks of 64 cells, so that skips are long, and one
    255 cell in a corner: the terrain box reaches height 1 and the cameras below start inside it.  Maps of 1024 cells
    or more along their longer side have a grid 2^30 model units wide (fx_bits = 30 - log2 size)."""
    rng = np.random.RandomState(seed)
    coarse = rng.randint(lo, hi + 1, size=(h // 64 + 1, w // 64 + 1))
    v = np.kron(coarse, np.ones((64, 64)))[:h, :w]
    v[0, -1] = 255
    hm = np.dstack([v, v, v]).astype(np.uint8)
    cm = rng.randint(0, 256, size=(h, w, 4)).astype(np.uint8)
    return hm, cm


def scene(name):
    """(height map, colour map, frame arguments, what the brute traversal's stats must show).  Grid width 1, heights
    span [0, 1].  The orthographic rays (hang 0: no motion along y) march along a 32768 x 16 strip.  Every camera is
    outside the terrain box: the march starts where a ray enters it."""
    if name == "ascending":
        # enters through the x = 0 face, ~0.43 height ranges up per step: V_z (1/16 Zq units, ~2^20 per height range)
        # passes 2^31 after ~5000 samples, x leaves the grid after ~48000, all inside the first window
        hm, cm = noise_maps(11, 16, 32768, 0, 100)
        fk = dict(projection=3, screen_width=6, screen_height=4, cam_pos=(-0.5, -8.0, 0.3), hang=0.0, vang=1.0,
                  ortho_width=0.05, step_dist=0.8)
        return hm, cm, fk, lambda st: st.max_steps > 40000
    if name == "ascending_steep":
        # passes 2^31 after a few hundred samples, then re-anchors with V_z out of range: the per-step loop finishes
        hm, cm = noise_maps(12, 16, 32768, 0, 100)
        fk = dict(projection=3, screen_width=5, screen_height=3, cam_pos=(-0.1, -8.0, 0.3), hang=0.0, vang=0.2,
                  ortho_width=0.02, step_dist=2.0)
        return hm, cm, fk, lambda st: st.max_steps > 70000
    if name == "big_steps":
        # 126 .. 132 cells per step along x on a 2048^2 map (fx_bits 19): just under and just over 2^26 units, some
        # pixels fit the model and some do not.  The top row descends by ~0.0002 per cell, the bottom row by ~0.04.
        hm, cm = noise_maps(13, 2048, 2048, 0, 200)
        fk = dict(projection=1, screen_width=32, screen_height=2, cam_pos=(-10.0, -1024.0, 0.9), hang=0.0,
                  vang=float(np.pi / 2 + 0.0195), hfov=0.6, step_dist=132.0)
        return hm, cm, fk, lambda st: st.max_steps > 8
    if name == "slow_descent":
        # enters through the top, then 1e-6 height per sample down towards terrain at <= 0.39: ~600000 samples,
        # several re-anchors of the model
        hm, cm = noise_maps(14, 16, 32768, 60, 100)
        fk = dict(projection=3, screen_width=4, screen_height=3, cam_pos=(20.0, -8.0, 1.2), hang=0.0,
                  vang=float(np.pi / 2 + 1e-4), ortho_width=0.05, step_dist=0.01)
        return hm, cm, fk, lambda st: st.max_steps > 3 * 65536
    raise KeyError(name)


@pytest.mark.parametrize("shrink", [None, "0.02"])
@pytest.mark.parametrize("name", ["ascending", "ascending_steep", "big_steps", "slow_descent"])
def test_lin_model_edges_match_brute_and_oracle(hmrm, oracle, name, shrink, monkeypatch):
    if shrink is not None:
        monkeypatch.setenv("HMRM_ZQ_RANGE_SHRINK", shrink)
    hm, cm, fk, exercised = scene(name)
    mn, mx = 0.0, 1.0
    fk = dict(dict(hfov=0.5, ortho_width=0.5), **fk, grid_width=1.0, bg=(4, 5, 6))
    of = oracle.make_frame(projection=fk["projection"], width=fk["screen_width"], height=fk["screen_height"],
                           pos=fk["cam_pos"], hang=fk["hang"], vang=fk["vang"], hfov=fk["hfov"],
                           ortho_width=fk["ortho_width"], grid_width=fk["grid_width"], step_dist=fk["step_dist"],
                           min_height=mn, max_height=mx, bg=fk["bg"])
    want, osteps, ost = oracle.render(of, oracle.update_heightmap(hm, LUM, mn, mx), cm)
    r = hmrm.Renderer(0)
    try:
        r.lum_r, r.lum_g, r.lum_b = LUM
        r.min_height, r.max_height = mn, mx
        r.set_maps(hm, cm)
        stats = {}
        for trav in (1, 2):
            f = r.frame(traversal=trav, flags=hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX, **fk)
            got = r.render(f).copy()
            st, si = r.stats(), r.step_index(f)
            tag = f"{name} shrink {shrink} traversal {trav}"
            assert np.array_equal(got, want), f"{tag}: {int((got != want).any(axis=2).sum())} pixels differ"
            assert np.array_equal(si, osteps), f"{tag}: step indices differ"
            assert (st.steps, st.box_hits, st.surf_hits, st.max_steps) == (ost.steps, ost.box_hits, ost.surf_hits, ost.max_steps), tag
            stats[trav] = st
    finally:
        r.close()
    assert exercised(stats[1]), (name, stats[1].max_steps, stats[1].box_hits)
