"""GPU: k2_render_lin's decision margins at their edges.  Every case of tests/golden/lin_margin_cases.json (made by
tools/lin_margin_search.py, checked on the CPU by tests/test_lin_model.py) puts pixel (0, 0)'s ray at a sample where the
integer model is more than one unit off in the direction that a one-unit-smaller margin would misjudge (the cell test,
the grid tests and the height tests), or at a sample placed ulp by ulp between the FP64 look's estimate and a cell edge
or the surface, where only the look's full error bound sends it on to advance_exact.  The map is built around that
sample, so a kernel with a margin one unit too small, or a look with a smaller bound, renders a different step index,
colour or step total there.

Each case is rendered by brute, skip, skip_fp64 and pack in the row-major and the 4x4-tiled pyramid layout; frame,
per-pixel step index and (steps, box_hits, surf_hits, max_steps) must equal the oracle's, and the device's ray and entry
point, from which the model's start P_0 = fl(e + fl(nudge d)) and step fl(step d) follow, must equal the oracle's."""
import json
from pathlib import Path

import numpy as np
import pytest

import lin_model as L

pytestmark = pytest.mark.gpu

CASES = json.loads((Path(__file__).resolve().parent / "golden" / "lin_margin_cases.json").read_text())["cases"]
TRAVERSALS = {1: "brute", 2: "skip", 3: "skip_fp64", 4: "pack"}
LAYOUTS = {0: "rowmajor", 1: "tile4"}


def frame_kwargs(c):
    f = c["frame"]
    return dict(projection=f["projection"], screen_width=f["screen_width"], screen_height=f["screen_height"],
                cam_pos=tuple(float.fromhex(v) for v in f["cam_pos"]), hang=float.fromhex(f["hang"]),
                vang=float.fromhex(f["vang"]), hfov=float.fromhex(f["hfov"]), ortho_width=float.fromhex(f["ortho_width"]),
                grid_width=float.fromhex(f["grid_width"]), step_dist=float.fromhex(f["step_dist"]), bg=tuple(f["bg"]))


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_margin_case_matches_oracle(hmrm, oracle, case):
    c = case
    fk = frame_kwargs(c)
    mn, mx = float.fromhex(c["min_height"]), float.fromhex(c["max_height"])
    hm, cm = L.case_maps(c["map"])
    w, h = c["map"]["w"], c["map"]["h"]
    of = oracle.make_frame(projection=fk["projection"], width=fk["screen_width"], height=fk["screen_height"],
                           pos=fk["cam_pos"], hang=fk["hang"], vang=fk["vang"], hfov=fk["hfov"],
                           ortho_width=fk["ortho_width"], grid_width=fk["grid_width"], step_dist=fk["step_dist"],
                           min_height=mn, max_height=mx, bg=fk["bg"])
    want, osteps, ost = oracle.render(of, oracle.update_heightmap(hm, L.LUM, mn, mx), cm)
    if "expect_first_hit" in c:
        assert osteps[0, 0] == c["expect_first_hit"], c["name"]
    r = hmrm.Renderer(0)
    try:
        r.lum_r, r.lum_g, r.lum_b = L.LUM
        r.min_height, r.max_height = mn, mx
        r.set_maps(hm, cm)
        # the model's inputs: the device's ray and box entry of pixel (0, 0) are the oracle's, bit for bit
        f = r.frame(traversal=2, flags=hmrm.FLAG_STATS | hmrm.FLAG_RAY_DUMP, **fk)
        r.render(f)
        dump = r.ray_dump(f)[0, 0]
        pos, d = oracle.get_ray(of, 0.0, 0.0)
        hit, e = oracle.intersection(pos, d, (0.0, 0.0, mn), (w * fk["grid_width"], -h * fk["grid_width"], mx))
        assert hit
        assert [float(v).hex() for v in dump[3:6]] == [v.hex() for v in d], c["name"]
        assert [float(v).hex() for v in dump[7:10]] == [v.hex() for v in e], c["name"]
        for layout, lname in LAYOUTS.items():
            r.set_layout(layout)
            for trav, tname in TRAVERSALS.items():
                f = r.frame(traversal=trav, flags=hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX, **fk)
                img = r.render(f).copy()
                st, si = r.stats(), r.step_index(f)
                tag = f"{c['name']} (sample {c['n']}, mutant {c['mutant']}) layout {lname} traversal {tname}"
                assert st.status & 8 == 0, f"{tag}: out-of-range index (status {st.status})"
                assert np.array_equal(si, osteps), f"{tag}: step indices {si.ravel()} != oracle {osteps.ravel()}"
                assert np.array_equal(img, want), f"{tag}: {int((img != want).any(axis=2).sum())} pixels differ"
                got = (st.steps, st.box_hits, st.surf_hits, st.max_steps)
                assert got == (ost.steps, ost.box_hits, ost.surf_hits, ost.max_steps), f"{tag}: stats {got} != oracle"
                if trav == 2 and c["band"].startswith("fp64"):
                    # the look refused sample n: the exact reconstruction decided it
                    assert r.debug_counters()[7] > 0, f"{tag}: no sample went to advance_exact"
    finally:
        r.close()
