"""GPU: the skip traversals against the brute kernel and the CPU oracle on maps larger than 1024 cells, at every
fixed-point resolution k = 20 .. 15, with 8-bit and 16-bit heights, in all three pyramid layouts.

The max-mip pyramid is observed only through its consumer: every case (tests/pyramid_cases.py) is rendered by brute,
skip, skip_fp64 and pack in every layout, and the 12 frames, per-pixel first-hit step indices and step totals must be
identical and equal to the oracle's.  The expected values come from oracle.update_heightmap (8-bit) or
height16_lib.heights16 (16-bit) and the oracle's loop; nothing the device computed feeds them."""
import numpy as np
import pytest

import height16_lib as H16
import pyramid_cases as PC

pytestmark = pytest.mark.gpu

SEEDS = (0, 1)
ORACLE_BUDGET = 200_000_000          # brute samples of one frame above which the oracle is not run
TRAVERSALS = {1: "brute", 2: "skip", 3: "skip_fp64", 4: "pack"}
LAYOUTS = {0: "rowmajor", 1: "tile4", 2: "zorder"}


def upload(hmrm, r, case):
    if case["upload"] == "device":
        import torch

        hm = np.ascontiguousarray(case["hm"])
        dh = torch.from_numpy(hm.view(np.int16) if case["depth"] == 16 else hm).cuda()
        dc = torch.from_numpy(np.ascontiguousarray(case["cm"])).cuda()
        (r.set_maps16_device if case["depth"] == 16 else r.set_maps_device)(dh, dc, case["w"], case["h"])
        torch.cuda.synchronize()
    elif case["depth"] == 16:
        r.set_maps16(case["hm"], case["cm"])
    else:
        r.set_maps(case["hm"], case["cm"])


def expected_heights(oracle, case, lum, mn, mx):
    if case["depth"] == 16:
        return H16.heights16(case["hm"], lum, mn, mx)
    return oracle.update_heightmap(case["hm"], lum, mn, mx)


def render_all(hmrm, r, fk, tag, tally):
    """12 renders (layout x traversal); all must agree.  Returns the brute render's (frame, step index, stats)."""
    kw = {k: v for k, v in fk.items() if k != "needle"}
    ref = None
    for layout, lname in LAYOUTS.items():
        r.set_layout(layout)
        for trav, tname in TRAVERSALS.items():
            f = r.frame(traversal=trav, flags=hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX, **kw)
            img = r.render(f).copy()
            st, si = r.stats(), r.step_index(f)
            where = f"{tag} layout {lname} traversal {tname}"
            assert st.status & 8 == 0, f"{where}: out-of-range index (status {st.status})"
            if trav == 2:
                dbg = r.debug_counters()
                tally["jumps"] += dbg[0]
                tally["exact"] += dbg[7]
                tally["skip_fetches"] += st.fetches
                tally["skip_steps"] += st.steps
            got = (img, si, (st.steps, st.box_hits, st.surf_hits, st.max_steps, st.status))
            if ref is None:
                ref = got
                continue
            assert np.array_equal(got[0], ref[0]), \
                f"{where}: {int((got[0] != ref[0]).any(axis=2).sum())} pixels differ from brute/rowmajor"
            assert np.array_equal(got[1], ref[1]), \
                f"{where}: {int((got[1] != ref[1]).sum())} step indices differ from brute/rowmajor"
            assert got[2] == ref[2], f"{where}: stats {got[2]} != brute/rowmajor {ref[2]}"
    r.set_layout(0)
    return ref


def check_case(hmrm, r, oracle, case, tally):
    settings = [(case["lum"], case["min_height"], case["max_height"])]
    if case["relum"] is not None:
        settings.append(case["relum"])
    for si_, (lum, mn, mx) in enumerate(settings):
        r.lum_r, r.lum_g, r.lum_b = lum
        r.min_height, r.max_height = mn, mx
        if si_ == 0:
            upload(hmrm, r, case)       # builds the pyramid with this setting
        else:
            r.update_heightmap()        # new lum / min / max over the maps already on the device
        heights = None
        for fi, fk in enumerate(case["frames"]):
            tag = (f"k {case['k']} depth {case['depth']} seed {case['seed']} case {case['index']} ({case['name']}) "
                   f"map {case['w']}x{case['h']} upload {case['upload']} setting {si_} lum {lum} h [{mn},{mx}] "
                   f"frame {fi} {fk}")
            img, steps, st = render_all(hmrm, r, fk, tag, tally)
            tally["frames"] += 1
            tally["hits"] += st[2] > 0
            tally["long"] += st[3] > 10_000
            if st[4] != 0 or st[0] > ORACLE_BUDGET:
                continue
            if heights is None:
                heights = expected_heights(oracle, case, lum, mn, mx)
            of = oracle.make_frame(projection=fk["projection"], width=fk["screen_width"], height=fk["screen_height"],
                                   pos=fk["cam_pos"], hang=fk["hang"], vang=fk["vang"], hfov=fk["hfov"],
                                   ortho_width=fk["ortho_width"], grid_width=fk["grid_width"],
                                   step_dist=fk["step_dist"], min_height=mn, max_height=mx, bg=fk["bg"])
            want, osteps, ost = oracle.render(of, heights, case["cm"])
            tally["oracle"] += 1
            assert np.array_equal(img, want), f"{tag}: {int((img != want).any(axis=2).sum())} pixels differ from the oracle"
            assert np.array_equal(steps, osteps), f"{tag}: {int((steps != osteps).sum())} step indices differ from the oracle"
            assert st[:4] == (ost.steps, ost.box_hits, ost.surf_hits, ost.max_steps), f"{tag}: stats {st} != oracle {ost}"
            if si_ == 0 and fk["needle"] is not None:
                nd = case["needles"][fi]
                seen = bool(np.all(want[:, :, :3] == np.array(nd["rgba"][:3], np.uint8), axis=2).any())
                tally["needles_missing"] += [] if seen else [f"{tag}: needle {nd} not in the oracle frame"]


@pytest.mark.parametrize("depth", (8, 16))
@pytest.mark.parametrize("k", PC.K_VALUES)
def test_traversals_match_oracle_over_large_maps(hmrm, renderer, oracle, k, depth):
    tally = dict(frames=0, oracle=0, hits=0, long=0, jumps=0, exact=0, skip_fetches=0, skip_steps=0,
                 needles_missing=[])
    try:
        for seed in SEEDS:
            for case in PC.cases(k, depth, seed):
                check_case(hmrm, renderer, oracle, case, tally)
    finally:
        renderer.set_layout(0)
    # not vacuous: most frames reach the oracle, some hit terrain and some march far, every needle is seen, the skip
    # traversal skipped, jumped and used its exact FP64 path
    assert tally["oracle"] >= 0.8 * tally["frames"], tally
    assert tally["hits"] > 0 and tally["long"] > 0, tally
    assert not tally["needles_missing"], tally["needles_missing"]
    assert tally["skip_fetches"] < tally["skip_steps"], tally
    assert tally["jumps"] > 0 and tally["exact"] > 0, tally


def test_pack_rebases_its_model_after_an_exact_decision(hmrm, renderer, oracle):
    """Found by this fuzz (edge case of k = 19, after the change of min / max): rays along -y exactly on the cell edges
    x = 1 and 4 cells need the exact FP64 reconstruction at every sample that the integer model cannot place.  After such
    a decision k2_render_pack rebuilt its model from the exact state that had been moved to the decided sample instead
    of the first sample of the model's window, so the model ran one step ahead: the rays left the grid early and the
    step totals fell short of the oracle's (14 instead of 22)."""
    w, h = 1025, 5
    hm = np.full((h, w, 3), 255, dtype=np.uint8)
    hm[:, 0] = 0
    cm = PC._colormap(np.random.RandomState(5), h, w)
    case = dict(k=19, depth=8, seed=0, index=0, name="pack_rebase", w=w, h=h, hm=hm, cm=cm, lum=PC.LUMS[0],
                min_height=-1.0, max_height=2.5, upload="host", relum=None, needles=[],
                frames=[dict(projection=3, screen_width=3, screen_height=2, cam_pos=(0.25, 0.5, 1.0),
                             hang=-np.pi / 2, vang=np.pi / 2, hfov=1.0, ortho_width=0.5, grid_width=0.25,
                             step_dist=0.125, bg=PC.BG, needle=None)])
    tally = dict(frames=0, oracle=0, hits=0, long=0, jumps=0, exact=0, skip_fetches=0, skip_steps=0, needles_missing=[])
    check_case(hmrm, renderer, oracle, case, tally)
    assert tally["oracle"] == 1 and tally["exact"] > 0, tally
