"""CPU: the case generator of tests/test_gpu_pyramid_fuzz.py keeps reaching the K1 branches it is meant to reach, at
every fixed-point resolution k and both height depths.  A generator that drifted into small or regular maps would
let the GPU fuzz pass without looking at anything."""
import numpy as np
import pytest

import pyramid_cases as PC

SEEDS = (0, 1)       # the seeds tests/test_gpu_pyramid_fuzz.py runs


def test_fx_bits_restates_the_product_formula():
    assert [PC.fx_bits(n, 1) for n in (1, 2, 1024, 1025, 2048, 2049, 32768)] == [20, 20, 20, 19, 19, 18, 15]
    for k, sizes in PC.SIZES.items():
        assert all(PC.fx_bits(n, 1) == k and PC.fx_bits(1, n) == k for n in sizes)
    assert all(PC.fx_bits(*wh) == k for k, wh in PC.MAP2D.items())


def summarise(k, depth):
    seen = dict(w_mod4=False, h_mod4=False, level_mod4_1=False, regions=0, levels=0, cells=0, needles=set(),
                uploads=set(), relum=0, cases=0)
    for seed in SEEDS:
        for case in PC.cases(k, depth, seed):
            w, h = case["w"], case["h"]
            assert case["hm"].shape[:2] == (h, w) and case["cm"].shape == (h, w, 4)
            assert case["hm"].dtype == (np.uint8 if depth == 8 else np.uint16)
            assert case["frames"], case["name"]
            shapes = PC.mip_shapes(w, h)
            seen["cases"] += 1
            seen["w_mod4"] |= w % 4 != 0
            seen["h_mod4"] |= h % 4 != 0
            seen["level_mod4_1"] |= any(lw % 4 == 1 and lw >= 5 for lw, _ in shapes[1:])
            seen["regions"] = max(seen["regions"], PC.mip_regions(w, h))
            seen["levels"] = max(seen["levels"], len(shapes))
            seen["cells"] = max(seen["cells"], w * h)
            seen["uploads"].add(case["upload"])
            seen["relum"] += case["relum"] is not None
            assert case["hm"].nbytes + case["cm"].nbytes + 8 * w * h < 1 << 30      # with the oracle's heights
            stride = PC.row_stride(w, h)
            colours = {}
            for nd in case["needles"]:
                seen["needles"].add(nd["placement"])
                x, y = nd["x"], nd["y"]
                assert 0 <= x < w and 0 <= y < h
                assert tuple(case["cm"][y, x]) == nd["rgba"]
                colours[nd["rgba"]] = (x, y)
                if nd["placement"] == "unsampled_row":
                    assert y % stride != 0
                    assert int(np.asarray(case["hm"])[y, x].ravel()[0]) > int(np.asarray(case["hm"])[0, 0].ravel()[0])
                if nd["placement"] == "last_col":
                    assert x == w - 1
                if nd["placement"] == "last_row":
                    assert y == h - 1
                if nd["placement"] == "region_seam":
                    assert x % 512 in (0, 511)
                if nd["placement"] == "block_seam":
                    assert x % 4 in (0, 3)
                if nd["placement"] == "level_last_col":
                    assert any(lw % 4 == 1 and (x >> l) == lw - 1 for l, (lw, _) in enumerate(shapes) if l >= 1)
            # needle colours are used by no other cell
            if colours:
                rgb = case["cm"][:, :, :3].reshape(-1, 3)
                for c in colours:
                    assert int(np.all(rgb == np.array(c[:3], np.uint8), axis=1).sum()) == 1, (case["name"], c)
                assert len(case["frames"]) == len(case["needles"])
    return seen


@pytest.mark.parametrize("depth", (8, 16))
@pytest.mark.parametrize("k", PC.K_VALUES)
def test_cases_reach_the_size_dependent_branches(k, depth):
    s = summarise(k, depth)
    assert s["w_mod4"] and s["h_mod4"], s
    assert s["level_mod4_1"], s                   # k1_dilate_levels' last column of a width = 1 (mod 4) level
    assert s["regions"] > 1, s                    # k1_mip_upper with more than one CTA
    assert s["levels"] > 10, s                    # k1_mip_upper's last-CTA levels >= 10
    assert s["uploads"] == {"host", "device"}, s
    assert s["relum"] >= s["cases"] // 3, s
    want = set(PC.PLACEMENTS)
    if k == 20:
        # a map of long side <= 1024 has at most 2^20 cells, and k1_range then reads every row
        assert s["cells"] <= 1 << 20
        want.discard("unsampled_row")
    else:
        assert s["cells"] > 1 << 20, s            # k1_range samples every row_stride-th row only
    assert want <= s["needles"], (want - s["needles"], s)


@pytest.mark.parametrize("k", PC.K_VALUES)
def test_edge_case_puts_a_sample_just_below_a_cell_edge(k):
    """Frame 1 of the edge case: sample 1 lies less than one unit below the edge of cell 1 (the reference's (int)
    truncation gives cell 0), and the integer model of k2_render_lin rounds it onto the edge."""
    case = next(c for c in PC.cases(k, 8, 0) if c["kind"] == "edge")
    f = case["frames"][0]
    gw = f["grid_width"]
    x0 = 0.0 + (gw * 0.01) * 1.0
    x1 = x0 + f["step_dist"] * 1.0
    assert int(x0 / gw) == 0 and int(x1 / gw) == 0 and int((x1 + f["step_dist"]) / gw) == 1
    X1 = x1 * 2.0 ** k / gw
    assert 2.0 ** k - 1.0 <= X1 < 2.0 ** k
    V0 = int(np.floor(x0 * 2.0 ** k / gw + 0.5))
    D = f["step_dist"] * 2.0 ** k / gw * 65536.0
    assert D == int(D)
    assert V0 + (int(D) + 32768) // 65536 == 1 << k
