"""CPU: the selection model of the destination tests (tests/destinations_model.py) against the two independent
statements of the same selections: the oracle's own cycle loop over a row band (oracle/hmap_oracle.c, render_core),
and multi_gpu.owned_pixel_rows for interleaved bands.  A wrong model would let the GPU tests agree with a wrong kernel."""
import itertools

import numpy as np
import pytest

import destinations_model as M


def _oracle_written(oracle, W, H, rows, cycle, period):
    """Pixels the oracle writes for this selection: it stores A = 255 on every pixel it renders."""
    rng = np.random.default_rng(W * 1000 + H)
    hm = rng.integers(0, 256, size=(6, 5, 3), dtype=np.uint8)
    cm = rng.integers(0, 256, size=(6, 5, 4), dtype=np.uint8)
    heights = oracle.update_heightmap(hm, max_height=1.0)
    f = oracle.make_frame(projection=oracle.PERSPECTIVE, width=W, height=H, pos=(-0.2, 0.2, 1.5), hang_deg=-45.0,
                          vang_deg=120.0, grid_width=0.05, step_dist=0.05, max_height=1.0, cycle=cycle,
                          cycle_period=period)
    fb = np.zeros((H, W, 4), dtype=np.uint8)
    oracle.render(f, heights, cm, want_steps=False, rows=rows, framebuf=fb)
    return fb[:, :, 3] == 255


@pytest.mark.parametrize("period", [1, 2, 3, 7, 47])
def test_cycle_and_row_band_match_the_oracle_loop(oracle, period):
    rng = np.random.default_rng(period)
    for W, H in [(2, 2), (3, 5), (8, 4), (13, 9), (33, 7), (65, 3)]:
        for cycle in sorted({0, period - 1, int(rng.integers(0, period))}):
            bands = [(0, H), (1, H), (H - 1, H), (0, 1)] + [tuple(sorted(rng.choice(H + 1, 2, replace=False)))
                                                           for _ in range(3)]
            for rb, re in bands:
                want = _oracle_written(oracle, W, H, (rb, re), cycle, period)
                got = M.selected(W, H, rb, re, cycle=cycle, period=period)
                assert np.array_equal(got, want), (W, H, rb, re, cycle, period)


def test_interleaved_bands_match_owned_pixel_rows(hmrm):
    from heightmap_ray_marcher_b200 import multi_gpu as MG

    for H in range(2, 27):
        for rb, re in [(0, H)] + [(a, b) for a, b in itertools.combinations(range(H + 1), 2) if (a + b) % 3 == 0]:
            for n in range(1, 6):
                for b in range(n):
                    mask = M.selected(3, H, rb, re, band_count=n, band_index=b)
                    rows = [int(r) for r in np.nonzero(mask.any(axis=1))[0]]
                    assert rows == [rb + r for r in MG.owned_pixel_rows(re - rb, b, n)], (H, rb, re, n, b)
                    assert mask[rows].all()


def test_bands_and_cycles_partition_the_row_band():
    """Every pixel of [row_begin, row_end) belongs to exactly one (band_index, cycle) pair, and no other pixel to any."""
    for W, H, rb, re in [(5, 9, 0, 9), (8, 13, 3, 11), (17, 6, 1, 2), (2, 21, 5, 21)]:
        for n, period in [(1, 1), (2, 3), (5, 7), (3, 47)]:
            count = sum(M.selected(W, H, rb, re, n, b, c, period).astype(int) for b in range(n) for c in range(period))
            want = np.zeros((H, W), dtype=int)
            want[rb:re] = 1
            assert np.array_equal(count, want), (W, H, rb, re, n, period)


def test_band_index_beyond_the_tile_rows_owns_nothing():
    assert not M.selected(9, 4, band_count=2, band_index=1).any()
    assert not M.selected(9, 11, 6, 11, band_count=3, band_index=2).any()
    assert M.selected(9, 11, 6, 11, band_count=3, band_index=1)[10:].all()


def test_expected_destination_writes_only_selected_pixel_bytes():
    fill = np.arange(1, 1 + 2 * 8 + 2 * 3 * 3, dtype=np.uint8)
    frame = np.full((2, 3, 4), 200, dtype=np.uint8)
    frame[:, :, 3] = 255
    mask = np.array([[True, False, False], [False, False, True]])
    out = M.expected_destination(fill, 8 + 1, frame, mask, 3)
    changed = np.nonzero(out != fill)[0].tolist()
    assert changed == [9, 10, 11, 24, 25, 26]
    out4 = M.expected_destination(np.zeros(30, dtype=np.uint8) + 7, 3, frame, mask, 4)
    assert out4[3:7].tolist() == [200, 200, 200, 255] and out4[23:27].tolist() == [200, 200, 200, 255]
    assert (np.delete(out4, list(range(3, 7)) + list(range(23, 27))) == 7).all()


def test_sentinel_bytes_avoid_0_and_255():
    b = M.sentinel_bytes(np.random.default_rng(0), 100000)
    assert b.min() == 1 and b.max() == 254
