"""CPU: the numpy model of a supersampled frame (include/hmrm.h: the box filter of the same camera's sW x sH frame) that
the device path is tested with (tests/test_gpu_supersample.py), proven here on hand-worked cases including the rounding
ties; the HMRM_FLAG_SUPERSAMPLE macros and their binding mirror; and hmap's --supersample usage refusals (no GPU needed
for any of them)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"


def box_reduce(frame, s: int, channels: int = 4):
    """[sH, sW, 3 | 4] uint8 frame -> [H, W, channels] uint8: each R, G, B is (sum + s*s/2) // (s*s) over the pixel's
    s x s subsamples, alpha 255 (include/hmrm.h)."""
    f = np.asarray(frame)
    sh, sw = f.shape[:2]
    assert sh % s == 0 and sw % s == 0, f"{sw}x{sh} is not a multiple of {s}"
    h, w = sh // s, sw // s
    n = s * s
    sums = f[:, :, :3].astype(np.int64).reshape(h, s, w, s, 3).sum(axis=(1, 3))
    out = np.empty((h, w, channels), dtype=np.uint8)
    out[:, :, :3] = (sums + n // 2) // n
    if channels == 4:
        out[:, :, 3] = 255
    return out


def _uniform_sum(s, total):
    """An s x s block (one output pixel) whose red channel sums to `total`, green to total + 1, blue to 0."""
    r = np.zeros(s * s, dtype=np.int64)
    g = np.zeros(s * s, dtype=np.int64)
    for k in range(total):
        r[k % (s * s)] += 1
    for k in range(total + 1):
        g[k % (s * s)] += 1
    px = np.zeros((s, s, 4), dtype=np.uint8)
    px[:, :, 0] = r.reshape(s, s)
    px[:, :, 1] = g.reshape(s, s)
    px[:, :, 3] = 255
    return px


@pytest.mark.parametrize("s,total,want", [
    (2, 1, 0), (2, 2, 1), (2, 5, 1), (2, 6, 2),          # (sum + 2) // 4
    (3, 4, 0), (3, 5, 1), (3, 13, 1), (3, 14, 2),        # (sum + 4) // 9
    (4, 7, 0), (4, 8, 1), (4, 23, 1), (4, 24, 2),        # (sum + 8) // 16
])
def test_box_reduce_rounding_ties(s, total, want):
    out = box_reduce(_uniform_sum(s, total), s)
    assert out.shape == (1, 1, 4)
    assert out[0, 0, 0] == want
    assert out[0, 0, 1] == (total + 1 + (s * s) // 2) // (s * s)
    assert out[0, 0, 2] == 0 and out[0, 0, 3] == 255


def test_box_reduce_hand_worked_2x2():
    # a 4 x 2 sub-frame, s = 2: output pixel 0 averages columns 0-1, pixel 1 columns 2-3
    f = np.zeros((2, 4, 4), dtype=np.uint8)
    f[:, :, 3] = 0                                   # the input's alpha is not used
    f[0, 0, :3] = (255, 0, 10)
    f[0, 1, :3] = (255, 0, 10)
    f[1, 0, :3] = (0, 255, 10)
    f[1, 1, :3] = (1, 255, 11)
    f[:, 2:, 0] = 100
    f[1, 3, 2] = 3
    out = box_reduce(f, 2)
    # R: (511 + 2) // 4 = 128; G: (510 + 2) // 4 = 128; B: (41 + 2) // 4 = 10
    assert out[0, 0].tolist() == [128, 128, 10, 255]
    # R: 400 // 4 = 100 (+2 rounds down); B: (3 + 2) // 4 = 1
    assert out[0, 1].tolist() == [100, 0, 1, 255]
    rgb = box_reduce(f, 2, channels=3)
    assert rgb.shape == (1, 2, 3) and rgb.tolist() == [[[128, 128, 10], [100, 0, 1]]]


def test_box_reduce_extremes_and_identity():
    for s in (1, 2, 3, 4):
        white = np.full((3 * s, 5 * s, 4), 255, dtype=np.uint8)
        assert (box_reduce(white, s) == 255).all()
        assert (box_reduce(np.zeros((2 * s, 2 * s, 3), np.uint8), s, channels=3) == 0).all()
    rng = np.random.default_rng(3)
    f = rng.integers(0, 256, size=(7, 9, 4), dtype=np.uint8)
    f[:, :, 3] = 255
    assert np.array_equal(box_reduce(f, 1), f)                      # s = 1 is the frame itself


def test_box_reduce_equals_float_mean_rounded_half_up():
    rng = np.random.default_rng(8)
    for s in (2, 3, 4):
        f = rng.integers(0, 256, size=(5 * s, 11 * s, 4), dtype=np.uint8)
        mean = f[:, :, :3].astype(np.float64).reshape(5, s, 11, s, 3).mean(axis=(1, 3))
        assert np.array_equal(box_reduce(f, s)[:, :, :3], np.floor(mean + 0.5).astype(np.uint8))


def _header_macros():
    """The values of the HMRM_FLAG_SUPERSAMPLE* macros as a C compiler sees include/hmrm.h."""
    import os
    import tempfile

    src = ('#include <stdio.h>\n#include "hmrm.h"\nint main(void) { printf("%u %u %u %u %u %u\\n", '
           "(unsigned)HMRM_FLAG_SUPERSAMPLE_SHIFT, (unsigned)HMRM_FLAG_SUPERSAMPLE_MASK, HMRM_FLAG_SUPERSAMPLE(1), "
           "HMRM_FLAG_SUPERSAMPLE(2), HMRM_FLAG_SUPERSAMPLE(3), HMRM_FLAG_SUPERSAMPLE(4)); return 0; }\n")
    with tempfile.TemporaryDirectory() as td:
        c, exe = os.path.join(td, "m.c"), os.path.join(td, "m")
        Path(c).write_text(src)
        subprocess.run(["cc", "-I", str(ROOT / "include"), "-o", exe, c], check=True)
        return [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]


def test_flag_macros_and_binding_mirror(hmrm):
    shift, mask, *flags = _header_macros()
    assert (shift, mask) == (8, 0xF00)
    assert flags == [0, 256, 512, 768]
    assert (hmrm.FLAG_SUPERSAMPLE_SHIFT, hmrm.FLAG_SUPERSAMPLE_MASK) == (shift, mask)
    assert [hmrm.supersample_flag(s) for s in (1, 2, 3, 4)] == flags
    # the supersample bits do not overlap the other flags
    assert mask & (hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX | hmrm.FLAG_RAY_DUMP) == 0
    for bad in (0, 5, -1, 2.0, True, "2"):
        with pytest.raises(ValueError):
            hmrm.supersample_flag(bad)


@pytest.mark.parametrize("args", [
    ["--headless", "o.png", "--supersample", "0"],
    ["--headless", "o.png", "--supersample", "5"],
    ["--headless", "o.png", "--supersample", "-2"],
    ["--headless", "o.png", "--supersample", "two"],
    ["--headless", "o.png", "--supersample"],
    ["--headless", "o.png", "--supersample", "2", "--gpus", "2"],
    ["--script", "frames.txt", "--video", "v.y4m", "--supersample", "5"],
])
def test_hmap_supersample_usage_refusals(hmrm, args, tmp_path):
    assert HMAP.exists(), "hmap host binary was not built"
    (tmp_path / "config.txt").write_text("resolution 64 48\n")
    (tmp_path / "frames.txt").write_text("hang 10\n")
    res = subprocess.run([str(HMAP), "config.txt", *args], capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 1
    assert res.stderr.splitlines()[0] == "USAGE: hmap.exe path/to/config.txt"
    assert "--supersample 1|2|3|4" in res.stderr and res.stdout == ""
    assert not (tmp_path / "o.png").exists() and not (tmp_path / "v.y4m").exists()


@pytest.mark.parametrize("n", ["1", "4"])
def test_hmap_supersample_accepted_by_the_option_checks(hmrm, n, tmp_path):
    (tmp_path / "config.txt").write_text("resolution 64 48\n")
    res = subprocess.run([str(HMAP), "config.txt", "--headless", "o.png", "--supersample", n, "--parse-only"],
                         capture_output=True, text=True, cwd=str(tmp_path))
    # past the option checks: the config is read and echoed (it names no maps, so the grammar check then fails)
    assert "USAGE" not in res.stderr and res.stdout.startswith("resolution 64 48")
