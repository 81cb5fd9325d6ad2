"""CPU: the numpy model of a motion-blurred frame (include/hmrm.h, hmrm_set_motion_blur: the rounded box average of the
reference's frames at several cameras) that tests/test_gpu_motion_blur.py checks the device against, proven here on
hand-worked rounding ties, against the float mean and against box_reduce; the collapse property that makes n identical
cameras the plain frame; the hmrm_camera layout and its binding mirror; and hmap's --motion-blur usage refusals."""
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from test_supersample import box_reduce

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"


def blur_reduce(subframes, s: int, channels: int = 4):
    """n sub-frames [sH, sW, 3 | 4] uint8 -> [H, W, channels] uint8: each R, G, B is (sum + N/2) // N with N = n*s*s and
    the sum over the s x s subsamples of the pixel in all n sub-frames, alpha 255 (include/hmrm.h)."""
    f = np.stack([np.asarray(x) for x in subframes])
    n, sh, sw = f.shape[:3]
    assert sh % s == 0 and sw % s == 0, f"{sw}x{sh} is not a multiple of {s}"
    h, w = sh // s, sw // s
    big_n = n * s * s
    sums = f[..., :3].astype(np.int64).reshape(n, h, s, w, s, 3).sum(axis=(0, 2, 4))
    out = np.empty((h, w, channels), dtype=np.uint8)
    out[:, :, :3] = (sums + big_n // 2) // big_n
    if channels == 4:
        out[:, :, 3] = 255
    return out


def blur_cameras(c0, c1, shutter: float, k: int):
    """hmap --motion-blur: sub-frame j of k uses t = (F * j) / k and c = c0 + t * (c1 - c0), per component of
    (x, y, z, hang, vang), in doubles and in that order."""
    out = []
    for j in range(k):
        t = (shutter * j) / k
        out.append(tuple(a + t * (b - a) for a, b in zip(c0, c1)))
    return out


def _pixel(values, s):
    """n sub-frames of one s x s block whose red subsamples are `values` (n*s*s of them), green 255 - red."""
    v = np.asarray(values, dtype=np.uint8).reshape(-1, s, s)
    f = np.zeros(v.shape + (4,), dtype=np.uint8)
    f[..., 0] = v
    f[..., 1] = 255 - v
    f[..., 3] = 7                                      # the input's alpha is not used
    return list(f)


@pytest.mark.parametrize("s,values,want", [
    (1, [0, 1], 1), (1, [0, 0], 0), (1, [3, 4], 4), (1, [254, 255], 255),           # (sum + 1) // 2
    (1, [0, 0, 1], 0), (1, [0, 1, 1], 1), (1, [1, 1, 2], 1), (1, [2, 2, 1], 2),     # (sum + 1) // 3
    (1, [0, 0, 1, 1], 1), (1, [0, 0, 0, 1], 0), (1, [1, 1, 1, 2], 1), (1, [2, 2, 2, 1], 2),   # (sum + 2) // 4
    (2, [0] * 6 + [1] * 2, 0), (2, [0] * 4 + [1] * 4, 1),                           # n = 2, s = 2: (sum + 4) // 8
    (2, [0] * 7 + [2], 0), (2, [0] * 6 + [2, 2], 1),
])
def test_blur_reduce_rounding_ties(s, values, want):
    out = blur_reduce(_pixel(values, s), s)
    n = len(values)
    assert out.shape == (1, 1, 4)
    assert out[0, 0].tolist() == [want, (255 * n - sum(values) + n // 2) // n, 0, 255]


def test_blur_reduce_hand_worked_two_frames():
    # two 4 x 2 sub-frames at s = 2: N = 8
    a = np.zeros((2, 4, 4), dtype=np.uint8)
    b = np.zeros((2, 4, 4), dtype=np.uint8)
    a[:, :2, 0] = 255                                 # left block of a: red 4 x 255
    b[0, 0, 0] = 3                                    # left block of b: red 3
    a[:, 2:, 2] = 10                                  # right block: blue 4 x 10 + 4 x 11
    b[:, 2:, 2] = 11
    out = blur_reduce([a, b], 2)
    # R: (1023 + 4) // 8 = 128; B: (84 + 4) // 8 = 11
    assert out.tolist() == [[[128, 0, 0, 255], [0, 0, 11, 255]]]
    assert blur_reduce([a[..., :3], b[..., :3]], 2, channels=3).tolist() == [[[128, 0, 0], [0, 0, 11]]]


def test_blur_reduce_equals_float_mean_rounded_half_up():
    rng = np.random.default_rng(11)
    for s in (1, 2, 3, 4):
        for n in (1, 2, 3, 5, 16):
            f = rng.integers(0, 256, size=(n, 3 * s, 7 * s, 4), dtype=np.uint8)
            mean = f[..., :3].astype(np.float64).reshape(n, 3, s, 7, s, 3).mean(axis=(0, 2, 4))
            assert np.array_equal(blur_reduce(list(f), s)[:, :, :3], np.floor(mean + 0.5).astype(np.uint8)), (s, n)


def test_blur_reduce_of_one_frame_is_box_reduce():
    rng = np.random.default_rng(12)
    for s in (1, 2, 3, 4):
        f = rng.integers(0, 256, size=(5 * s, 9 * s, 4), dtype=np.uint8)
        for ch in (3, 4):
            assert np.array_equal(blur_reduce([f], s, ch), box_reduce(f, s, ch))


def test_identical_cameras_collapse_to_the_plain_frame():
    """n copies of one sub-frame give box_reduce of it, for every s <= 4, n <= 16 and every possible block sum."""
    for s in (1, 2, 3, 4):
        q = s * s
        total = np.arange(255 * q + 1, dtype=np.int64)
        plain = (total + q // 2) // q
        for n in range(1, 17):
            assert np.array_equal((n * total + (n * q) // 2) // (n * q), plain), (s, n)
    rng = np.random.default_rng(13)
    f = rng.integers(0, 256, size=(2 * 3, 3 * 3, 4), dtype=np.uint8)
    assert np.array_equal(blur_reduce([f] * 16, 3), box_reduce(f, 3))


def test_blur_cameras_hand_worked():
    cams = blur_cameras((0.0, 1.0, 2.0, 0.5, 1.0), (4.0, 1.0, 0.0, 1.5, 1.0), 0.5, 4)
    assert cams[0] == (0.0, 1.0, 2.0, 0.5, 1.0)       # t = 0: this frame's camera
    assert cams[2] == (1.0, 1.0, 1.5, 0.75, 1.0)      # t = 0.25
    assert len(cams) == 4 and cams[3][0] == 1.5       # t = 0.375: the shutter closes before the next frame


def _camera_layout():
    """sizeof(hmrm_camera) and the offsets of its fields as a C compiler sees include/hmrm.h."""
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "hmrm.h"\nint main(void) { printf("%zu %zu %zu %zu\\n", '
           "sizeof(hmrm_camera), offsetof(hmrm_camera, cam_pos), offsetof(hmrm_camera, hang), "
           "offsetof(hmrm_camera, vang)); return 0; }\n")
    with tempfile.TemporaryDirectory() as td:
        c, exe = os.path.join(td, "m.c"), os.path.join(td, "m")
        Path(c).write_text(src)
        subprocess.run(["cc", "-I", str(ROOT / "include"), "-o", exe, c], check=True)
        return [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]


def test_camera_layout_and_binding_mirror(hmrm):
    import ctypes as C

    size, pos, hang, vang = _camera_layout()
    assert (size, pos, hang, vang) == (40, 0, 24, 32)
    cam = hmrm.Camera
    assert C.sizeof(cam) == size
    assert (cam.cam_pos.offset, cam.hang.offset, cam.vang.offset) == (pos, hang, vang)


def test_binding_rejects_malformed_cameras_before_the_library(hmrm):
    # shape errors are found in Python; a Renderer (and so a GPU) is not needed to see them
    r = hmrm.Renderer.__new__(hmrm.Renderer)
    two = ((0.0, 0.0), 0.0, 0.0)
    four = ((0.0, 0.0, 0.0, 0.0), 0.0, 0.0)
    # five 2-component positions are 20 numbers, five 4-component ones 30: neither may pass as 4 or 6 other cameras
    for bad in (np.zeros((2, 4)), np.zeros(5), [two], [two] * 5, [four] * 5, [((0.0, 0.0, 0.0), 0.0, 0.0), two]):
        with pytest.raises(ValueError):
            r.set_motion_blur(bad)


@pytest.mark.parametrize("args", [
    ["--script", "frames.txt", "--motion-blur", "0"],
    ["--script", "frames.txt", "--motion-blur", "17"],
    ["--script", "frames.txt", "--motion-blur", "-1"],
    ["--script", "frames.txt", "--motion-blur", "two"],
    ["--script", "frames.txt", "--motion-blur"],
    ["--headless", "o.png", "--motion-blur", "4"],
    ["--headless", "o.png", "--script", "frames.txt", "--motion-blur", "4"],
    ["--motion-blur", "4", "--parse-only"],
    ["--script", "frames.txt", "--shutter", "0.5"],
    ["--script", "frames.txt", "--motion-blur", "4", "--shutter", "0"],
    ["--script", "frames.txt", "--motion-blur", "4", "--shutter", "1.5"],
    ["--script", "frames.txt", "--motion-blur", "4", "--shutter", "-0.25"],
    ["--script", "frames.txt", "--motion-blur", "4", "--shutter", "half"],
    ["--script", "frames.txt", "--motion-blur", "4", "--shutter", "nan"],
    ["--script", "frames.txt", "--video", "v.y4m", "--motion-blur", "4", "--shutter"],
])
def test_hmap_motion_blur_usage_refusals(hmrm, args, tmp_path):
    assert HMAP.exists(), "hmap host binary was not built"
    (tmp_path / "config.txt").write_text("resolution 64 48\n")
    (tmp_path / "frames.txt").write_text("hang 10\n")
    res = subprocess.run([str(HMAP), "config.txt", *args], capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 1
    assert res.stderr.splitlines()[0] == "USAGE: hmap.exe path/to/config.txt"
    assert "--motion-blur 1..16 [--shutter F]" in res.stderr and res.stdout == ""
    assert not (tmp_path / "o.png").exists() and not (tmp_path / "v.y4m").exists()


@pytest.mark.parametrize("extra", [["--motion-blur", "1"], ["--motion-blur", "16", "--shutter", "1"],
                                   ["--motion-blur", "4", "--shutter", "0.125", "--video", "-"]])
def test_hmap_motion_blur_accepted_by_the_option_checks(hmrm, extra, tmp_path):
    (tmp_path / "config.txt").write_text("resolution 64 48\n")
    res = subprocess.run([str(HMAP), "config.txt", "--script", "frames.txt", *extra, "--parse-only"],
                         capture_output=True, text=True, cwd=str(tmp_path))
    # past the option checks: the config is read and echoed (it names no maps, so the grammar check then fails)
    assert "USAGE" not in res.stderr and "resolution 64 48" in res.stdout + res.stderr
