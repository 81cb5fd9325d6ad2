"""GPU: the `hmap` binary end to end (config file -> PNG) against the reference's frames."""
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest
from PIL import Image

import helpers as H
import scenes as S
from test_gpu_png import assert_equals_model

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"


def write_scene(oracle, scene, tmp_path):
    hm, cm = H.load_scene_maps(scene, oracle)
    oracle.write_png(tmp_path / "h.png", hm)
    oracle.write_png(tmp_path / "c.png", cm)
    cfg = tmp_path / "config.txt"
    # the reference's default cycle (47) stays in the file: headless frames are complete images regardless
    text = oracle.config_text(S.frame_kwargs(scene), "h.png", "c.png", lum=scene["lum"]).replace("cycle 1\n", "")
    cfg.write_text(text)
    return cfg


@pytest.mark.parametrize("name", ["persp_basic", "spher_wide", "ortho_fine", "noise_lum_neg", "min_height_twice",
                                  "alpha_zero_centre"])
def test_headless_png_matches_reference_frame(hmrm, oracle, name, tmp_path):
    scene = S.SCENE_BY_NAME[name]
    cfg = write_scene(oracle, scene, tmp_path)
    out = tmp_path / "out.png"
    stats = tmp_path / "stats.json"
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--projection", str(scene["projection"]),
                          "--stats-json", str(stats)], capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr
    assert f"Saved screenshot at {out}" in res.stdout            # main/hmap.cpp:166
    got = np.asarray(Image.open(out).convert("RGBA"))
    assert np.array_equal(got, H.golden_frames()[name])
    assert_equals_model(out.read_bytes(), H.golden_frames()[name], name)
    meta = H.golden_meta()[name]
    st = json.loads(stats.read_text())
    assert (st["rays"], st["box_hits"], st["surf_hits"], st["steps"]) == (
        meta["rays"], meta["box_hits"], meta["surf_hits"], meta["steps"])


def test_script_recording_matches_oracle_per_frame(hmrm, oracle, tmp_path):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    cfg = write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6, 0.6, 3.2), hang_deg=-45.0), dict(pos=(-0.2, 0.9, 3.0), hang_deg=-60.0),
              dict(pos=(0.4, 1.0, 2.8), hang_deg=-80.0), dict(pos=(0.4, 1.0, 2.8), hang_deg=-80.0, max_height=1.5)]
    lines = ["pos %r %r %r hang %r" % (*s["pos"], s["hang_deg"]) + (" max_height %r" % s["max_height"] if "max_height" in s else "")
             for s in states]
    (tmp_path / "frames.txt").write_text("\n".join(lines) + "\n")
    res = subprocess.run([str(HMAP), str(cfg), "--script", "frames.txt", "--out-prefix", str(tmp_path / "f_")],
                         capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr
    assert res.stdout.rstrip().endswith("Done recording.")          # main/hmap.cpp:1142
    maps = H.load_scene_maps(scene, oracle)
    for i, s in enumerate(states):
        want, _, _ = H.oracle_render_scene(oracle, dict(scene, **s), maps)
        got = np.asarray(Image.open(tmp_path / f"f_{i}.png").convert("RGBA"))
        assert np.array_equal(got, want), f"frame {i}"
        assert_equals_model((tmp_path / f"f_{i}.png").read_bytes(), want, f"frame {i}")


def test_brute_and_fp64_flags(hmrm, oracle, tmp_path):
    scene = S.SCENE_BY_NAME["spher_basic"]
    cfg = write_scene(oracle, scene, tmp_path)
    out = tmp_path / "b.png"
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--projection", "2", "--traversal", "brute",
                          "--precision", "fp64"], capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr
    assert np.array_equal(np.asarray(Image.open(out).convert("RGBA")), H.golden_frames()["spher_basic"])
    assert_equals_model(out.read_bytes(), H.golden_frames()["spher_basic"], "brute fp64")


@pytest.mark.parametrize("name,gpus", [("persp_basic", 2), ("spher_wide", 3), ("ortho_fine", 5)])
def test_one_frame_over_several_devices_equals_the_reference_frame(hmrm, oracle, name, gpus, tmp_path):
    """--gpus N on one frame: its tile rows are dealt round-robin to N contexts, each of which copies its own rows
    into the one host frame.  HMAP_DEVICE_LIST lets the contexts share cuda:0 on a one-GPU box."""
    import os

    scene = S.SCENE_BY_NAME[name]
    cfg = write_scene(oracle, scene, tmp_path)
    out = tmp_path / "out.png"
    stats = tmp_path / "stats.json"
    env = dict(os.environ, HMAP_DEVICE_LIST=",".join(["0"] * gpus))
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--projection", str(scene["projection"]),
                          "--gpus", str(gpus), "--stats-json", str(stats)], capture_output=True, text=True,
                         cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr
    assert np.array_equal(np.asarray(Image.open(out).convert("RGBA")), H.golden_frames()[name])
    assert_equals_model(out.read_bytes(), H.golden_frames()[name], f"{name} over {gpus} devices")
    meta = H.golden_meta()[name]
    st = json.loads(stats.read_text())
    assert (st["rays"], st["box_hits"], st["surf_hits"], st["steps"]) == (
        meta["rays"], meta["box_hits"], meta["surf_hits"], meta["steps"])


def test_recording_over_several_devices(hmrm, oracle, tmp_path):
    import os

    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    cfg = write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6 + 0.1 * i, 0.6, 3.2), hang_deg=-45.0 - 3.0 * i) for i in range(7)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"]) for s in states))
    env = dict(os.environ, HMAP_DEVICE_LIST="0,0,0")
    res = subprocess.run([str(HMAP), str(cfg), "--script", "frames.txt", "--out-prefix", str(tmp_path / "f_"), "--gpus", "3"],
                         capture_output=True, text=True, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr
    maps = H.load_scene_maps(scene, oracle)
    for i, s in enumerate(states):
        want, _, _ = H.oracle_render_scene(oracle, dict(scene, **s), maps)
        got = np.asarray(Image.open(tmp_path / f"f_{i}.png").convert("RGBA"))
        assert np.array_equal(got, want), f"frame {i}"
        assert_equals_model((tmp_path / f"f_{i}.png").read_bytes(), want, f"frame {i}")
