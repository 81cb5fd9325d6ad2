"""GPU: the interactive shell of `hmap` (host/hmap_sdl.cpp, -DHMAP_WITH_SDL) against the UNMODIFIED reference, both
linked with the same scripted fake SDL (oracle/shim) and driven by the same event script: keys, mouse look, wheel
zoom, WASD movement, console commands, projection switches, window resize, progressive `cycle` rendering.
Every frame both programs hand to SDL_UpdateTexture is compared byte for byte (events -> state -> frame parity,
including the reference's one-frame look/up lag, SURVEY.md D-6): with the reference's recorded frames and console
output (tests/golden/replays.json), and with the reference run now where oracle/_ref is built."""
import importlib.util
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import helpers as H
import scenes as S

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "heightmap-ray-marcher_b200"
SHIM = ROOT / "oracle" / "shim"


def build_shell(out_dir: Path) -> Path:
    obj = out_dir / "fake_sdl.o"
    subprocess.run(["g++", "-std=c++11", "-O2", "-c", "-I", str(SHIM), "-o", str(obj), str(SHIM / "fake_sdl.cpp")], check=True)
    spec = importlib.util.spec_from_file_location("hmrm_build", PKG / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build_hmap_fake_sdl(SHIM, obj, out_dir / "hmap_sdl")


@pytest.fixture(scope="module")
def shell_binary(hmrm, tmp_path_factory):
    return build_shell(tmp_path_factory.mktemp("hmap_sdl"))


EVENTS = """0 key 1
1 motion 40 -25
2 wheel 2
3 hold w 1
5 hold w 0
5 hold d 1
6 hold d 0
6 key 2
7 key backquote
7 text hang -60 pos -0.3 0.8 3.0 bg_color 20 40 60
7 key return
8 key 3
9 wheel -3
10 hold space 1
11 hold space 0
11 key 1
12 key backquote
12 text step_dist 0.02
12 key backspace
12 key backspace
12 text 11 max_height 2.0
12 key return
13 key 2 ctrl
14 hold a 1
"""
RESIZE_EVENTS = "0 key 2\n6 motion -30 10\n9 resize 200 120\n14 wheel 1\n"
# the reference's framebuf starts uninitialised (main/hmap.cpp:612, and again after a resize :699): with a 3-frame
# cycle, frames are compared once every phase has been drawn
RESIZE_COMPARED = list(range(3, 9)) + list(range(12, 18))


def write_inputs(oracle, tmp_path, config_extra, events) -> None:
    """Maps, config and event script of a shell run in tmp_path."""
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    hm, cm = H.load_scene_maps(scene, oracle)
    oracle.write_png(tmp_path / "h.png", hm)
    oracle.write_png(tmp_path / "c.png", cm)
    text = oracle.config_text(S.frame_kwargs(scene), "h.png", "c.png", lum=scene["lum"], extra="move 0.004 " + config_extra)
    (tmp_path / "config.txt").write_text(text)
    (tmp_path / "events.txt").write_text(events)


def run_shell(binary, tmp_path, frames):
    """-> (the RGBA8 frames `binary` hands to SDL_UpdateTexture, its stdout), inputs from write_inputs."""
    d = tmp_path / Path(binary).name
    d.mkdir()
    env = dict(os.environ, HMRM_FAKE_FRAMES=str(frames), HMRM_FAKE_EVENTS=str(tmp_path / "events.txt"),
               HMRM_FAKE_DUMP=str(d / "frame_"), HMRM_FAKE_PROJ="1")
    res = subprocess.run([str(binary), str(tmp_path / "config.txt")], cwd=str(tmp_path), env=env, capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    return [np.fromfile(d / f"frame_{i}.rgba", dtype=np.uint8) for i in range(frames)], res.stdout


def test_shell_frames_match_reference_under_scripted_events(oracle, shell_binary, tmp_path):
    write_inputs(oracle, tmp_path, "", EVENTS)
    ours, ours_out = run_shell(shell_binary, tmp_path, 16)
    rec = H.golden_replays()["shell_events"]
    differ = [i for i, f in enumerate(ours) if H.sha(f) != rec["frame_sha256"][i]]
    assert not differ, f"frames {differ} differ from the reference's"
    # the console echo (config grammar) is the same text on stdout
    assert ours_out == rec["stdout"]
    # the script really changed the picture from frame to frame
    assert sum(rec["frame_sha256"][i] != rec["frame_sha256"][i + 1] for i in range(15)) >= 8
    if oracle.REF_BIN.exists():
        ref, ref_out = run_shell(oracle.REF_BIN, tmp_path, 16)
        for i, (a, b) in enumerate(zip(ref, ours)):
            assert a.size == b.size, f"frame {i}: size {b.size} != {a.size}"
            assert np.array_equal(a, b), f"frame {i}: {int((a != b).reshape(-1, 4).any(axis=1).sum())} pixels differ"
        assert ours_out == ref_out


def test_shell_resize_and_progressive_cycle(oracle, shell_binary, tmp_path):
    write_inputs(oracle, tmp_path, "cycle 3", RESIZE_EVENTS)
    ours, _ = run_shell(shell_binary, tmp_path, 18)
    rec = H.golden_replays()["shell_resize_cycle"]
    for i in RESIZE_COMPARED:
        assert ours[i].size == rec["frame_size"][str(i)], f"frame {i}"
        assert H.sha(ours[i]) == rec["frame_sha256"][str(i)], f"frame {i}"
    assert rec["frame_size"]["8"] == 160 * 90 * 4 and rec["frame_size"]["12"] == 200 * 120 * 4
    if oracle.REF_BIN.exists():
        ref, _ = run_shell(oracle.REF_BIN, tmp_path, 18)
        for i in RESIZE_COMPARED:
            assert ref[i].size == ours[i].size
            assert np.array_equal(ref[i], ours[i]), f"frame {i}"
