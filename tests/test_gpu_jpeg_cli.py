"""GPU: `hmap --jpeg Q`: JPEG stills (--headless, --script with --out-prefix or --record) and Motion-JPEG video
(--video with --jpeg), over one or several devices.  Every file must equal Pillow's encoding of the oracle's frame."""
import io
import json
import os
import subprocess
from pathlib import Path

import pytest
from PIL import Image

import helpers as H
import scenes as S
from test_gpu_png import _write_scene
from test_jpeg_model import pil_jpeg

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"


def _run(args, tmp_path, gpus=1, text=True):
    env = dict(os.environ, HMAP_DEVICE_LIST=",".join(["0"] * gpus))
    return subprocess.run([str(HMAP), "config.txt", "--gpus", str(gpus), *args], capture_output=True, text=text,
                          cwd=str(tmp_path), env=env)


def _script_scene(oracle, tmp_path, n):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    _write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6 + 0.07 * i, 0.6, 3.2), hang_deg=-45.0 - 5.0 * i) for i in range(n)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"]) for s in states))
    maps = H.load_scene_maps(scene, oracle)
    return [H.oracle_render_scene(oracle, dict(scene, **s), maps)[0] for s in states]


@pytest.mark.parametrize("gpus", [1, 2])
def test_headless_jpeg(hmrm, oracle, gpus, tmp_path):
    """One device renders and encodes; two deal the frame's tile rows and device 0 encodes the assembled frame."""
    scene = S.SCENE_BY_NAME["ortho_basic"]
    _write_scene(oracle, scene, tmp_path)
    want = H.golden_frames()["ortho_basic"]
    for q, chroma, s420 in ((90, "420", True), (60, "444", False)):
        res = _run(["--headless", "out.jpg", "--projection", "3", "--jpeg", str(q), "--jpeg-chroma", chroma,
                    "--stats-json", "stats.json"], tmp_path, gpus)
        assert res.returncode == 0, res.stderr
        data = (tmp_path / "out.jpg").read_bytes()
        assert data == pil_jpeg(want, q, s420), f"q{q} {chroma}"
        st = json.loads((tmp_path / "stats.json").read_text())
        assert st["jpeg_bytes"] == len(data) and st["png_bytes"] == 0
        assert "Saved screenshot at out.jpg" in res.stdout


@pytest.mark.parametrize("gpus", [1, 2])
def test_script_out_prefix_and_record(hmrm, oracle, gpus, tmp_path):
    frames = _script_scene(oracle, tmp_path, 7)
    res = _run(["--script", "frames.txt", "--out-prefix", "s_", "--jpeg", "75", "--stats-json", "stats.json"], tmp_path,
               gpus)
    assert res.returncode == 0, res.stderr
    for i, px in enumerate(frames):
        assert (tmp_path / f"s_{i}.jpg").read_bytes() == pil_jpeg(px, 75, True), f"frame {i}"
    assert not list(tmp_path.glob("s_*.png"))
    st = json.loads((tmp_path / "stats.json").read_text())
    assert st["frames"] == 7 and st["jpeg_bytes"] == sum((tmp_path / f"s_{i}.jpg").stat().st_size for i in range(7))
    (tmp_path / "screenshots").mkdir()
    res = _run(["--script", "frames.txt", "--record", "--jpeg", "75"], tmp_path, gpus)
    assert res.returncode == 0, res.stderr
    assert res.stdout.rstrip().endswith("Done recording.")
    assert res.stdout.count("Saved screenshot at ") == 7
    files = sorted((tmp_path / "screenshots").glob("hmap_*.jpg"), key=lambda p: int(p.stem.rsplit("_", 1)[1]))
    assert len(files) == 7
    for i, p in enumerate(files):
        assert p.read_bytes() == pil_jpeg(frames[i], 75, True), f"frame {i}"


@pytest.mark.parametrize("gpus", [1, 3])
def test_motion_jpeg_video(hmrm, oracle, gpus, tmp_path):
    frames = _script_scene(oracle, tmp_path, 9)
    res = _run(["--script", "frames.txt", "--video", "-", "--jpeg", "75", "--stats-json", "stats.json"], tmp_path, gpus,
               text=False)
    assert res.returncode == 0, res.stderr
    want = [pil_jpeg(px, 75, True) for px in frames]
    assert res.stdout == b"".join(want)
    assert res.stdout.count(b"\xff\xd8\xff\xe0") == len(frames)
    # split at SOI / EOI: each piece is one frame's file
    pieces, pos = [], 0
    for w in want:
        end = pos + len(w)
        assert res.stdout[pos:pos + 2] == b"\xff\xd8" and res.stdout[end - 2:end] == b"\xff\xd9"
        pieces.append(res.stdout[pos:end])
        pos = end
    for p in pieces:
        assert Image.open(io.BytesIO(p)).size == (160, 90)
    assert b"Saved video at - (9 frames)" in res.stderr
    st = json.loads((tmp_path / "stats.json").read_text())
    assert st["video_bytes"] == len(res.stdout) == st["jpeg_bytes"]


def test_supersample_and_height_bits_16(hmrm, renderer, oracle, tmp_path):
    scene = S.SCENE_BY_NAME["persp_basic"]
    _write_scene(oracle, scene, tmp_path)
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    f = H.product_frame(hmrm, renderer, scene)
    f.flags = hmrm.supersample_flag(2)
    want = renderer.render(f).copy()
    res = _run(["--headless", "ss.jpg", "--jpeg", "85", "--supersample", "2"], tmp_path)
    assert res.returncode == 0, res.stderr
    assert (tmp_path / "ss.jpg").read_bytes() == pil_jpeg(want, 85, True)
    res = _run(["--headless", "h16.jpg", "--jpeg", "85", "--height-bits", "16"], tmp_path)
    assert res.returncode == 0, res.stderr
    im = Image.open(tmp_path / "h16.jpg")
    assert im.size == (scene["width"], scene["height"])
    raw = tmp_path / "h16.raw"
    dec = subprocess.run([str(HMAP), "--decode-image", str(tmp_path / "h16.jpg"), "4", str(raw)], capture_output=True,
                         text=True)
    assert dec.returncode == 0, dec.stderr
    assert raw.stat().st_size == scene["width"] * scene["height"] * 4


def test_option_refusals(hmrm, oracle, tmp_path):
    _script_scene(oracle, tmp_path, 2)
    for extra in (["--fps", "24"], ["--video-matrix", "bt601"]):
        res = _run(["--script", "frames.txt", "--video", "out.mjpg", "--jpeg", "75", *extra], tmp_path)
        assert res.returncode == 1 and "Motion-JPEG" in res.stderr, extra
        assert not (tmp_path / "out.mjpg").exists()
    res = _run(["--script", "frames.txt", "--out-prefix", "q_", "--jpeg", "0"], tmp_path)
    assert res.returncode == 1 and not list(tmp_path.glob("q_*"))
    # --jpeg-chroma only means something for JPEG files
    res = _run(["--script", "frames.txt", "--out-prefix", "c_", "--jpeg-chroma", "444"], tmp_path)
    assert res.returncode == 1 and "needs --jpeg" in res.stderr and not list(tmp_path.glob("c_*"))
