"""GPU: 4:2:0 video planes converted on the device (hmrm_render_yuv420_async, hmrm_convert_yuv420, and `hmap --video`
writing Y4M through them).  Every plane is compared byte for byte with the numpy model of tests/test_yuv420.py."""
import json
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import helpers as H
import scenes as S
from test_gpu_png import _write_scene
from test_png_encode import check_png
from test_yuv420 import BT601, BT709, i420, read_y4m, yuv420_model

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"
GOLDEN_NAMES = sorted(H.golden_frames().files)


def assert_planes(got, px, matrix, what=""):
    want = yuv420_model(px, matrix)
    for name, g, w in zip(("Y", "Cb", "Cr"), got, want):
        assert g.shape == w.shape, f"{what} {name}: shape {g.shape} != {w.shape}"
        bad = np.argwhere(g != w)
        assert bad.size == 0, f"{what} {name}: {len(bad)} bytes differ, first at {tuple(bad[0])}"


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_reference_frames_through_render_yuv420(hmrm, renderer, oracle, name):
    scene = S.SCENE_BY_NAME[name]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    want = H.golden_frames()[name]
    for fmt in (hmrm.PIXEL_RGBA8, hmrm.PIXEL_RGB8):
        for matrix in (hmrm.YUV_BT601, hmrm.YUV_BT709):
            got = renderer.render_yuv420(H.product_frame(hmrm, renderer, scene, pixel_format=fmt), matrix=matrix)
            assert_planes(got, want, matrix, f"{name} format {fmt} matrix {matrix}")


def _case(kind, h, w, ch, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, size=(h, w, ch), dtype=np.uint8)
    if kind == "constant":
        return np.full((h, w, ch), (201, 17, 90, 255)[:ch], dtype=np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "grey":
        v = ((xx * 3 + yy * 5) % 256).astype(np.uint8)
        return np.repeat(v[:, :, None], ch, axis=2)
    return np.stack([(xx * 7 + k * 60) % 256 if k % 2 == 0 else (yy * 3 + xx // 5) % 256 for k in range(ch)],
                    axis=2).astype(np.uint8)


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("h,w", [(1, 1), (1, 2), (2, 1), (3, 5), (181, 243), (8, 8200), (4320, 7680)])
def test_convert_yuv420_shapes_and_content(hmrm, renderer, h, w, ch):
    for kind in ("noise", "constant", "grey", "gradient"):
        px = _case(kind, h, w, ch, seed=h * 7 + w + ch)
        for matrix in (hmrm.YUV_BT601, hmrm.YUV_BT709):
            got = renderer.convert_yuv420(px, matrix)
            assert_planes(got, px, matrix, f"{kind} {h}x{w}x{ch} matrix {matrix}")
            if kind == "grey":
                assert (got[1] == 128).all() and (got[2] == 128).all()


def _flythrough(hmrm, renderer, oracle, n):
    scene = dict(S.SCENE_BY_NAME["persp_basic"])
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    return scene, [H.product_frame(hmrm, renderer, dict(scene, pos=(-0.6 + 0.05 * i, 0.6, 3.2 - 0.1 * i),
                                                        hang_deg=-45.0 - 7.0 * i)) for i in range(n)]


def _split(buf, w, h):
    """I420 bytes -> (Y, Cb, Cr)"""
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return (buf[:w * h].reshape(h, w), buf[w * h:w * h + cw * ch].reshape(ch, cw),
            buf[w * h + cw * ch:w * h + 2 * cw * ch].reshape(ch, cw))


def test_streaming_four_frames_in_flight(hmrm, renderer, oracle):
    scene, frames = _flythrough(hmrm, renderer, oracle, 7)
    w, h = scene["width"], scene["height"]
    want = [renderer.render(f).copy() for f in frames]
    assert len({H.sha(x) for x in want}) == len(want)
    bufs = [hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),)) for _ in range(4)]
    pending = []
    for i, f in enumerate(frames):
        if len(pending) == 4:
            renderer.wait_pending(3)
            j = pending.pop(0)
            assert_planes(_split(bufs[j % 4], w, h), want[j], BT709, f"frame {j}")
        renderer.render_yuv420_async(f, bufs[i % 4], BT709)
        pending.append(i)
    renderer.wait()
    for j in pending:
        assert_planes(_split(bufs[j % 4], w, h), want[j], BT709, f"frame {j}")


def test_yuv_and_png_frames_interleaved_in_flight(hmrm, renderer, oracle):
    scene, frames = _flythrough(hmrm, renderer, oracle, 8)
    w, h = scene["width"], scene["height"]
    want = [renderer.render(f).copy() for f in frames]
    yuv = [hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),)) for _ in range(4)]
    png = [hmrm.pinned_empty((hmrm.png_bound(w, h, 4),)) for _ in range(4)]
    sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]

    def check(j):
        if j % 2 == 0:
            assert_planes(_split(yuv[j % 4], w, h), want[j], BT601, f"frame {j}")
        else:
            data = png[j % 4][:int(sizes[j % 4][0])].tobytes()
            assert np.array_equal(check_png(data)[0], want[j]), f"frame {j}"

    pending = []
    for i, f in enumerate(frames):
        if len(pending) == 4:
            renderer.wait_pending(3)
            check(pending.pop(0))
        if i % 2 == 0:
            renderer.render_yuv420_async(f, yuv[i % 4], BT601)
        else:
            renderer.render_png_async(f, png[i % 4], sizes[i % 4])
        pending.append(i)
    renderer.wait()
    for j in pending:
        check(j)


def test_render_yuv420_into_cuda_tensor(hmrm, renderer, oracle):
    import torch

    scene = S.SCENE_BY_NAME["spher_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    f = H.product_frame(hmrm, renderer, scene)
    w, h = scene["width"], scene["height"]
    n = hmrm.yuv420_bytes(w, h)
    out = torch.zeros(n + 3, dtype=torch.uint8, device="cuda:0")
    renderer.render_yuv420_async(f, out.data_ptr() + 3, BT709, capacity=n)        # an unaligned destination
    renderer.wait()
    want = H.golden_frames()["spher_basic"]
    assert_planes(_split(out[3:].cpu().numpy(), w, h), want, BT709, "unaligned tensor")
    assert int(out[:3].sum()) == 0
    # a tensor reports its own size: one byte short is refused, not overrun
    with pytest.raises(hmrm.HmrmError):
        renderer.render_yuv420_async(f, out[:n - 1], BT709)
    with pytest.raises(ValueError):
        renderer.render_yuv420_async(f, out.data_ptr(), BT709)         # a raw address without its capacity
    exact = torch.empty(n, dtype=torch.uint8, device="cuda:0")
    renderer.render_yuv420_async(f, exact, BT601)
    renderer.wait()
    assert_planes(_split(exact.cpu().numpy(), w, h), want, BT601, "tensor")


def test_refusals(hmrm, renderer, oracle):
    import ctypes as C

    scene = S.SCENE_BY_NAME["persp_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    lib = hmrm.load_library()
    w, h = scene["width"], scene["height"]
    n = hmrm.yuv420_bytes(w, h)
    pinned = hmrm.pinned_empty((n,))
    pageable = np.zeros(n, dtype=np.uint8)

    def call(frame, out=pinned, cap=n, matrix=BT709):
        return lib.hmrm_render_yuv420_async(renderer._h, C.byref(frame), matrix, out.ctypes.data, cap)

    f = H.product_frame(hmrm, renderer, scene)
    assert call(f, cap=n - 1) == 1
    assert call(f, out=pageable) == 1
    assert lib.hmrm_render_yuv420_async(renderer._h, C.byref(f), BT709, None, n) == 1
    assert call(f, matrix=2) == 1 and call(f, matrix=-1) == 1
    assert call(H.product_frame(hmrm, renderer, scene, cycle_period=3)) == 1
    assert call(H.product_frame(hmrm, renderer, scene, band_count=2, band_index=0)) == 1
    assert call(H.product_frame(hmrm, renderer, scene, row_begin=0, row_end=h // 2)) == 1
    assert call(H.product_frame(hmrm, renderer, scene, row_begin=4, row_end=h)) == 1
    assert call(H.product_frame(hmrm, renderer, scene, flags=hmrm.FLAG_STEP_INDEX)) == 1
    assert call(H.product_frame(hmrm, renderer, scene, flags=hmrm.FLAG_RAY_DUMP)) == 1
    px = np.zeros((10, 10, 4), dtype=np.uint8)
    m = hmrm.yuv420_bytes(10, 10)

    def conv(ch=4, matrix=BT709, out=pinned, cap=m, width=10, height=10):
        return lib.hmrm_convert_yuv420(renderer._h, px.ctypes.data, width, height, ch, matrix, out.ctypes.data, cap)

    assert conv(ch=2) == 1 and conv(ch=5) == 1 and conv(ch=1) == 1
    assert conv(matrix=7) == 1
    assert conv(cap=m - 1) == 1
    assert conv(out=pageable) == 1
    assert conv(width=0) == 1 and conv(height=65537) == 1
    assert lib.hmrm_convert_yuv420(renderer._h, None, 10, 10, 4, BT709, pinned.ctypes.data, m) == 1
    # the context still works after the refusals
    assert_planes(renderer.render_yuv420(f, matrix=BT709), H.golden_frames()["persp_basic"], BT709, "after refusals")
    assert conv() == 0


# ---- hmap --video ----
def _video_scene(oracle, tmp_path, n, width=160, height=90):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=width, height=height)
    cfg = _write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6 + 0.07 * i, 0.6, 3.2), hang_deg=-45.0 - 5.0 * i) for i in range(n)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"]) for s in states))
    return scene, cfg, states


def _hmap(args, tmp_path, gpus=1, text=True):
    env = dict(os.environ, HMAP_DEVICE_LIST=",".join(["0"] * gpus))
    return subprocess.run([str(HMAP), "config.txt", "--script", "frames.txt", "--gpus", str(gpus), *args],
                          capture_output=True, text=text, cwd=str(tmp_path), env=env)


def _want_frames(oracle, scene, states, matrix):
    maps = H.load_scene_maps(scene, oracle)
    return [i420(yuv420_model(H.oracle_render_scene(oracle, dict(scene, **s), maps)[0], matrix)) for s in states]


def test_hmap_video_over_several_devices_equals_oracle(hmrm, oracle, tmp_path):
    scene, cfg, states = _video_scene(oracle, tmp_path, 11)
    res = _hmap(["--video", "out.y4m", "--stats-json", "stats.json"], tmp_path, gpus=3)
    assert res.returncode == 0, res.stderr
    data = (tmp_path / "out.y4m").read_bytes()
    assert data.startswith(b"YUV4MPEG2 W160 H90 F30:1 Ip A1:1 C420jpeg XCOLORRANGE=LIMITED\n")
    header, frames = read_y4m(data)
    assert (header["W"], header["H"], header["C"], header["X"]) == ("160", "90", "420jpeg", ["COLORRANGE=LIMITED"])
    want = _want_frames(oracle, scene, states, BT709)
    assert len(frames) == len(want) == 11
    for i, (g, w) in enumerate(zip(frames, want)):
        assert g == w, f"frame {i}"
    assert res.stdout.rstrip().endswith("Saved video at out.y4m (11 frames)")
    assert "Saved screenshot" not in res.stdout
    st = json.loads((tmp_path / "stats.json").read_text())
    assert st["frames"] == 11 and st["video_bytes"] == len(data)


def test_hmap_video_to_stdout_equals_file(hmrm, oracle, tmp_path):
    _video_scene(oracle, tmp_path, 5)
    to_file = _hmap(["--video", "out.y4m"], tmp_path, gpus=2, text=False)
    assert to_file.returncode == 0, to_file.stderr
    to_pipe = _hmap(["--video", "-"], tmp_path, gpus=2, text=False)
    assert to_pipe.returncode == 0, to_pipe.stderr
    assert to_pipe.stdout == (tmp_path / "out.y4m").read_bytes()
    # the config echo and the messages went to stderr instead of stdout
    echo = to_file.stdout.decode().replace("Saved video at out.y4m (5 frames)\n", "")
    assert echo.strip() and echo in to_pipe.stderr.decode()
    assert "Saved video at - (5 frames)" in to_pipe.stderr.decode()


def test_hmap_video_fps_and_bt601(hmrm, oracle, tmp_path):
    scene, cfg, states = _video_scene(oracle, tmp_path, 4, width=99, height=37)
    res = _hmap(["--video", "out.y4m", "--fps", "24", "--video-matrix", "bt601"], tmp_path)
    assert res.returncode == 0, res.stderr
    data = (tmp_path / "out.y4m").read_bytes()
    assert data.startswith(b"YUV4MPEG2 W99 H37 F24:1 Ip A1:1 C420jpeg XCOLORRANGE=LIMITED\n")
    _, frames = read_y4m(data)
    assert frames == _want_frames(oracle, scene, states, BT601)


def test_hmap_video_resolution_change_keeps_earlier_frames(hmrm, oracle, tmp_path):
    scene, cfg, states = _video_scene(oracle, tmp_path, 6)
    lines = (tmp_path / "frames.txt").read_text().splitlines()
    lines[4] = "resolution 120 90 " + lines[4]
    (tmp_path / "frames.txt").write_text("\n".join(lines) + "\n")
    res = _hmap(["--video", "out.y4m"], tmp_path, gpus=2)
    assert res.returncode == 1
    assert "frame 4" in res.stderr and "resolution" in res.stderr
    header, frames = read_y4m((tmp_path / "out.y4m").read_bytes())
    assert (header["W"], header["H"]) == ("160", "90")
    assert frames == _want_frames(oracle, scene, states[:4], BT709)


def test_hmap_stats_json_has_video_bytes_only_with_video(hmrm, oracle, tmp_path):
    _video_scene(oracle, tmp_path, 3)
    res = _hmap(["--video", "v.y4m", "--stats-json", "with.json"], tmp_path)
    assert res.returncode == 0, res.stderr
    assert json.loads((tmp_path / "with.json").read_text())["video_bytes"] == (tmp_path / "v.y4m").stat().st_size
    res = _hmap(["--out-prefix", "p_", "--stats-json", "without.json"], tmp_path)
    assert res.returncode == 0, res.stderr
    st = json.loads((tmp_path / "without.json").read_text())
    assert "video_bytes" not in st and list(st)[-1] == "png_bytes"
