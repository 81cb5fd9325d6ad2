"""GPU: supersampled frames (HMRM_FLAG_SUPERSAMPLE, kernel K5) through every path: hmrm_render, the frame ring with raw,
PNG and YUV outputs, hmrm_render_device, the statistics, the refusals and `hmap --supersample`.  Every expected pixel is
the numpy box filter (tests/test_supersample.py) of the CPU oracle's frame at sW x sH; nothing the device computed feeds
an expectation."""
import ctypes as C
import functools
import io
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
from test_supersample import box_reduce
from test_yuv420 import BT709, i420, read_y4m, yuv420_model

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"


@functools.lru_cache(maxsize=None)
def _maps(oracle, name):
    return H.load_scene_maps(S.SCENE_BY_NAME[name], oracle)


def _sub(oracle, scene, s):
    """The oracle's frame of `scene` at s times its size, and its statistics."""
    big = dict(scene, width=scene["width"] * s, height=scene["height"] * s)
    fb, _, st = H.oracle_render_scene(oracle, big, _maps(oracle, scene["name"]))
    return fb, st


def expected(oracle, scene, s, channels=4):
    return box_reduce(_sub(oracle, scene, s)[0], s, channels)


def _frame(hmrm, renderer, scene, s, **extra):
    return H.product_frame(hmrm, renderer, scene, flags=hmrm.supersample_flag(s) | extra.pop("flags", 0), **extra)


def _configure(renderer, oracle, name):
    H.configure(renderer, S.SCENE_BY_NAME[name], _maps(oracle, name))


def _assert_same(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = np.argwhere((got != want).any(axis=-1))
    assert bad.size == 0, f"{what}: {len(bad)} pixels differ, first at {tuple(bad[0])}"


# ---- 1. every scene, every projection, s = 2, 3, 4, RGBA8 and RGB8 ----
@pytest.mark.parametrize("scene", S.SCENES, ids=lambda s: s["name"])
def test_render_equals_box_filter_of_oracle(hmrm, renderer, oracle, scene):
    _configure(renderer, oracle, scene["name"])
    for s in (2, 3, 4):
        want = expected(oracle, scene, s)
        for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
            got = renderer.render(_frame(hmrm, renderer, scene, s, pixel_format=fmt))
            _assert_same(got, want[:, :, :ch], f"{scene['name']} s={s} channels={ch}")


@pytest.mark.parametrize("w,h", [(2, 2), (3, 2), (5, 7), (13, 3), (161, 91)])
def test_small_and_odd_frames(hmrm, renderer, oracle, w, h):
    for name in ("persp_basic", "spher_basic", "ortho_basic"):
        scene = dict(S.SCENE_BY_NAME[name], width=w, height=h)
        _configure(renderer, oracle, name)
        for s in (2, 3, 4):
            want = expected(oracle, scene, s)
            for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
                got = renderer.render(_frame(hmrm, renderer, scene, s, pixel_format=fmt))
                _assert_same(got, want[:, :, :ch], f"{name} {w}x{h} s={s} channels={ch}")


# ---- 2. the 4K flythrough at s = 2 over the 16384^2 map: sampled rows against the oracle's sub-rows ----
def test_flythrough4k_s2_sampled_rows_match_oracle(hmrm, oracle):
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    wl = bench.WORKLOADS["flythrough4k"]
    W, Hh = wl["W"], wl["H"]
    c = bench.camera(wl, 7)
    r = hmrm.Renderer(0)
    try:
        r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
        r.synth_maps(wl["log2n"], bench.SEED)
        f = r.frame(projection=wl["projection"], screen_width=W, screen_height=Hh, cam_pos=c["pos"],
                    hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                    ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"], supersample=2)
        got = r.render(f).copy()
    finally:
        r.close()
    terrain = np.nonzero((got[:, :, :3] != 0).any(axis=(1, 2)))[0]
    assert terrain.size > 0
    first = int(terrain[0])
    rows = sorted({0, max(first - 1, 0), first, min(first + 1, Hh - 1), min(first + 20, Hh - 1), Hh // 2,
                   (3 * Hh) // 4, Hh - 1})
    of = oracle.make_frame(projection=wl["projection"], width=2 * W, height=2 * Hh, grid_width=bench.GRID_WIDTH,
                           step_dist=wl["step_dist"], min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT, **c)
    hits = 0
    for py in rows:
        ofb, _, ost = oracle.render_synth(of, wl["log2n"], bench.SEED, rows=(2 * py, 2 * py + 2), want_steps=False)
        _assert_same(got[py:py + 1], box_reduce(ofb[2 * py:2 * py + 2], 2), f"flythrough4k s=2 row {py}")
        hits += ost.surf_hits
    assert hits > 0


# ---- 3. PNG and 4. YUV at s = 2 ----
@pytest.mark.parametrize("name", ["persp_basic", "spher_wide", "defaults_grid"])
def test_render_png_s2_decodes_to_filtered_frame(hmrm, renderer, oracle, name):
    from PIL import Image

    scene = S.SCENE_BY_NAME[name]
    _configure(renderer, oracle, name)
    want = expected(oracle, scene, 2)
    for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
        data = renderer.render_png(_frame(hmrm, renderer, scene, 2, pixel_format=fmt))
        _assert_same(check_png(data)[0], want[:, :, :ch], f"{name} channels={ch} (checker)")
        _assert_same(np.asarray(Image.open(io.BytesIO(data))), want[:, :, :ch], f"{name} channels={ch} (PIL)")


@pytest.mark.parametrize("name", ["persp_basic", "ortho_fine", "defaults_grid"])
def test_render_yuv420_s2_equals_model_of_filtered_frame(hmrm, renderer, oracle, name):
    scene = S.SCENE_BY_NAME[name]
    _configure(renderer, oracle, name)
    want = expected(oracle, scene, 2)
    for fmt in (hmrm.PIXEL_RGBA8, hmrm.PIXEL_RGB8):
        for matrix in (hmrm.YUV_BT601, hmrm.YUV_BT709):
            got = renderer.render_yuv420(_frame(hmrm, renderer, scene, 2, pixel_format=fmt), matrix=matrix)
            for plane, g, w in zip("Y Cb Cr".split(), got, yuv420_model(want, matrix)):
                assert np.array_equal(g, w), f"{name} format {fmt} matrix {matrix} plane {plane}"


# ---- 5. hmrm_render_device: supersampled frames back to back on one stream ----
def _cams(n):
    return [dict(pos=(-0.6 + 0.05 * i, 0.6, 3.2 - 0.1 * i), hang_deg=-45.0 - 7.0 * i) for i in range(n)]


def test_render_device_back_to_back_frames(hmrm, renderer, oracle):
    import torch

    base = dict(S.SCENE_BY_NAME["persp_basic"], width=161, height=90)
    _configure(renderer, oracle, "persp_basic")
    cams = _cams(7)
    ss = [2, 2, 2, 2, 2, 2, 3]                         # more frames than sub-frame scratches, no wait in between
    scenes = [dict(base, **c) for c in cams]
    want = [expected(oracle, sc, s) for sc, s in zip(scenes, ss)]
    w, h = base["width"], base["height"]
    outs = [torch.zeros(h * w * 4 + 3, dtype=torch.uint8, device="cuda:0") for _ in cams]
    for i, (sc, s) in enumerate(zip(scenes, ss)):
        off = 3 if i == 1 else 0                       # one unaligned destination
        renderer.render_device(_frame(hmrm, renderer, sc, s), outs[i].data_ptr() + off)
    renderer.wait()
    for i, o in enumerate(outs):
        off = 3 if i == 1 else 0
        got = o[off:off + h * w * 4].cpu().numpy().reshape(h, w, 4)
        _assert_same(got, want[i], f"frame {i} s={ss[i]}")
    # RGB8 into a tensor on a caller's stream
    st = torch.cuda.Stream()
    out = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:0")
    renderer.render_device(_frame(hmrm, renderer, scenes[0], 2, pixel_format=hmrm.PIXEL_RGB8), out, st.cuda_stream)
    st.synchronize()
    _assert_same(out.cpu().numpy(), want[0][:, :, :3], "RGB8 on a caller stream")


# ---- 6. four frames in flight through the ring: s = 1, 2, 4 with raw, PNG and YUV outputs ----
def test_ring_mixes_factors_and_outputs(hmrm, renderer, oracle):
    base = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    _configure(renderer, oracle, "persp_basic")
    n = 9
    scenes = [dict(base, **c) for c in _cams(n)]
    ss = [(1, 2, 4)[i % 3] for i in range(n)]
    kinds = [("raw", "png", "yuv", "png")[i % 4] for i in range(n)]
    want = [expected(oracle, sc, s) for sc, s in zip(scenes, ss)]
    w, h = base["width"], base["height"]
    raw = [hmrm.pinned_empty((h, w, 4)) for _ in range(4)]
    png = [hmrm.pinned_empty((hmrm.png_bound(w, h, 4),)) for _ in range(4)]
    sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]
    yuv = [hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),)) for _ in range(4)]

    def check(j):
        what = f"frame {j} s={ss[j]} {kinds[j]}"
        if kinds[j] == "raw":
            _assert_same(raw[j % 4], want[j], what)
        elif kinds[j] == "png":
            _assert_same(check_png(png[j % 4][:int(sizes[j % 4][0])].tobytes())[0], want[j], what)
        else:
            assert i420(yuv420_model(want[j], BT709)) == yuv[j % 4].tobytes(), what

    pending = []
    for i, sc in enumerate(scenes):
        if len(pending) == 4:
            renderer.wait_pending(3)
            check(pending.pop(0))
        f = _frame(hmrm, renderer, sc, ss[i])
        if kinds[i] == "raw":
            renderer.render_async(f, raw[i % 4])
        elif kinds[i] == "png":
            renderer.render_png_async(f, png[i % 4], sizes[i % 4])
        else:
            renderer.render_yuv420_async(f, yuv[i % 4], BT709)
        pending.append(i)
    renderer.wait()
    for j in pending:
        check(j)


# ---- 7. statistics describe the sub-frame render ----
@pytest.mark.parametrize("name", ["persp_graze", "spher_fine", "ortho_basic"])
def test_stats_describe_the_sub_frame(hmrm, renderer, oracle, name):
    scene = S.SCENE_BY_NAME[name]
    _configure(renderer, oracle, name)
    for s in (2, 3):
        _, ost = _sub(oracle, scene, s)
        renderer.render(_frame(hmrm, renderer, scene, s, flags=hmrm.FLAG_STATS))
        st = renderer.stats()
        assert st.rays == s * s * scene["width"] * scene["height"]
        assert (st.steps, st.surf_hits, st.box_hits) == (ost.steps, ost.surf_hits, ost.box_hits), f"{name} s={s}"
        assert st.status == 0 and st.kernel_ms > 0.0


# ---- 8. refusals ----
def test_refusals_leave_the_context_usable(hmrm, renderer, oracle):
    import torch

    scene = S.SCENE_BY_NAME["persp_basic"]
    _configure(renderer, oracle, "persp_basic")
    lib = hmrm.load_library()
    w, h = scene["width"], scene["height"]
    host = hmrm.pinned_empty((h, w, 4))
    png = hmrm.pinned_empty((hmrm.png_bound(w, h, 4),))
    size = hmrm.pinned_empty((1,), dtype=np.uint64)
    yuv = hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),))
    dev = torch.zeros(h * w * 4 + 256, dtype=torch.uint8, device="cuda:0")
    stage = torch.zeros(h * w * 4, dtype=torch.uint8, device="cuda:0")

    def calls(f):
        fp = C.byref(f)
        return [lib.hmrm_render(renderer._h, fp, host.ctypes.data),
                lib.hmrm_render_async(renderer._h, fp, host.ctypes.data),
                lib.hmrm_render_device(renderer._h, fp, dev.data_ptr(), None),
                lib.hmrm_render_png_async(renderer._h, fp, png.ctypes.data, png.nbytes, size.ctypes.data),
                lib.hmrm_render_yuv420_async(renderer._h, fp, BT709, yuv.ctypes.data, yuv.nbytes)]

    def frame(**kw):
        return H.product_frame(hmrm, renderer, scene, **kw)

    s2 = hmrm.supersample_flag(2)
    bad = {
        "field 4 (s = 5)": frame(flags=4 << hmrm.FLAG_SUPERSAMPLE_SHIFT),
        "field 15": frame(flags=hmrm.FLAG_SUPERSAMPLE_MASK),
        "sW > 65536": frame(flags=hmrm.supersample_flag(4), screen_width=16385, screen_height=8),
        "sH > 65536": frame(flags=s2, screen_width=8, screen_height=32769),
        "cycle_period 3": frame(flags=s2, cycle_period=3),
        "band_count 2": frame(flags=s2, band_count=2, band_index=0),
        "row band top": frame(flags=s2, row_begin=0, row_end=h // 2),
        "row band bottom": frame(flags=s2, row_begin=4, row_end=h),
        "step index": frame(flags=s2 | hmrm.FLAG_STEP_INDEX),
        "ray dump": frame(flags=s2 | hmrm.FLAG_RAY_DUMP),
    }
    for what, f in bad.items():
        assert calls(f) == [1] * 5, what
        assert lib.hmrm_last_error(renderer._h)
    f2 = frame(flags=s2)
    ctrl = torch.zeros(256, dtype=torch.uint8, device="cuda:0")
    assert lib.hmrm_render_peer(renderer._h, C.byref(f2), dev.data_ptr(), ctrl.data_ptr(), 1, None) == 1
    assert b"supersampling" in lib.hmrm_last_error(renderer._h)
    assert lib.hmrm_render_peer_staged(renderer._h, C.byref(f2), stage.data_ptr(), dev.data_ptr(), ctrl.data_ptr(), 1,
                                       None) == 1
    assert int(ctrl.sum()) == 0 and int(dev.sum()) == 0
    # the context still works, supersampled and not
    want = expected(oracle, scene, 2)
    _assert_same(renderer.render(f2), want, "s=2 after refusals")
    _assert_same(renderer.render(frame()), H.golden_frames()["persp_basic"], "s=1 after refusals")


# ---- 9. hmap --headless --supersample 2 ----
def test_hmap_headless_supersample(hmrm, oracle, tmp_path):
    scene = S.SCENE_BY_NAME["persp_basic"]
    cfg = _write_scene(oracle, scene, tmp_path)
    out, stats = tmp_path / "out.png", tmp_path / "stats.json"
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--supersample", "2", "--stats-json", str(stats)],
                         capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr
    _assert_same(check_png(out.read_bytes())[0], expected(oracle, scene, 2), "hmap --headless --supersample 2")
    st = json.loads(stats.read_text())
    assert st["supersample"] == 2 and st["rays"] == 4 * scene["width"] * scene["height"]
    # without the option the statistics do not name it
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--stats-json", str(stats)], capture_output=True,
                         text=True, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr
    assert "supersample" not in json.loads(stats.read_text())
    _assert_same(check_png(out.read_bytes())[0], H.golden_frames()["persp_basic"], "hmap --headless")


# ---- 10. hmap --script --video - --supersample 2 over several contexts ----
def test_hmap_video_supersample_over_several_devices(hmrm, oracle, tmp_path):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    _write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6 + 0.07 * i, 0.6, 3.2), hang_deg=-45.0 - 5.0 * i) for i in range(7)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"]) for s in states))
    env = dict(os.environ, HMAP_DEVICE_LIST="0,0,0")
    res = subprocess.run([str(HMAP), "config.txt", "--script", "frames.txt", "--gpus", "3", "--video", "-",
                          "--supersample", "2", "--stats-json", "stats.json"], capture_output=True, cwd=str(tmp_path),
                         env=env)
    assert res.returncode == 0, res.stderr.decode()
    header, frames = read_y4m(res.stdout)
    assert (header["W"], header["H"]) == ("160", "90")
    want = [i420(yuv420_model(expected(oracle, dict(scene, **s), 2), BT709)) for s in states]
    assert len(frames) == len(want)
    for i, (g, w) in enumerate(zip(frames, want)):
        assert g == w, f"frame {i}"
    st = json.loads((tmp_path / "stats.json").read_text())
    assert st["supersample"] == 2 and st["video_bytes"] == len(res.stdout) and st["frames"] == len(states)
    assert st["rays"] == 4 * 160 * 90 * len(states)
