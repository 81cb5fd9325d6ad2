"""GPU: motion-blurred frames (hmrm_set_motion_blur, kernel K5) through every path: hmrm_render, the frame ring with raw,
PNG, YUV and JPEG outputs, hmrm_render_device, the statistics, the refusals and `hmap --motion-blur`.  Every expected
pixel is blur_reduce (tests/test_motion_blur.py) of the CPU oracle's frames at the sub-frame cameras; nothing the device
computed feeds an expectation."""
import ctypes as C
import functools
import io
import json
import math
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import helpers as H
import jpeg_model as J
import scenes as S
from test_gpu_png import _write_scene, assert_equals_model
from test_motion_blur import blur_cameras, blur_reduce
from test_png_encode import check_png
from test_yuv420 import BT709, i420, read_y4m, yuv420_model

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"
PAIRS = [(n, s) for n in (1, 2, 3, 5, 16) for s in (1, 2, 3, 4)]


@pytest.fixture(autouse=True)
def _blur_off(renderer):
    """The session's renderer leaves every test without blur, whatever the test did."""
    yield
    renderer.set_motion_blur([])


@functools.lru_cache(maxsize=None)
def _maps(oracle, name):
    return H.load_scene_maps(S.SCENE_BY_NAME[name], oracle)


def _configure(renderer, oracle, name):
    H.configure(renderer, S.SCENE_BY_NAME[name], _maps(oracle, name))


def camera_of(oracle, scene):
    """(x, y, z, hang, vang) of a scene, angles in radians as the config grammar converts them."""
    return (*[float(v) for v in scene["pos"]], oracle.deg2rad(scene["hang_deg"]), oracle.deg2rad(scene["vang_deg"]))


def scene_cams(oracle, scene, n, step=1.0):
    """n sub-frame cameras moving away from the scene's camera: a few cells and a degree or so per sub-frame."""
    x, y, z, hang, vang = camera_of(oracle, scene)
    return [(x + 0.011 * step * j, y - 0.007 * step * j, z + 0.004 * step * j, hang + 0.013 * step * j,
             vang - 0.005 * step * j) for j in range(n)]


@functools.lru_cache(maxsize=None)
def _oracle_sub(oracle, key, cam, s):
    """The oracle's frame (and statistics) of scene `key` (name, width, height) at camera `cam`, s times its size."""
    name, w, h = key
    scene = S.SCENE_BY_NAME[name]
    kw = S.frame_kwargs(scene)
    for k in ("pos", "hang_deg", "vang_deg", "width", "height"):
        kw.pop(k)
    hm, cm = _maps(oracle, name)
    heights = oracle.update_heightmap(hm, scene["lum"], scene["min_height"], scene["max_height"])
    f = oracle.make_frame(projection=scene["projection"], width=w * s, height=h * s, pos=cam[:3], hang=cam[3],
                          vang=cam[4], **kw)
    fb, _, st = oracle.render(f, heights, cm, want_steps=False)
    return fb, st


def expected(oracle, scene, cams, s, channels=4):
    key = (scene["name"], scene["width"], scene["height"])
    return blur_reduce([_oracle_sub(oracle, key, tuple(c), s)[0] for c in cams], s, channels)


def _frame(hmrm, renderer, scene, s=1, **extra):
    return H.product_frame(hmrm, renderer, scene, flags=hmrm.supersample_flag(s) | extra.pop("flags", 0), **extra)


def _set(renderer, cams):
    renderer.set_motion_blur([(c[:3], c[3], c[4]) for c in cams])


def _assert_same(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = np.argwhere((got != want).any(axis=-1))
    assert bad.size == 0, f"{what}: {len(bad)} pixels differ, first at {tuple(bad[0])}"


def _fit(scene, n, s, budget=1_500_000):
    """The scene at a size whose n * s * s sub-frame rays stay within the oracle's budget (odd sizes kept odd)."""
    w, h = scene["width"], scene["height"]
    k = math.sqrt(budget / (n * s * s * w * h))
    if k < 1.0:
        w, h = max(2, int(w * k) | 1), max(2, int(h * k) | 1)
    return dict(scene, width=w, height=h)


# ---- 1. every scene and projection; n in {1, 2, 3, 5, 16} x s in {1, 2, 3, 4} dealt over the scenes ----
@pytest.mark.parametrize("i,scene", list(enumerate(S.SCENES)), ids=lambda v: v["name"] if isinstance(v, dict) else "")
def test_render_equals_blur_of_oracle(hmrm, renderer, oracle, i, scene):
    _configure(renderer, oracle, scene["name"])
    for n, s in (PAIRS[i % len(PAIRS)], PAIRS[(i + 7) % len(PAIRS)]):
        sc = _fit(scene, n, s)
        cams = scene_cams(oracle, sc, n)
        want = expected(oracle, sc, cams, s)
        _set(renderer, cams)
        for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
            got = renderer.render(_frame(hmrm, renderer, sc, s, pixel_format=fmt))
            _assert_same(got, want[:, :, :ch], f"{scene['name']} {sc['width']}x{sc['height']} n={n} s={s} ch={ch}")


def test_every_pair_is_dealt():
    assert {PAIRS[i % 20] for i in range(len(S.SCENES))} | {PAIRS[(i + 7) % 20] for i in range(len(S.SCENES))} == \
        set(PAIRS)


@pytest.mark.parametrize("w,h", [(2, 2), (3, 2), (5, 7), (13, 3), (37, 21)])
def test_small_and_odd_frames(hmrm, renderer, oracle, w, h):
    for name in ("persp_basic", "spher_basic", "ortho_basic"):
        scene = dict(S.SCENE_BY_NAME[name], width=w, height=h)
        _configure(renderer, oracle, name)
        for n, s in PAIRS:
            cams = scene_cams(oracle, scene, n, step=3.0)
            want = expected(oracle, scene, cams, s)
            _set(renderer, cams)
            for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
                got = renderer.render(_frame(hmrm, renderer, scene, s, pixel_format=fmt))
                _assert_same(got, want[:, :, :ch], f"{name} {w}x{h} n={n} s={s} channels={ch}")


# ---- 2. the 4K flythrough at n = 8 between two consecutive bench cameras: sampled rows against the oracle ----
def test_flythrough4k_n8_sampled_rows_match_oracle(hmrm, oracle):
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    wl = bench.WORKLOADS["flythrough4k"]
    W, Hh = wl["W"], wl["H"]
    c0, c1 = bench.camera(wl, 7), bench.camera(wl, 8)

    def cam(c):
        return (*[float(v) for v in c["pos"]], oracle.deg2rad(c["hang_deg"]), oracle.deg2rad(c["vang_deg"]))

    cams = blur_cameras(cam(c0), cam(c1), 0.5, 8)
    r = hmrm.Renderer(0)
    try:
        r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
        r.synth_maps(wl["log2n"], bench.SEED)
        f = r.frame(projection=wl["projection"], screen_width=W, screen_height=Hh, cam_pos=c0["pos"],
                    hang=hmrm.deg2rad(c0["hang_deg"]), vang=hmrm.deg2rad(c0["vang_deg"]),
                    hfov=hmrm.deg2rad(c0["hfov_deg"]), ortho_width=c0["ortho_width"], grid_width=bench.GRID_WIDTH,
                    step_dist=wl["step_dist"])
        _set(r, cams)
        got = r.render(f).copy()
    finally:
        r.close()
    terrain = np.nonzero((got[:, :, :3] != 0).any(axis=(1, 2)))[0]
    assert terrain.size > 0
    first = int(terrain[0])
    rows = sorted({0, max(first - 1, 0), first, min(first + 1, Hh - 1), min(first + 20, Hh - 1), Hh // 2, Hh - 1})
    hits = 0
    for py in rows:
        subs = []
        for c in cams:
            of = oracle.make_frame(projection=wl["projection"], width=W, height=Hh, pos=c[:3], hang=c[3], vang=c[4],
                                   hfov_deg=c0["hfov_deg"], ortho_width=c0["ortho_width"], grid_width=bench.GRID_WIDTH,
                                   step_dist=wl["step_dist"], min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT)
            ofb, _, ost = oracle.render_synth(of, wl["log2n"], bench.SEED, rows=(py, py + 1), want_steps=False)
            subs.append(ofb[py:py + 1])
            hits += ost.surf_hits
        _assert_same(got[py:py + 1], blur_reduce(subs, 1), f"flythrough4k n=8 row {py}")
    assert hits > 0


# ---- 3. the collapse property and turning blur off ----
@pytest.mark.parametrize("name", ["persp_basic", "spher_fine", "ortho_basic"])
def test_identical_cameras_give_the_plain_frame_and_clearing_restores_it(hmrm, renderer, oracle, name):
    scene = dict(S.SCENE_BY_NAME[name], width=96, height=54)
    _configure(renderer, oracle, name)
    cam = camera_of(oracle, scene)
    for s in (1, 2, 3, 4):
        renderer.set_motion_blur([])
        plain = renderer.render(_frame(hmrm, renderer, scene, s)).copy()
        for n in (1, 2, 5, 16):
            _set(renderer, [cam] * n)
            _assert_same(renderer.render(_frame(hmrm, renderer, scene, s)), plain, f"{name} s={s} n={n}")
    _set(renderer, scene_cams(oracle, scene, 3))
    blurred = renderer.render(_frame(hmrm, renderer, scene)).copy()
    renderer.set_motion_blur(np.zeros((0, 5)))
    _assert_same(renderer.render(_frame(hmrm, renderer, scene)), expected(oracle, scene, [cam], 1), f"{name} cleared")
    assert (blurred != renderer.render(_frame(hmrm, renderer, scene))).any(), "the cameras should move the picture"


def test_array_and_sequence_forms_agree(hmrm, renderer, oracle):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=64, height=36)
    _configure(renderer, oracle, "persp_basic")
    cams = scene_cams(oracle, scene, 5)
    renderer.set_motion_blur(np.array(cams, dtype=np.float64))
    a = renderer.render(_frame(hmrm, renderer, scene)).copy()
    _set(renderer, cams)
    _assert_same(renderer.render(_frame(hmrm, renderer, scene)), a, "[n, 5] array against (pos, hang, vang)")
    _assert_same(a, expected(oracle, scene, cams, 1), "against the oracle")


# ---- 4. PNG, YUV and JPEG outputs ----
@pytest.mark.parametrize("name,n,s", [("persp_basic", 4, 1), ("spher_wide", 5, 2), ("defaults_grid", 2, 1)])
def test_encoded_outputs_are_of_the_blurred_frame(hmrm, renderer, oracle, name, n, s):
    from PIL import Image

    scene = _fit(S.SCENE_BY_NAME[name], n, s)
    _configure(renderer, oracle, name)
    cams = scene_cams(oracle, scene, n)
    want = expected(oracle, scene, cams, s)
    _set(renderer, cams)
    for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
        f = _frame(hmrm, renderer, scene, s, pixel_format=fmt)
        data = renderer.render_png(f)
        _assert_same(check_png(data)[0], want[:, :, :ch], f"{name} PNG channels={ch} (checker)")
        _assert_same(np.asarray(Image.open(io.BytesIO(data))), want[:, :, :ch], f"{name} PNG channels={ch} (PIL)")
        assert_equals_model(data, want, f"{name} PNG channels={ch}")
        for matrix in (hmrm.YUV_BT601, hmrm.YUV_BT709):
            got = renderer.render_yuv420(f, matrix=matrix)
            for plane, g, w in zip("Y Cb Cr".split(), got, yuv420_model(want, matrix)):
                assert np.array_equal(g, w), f"{name} YUV format {fmt} matrix {matrix} plane {plane}"
        for q, chroma, sub in ((75, hmrm.JPEG_420, True), (90, hmrm.JPEG_444, False)):
            assert renderer.render_jpeg(f, quality=q, chroma=chroma) == J.write(want, q, sub), f"{name} JPEG q={q}"


# ---- 5. hmrm_render_device at byte offsets 0-3 with guard bytes, on the context's and a caller's stream ----
def test_render_device_offsets_and_streams(hmrm, renderer, oracle):
    import torch

    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=61, height=35)
    _configure(renderer, oracle, "persp_basic")
    w, h, guard = scene["width"], scene["height"], 64
    cases = [(n, s, ch) for n, s, ch in ((2, 1, 4), (5, 2, 3), (3, 3, 4), (6, 1, 3))]
    want = [expected(oracle, scene, scene_cams(oracle, scene, n), s, ch) for n, s, ch in cases]
    st = torch.cuda.Stream()
    for stream in (None, st):
        bufs = []
        for (n, s, ch), off in zip(cases, range(4)):
            buf = torch.full((2 * guard + off + h * w * ch,), 0xA5, dtype=torch.uint8, device="cuda:0")
            _set(renderer, scene_cams(oracle, scene, n))
            fmt = hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8
            renderer.render_device(_frame(hmrm, renderer, scene, s, pixel_format=fmt), buf.data_ptr() + guard + off,
                                   None if stream is None else stream.cuda_stream)
            bufs.append((buf, off, ch))
        if stream is None:
            renderer.wait()
        else:
            stream.synchronize()
        for i, (buf, off, ch) in enumerate(bufs):
            b = buf.cpu().numpy()
            what = f"case {i} offset {off} stream {'caller' if stream else 'context'}"
            assert (b[:guard + off] == 0xA5).all() and (b[guard + off + h * w * ch:] == 0xA5).all(), what + " guard"
            _assert_same(b[guard + off:guard + off + h * w * ch].reshape(h, w, ch), want[i], what)


# ---- 6. frames in flight: blurred (different camera sets), plain and supersampled; raw, PNG, YUV and JPEG ----
def test_frames_in_flight_keep_their_own_state(hmrm, renderer, oracle):
    base = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    _configure(renderer, oracle, "persp_basic")
    plan = [(4, 1), (0, 1), (8, 1), (0, 2), (3, 2), (16, 1), (1, 1), (2, 3), (5, 1), (0, 1)]   # (n, s); n = 0: plain
    kinds = ["raw", "png", "yuv", "jpeg"]
    w, h = base["width"], base["height"]
    want, sets = [], []
    for i, (n, s) in enumerate(plan):
        sc = dict(base, pos=(-0.6 + 0.05 * i, 0.6, 3.2 - 0.1 * i), hang_deg=-45.0 - 7.0 * i)
        cams = scene_cams(oracle, sc, n, step=1.0 + i) if n else [camera_of(oracle, sc)]
        sets.append((sc, cams))
        want.append(expected(oracle, sc, cams, s))
    raw = [hmrm.pinned_empty((h, w, 4)) for _ in range(4)]
    files = [hmrm.pinned_empty((max(hmrm.png_bound(w, h, 4), hmrm.jpeg_bound(w, h)),)) for _ in range(4)]
    sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]
    yuv = [hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),)) for _ in range(4)]

    def check(j):
        k, what = kinds[j % 4], f"frame {j} n={plan[j][0]} s={plan[j][1]} {kinds[j % 4]}"
        if k == "raw":
            _assert_same(raw[j % 4], want[j], what)
        elif k == "png":
            data = files[j % 4][:int(sizes[j % 4][0])].tobytes()
            _assert_same(check_png(data)[0], want[j], what)
            assert_equals_model(data, want[j], what)
        elif k == "yuv":
            assert i420(yuv420_model(want[j], BT709)) == yuv[j % 4].tobytes(), what
        else:
            assert files[j % 4][:int(sizes[j % 4][0])].tobytes() == J.write(want[j], 80, True), what

    pending = []
    for i, (n, s) in enumerate(plan):
        if len(pending) == 4:
            renderer.wait_pending(3)
            check(pending.pop(0))
        sc, cams = sets[i]
        if n:
            _set(renderer, cams)
        else:
            renderer.set_motion_blur([])
        f = _frame(hmrm, renderer, sc, s)
        k = kinds[i % 4]
        if k == "raw":
            renderer.render_async(f, raw[i % 4])
        elif k == "png":
            renderer.render_png_async(f, files[i % 4], sizes[i % 4])
        elif k == "yuv":
            renderer.render_yuv420_async(f, yuv[i % 4], BT709)
        else:
            renderer.render_jpeg_async(f, files[i % 4], sizes[i % 4], quality=80)
        pending.append(i)
    renderer.wait()
    for j in pending:
        check(j)


# ---- 7. statistics are sums over the sub-frame renders ----
@pytest.mark.parametrize("name", ["persp_graze", "spher_fine", "ortho_basic"])
def test_stats_sum_over_sub_frames(hmrm, renderer, oracle, name):
    scene = _fit(S.SCENE_BY_NAME[name], 16, 2, budget=3_000_000)
    _configure(renderer, oracle, name)
    for n, s in ((3, 1), (5, 2), (12, 1)):
        cams = scene_cams(oracle, scene, n)
        _set(renderer, cams)
        renderer.render(_frame(hmrm, renderer, scene, s, flags=hmrm.FLAG_STATS))
        st = renderer.stats()
        what = f"{name} n={n} s={s}"
        assert st.rays == n * s * s * scene["width"] * scene["height"], what
        key = (scene["name"], scene["width"], scene["height"])
        ost = [_oracle_sub(oracle, key, tuple(c), s)[1] for c in cams]
        assert st.steps == sum(o.steps for o in ost), what
        assert (st.box_hits, st.surf_hits) == (sum(o.box_hits for o in ost), sum(o.surf_hits for o in ost)), what
        assert st.max_steps == max(o.max_steps for o in ost), what
        assert st.status == 0
        # kernel_ms runs from the first sub-frame's start to the last one's end: at least most of the sum of the same
        # sub-frames rendered one by one (one sub-frame's time alone would be about 1/n of it)
        renderer.set_motion_blur([])
        alone = 0.0
        for c in cams:
            f = _frame(hmrm, renderer, scene, s, flags=hmrm.FLAG_STATS, hang=c[3], vang=c[4])
            f.cam_pos[:] = list(c[:3])
            renderer.render(f)
            alone += renderer.stats().kernel_ms
        assert st.kernel_ms >= 0.5 * alone > 0.0, f"{what}: {st.kernel_ms} ms against {alone} ms one by one"


# ---- 8. refusals: nothing written, the state unchanged ----
def test_refusals(hmrm, renderer, oracle):
    import torch

    scene = S.SCENE_BY_NAME["persp_basic"]
    _configure(renderer, oracle, "persp_basic")
    lib = hmrm.load_library()
    w, h = scene["width"], scene["height"]
    host = hmrm.pinned_empty((h, w, 4))
    png = hmrm.pinned_empty((hmrm.png_bound(w, h, 4),))
    jpg = hmrm.pinned_empty((hmrm.jpeg_bound(w, h),))
    size = hmrm.pinned_empty((1,), dtype=np.uint64)
    yuv = hmrm.pinned_empty((hmrm.yuv420_bytes(w, h),))
    dev = torch.zeros(h * w * 4 + 256, dtype=torch.uint8, device="cuda:0")
    stage = torch.zeros(h * w * 4, dtype=torch.uint8, device="cuda:0")
    ctrl = torch.zeros(256, dtype=torch.uint8, device="cuda:0")
    cams = scene_cams(oracle, scene, 3)
    want = expected(oracle, scene, cams, 1)

    def calls(f):
        fp = C.byref(f)
        return [lib.hmrm_render(renderer._h, fp, host.ctypes.data),
                lib.hmrm_render_async(renderer._h, fp, host.ctypes.data),
                lib.hmrm_render_device(renderer._h, fp, dev.data_ptr(), None),
                lib.hmrm_render_png_async(renderer._h, fp, png.ctypes.data, png.nbytes, size.ctypes.data),
                lib.hmrm_render_yuv420_async(renderer._h, fp, BT709, yuv.ctypes.data, yuv.nbytes),
                lib.hmrm_render_jpeg_async(renderer._h, fp, 75, hmrm.JPEG_420, jpg.ctypes.data, jpg.nbytes,
                                           size.ctypes.data)]

    def frame(**kw):
        return H.product_frame(hmrm, renderer, scene, **kw)

    _set(renderer, cams)
    for arr in (host, png, jpg, size, yuv):
        arr[...] = 0
    bad = {
        "cycle_period 3": frame(cycle_period=3),
        "band_count 2": frame(band_count=2, band_index=0),
        "row band top": frame(row_begin=0, row_end=h // 2),
        "row band bottom": frame(row_begin=4, row_end=h),
        "step index": frame(flags=hmrm.FLAG_STEP_INDEX),
        "ray dump": frame(flags=hmrm.FLAG_RAY_DUMP),
        "cycle_period 3, s = 2": frame(flags=hmrm.supersample_flag(2), cycle_period=3),
    }
    for what, f in bad.items():
        assert calls(f) == [1] * 6, what
        assert b"motion-blurred" in lib.hmrm_last_error(renderer._h), what
    f = frame()
    assert lib.hmrm_render_peer(renderer._h, C.byref(f), dev.data_ptr(), ctrl.data_ptr(), 1, None) == 1
    assert b"motion blur" in lib.hmrm_last_error(renderer._h)
    assert lib.hmrm_render_peer_staged(renderer._h, C.byref(f), stage.data_ptr(), dev.data_ptr(), ctrl.data_ptr(), 1,
                                       None) == 1
    renderer.wait()
    assert int(ctrl.sum()) == 0 and int(dev.sum()) == 0 and int(stage.sum()) == 0
    for arr in (host, png, jpg, size, yuv):
        assert not arr.any()
    # hmrm_set_motion_blur's own refusals leave the cameras in place
    arr = (hmrm.Camera * 17)()
    assert lib.hmrm_set_motion_blur(renderer._h, arr, 17) == 1
    assert lib.hmrm_set_motion_blur(renderer._h, arr, -1) == 1
    assert lib.hmrm_set_motion_blur(renderer._h, None, 2) == 1
    assert lib.hmrm_set_motion_blur(None, arr, 1) == 1
    with pytest.raises(hmrm.HmrmError):
        renderer.set_motion_blur([((0.0, 0.0, 0.0), 0.0, 0.0)] * 17)
    _assert_same(renderer.render(frame()), want, "blurred after refusals")
    # a non-finite sub-frame camera is refused before anything is enqueued
    _set(renderer, [cams[0], (math.nan, 0.0, 0.0, 0.0, 0.0)])
    host[...] = 0
    assert lib.hmrm_render(renderer._h, C.byref(frame()), host.ctypes.data) == 1 and not host.any()
    renderer.set_motion_blur([])
    _assert_same(renderer.render(frame()), H.golden_frames()["persp_basic"], "plain after refusals")


# ---- 9. hmap --script --motion-blur 4 --shutter 0.5 ----
def _script(oracle, tmp_path, scene, n):
    _write_scene(oracle, scene, tmp_path)
    states = [dict(pos=(-0.6 + 0.09 * i, 0.6 - 0.02 * i, 3.2 - 0.05 * i), hang_deg=-45.0 - 6.0 * i) for i in range(n)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"])
                                                 for s in states))
    return states


def _script_expected(oracle, scene, states, k, shutter):
    """Frame n: blur_reduce of the oracle at the cameras of hmap's formula between states n and n + 1; the last plain."""
    vang = oracle.deg2rad(scene["vang_deg"])
    cams = [(*[float(v) for v in st["pos"]], oracle.deg2rad(st["hang_deg"]), vang) for st in states]
    out = []
    for i, c in enumerate(cams):
        sub = blur_cameras(c, cams[i + 1], shutter, k) if i + 1 < len(cams) else [c]
        out.append(expected(oracle, scene, sub, 1))
    return out


def _run(args, cwd, gpus=1, text=True):
    env = dict(os.environ, HMAP_DEVICE_LIST=",".join(["0"] * gpus))
    return subprocess.run([str(HMAP), "config.txt", "--script", "frames.txt", "--gpus", str(gpus), *args],
                          capture_output=True, text=text, cwd=str(cwd), env=env)


@pytest.mark.parametrize("gpus", [1, 3])
def test_hmap_motion_blur_png_y4m_mjpeg_jpeg(hmrm, oracle, gpus, tmp_path):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    states = _script(oracle, tmp_path, scene, 6)
    want = _script_expected(oracle, scene, states, 4, 0.5)
    blur = ["--motion-blur", "4", "--shutter", "0.5"]
    res = _run(["--out-prefix", "f_", *blur, "--stats-json", "stats.json"], tmp_path, gpus)
    assert res.returncode == 0, res.stderr
    # want[-1], the last frame, is the oracle's plain frame of the last camera: it has no successor to blur towards
    for i, w in enumerate(want):
        _assert_same(check_png((tmp_path / f"f_{i}.png").read_bytes())[0], w, f"PNG frame {i}")
        assert_equals_model((tmp_path / f"f_{i}.png").read_bytes(), w, f"PNG frame {i}")
    st = json.loads((tmp_path / "stats.json").read_text())
    assert st["motion_blur"] == 4 and st["shutter"] == 0.5 and st["frames"] == len(states)
    assert st["rays"] == 160 * 90 * (4 * (len(states) - 1) + 1)
    res = _run(["--video", "-", *blur], tmp_path, gpus, text=False)
    assert res.returncode == 0, res.stderr.decode()
    header, frames = read_y4m(res.stdout)
    assert (header["W"], header["H"]) == ("160", "90") and len(frames) == len(want)
    for i, (g, w) in enumerate(zip(frames, want)):
        assert g == i420(yuv420_model(w, BT709)), f"Y4M frame {i}"
    res = _run(["--video", "-", "--jpeg", "75", *blur], tmp_path, gpus, text=False)
    assert res.returncode == 0, res.stderr.decode()
    assert res.stdout == b"".join(J.write(w, 75, True) for w in want)
    # JPEG stills: one file per frame
    res = _run(["--out-prefix", "j_", "--jpeg", "80", *blur], tmp_path, gpus)
    assert res.returncode == 0, res.stderr
    for i, w in enumerate(want):
        assert (tmp_path / f"j_{i}.jpg").read_bytes() == J.write(w, 80, True), f"JPEG frame {i}"


def test_hmap_motion_blur_1_is_byte_identical(hmrm, oracle, tmp_path):
    scene = dict(S.SCENE_BY_NAME["ortho_basic"], width=96, height=54)
    outs = []
    for sub, extra in (("plain", []), ("blur1", ["--motion-blur", "1"])):
        d = tmp_path / sub
        d.mkdir()
        _script(oracle, d, scene, 5)
        for args in (["--out-prefix", "f_"], ["--video", "v.y4m"], ["--video", "-", "--jpeg", "80"]):
            res = _run([*args, "--projection", "3", *extra], d, text=False)
            assert res.returncode == 0, res.stderr.decode()
            files = {p.name: p.read_bytes() for p in sorted(d.iterdir()) if p.suffix in (".png", ".y4m")}
            outs.append((sub, args, res.stdout, res.stderr, files))
    for a, b in zip(outs[:3], outs[3:]):
        assert a[2:] == b[2:], f"{a[1]}: --motion-blur 1 differs from no option"
