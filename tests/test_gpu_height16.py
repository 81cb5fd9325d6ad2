"""GPU: 16-bit height maps (hmrm_set_maps16 / hmrm_set_maps16_device / hmrm_synth_maps16, kernels k1_range<Grey16Cells>,
k1_build16) against the numpy model of include/hmrm.h's definition, against the pinned 8-bit path for
widened grey maps, and against the CPU oracle rendering the model's heights; and `hmap --height-bits 16`."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import height16_lib as H16
import helpers as H
import scenes as S
from test_gpu_round2 import load_bench
from test_gpu_sdl_shell import build_shell
from test_png_encode import check_png
from test_supersample import box_reduce
from test_yuv420 import BT709, i420, read_y4m, yuv420_model

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"

TRAVERSALS = [1, 2, 3, 4]          # brute, skip, skip_fp64, pack
UNIT_LUM = (1.0, 0.0, 0.0)


def same_bits(a, b) -> bool:
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


def set_heights16(r, x, cm, lum, lo, hi):
    r.lum_r, r.lum_g, r.lum_b = lum
    r.min_height, r.max_height = lo, hi
    r.set_maps16(x, cm)


# ---- heights --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["persp_basic", "persp_graze", "noise_lum", "noise_lum_neg", "crop_ortho",
                                  "min_height_twice", "min_height_negative"])
def test_heights_equal_model_on_scene_maps(hmrm, renderer, oracle, name):
    sc = S.SCENE_BY_NAME[name]
    hm, cm = H.load_scene_maps(sc, oracle)
    x = (hm[:, :, 1].astype(np.uint16) * 257) ^ (hm[:, :, 0].astype(np.uint16) * 3)     # full-precision samples
    set_heights16(renderer, x, cm, sc["lum"], sc["min_height"], sc["max_height"])
    assert same_bits(renderer.heights(), H16.heights16(x, sc["lum"], sc["min_height"], sc["max_height"]))


@pytest.mark.parametrize("w,h", [(1, 1), (1, 37), (41, 1), (2, 2), (5, 3), (13, 7), (255, 17), (256, 256), (4097, 3),
                                 (3, 4097), (300, 301)])
@pytest.mark.parametrize("lum,lo,hi", [((0.299, 0.587, 0.114), 0.0, 10.0), ((-0.2, 1.4, 0.1), -1.25, 1.5),
                                       ((1.7, 2.3, 0.9), 3.0, -2.0)])
def test_heights_equal_model_on_noise_every_value(hmrm, renderer, w, h, lum, lo, hi):
    n = w * h
    rng = np.random.default_rng(w * 7919 + h)
    x = rng.integers(0, 65536, size=n, dtype=np.uint16)
    x[: min(n, 65536)] = rng.permutation(65536)[: min(n, 65536)].astype(np.uint16)   # all 65536 values when n allows
    x = x.reshape(h, w)
    cm = rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8)
    set_heights16(renderer, x, cm, lum, lo, hi)
    assert same_bits(renderer.heights(), H16.heights16(x, lum, lo, hi))


def test_set_maps16_device_and_synth_maps16(hmrm, renderer):
    import torch

    x, cm = H16.synth_maps16(9, 77)
    renderer.lum_r, renderer.lum_g, renderer.lum_b = S.DEFAULT_LUM
    renderer.min_height, renderer.max_height = 0.0, 2.0
    renderer.synth_maps16(9, 77)
    want = H16.heights16(x, S.DEFAULT_LUM, 0.0, 2.0)
    assert same_bits(renderer.heights(), want)
    dx = torch.from_numpy(x.view(np.int16)).cuda()
    dc = torch.from_numpy(cm).cuda()
    renderer.set_maps16_device(dx, dc, 512, 512)
    assert same_bits(renderer.heights(), want)


# ---- equivalence with the 8-bit path -------------------------------------------------------------------------------
def _render_pair(hmrm, r, sc, hm, cm, traversal, pixel_format):
    lum, lo, hi = UNIT_LUM, sc["min_height"], sc["max_height"]
    flags = hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX
    r.lum_r, r.lum_g, r.lum_b = lum
    r.min_height, r.max_height = lo, hi
    grey = np.repeat(hm[:, :, :1], 3, axis=2)
    r.set_maps(grey, cm)
    f = H.product_frame(hmrm, r, sc, traversal=traversal, pixel_format=pixel_format, flags=flags)
    a, sa, ta = r.render(f).copy(), r.step_index(f).copy(), r.stats()
    r.set_maps16(hm[:, :, 0].astype(np.uint16) * 257, cm)
    b, sb, tb = r.render(f).copy(), r.step_index(f).copy(), r.stats()
    return (a, sa, ta), (b, sb, tb)


@pytest.mark.parametrize("pixel_format", [0, 1])
@pytest.mark.parametrize("traversal", TRAVERSALS)
@pytest.mark.parametrize("name", [s["name"] for s in S.SCENES])
def test_widened_grey_matches_8bit_path(hmrm, renderer, oracle, name, traversal, pixel_format):
    sc = S.SCENE_BY_NAME[name]
    hm, cm = H.load_scene_maps(sc, oracle)
    (a, sa, ta), (b, sb, tb) = _render_pair(hmrm, renderer, sc, hm, cm, traversal, pixel_format)
    assert np.array_equal(a, b)
    assert np.array_equal(sa, sb)
    assert (ta.rays, ta.steps, ta.fetches, ta.surf_hits) == (tb.rays, tb.steps, tb.fetches, tb.surf_hits)


@pytest.mark.parametrize("layout", [0, 1, 2])
@pytest.mark.parametrize("name", ["persp_graze", "crop_ortho"])
def test_widened_grey_matches_8bit_path_in_every_layout(hmrm, oracle, name, layout):
    sc = S.SCENE_BY_NAME[name]
    hm, cm = H.load_scene_maps(sc, oracle)
    r = hmrm.Renderer(0)
    try:
        r.set_layout(layout)
        for traversal in (2, 4):
            (a, sa, ta), (b, sb, tb) = _render_pair(hmrm, r, sc, hm, cm, traversal, 0)
            assert r.get_layout() == layout
            assert np.array_equal(a, b) and np.array_equal(sa, sb)
            assert (ta.steps, ta.fetches) == (tb.steps, tb.fetches)
    finally:
        r.close()


# ---- oracle parity over the model's heights ------------------------------------------------------------------------
SYNTH16 = {8: H16.synth_maps16(8, 1234), 9: H16.synth_maps16(9, 77)}


def _synth_scene(sc):
    return dict(sc, lum=S.DEFAULT_LUM, maps=dict(kind="synth16", log2n=9 if sc["maps"].get("log2n") == 9 else 8))


def _oracle16(oracle, sc, **extra):
    x, cm = SYNTH16[sc["maps"]["log2n"]]
    heights = H16.heights16(x, sc["lum"], sc["min_height"], sc["max_height"])
    return oracle.render(H.oracle_frame(oracle, sc, **extra), heights, cm)


def _configure16(renderer, sc):
    log2n = sc["maps"]["log2n"]
    renderer.lum_r, renderer.lum_g, renderer.lum_b = sc["lum"]
    renderer.min_height, renderer.max_height = sc["min_height"], sc["max_height"]
    renderer.synth_maps16(log2n, 1234 if log2n == 8 else 77)


@pytest.mark.parametrize("name", [s["name"] for s in S.SCENES])
def test_synth16_frames_match_oracle(hmrm, renderer, oracle, name):
    sc = _synth_scene(S.SCENE_BY_NAME[name])
    _configure16(renderer, sc)
    want, wsteps, wst = _oracle16(oracle, sc)
    f = H.product_frame(hmrm, renderer, sc, flags=hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX)
    got = renderer.render(f)
    assert np.array_equal(got, want), f"{int((got != want).any(axis=2).sum())} pixels differ"
    assert np.array_equal(renderer.step_index(f), wsteps)
    assert renderer.stats().steps == wst.steps


@pytest.mark.parametrize("name", ["persp_basic", "spher_wide"])
def test_synth16_supersampled_matches_box_filter_of_oracle(hmrm, renderer, oracle, name):
    sc = _synth_scene(S.SCENE_BY_NAME[name])
    _configure16(renderer, sc)
    sub = dict(sc, width=2 * sc["width"], height=2 * sc["height"])
    want = box_reduce(_oracle16(oracle, sub)[0], 2)
    f = H.product_frame(hmrm, renderer, sc, flags=hmrm.supersample_flag(2))
    assert np.array_equal(renderer.render(f), want)


def test_flythrough4k_bands_over_synth16_match_oracle(hmrm, oracle):
    """BASELINE configs[3]'s camera over synth_maps16(14): sampled 4-row bands, pixels and step indices."""
    bench = load_bench()
    wl = bench.WORKLOADS["flythrough4k"]
    W, Hh = wl["W"], wl["H"]
    c = bench.camera(wl, 7)
    r = hmrm.Renderer(0)
    try:
        r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
        r.synth_maps16(wl["log2n"], bench.SEED)
        f = r.frame(projection=wl["projection"], screen_width=W, screen_height=Hh, cam_pos=c["pos"],
                    hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                    ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                    flags=hmrm.FLAG_STATS | hmrm.FLAG_STEP_INDEX)
        got = r.render(f).copy()
        steps = r.step_index(f).copy()
        assert r.stats().status == 0
    finally:
        r.close()
    x, cm = H16.synth_maps16(wl["log2n"], bench.SEED)
    heights = H16.c_heights16(x, S.DEFAULT_LUM, bench.MIN_HEIGHT, bench.MAX_HEIGHT)
    del x
    hit_rows = np.nonzero((steps >= 0).any(axis=1))[0]
    assert hit_rows.size > 0
    first = int(hit_rows[0])
    starts = sorted({0, max(first - 2, 0), min(first + 40, Hh - 4), Hh // 2, (3 * Hh) // 4, Hh - 4})
    of = oracle.make_frame(projection=wl["projection"], width=W, height=Hh, grid_width=bench.GRID_WIDTH,
                           step_dist=wl["step_dist"], min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT, **c)
    total_hits = 0
    for a in starts:
        ofb, osteps, ost = oracle.render(of, heights, cm, rows=(a, a + 4))
        assert np.array_equal(got[a:a + 4], ofb[a:a + 4]), f"rows {a}..{a + 3} differ from the oracle"
        assert np.array_equal(steps[a:a + 4], osteps[a:a + 4]), f"step indices of rows {a}..{a + 3}"
        total_hits += ost.surf_hits
    assert total_hits > 0


# ---- one context ----------------------------------------------------------------------------------------------------
def test_switching_depths_in_one_context(hmrm, oracle):
    sc8 = S.SCENE_BY_NAME["persp_graze"]
    sc16 = _synth_scene(sc8)
    hm, cm = H.load_scene_maps(sc8, oracle)
    r = hmrm.Renderer(0)
    try:
        for _ in range(2):
            _configure16(r, sc16)
            assert np.array_equal(r.render(H.product_frame(hmrm, r, sc16)), _oracle16(oracle, sc16)[0])
            with pytest.raises(hmrm.HmrmError) as e:
                r.get_maps()
            assert e.value.code == 3 and "16-bit" in str(e.value)
            H.configure(r, sc8, (hm, cm))
            assert np.array_equal(r.render(H.product_frame(hmrm, r, sc8)), H.oracle_render_scene(oracle, sc8, (hm, cm))[0])
            ghm, gcm = r.get_maps()
            assert np.array_equal(ghm, hm) and np.array_equal(gcm, cm)
    finally:
        r.close()


def test_refusals(hmrm):
    r = hmrm.Renderer(0)
    try:
        lum = (C.c_double * 3)(0.299, 0.587, 0.114)
        assert r._lib.hmrm_update_heightmap(r._h, lum, 0.0, 10.0) == 3
        x = np.zeros((4, 4), np.uint16)
        cm = np.zeros((4, 4, 4), np.uint8)
        assert r._lib.hmrm_set_maps16(r._h, None, cm.ctypes.data, 4, 4) == 1
        assert r._lib.hmrm_set_maps16(r._h, x.ctypes.data, None, 4, 4) == 1
        assert r._lib.hmrm_set_maps16_device(r._h, None, None, 4, 4) == 1
        for w, h in ((0, 4), (4, 0), (32769, 1), (1, 32769), (-1, 4)):
            assert r._lib.hmrm_set_maps16(r._h, x.ctypes.data, cm.ctypes.data, w, h) == 1
        assert r._lib.hmrm_synth_maps16(r._h, 3, 1) == 1
        assert r._lib.hmrm_synth_maps16(r._h, 16, 1) == 1
        # a 16-bit map's colormap is still downloadable
        r.set_maps16(x + 7, cm + 3)
        out = np.empty((4, 4, 4), np.uint8)
        assert r._lib.hmrm_get_maps(r._h, None, out.ctypes.data) == 0
        assert (out == 3).all()
    finally:
        r.close()


# ---- hmap -----------------------------------------------------------------------------------------------------------
def _write16(oracle, tmp_path, sc, x, cm, lum=None, name="h16.png"):
    H16.write_png16(tmp_path / name, x)
    oracle.write_png(tmp_path / "c.png", cm)
    (tmp_path / "config.txt").write_text(oracle.config_text(S.frame_kwargs(sc), name, "c.png", lum=lum))
    return tmp_path / "config.txt"


def _hmap(args, tmp_path, env=None):
    res = subprocess.run([str(HMAP), *args], capture_output=True, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr.decode()
    return res


def test_hmap_headless_16bit_png_matches_oracle(hmrm, oracle, tmp_path):
    sc = _synth_scene(S.SCENE_BY_NAME["persp_graze"])
    x, cm = SYNTH16[9]
    _write16(oracle, tmp_path, sc, x, cm, lum=sc["lum"])
    _hmap(["config.txt", "--headless", "out.png", "--height-bits", "16"], tmp_path)
    assert np.array_equal(check_png((tmp_path / "out.png").read_bytes())[0], _oracle16(oracle, sc)[0])
    # the same frame over three contexts (tile-row bands)
    env = dict(os.environ, HMAP_DEVICE_LIST="0,0,0")
    _hmap(["config.txt", "--headless", "out3.png", "--height-bits", "16", "--gpus", "3"], tmp_path, env)
    assert np.array_equal(check_png((tmp_path / "out3.png").read_bytes())[0], _oracle16(oracle, sc)[0])


def test_hmap_8bit_grey_png_same_file_at_either_depth(hmrm, oracle, tmp_path):
    sc = S.SCENE_BY_NAME["persp_basic"]
    hm, cm = H.load_scene_maps(sc, oracle)
    oracle.write_png(tmp_path / "g8.png", hm[:, :, 0])
    oracle.write_png(tmp_path / "c.png", cm)
    (tmp_path / "config.txt").write_text(oracle.config_text(S.frame_kwargs(sc), "g8.png", "c.png", lum=UNIT_LUM))
    _hmap(["config.txt", "--headless", "a.png"], tmp_path)
    _hmap(["config.txt", "--headless", "b.png", "--height-bits", "16"], tmp_path)
    assert (tmp_path / "a.png").read_bytes() == (tmp_path / "b.png").read_bytes()


def test_hmap_script_loads_another_16bit_map(hmrm, oracle, tmp_path):
    sc = _synth_scene(dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90))
    x, cm = SYNTH16[8]
    _write16(oracle, tmp_path, sc, x, cm, lum=sc["lum"])
    y = np.ascontiguousarray(x[::-1])
    H16.write_png16(tmp_path / "other.png", y)
    (tmp_path / "frames.txt").write_text("hang -40\nheightmap other.png\nhang -35\n")
    _hmap(["config.txt", "--script", "frames.txt", "--out-prefix", "f", "--height-bits", "16"], tmp_path)
    for i, (hang, hmap16) in enumerate([(-40.0, x), (-40.0, y), (-35.0, y)]):
        s = dict(sc, hang_deg=hang)
        heights = H16.heights16(hmap16, s["lum"], s["min_height"], s["max_height"])
        want = oracle.render(H.oracle_frame(oracle, s), heights, cm)[0]
        assert np.array_equal(check_png((tmp_path / f"f{i}.png").read_bytes())[0], want), f"frame {i}"


def test_hmap_video_16bit(hmrm, oracle, tmp_path):
    sc = _synth_scene(dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90))
    x, cm = SYNTH16[8]
    _write16(oracle, tmp_path, sc, x, cm, lum=sc["lum"])
    states = [-45.0 - 5.0 * i for i in range(4)]
    (tmp_path / "frames.txt").write_text("".join(f"hang {h!r}\n" for h in states))
    res = _hmap(["config.txt", "--script", "frames.txt", "--video", "-", "--height-bits", "16"], tmp_path)
    header, frames = read_y4m(res.stdout)
    want = [i420(yuv420_model(_oracle16(oracle, dict(sc, hang_deg=h))[0], BT709)) for h in states]
    assert len(frames) == len(want)
    for i, (g, w) in enumerate(zip(frames, want)):
        assert g == w, f"frame {i}"


def test_shell_shows_16bit_map(hmrm, oracle, tmp_path):
    binary = build_shell(tmp_path)
    sc = _synth_scene(dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90))
    x, cm = SYNTH16[8]
    _write16(oracle, tmp_path, sc, x, cm, lum=sc["lum"])
    (tmp_path / "events.txt").write_text("")
    d = tmp_path / "dump"
    d.mkdir()
    env = dict(os.environ, HMRM_FAKE_FRAMES="1", HMRM_FAKE_EVENTS=str(tmp_path / "events.txt"),
               HMRM_FAKE_DUMP=str(d / "frame_"), HMRM_FAKE_PROJ="1")
    res = subprocess.run([str(binary), "config.txt", "--height-bits", "16"], cwd=str(tmp_path), env=env,
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    got = np.fromfile(d / "frame_0.rgba", dtype=np.uint8).reshape(90, 160, 4)
    assert np.array_equal(got, _oracle16(oracle, sc)[0])
