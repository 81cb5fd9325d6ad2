"""CPU: the oracle (oracle/hmap_oracle.c) against the committed fixtures that were produced by the
UNMODIFIED reference (tests/golden/make_golden.py) or recorded where it matched the reference
(tests/golden/replays.json, tests/golden/make_golden_replays.py), and — when oracle/_ref is present — against
the reference build itself, live."""
import numpy as np
import pytest

import helpers as H
import scenes as S


@pytest.mark.parametrize("scene", S.SCENES, ids=lambda s: s["name"])
def test_oracle_frame_matches_reference_golden(oracle, scene):
    meta = H.golden_meta()[scene["name"]]
    maps = H.load_scene_maps(scene, oracle)
    fb, steps, st = H.oracle_render_scene(oracle, scene, maps)
    assert H.sha(fb) == meta["sha256"]
    assert np.array_equal(fb, H.golden_frames()[scene["name"]])
    assert (st.rays, st.box_hits, st.surf_hits, st.steps, st.max_steps) == (
        meta["rays"], meta["box_hits"], meta["surf_hits"], meta["steps"], meta["max_steps"])
    assert H.sha(steps) == meta["step_index_sha256"]
    assert st.status == 0


def test_oracle_deg2rad_kat(oracle):
    for rec in H.golden_kat()["deg2rad"]:
        assert H.same(oracle.deg2rad(H.fx(rec["deg"])), rec["rad"])


def test_oracle_rays_kat(oracle):
    for rec in H.golden_kat()["rays"]:
        f = oracle.make_frame(projection=rec["projection"], width=rec["W"], height=rec["H"],
                              pos=[float.fromhex(v) for v in rec["pos"]], hang=float.fromhex(rec["hang"]),
                              vang=float.fromhex(rec["vang"]), hfov=float.fromhex(rec["hfov"]),
                              ortho_width=float.fromhex(rec["ortho_width"]))
        pos, d = oracle.get_ray(f, float.fromhex(rec["w"]), float.fromhex(rec["h"]))
        assert all(H.same(v, g) for v, g in zip(pos, rec["ray_pos"])), rec
        assert all(H.same(v, g) for v, g in zip(d, rec["ray_dir"])), rec


def test_oracle_aabb_kat(oracle):
    for rec in H.golden_kat()["aabb"]:
        args = [[float.fromhex(v) for v in rec[k]] for k in ("pos", "dir", "c0", "c1")]
        d = oracle.distance(*args)
        assert H.same(d, rec["distance"]), rec
        hit, pt = oracle.intersection(*args)
        assert int(hit) == rec["hit"]
        if hit:
            assert all(H.same(v, g) for v, g in zip(pt, rec["point"]))


def test_oracle_heights_kat(oracle):
    for rec in H.golden_kat()["heights"]:
        rgb = np.random.RandomState(rec["rgb_seed"]).randint(0, 256, size=(64, 64, 3)).astype(np.uint8)
        rgb[0, :8] = [[0, 0, 0], [255, 255, 255], [255, 0, 0], [0, 255, 0], [0, 0, 255], [1, 1, 1],
                      [254, 255, 253], [128, 128, 128]]
        h = oracle.update_heightmap(rgb, [float.fromhex(v) for v in rec["lum"]],
                                    float.fromhex(rec["min_height"]), float.fromhex(rec["max_height"]))
        assert all(H.same(float(v), g) for v, g in zip(h[0, :16], rec["first_row"]))
        assert H.sha(h) == rec["sha256"]


def test_cycle_interleave_and_row_band(oracle):
    """cycle/cycle_period (main/hmap.cpp:976-981) only selects pixels: phases tile the full frame."""
    scene = S.SCENE_BY_NAME["persp_basic"]
    maps = H.load_scene_maps(scene, oracle)
    full, _, _ = H.oracle_render_scene(oracle, scene, maps)
    acc = np.zeros_like(full)
    hm, cm = maps
    heights = oracle.update_heightmap(hm, scene["lum"], scene["min_height"], scene["max_height"])
    for phase in range(7):
        oracle.render(H.oracle_frame(oracle, scene, cycle=phase, cycle_period=7), heights, cm, framebuf=acc)
    assert np.array_equal(acc, full)
    band = np.zeros_like(full)
    oracle.render(H.oracle_frame(oracle, scene), heights, cm, rows=(40, 100), framebuf=band)
    assert np.array_equal(band[40:100], full[40:100]) and not band[:40].any() and not band[100:].any()


@pytest.mark.parametrize("name", ["persp_basic", "spher_fine", "ortho_basic", "noise_lum_neg", "min_height_twice"])
def test_oracle_matches_live_reference(oracle, name, tmp_path):
    """Oracle A (unmodified reference under the fake SDL): its stored frame (tests/golden/frames.npz), and both
    builds rendered now where oracle/_ref is built."""
    scene = S.SCENE_BY_NAME[name]
    hm, cm = H.load_scene_maps(scene, oracle)
    fb, _, _ = H.oracle_render_scene(oracle, scene, (hm, cm))
    assert np.array_equal(H.golden_frames()[name], fb)
    if not oracle.have_ref():
        return
    oracle.write_png(tmp_path / "h.png", hm)
    oracle.write_png(tmp_path / "c.png", cm)
    kw = S.frame_kwargs(scene)
    cfg = oracle.config_text(kw, tmp_path / "h.png", tmp_path / "c.png", lum=scene["lum"])
    for binary in (oracle.REF_BIN, oracle.REF_BIN_O2):
        frames, _ = oracle.run_ref(cfg, scene["projection"], kw["width"], kw["height"], binary=binary)
        assert np.array_equal(frames[0], fb)


FLY_SCENE = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
FLY_STATES = [dict(pos=(-0.6, 0.6, 3.2), hang_deg=-45.0), dict(pos=(-0.2, 0.9, 3.0), hang_deg=-60.0),
              dict(pos=(0.4, 1.0, 2.8), hang_deg=-80.0)]


def flythrough_oracle_frames(oracle, maps):
    return [H.oracle_render_scene(oracle, dict(FLY_SCENE, **s), maps)[0] for s in FLY_STATES]


def test_reference_scripted_flythrough_matches_oracle(oracle, tmp_path):
    """Console-driven camera changes in the unmodified reference (main/hmap.cpp:760-804) reproduce
    per-frame oracle renders (each state rendered twice because of the one-frame look/up lag): against the
    reference's recorded frames, and rendered now where oracle/_ref is built."""
    hm, cm = H.load_scene_maps(FLY_SCENE, oracle)
    want = flythrough_oracle_frames(oracle, (hm, cm))
    assert [H.sha(fb) for fb in want] == H.golden_replays()["flythrough"]
    if not oracle.have_ref():
        return
    oracle.write_png(tmp_path / "h.png", hm)
    oracle.write_png(tmp_path / "c.png", cm)
    kw = S.frame_kwargs(FLY_SCENE)
    cfg = oracle.config_text(kw, tmp_path / "h.png", tmp_path / "c.png", lum=FLY_SCENE["lum"])
    script = ["pos %r %r %r hang %r" % (*s["pos"], s["hang_deg"]) for s in FLY_STATES]
    frames, _ = oracle.run_ref(cfg, 1, kw["width"], kw["height"], script=script)
    for got, fb in zip(frames, want):
        assert np.array_equal(got, fb)


def random_scene(rng, i):
    """A random small scene: any projection, camera anywhere around (or inside, or below) the box, any look direction,
    random luminance weights / height range / step / background."""
    maps = [S.SYNTH8, S.NOISE, S.CROP][i % 3]
    extent = 2.56 if maps is S.SYNTH8 else 2.0
    lo = float(rng.uniform(-1.0, 1.0))
    return S._scene(f"random_{i}", 1 + i % 3, maps, width=int(rng.integers(24, 97)), height=int(rng.integers(16, 55)),
                    pos=(float(rng.uniform(-1.5, extent + 1.5)), float(rng.uniform(-extent - 1.5, 1.5)), float(rng.uniform(-1.0, 5.0))),
                    hang_deg=float(rng.uniform(-180.0, 180.0)), vang_deg=float(rng.uniform(5.0, 175.0)),
                    hfov_deg=float(rng.uniform(20.0, 150.0)), grid_width=float(rng.choice([0.01, 0.013, 0.02])),
                    step_dist=float(rng.choice([0.05, 0.02, 0.004, 0.11])), ortho_width=float(rng.uniform(0.005, 0.05)),
                    min_height=lo, max_height=lo + float(rng.uniform(0.2, 3.0)),
                    lum=tuple(float(v) for v in rng.uniform(-0.3, 1.2, size=3)), bg=tuple(int(v) for v in rng.integers(0, 256, size=3)))


def random_scenes():
    rng = np.random.default_rng(424242)
    return [random_scene(rng, i) for i in range(18)]


def test_oracle_matches_live_reference_on_random_scenes(oracle, tmp_path):
    """The restatement against the unmodified reference on 18 random scenes beyond the committed golden frames: against
    the reference's recorded frames, and rendered now where oracle/_ref is built."""
    recorded = H.golden_replays()["random_scenes"]
    assert len(recorded) == 18
    for scene, want_sha in zip(random_scenes(), recorded):
        hm, cm = H.load_scene_maps(scene, oracle)
        fb, _, _ = H.oracle_render_scene(oracle, scene, (hm, cm))
        assert H.sha(fb) == want_sha, scene
        if not oracle.have_ref():
            continue
        oracle.write_png(tmp_path / "h.png", hm)
        oracle.write_png(tmp_path / "c.png", cm)
        kw = S.frame_kwargs(scene)
        cfg = oracle.config_text(kw, tmp_path / "h.png", tmp_path / "c.png", lum=scene["lum"])
        frames, _ = oracle.run_ref(cfg, scene["projection"], kw["width"], kw["height"], binary=oracle.REF_BIN_O2)
        assert np.array_equal(frames[0], fb), scene
