"""GPU: many cameras in one launch (hmrm_render_views / hmrm_render_views_device, k2_render_lin with kViews).  Every
view must equal the CPU oracle's frame of that camera byte for byte; views of very different cost (grazing, sky, a
total miss, from below the terrain, inside the box) share each batch, and the shapes put partial tiles and partial tile
rows at view boundaries."""
import ctypes as C
import functools
import math

import numpy as np
import pytest

import helpers as H
import scenes as S

pytestmark = pytest.mark.gpu

# cameras of scenes with very different costs per ray: (scene whose pos / hang / vang is taken)
MIX = ["persp_graze", "looking_up_sky", "looking_down_miss", "from_below", "camera_inside_box", "persp_basic"]


@functools.lru_cache(maxsize=None)
def _maps(oracle, name):
    return H.load_scene_maps(S.SCENE_BY_NAME[name], oracle)


@functools.lru_cache(maxsize=None)
def _heights(oracle, name):
    sc = S.SCENE_BY_NAME[name]
    return oracle.update_heightmap(_maps(oracle, name)[0], sc["lum"], sc["min_height"], sc["max_height"])


def _configure(renderer, oracle, name):
    H.configure(renderer, S.SCENE_BY_NAME[name], _maps(oracle, name))


def cam_of(oracle, name, dx=0.0, dhang=0.0):
    sc = S.SCENE_BY_NAME[name]
    x, y, z = (float(v) for v in sc["pos"])
    return (x + dx, y, z, oracle.deg2rad(sc["hang_deg"]) + dhang, oracle.deg2rad(sc["vang_deg"]))


def mix_cams(oracle, n):
    """n cameras cycling through MIX, each pass moved a little so that no two are the same."""
    return [cam_of(oracle, MIX[j % len(MIX)], dx=0.013 * (j // len(MIX)), dhang=0.011 * (j // len(MIX)))
            for j in range(n)]


@functools.lru_cache(maxsize=None)
def _oracle_view(oracle, name, w, h, cam):
    """The oracle's RGBA8 frame and statistics of scene `name` at size w x h and camera cam = (x, y, z, hang, vang)."""
    kw = S.frame_kwargs(S.SCENE_BY_NAME[name])
    for k in ("pos", "hang_deg", "vang_deg", "width", "height"):
        kw.pop(k)
    f = oracle.make_frame(projection=S.SCENE_BY_NAME[name]["projection"], width=w, height=h, pos=cam[:3], hang=cam[3],
                          vang=cam[4], **kw)
    fb, _, st = oracle.render(f, _heights(oracle, name), _maps(oracle, name)[1], want_steps=False)
    return fb, st


def expected(oracle, name, w, h, cams, channels=4):
    return np.stack([_oracle_view(oracle, name, w, h, tuple(c))[0][:, :, :channels] for c in cams])


def _frame(hmrm, renderer, name, w, h, **extra):
    return H.product_frame(hmrm, renderer, dict(S.SCENE_BY_NAME[name], width=w, height=h), **extra)


def _assert_views(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = np.argwhere((got != want).any(axis=-1))
    assert bad.size == 0, f"{what}: {len(bad)} pixels differ, first at (view, y, x) = {tuple(bad[0])}"


def _plain(hmrm, renderer, f, cam, flags=0):
    """hmrm_render of f at one camera (a copy of the frame, f itself unchanged)."""
    g = type(f).from_buffer_copy(f)
    g.cam_pos[:] = list(cam[:3])
    g.hang, g.vang = cam[3], cam[4]
    g.flags = flags
    return renderer.render(g).copy()


# ---- 1. scenes of all three projections, views of very different costs, RGBA8 and RGB8 ----
@pytest.mark.parametrize("name", ["persp_basic", "spher_basic", "ortho_basic", "spher_fine", "noise_lum", "crop_ortho",
                                  "defaults_grid"])
def test_views_equal_oracle(hmrm, renderer, oracle, name):
    _configure(renderer, oracle, name)
    w, h = 37, 21                 # W % 8, W % 4, H % 4 != 0; W * H * 3 = 3 (mod 4): RGB8 views take all four alignments
    cams = mix_cams(oracle, 12)
    want = expected(oracle, name, w, h, cams)
    for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
        got = renderer.render_views(np.array(cams), _frame(hmrm, renderer, name, w, h, pixel_format=fmt))
        _assert_views(got, want[..., :ch], f"{name} channels={ch}")


# ---- 2. device destinations at byte offsets 0..3 with canaries; n = 1, a few, and a batch above 100000 tiles ----
# (W % 4 == 0 with RGB8: whole tile rows go out as 32-bit words where the view's base is 4-aligned, byte by byte
# elsewhere; W * H * 3 is then a multiple of 4, so all views of a batch share the alignment of the buffer offset)
@pytest.mark.parametrize("w,h,n", [(37, 21, 1), (37, 21, 7), (13, 6, 5), (61, 35, 5), (40, 21, 6), (64, 13, 9),
                                   (37, 21, 3400)])
def test_device_offsets_shapes_and_large_batches(hmrm, renderer, oracle, w, h, n):
    import torch

    name = "persp_basic"
    _configure(renderer, oracle, name)
    if n > 100:
        assert n * ((w + 7) // 8) * ((h + 3) // 4) >= 100000   # the batch runs the large-launch shape
    cams = mix_cams(oracle, min(n, 24))
    cams = [cams[j % len(cams)] for j in range(n)]
    want = expected(oracle, name, w, h, cams)
    guard = 64
    for ch in (4, 3):
        f = _frame(hmrm, renderer, name, w, h, pixel_format=hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8)
        size = n * h * w * ch
        for off in range(4):
            buf = torch.full((2 * guard + off + size,), 0xA5, dtype=torch.uint8, device="cuda:0")
            renderer.render_views_device(f, np.array(cams), buf.data_ptr() + guard + off)
            renderer.wait()
            torch.cuda.synchronize()
            b = buf.cpu().numpy()
            what = f"{w}x{h} n={n} channels={ch} offset={off}"
            assert (b[:guard + off] == 0xA5).all() and (b[guard + off + size:] == 0xA5).all(), what + " canary"
            _assert_views(b[guard + off:guard + off + size].reshape(n, h, w, ch), want[..., :ch], what)


def test_one_view_of_the_frames_own_camera_is_hmrm_render(hmrm, renderer, oracle):
    for name in ("persp_graze", "spher_wide", "ortho_fine"):
        _configure(renderer, oracle, name)
        sc = S.SCENE_BY_NAME[name]
        f = H.product_frame(hmrm, renderer, sc)
        cam = (*f.cam_pos, f.hang, f.vang)
        for fmt in (hmrm.PIXEL_RGBA8, hmrm.PIXEL_RGB8):
            f.pixel_format = fmt
            plain = renderer.render(f).copy()
            _assert_views(renderer.render_views(np.array([cam]), f), plain[None], f"{name} format {fmt}")


# ---- 3. pyramid layouts and 16-bit maps ----
def test_every_layout(hmrm, renderer, oracle):
    name = "spher_fine"
    _configure(renderer, oracle, name)
    w, h = 45, 27
    cams = mix_cams(oracle, 9)
    want = expected(oracle, name, w, h, cams)
    before = renderer.get_layout()
    try:
        for layout in (hmrm.LAYOUT_ROWMAJOR, hmrm.LAYOUT_TILE4, hmrm.LAYOUT_ZORDER):
            renderer.set_layout(layout)
            _assert_views(renderer.render_views(np.array(cams), _frame(hmrm, renderer, name, w, h)), want, f"layout {layout}")
    finally:
        renderer.set_layout(before)


def test_16_bit_map(hmrm, renderer, oracle):
    import height16_lib as H16

    sc = dict(S.SCENE_BY_NAME["persp_basic"], width=53, height=30)
    x, cm = H16.synth_maps16(8, 1234)
    heights = H16.heights16(x, sc["lum"], sc["min_height"], sc["max_height"])
    renderer.lum_r, renderer.lum_g, renderer.lum_b = sc["lum"]
    renderer.min_height, renderer.max_height = sc["min_height"], sc["max_height"]
    renderer.synth_maps16(8, 1234)
    cams = mix_cams(oracle, 8)
    want = []
    for c in cams:
        f = oracle.make_frame(projection=1, width=53, height=30, pos=c[:3], hang=c[3], vang=c[4],
                              hfov_deg=sc["hfov_deg"], grid_width=sc["grid_width"], step_dist=sc["step_dist"],
                              ortho_width=sc["ortho_width"], min_height=sc["min_height"], max_height=sc["max_height"])
        want.append(oracle.render(f, heights, cm, want_steps=False)[0])
    _assert_views(renderer.render_views(np.array(cams), H.product_frame(hmrm, renderer, sc)), np.stack(want), "16-bit map")


# ---- 4. statistics ----
@pytest.mark.parametrize("name", ["persp_basic", "spher_fine", "ortho_basic"])
def test_stats_are_sums_over_views(hmrm, renderer, oracle, name):
    _configure(renderer, oracle, name)
    w, h = 37, 21
    cams = mix_cams(oracle, 10)
    renderer.render_views(np.array(cams), _frame(hmrm, renderer, name, w, h, flags=hmrm.FLAG_STATS))
    st = renderer.stats()
    ost = [_oracle_view(oracle, name, w, h, tuple(c))[1] for c in cams]
    assert st.rays == len(cams) * w * h
    assert st.steps == sum(o.steps for o in ost)
    assert (st.box_hits, st.surf_hits) == (sum(o.box_hits for o in ost), sum(o.surf_hits for o in ost))
    assert st.max_steps == max(o.max_steps for o in ost)
    assert st.status == 0 and st.kernel_ms > 0.0
    # per-view hmrm_render statistics add up to the batch's, fetches included
    f = _frame(hmrm, renderer, name, w, h)
    fetches = 0
    for c in cams:
        _plain(hmrm, renderer, f, c, hmrm.FLAG_STATS)
        fetches += renderer.stats().fetches
    assert st.fetches == fetches
    # after a batch there is no step index or ray dump, even when the render before it had both
    lib = hmrm.load_library()
    out = np.zeros(w * h * 10, dtype=np.float64)
    _plain(hmrm, renderer, f, cams[0], hmrm.FLAG_STEP_INDEX | hmrm.FLAG_RAY_DUMP)
    assert lib.hmrm_get_step_index(renderer._h, out.ctypes.data) == 0
    renderer.render_views(np.array(cams), _frame(hmrm, renderer, name, w, h, flags=hmrm.FLAG_STATS))
    assert lib.hmrm_get_step_index(renderer._h, out.ctypes.data) == 3
    assert lib.hmrm_get_ray_dump(renderer._h, out.ctypes.data) == 3


def test_nonterminating_view_is_flagged_and_the_others_stay_exact(hmrm, renderer):
    hm = np.zeros((32, 32, 3), dtype=np.uint8)
    cm = np.full((32, 32, 4), 255, dtype=np.uint8)
    renderer.lum_r, renderer.lum_g, renderer.lum_b = 0.0, 0.0, 0.0
    renderer.min_height, renderer.max_height = 0.0, 10.0
    renderer.set_maps(hm, cm)
    f = renderer.frame(projection=3, screen_width=16, screen_height=8, ortho_width=0.01, grid_width=0.05,
                       step_dist=0.25, flags=hmrm.FLAG_STATS)
    stuck = (0.8, -0.8, -3.0, 0.0, 0.0)          # straight up under a flat terrain: never leaves the grid
    others = [(0.8, -0.8, 3.0, 0.0, math.pi), (0.5, -0.5, 2.0, 0.3, 2.5), (-1.0, 1.0, 1.0, -0.7, 2.2)]
    cams = [others[0], stuck, others[1], others[2]]
    got = renderer.render_views(np.array(cams), f).copy()
    assert renderer.stats().status == 4          # HMRM_ERR_NONTERMINATING
    for j, c in enumerate(cams):
        if c is not stuck:
            _assert_views(got[j:j + 1], _plain(hmrm, renderer, f, c)[None], f"view {j}")
    assert (got[..., 3] == 255).all()


# ---- 5. refusals: the code, nothing written, the context still renders ----
def test_refusals(hmrm, renderer, oracle):
    import torch

    name = "persp_basic"
    _configure(renderer, oracle, name)
    lib = hmrm.load_library()
    w, h = 37, 21
    cams = mix_cams(oracle, 3)
    arr = (hmrm.Camera * 3)()
    for i, c in enumerate(cams):
        arr[i].cam_pos[:] = list(c[:3])
        arr[i].hang, arr[i].vang = c[3], c[4]
    host = np.full(3 * h * w * 4, 0xA5, dtype=np.uint8)
    dev = torch.full((3 * h * w * 4,), 0xA5, dtype=torch.uint8, device="cuda:0")

    def calls(f, cams_arr=arr, n=3, out_host=None, out_dev=None):
        fp = C.byref(f) if f is not None else None
        return [lib.hmrm_render_views(renderer._h, fp, cams_arr, n, host.ctypes.data if out_host is None else out_host),
                lib.hmrm_render_views_device(renderer._h, fp, cams_arr, n, dev.data_ptr() if out_dev is None else out_dev,
                                             None)]

    def frame(**kw):
        return _frame(hmrm, renderer, name, w, h, **kw)

    invalid = {
        "cycle_period 3": (frame(cycle_period=3),),
        "band_count 2": (frame(band_count=2, band_index=0),),
        "row band": (frame(row_begin=0, row_end=h // 2),),
        "step index": (frame(flags=hmrm.FLAG_STEP_INDEX),),
        "ray dump": (frame(flags=hmrm.FLAG_RAY_DUMP),),
        "supersample 2": (frame(flags=hmrm.supersample_flag(2)),),
        "traversal brute": (frame(traversal=hmrm.TRAVERSAL_BRUTE),),
        "traversal fp64 skip": (frame(traversal=hmrm.TRAVERSAL_SKIP_FP64),),
        "traversal pack": (frame(traversal=hmrm.TRAVERSAL_PACK),),
        "traversal 9": (frame(traversal=9),),
        "NULL frame": (None,),
        "resolution 1": (frame(screen_width=1),),
        "tiny grid_width": (frame(grid_width=1e-306, step_dist=1e-306),),
        "n 0": (frame(), arr, 0),
        "n 65537": (frame(), arr, 65537),
        "NULL cams": (frame(), None, 3),
        "NULL output": (frame(), arr, 3, 0, 0),
    }
    for what, args in invalid.items():
        assert calls(*args) == [1, 1], what
    bad = (hmrm.Camera * 3)()
    for field in ("x", "hang", "vang"):
        C.memmove(bad, arr, C.sizeof(arr))
        if field == "x":
            bad[2].cam_pos[0] = math.inf
        else:
            setattr(bad[1], field, math.nan)
        assert calls(frame(), bad) == [1, 1], f"non-finite {field}"
    # more than 2^26 tiles: 65536 views of 8200 x 4 are 65536 * 1025 tiles
    many = (hmrm.Camera * 65536)()
    for j in range(65536):
        C.memmove(C.byref(many, j * C.sizeof(hmrm.Camera)), arr, C.sizeof(hmrm.Camera))
    assert calls(frame(screen_width=8200, screen_height=4), many, 65536) == [1, 1]
    assert b"2^26" in lib.hmrm_last_error(renderer._h)
    renderer.set_motion_blur([(cams[0][:3], cams[0][3], cams[0][4])])
    try:
        assert calls(frame()) == [1, 1], "motion blur set"
    finally:
        renderer.set_motion_blur([])
    torch.cuda.synchronize()
    assert (host == 0xA5).all() and (dev.cpu().numpy() == 0xA5).all()
    _assert_views(renderer.render_views(np.array(cams), frame()), expected(oracle, name, w, h, cams), "after the refusals")


def test_unquantisable_maps_are_a_state_error(hmrm, oracle, monkeypatch):
    """A height range the 16-bit quantiser cannot map (forced through the HMRM_ZQ_RANGE_SHRINK test hook, read when
    the context is created): no skip traversal, so views are refused with HMRM_ERR_STATE, nothing is written, and
    the context still renders plain frames (with the brute traversal)."""
    import torch

    monkeypatch.setenv("HMRM_ZQ_RANGE_SHRINK", "inf")
    name = "persp_basic"
    r = hmrm.Renderer(0)
    try:
        _configure(r, oracle, name)
        lib = hmrm.load_library()
        w, h = 37, 21
        cams = mix_cams(oracle, 3)
        n = len(cams)
        arr = (hmrm.Camera * n)()
        for i, c in enumerate(cams):
            arr[i].cam_pos[:] = list(c[:3])
            arr[i].hang, arr[i].vang = c[3], c[4]
        host = np.full(n * h * w * 4, 0xA5, dtype=np.uint8)
        dev = torch.full((n * h * w * 4,), 0xA5, dtype=torch.uint8, device="cuda:0")
        f = _frame(hmrm, r, name, w, h)
        assert lib.hmrm_render_views(r._h, C.byref(f), arr, n, host.ctypes.data) == 3
        assert b"quantised" in lib.hmrm_last_error(r._h)
        assert lib.hmrm_render_views_device(r._h, C.byref(f), arr, n, dev.data_ptr(), None) == 3
        torch.cuda.synchronize()
        assert (host == 0xA5).all() and (dev.cpu().numpy() == 0xA5).all()
        for j, c in enumerate(cams):
            _assert_views(_plain(hmrm, r, f, c)[None], expected(oracle, name, w, h, [c]), f"plain frame {j} afterwards")
    finally:
        r.close()


# ---- 6. interplay with the frame ring, and batches that grow and shrink ----
def test_batches_between_frames_in_flight_and_changing_n(hmrm, renderer, oracle):
    name = "persp_basic"
    _configure(renderer, oracle, name)
    w, h = 61, 35
    frames = [hmrm.pinned_empty((h, w, 4)) for _ in range(4)]
    ring_cams = mix_cams(oracle, 4)
    f = _frame(hmrm, renderer, name, w, h)
    for i, c in enumerate(ring_cams):
        g = type(f).from_buffer_copy(f)
        g.cam_pos[:] = list(c[:3])
        g.hang, g.vang = c[3], c[4]
        renderer.render_async(g, frames[i])
    cams = mix_cams(oracle, 18)
    got = renderer.render_views(np.array(cams), f).copy()
    renderer.wait()
    for i, c in enumerate(ring_cams):
        _assert_views(frames[i][None], expected(oracle, name, w, h, [c]), f"ring frame {i}")
    _assert_views(got, expected(oracle, name, w, h, cams), "batch between ring frames")
    for n in (1, 18, 300, 2, 40, 1):
        cs = [cams[j % len(cams)] for j in range(n)]
        for fmt, ch in ((hmrm.PIXEL_RGB8, 3), (hmrm.PIXEL_RGBA8, 4)):
            got = renderer.render_views(np.array(cs), _frame(hmrm, renderer, name, w, h, pixel_format=fmt))
            _assert_views(got, expected(oracle, name, w, h, cs, ch), f"n={n} channels={ch}")


# ---- 7. the binding ----
def test_binding_forms_and_shape_errors(hmrm, renderer, oracle):
    import torch

    name = "spher_basic"
    _configure(renderer, oracle, name)
    w, h = 40, 24
    cams = mix_cams(oracle, 5)
    want = expected(oracle, name, w, h, cams)
    f = _frame(hmrm, renderer, name, w, h)
    _assert_views(renderer.render_views(np.array(cams, dtype=np.float64), f), want, "[n, 5] array")
    _assert_views(renderer.render_views([(c[:3], c[3], c[4]) for c in cams], f), want, "(pos, hang, vang)")
    _assert_views(renderer.render_views([list(c) for c in cams], f), want, "a list of five-number rows")
    out = np.zeros((5, h, w, 4), dtype=np.uint8)
    assert renderer.render_views(np.array(cams), f, out=out) is not None and np.array_equal(out, want)
    t = torch.zeros((5, h, w, 4), dtype=torch.uint8, device="cuda:0")
    st = torch.cuda.Stream()
    renderer.render_views_device(f, np.array(cams), t, st.cuda_stream)
    st.synchronize()
    _assert_views(t.cpu().numpy(), want, "torch tensor on a caller's stream")
    small = torch.full((5 * h * w * 4 - 1,), 7, dtype=torch.uint8, device="cuda:0")
    for bad_call in (lambda: renderer.render_views(np.zeros((3, 4)), f),
                     lambda: renderer.render_views([((0.0, 1.0), 0.0, 0.0)], f),
                     lambda: renderer.render_views_device(f, np.zeros((2, 6)), t),
                     lambda: renderer.render_views_device(f, np.array(cams), small),
                     lambda: renderer.render_views(np.array(cams), f, out=np.zeros((4, h, w, 4), dtype=np.uint8))):
        with pytest.raises(ValueError):
            bad_call()
    torch.cuda.synchronize()
    assert (small.cpu().numpy() == 7).all()
