"""GPU: the last step of every render call — where its pixels go.

Every destination is an allocation filled with sentinel bytes (never 0 or 255), with at least 64 guard bytes before
and after the frame.  The expected allocation is the fill with the CPU oracle's bytes written at exactly the pixels the
selection model (tests/destinations_model.py, checked on the CPU by tests/test_destinations_model.py) says the call
writes; every byte of the allocation is compared, guards included.  Nothing the device computed feeds an expectation.

Covered: hmrm_render_device at byte offsets 0, 1, 2, 3, 4, 8 and 12 (the context's stream and a caller's), hmrm_render
and hmrm_render_async into host memory at offsets 0 to 3, RGBA8 and RGB8, all four traversals, row bands, interleaved
bands, the progressive interleave and their combinations, supersample factors 2 to 4, peer frames at unaligned
offsets, and frames at the 65536-pixel axis limit (up to 65536 x 16384, 4 GiB)."""
import functools

import numpy as np
import pytest

import destinations_model as M
import helpers as H
import scenes as S
from test_png_encode import check_png
from test_supersample import box_reduce
from test_yuv420 import BT601, BT709, yuv420_model

pytestmark = pytest.mark.gpu

GUARD = 64
DEVICE_OFFSETS = (0, 1, 2, 3, 4, 8, 12)
HOST_OFFSETS = (0, 1, 2, 3)
WIDTHS = tuple(range(2, 18)) + (31, 32, 33, 63, 65)          # every W mod 8 and W mod 4
HEIGHTS = tuple(range(2, 10)) + (11, 13, 15, 17, 23, 25)     # ragged last tile rows: 4k +- 1
TRAVERSALS = {"brute": 1, "skip": 2, "skip_fp64": 3, "pack": 4}
PERIODS = (1, 2, 3, 7, 47)
DESTS = ("device", "device_stream", "host", "host_async")
DEVICE_KINDS = ("whole", "rows", "bands", "cycle", "rows+bands", "rows+cycle", "rows+bands+cycle")
# the host copy-out writes whole rows of the band; the header leaves the progressive interleave there unspecified
HOST_KINDS = ("whole", "rows", "bands", "rows+bands")
N_CASES = 640

# the scenes' maps plus one more non-square noise map
NOISE_SMALL = dict(S.SCENE_BY_NAME["noise_lum"], name="noise_77x45", maps=dict(kind="noise", w=77, h=45, seed=11),
                   pos=(-0.3, 0.3, 1.4), vang_deg=110.0)
SCENES = {s["name"]: s for s in S.SCENES + [NOISE_SMALL]}


@functools.lru_cache(maxsize=None)
def _maps(oracle, name):
    return H.load_scene_maps(SCENES[name], oracle)


class _Configured:
    """The renderer's maps follow the scene of the case; set_maps only when the scene changes."""

    def __init__(self, renderer, oracle):
        self.r, self.oracle, self.name = renderer, oracle, None

    def __call__(self, name):
        if name != self.name:
            H.configure(self.r, SCENES[name], _maps(self.oracle, name))
            self.name = name


def _oracle(oracle, scene, s=1):
    """The oracle's W x H frame of `scene` (the box filter of its sW x sH frame for s > 1) and its statistics."""
    big = dict(scene, width=scene["width"] * s, height=scene["height"] * s)
    fb, _, st = H.oracle_render_scene(oracle, big, _maps(oracle, scene["name"]))
    return (fb if s == 1 else box_reduce(fb, s, 4)), st


def _assert_bytes(got, want, what, start, shape):
    """Every byte of the allocation; on failure, where the first wrong byte is (guard or pixel)."""
    if np.array_equal(got, want):
        return
    bad = np.nonzero(got != want)[0]
    i = int(bad[0])
    h, w, ch = shape
    if i < start or i >= start + h * w * ch:
        where = f"guard byte {i - start if i < start else i - (start + h * w * ch)} {'before' if i < start else 'after'}"
    else:
        p = (i - start) // ch
        where = f"pixel (x {p % w}, y {p // w}) byte {(i - start) % ch}"
    pytest.fail(f"{what}: {bad.size} bytes differ, first at {where}: got {got[i]}, want {want[i]}")


# ---- 1. sampled cases: shapes x cameras x destinations x offsets x formats x traversals x selections ----
def _selection(rng, kind, h):
    sel = dict(row_begin=0, row_end=0, band_count=0, band_index=0, cycle=0, cycle_period=1)
    if "rows" in kind:
        rb = int(rng.choice([r for r in range(1, h) if r % 4] or [1]))
        sel.update(row_begin=rb, row_end=int(rng.integers(rb + 1, h + 1)))
    if "bands" in kind:
        n = int(rng.integers(1, 6))
        # the last band often owns no tile row of a short band
        b = n - 1 if rng.random() < 0.3 else int(rng.integers(0, n))
        sel.update(band_count=n, band_index=b)
    if "cycle" in kind:
        period = int(rng.choice(PERIODS))
        sel.update(cycle_period=period, cycle=int(rng.integers(0, period)))
    return sel


def _cases():
    rng = np.random.default_rng(20261021)
    names = sorted(SCENES)
    cases = []
    for i in range(N_CASES):
        dest = DESTS[i % 4]
        device = dest.startswith("device")
        scene = SCENES[names[int(rng.integers(0, len(names)))]]
        w, h = int(rng.choice(WIDTHS)), int(rng.choice(HEIGHTS))
        bg = [scene["bg"], (0, 0, 0), tuple(int(v) for v in rng.integers(0, 256, 3))][int(rng.integers(0, 3))]
        kinds = DEVICE_KINDS if device else HOST_KINDS
        kind = kinds[int(rng.integers(0, len(kinds)))]
        s = int(rng.choice([2, 3, 4])) if kind == "whole" and rng.random() < 0.4 else 1
        cases.append(dict(
            i=i, dest=dest, scene=dict(scene, width=w, height=h, bg=bg), kind=kind, s=s,
            traversal=list(TRAVERSALS)[(i // 4) % 4], channels=(4, 3)[(i // 16) % 2],
            offset=int(rng.choice(DEVICE_OFFSETS if device else HOST_OFFSETS)),
            sel=_selection(rng, kind, h), seed=int(rng.integers(0, 2**31))))
    return sorted(cases, key=lambda c: c["scene"]["name"])


def test_sampled_destinations_match_oracle(hmrm, renderer, oracle):
    import torch

    configure = _Configured(renderer, oracle)
    stream = torch.cuda.Stream(device=0)
    pinned = hmrm.pinned_empty((2 * GUARD + 16 + 65 * 25 * 4,))
    seen = {k: set() for k in ("device_offsets", "host_offsets", "w_mod_8", "traversal", "device_kind", "host_kind",
                               "period", "band_count", "s_device", "s_host", "unaligned_ss")}
    empty_band = rays = misses = surf = sky_in_box = black_sky = 0
    for c in _cases():
        scene, sel, ch, off = c["scene"], c["sel"], c["channels"], c["offset"]
        w, h = scene["width"], scene["height"]
        configure(scene["name"])
        frame, st = _oracle(oracle, scene, c["s"])
        mask = M.selected(w, h, sel["row_begin"], sel["row_end"], sel["band_count"], sel["band_index"], sel["cycle"],
                          sel["cycle_period"])
        start = GUARD + off
        fill = M.sentinel_bytes(np.random.default_rng(c["seed"]), start + h * w * ch + GUARD)
        want = M.expected_destination(fill, start, frame, mask, ch)
        f = H.product_frame(hmrm, renderer, scene, traversal=TRAVERSALS[c["traversal"]],
                            pixel_format=hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8,
                            flags=hmrm.supersample_flag(c["s"]), **sel)
        if c["dest"].startswith("device"):
            buf = torch.from_numpy(fill).to("cuda:0")
            torch.cuda.synchronize()
            assert (buf.data_ptr() + start) % 4 == off % 4
            if c["dest"] == "device":
                renderer.render_device(f, buf.data_ptr() + start)
                renderer.wait()
            else:
                renderer.render_device(f, buf.data_ptr() + start, stream.cuda_stream)
                stream.synchronize()
            got = buf.cpu().numpy()
        elif c["dest"] == "host":
            got = fill.copy()
            assert got.ctypes.data % 4 == 0
            renderer.render(f, out=got[start:start + h * w * ch].reshape(h, w, ch))
        else:
            got = pinned[:fill.size]
            got[:] = fill
            renderer.render_async(f, got[start:])
            renderer.wait()
            got = got.copy()
        assert renderer.stats().status == 0, c
        what = (f"case {c['i']} {c['dest']} offset {off} {scene['name']} {w}x{h} bg {scene['bg']} channels {ch} "
                f"{c['traversal']} {c['kind']} {sel} s={c['s']}")
        _assert_bytes(got, want, what, start, (h, w, ch))

        device = c["dest"].startswith("device")
        seen["device_offsets" if device else "host_offsets"].add((off, ch))
        seen["w_mod_8"].add(w % 8)
        seen["traversal"].add(c["traversal"])
        seen["device_kind" if device else "host_kind"].add(c["kind"])
        seen["period"].add(sel["cycle_period"])
        seen["band_count"].add(sel["band_count"])
        if c["s"] > 1:
            seen["s_device" if device else "s_host"].add(c["s"])
            if off % 4:
                seen["unaligned_ss"].add(ch)
        empty_band += sel["band_count"] > 1 and not mask.any()
        rays += st.rays
        misses += st.rays - st.box_hits
        surf += st.surf_hits
        sky_in_box += st.box_hits - st.surf_hits
        black_sky += tuple(scene["bg"]) == (0, 0, 0) and st.rays > st.surf_hits

    # the sample reached every dimension it is meant to cover
    assert seen["device_offsets"] == {(o, ch) for o in DEVICE_OFFSETS for ch in (3, 4)}
    assert seen["host_offsets"] == {(o, ch) for o in HOST_OFFSETS for ch in (3, 4)}
    assert seen["w_mod_8"] == set(range(8))
    assert seen["traversal"] == set(TRAVERSALS)
    assert seen["device_kind"] == set(DEVICE_KINDS) and seen["host_kind"] == set(HOST_KINDS)
    assert seen["period"] == set(PERIODS) and seen["band_count"] >= {1, 2, 3, 4, 5}
    assert seen["s_device"] == seen["s_host"] == {2, 3, 4} and seen["unaligned_ss"] == {3, 4}
    assert empty_band > 0
    assert misses > 0 and surf > 0 and sky_in_box > 0 and black_sky > 0, (rays, misses, surf, sky_in_box, black_sky)


# ---- 2. peer frames into unaligned device frames: emulated ranks in one stream ----
@pytest.mark.parametrize("offset", [1, 2, 3])
def test_peer_frames_at_unaligned_offsets(hmrm, renderer, oracle, offset):
    """hmrm_render_peer and hmrm_render_peer_staged (ranks 0, 2 and 1 of three) into d_frame and d_stage at `offset`
    bytes past a 4-byte boundary.  As in test_gpu_peer_frame.py, every call is in ONE stream, so every device-side wait
    is already satisfied by work earlier in that stream and nothing spins on another launch."""
    import torch

    ranks = 3
    configure = _Configured(renderer, oracle)
    stream = torch.cuda.Stream(device=0)
    ctrl = renderer.device_alloc(256)            # zero-filled: arrived = released = error = 0
    rng = np.random.default_rng(offset)
    use = 0
    try:
        for name, w, h in (("persp_basic", 61, 23), ("spher_fine", 64, 18), ("ortho_basic", 35, 9)):
            configure(name)
            scene = dict(SCENES[name], width=w, height=h)
            frame, _ = _oracle(oracle, scene)
            for ch in (4, 3):
                for trav in TRAVERSALS:
                    use += 1
                    start = GUARD + offset
                    fill = M.sentinel_bytes(rng, start + h * w * ch + GUARD)
                    stage_fill = M.sentinel_bytes(rng, fill.size)
                    d_frame = torch.from_numpy(fill).to("cuda:0")
                    d_stage = torch.from_numpy(stage_fill).to("cuda:0")
                    torch.cuda.synchronize()
                    for rk in (2, 0, 1):
                        f = H.product_frame(hmrm, renderer, scene, band_count=ranks, band_index=rk,
                                            traversal=TRAVERSALS[trav],
                                            pixel_format=hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8)
                        if rk == 1:
                            renderer.render_peer_staged(f, d_stage.data_ptr() + start, d_frame.data_ptr() + start, ctrl,
                                                        use, stream.cuda_stream)
                        else:
                            renderer.render_peer(f, d_frame.data_ptr() + start, ctrl, use, stream.cuda_stream)
                        assert renderer.stats().status == 0
                    renderer.peer_wait(ctrl, use, ranks, stream.cuda_stream)
                    renderer.peer_release(ctrl, use, stream.cuda_stream)
                    stream.synchronize()
                    what = f"{name} {w}x{h} channels {ch} {trav} offset {offset}"
                    _assert_bytes(d_frame.cpu().numpy(), M.expected_destination(fill, start, frame, np.ones((h, w), bool), ch),
                                  what + " d_frame", start, (h, w, ch))
                    band1 = M.selected(w, h, band_count=ranks, band_index=1)
                    _assert_bytes(d_stage.cpu().numpy(), M.expected_destination(stage_fill, start, frame, band1, ch),
                                  what + " d_stage", start, (h, w, ch))
        _, released, error = renderer.peer_status(ctrl)
        assert (released, error) == (use, 0)
    finally:
        renderer.device_free(ctrl)


# ---- 3. frames at the size limits ----
@pytest.mark.parametrize("w,h", [(65536, 2), (2, 65536)])
def test_axis_limit_frames_match_oracle(hmrm, renderer, oracle, w, h):
    """tiles_x = 8192 with one tile row, and tiles_x = 1 with 16384 tile rows: tile_row_col's float quotient, the
    reciprocal 1 / tiles_x, and pack's (py << 16) | px pixel word at px or py = 65535.  Every pixel, every traversal,
    RGBA8 and RGB8, at offsets 0 to 3."""
    import torch

    configure = _Configured(renderer, oracle)
    hits = 0
    for name in ("persp_basic", "spher_basic", "ortho_basic"):
        configure(name)
        # (a narrower field of view turns the two columns of the tall frame towards the terrain)
        scene = dict(SCENES[name], width=w, height=h, **({"hfov_deg": 20.0} if w == 2 else {}))
        frame, st = _oracle(oracle, scene)
        hits += st.surf_hits
        for i, trav in enumerate(TRAVERSALS):
            for ch in (4, 3):
                off = (i + ch) % 4
                start = GUARD + off
                fill = M.sentinel_bytes(np.random.default_rng(i * 8 + ch), start + h * w * ch + GUARD)
                buf = torch.from_numpy(fill).to("cuda:0")
                torch.cuda.synchronize()
                f = H.product_frame(hmrm, renderer, scene, traversal=TRAVERSALS[trav],
                                    pixel_format=hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8)
                renderer.render_device(f, buf.data_ptr() + start)
                renderer.wait()
                assert renderer.stats().status == 0
                _assert_bytes(buf.cpu().numpy(), M.expected_destination(fill, start, frame, np.ones((h, w), bool), ch),
                              f"{name} {w}x{h} {trav} channels {ch} offset {off}", start, (h, w, ch))
    assert hits > 0


def test_4gib_frames_through_render_device(hmrm, renderer, oracle):
    """65536 x 16384: 2^25 tiles (above 2^24, __uint2float_rz(tile) is no longer exact) and 4 GiB of RGBA8 / 3 GiB of
    RGB8 (every index above 2^31 bytes).  On the device: every ray counted, every alpha byte written, the guards intact;
    on the host: sampled tile rows and the first and last 8 columns against the oracle."""
    import torch

    w, h = 65536, 16384
    name = "persp_basic"
    _Configured(renderer, oracle)(name)
    scene = dict(SCENES[name], width=w, height=h)
    hm, cm = _maps(oracle, name)
    heights = oracle.update_heightmap(hm, scene["lum"], scene["min_height"], scene["max_height"])
    # a lazily committed host frame: only the sampled rows and columns are ever touched
    want = np.zeros((h, w, 4), dtype=np.uint8)
    rows = [(0, 4), (h // 2, h // 2 + 4), (h - 4, h)]
    cols = list(range(8)) + list(range(w - 8, w))
    for r0, r1 in rows:
        oracle.render(H.oracle_frame(oracle, scene), heights, cm, want_steps=False, rows=(r0, r1), framebuf=want)
    for x in cols:       # cycle_period W: pixel x of every row
        oracle.render(H.oracle_frame(oracle, scene, cycle=x, cycle_period=w), heights, cm, want_steps=False, framebuf=want)

    rgba = None
    for ch in (4, 3):
        n = h * w * ch
        guards = torch.from_numpy(M.sentinel_bytes(np.random.default_rng(ch), 2 * GUARD)).to("cuda:0")
        buf = torch.empty(n + 2 * GUARD, dtype=torch.uint8, device="cuda:0")
        buf.fill_(0xA5)
        buf[:GUARD] = guards[:GUARD]
        buf[GUARD + n:] = guards[GUARD:]
        out = buf[GUARD:GUARD + n].view(h, w, ch)
        if ch == 4:
            out[:, :, 3] = 0                         # an alpha the renderer never writes
        torch.cuda.synchronize()
        f = H.product_frame(hmrm, renderer, scene, traversal=hmrm.TRAVERSAL_SKIP, flags=hmrm.FLAG_STATS,
                            pixel_format=hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8)
        renderer.render_device(f, buf.data_ptr() + GUARD)
        renderer.wait()
        st = renderer.stats()
        assert st.rays == w * h and st.status == 0, (ch, st.rays, st.status)
        assert torch.equal(buf[:GUARD], guards[:GUARD]) and torch.equal(buf[GUARD + n:], guards[GUARD:]), ch
        for r0, r1 in rows:
            got = out[r0:r1].cpu().numpy()
            assert np.array_equal(got, want[r0:r1, :, :ch]), (ch, r0, r1, int((got != want[r0:r1, :, :ch]).sum()))
        for lo, hi in ((0, 8), (w - 8, w)):
            got = out[:, lo:hi].cpu().numpy()
            assert np.array_equal(got, want[:, lo:hi, :ch]), (ch, lo, int((got != want[:, lo:hi, :ch]).sum()))
        if ch == 4:
            assert bool((out[:, :, 3] == 255).all())
            rgba = buf
        else:
            # every RGB8 pixel was written: the RGBA8 frame above is complete (alpha) and matches the oracle's samples
            assert torch.equal(out, rgba[GUARD:GUARD + h * w * 4].view(h, w, 4)[:, :, :3])
        del out
    del buf, rgba
    torch.cuda.empty_cache()


@pytest.mark.parametrize("w,h", [(16384, 2), (2, 16384)])
def test_supersample4_subframe_at_the_axis_limit(hmrm, renderer, oracle, w, h):
    """s = 4 of 16384 x 2 and 2 x 16384: the sub-frame is 65536 pixels long.  Every pixel against the box filter of the
    oracle's sub-frame, into device memory at offsets 0 and 3 and into host memory."""
    import torch

    _Configured(renderer, oracle)("persp_basic")
    scene = dict(SCENES["persp_basic"], width=w, height=h, **({"hfov_deg": 20.0} if w == 2 else {}))
    frame, st = _oracle(oracle, scene, 4)
    assert st.surf_hits > 0 and st.rays > st.surf_hits
    for ch in (4, 3):
        fmt = hmrm.PIXEL_RGB8 if ch == 3 else hmrm.PIXEL_RGBA8
        f = H.product_frame(hmrm, renderer, scene, pixel_format=fmt, flags=hmrm.supersample_flag(4))
        for off in (0, 3):
            start = GUARD + off
            fill = M.sentinel_bytes(np.random.default_rng(off + ch), start + h * w * ch + GUARD)
            buf = torch.from_numpy(fill).to("cuda:0")
            torch.cuda.synchronize()
            renderer.render_device(f, buf.data_ptr() + start)
            renderer.wait()
            _assert_bytes(buf.cpu().numpy(), M.expected_destination(fill, start, frame, np.ones((h, w), bool), ch),
                          f"s=4 {w}x{h} channels {ch} offset {off}", start, (h, w, ch))
        got = renderer.render(f)
        assert np.array_equal(got, frame[:, :, :ch]), f"s=4 {w}x{h} channels {ch} hmrm_render"


@pytest.mark.parametrize("w,h", [(65536, 3), (3, 65536)])
def test_png_and_yuv_at_the_axis_limit(renderer, w, h):
    """hmrm_encode_png and hmrm_convert_yuv420 on odd images at the 65536 axis limit."""
    from PIL import Image
    import io

    rng = np.random.default_rng(w)
    for ch in (3, 4):
        y, x, c = np.meshgrid(np.arange(h), np.arange(w), np.arange(ch), indexing="ij")
        px = ((3 * x + 5 * y + 40 * c) % 256).astype(np.uint8)
        noisy = rng.random((h, w)) < 0.25
        px[noisy] = rng.integers(0, 256, (int(noisy.sum()), ch), dtype=np.uint8)
        data = renderer.encode_png(px)
        assert np.array_equal(check_png(data)[0], px), (w, h, ch)
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(data))), px), (w, h, ch)
        for matrix in (BT601, BT709):
            got = renderer.convert_yuv420(px, matrix)
            for plane, g, want in zip(("Y", "Cb", "Cr"), got, yuv420_model(px, matrix)):
                assert np.array_equal(g, want), (w, h, ch, matrix, plane)
