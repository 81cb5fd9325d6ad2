"""GPU: JPEG frames encoded on the device (hmrm_render_jpeg_async, hmrm_encode_jpeg).  Every expected file is Pillow's
(libjpeg-turbo) encoding of the same pixels, never the device's; only past libjpeg-turbo's 65500-pixel limit is it the
model's.  Files are also decoded by PIL and by `hmap --decode-image` (the repository's stb-exact decoder, restart
markers included) and must have the frame's size."""
import io
import subprocess
from pathlib import Path

import numpy as np
import pytest
from PIL import Image

import helpers as H
import scenes as S
from test_jpeg_model import expected_bound, pil_jpeg

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"
GOLDEN_NAMES = sorted(H.golden_frames().files)


def _case(kind, h, w, ch, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, size=(h, w, ch), dtype=np.uint8)
    if kind == "constant":
        return np.full((h, w, ch), 77, dtype=np.uint8)
    if kind == "rows":
        return np.broadcast_to(rng.integers(0, 256, size=(1, w, ch), dtype=np.uint8), (h, w, ch)).copy()
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(xx + k * 30) % 256 if k % 2 == 0 else (yy * 3 + xx // 7) % 256 for k in range(ch)],
                    axis=2).astype(np.uint8)


def check_decodes_hmap(data: bytes, w: int, h: int, tmp_path):
    path, raw = tmp_path / "f.jpg", tmp_path / "f.raw"
    path.write_bytes(data)
    res = subprocess.run([str(HMAP), "--decode-image", str(path), "4", str(raw)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    assert res.stdout.split() == [str(w), str(h), "4"] and raw.stat().st_size == w * h * 4


def check_decodes(data: bytes, w: int, h: int, tmp_path=None):
    im = Image.open(io.BytesIO(data))
    im.load()
    assert im.size == (w, h) and im.mode == "RGB"
    if tmp_path is not None:
        check_decodes_hmap(data, w, h, tmp_path)


def encode_both(renderer, hmrm, px, q, s420, tmp_path):
    """The device's file equals Pillow's and decodes, with PIL and with hmap, to the image's size."""
    want = pil_jpeg(px, q, s420)
    got = renderer.encode_jpeg(px, q, hmrm.JPEG_420 if s420 else hmrm.JPEG_444)
    assert got == want, f"{px.shape} q{q} {'4:2:0' if s420 else '4:4:4'}: {len(got)} vs Pillow's {len(want)} bytes"
    assert len(got) <= expected_bound(px.shape[1], px.shape[0], s420)
    check_decodes(got, px.shape[1], px.shape[0], tmp_path)
    return got


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("kind", ["noise", "constant", "rows", "gradient"])
def test_encode_jpeg_equals_pillow(hmrm, renderer, kind, ch, tmp_path):
    px = _case(kind, 181, 243, ch, seed=ch)
    for q in (1, 50, 75, 90, 100):
        for s420 in (True, False):
            encode_both(renderer, hmrm, px, q, s420, tmp_path)


@pytest.mark.parametrize("h,w", [(1, 1), (9, 7), (33, 17), (1, 40), (40, 1), (16, 16), (31, 47), (243, 181)])
def test_encode_jpeg_small_and_odd_shapes(hmrm, renderer, h, w, tmp_path):
    for ch in (3, 4):
        for kind in ("noise", "gradient"):
            px = _case(kind, h, w, ch, seed=h * 1000 + w)
            for q in (1, 75, 100):
                for s420 in (True, False):
                    encode_both(renderer, hmrm, px, q, s420, tmp_path)


def test_encode_jpeg_from_device_memory(hmrm, renderer, tmp_path):
    import torch

    for ch in (3, 4):
        px = _case("noise", 97, 131, ch, seed=5)
        px[20:60] = _case("gradient", 40, 131, ch)
        d = torch.from_numpy(px).to("cuda:0")
        for s420, chroma in ((True, hmrm.JPEG_420), (False, hmrm.JPEG_444)):
            data = renderer.encode_jpeg(d, 90, chroma)
            assert data == pil_jpeg(px, 90, s420)
            check_decodes(data, 131, 97, tmp_path)


def test_encode_jpeg_axis_limits(hmrm, renderer, tmp_path):
    """65535 per axis, SOF0's limit.  libjpeg-turbo refuses more than 65500, so Pillow checks 65500 and the model
    (pinned to Pillow by tests/test_jpeg_model.py) checks 65535, whose files the repository's decoder also reads."""
    import jpeg_model as M

    for h, w in ((2, 65500), (65500, 2), (2, 65535), (65535, 2)):
        px = _case("gradient", h, w, 3)
        px[::3, ::5, 1] = 200
        for s420, chroma in ((True, hmrm.JPEG_420), (False, hmrm.JPEG_444)):
            if max(h, w) <= 65500:
                encode_both(renderer, hmrm, px, 75, s420, tmp_path)
                continue
            got = renderer.encode_jpeg(px, 75, chroma)
            assert got == M.write(px, 75, s420), f"{w}x{h} {'4:2:0' if s420 else '4:4:4'}"
            check_decodes_hmap(got, w, h, tmp_path)
    with pytest.raises(ValueError):
        renderer.encode_jpeg(np.zeros((2, 65536, 3), dtype=np.uint8))


def test_encode_jpeg_bit_offsets_past_2_32(hmrm, renderer):
    """16384 x 8192 noise at q = 100 in 4:4:4: a ~550 MB file, past 2^32 bits."""
    import torch

    px = _case("noise", 8192, 16384, 3, seed=11)
    want = pil_jpeg(px, 100, False)
    assert len(want) * 8 > 2 ** 32
    got = renderer.encode_jpeg(torch.from_numpy(px).to("cuda:0"), 100, hmrm.JPEG_444)
    assert len(got) == len(want) and got == want
    renderer._pinned_cache.pop("jpeg", None)


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_reference_frames_through_render_jpeg(hmrm, renderer, oracle, name, tmp_path):
    scene = S.SCENE_BY_NAME[name]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    want = H.golden_frames()[name]
    for q, chroma, s420 in ((90, hmrm.JPEG_420, True), (75, hmrm.JPEG_444, False)):
        files = [renderer.render_jpeg(H.product_frame(hmrm, renderer, scene, pixel_format=fmt), q, chroma)
                 for fmt in (hmrm.PIXEL_RGBA8, hmrm.PIXEL_RGB8)]
        assert files[0] == files[1], f"{name}: RGBA8 and RGB8 files differ"
        assert files[0] == pil_jpeg(want, q, s420), f"{name} q{q}"
        check_decodes(files[0], want.shape[1], want.shape[0], tmp_path)


@pytest.mark.parametrize("s", [2, 3, 4])
def test_supersampled_frames(hmrm, renderer, oracle, s, tmp_path):
    scene = dict(S.SCENE_BY_NAME["persp_basic"])
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    f = H.product_frame(hmrm, renderer, scene)
    f.flags = hmrm.supersample_flag(s)
    px = renderer.render(f).copy()
    for q, chroma, s420 in ((90, hmrm.JPEG_420, True), (90, hmrm.JPEG_444, False)):
        data = renderer.render_jpeg(f, q, chroma)
        assert data == pil_jpeg(px, q, s420)
        check_decodes(data, px.shape[1], px.shape[0], tmp_path)


def test_destinations(hmrm, renderer, oracle):
    import torch

    scene = S.SCENE_BY_NAME["spher_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    f = H.product_frame(hmrm, renderer, scene)
    W, Hh = scene["width"], scene["height"]
    want = pil_jpeg(H.golden_frames()["spher_basic"], 75, True)
    bound = hmrm.jpeg_bound(W, Hh, hmrm.JPEG_420)
    guard = 64
    # pinned host memory with sentinel bytes around the file
    host = hmrm.pinned_empty((bound + 2 * guard,))
    host[:] = 0xA5
    size = hmrm.pinned_empty((1,), dtype=np.uint64)
    renderer.render_jpeg_async(f, host.ctypes.data + guard, size, 75, hmrm.JPEG_420, capacity=bound)
    renderer.wait()
    n = int(size[0])
    assert n == len(want) and host[guard:guard + n].tobytes() == want
    assert (host[:guard] == 0xA5).all() and (host[guard + n:] == 0xA5).all()
    # device memory at several byte offsets
    for off in (0, 1, 3, 8):
        out = torch.full((bound + off + guard,), 0x5A, dtype=torch.uint8, device="cuda:0")
        dsize = torch.zeros(1, dtype=torch.int64, device="cuda:0")
        renderer.render_jpeg_async(f, out.data_ptr() + off, dsize.data_ptr(), 75, hmrm.JPEG_420, capacity=bound)
        renderer.wait()
        n = int(dsize.item())
        got = out.cpu().numpy()
        assert n == len(want) and got[off:off + n].tobytes() == want, f"offset {off}"
        assert (got[:off] == 0x5A).all() and (got[off + n:] == 0x5A).all(), f"offset {off}: bytes outside the file"
    # exactly the bound is accepted, one byte less refused
    out = torch.zeros(bound, dtype=torch.uint8, device="cuda:0")
    renderer.render_jpeg_async(f, out, dsize, 75, hmrm.JPEG_420)
    renderer.wait()
    assert out[:int(dsize.item())].cpu().numpy().tobytes() == want
    with pytest.raises(hmrm.HmrmError):
        renderer.render_jpeg_async(f, out[:bound - 1], dsize, 75, hmrm.JPEG_420)
    with pytest.raises(ValueError):
        renderer.render_jpeg_async(f, out.data_ptr(), dsize, 75, hmrm.JPEG_420)    # a raw address without its capacity
    # encode_jpeg's synchronous path on the context's stream after work on a caller's stream
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        px = torch.from_numpy(H.golden_frames()["spher_basic"]).to("cuda:0")
    s.synchronize()
    assert renderer.encode_jpeg(px, 75, hmrm.JPEG_420) == want


def test_four_frames_in_flight_with_raw_png_and_yuv(hmrm, renderer, oracle):
    scene = dict(S.SCENE_BY_NAME["persp_basic"])
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    W, Hh = scene["width"], scene["height"]
    frames = [H.product_frame(hmrm, renderer, dict(scene, pos=(-0.6 + 0.05 * i, 0.6, 3.2 - 0.1 * i),
                                                   hang_deg=-45.0 - 7.0 * i)) for i in range(10)]
    alone = [renderer.render(f).copy() for f in frames]
    kinds = ["jpeg", "raw", "jpeg", "png", "yuv", "jpeg", "jpeg", "raw", "png", "jpeg"]
    bufs = []
    for k in kinds:
        if k == "jpeg":
            bufs.append((hmrm.pinned_empty((hmrm.jpeg_bound(W, Hh),)), hmrm.pinned_empty((1,), dtype=np.uint64)))
        elif k == "png":
            bufs.append((hmrm.pinned_empty((hmrm.png_bound(W, Hh, 4),)), hmrm.pinned_empty((1,), dtype=np.uint64)))
        elif k == "yuv":
            bufs.append((hmrm.pinned_empty((hmrm.yuv420_bytes(W, Hh),)), None))
        else:
            bufs.append((hmrm.pinned_empty((Hh, W, 4)), None))

    def check(i):
        k, (out, size) = kinds[i], bufs[i]
        if k == "jpeg":
            assert out[:int(size[0])].tobytes() == pil_jpeg(alone[i], 85, True), f"frame {i}"
        elif k == "png":
            assert np.array_equal(np.asarray(Image.open(io.BytesIO(out[:int(size[0])].tobytes()))), alone[i])
        elif k == "yuv":
            want = renderer.convert_yuv420(alone[i])
            assert out.tobytes() == b"".join(p.tobytes() for p in want), f"frame {i}"
        else:
            assert np.array_equal(out, alone[i]), f"frame {i}"

    pending = []
    for i, (k, f) in enumerate(zip(kinds, frames)):
        if len(pending) == 4:
            renderer.wait_pending(3)
            pending.pop(0)
        out, size = bufs[i]
        if k == "jpeg":
            renderer.render_jpeg_async(f, out, size, 85, hmrm.JPEG_420)
        elif k == "png":
            renderer.render_png_async(f, out, size)
        elif k == "yuv":
            renderer.render_yuv420_async(f, out, hmrm.YUV_BT709)
        else:
            renderer.render_async(f, out)
        pending.append(i)
    renderer.wait()
    for i in range(len(kinds)):
        check(i)


@pytest.mark.parametrize("s420", [True, False])
def test_flythrough_4k_frame(hmrm, s420):
    import bench

    wl = bench.WORKLOADS["flythrough4k"]
    with hmrm.Renderer(0) as r:
        r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
        r.synth_maps(wl["log2n"], bench.SEED)
        c = bench.camera(wl, 17)
        f = r.frame(projection=wl["projection"], screen_width=wl["W"], screen_height=wl["H"], cam_pos=c["pos"],
                    hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                    ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"])
        px = r.render(f).copy()
        assert r.render_jpeg(f, 90, hmrm.JPEG_420 if s420 else hmrm.JPEG_444) == pil_jpeg(px, 90, s420)


def test_refusals(hmrm, renderer, oracle):
    import ctypes as C

    scene = S.SCENE_BY_NAME["persp_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    lib = hmrm.load_library()
    bound = hmrm.jpeg_bound(scene["width"], scene["height"])
    pinned = hmrm.pinned_empty((bound,))
    size = hmrm.pinned_empty((1,), dtype=np.uint64)
    pageable = np.zeros(bound, dtype=np.uint8)
    pageable_size = np.zeros(1, dtype=np.uint64)

    def call(frame, out, cap, sz, q=90, chroma=0):
        return lib.hmrm_render_jpeg_async(renderer._h, C.byref(frame), q, chroma, out.ctypes.data, cap, sz.ctypes.data)

    f = H.product_frame(hmrm, renderer, scene)
    assert call(f, pinned, bound - 1, size) == 1
    assert call(f, pageable, bound, size) == 1
    assert call(f, pinned, bound, pageable_size) == 1
    assert lib.hmrm_render_jpeg_async(renderer._h, C.byref(f), 90, 0, pinned.ctypes.data, bound,
                                      size.ctypes.data + 4) == 1                       # size word not 8-byte aligned
    assert call(H.product_frame(hmrm, renderer, scene, cycle_period=3), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, band_count=2, band_index=0), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, flags=hmrm.FLAG_STEP_INDEX), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, flags=hmrm.FLAG_RAY_DUMP), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, row_begin=0, row_end=8), pinned, bound, size) == 1
    for q, chroma in ((0, 0), (101, 0), (90, 2), (90, -1)):
        assert call(f, pinned, bound, size, q, chroma) == 1
    assert call(H.product_frame(hmrm, renderer, scene, screen_width=65536, screen_height=2), pinned, bound, size) == 1
    px = np.zeros((10, 10, 4), dtype=np.uint8)
    small = hmrm.jpeg_bound(10, 10)
    assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, 10, 10, 4, 90, 0, pinned.ctypes.data, small - 1,
                                size.ctypes.data) == 1
    assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, 10, 10, 4, 90, 0, pageable.ctypes.data, bound,
                                size.ctypes.data) == 1
    assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, 10, 10, 2, 90, 0, pinned.ctypes.data, bound,
                                size.ctypes.data) == 1
    assert lib.hmrm_encode_jpeg(renderer._h, None, 10, 10, 4, 90, 0, pinned.ctypes.data, bound, size.ctypes.data) == 1
    # every limit of hmrm_encode_jpeg, through the C entry point with a live context
    for w, h, ch, q, chroma in ((10, 10, 4, 0, 0), (10, 10, 4, 101, 0), (10, 10, 4, 90, 2), (10, 10, 4, 90, -1),
                                (65536, 1, 4, 90, 0), (1, 65536, 4, 90, 1), (0, 10, 4, 90, 0), (10, 10, 5, 90, 0)):
        assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, w, h, ch, q, chroma, pinned.ctypes.data, bound,
                                    size.ctypes.data) == 1, (w, h, ch, q, chroma)
    assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, 10, 10, 4, 90, 0, None, bound, size.ctypes.data) == 1
    assert lib.hmrm_encode_jpeg(renderer._h, px.ctypes.data, 10, 10, 4, 90, 0, pinned.ctypes.data, bound, None) == 1
    # the context still works after the refusals
    assert renderer.render_jpeg(f, 90) == pil_jpeg(H.golden_frames()["persp_basic"], 90, True)
