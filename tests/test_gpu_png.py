"""GPU: PNG frames deflated on the device (hmrm_render_png_async, hmrm_encode_png, and `hmap` writing through them).
Every file is checked by the independent checker of tests/test_png_encode.py (chunk CRCs, IHDR, zlib with its
Adler-32, the five filters undone in Python) and by PIL; the decoded pixels must be the frame, byte for byte.  And every
file must be the PNG model's (tests/png_model.py) byte for byte: whole, or for frames too large for the model, its
first and last segments, every segment that starts in a row repeated from the row above and 64 seeded random ones."""
import io
import json
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
from PIL import Image

import helpers as H
import png_model as M
import scenes as S
from test_png_encode import check_png, expected_bound, png_chunks
from test_png_model import (content, filter_tie_pixels, literal_edge_pixels, match_length_pixels, row_distance_pixels,
                            tie_pixels)

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"
GOLDEN_NAMES = sorted(H.golden_frames().files)


def pil_pixels(data: bytes) -> np.ndarray:
    return np.asarray(Image.open(io.BytesIO(data)))


def _chunks(data: bytes) -> list:
    """The file's chunks as they are (length, type, data, CRC), nothing verified."""
    pos, out = 8, []
    while pos < len(data):
        end = pos + 12 + int.from_bytes(data[pos:pos + 4], "big")
        out.append(data[pos:end])
        pos = end
    return out


def assert_equals_model(data: bytes, pixels: np.ndarray, what: str = ""):
    """The file is the model's file of the pixels (the channels its IHDR names), byte for byte; a difference is
    reported by the first chunk (segment) in which it occurs."""
    ch = 4 if data[25] == 6 else 3
    want = M.write(np.ascontiguousarray(pixels[:, :, :ch]))
    if data != want:
        got, ref = _chunks(data), _chunks(want)
        k = next((k for k, (a, b) in enumerate(zip(got, ref)) if a != b), min(len(got), len(ref)))
        raise AssertionError(f"{what}: not the model's file: {len(got)} chunks, the model's {len(ref)}; chunk {k} "
                             f"(segment {k - 1}) differs first")


def assert_sampled_segments_equal_model(data: bytes, px: np.ndarray, seed: int = 0, count: int = 64):
    """For frames too large for the whole model: the head, the chunk count, the first and last segments, every segment
    that starts inside a row repeated from the row above and `count` seeded random segments equal the model's."""
    h, w, ch = px.shape
    rowlen = w * ch + 1
    nseg = M.segment_count(px)
    chunks = _chunks(data)
    assert data.startswith(M.head(w, h, ch)) and len(chunks) == nseg + 3
    repeated = np.flatnonzero((px[1:] == px[:-1]).reshape(h - 1, -1).all(axis=1)) + 1
    starts = np.arange(nseg, dtype=np.int64) * M.SEG
    picks = {0, nseg - 1} | set(np.flatnonzero(np.isin(starts // rowlen, repeated)).tolist())
    picks |= set(np.random.default_rng(seed).integers(0, nseg, size=count).tolist())
    for k in sorted(picks):
        assert chunks[1 + k] == M.segment_chunk(px, k), f"segment {k} of {nseg} differs from the model's"


def roundtrip(renderer, px: np.ndarray, unfilter: bool = True, model: str = "whole") -> bytes:
    data = renderer.encode_png(px)
    h, w, ch = px.shape
    assert len(data) <= expected_bound(w, h, ch)
    got, _ = check_png(data, unfilter=unfilter)
    if unfilter:
        assert np.array_equal(got, px)
    assert np.array_equal(pil_pixels(data), px)
    if model == "whole":
        assert_equals_model(data, px, f"{w}x{h}x{ch}")
    else:
        assert_sampled_segments_equal_model(data, px)
    return data


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_reference_frames_through_render_png(hmrm, renderer, oracle, name, tmp_path):
    scene = S.SCENE_BY_NAME[name]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    want = H.golden_frames()[name]
    for fmt, ch in ((hmrm.PIXEL_RGBA8, 4), (hmrm.PIXEL_RGB8, 3)):
        data = renderer.render_png(H.product_frame(hmrm, renderer, scene, pixel_format=fmt))
        assert len(data) <= expected_bound(want.shape[1], want.shape[0], ch)
        got, _ = check_png(data)
        assert np.array_equal(got, want[:, :, :ch]), f"{name} {ch} channels: checker"
        assert np.array_equal(pil_pixels(data), want[:, :, :ch]), f"{name} {ch} channels: PIL"
        assert_equals_model(data, want, f"{name} {ch} channels")
        path = tmp_path / f"f{ch}.png"
        path.write_bytes(data)
        raw = tmp_path / f"f{ch}.raw"
        res = subprocess.run([str(HMAP), "--decode-image", str(path), "4", str(raw)], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        ours = np.fromfile(raw, dtype=np.uint8).reshape(want.shape[0], want.shape[1], 4)
        assert np.array_equal(ours[:, :, :ch], want[:, :, :ch]) and (ours[:, :, 3] == 255).all(), f"{name}: hmap decode"


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("kind", ["noise", "constant", "rows", "gradient", "repeat"])
def test_encode_png_content_kinds(renderer, kind, ch):
    px = content(kind, 181, 243, ch, seed=ch)
    data = roundtrip(renderer, px)
    raw = px.size + px.shape[0]
    if kind in ("noise", "repeat"):
        assert len(data) <= expected_bound(243, 181, ch)           # stored segments: raw size plus framing
    else:
        assert len(data) < raw // 4, f"{kind}: {len(data)} bytes for {raw} filtered bytes"


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("h,w", [(1, 1), (5, 1), (7, 2), (9, 3), (1, 5), (2, 2), (33, 17), (101, 77)])
def test_encode_png_small_and_odd_shapes(renderer, h, w, ch):
    for kind in ("noise", "gradient", "constant"):
        roundtrip(renderer, content(kind, h, w, ch, seed=h * 1000 + w))


def test_encode_png_row_distance_beyond_deflate_window(renderer):
    """8200 x 8 RGBA: row_bytes + 1 > 32768, so the one-row-up candidate must not be used."""
    px = content("rows", 8, 8200, 4, seed=3)
    px[:, ::97] = 5
    roundtrip(renderer, px)
    roundtrip(renderer, content("noise", 8, 8200, 4, seed=4))


def test_encode_png_8k_frame(renderer):
    """7680 x 4320 RGBA: offsets beyond 2^32 bits, 32 K segments.  Checked by the checker's structure pass, by PIL and
    by zlib-level decode of the filtered stream, and by segments sampled against the model."""
    px = content("gradient", 4320, 7680, 4)
    px[::7, ::5, 1] = np.random.default_rng(8).integers(0, 256, size=px[::7, ::5, 1].shape, dtype=np.uint8)
    px[1000:1003] = px[999]                  # segments starting in rows repeated from the row above
    roundtrip(renderer, px, unfilter=False, model="sampled")


@pytest.mark.parametrize("w,ch", [(8191, 4), (8192, 4), (10922, 3), (10923, 3)])
def test_encode_png_row_distance_at_the_window_limit(renderer, w, ch):
    """W * C + 1 = 32765 and 32767 (the row-up candidate is used), 32769 and 32770 (it is not); the filtered rows
    repeat, so where the candidate is allowed it wins."""
    roundtrip(renderer, row_distance_pixels(w, ch))


# filtered stream of exactly 4096 k bytes, 4096 k +- 1 (the last segment 1 byte), and shorter than one segment
SEGMENT_SHAPES = [(1, 1365, 3), (2, 1365, 3), (4, 1365, 3), (16, 341, 3), (1024, 5, 3), (256, 21, 3),
                  (17, 80, 3), (3, 910, 3), (5, 819, 4), (3, 341, 4), (11, 279, 4), (7, 20, 4), (1, 1, 3)]


@pytest.mark.parametrize("h,w,ch", SEGMENT_SHAPES)
def test_encode_png_segment_boundaries(renderer, h, w, ch):
    total = h * (w * ch + 1)
    assert total % M.SEG in (0, 1, M.SEG - 1) or total < M.SEG
    for kind in ("rows", "repeat", "constant", "noise", "gradient"):
        roundtrip(renderer, content(kind, h, w, ch, seed=total))


@pytest.mark.parametrize("ch", [3, 4])
def test_encode_png_match_lengths_literals_and_filter_ties(renderer, ch):
    """Matches of exactly 258 (the cap), 257, 11, 10 and 3 bytes; literals on both sides of 143 / 144; every pair of
    filter types tied for the smallest sum; constant rows under an identical row (Up and Paeth tie at zero)."""
    roundtrip(renderer, match_length_pixels(ch))
    roundtrip(renderer, literal_edge_pixels(9, 31, ch))
    roundtrip(renderer, filter_tie_pixels(ch))
    roundtrip(renderer, content("constant", 6, 50, ch))


def test_encode_png_coded_stored_tie_stays_coded(renderer):
    """A segment whose fixed-Huffman block takes exactly as many bytes as its stored block is coded (BTYPE 01)."""
    px = tie_pixels()
    data = roundtrip(renderer, px)
    idats = [b for t, b in png_chunks(data) if t == b"IDAT"]
    assert len(idats) == 2 and idats[0][:2] == b"\x78\x01" and idats[0][2] & 7 == 2
    assert len(idats[0]) == 2 + 5 + px.size + 1


def test_streaming_four_frames_in_flight(hmrm, renderer, oracle):
    scene = dict(S.SCENE_BY_NAME["persp_basic"])
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    frames = [H.product_frame(hmrm, renderer, dict(scene, pos=(-0.6 + 0.05 * i, 0.6, 3.2 - 0.1 * i),
                                                   hang_deg=-45.0 - 7.0 * i)) for i in range(6)]
    want = [renderer.render(f).copy() for f in frames]
    bound = hmrm.png_bound(scene["width"], scene["height"], 4)
    bufs = [hmrm.pinned_empty((bound,)) for _ in range(4)]
    sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]
    pending = []
    for i, f in enumerate(frames):
        if len(pending) == 4:
            renderer.wait_pending(3)
            j = pending.pop(0)
            data = bufs[j % 4][:int(sizes[j % 4][0])].tobytes()
            assert np.array_equal(check_png(data)[0], want[j]), f"frame {j}"
            assert_equals_model(data, want[j], f"frame {j}")
        renderer.render_png_async(f, bufs[i % 4], sizes[i % 4])
        pending.append(i)
    renderer.wait()
    for j in pending:
        data = bufs[j % 4][:int(sizes[j % 4][0])].tobytes()
        assert int(sizes[j % 4][0]) == len(data) and data.endswith(b"IEND\xaeB`\x82")
        assert np.array_equal(check_png(data)[0], want[j]), f"frame {j}"
        assert_equals_model(data, want[j], f"frame {j}")
    assert len({H.sha(w) for w in want}) == len(want)


def test_render_png_into_device_memory(hmrm, renderer, oracle):
    import torch

    scene = S.SCENE_BY_NAME["spher_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    f = H.product_frame(hmrm, renderer, scene)
    bound = hmrm.png_bound(scene["width"], scene["height"], 4)
    out = torch.zeros(bound + 3, dtype=torch.uint8, device="cuda:0")
    size = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    renderer.render_png_async(f, out.data_ptr() + 3, size.data_ptr(), capacity=bound)   # an unaligned destination
    renderer.wait()
    n = int(size.item())
    data = out[3:3 + n].cpu().numpy().tobytes()
    assert np.array_equal(check_png(data)[0], H.golden_frames()["spher_basic"])
    assert_equals_model(data, H.golden_frames()["spher_basic"], "device destination")
    # a tensor reports its own size: one byte short of the bound is refused, not overrun
    with pytest.raises(hmrm.HmrmError):
        renderer.render_png_async(f, out[:bound - 1], size)
    with pytest.raises(ValueError):
        renderer.render_png_async(f, out.data_ptr(), size)             # a raw address without its capacity
    with pytest.raises(ValueError):
        renderer.render_png_async(f, out, torch.zeros(1, dtype=torch.int32, device="cuda:0"))
    renderer.render_png_async(f, out, size)
    renderer.wait()
    assert int(size.item()) == n


def test_refusals(hmrm, renderer, oracle):
    import ctypes as C

    scene = S.SCENE_BY_NAME["persp_basic"]
    H.configure(renderer, scene, H.load_scene_maps(scene, oracle))
    lib = hmrm.load_library()
    bound = hmrm.png_bound(scene["width"], scene["height"], 4)
    pinned = hmrm.pinned_empty((bound,))
    size = hmrm.pinned_empty((1,), dtype=np.uint64)
    pageable = np.zeros(bound, dtype=np.uint8)
    pageable_size = np.zeros(1, dtype=np.uint64)

    def call(frame, out, cap, sz):
        return lib.hmrm_render_png_async(renderer._h, C.byref(frame), out.ctypes.data, cap, sz.ctypes.data)

    f = H.product_frame(hmrm, renderer, scene)
    assert call(f, pinned, bound - 1, size) == 1
    assert call(f, pageable, bound, size) == 1
    assert call(f, pinned, bound, pageable_size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, cycle_period=3), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, band_count=2, band_index=0), pinned, bound, size) == 1
    assert call(H.product_frame(hmrm, renderer, scene, flags=hmrm.FLAG_STEP_INDEX), pinned, bound, size) == 1
    px = np.zeros((10, 10, 4), dtype=np.uint8)
    assert lib.hmrm_encode_png(renderer._h, px.ctypes.data, 10, 10, 4, pinned.ctypes.data,
                               hmrm.png_bound(10, 10, 4) - 1, size.ctypes.data) == 1
    assert lib.hmrm_encode_png(renderer._h, px.ctypes.data, 10, 10, 4, pageable.ctypes.data, bound,
                               size.ctypes.data) == 1
    assert lib.hmrm_encode_png(renderer._h, px.ctypes.data, 10, 10, 2, pinned.ctypes.data, bound, size.ctypes.data) == 1
    # the context still works after the refusals
    data = renderer.render_png(f)
    assert np.array_equal(check_png(data)[0], H.golden_frames()["persp_basic"])


def _write_scene(oracle, scene, tmp_path):
    hm, cm = H.load_scene_maps(scene, oracle)
    oracle.write_png(tmp_path / "h.png", hm)
    oracle.write_png(tmp_path / "c.png", cm)
    cfg = tmp_path / "config.txt"
    cfg.write_text(oracle.config_text(S.frame_kwargs(scene), "h.png", "c.png", lum=scene["lum"]))
    return cfg


@pytest.mark.parametrize("gpus", [1, 3])
def test_hmap_stats_json_reports_png_bytes(hmrm, oracle, gpus, tmp_path):
    scene = S.SCENE_BY_NAME["ortho_basic"]
    cfg = _write_scene(oracle, scene, tmp_path)
    out, stats = tmp_path / "out.png", tmp_path / "stats.json"
    env = dict(os.environ, HMAP_DEVICE_LIST=",".join(["0"] * gpus))
    res = subprocess.run([str(HMAP), str(cfg), "--headless", str(out), "--projection", "3", "--gpus", str(gpus),
                          "--stats-json", str(stats)], capture_output=True, text=True, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr
    assert json.loads(stats.read_text())["png_bytes"] == out.stat().st_size
    assert np.array_equal(check_png(out.read_bytes())[0], H.golden_frames()["ortho_basic"])
    assert_equals_model(out.read_bytes(), H.golden_frames()["ortho_basic"], "hmap --headless")
    # a script: the sum over its files
    (tmp_path / "frames.txt").write_text("".join("hang %r\n" % (-45.0 - 4.0 * i) for i in range(6)))
    res = subprocess.run([str(HMAP), str(cfg), "--script", "frames.txt", "--out-prefix", str(tmp_path / "s_"),
                          "--gpus", str(gpus), "--stats-json", str(stats)], capture_output=True, text=True,
                         cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr
    st = json.loads(stats.read_text())
    assert st["frames"] == 6
    assert st["png_bytes"] == sum((tmp_path / f"s_{i}.png").stat().st_size for i in range(6))


def test_hmap_record_over_several_devices_equals_oracle(hmrm, oracle, tmp_path):
    scene = dict(S.SCENE_BY_NAME["persp_basic"], width=160, height=90)
    cfg = _write_scene(oracle, scene, tmp_path)
    (tmp_path / "screenshots").mkdir()
    states = [dict(pos=(-0.6 + 0.07 * i, 0.6, 3.2), hang_deg=-45.0 - 5.0 * i) for i in range(11)]
    (tmp_path / "frames.txt").write_text("".join("pos %r %r %r hang %r\n" % (*s["pos"], s["hang_deg"]) for s in states))
    env = dict(os.environ, HMAP_DEVICE_LIST="0,0,0")
    res = subprocess.run([str(HMAP), str(cfg), "--script", "frames.txt", "--record", "--gpus", "3"],
                         capture_output=True, text=True, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stderr
    assert res.stdout.rstrip().endswith("Done recording.")
    files = sorted((tmp_path / "screenshots").glob("hmap_*.png"), key=lambda p: int(p.stem.rsplit("_", 1)[1]))
    assert len(files) == len(states)
    assert res.stdout.count("Saved screenshot at ") == len(states)
    maps = H.load_scene_maps(scene, oracle)
    for i, s in enumerate(states):
        want, _, _ = H.oracle_render_scene(oracle, dict(scene, **s), maps)
        got, _ = check_png(files[i].read_bytes())
        assert np.array_equal(got, want), f"frame {i}"
        assert_equals_model(files[i].read_bytes(), want, f"frame {i}")


def test_sdl_shell_screenshot_and_recording_are_device_encoded(hmrm, oracle, tmp_path):
    """The interactive shell (fake SDL): F12 saves the previous frame and Ctrl+Shift+R records frames, both through
    hmrm_encode_png; every file decodes to the frame the shell handed to SDL."""
    from test_gpu_sdl_shell import build_shell, run_shell, write_inputs

    (tmp_path / "build").mkdir()
    binary = build_shell(tmp_path / "build")
    write_inputs(oracle, tmp_path, "recording_frame_count 3", "1 key 2\n3 key f12\n4 key r ctrl shift\n")
    (tmp_path / "screenshots").mkdir()
    frames, out = run_shell(binary, tmp_path, 9)
    shots = sorted((tmp_path / "screenshots").glob("hmap_*.png"))
    assert out.count("Saved screenshot at ") == 4 and "Done recording." in out
    stills = [p for p in shots if p.stem.count("_") == 1]
    recorded = sorted((p for p in shots if p.stem.count("_") == 2), key=lambda p: int(p.stem.rsplit("_", 1)[1]))
    assert len(stills) == 1 and len(recorded) == 3
    decoded = {H.sha(check_png(p.read_bytes())[0]) for p in shots}
    for p in shots:
        assert_equals_model(p.read_bytes(), check_png(p.read_bytes())[0], p.name)
    shown = {H.sha(f): i for i, f in enumerate(frames)}
    assert decoded <= set(shown), "a saved file is not one of the frames the shell displayed"
