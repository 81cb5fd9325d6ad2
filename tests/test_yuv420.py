"""CPU: the numpy model of the 4:2:0 conversion (include/hmrm.h's integer definition) and the Y4M reader that the device
conversion and `hmap --video` are tested with (tests/test_gpu_yuv.py); the model is proven here against the float
BT.601 / BT.709 definitions and hand-worked edge cases, the reader against hand-built streams.  Also hmrm_yuv420_bytes,
the NULL-context refusals of the new entry points and hmap's --video usage refusals (no GPU needed for any of them)."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"

BT601, BT709 = 0, 1
# (Y, Cb, Cr) rows of (R, G, B) weights in 2^-14 fixed point, as include/hmrm.h lists them
COEF = {
    BT601: ((4207, 8260, 1604), (-2428, -4768, 7196), (7196, -6026, -1170)),
    BT709: ((2991, 10064, 1016), (-1649, -5547, 7196), (7196, -6536, -660)),
}
KR_KB = {BT601: (0.299, 0.114), BT709: (0.2126, 0.0722)}


def yuv420_model(px, matrix: int):
    """[H, W, 3 | 4] uint8 -> (Y [H, W], Cb [ceil(H/2), ceil(W/2)], Cr) uint8, exactly as include/hmrm.h defines them."""
    px = np.asarray(px)
    h, w = px.shape[:2]
    ch, cw = (h + 1) // 2, (w + 1) // 2
    r, g, b = (px[:, :, k].astype(np.int32) for k in range(3))
    ky, kcb, kcr = COEF[matrix]
    y = ((ky[0] * r + ky[1] * g + ky[2] * b + (1 << 13)) >> 14) + 16
    rows = np.minimum(np.arange(2 * ch), h - 1)
    cols = np.minimum(np.arange(2 * cw), w - 1)

    def box(p):     # sum of each 2x2 block, indices clamped (odd sizes replicate the last row / column)
        return p[rows][:, cols].reshape(ch, 2, cw, 2).sum(axis=(1, 3))

    sr, sg, sb = box(r), box(g), box(b)
    cb = ((kcb[0] * sr + kcb[1] * sg + kcb[2] * sb + (1 << 15)) >> 16) + 128
    cr = ((kcr[0] * sr + kcr[1] * sg + kcr[2] * sb + (1 << 15)) >> 16) + 128
    return y.astype(np.uint8), cb.astype(np.uint8), cr.astype(np.uint8)


def i420(planes) -> bytes:
    return b"".join(np.ascontiguousarray(p).tobytes() for p in planes)


def read_y4m(data: bytes):
    """-> (header, frames): header maps each parameter letter of the stream header to its text ("X" to a list), frames
    are the bytes of each frame's planes.  Only 4:2:0 streams; asserts the structure."""
    end = data.index(b"\n")
    tokens = data[:end].decode("ascii").split(" ")
    assert tokens[0] == "YUV4MPEG2", "stream magic"
    header = {"X": []}
    for t in tokens[1:]:
        assert t, "empty header token"
        if t[0] == "X":
            header["X"].append(t[1:])
        else:
            assert t[0] not in header, f"repeated header parameter {t[0]}"
            header[t[0]] = t[1:]
    w, h = int(header["W"]), int(header["H"])
    assert header.get("C", "420jpeg").startswith("420")
    size = w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)
    frames, pos = [], end + 1
    while pos < len(data):
        nl = data.index(b"\n", pos)
        assert data[pos:nl].split(b" ")[0] == b"FRAME", f"frame marker at byte {pos}"
        assert nl + 1 + size <= len(data), "truncated frame"
        frames.append(data[nl + 1:nl + 1 + size])
        pos = nl + 1 + size
    return header, frames


# ---- the model against the float definitions ----
def _float_yuv(rgb_mean, matrix):
    kr, kb = KR_KB[matrix]
    kg = 1.0 - kr - kb
    r, g, b = (rgb_mean[..., k] / 255.0 for k in range(3))
    y = kr * r + kg * g + kb * b
    return 16 + 219 * y, 128 + 224 * (b - y) / (2 * (1 - kb)), 128 + 224 * (r - y) / (2 * (1 - kr))


@pytest.mark.parametrize("matrix", [BT601, BT709])
def test_model_luma_within_half_a_step_of_float_for_every_colour(matrix):
    v = np.arange(1 << 24, dtype=np.uint32)
    px = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], axis=1).astype(np.uint8).reshape(4096, 4096, 3)
    y, _, _ = yuv420_model(px, matrix)
    yf, _, _ = _float_yuv(px.astype(np.float64), matrix)
    err = np.abs(y - yf)
    assert err.max() <= 0.51, err.max()
    assert y.min() >= 16 and y.max() <= 235


@pytest.mark.parametrize("matrix", [BT601, BT709])
def test_model_chroma_within_half_a_step_of_float_block_mean(matrix):
    rng = np.random.default_rng(11 + matrix)
    n = 1 << 20
    blocks = rng.integers(0, 256, size=(n, 2, 2, 3), dtype=np.uint8)
    blocks[:4096] = rng.integers(0, 2, size=(4096, 2, 2, 3), dtype=np.uint8) * 255        # extremes
    # n blocks side by side: a 2 x 2n image whose 2x2 block j is blocks[j]
    px = blocks.transpose(1, 0, 2, 3).reshape(2, 2 * n, 3)
    _, cb, cr = yuv420_model(px, matrix)
    _, cbf, crf = _float_yuv(blocks.astype(np.float64).mean(axis=(1, 2)), matrix)
    assert np.abs(cb[0] - cbf).max() <= 0.51 and np.abs(cr[0] - crf).max() <= 0.51
    for c in (cb, cr):
        assert c.min() >= 16 and c.max() <= 240


@pytest.mark.parametrize("matrix", [BT601, BT709])
def test_model_grey_has_neutral_chroma(matrix):
    grey = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, axis=1).reshape(16, 16, 3)
    y, cb, cr = yuv420_model(grey, matrix)
    assert (cb == 128).all() and (cr == 128).all()
    assert y[0, 0] == 16 and y[-1, -1] == 235 and (np.diff(y.ravel().astype(int)) >= 0).all()


RED, BLACK, BLUE = (255, 0, 0), (0, 0, 0), (0, 0, 255)


def test_model_hand_worked_1x1():
    for matrix in (BT601, BT709):
        y, cb, cr = yuv420_model(np.full((1, 1, 4), 255, np.uint8), matrix)     # white: (14071*255 + 8192) >> 14 = 219
        assert (y.tolist(), cb.tolist(), cr.tolist()) == ([[235]], [[128]], [[128]])
    # BT.601 red: Y = (4207*255 + 8192) >> 14 = 65, + 16; the block is 4 x red: Cb = (-2428*1020 + 32768) >> 16 = -38
    y, cb, cr = yuv420_model(np.array([[RED]], np.uint8), BT601)
    assert (y.tolist(), cb.tolist(), cr.tolist()) == ([[81]], [[90]], [[240]])


def test_model_hand_worked_1x3_and_3x1():
    # BT.601.  Block 0 = 2 x (red + black): SR = 510 -> Cb = (-2428*510 + 32768) >> 16 = -19, Cr = 56.
    # Block 1 covers columns 2 and 3 -> 2 (clamped) and rows 0, 1 -> 0: 4 x blue, SB = 1020 -> Cb = 112, Cr = -18.
    px = np.array([[RED, BLACK, BLUE]], np.uint8)
    y, cb, cr = yuv420_model(px, BT601)
    assert y.tolist() == [[81, 16, 41]]
    assert cb.tolist() == [[109, 240]] and cr.tolist() == [[184, 110]]
    y, cb, cr = yuv420_model(px.transpose(1, 0, 2), BT601)
    assert y.tolist() == [[81], [16], [41]]
    assert cb.tolist() == [[109], [240]] and cr.tolist() == [[184], [110]]


def test_model_hand_worked_3x3():
    px = np.zeros((3, 3, 3), np.uint8)
    px[0, 0] = RED
    px[2, 2] = BLUE
    px[0, 2] = px[2, 0] = RED
    y, cb, cr = yuv420_model(px, BT601)
    assert y.tolist() == [[81, 16, 81], [16, 16, 16], [81, 16, 41]]
    # block (0,0): one red of four -> SR = 255; (0,1): column 2 twice, rows 0..1 -> 2 x red; (1,0): row 2 twice,
    # column 0..1 -> 2 x red; (1,1): pixel (2,2) four times -> 4 x blue
    assert cb.tolist() == [[(-2428 * 255 + 32768 >> 16) + 128, 109], [109, 240]]
    assert cr.tolist() == [[(7196 * 255 + 32768 >> 16) + 128, 184], [184, 110]]


# ---- the Y4M reader ----
def _stream(w, h, frames, head_extra=" F30:1 Ip A1:1 C420jpeg XCOLORRANGE=LIMITED", frame_params=b""):
    return (f"YUV4MPEG2 W{w} H{h}{head_extra}\n".encode() + b"".join(b"FRAME" + frame_params + b"\n" + f for f in frames))


def test_read_y4m_hand_built_streams():
    rng = np.random.default_rng(5)
    for w, h in ((1, 1), (3, 5), (4, 2), (17, 9)):
        size = w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)
        frames = [rng.integers(0, 256, size, dtype=np.uint8).tobytes() for _ in range(3)]
        frames[1] = b"FRAME\n" * (size // 6) + b"F" * (size % 6)            # frame data that looks like markers
        header, got = read_y4m(_stream(w, h, frames))
        assert got == frames
        assert (header["W"], header["H"], header["F"], header["I"], header["A"], header["C"]) == (
            str(w), str(h), "30:1", "p", "1:1", "420jpeg")
        assert header["X"] == ["COLORRANGE=LIMITED"]
        assert read_y4m(_stream(w, h, frames, frame_params=b" Ixyz"))[1] == frames
    assert read_y4m(_stream(6, 4, []))[1] == []
    header, _ = read_y4m(_stream(2, 2, [], head_extra=" F24:1 C420"))
    assert header["F"] == "24:1" and header["X"] == []


def test_read_y4m_rejects_damage():
    good = _stream(4, 4, [bytes(24), bytes(24)])
    read_y4m(good)
    for bad in (good[:-1], b"YUV4MPEG3" + good[9:], good.replace(b"FRAME\n", b"FRAMX\n", 1),
                _stream(4, 4, [], head_extra=" C444")):
        with pytest.raises((AssertionError, ValueError)):
            read_y4m(bad)


# ---- the library's size function and refusals ----
def _expected_bytes(w, h):
    return w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)


@pytest.mark.parametrize("w,h", [(1, 1), (1, 2), (2, 1), (3, 5), (5, 3), (2, 2), (243, 181), (8200, 8), (3840, 2160),
                                 (7680, 4320), (1, 65536), (65536, 1), (65535, 65535), (65536, 65536)])
def test_yuv420_bytes_formula(hmrm, w, h):
    assert hmrm.yuv420_bytes(w, h) == _expected_bytes(w, h)


@pytest.mark.parametrize("w,h", [(0, 1), (1, 0), (0, 0), (-1, 5), (5, -2), (65537, 1), (1, 65537), (-2**31, 4)])
def test_yuv420_bytes_refuses_other_shapes(hmrm, w, h):
    assert hmrm.yuv420_bytes(w, h) == 0


def test_yuv_entry_points_refuse_null_context(hmrm):
    lib = hmrm.load_library()
    f = hmrm.Frame()
    lib.hmrm_frame_defaults(C.byref(f))
    buf = (C.c_uint8 * 64)()
    assert lib.hmrm_render_yuv420_async(None, C.byref(f), hmrm.YUV_BT709, buf, 64) == 1      # HMRM_ERR_INVALID
    px = (C.c_uint8 * 12)()
    assert lib.hmrm_convert_yuv420(None, px, 2, 2, 3, hmrm.YUV_BT709, buf, 64) == 1
    assert (hmrm.YUV_BT601, hmrm.YUV_BT709) == (BT601, BT709)


@pytest.mark.parametrize("args", [
    ["--video", "v.y4m"],                                                    # no --script
    ["--script", "frames.txt", "--video", "v.y4m", "--headless", "o.png"],
    ["--script", "frames.txt", "--video", "v.y4m", "--record"],
    ["--script", "frames.txt", "--video", "v.y4m", "--out-prefix", "p_"],
    ["--script", "frames.txt", "--video", "v.y4m", "--fps", "0"],
    ["--script", "frames.txt", "--video", "v.y4m", "--fps", "-3"],
    ["--script", "frames.txt", "--video", "v.y4m", "--fps", "many"],
    ["--script", "frames.txt", "--video", "v.y4m", "--video-matrix", "bt2020"],
    ["--script", "frames.txt", "--video", "v.y4m", "--video-matrix"],
])
def test_hmap_video_usage_refusals(hmrm, args, tmp_path):
    assert HMAP.exists(), "hmap host binary was not built"
    (tmp_path / "config.txt").write_text("resolution 64 48\n")
    (tmp_path / "frames.txt").write_text("hang 10\n")
    res = subprocess.run([str(HMAP), "config.txt", *args], capture_output=True, text=True, cwd=str(tmp_path))
    assert res.returncode == 1
    assert res.stderr.splitlines()[0] == "USAGE: hmap.exe path/to/config.txt"
    assert "--video FILE|-" in res.stderr and res.stdout == ""
    assert not (tmp_path / "v.y4m").exists()
