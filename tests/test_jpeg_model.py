"""CPU: the JPEG model (tests/jpeg_model.py) against Pillow's libjpeg-turbo byte for byte, so that the device encoder
(K6) is tested against files whose definition is known to be right; hmrm_jpeg_bound's formula and that it holds the
model's largest files; the JPEG entry points refuse their limits and a NULL context; the exact-reciprocal quantiser
and jfdctint's 32-bit arithmetic, checked exhaustively."""
import io

import numpy as np
import pytest
from PIL import Image

import jpeg_model as M


def pil_jpeg(rgb: np.ndarray, q: int, s420: bool) -> bytes:
    b = io.BytesIO()
    Image.fromarray(np.ascontiguousarray(rgb[:, :, :3])).save(b, format="JPEG", quality=q, subsampling=2 if s420 else 0,
                                                               restart_marker_rows=1)
    return b.getvalue()


def content(kind: str, h: int, w: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3)).astype(np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(xx * 5 + yy * 3) % 256, (yy * 7) % 256, (xx * xx + yy) % 256], 2).astype(np.uint8)


GRID_SHAPES = [(8, 8), (16, 16), (37, 53), (1, 1), (17, 33), (31, 9), (64, 48), (23, 101), (40, 130), (130, 17)]


@pytest.mark.parametrize("h,w", GRID_SHAPES)
def test_model_equals_pillow_grid(h, w):
    """sizes x {noise, smooth} x q {1, 10, 50, 75, 90, 100} x {4:4:4, 4:2:0} x restart intervals {one MCU row, none,
    1 MCU, 3 MCUs}: 960 files over the ten shapes."""
    for kind in ("noise", "smooth"):
        a = content(kind, h, w, seed=h * 1000 + w)
        for q in (1, 10, 50, 75, 90, 100):
            for ss in (0, 2):
                for rst in (None, 0, 1, 3):
                    kw = dict(restart_marker_rows=1) if rst is None else dict(restart_marker_blocks=rst) if rst else {}
                    b = io.BytesIO()
                    Image.fromarray(a).save(b, format="JPEG", quality=q, subsampling=ss, **kw)
                    assert M.write(a, q, ss == 2, rst) == b.getvalue(), (kind, q, ss, rst)


@pytest.mark.parametrize("q", [1, 49, 50, 51, 100])
@pytest.mark.parametrize("s420", [False, True])
def test_model_equals_pillow_at_quality_edges(q, s420):
    for kind in ("noise", "smooth"):
        a = content(kind, 29, 45, seed=q)
        assert M.write(a, q, s420) == pil_jpeg(a, q, s420)


@pytest.mark.parametrize("h,w", [(1, 7), (1, 40), (7, 1), (40, 1), (1, 17), (17, 1)])
@pytest.mark.parametrize("s420", [False, True])
def test_model_equals_pillow_one_pixel_wide(h, w, s420):
    for kind in ("noise", "smooth"):
        a = content(kind, h, w, seed=h + w)
        assert M.write(a, 75, s420) == pil_jpeg(a, 75, s420)


@pytest.mark.parametrize("h,w", [(9, 17), (25, 41), (15, 31), (47, 15), (16, 32), (48, 16)])   # 1 mod 8, 15 mod 16, 0 mod 16
@pytest.mark.parametrize("s420", [False, True])
def test_model_equals_pillow_edge_sizes(h, w, s420):
    for kind in ("noise", "smooth"):
        a = content(kind, h, w, seed=h * w)
        assert M.write(a, 90, s420) == pil_jpeg(a, 90, s420)


def expected_bound(w, h, s420):
    m = 16 if s420 else 8
    mcus = -(-w // m) * -(-h // m)
    return 631 + 415 * mcus * (6 if s420 else 3) + 4 * -(-h // m)


@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (17, 33), (181, 243), (1920, 1080), (3840, 2160), (65535, 2),
                                 (2, 65535), (16384, 8192), (65535, 65535)])
def test_jpeg_bound_formula(hmrm, w, h):
    assert hmrm.jpeg_bound(w, h, hmrm.JPEG_420) == expected_bound(w, h, True)
    assert hmrm.jpeg_bound(w, h, hmrm.JPEG_444) == expected_bound(w, h, False)


@pytest.mark.parametrize("h,w", [(8, 8), (37, 53), (64, 48), (130, 17)])
def test_jpeg_bound_holds_noise_at_quality_100(hmrm, h, w):
    a = content("noise", h, w, seed=7)
    for s420, chroma in ((True, hmrm.JPEG_420), (False, hmrm.JPEG_444)):
        assert len(M.write(a, 100, s420)) <= hmrm.jpeg_bound(w, h, chroma)


@pytest.mark.parametrize("w,h,chroma", [(0, 5, 0), (5, 0, 1), (-1, 5, 0), (65536, 2, 0), (2, 65536, 1), (5, 5, 2),
                                        (5, 5, -1)])
def test_jpeg_bound_refuses_other_shapes(hmrm, w, h, chroma):
    assert hmrm.jpeg_bound(w, h, chroma) == 0


def test_jpeg_entry_points_refuse_limits_and_null_context(hmrm):
    import ctypes as C

    lib = hmrm.load_library()
    f = hmrm.Frame()
    lib.hmrm_frame_defaults(C.byref(f))
    buf = (C.c_uint8 * 4096)()
    size = C.c_uint64()
    px = (C.c_uint8 * 12)()
    for q, chroma in ((90, 0), (0, 0), (101, 0), (90, 2)):
        assert lib.hmrm_render_jpeg_async(None, C.byref(f), q, chroma, buf, 4096, C.byref(size)) == 1  # HMRM_ERR_INVALID
        assert lib.hmrm_encode_jpeg(None, px, 2, 2, 3, q, chroma, buf, 4096, C.byref(size)) == 1
    assert lib.hmrm_encode_jpeg(None, px, 65536, 1, 3, 90, 0, buf, 4096, C.byref(size)) == 1
    assert lib.hmrm_encode_jpeg(None, None, 2, 2, 3, 90, 0, None, 4096, None) == 1
    assert lib.hmrm_render_jpeg_async(None, None, 90, 0, None, 0, None) == 1


def test_reciprocal_quantiser_is_exact():
    """k6_jpeg_blocks divides a = |c| + 4t by 8t as umulhi(a, ceil(2^32 / 8t)): equal to the division for every
    |c| <= 2^15 and every table entry t (jfdctint's |c| is at most 8192)."""
    c = np.arange(0, (1 << 15) + 1, dtype=np.uint64)
    for t in range(1, 256):
        d = np.uint64(8 * t)
        m = np.uint64(((1 << 32) + 8 * t - 1) // (8 * t))
        a = c + np.uint64(4 * t)
        assert np.array_equal((a * m) >> np.uint64(32), a // d), t


def _fdct1(v, pass1: bool):
    """jfdctint's 1-D pass on 8 linear forms -> (every intermediate before a descale, the 8 outputs)."""
    t0, t7, t1, t6, t2, t5, t3, t4 = (v[0] + v[7], v[0] - v[7], v[1] + v[6], v[1] - v[6], v[2] + v[5], v[2] - v[5],
                                      v[3] + v[4], v[3] - v[4])
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    z1 = (t12 + t13) * 4433
    z5 = (t4 + t6 + t5 + t7) * 9633
    a4, a5, a6, a7 = t4 * 2446, t5 * 16819, t6 * 25172, t7 * 12299
    y1, y2 = (t4 + t7) * -7373, (t5 + t6) * -20995
    y3, y4 = (t4 + t6) * -16069 + z5, (t5 + t7) * -3196 + z5
    e2, e6 = z1 + t13 * 6270, z1 - t12 * 15137
    o7, o5, o3, o1 = a4 + y1 + y3, a5 + y2 + y4, a6 + y2 + y3, a7 + y1 + y4
    inter = [t0, t7, t1, t6, t2, t5, t3, t4, t10, t13, t11, t12, z1, z5, a4, a5, a6, a7, y1, y2, y3, y4, e2, e6,
             o7, o5, o3, o1]
    sh = 2.0 ** (11 if pass1 else 15)
    even = 4.0 if pass1 else 0.25
    return inter, [(t10 + t11) * even, o1 / sh, e2 / sh, o3 / sh, (t10 - t11) * even, o5 / sh, e6 / sh, o7 / sh]


def test_fdct_fits_32_bits():
    """Every intermediate of jfdctint is a linear form of the 64 level-shifted samples (|x| <= 128) plus, in pass 2,
    the effect of pass 1's rounding (at most 1/2 per pass-1 output); the largest magnitude of a form is 128 times the
    sum of its |weights|.  K6 computes in 32-bit integers, so each must stay below 2^31."""
    unit = np.eye(64).reshape(8, 8, 64)
    pass1 = [_fdct1([unit[r, c] for c in range(8)], True) for r in range(8)]
    big1 = max(128 * np.abs(x).sum() for inter, _ in pass1 for x in inter)
    big2 = max(128 * np.abs(x).sum() for c in range(8) for x in _fdct1([pass1[r][1][c] for r in range(8)], False)[0])
    eye8 = np.eye(8)
    slack = max(0.5 * np.abs(x).sum() for x in _fdct1([eye8[r] for r in range(8)], False)[0])
    assert big1 < 2 ** 23.5
    assert big2 + slack < 2 ** 28.5
