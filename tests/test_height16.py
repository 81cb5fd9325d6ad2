"""CPU: the 16-bit height definition (include/hmrm.h, hmrm_set_maps16), the synthetic 16-bit map, `hmap`'s 16-bit
heightmap ingest (--decode-image ... h16, --height-bits) and the NULL-context refusals of the new entry points."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import height16_lib as H

ROOT = Path(__file__).resolve().parent.parent
HMAP = ROOT / "heightmap-ray-marcher_b200" / "hmap"

UNIT_LUMS = [(1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0)]
RANGES = [(0.0, 10.0), (0.0, 2.5), (-1.25, 1.5), (0.75, 2.5), (3.0, -2.0)]
LUMS = [(0.299, 0.587, 0.114), (-0.2, 1.4, 0.1), (1.7, 2.3, 0.9), (-1.0, -0.5, -0.25), (0.9, 0.05, 0.3)]


def same_bits(a, b) -> bool:
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


@pytest.mark.parametrize("lum", UNIT_LUMS)
@pytest.mark.parametrize("rng", RANGES)
def test_model_equals_8bit_oracle_for_widened_grey(oracle, lum, rng):
    """x = 257 v8 with a unit lum vector: v / 65535 and v8 / 255 are the same correctly rounded number."""
    v8 = np.arange(256, dtype=np.uint8)
    want = oracle.update_heightmap(np.repeat(v8[None, :, None], 3, axis=2), lum, *rng)[0]
    got = H.heights16(v8.astype(np.uint16) * 257, lum, *rng)
    assert same_bits(got, want)


@pytest.mark.parametrize("lum", LUMS)
@pytest.mark.parametrize("rng", RANGES)
def test_model_equals_c_statement_for_every_sample(lum, rng):
    x = np.arange(65536, dtype=np.uint16)
    assert same_bits(H.heights16(x, lum, *rng), H.c_heights16(x, lum, *rng))


def test_synth_height16_tracks_synth_height(oracle):
    hm8, cm8 = oracle.synth_maps(8, 1234)
    hm16, cm16 = H.synth_maps16(8, 1234)
    d = (hm16 >> 8).astype(np.int32) - hm8[:, :, 0].astype(np.int32)
    assert np.abs(d).max() <= 1
    assert np.array_equal(cm16, cm8)              # the same colormap as hmrm_synth_maps
    assert len(np.unique(hm16)) > 4 * len(np.unique(hm8))


# ---- ingest ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hmap(hmrm):
    assert HMAP.exists(), "hmap host binary was not built"
    return HMAP


def decode16(hmap, path, tmp_path):
    out = tmp_path / "out.raw"
    res = subprocess.run([str(hmap), "--decode-image", str(path), "h16", str(out)], capture_output=True, text=True)
    if res.returncode != 0:
        return None, res.stderr
    w, h, c = (int(v) for v in res.stdout.split())
    assert c == 1
    return np.fromfile(out, dtype="<u2").reshape(h, w), res.stderr


def noise16(h, w, seed=3):
    return np.random.default_rng(seed).integers(0, 65536, size=(h, w), dtype=np.uint16)


@pytest.mark.parametrize("interlace", [False, True])
@pytest.mark.parametrize("filt", [0, 1, 2, 3, 4, None])
def test_decode_grey16_png(hmap, tmp_path, filt, interlace):
    x = noise16(19, 23)
    x[0, :4] = [0, 1, 65534, 65535]
    p = tmp_path / "g.png"
    H.write_png16(p, x, filters=(0, 1, 2, 3, 4) if filt is None else (filt,), interlace=interlace)
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)


@pytest.mark.parametrize("interlace", [False, True])
def test_decode_grey_alpha16_png_drops_alpha(hmap, tmp_path, interlace):
    x = noise16(17, 9, seed=4)
    a = noise16(17, 9, seed=5)
    p = tmp_path / "ga.png"
    H.write_png16(p, np.stack([x, a], axis=2), interlace=interlace)
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)


@pytest.mark.parametrize("channels", [3, 4])
def test_decode_rgb16_png_grey_accepted_colour_refused(hmap, tmp_path, channels):
    x = noise16(11, 13, seed=6)
    planes = [x, x, x] + ([noise16(11, 13, seed=7)] if channels == 4 else [])
    p = tmp_path / "rgb.png"
    H.write_png16(p, np.stack(planes, axis=2))
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)
    g = x.copy()
    g[5, 7] ^= 1                                   # one pixel with R != G
    planes[1] = g
    q = tmp_path / "colour.png"
    H.write_png16(q, np.stack(planes, axis=2))
    got, err = decode16(hmap, q, tmp_path)
    assert got is None
    assert str(q) in err and "not grey" in err


@pytest.mark.parametrize("interlace", [False, True])
def test_decode_16bit_png_with_colour_key(hmap, tmp_path, interlace):
    """A tRNS colour key adds an alpha channel to the decoded pixels, not to the file's 16-bit samples."""
    x = noise16(9, 11, seed=11)
    key = int(x[4, 5])
    p = tmp_path / "g_trns.png"
    H.write_png16(p, x, interlace=interlace, trns=(key,))
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)
    q = tmp_path / "rgb_trns.png"
    H.write_png16(q, np.stack([x, x, x], axis=2), interlace=interlace, trns=(key, key, key))
    got, err = decode16(hmap, q, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)
    g = x.copy()
    g[2, 3] ^= 1
    r = tmp_path / "colour_trns.png"
    H.write_png16(r, np.stack([x, g, x], axis=2), interlace=interlace, trns=(key, key, key))
    got, err = decode16(hmap, r, tmp_path)
    assert got is None
    assert str(r) in err and "not grey" in err


def test_decode_ppm16_grey_accepted_colour_refused(hmap, tmp_path):
    x = noise16(6, 13, seed=12)
    p = tmp_path / "g.ppm"
    H.write_pgm16(p, np.stack([x, x, x], axis=2))
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)
    g = x.copy()
    g[1, 1] ^= 256
    q = tmp_path / "colour.ppm"
    H.write_pgm16(q, np.stack([x, g, x], axis=2))
    got, err = decode16(hmap, q, tmp_path)
    assert got is None
    assert str(q) in err and "not grey" in err


@pytest.mark.parametrize("maxval", [65535, 1000, 256])
def test_decode_pgm16_keeps_samples(hmap, tmp_path, maxval):
    x = (noise16(7, 31, seed=8).astype(np.uint32) % (maxval + 1)).astype(np.uint16)
    p = tmp_path / "g.pgm"
    H.write_pgm16(p, x, maxval)
    got, err = decode16(hmap, p, tmp_path)
    assert got is not None, err
    assert np.array_equal(got, x)


def test_decode_8bit_grey_files_widened(hmap, oracle, tmp_path):
    from PIL import Image

    v8 = np.random.default_rng(9).integers(0, 256, size=(21, 14), dtype=np.uint8)
    want = v8.astype(np.uint16) * 257
    files = []
    p = tmp_path / "g8.png"
    Image.fromarray(v8, "L").save(p)
    files.append(p)
    p = tmp_path / "g8.pgm"
    p.write_bytes(b"P5\n14 21\n255\n" + v8.tobytes())
    files.append(p)
    p = tmp_path / "rgb8.bmp"
    Image.fromarray(np.repeat(v8[:, :, None], 3, axis=2), "RGB").save(p)
    files.append(p)
    p = tmp_path / "rgb8.ppm"
    oracle.write_ppm(p, np.repeat(v8[:, :, None], 3, axis=2))
    files.append(p)
    for f in files:
        got, err = decode16(hmap, f, tmp_path)
        assert got is not None, (f, err)
        assert np.array_equal(got, want), f


def test_decode_8bit_colour_refused(hmap, oracle, tmp_path):
    rgb = np.random.default_rng(10).integers(0, 256, size=(6, 8, 3), dtype=np.uint8)
    p = tmp_path / "colour.png"
    oracle.write_png(p, rgb)
    got, err = decode16(hmap, p, tmp_path)
    assert got is None
    assert str(p) in err and "not grey" in err


def test_decode_unreadable_refused(hmap, tmp_path):
    p = tmp_path / "junk.png"
    p.write_bytes(b"\x89PNG\r\n\x1a\n" + b"\0" * 20)
    got, err = decode16(hmap, p, tmp_path)
    assert got is None and str(p) in err
    got, err = decode16(hmap, tmp_path / "missing.png", tmp_path)
    assert got is None and "missing.png" in err


# ---- hmap options ---------------------------------------------------------------------------------------------------
def write_config(tmp_path, hm, cm) -> Path:
    cfg = tmp_path / "config.txt"
    cfg.write_text(f"resolution 64 48\nheightmap {hm}\ncolormap {cm}\n")
    return cfg


@pytest.mark.parametrize("bits", ["12", "0", "sixteen", "-16"])
def test_height_bits_other_values_are_usage_errors(hmap, oracle, tmp_path, bits):
    hm = tmp_path / "h.png"
    H.write_png16(hm, noise16(8, 8))
    cm = tmp_path / "c.png"
    oracle.write_png(cm, np.zeros((8, 8, 4), np.uint8))
    res = subprocess.run([str(hmap), str(write_config(tmp_path, hm, cm)), "--height-bits", bits, "--parse-only"],
                         capture_output=True, text=True)
    assert res.returncode == 1 and "USAGE" in res.stderr


def test_parse_only_height_bits_16(hmap, oracle, tmp_path):
    cm = tmp_path / "c.png"
    oracle.write_png(cm, np.zeros((8, 8, 4), np.uint8))
    grey = tmp_path / "h.png"
    H.write_png16(grey, noise16(8, 8))
    cfg = write_config(tmp_path, grey, cm)
    res = subprocess.run([str(hmap), str(cfg), "--height-bits", "16", "--parse-only"], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    # an 8-bit reader of the same file works too (stb keeps the high byte)
    res = subprocess.run([str(hmap), str(cfg), "--parse-only"], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    # a colour heightmap is refused at 16 bits, naming the file
    colour = tmp_path / "colour.png"
    oracle.write_png(colour, np.random.default_rng(1).integers(0, 256, size=(8, 8, 3), dtype=np.uint8))
    cfg = write_config(tmp_path, colour, cm)
    res = subprocess.run([str(hmap), str(cfg), "--height-bits", "16", "--parse-only"], capture_output=True, text=True)
    assert res.returncode == 1
    assert f"Failed to load image for heightmap from {colour}" in res.stderr and "not grey" in res.stderr
    # the size check uses the 16-bit map
    small = tmp_path / "small.png"
    H.write_png16(small, noise16(5, 7))
    cfg = write_config(tmp_path, small, cm)
    res = subprocess.run([str(hmap), str(cfg), "--height-bits", "16", "--parse-only"], capture_output=True, text=True)
    assert res.returncode == 1
    assert "heightmap dimensions (7x5) must match colormap dimensions (8x8)" in res.stderr


def test_new_entry_points_refuse_null_context(hmrm):
    lib = hmrm.load_library()
    buf16 = np.zeros(4, np.uint16)
    buf8 = np.zeros(16, np.uint8)
    assert lib.hmrm_set_maps16(None, buf16.ctypes.data, buf8.ctypes.data, 2, 2) == 1
    assert lib.hmrm_set_maps16_device(None, buf16.ctypes.data, buf8.ctypes.data, 2, 2) == 1
    assert lib.hmrm_synth_maps16(None, 8, 1234) == 1
