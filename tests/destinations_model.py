"""Which pixels a render call writes, restated from include/hmrm.h, and the destination bytes expected after it.

The GPU destination tests (tests/test_gpu_destinations.py) build every expected byte from this model and the CPU
oracle's frame alone; tests/test_destinations_model.py checks the model against the oracle's own cycle loop and
multi_gpu.owned_pixel_rows, so that a wrong model cannot make the GPU tests agree with a wrong kernel.
"""
from __future__ import annotations

import numpy as np

TILE_ROWS = 4      # screen tiles are 8 x 4 pixels


def selected(W, H, row_begin=0, row_end=0, band_count=0, band_index=0, cycle=0, period=1) -> np.ndarray:
    """bool [H, W]: the pixels of a W x H frame that a render call with this selection writes.

    - the row band [row_begin, row_end) (0, 0 = all rows);
    - band_count > 1: tile rows of 4 pixel rows are counted from row_begin, and band b owns tile rows t with
      t % band_count == b;
    - pixel p = py * W + px is selected when p >= cycle and (p - cycle) % period == 0."""
    if row_begin == 0 and row_end == 0:
        row_end = H
    py = np.arange(H, dtype=np.int64)[:, None]
    px = np.arange(W, dtype=np.int64)[None, :]
    rows = (py >= row_begin) & (py < row_end)
    if band_count > 1:
        rows &= ((py - row_begin) // TILE_ROWS) % band_count == band_index
    p = py * W + px
    return rows & (p >= cycle) & ((p - cycle) % period == 0)


def sentinel_bytes(rng, n: int) -> np.ndarray:
    """n guard / fill bytes, none of them 0 or 255 (the values a wrong store of black or of alpha would leave)."""
    return rng.integers(1, 255, size=n, dtype=np.uint8)


def expected_destination(fill: np.ndarray, offset: int, frame: np.ndarray, mask: np.ndarray, channels: int) -> np.ndarray:
    """The allocation `fill` after a render into it at byte `offset`: the `channels` first bytes of each pixel of
    `frame` ([H, W, >= channels]) at the pixels of `mask`, every other byte as filled."""
    H, W = mask.shape
    out = fill.copy()
    view = out[offset:offset + H * W * channels].reshape(H, W, channels)
    view[mask] = frame[mask][:, :channels]
    return out
