"""Glue between the parity scenes (tests/scenes.py) and the product API."""
from __future__ import annotations

import hashlib
import json
from pathlib import Path

import numpy as np

import scenes as S

GOLDEN = Path(__file__).resolve().parent / "golden"


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def golden_meta() -> dict:
    return json.loads((GOLDEN / "frames.json").read_text())


def golden_frames():
    return np.load(GOLDEN / "frames.npz")


def golden_replays() -> dict:
    return json.loads((GOLDEN / "replays.json").read_text())


def golden_kat() -> dict:
    return json.loads((GOLDEN / "kat.json").read_text())


def load_scene_maps(scene, oracle):
    return S.build_maps(scene["maps"], oracle.synth_maps)


def configure(renderer, scene, maps) -> None:
    """Set maps + lum/min/max on a product Renderer exactly as the scene's config file would."""
    hm, cm = maps
    renderer.lum_r, renderer.lum_g, renderer.lum_b = scene["lum"]
    renderer.min_height, renderer.max_height = scene["min_height"], scene["max_height"]
    renderer.set_maps(hm, cm)


def product_frame(hmrm, renderer, scene, **extra):
    kw = S.frame_kwargs(scene)
    f = renderer.frame(projection=scene["projection"], screen_width=kw["width"], screen_height=kw["height"],
                       cam_pos=kw["pos"], hang=hmrm.deg2rad(kw["hang_deg"]), vang=hmrm.deg2rad(kw["vang_deg"]),
                       hfov=hmrm.deg2rad(kw["hfov_deg"]), ortho_width=kw["ortho_width"],
                       grid_width=kw["grid_width"], step_dist=kw["step_dist"], bg=kw["bg"], cycle=0, cycle_period=1)
    for k, v in extra.items():
        setattr(f, k, v)
    return f


def oracle_frame(oracle, scene, **extra):
    return oracle.make_frame(projection=scene["projection"], **S.frame_kwargs(scene), **extra)


def oracle_render_scene(oracle, scene, maps, **extra):
    hm, cm = maps
    heights = oracle.update_heightmap(hm, scene["lum"], scene["min_height"], scene["max_height"])
    return oracle.render(oracle_frame(oracle, scene, **extra), heights, cm)


def fx(s: str) -> float:
    """C99 hex float text (printf %a or float.hex) -> float."""
    return float.fromhex(s)


def bits(v: float) -> int:
    """Bit pattern of a double; every NaN maps to one value (sign/payload of NaN are not part of the contract)."""
    import math
    import struct

    if math.isnan(v):
        return -1
    return struct.unpack("<q", struct.pack("<d", v))[0]


def same(v: float, golden_hex: str) -> bool:
    return bits(v) == bits(fx(golden_hex))
