"""heightmap-ray-marcher_b200 — host-side mirror of the reference's render interface over
libhmrm.so (hand-written sm_100a CUDA behind the C ABI in include/hmrm.h).

The reference (Costava/heightmap-ray-marcher) drives its hot path through global
variables set by a config grammar (main/hmap.cpp:28-112, :309-520).  `Renderer`
keeps the same names and meanings as attributes; `Renderer.render()` is the
replacement for the frame body main/hmap.cpp:952-1058.

There is no CPU path here: importing works anywhere, but creating a Renderer
without the built library or without a CUDA device raises.
"""
from __future__ import annotations

from .binding import (  # noqa: F401
    FP32_FAST,
    FP64_EXACT,
    FLAG_RAY_DUMP,
    FLAG_STATS,
    FLAG_STEP_INDEX,
    FLAG_SUPERSAMPLE_MASK,
    FLAG_SUPERSAMPLE_SHIFT,
    JPEG_420,
    JPEG_444,
    LAYOUT_ROWMAJOR,
    LAYOUT_TILE4,
    LAYOUT_ZORDER,
    PIXEL_RGB8,
    PIXEL_RGBA8,
    ORTHOGRAPHIC,
    PERSPECTIVE,
    SPHERICAL,
    TRAVERSAL_AUTO,
    TRAVERSAL_BRUTE,
    TRAVERSAL_PACK,
    TRAVERSAL_SKIP,
    TRAVERSAL_SKIP_FP64,
    YUV_BT601,
    YUV_BT709,
    Camera,
    Frame,
    HmrmError,
    Renderer,
    Stats,
    camera_basis,
    deg2rad,
    get_ray,
    jpeg_bound,
    library_path,
    load_library,
    pinned_empty,
    png_bound,
    supersample_flag,
    yuv420_bytes,
)

__all__ = [
    "Renderer", "Frame", "Camera", "Stats", "HmrmError", "load_library", "library_path", "deg2rad", "camera_basis",
    "get_ray", "png_bound", "yuv420_bytes", "pinned_empty", "PERSPECTIVE", "SPHERICAL", "ORTHOGRAPHIC", "FP64_EXACT", "FP32_FAST", "TRAVERSAL_AUTO",
    "TRAVERSAL_BRUTE", "TRAVERSAL_SKIP", "TRAVERSAL_PACK", "FLAG_STATS", "FLAG_STEP_INDEX", "FLAG_RAY_DUMP", "PIXEL_RGBA8", "PIXEL_RGB8",
    "LAYOUT_ROWMAJOR", "LAYOUT_TILE4", "LAYOUT_ZORDER", "YUV_BT601", "YUV_BT709",
    "FLAG_SUPERSAMPLE_SHIFT", "FLAG_SUPERSAMPLE_MASK", "supersample_flag", "jpeg_bound", "JPEG_420", "JPEG_444",
]
