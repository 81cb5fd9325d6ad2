"""ctypes binding of include/hmrm.h and the `Renderer` host object.

Everything that computes happens inside libhmrm.so on the GPU; this file only
marshals arguments.  numpy arrays are used for host buffers; torch tensors can be
passed through their data_ptr() to the *_device entry points (bench.py does that
for the NCCL band gather).
"""
from __future__ import annotations

import ctypes as C
import math
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent

PERSPECTIVE, SPHERICAL, ORTHOGRAPHIC = 1, 2, 3          # main/hmap.cpp:104-106
FP64_EXACT, FP32_FAST = 0, 1
TRAVERSAL_AUTO, TRAVERSAL_BRUTE, TRAVERSAL_SKIP, TRAVERSAL_SKIP_FP64, TRAVERSAL_PACK = 0, 1, 2, 3, 4
FLAG_STATS, FLAG_STEP_INDEX, FLAG_RAY_DUMP = 1, 2, 4
FLAG_SUPERSAMPLE_SHIFT = 8                               # flags bits 8-11 hold s - 1 (include/hmrm.h)
FLAG_SUPERSAMPLE_MASK = 15 << FLAG_SUPERSAMPLE_SHIFT
PIXEL_RGBA8, PIXEL_RGB8 = 0, 1
LAYOUT_ROWMAJOR, LAYOUT_TILE4, LAYOUT_ZORDER = 0, 1, 2
YUV_BT601, YUV_BT709 = 0, 1
JPEG_420, JPEG_444 = 0, 1


class HmrmError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"hmrm error {code}: {message}")
        self.code = code


class Frame(C.Structure):
    """`hmrm_frame` — the reference's per-frame render globals (main/hmap.cpp:28-112)."""

    _fields_ = [
        ("projection", C.c_int32),
        ("screen_width", C.c_int32),
        ("screen_height", C.c_int32),
        ("precision", C.c_int32),
        ("cam_pos", C.c_double * 3),
        ("hang", C.c_double),
        ("vang", C.c_double),
        ("hfov", C.c_double),
        ("ortho_width", C.c_double),
        ("grid_width", C.c_double),
        ("step_dist", C.c_double),
        ("bg", C.c_uint8 * 3),
        ("pixel_format", C.c_uint8),
        ("cycle", C.c_int32),
        ("cycle_period", C.c_int32),
        ("row_begin", C.c_int32),
        ("row_end", C.c_int32),
        ("traversal", C.c_int32),
        ("flags", C.c_uint32),
        ("band_count", C.c_int32),
        ("band_index", C.c_int32),
    ]


class Stats(C.Structure):
    """`hmrm_stats`."""

    _fields_ = [
        ("rays", C.c_int64),
        ("box_hits", C.c_int64),
        ("surf_hits", C.c_int64),
        ("steps", C.c_int64),
        ("fetches", C.c_int64),
        ("max_steps", C.c_int64),
        ("status", C.c_int32),
        ("reserved0", C.c_int32),
        ("kernel_ms", C.c_double),
    ]


# name -> (restype, argtypes); kept in step with include/hmrm.h (tests/test_abi.py checks both ways)
PROTOTYPES = {
    "hmrm_abi_version": (C.c_int, []),
    "hmrm_device_count": (C.c_int, []),
    "hmrm_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "hmrm_destroy": (None, [C.c_void_p]),
    "hmrm_last_error": (C.c_char_p, [C.c_void_p]),
    "hmrm_set_maps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "hmrm_set_maps_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "hmrm_synth_maps": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "hmrm_get_maps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "hmrm_set_maps16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "hmrm_set_maps16_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "hmrm_synth_maps16": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "hmrm_set_layout": (C.c_int, [C.c_void_p, C.c_int]),
    "hmrm_get_layout": (C.c_int, [C.c_void_p]),
    "hmrm_update_heightmap": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_double, C.c_double]),
    "hmrm_get_heights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmrm_frame_defaults": (None, [C.POINTER(Frame)]),
    "hmrm_render": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p]),
    "hmrm_render_device": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p, C.c_void_p]),
    "hmrm_render_async": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p]),
    "hmrm_wait": (C.c_int, [C.c_void_p]),
    "hmrm_wait_pending": (C.c_int, [C.c_void_p, C.c_int]),
    "hmrm_png_bound": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "hmrm_render_png_async": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p, C.c_size_t, C.c_void_p]),
    "hmrm_encode_png": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                  C.c_void_p]),
    "hmrm_jpeg_bound": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "hmrm_render_jpeg_async": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                         C.c_void_p]),
    "hmrm_encode_jpeg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "hmrm_yuv420_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "hmrm_render_yuv420_async": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_int32, C.c_void_p, C.c_size_t]),
    "hmrm_convert_yuv420": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_size_t]),
    "hmrm_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "hmrm_get_step_index": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmrm_get_ray_dump": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmrm_get_debug_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "hmrm_deg2rad": (C.c_double, [C.c_double]),
    "hmrm_camera_basis": (None, [C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "hmrm_get_ray": (C.c_int, [C.POINTER(Frame), C.c_double, C.c_double, C.POINTER(C.c_double),
                               C.POINTER(C.c_double)]),
    "hmrm_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "hmrm_host_alloc_flags": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t, C.c_uint32]),
    "hmrm_host_free": (None, [C.c_void_p]),
    "hmrm_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "hmrm_host_unregister": (C.c_int, [C.c_void_p]),
    "hmrm_device_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "hmrm_device_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmrm_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "hmrm_ipc_open": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "hmrm_ipc_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmrm_render_peer": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "hmrm_render_peer_staged": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                          C.c_void_p]),
    "hmrm_peer_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p]),
    "hmrm_peer_release": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "hmrm_peer_status": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]),
    "hmrm_peer_sync_mode": (C.c_int, [C.c_void_p]),
    "hmrm_debug_aabb": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


def library_path() -> Path:
    # HMRM_LIBRARY: another build of the SAME library (kernel experiments of tools/, e.g. variants/libhmrm_x.so)
    import os

    override = os.environ.get("HMRM_LIBRARY")
    return Path(override) if override else PKG / "libhmrm.so"


def load_library() -> C.CDLL:
    """Load libhmrm.so.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        path = library_path()
        if not path.exists():
            raise HmrmError(-1, f"{path} is missing: build it with `python {PKG.name}/build.py` "
                                "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(str(path))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def deg2rad(degrees: float) -> float:
    """DegreesToRads, main/hmap.cpp:131-133 (host arithmetic, identical rounding)."""
    return load_library().hmrm_deg2rad(float(degrees))


def camera_basis(hang: float, vang: float):
    look = (C.c_double * 3)()
    up = (C.c_double * 3)()
    load_library().hmrm_camera_basis(hang, vang, look, up)
    return tuple(look), tuple(up)


def get_ray(frame: Frame, w: float, h: float):
    """ImagePlane::GetRay of the plane `frame` describes (src/ImagePlane.hpp:10)."""
    pos = (C.c_double * 3)()
    d = (C.c_double * 3)()
    rc = load_library().hmrm_get_ray(C.byref(frame), w, h, pos, d)
    if rc:
        raise HmrmError(rc, "hmrm_get_ray: invalid frame")
    return tuple(pos), tuple(d)


def supersample_flag(s: int) -> int:
    """The flags bits of supersampling factor s (1..4): HMRM_FLAG_SUPERSAMPLE(s).  The frame stays W x H; each pixel is
    the box filter of the s x s pixels of the same camera's sW x sH frame."""
    if not isinstance(s, (int, np.integer)) or isinstance(s, bool) or not 1 <= int(s) <= 4:
        raise ValueError(f"supersample factor {s!r} is not one of 1, 2, 3, 4")
    return (int(s) - 1) << FLAG_SUPERSAMPLE_SHIFT


def png_bound(width: int, height: int, channels: int) -> int:
    """Worst-case PNG file size of a width x height x channels (3 | 4) frame (hmrm_png_bound); 0 for other shapes."""
    return int(load_library().hmrm_png_bound(int(width), int(height), int(channels)))


def jpeg_bound(width: int, height: int, chroma: int = JPEG_420) -> int:
    """Worst-case JPEG file size of a width x height frame in chroma mode JPEG_420 | JPEG_444 (hmrm_jpeg_bound);
    0 outside [1, 65535] per axis or for another chroma value."""
    return int(load_library().hmrm_jpeg_bound(int(width), int(height), int(chroma)))


def yuv420_bytes(width: int, height: int) -> int:
    """Bytes of the I420 planes of a width x height frame (hmrm_yuv420_bytes); 0 outside [1, 65536] per axis."""
    return int(load_library().hmrm_yuv420_bytes(int(width), int(height)))


def yuv420_planes(buf: np.ndarray, width: int, height: int):
    """(Y [H, W], Cb [ceil(H/2), ceil(W/2)], Cr) views of I420 bytes."""
    cw, ch = (width + 1) // 2, (height + 1) // 2
    y = buf[:width * height].reshape(height, width)
    cb = buf[width * height:width * height + cw * ch].reshape(ch, cw)
    cr = buf[width * height + cw * ch:width * height + 2 * cw * ch].reshape(ch, cw)
    return y, cb, cr


def _nbytes(a):
    """Size in bytes of a numpy array or torch tensor; None for a raw address."""
    if isinstance(a, np.ndarray):
        return a.nbytes
    if hasattr(a, "numel") and hasattr(a, "element_size"):
        return int(a.numel()) * int(a.element_size())
    return None


def _ptr(a) -> int:
    if a is None:
        return 0
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return int(a.data_ptr())
    return int(a)


class Renderer:
    """One rendering context on one CUDA device.

    Attribute names follow the reference's globals: screen_width, screen_height, hfov, hang,
    vang (radians), cam_pos, grid_width, step_dist, ortho_width, min_height, max_height,
    lum_r/g/b, bg_r/g/b, cycle, cycle_period, image_plane.  Defaults are the reference's
    (main/hmap.cpp:31-112) except cycle_period = 1.
    """

    def __init__(self, device: int = 0):
        self._lib = load_library()
        handle = C.c_void_p()
        rc = self._lib.hmrm_create(int(device), C.byref(handle))
        if rc:
            raise HmrmError(rc, self._lib.hmrm_last_error(None).decode())
        self._h = handle
        self.device = device
        f = Frame()
        self._lib.hmrm_frame_defaults(C.byref(f))
        self.screen_width, self.screen_height = f.screen_width, f.screen_height
        self.image_plane = f.projection
        self.cam_pos = list(f.cam_pos)
        self.hang, self.vang, self.hfov = f.hang, f.vang, f.hfov
        self.grid_width, self.step_dist, self.ortho_width = f.grid_width, f.step_dist, f.ortho_width
        self.bg_r = self.bg_g = self.bg_b = 0
        self.cycle, self.cycle_period = 0, 1
        self.min_height, self.max_height = 0.0, 10.0
        self.lum_r, self.lum_g, self.lum_b = 0.299, 0.587, 0.114
        self.precision = FP64_EXACT
        self.traversal = TRAVERSAL_AUTO
        self.map_width = self.map_height = 0

    # -- lifetime -------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.hmrm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int) -> None:
        if rc:
            raise HmrmError(rc, self._lib.hmrm_last_error(self._h).decode())

    # -- maps + prepass -------------------------------------------------------------------
    def set_maps(self, height_rgb8: np.ndarray, color_rgba8: np.ndarray) -> None:
        """heightmap / colormap as stb_image decodes them (main/hmap.cpp:320-321, :341-342)."""
        hm = np.ascontiguousarray(height_rgb8, dtype=np.uint8)
        cm = np.ascontiguousarray(color_rgba8, dtype=np.uint8)
        if hm.ndim != 3 or hm.shape[2] != 3 or cm.ndim != 3 or cm.shape[2] != 4:
            raise ValueError("height map must be [H,W,3] uint8 and colormap [H,W,4] uint8")
        if hm.shape[:2] != cm.shape[:2]:
            # main/hmap.cpp:503-515
            raise ValueError(f"heightmap dimensions ({hm.shape[1]}x{hm.shape[0]}) must match colormap "
                             f"dimensions ({cm.shape[1]}x{cm.shape[0]})")
        self._check(self._lib.hmrm_set_maps(self._h, hm.ctypes.data, cm.ctypes.data, hm.shape[1], hm.shape[0]))
        self.map_height, self.map_width = hm.shape[:2]
        self.update_heightmap()

    def set_maps_device(self, d_height_rgb8, d_color_rgba8, width: int, height: int) -> None:
        self._check(self._lib.hmrm_set_maps_device(self._h, _ptr(d_height_rgb8), _ptr(d_color_rgba8), width, height))
        self.map_height, self.map_width = height, width
        self.update_heightmap()

    def synth_maps(self, log2n: int, seed: int = 1234) -> None:
        """Synthetic fBm maps of size 2^log2n generated on the device (csrc/synth_fbm.h)."""
        self._check(self._lib.hmrm_synth_maps(self._h, log2n, seed))
        self.map_height = self.map_width = 1 << log2n
        self.update_heightmap()

    def set_maps16(self, height_u16: np.ndarray, color_rgba8: np.ndarray) -> None:
        """16-bit height samples [H,W] (used as R = G = B on the 0..65535 scale, include/hmrm.h) and the colormap."""
        hm = np.ascontiguousarray(height_u16, dtype=np.uint16)
        cm = np.ascontiguousarray(color_rgba8, dtype=np.uint8)
        if hm.ndim != 2 or cm.ndim != 3 or cm.shape[2] != 4:
            raise ValueError("height map must be [H,W] uint16 and colormap [H,W,4] uint8")
        if hm.shape != cm.shape[:2]:
            raise ValueError(f"heightmap dimensions ({hm.shape[1]}x{hm.shape[0]}) must match colormap "
                             f"dimensions ({cm.shape[1]}x{cm.shape[0]})")
        self._check(self._lib.hmrm_set_maps16(self._h, hm.ctypes.data, cm.ctypes.data, hm.shape[1], hm.shape[0]))
        self.map_height, self.map_width = hm.shape
        self.update_heightmap()

    def set_maps16_device(self, d_height_u16, d_color_rgba8, width: int, height: int) -> None:
        self._check(self._lib.hmrm_set_maps16_device(self._h, _ptr(d_height_u16), _ptr(d_color_rgba8), width, height))
        self.map_height, self.map_width = height, width
        self.update_heightmap()

    def synth_maps16(self, log2n: int, seed: int = 1234) -> None:
        """Synthetic 16-bit fBm height (hmrm_synth_height16) with synth_maps' colormap, generated on the device."""
        self._check(self._lib.hmrm_synth_maps16(self._h, log2n, seed))
        self.map_height = self.map_width = 1 << log2n
        self.update_heightmap()

    def get_maps(self):
        hm = np.empty((self.map_height, self.map_width, 3), dtype=np.uint8)
        cm = np.empty((self.map_height, self.map_width, 4), dtype=np.uint8)
        self._check(self._lib.hmrm_get_maps(self._h, hm.ctypes.data, cm.ctypes.data))
        return hm, cm

    def update_heightmap(self) -> None:
        """UpdateHeightmap (main/hmap.cpp:171-191) with the current lum_*/min_height/max_height."""
        lum = (C.c_double * 3)(self.lum_r, self.lum_g, self.lum_b)
        self._check(self._lib.hmrm_update_heightmap(self._h, lum, self.min_height, self.max_height))

    def set_layout(self, layout: int) -> None:
        """Layout of the height pyramid (LAYOUT_*); rebuilds the pyramid."""
        self._check(self._lib.hmrm_set_layout(self._h, int(layout)))
        if self.map_width:
            self.update_heightmap()

    def get_layout(self) -> int:
        return int(self._lib.hmrm_get_layout(self._h))

    def heights(self) -> np.ndarray:
        out = np.empty((self.map_height, self.map_width), dtype=np.float64)
        self._check(self._lib.hmrm_get_heights(self._h, out.ctypes.data))
        return out

    # -- render ---------------------------------------------------------------------------
    def frame(self, supersample: int | None = None, **overrides) -> Frame:
        """The hmrm_frame of the current attributes; `overrides` set Frame fields, `supersample` (1..4) the
        supersampling bits of its flags (the output size stays screen_width x screen_height)."""
        f = Frame()
        f.projection = self.image_plane
        f.screen_width, f.screen_height = self.screen_width, self.screen_height
        f.precision = self.precision
        f.cam_pos[:] = [float(v) for v in self.cam_pos]
        f.hang, f.vang, f.hfov = self.hang, self.vang, self.hfov
        f.ortho_width, f.grid_width, f.step_dist = self.ortho_width, self.grid_width, self.step_dist
        f.bg[:] = [self.bg_r & 255, self.bg_g & 255, self.bg_b & 255]
        f.cycle, f.cycle_period = self.cycle, self.cycle_period
        f.traversal = self.traversal
        for k, v in overrides.items():
            if k in ("cam_pos", "bg"):
                getattr(f, k)[:] = list(v)
            else:
                setattr(f, k, v)
        if supersample is not None:
            f.flags = (f.flags & ~FLAG_SUPERSAMPLE_MASK) | supersample_flag(supersample)
        return f

    def render(self, frame: Frame | None = None, out: np.ndarray | None = None, **overrides) -> np.ndarray:
        """One frame (main/hmap.cpp:952-1058) into a host RGBA8 [H,W,4] array."""
        f = frame if frame is not None else self.frame(**overrides)
        channels = 3 if f.pixel_format == PIXEL_RGB8 else 4
        if out is None:
            out = np.zeros((f.screen_height, f.screen_width, channels), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size == f.screen_height * f.screen_width * channels
        self._check(self._lib.hmrm_render(self._h, C.byref(f), out.ctypes.data))
        return out

    def render_async(self, frame: Frame, out) -> None:
        self._check(self._lib.hmrm_render_async(self._h, C.byref(frame), _ptr(out)))

    def wait(self) -> None:
        self._check(self._lib.hmrm_wait(self._h))

    def wait_pending(self, max_pending: int) -> None:
        """Streaming: return once at most `max_pending` (0..3) frames of render_async / render_png_async /
        render_yuv420_async / render_jpeg_async are still in flight."""
        self._check(self._lib.hmrm_wait_pending(self._h, max_pending))

    # -- PNG frames, deflated on the device -------------------------------------------------------
    def render_png_async(self, frame: Frame, out, size_out, capacity: int | None = None) -> None:
        """hmrm_render_png_async: `out` (pinned host or device memory of png_bound bytes or more) receives the PNG file,
        `size_out` (one uint64 in the same kinds of memory) its size, once wait / wait_pending covers the frame.
        numpy arrays and torch tensors report their own sizes; a raw address needs `capacity`."""
        capacity = self._file_capacity("render_png_async", out, size_out, capacity)
        self._check(self._lib.hmrm_render_png_async(self._h, C.byref(frame), _ptr(out), int(capacity), _ptr(size_out)))

    def render_png(self, frame: Frame | None = None, **overrides) -> bytes:
        """One frame as a complete PNG file (the decoded pixels are render()'s)."""
        f = frame if frame is not None else self.frame(**overrides)
        out, size = self._png_buffers(f.screen_width, f.screen_height, 3 if f.pixel_format == PIXEL_RGB8 else 4)
        self.render_png_async(f, out, size)
        self.wait()
        return out[:int(size[0])].tobytes()

    def encode_png(self, pixels: np.ndarray) -> bytes:
        """[H, W, 3 | 4] uint8 pixels -> PNG file, encoded on this context's device."""
        px = np.ascontiguousarray(pixels, dtype=np.uint8)
        if px.ndim != 3 or px.shape[2] not in (3, 4):
            raise ValueError("pixels must be [H, W, 3] or [H, W, 4] uint8")
        h, w, ch = px.shape
        out, size = self._png_buffers(w, h, ch)
        self._check(self._lib.hmrm_encode_png(self._h, px.ctypes.data, w, h, ch, out.ctypes.data, out.nbytes,
                                              size.ctypes.data))
        return out[:int(size[0])].tobytes()

    def _png_buffers(self, width: int, height: int, channels: int):
        """Pinned file + size buffers, kept for the last shape: pinning ~33 MB per 4K call would cost more than the
        encode."""
        bound = png_bound(width, height, channels)
        if bound == 0:
            raise ValueError(f"no PNG of {width}x{height}x{channels}")
        cached = getattr(self, "_png_cache", None)
        if cached is None or cached[0].nbytes < bound:
            cached = (pinned_empty((bound,)), pinned_empty((1,), dtype=np.uint64))
            self._png_cache = cached
        return cached

    # -- JPEG frames, encoded on the device ---------------------------------------------------------
    def render_jpeg_async(self, frame: Frame, out, size_out, quality: int = 90, chroma: int = JPEG_420,
                          capacity: int | None = None) -> None:
        """hmrm_render_jpeg_async: `out` (pinned host or device memory of jpeg_bound bytes or more) receives the JPEG
        file, `size_out` (one uint64 in the same kinds of memory) its size, once wait / wait_pending covers the frame.
        numpy arrays and torch tensors report their own sizes; a raw address needs `capacity`."""
        capacity = self._file_capacity("render_jpeg_async", out, size_out, capacity)
        self._check(self._lib.hmrm_render_jpeg_async(self._h, C.byref(frame), int(quality), int(chroma), _ptr(out),
                                                     int(capacity), _ptr(size_out)))

    def render_jpeg(self, frame: Frame | None = None, quality: int = 90, chroma: int = JPEG_420, **overrides) -> bytes:
        """One frame as a complete JPEG file (include/hmrm.h defines it to the byte)."""
        f = frame if frame is not None else self.frame(**overrides)
        out, size = self._jpeg_buffers(f.screen_width, f.screen_height, chroma)
        self.render_jpeg_async(f, out, size, quality, chroma)
        self.wait()
        return out[:int(size[0])].tobytes()

    def encode_jpeg(self, pixels, quality: int = 90, chroma: int = JPEG_420) -> bytes:
        """[H, W, 3 | 4] uint8 pixels (a numpy array, or a contiguous uint8 CUDA tensor of this device) -> JPEG file,
        encoded on this context's device."""
        if hasattr(pixels, "data_ptr") and getattr(pixels, "is_cuda", False):
            if pixels.dim() != 3 or pixels.shape[2] not in (3, 4) or not pixels.is_contiguous() or \
                    str(pixels.dtype) != "torch.uint8":
                raise ValueError("pixels must be a contiguous [H, W, 3] or [H, W, 4] uint8 tensor")
            h, w, ch = (int(v) for v in pixels.shape)
            ptr = int(pixels.data_ptr())
        else:
            px = np.ascontiguousarray(pixels, dtype=np.uint8)
            if px.ndim != 3 or px.shape[2] not in (3, 4):
                raise ValueError("pixels must be [H, W, 3] or [H, W, 4] uint8")
            h, w, ch = px.shape
            ptr = px.ctypes.data
        out, size = self._jpeg_buffers(w, h, chroma)
        self._check(self._lib.hmrm_encode_jpeg(self._h, ptr, w, h, ch, int(quality), int(chroma), out.ctypes.data,
                                               out.nbytes, size.ctypes.data))
        return out[:int(size[0])].tobytes()

    def _jpeg_buffers(self, width: int, height: int, chroma: int):
        """Pinned file + size buffers, kept while they are large enough (as _png_buffers)."""
        bound = jpeg_bound(width, height, chroma)
        if bound == 0:
            raise ValueError(f"no JPEG of {width}x{height} in chroma mode {chroma}")
        cached = getattr(self, "_jpeg_cache", None)
        if cached is None or cached[0].nbytes < bound:
            cached = (pinned_empty((bound,)), pinned_empty((1,), dtype=np.uint64))
            self._jpeg_cache = cached
        return cached[0][:bound], cached[1]

    @staticmethod
    def _file_capacity(name: str, out, size_out, capacity):
        """The capacity of a file destination (its own size unless given), after checking the size word."""
        if capacity is None:
            capacity = _nbytes(out)
            if capacity is None:
                raise ValueError(f"{name}: pass capacity= with a raw output address")
        size_bytes = _nbytes(size_out)
        if size_bytes is not None and (size_bytes < 8 or str(getattr(size_out, "dtype", "")).split(".")[-1]
                                       not in ("uint64", "int64")):
            raise ValueError(f"{name}: size_out must hold one 64-bit integer")
        return capacity

    # -- 4:2:0 video planes, converted on the device ----------------------------------------------
    def render_yuv420_async(self, frame: Frame, out, matrix: int = YUV_BT709, capacity: int | None = None) -> None:
        """hmrm_render_yuv420_async: `out` (pinned host or device memory of yuv420_bytes or more) receives the I420 planes
        once wait / wait_pending covers the frame.  numpy arrays and torch tensors report their own sizes; a raw address
        needs `capacity`."""
        if capacity is None:
            capacity = _nbytes(out)
            if capacity is None:
                raise ValueError("render_yuv420_async: pass capacity= with a raw output address")
        self._check(self._lib.hmrm_render_yuv420_async(self._h, C.byref(frame), int(matrix), _ptr(out), int(capacity)))

    def render_yuv420(self, frame: Frame | None = None, matrix: int = YUV_BT709, **overrides):
        """One frame as (Y, Cb, Cr) uint8 planes.  They are views of one pinned buffer that the next render_yuv420 or
        convert_yuv420 call overwrites: copy them to keep them."""
        f = frame if frame is not None else self.frame(**overrides)
        out = self._yuv_buffer(f.screen_width, f.screen_height)
        self.render_yuv420_async(f, out, matrix)
        self.wait()
        return yuv420_planes(out, f.screen_width, f.screen_height)

    def convert_yuv420(self, pixels: np.ndarray, matrix: int = YUV_BT709):
        """[H, W, 3 | 4] uint8 pixels -> (Y, Cb, Cr) planes, converted on this context's device; the same buffer as
        render_yuv420's."""
        px = np.ascontiguousarray(pixels, dtype=np.uint8)
        if px.ndim != 3 or px.shape[2] not in (3, 4):
            raise ValueError("pixels must be [H, W, 3] or [H, W, 4] uint8")
        h, w, ch = px.shape
        out = self._yuv_buffer(w, h)
        self._check(self._lib.hmrm_convert_yuv420(self._h, px.ctypes.data, w, h, ch, int(matrix), out.ctypes.data,
                                                  out.nbytes))
        return yuv420_planes(out, w, h)

    def _yuv_buffer(self, width: int, height: int) -> np.ndarray:
        """Pinned planes buffer of exactly the frame's size, kept while the shape repeats (as _png_buffers)."""
        n = yuv420_bytes(width, height)
        if n == 0:
            raise ValueError(f"no YUV frame of {width}x{height}")
        cached = getattr(self, "_yuv_cache", None)
        if cached is None or cached.nbytes < n:
            cached = pinned_empty((n,))
            self._yuv_cache = cached
        return cached[:n]

    def render_device(self, frame: Frame, d_out, stream=None) -> None:
        self._check(self._lib.hmrm_render_device(self._h, C.byref(frame), _ptr(d_out), _ptr(stream)))

    def stats(self) -> Stats:
        st = Stats()
        self._check(self._lib.hmrm_get_stats(self._h, C.byref(st)))
        return st

    def debug_counters(self) -> list:
        out = (C.c_int64 * 12)()
        self._check(self._lib.hmrm_get_debug_counters(self._h, out))
        return list(out)

    # ---- peer frames (one frame rendered by several GPUs, see include/hmrm.h) ----
    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self._lib.hmrm_device_alloc(self._h, nbytes, C.byref(p)))
        return int(p.value)

    def device_free(self, dptr: int) -> None:
        self._check(self._lib.hmrm_device_free(self._h, C.c_void_p(dptr)))

    def ipc_export(self, dptr: int) -> bytes:
        buf = (C.c_uint8 * 64)()
        self._check(self._lib.hmrm_ipc_export(self._h, C.c_void_p(dptr), buf))
        return bytes(buf)

    def ipc_open(self, handle: bytes) -> int:
        buf = (C.c_uint8 * 64).from_buffer_copy(handle)
        p = C.c_void_p()
        self._check(self._lib.hmrm_ipc_open(self._h, buf, C.byref(p)))
        return int(p.value)

    def ipc_close(self, dptr: int) -> None:
        self._check(self._lib.hmrm_ipc_close(self._h, C.c_void_p(dptr)))

    def ray_dump(self, frame: Frame) -> np.ndarray:
        """[H, W, 10] float64 of the last FLAG_RAY_DUMP render: pos, dir, distance(), entry point — as the DEVICE computed them."""
        out = np.empty((frame.screen_height, frame.screen_width, 10), dtype=np.float64)
        self._check(self._lib.hmrm_get_ray_dump(self._h, out.ctypes.data))
        return out

    def render_peer(self, frame: Frame, d_frame: int, d_ctrl: int, use: int, stream=None) -> None:
        self._check(self._lib.hmrm_render_peer(self._h, C.byref(frame), C.c_void_p(d_frame), C.c_void_p(d_ctrl), use,
                                               _ptr(stream)))

    def render_peer_staged(self, frame: Frame, d_stage, d_frame: int, d_ctrl: int, use: int, stream=None) -> None:
        self._check(self._lib.hmrm_render_peer_staged(self._h, C.byref(frame), _ptr(d_stage), C.c_void_p(d_frame),
                                                      C.c_void_p(d_ctrl), use, _ptr(stream)))

    def peer_wait(self, d_ctrl: int, use: int, ranks: int, stream=None) -> None:
        self._check(self._lib.hmrm_peer_wait(self._h, C.c_void_p(d_ctrl), use, ranks, _ptr(stream)))

    def peer_release(self, d_ctrl: int, use: int, stream=None) -> None:
        self._check(self._lib.hmrm_peer_release(self._h, C.c_void_p(d_ctrl), use, _ptr(stream)))

    def peer_sync_mode(self) -> str:
        """Which implementation of the peer-frame protocol this context uses: "memops" or "kernels"."""
        return "memops" if self._lib.hmrm_peer_sync_mode(self._h) == 1 else "kernels"

    def peer_status(self, d_ctrl: int):
        out = (C.c_uint32 * 3)()
        self._check(self._lib.hmrm_peer_status(self._h, C.c_void_p(d_ctrl), out))
        return tuple(out)

    def debug_aabb(self, rays: np.ndarray, boxes: np.ndarray) -> np.ndarray:
        """The device's slab test on [n,6] rays (pos, dir) and [n,6] boxes (c0, c1) -> [n,5] (distance, hit, entry)."""
        rays = np.ascontiguousarray(rays, dtype=np.float64)
        boxes = np.ascontiguousarray(boxes, dtype=np.float64)
        out = np.empty((rays.shape[0], 5), dtype=np.float64)
        self._check(self._lib.hmrm_debug_aabb(self._h, rays.shape[0], rays.ctypes.data, boxes.ctypes.data, out.ctypes.data))
        return out

    def step_index(self, frame: Frame) -> np.ndarray:
        out = np.empty((frame.screen_height, frame.screen_width), dtype=np.int32)
        self._check(self._lib.hmrm_get_step_index(self._h, out.ctypes.data))
        return out


def pinned_empty(shape, dtype=np.uint8, write_combined: bool = False) -> np.ndarray:
    """numpy array over page-locked host memory (hmrm_host_alloc); freed when garbage collected."""
    lib = load_library()
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    rc = lib.hmrm_host_alloc_flags(C.byref(p), nbytes, 1 if write_combined else 0)
    if rc:
        raise HmrmError(rc, lib.hmrm_last_error(None).decode())
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib.hmrm_host_free(self.ptr)
            except Exception:
                pass

    _owners[id(buf)] = _Owner(p)
    return arr


_owners: dict = {}
