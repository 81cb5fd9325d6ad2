"""4:2:0 video output of the bench's flythrough4k cameras on one GPU; prints one JSON line.

    python tools/yuv_probe.py [--frames 240] [--out FILE]

- k4_yuv420 per 4K frame: kernel durations from torch.profiler (CUPTI device timestamps) over --frames render + YUV
  frames, after a warm-up; the render kernel's time in the same window for comparison;
- frames per second, 4 in flight into pinned host memory, of render + YUV (hmrm_render_yuv420_async), render + raw RGB8,
  render + raw RGBA8 (hmrm_render_async) and render + PNG (hmrm_render_png_async): host clock around the whole window,
  which ends in a synchronise; each measured twice, the four alternating;
- `hmap --script --video` (one Y4M file) against `hmap --script` (one PNG file per frame), both writing to /dev/shm:
  seconds per frame after start-up;
- the goals: K4 <= 25 us per 4K frame, and render + YUV frames/s >= render + raw RGB8 frames/s.
A sample of the frames is checked against the numpy model of tests/test_yuv420.py.
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import bench  # noqa: E402
import hmrm_pkg  # noqa: E402
from png_probe import card, kernel_us  # noqa: E402

K4_GOAL_US = 25.0


def hmap_script_seconds(hmap: Path, frames: int, wl: dict, hm, cm, O) -> dict:
    """Wall time of `hmap --script` for 1 and for all frames, as a Y4M video and as PNG files."""
    with tempfile.TemporaryDirectory(prefix="hmrm_yuv_", dir="/dev/shm") as td:
        td = Path(td)
        with open(td / "height.pgm", "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (hm.shape[1], hm.shape[0]))
            f.write(np.ascontiguousarray(hm[:, :, 0]).tobytes())
        O.write_tga_rgba(td / "color.tga", cm)
        cams = [bench.camera(wl, i) for i in range(frames)]
        kw = dict(width=wl["W"], height=wl["H"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                  min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT, **cams[0])
        (td / "config.txt").write_text(O.config_text(kw, td / "height.pgm", td / "color.tga"))
        (td / "frames.txt").write_text("".join("pos %r %r %r hang %r vang %r\n" % (*c["pos"], c["hang_deg"], c["vang_deg"])
                                               for c in cams))
        res = {}
        for kind, out in (("video", ["--video", str(td / "v.y4m")]), ("png", ["--out-prefix", str(td / "f_")])):
            r = {}
            for label, extra in (("one_frame_s", ["--frames", "1"]), ("all_frames_s", [])):
                t0 = time.perf_counter()
                subprocess.run([str(hmap), "config.txt", "--script", "frames.txt"] + out + extra, cwd=str(td), check=True,
                               stdout=subprocess.DEVNULL)
                r[label] = time.perf_counter() - t0
            r["s_per_frame_after_startup"] = (r["all_frames_s"] - r["one_frame_s"]) / max(1, frames - 1)
            if kind == "video":
                r["file_mb"] = (td / "v.y4m").stat().st_size / 1e6
            else:
                r["mean_file_mb"] = sum(p.stat().st_size for p in td.glob("f_*.png")) / frames / 1e6
            res[kind] = r
        res["frames"] = frames
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=240)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import oracle_lib as O
    from test_yuv420 import yuv420_model

    hmrm = hmrm_pkg.load()
    wl = bench.WORKLOADS["flythrough4k"]
    W, H, F = wl["W"], wl["H"], args.frames
    r = hmrm.Renderer(0)
    r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r.synth_maps(wl["log2n"], bench.SEED)

    def frame(n, fmt=hmrm.PIXEL_RGBA8):
        c = bench.camera(wl, n)
        return r.frame(projection=wl["projection"], screen_width=W, screen_height=H, cam_pos=c["pos"],
                       hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                       ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                       pixel_format=fmt)

    frames = [frame(n) for n in range(F)]
    frames_rgb8 = [frame(n, hmrm.PIXEL_RGB8) for n in range(F)]
    yuv_bufs = [hmrm.pinned_empty((hmrm.yuv420_bytes(W, H),)) for _ in range(4)]
    rgb8_bufs = [hmrm.pinned_empty((H, W, 3)) for _ in range(4)]
    rgba8_bufs = [hmrm.pinned_empty((H, W, 4)) for _ in range(4)]
    png_bufs = [hmrm.pinned_empty((hmrm.png_bound(W, H, 4),)) for _ in range(4)]
    png_sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]

    def stream(submit):
        for n in range(F):
            if n >= 4:
                r.wait_pending(3)
            submit(n)
        r.wait()

    runs = {
        "yuv": lambda: stream(lambda n: r.render_yuv420_async(frames[n], yuv_bufs[n % 4], hmrm.YUV_BT709)),
        "raw_rgb8": lambda: stream(lambda n: r.render_async(frames_rgb8[n], rgb8_bufs[n % 4])),
        "raw_rgba8": lambda: stream(lambda n: r.render_async(frames[n], rgba8_bufs[n % 4])),
        "png": lambda: stream(lambda n: r.render_png_async(frames[n], png_bufs[n % 4], png_sizes[n % 4])),
    }
    for run in runs.values():     # warm-up: every kernel, every scratch buffer allocated
        run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        runs["yuv"]()
        torch.cuda.synchronize()
    k4_us = kernel_us(prof, "k4_yuv420") / F
    render_us = kernel_us(prof, "k2_render") / F

    fps = {k: [] for k in runs}
    for _ in range(2):
        for k, run in runs.items():
            t0 = time.perf_counter()
            run()
            fps[k].append(F / (time.perf_counter() - t0))

    # the device's planes are the model's planes of the rendered pixels
    checked = 0
    for n in range(0, F, max(1, F // 6)):
        px = r.render(frames[n])
        got = r.render_yuv420(frames[n], matrix=hmrm.YUV_BT709)
        for g, w in zip(got, yuv420_model(px, hmrm.YUV_BT709)):
            assert np.array_equal(g, w), f"frame {n}"
        checked += 1
    r.close()

    yuv_fps, rgb8_fps = min(fps["yuv"]), max(fps["raw_rgb8"])
    out = dict(
        card=card(),
        workload=f"flythrough4k cameras, {W}x{H}, {F} frames; YUV: BT.709 from RGBA8 framebuffers",
        k4_yuv420_us_per_frame=k4_us,
        render_kernel_us_per_frame=render_us,
        k4_over_render=k4_us / render_us if render_us else None,
        fps=fps,
        yuv_frame_bytes=hmrm.yuv420_bytes(W, H),
        rgb8_frame_bytes=W * H * 3,
        frames_checked_against_model=checked,
        goals=dict(
            k4_le_25us=dict(met=k4_us <= K4_GOAL_US, value_us=k4_us, goal_us=K4_GOAL_US),
            yuv_fps_ge_raw_rgb8_fps=dict(met=yuv_fps >= rgb8_fps, yuv_fps_worst=yuv_fps, raw_rgb8_fps_best=rgb8_fps),
        ),
        timing="K4 / render kernels: torch.profiler CUDA activity (CUPTI); fps: host clock over the window, ending in "
               "hmrm_wait",
    )
    hm, cm = O.synth_maps(wl["log2n"], bench.SEED)
    out["hmap_script"] = hmap_script_seconds(ROOT / "heightmap-ray-marcher_b200" / "hmap", F, wl, hm, cm, O)
    line = json.dumps(out)
    print(line)
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
