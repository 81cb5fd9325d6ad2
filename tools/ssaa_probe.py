"""Supersampled frames (HMRM_FLAG_SUPERSAMPLE, kernel K5) on the bench's flythrough4k cameras, one GPU; prints one JSON
line.

    python tools/ssaa_probe.py [--frames 120] [--hmap-frames 720] [--out FILE]

- k5_downsample per 4K frame for s = 2, 3, 4 (RGB8 output): kernel durations from torch.profiler (CUPTI device
  timestamps) over --frames hmrm_render_device frames after a warm-up, against the byte floor (s*s*W*H*4 bytes read +
  W*H*3 written, over 6546 GB/s, the measured HBM peak the bench reports, profiles/r01_bench_line_*.json); the
  sub-frame render kernel's time in the same window;
- frames per second at s = 2, 4 in flight into pinned host memory, of render + filter + YUV (hmrm_render_yuv420_async)
  and render + filter + PNG (hmrm_render_png_async), against hmrm_render_device of the 7680x4320 sub-frame alone: host
  clock around the whole window, which ends in a synchronise; each measured twice, alternating;
- `hmap --script --video --supersample 2` writing to /dev/null: milliseconds per frame after start-up (the best of two
  runs of 1 frame and of all frames; the 5-6 s start-up varies by more than a short run takes), beside the same runs
  without --supersample;
- the goals: K5 within 1.5x of the byte floor, and the s = 2 YUV path at >= 95 % of the bare sub-frame render rate.
A sample of the frames is checked against the box filter of the same device's sub-frame (a consistency check; the
oracle comparisons are in tests/test_gpu_supersample.py).
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
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402
import hmrm_pkg  # noqa: E402
from png_probe import card, kernel_us  # noqa: E402

COPY_PEAK_GBS = 6546.0
K5_GOAL_OVER_FLOOR = 1.5
YUV_GOAL_SHARE = 0.95


def hmap_video_seconds(hmap: Path, frames: int, wl: dict, hm, cm, O) -> dict:
    """Wall time of `hmap --script --video /dev/null` for 1 and for all frames (best of two each), with and without
    --supersample 2."""
    with tempfile.TemporaryDirectory(prefix="hmrm_ssaa_", dir="/dev/shm") as td:
        td = Path(td)
        with open(td / "height.pgm", "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (hm.shape[1], hm.shape[0]))
            f.write(np.ascontiguousarray(hm[:, :, 0]).tobytes())
        O.write_tga_rgba(td / "color.tga", cm)
        cams = [bench.camera(wl, i % wl["frames"]) for i in range(frames)]
        kw = dict(width=wl["W"], height=wl["H"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                  min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT, **cams[0])
        (td / "config.txt").write_text(O.config_text(kw, td / "height.pgm", td / "color.tga"))
        (td / "frames.txt").write_text("".join("pos %r %r %r hang %r vang %r\n" % (*c["pos"], c["hang_deg"], c["vang_deg"])
                                               for c in cams))
        res = {}
        for label, extra in (("supersample_2", ["--supersample", "2"]), ("supersample_1", [])):
            r = {}
            for run, more in (("one_frame_s", ["--frames", "1"]), ("all_frames_s", [])):
                best = None
                for _ in range(2):
                    t0 = time.perf_counter()
                    subprocess.run([str(hmap), "config.txt", "--script", "frames.txt", "--video", "/dev/null"] + extra
                                   + more, cwd=str(td), check=True, stdout=subprocess.DEVNULL)
                    t = time.perf_counter() - t0
                    best = t if best is None else min(best, t)
                r[run] = best
            r["ms_per_frame_after_startup"] = 1e3 * (r["all_frames_s"] - r["one_frame_s"]) / max(1, frames - 1)
            res[label] = r
        res["frames"] = frames
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=120)
    ap.add_argument("--hmap-frames", type=int, default=720)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import oracle_lib as O
    from test_supersample import box_reduce
    from test_yuv420 import yuv420_model

    hmrm = hmrm_pkg.load()
    wl = bench.WORKLOADS["flythrough4k"]
    W, H, F = wl["W"], wl["H"], args.frames
    r = hmrm.Renderer(0)
    r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r.synth_maps(wl["log2n"], bench.SEED)

    def frame(n, s=1, fmt=hmrm.PIXEL_RGBA8, w=W, h=H):
        c = bench.camera(wl, n)
        return r.frame(projection=wl["projection"], screen_width=w, screen_height=h, cam_pos=c["pos"],
                       hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                       ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                       pixel_format=fmt, supersample=s)

    # ---- K5 and the sub-frame render per s, RGB8 output into a device tensor ----
    d_out = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda:0")
    k5 = {}
    for s in (2, 3, 4):
        frames = [frame(n, s, hmrm.PIXEL_RGB8) for n in range(F)]
        for f in frames[:8]:                         # warm-up: tables, scratches, modules
            r.render_device(f, d_out)
        r.wait()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for f in frames:
                r.render_device(f, d_out)
            r.wait()
            torch.cuda.synchronize()
        k5_us = kernel_us(prof, "k5_downsample") / F
        render_us = kernel_us(prof, "k2_render") / F
        floor_bytes = s * s * W * H * 4 + W * H * 3
        floor_us = floor_bytes / (COPY_PEAK_GBS * 1e3)
        k5[str(s)] = dict(k5_us_per_frame=k5_us, floor_bytes=floor_bytes, floor_us=floor_us,
                          k5_over_floor=k5_us / floor_us if floor_us else None,
                          achieved_gbs=floor_bytes / (k5_us * 1e3) if k5_us else None,
                          sub_frame_render_us_per_frame=render_us, k5_over_render=k5_us / render_us if render_us else None)

    # ---- s = 2 streams against the bare 7680x4320 render ----
    frames_s2 = [frame(n, 2) for n in range(F)]
    frames_8k = [frame(n, 1, w=2 * W, h=2 * H) for n in range(F)]
    d_8k = torch.empty((2 * H, 2 * W, 4), dtype=torch.uint8, device="cuda:0")
    yuv_bufs = [hmrm.pinned_empty((hmrm.yuv420_bytes(W, H),)) for _ in range(4)]
    png_bufs = [hmrm.pinned_empty((hmrm.png_bound(W, H, 4),)) for _ in range(4)]
    png_sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]

    def stream(submit):
        for n in range(F):
            if n >= 4:
                r.wait_pending(3)
            submit(n)
        r.wait()

    def bare():
        for n in range(F):
            r.render_device(frames_8k[n], d_8k)
        r.wait()

    runs = {
        "sub_frame_render_7680x4320": bare,
        "yuv_s2": lambda: stream(lambda n: r.render_yuv420_async(frames_s2[n], yuv_bufs[n % 4], hmrm.YUV_BT709)),
        "png_s2": lambda: stream(lambda n: r.render_png_async(frames_s2[n], png_bufs[n % 4], png_sizes[n % 4])),
    }
    for run in runs.values():
        run()
    fps = {k: [] for k in runs}
    for _ in range(2):
        for k, run in runs.items():
            t0 = time.perf_counter()
            run()
            fps[k].append(F / (time.perf_counter() - t0))

    # consistency: the filtered frame is the box filter of the same device's sub-frame, and the YUV planes its model
    checked = 0
    for n in range(0, F, max(1, F // 4)):
        sub = r.render(frame(n, 1, w=2 * W, h=2 * H)).copy()
        got = r.render(frames_s2[n]).copy()
        assert np.array_equal(got, box_reduce(sub, 2)), f"frame {n}"
        planes = r.render_yuv420(frames_s2[n], matrix=hmrm.YUV_BT709)
        for g, w in zip(planes, yuv420_model(got, hmrm.YUV_BT709)):
            assert np.array_equal(g, w), f"frame {n} planes"
        checked += 1
    r.close()

    yuv_share = min(fps["yuv_s2"]) / max(fps["sub_frame_render_7680x4320"])
    worst = max(v["k5_over_floor"] for v in k5.values())
    out = dict(
        card=card(),
        workload=f"flythrough4k cameras, {W}x{H} output, {F} frames per window",
        k5=k5,
        fps=fps,
        yuv_s2_share_of_bare_render=yuv_share,
        png_s2_share_of_bare_render=min(fps["png_s2"]) / max(fps["sub_frame_render_7680x4320"]),
        frames_checked=checked,
        goals=dict(
            k5_within_1_5x_floor=dict(met=worst <= K5_GOAL_OVER_FLOOR, worst_over_floor=worst),
            yuv_s2_ge_95pct_of_bare_render=dict(met=yuv_share >= YUV_GOAL_SHARE, share=yuv_share),
        ),
        timing="K5 / render kernels: torch.profiler CUDA activity (CUPTI); fps: host clock over the window, ending in "
               "hmrm_wait; floor at %.0f GB/s" % COPY_PEAK_GBS,
    )
    hm, cm = O.synth_maps(wl["log2n"], bench.SEED)
    out["hmap_script_video"] = hmap_video_seconds(ROOT / "heightmap-ray-marcher_b200" / "hmap", args.hmap_frames, wl, hm,
                                                  cm, O)
    line = json.dumps(out)
    print(line)
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
