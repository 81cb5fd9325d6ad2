"""Motion-blurred frames (hmrm_set_motion_blur, kernel K5) on the bench's flythrough4k cameras, one GPU; prints one JSON
line.

    python tools/blur_probe.py [--frames 48] [--hmap-frames 240] [--out FILE]   (writes profiles/r11_blur_probe.txt)
    python tools/blur_probe.py --k5-only          (K5 without blur, s = 2, 3, 4: runs against older builds too)

Frame i blurs from bench camera i (c_n) towards camera i + 1 (c_{n+1}) with hmap's formula at shutter 0.5.
- K5 per output frame at (n, s) = (4, 1), (8, 1), (4, 2), RGB8 output, against the n sub-frame renders of the same
  frame: kernel durations from torch.profiler (CUPTI device timestamps) over --frames hmrm_render_device frames after a
  warm-up.  Goal: K5 <= 3 % of the sub-frame render time.
- frames per second, four in flight into pinned host memory, of blurred render + YUV (hmrm_render_yuv420_async) at n = 8
  against plain render + YUV, in the same session, each measured twice, alternating.  Goal: >= 0.95 x plain / 8.
- `hmap --script --video /dev/null --motion-blur 8`: milliseconds per frame after start-up (the best of two runs of 1
  frame and of all frames), beside the same runs without the option.
- K5 without blur, s = 2, 3, 4 (what tools/ssaa_probe.py measures), for an A/B against an older build through
  HMRM_LIBRARY.
A sample of the blurred frames is checked against the rounded average of the same device's plain sub-frames (a
consistency check; the oracle comparisons are in tests/test_gpu_motion_blur.py).
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

SHUTTER = 0.5
K5_GOAL_SHARE = 0.03
YUV_GOAL = 0.95


def hmap_video_seconds(hmap: Path, frames: int, wl: dict, hm, cm, O) -> dict:
    with tempfile.TemporaryDirectory(prefix="hmrm_blur_", dir="/dev/shm") as td:
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
        for label, extra in (("motion_blur_8", ["--motion-blur", "8"]), ("plain", [])):
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
    ap.add_argument("--frames", type=int, default=48)
    ap.add_argument("--hmap-frames", type=int, default=240)
    ap.add_argument("--k5-only", action="store_true")
    ap.add_argument("--out", type=Path, default=None, help="default: profiles/r11_blur_probe.txt (none with --k5-only)")
    args = ap.parse_args()
    if args.out is None and not args.k5_only:
        args.out = ROOT / "profiles" / "r11_blur_probe.txt"
    import torch
    from torch.profiler import ProfilerActivity, profile

    hmrm = hmrm_pkg.load()
    wl = bench.WORKLOADS["flythrough4k"]
    W, H, F = wl["W"], wl["H"], args.frames
    r = hmrm.Renderer(0)
    r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r.synth_maps(wl["log2n"], bench.SEED)

    def frame(i, s=1, fmt=hmrm.PIXEL_RGBA8):
        c = bench.camera(wl, i)
        return r.frame(projection=wl["projection"], screen_width=W, screen_height=H, cam_pos=c["pos"],
                       hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                       ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"],
                       pixel_format=fmt, supersample=s)

    def cams(i, k):
        a, b = bench.camera(wl, i), bench.camera(wl, i + 1)
        ca = (*a["pos"], hmrm.deg2rad(a["hang_deg"]), hmrm.deg2rad(a["vang_deg"]))
        cb = (*b["pos"], hmrm.deg2rad(b["hang_deg"]), hmrm.deg2rad(b["vang_deg"]))
        return np.array([[x + ((SHUTTER * j) / k) * (y - x) for x, y in zip(ca, cb)] for j in range(k)])

    d_out = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda:0")

    def profiled(submit):
        for i in range(min(8, F)):                   # warm-up: tables, scratches, modules
            submit(i)
        r.wait()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(F):
                submit(i)
            r.wait()
            torch.cuda.synchronize()
        return kernel_us(prof, "k5_downsample") / F, kernel_us(prof, "k2_render") / F

    out = dict(card=card(), workload=f"flythrough4k cameras, {W}x{H} output, {F} frames per window")
    k5_plain = {}
    for s in (2, 3, 4):
        k5_us, render_us = profiled(lambda i: r.render_device(frame(i, s, hmrm.PIXEL_RGB8), d_out))
        k5_plain[str(s)] = dict(k5_us_per_frame=k5_us, sub_frame_render_us_per_frame=render_us)
    out["k5_without_blur"] = k5_plain
    if not args.k5_only:
        k5 = {}
        for n, s in ((4, 1), (8, 1), (4, 2)):
            def submit(i):
                r.set_motion_blur(cams(i, n))
                r.render_device(frame(i, s, hmrm.PIXEL_RGB8), d_out)
            k5_us, render_us = profiled(submit)
            k5[f"n{n}_s{s}"] = dict(k5_us_per_frame=k5_us, sub_frame_renders_us_per_frame=render_us,
                                    k5_share_of_render=k5_us / render_us if render_us else None)
        r.set_motion_blur([])
        out["k5_blur"] = k5

        yuv_bufs = [hmrm.pinned_empty((hmrm.yuv420_bytes(W, H),)) for _ in range(4)]
        frames = [frame(i) for i in range(F)]
        sets = [cams(i, 8) for i in range(F)]

        def stream(blur):
            for i in range(F):
                if i >= 4:
                    r.wait_pending(3)
                r.set_motion_blur(sets[i] if blur else [])
                r.render_yuv420_async(frames[i], yuv_bufs[i % 4], hmrm.YUV_BT709)
            r.wait()

        runs = {"plain_yuv": lambda: stream(False), "blur8_yuv": lambda: stream(True)}
        for run in runs.values():
            run()
        fps = {k: [] for k in runs}
        for _ in range(2):
            for k, run in runs.items():
                t0 = time.perf_counter()
                run()
                fps[k].append(F / (time.perf_counter() - t0))
        r.set_motion_blur([])
        share = min(fps["blur8_yuv"]) / (max(fps["plain_yuv"]) / 8)
        out["fps"] = fps
        out["blur8_yuv_over_plain_div_8"] = share

        # consistency: a blurred frame is the rounded average of the same device's plain sub-frames
        checked = 0
        for i in range(0, F, max(1, F // 3)):
            subs = []
            for c in sets[i]:
                f = frame(i)
                f.cam_pos[:] = list(c[:3])
                f.hang, f.vang = float(c[3]), float(c[4])
                subs.append(r.render(f)[:, :, :3].astype(np.int64))
            r.set_motion_blur(sets[i])
            got = r.render(frame(i)).copy()
            r.set_motion_blur([])
            assert np.array_equal(got[:, :, :3], (sum(subs) + 4) // 8), f"frame {i}"
            checked += 1
        out["frames_checked"] = checked
        worst = max(v["k5_share_of_render"] for v in k5.values())
        out["goals"] = dict(k5_le_3pct_of_render=dict(met=worst <= K5_GOAL_SHARE, worst=worst),
                            blur8_yuv_ge_95pct_of_plain_div_8=dict(met=share >= YUV_GOAL, share=share))
        import oracle_lib as O

        hm, cm = O.synth_maps(wl["log2n"], bench.SEED)
        out["hmap_script_video"] = hmap_video_seconds(ROOT / "heightmap-ray-marcher_b200" / "hmap", args.hmap_frames,
                                                      wl, hm, cm, O)
    r.close()
    out["timing"] = ("K5 / render kernels: torch.profiler CUDA activity (CUPTI); fps: host clock over the window, ending "
                     "in hmrm_wait")
    line = json.dumps(out)
    print(line)
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
