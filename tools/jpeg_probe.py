"""JPEG output of the bench's flythrough4k cameras on one GPU; prints one JSON line.

    python tools/jpeg_probe.py [--frames 240] [--out FILE]

- encode kernels (k6_jpeg_*, and k3_png_gather, which writes the file) per 4K frame, for q = 75 and 90 in 4:2:0 and
  4:4:4: kernel durations from torch.profiler (CUPTI device timestamps) over --frames render + JPEG frames, after a
  warm-up; the render kernel's time in the same window;
- frames per second of render + JPEG (q 90, 4:2:0) into pinned host memory against render + YUV (hmrm_render_yuv420_async)
  in the same session, alternated, 4 frames in flight each; host clock around each window, which ends in a synchronise;
- mean JPEG size per frame, against the mean PNG size of the same frames (hmrm_render_png_async);
- the bytes-over-HBM floor of the encode: the RGBA8 frame read plus the file written, at 7.7 TB/s;
- `hmap --script --jpeg 90` and `hmap --script` (PNG) wall time per frame after start-up, files in /dev/shm.
The card's name, power limit and clocks are read in the same run.
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

HBM_BYTES_PER_S = 7.7e12


def hmap_script_s_per_frame(frames: int, wl: dict, hm, cm, O, extra: list) -> dict:
    hmap = ROOT / "heightmap-ray-marcher_b200" / "hmap"
    with tempfile.TemporaryDirectory(prefix="hmrm_jpeg_", dir="/dev/shm") as td:
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
        for label, more in (("one_frame_s", ["--frames", "1"]), ("all_frames_s", [])):
            t0 = time.perf_counter()
            subprocess.run([str(hmap), "config.txt", "--script", "frames.txt", "--out-prefix", str(td / "f_")] + extra +
                           more, cwd=str(td), check=True, stdout=subprocess.DEVNULL)
            res[label] = time.perf_counter() - t0
        files = list(td.glob("f_*"))
        res["mean_file_mb"] = sum(p.stat().st_size for p in files) / max(1, len(files)) / 1e6
        res["ms_per_frame_after_startup"] = 1e3 * (res["all_frames_s"] - res["one_frame_s"]) / max(1, frames - 1)
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=240)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import oracle_lib as O

    hmrm = hmrm_pkg.load()
    wl = bench.WORKLOADS["flythrough4k"]
    W, H, F = wl["W"], wl["H"], args.frames
    r = hmrm.Renderer(0)
    r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r.synth_maps(wl["log2n"], bench.SEED)

    def frame(n):
        c = bench.camera(wl, n)
        return r.frame(projection=wl["projection"], screen_width=W, screen_height=H, cam_pos=c["pos"],
                       hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]), hfov=hmrm.deg2rad(c["hfov_deg"]),
                       ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"])

    frames = [frame(n) for n in range(F)]
    bound = hmrm.jpeg_bound(W, H, hmrm.JPEG_444)
    bufs = [hmrm.pinned_empty((bound,)) for _ in range(4)]
    sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]
    yuv_bufs = [hmrm.pinned_empty((hmrm.yuv420_bytes(W, H),)) for _ in range(4)]
    png_bound = hmrm.png_bound(W, H, 4)
    png_bufs = [hmrm.pinned_empty((png_bound,)) for _ in range(4)]

    def run(kind, q=90, chroma=hmrm.JPEG_420, collect=None):
        for n, f in enumerate(frames):
            if n >= 4:
                r.wait_pending(3)
                if collect is not None:
                    collect.append(int(sizes[(n - 4) % 4][0]))
            if kind == "jpeg":
                r.render_jpeg_async(f, bufs[n % 4], sizes[n % 4], q, chroma)
            elif kind == "png":
                r.render_png_async(f, png_bufs[n % 4], sizes[n % 4])
            else:
                r.render_yuv420_async(f, yuv_bufs[n % 4])
        r.wait()
        if collect is not None:
            collect.extend(int(sizes[n % 4][0]) for n in range(max(0, F - 4), F))

    modes = [(75, hmrm.JPEG_420, "q75_420"), (90, hmrm.JPEG_420, "q90_420"), (75, hmrm.JPEG_444, "q75_444"),
             (90, hmrm.JPEG_444, "q90_444")]
    for q, chroma, _ in modes:          # warm-up: every kernel, scratch allocated
        run("jpeg", q, chroma)
    run("yuv")
    run("png")
    torch.cuda.synchronize()
    kernels = {}
    sizes_by_mode = {}
    for q, chroma, name in modes:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run("jpeg", q, chroma)
            torch.cuda.synchronize()
        enc = {k: kernel_us(prof, k) / F for k in ("k6_jpeg_blocks", "k6_jpeg_rows", "k6_jpeg_finish", "k3_png_gather")}
        kernels[name] = dict(enc, total=sum(enc.values()), render=kernel_us(prof, "k2_render") / F)
        got = []
        run("jpeg", q, chroma, got)
        sizes_by_mode[name] = float(np.mean(got))
        floor_us = (W * H * 4 + sizes_by_mode[name]) / HBM_BYTES_PER_S * 1e6
        kernels[name]["hbm_floor_us"] = floor_us

    fps = {"jpeg_q90_420": [], "yuv": []}
    for _ in range(3):              # alternated windows
        for kind in ("jpeg", "yuv"):
            t0 = time.perf_counter()
            run(kind)
            fps["jpeg_q90_420" if kind == "jpeg" else "yuv"].append(F / (time.perf_counter() - t0))
    png_sizes = []
    run("png", collect=png_sizes)
    r.close()

    out = dict(
        card=card(),
        workload=f"flythrough4k cameras, {W}x{H} RGBA8, {F} frames",
        encode_kernels_us_per_frame=kernels,
        render_jpeg_fps=fps["jpeg_q90_420"],
        render_yuv_fps=fps["yuv"],
        jpeg_over_yuv_fps=float(np.mean(fps["jpeg_q90_420"]) / np.mean(fps["yuv"])),
        jpeg_mean_bytes=sizes_by_mode,
        png_mean_bytes=float(np.mean(png_sizes)),
        timing="encode / render kernels: torch.profiler CUDA activity (CUPTI); fps: host clock over the window, ending "
               "in hmrm_wait; hbm_floor_us: (RGBA8 frame + mean file) / 7.7 TB/s",
    )
    hm, cm = O.synth_maps(wl["log2n"], bench.SEED)
    out["hmap_script_jpeg90"] = hmap_script_s_per_frame(F, wl, hm, cm, O, ["--jpeg", "90"])
    out["hmap_script_png"] = hmap_script_s_per_frame(F, wl, hm, cm, O, [])
    line = json.dumps(out)
    print(line)
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
