"""PNG output of the bench's flythrough4k cameras on one GPU; prints one JSON line.

    python tools/png_probe.py [--frames 240] [--hmap-before DIR/hmap] [--out FILE]

- encode kernels (k3_png_*) per 4K frame: kernel durations from torch.profiler (CUPTI device timestamps) over --frames
  render + PNG frames, after a warm-up; the render kernel's time in the same window for comparison;
- frames per second of render + PNG into pinned host memory (hmrm_render_png_async, 4 in flight) and of render + raw
  RGBA8 D2H (hmrm_render_async, 4 in flight), host clock around the whole window, which ends in a synchronise;
- mean PNG size against the raw frame and against zlib level 1 on the same pixels (Python zlib on this host, filter
  None on every row: what `hmap` wrote before frames were encoded on the device), and zlib's time per frame;
- `hmap --script` wall time for --frames 4K frames written to /dev/shm, for this tree's hmap and, with --hmap-before,
  for another build (e.g. the parent commit's), run in the same session.
"""
import argparse
import io
import json
import subprocess
import sys
import tempfile
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import bench  # noqa: E402
import hmrm_pkg  # noqa: E402


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the probe still measures; the card is then unknown
        return dict(name="unknown", error=str(e))


def kernel_us(prof, pattern: str) -> float:
    tot = 0.0
    for e in prof.key_averages():
        if pattern in e.key:
            tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return tot


def hmap_script_seconds(hmap: Path, frames: int, wl: dict, hm, cm, O) -> dict:
    with tempfile.TemporaryDirectory(prefix="hmrm_png_", dir="/dev/shm") as td:
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
        for label, extra in (("one_frame_s", ["--frames", "1"]), ("all_frames_s", [])):
            t0 = time.perf_counter()
            subprocess.run([str(hmap), "config.txt", "--script", "frames.txt", "--out-prefix", str(td / "f_")] + extra,
                           cwd=str(td), check=True, stdout=subprocess.DEVNULL)
            res[label] = time.perf_counter() - t0
        res["frames"] = frames
        res["mean_file_mb"] = sum(p.stat().st_size for p in td.glob("f_*.png")) / frames / 1e6
        res["s_per_frame_after_startup"] = (res["all_frames_s"] - res["one_frame_s"]) / max(1, frames - 1)
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=240)
    ap.add_argument("--hmap-before", type=Path, default=None)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    from PIL import Image

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
    bound = hmrm.png_bound(W, H, 4)
    png_bufs = [hmrm.pinned_empty((bound,)) for _ in range(4)]
    png_sizes = [hmrm.pinned_empty((1,), dtype=np.uint64) for _ in range(4)]
    raw_bufs = [hmrm.pinned_empty((H, W, 4)) for _ in range(4)]

    def run_png(collect=None):
        for n, f in enumerate(frames):
            if n >= 4:
                r.wait_pending(3)
                if collect is not None:
                    collect.append(int(png_sizes[(n - 4) % 4][0]))
            r.render_png_async(f, png_bufs[n % 4], png_sizes[n % 4])
        r.wait()
        if collect is not None:
            collect.extend(int(png_sizes[n % 4][0]) for n in range(max(0, F - 4), F))

    def run_raw():
        for n, f in enumerate(frames):
            if n >= 4:
                r.wait_pending(3)
            r.render_async(f, raw_bufs[n % 4])
        r.wait()

    run_png()        # warm-up: every kernel, scratch allocated
    run_raw()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_png()
        torch.cuda.synchronize()
    enc_us = {k: kernel_us(prof, k) / F for k in ("k3_png_filter", "k3_png_deflate", "k3_png_finish", "k3_png_gather")}
    render_us = kernel_us(prof, "k2_render") / F

    sizes = []
    t0 = time.perf_counter()
    run_png(sizes)
    png_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    run_raw()
    raw_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    run_png()
    png_s2 = time.perf_counter() - t0

    # zlib level 1 on a sample of the same frames (filter None on every row)
    zs, zt = [], []
    for n in range(0, F, max(1, F // 8)):
        px = r.render(frames[n])
        stream = np.concatenate([np.zeros((H, 1), np.uint8), px.reshape(H, W * 4)], axis=1).tobytes()
        t = time.perf_counter()
        zs.append(len(zlib.compress(stream, 1)))
        zt.append(time.perf_counter() - t)
        data = r.render_png(frames[n])
        # the device's file decodes to the same pixels (PIL here; tests/test_gpu_png.py checks every byte path)
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(data))), px)
    r.close()

    out = dict(
        card=card(),
        workload=f"flythrough4k cameras, {W}x{H} RGBA8, {F} frames",
        encode_kernels_us_per_frame=dict(enc_us, total=sum(enc_us.values())),
        render_kernel_us_per_frame=render_us,
        render_png_fps=[F / png_s, F / png_s2],
        render_raw_fps=F / raw_s,
        png_mean_bytes=float(np.mean(sizes)),
        raw_frame_bytes=W * H * 4,
        png_over_raw=float(np.mean(sizes)) / (W * H * 4),
        zlib1_mean_bytes=float(np.mean(zs)),
        png_over_zlib1=float(np.mean(sizes)) / float(np.mean(zs)),
        zlib1_host_s_per_frame=float(np.mean(zt)),
        timing="encode / render kernels: torch.profiler CUDA activity (CUPTI); fps: host clock over the window, ending "
               "in hmrm_wait",
    )
    hm, cm = O.synth_maps(wl["log2n"], bench.SEED)
    out["hmap_script"] = hmap_script_seconds(ROOT / "heightmap-ray-marcher_b200" / "hmap", F, wl, hm, cm, O)
    if args.hmap_before is not None:
        out["hmap_script_before"] = hmap_script_seconds(args.hmap_before.resolve(), F, wl, hm, cm, O)
        out["hmap_script_speedup"] = (out["hmap_script_before"]["all_frames_s"] / out["hmap_script"]["all_frames_s"])
    line = json.dumps(out)
    print(line)
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
