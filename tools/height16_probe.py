"""16-bit height maps (hmrm_synth_maps16, kernel k1_build16) against the 8-bit path, one GPU; prints one
JSON line (and writes it, after a header naming the card, to --out).

    python tools/height16_probe.py [--reps 24] [--frames 120] [--out FILE]

- K1 at 16384^2: hmrm_update_heightmap on synth_maps(14) and synth_maps16(14), held by two contexts and called
  alternately, --reps times each; host clock around the call, which ends in a device synchronise.  Median and spread
  (min, max).  Goal: the 16-bit total <= the 8-bit total of the same session.
- Per-kernel breakdown of K1 from torch.profiler (CUPTI device timestamps), in a separate run of 5 calls per context.
- Render: the flythrough4k cameras over both maps, 3840x2160, device-resident (hmrm_render_device), CUDA events
  around --frames frames after a warm-up: Grays/s; then the same frames with HMRM_FLAG_STATS for the reference steps,
  fetches and the debug counter of samples the exact FP64 expressions decided.  No goal: the terrain differs.
"""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402
import hmrm_pkg  # noqa: E402
from png_probe import card  # noqa: E402

LOG2N = 14


def k1_times(r8, r16, reps):
    t = {8: [], 16: []}
    for _ in range(reps):
        for bits, r in ((8, r8), (16, r16)):
            t0 = time.perf_counter()
            r.update_heightmap()
            t[bits].append((time.perf_counter() - t0) * 1e3)
    return {str(b): dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v), n=len(v)) for b, v in t.items()}


def k1_kernels(r8, r16):
    from torch.profiler import ProfilerActivity, profile

    out = {}
    for bits, r in ((8, r8), (16, r16)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                r.update_heightmap()
        ks = {}
        for e in prof.key_averages():
            us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            if us > 0:
                ks[e.key[:60]] = us / 5.0
        out[str(bits)] = dict(per_call_us=ks, total_us=sum(ks.values()))
    return out


def render(hmrm, r, frames):
    import torch

    wl = bench.WORKLOADS["flythrough4k"]
    W, H = wl["W"], wl["H"]
    d_out = torch.empty(W * H * 4, dtype=torch.uint8, device="cuda")

    def frame(n, flags=0):
        c = bench.camera(wl, n % wl["frames"])
        return r.frame(projection=wl["projection"], screen_width=W, screen_height=H, cam_pos=c["pos"],
                       hang=hmrm.deg2rad(c["hang_deg"]), vang=hmrm.deg2rad(c["vang_deg"]),
                       hfov=hmrm.deg2rad(c["hfov_deg"]), ortho_width=c["ortho_width"], grid_width=bench.GRID_WIDTH,
                       step_dist=wl["step_dist"], flags=flags)

    fs = [frame(n) for n in range(frames)]
    for f in fs[:10]:
        r.render_device(f, d_out)
    r.wait()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for f in fs:
        r.render_device(f, d_out, torch.cuda.current_stream().cuda_stream)
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b)
    steps = fetches = fp64 = 0
    for n in range(frames):
        f = frame(n, hmrm.FLAG_STATS)
        r.render_device(f, d_out, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        st = r.stats()
        steps += st.steps
        fetches += st.fetches
        fp64 += r.debug_counters()[7]
    return dict(ms_per_frame=ms / frames, grays_per_s=W * H * frames / (ms * 1e-3) / 1e9,
                ref_steps_per_frame=steps / frames, fetches_per_frame=fetches / frames,
                fp64_decided_samples_per_frame=fp64 / frames, fp64_decided_per_ref_step=fp64 / max(steps, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=24)
    ap.add_argument("--frames", type=int, default=120)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    hmrm = hmrm_pkg.load()
    r8, r16 = hmrm.Renderer(0), hmrm.Renderer(0)
    for r in (r8, r16):
        r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r8.synth_maps(LOG2N, bench.SEED)
    r16.synth_maps16(LOG2N, bench.SEED)
    res = dict(card=card(), map=f"{1 << LOG2N}^2 synthetic fBm, seed {bench.SEED}")
    k1_times(r8, r16, 3)                       # warm-up (lazy allocations, first-launch costs)
    res["k1_host_clock"] = k1_times(r8, r16, args.reps)
    res["k1_kernels"] = k1_kernels(r8, r16)
    m8, m16 = res["k1_host_clock"]["8"]["median_ms"], res["k1_host_clock"]["16"]["median_ms"]
    res["k1_goal_16_le_8"] = dict(met=m16 <= m8, ratio_16_over_8=m16 / m8)
    res["render_flythrough4k"] = {"8": render(hmrm, r8, args.frames), "16": render(hmrm, r16, args.frames)}
    res["timing"] = ("K1: host clock around hmrm_update_heightmap (ends in a device synchronise), calls alternating "
                     "between the two contexts; kernels: torch.profiler CUDA activity; render: CUDA events around "
                     "hmrm_render_device frames on one stream")
    r8.close()
    r16.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        c = res["card"]
        head = (f"# on one {c.get('name')} ({c.get('power_limit')} power limit, max SM clock {c.get('max_sm_clock')}), "
                f"one session: python tools/height16_probe.py\n"
                f"# K1 goal (16-bit total <= 8-bit total): {'MET' if res['k1_goal_16_le_8']['met'] else 'MISSED'} "
                f"({m16:.3f} vs {m8:.3f} ms median, host clock)\n")
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(head + line + "\n")


if __name__ == "__main__":
    main()
