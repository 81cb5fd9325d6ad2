#!/usr/bin/env python
"""bench.py — Mrays/s (and march-steps/s) of the heightmap ray-march hot path at 4K on N B200s.

Workload (BASELINE.json configs[3], SURVEY.md §8d-4): perspective 3840x2160 flythrough over a 16384^2
synthetic fBm heightmap + colormap (csrc/synth_fbm.h, seed 1234), min_height 0, max_height 10, grid_width 0.01,
step_dist 0.05, orbit camera frame n of 240: pos = (81.92 + 140 cos 2πt, -81.92 + 140 sin 2πt, 40), hang toward the
map centre, vang 110°, hfov 90°.  One step = one full 4K frame per GPU; frames are sharded round-robin
(frame = step*N + rank), maps replicated per GPU, no data-path collective (weak scaling).  At N > 1 the line also
carries a `bands8k` sub-record: BASELINE configs[4], one 7680x4320 frame over a 32768^2 map split into interleaved
4-row tile bands over the N GPUs, every rank's kernel storing its RGB8 bands straight into rank 0's frame over NVLink
peer memory with a device-side completion (strong scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload flythrough4k|...]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` is timed with CUDA events around K frames rendered into device memory
(inputs resident in HBM); `e2e` times the same frames through the C-ABI call with a host output buffer (the D2H
of every frame inside the timed region).  `--impl reference` times the UNMODIFIED reference
(oracle/_ref/hmap_ref*, built from /root/reference by oracle/Makefile) on the host cores, on a bounded sample.

`--dump-outputs DIR` writes rank 0's frame of the last timed step, as the caller of the timed path receives it, to
DIR/frame.npy (float32 [n, channels]: the pixels at DIR/pixel_index.npy, float64 [n] row-major indices y*W + x, a fixed
seeded sample of at most 2^21 pixels, every pixel of a smaller frame).  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOADS = {
    # name: (log2n, W, H, projection, step_dist, frames)
    "flythrough4k": dict(log2n=14, W=3840, H=2160, projection=1, step_dist=0.05, frames=240,
                         desc="perspective 3840x2160, 240-frame orbit over a 16384^2 fBm heightmap (BASELINE configs[3])"),
    "sample720": dict(log2n=10, W=1280, H=720, projection=1, step_dist=0.05, frames=240, camera="sample",
                      desc="sample_config.txt camera (pos -5 5 0, hang -45, vang 90, hfov 90), perspective 1280x720 over a "
                           "1024^2 fBm heightmap (BASELINE configs[0]); the camera does not move"),
    "spherical1080": dict(log2n=12, W=1920, H=1080, projection=2, step_dist=0.05, frames=240,
                          desc="spherical 1920x1080 over a 4096^2 fBm heightmap (BASELINE configs[1])"),
    "ortho4k": dict(log2n=13, W=3840, H=2160, projection=3, step_dist=0.00625, frames=240,
                    desc="orthographic 3840x2160 over an 8192^2 fBm heightmap, step_dist/8 (BASELINE configs[2])"),
    "bands8k": dict(log2n=15, W=7680, H=4320, projection=1, step_dist=0.05, frames=240, mode="bands",
                    desc="perspective 7680x4320 single frames over a 32768^2 fBm heightmap, interleaved 4-row tile bands "
                         "over the GPUs, stored into rank 0's frame over NVLink (BASELINE configs[4])"),
    "smoke": dict(log2n=10, W=640, H=360, projection=1, step_dist=0.05, frames=240,
                  desc="small debugging workload"),
    "smokebands": dict(log2n=10, W=640, H=360, projection=1, step_dist=0.05, frames=240, mode="bands",
                       desc="small debugging workload, bands mode"),
}
GRID_WIDTH = 0.01
MIN_HEIGHT, MAX_HEIGHT = 0.0, 10.0
SEED = 1234
REF_SAMPLE_DIV = 4          # the CPU arms render every frame at W/4 x H/4 (1/16 as many rays, same cameras)
SM_COUNT_FALLBACK = 148
DUMP_MAX_PIXELS = 1 << 21   # --dump-outputs: 2^21 pixels x 4 channels in float32 + their float64 indices = 48 MiB
DUMP_SEED = 20240601


def dump_frame(dump_dir: str, frame) -> None:
    """frame: uint8 [H, W, C] -> DIR/frame.npy (float32 [n, C]) and DIR/pixel_index.npy (float64 [n]), a fixed seeded
    sample of the pixels in row-major order."""
    import numpy as np

    h, w, c = frame.shape
    if h * w <= DUMP_MAX_PIXELS:
        idx = np.arange(h * w)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, size=DUMP_MAX_PIXELS, replace=False))
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, "frame.npy"), frame.reshape(h * w, c)[idx].astype(np.float32))
    np.save(os.path.join(dump_dir, "pixel_index.npy"), idx.astype(np.float64))


def camera(wl: dict, n: int) -> dict:
    """Camera of frame n (config-grammar values: degrees)."""
    if wl.get("camera") == "sample":
        # the reference's defaults (main/hmap.cpp:75,80,85) with sample_config.txt's hfov
        return dict(pos=(-5.0, 5.0, 0.0), hang_deg=-45.0, vang_deg=90.0, hfov_deg=90.0, ortho_width=0.1)
    extent = (1 << wl["log2n"]) * GRID_WIDTH
    cx, cy = extent / 2.0, -extent / 2.0
    t = (n % wl["frames"]) / wl["frames"]
    radius = extent * (140.0 / 163.84)
    px, py = cx + radius * math.cos(2 * math.pi * t), cy + radius * math.sin(2 * math.pi * t)
    hang_deg = math.degrees(math.atan2(cy - py, cx - px))
    if wl["projection"] == 3:
        return dict(pos=(px, py, 30.0), hang_deg=hang_deg, vang_deg=125.0, hfov_deg=90.0,
                    ortho_width=extent * 1.2 / wl["W"])
    return dict(pos=(px, py, 40.0 * extent / 163.84 + 10.0 * (1 - extent / 163.84)), hang_deg=hang_deg,
                vang_deg=110.0, hfov_deg=90.0, ortho_width=0.03)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        sm, smax, reasons = [], [], set()
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/_ref) or, if it was not built, the oracle port
# ------------------------------------------------------------------------------------------------
def run_cpu_reference(wl: dict, frame_ids: list[int], warmup: int, workdir: Path) -> dict:
    """Times frames `frame_ids` at (W/4 x H/4) on the host cores.  Returns dict with per-frame ms, rays, kind."""
    import numpy as np

    import oracle_lib as O

    W, H = wl["W"] // REF_SAMPLE_DIV, wl["H"] // REF_SAMPLE_DIV
    cores = os.cpu_count() or 1
    sample = (f"{len(frame_ids)} frames of the workload's camera path rendered at {W}x{H}: the same cameras at 1/"
              f"{REF_SAMPLE_DIV} of the resolution per axis, i.e. 1/{REF_SAMPLE_DIV ** 2} as many rays covering the same "
              f"field of view (not a subset of the full-resolution rays: w = px/(W-1))")

    # The reference cannot load a 32768^2 map at all (stb_image caps, int indices: SURVEY.md D-9): port only, and
    # the port reads the procedural map's texels on the fly unless the host has room for 15 GiB of arrays.
    if wl["log2n"] >= 15:
        import psutil

        room = psutil.virtual_memory().available >= (48 << 30)
        t0 = time.perf_counter()
        heights = cm = None
        if room:
            hm, cm = O.synth_maps(wl["log2n"], SEED)
            heights = O.update_heightmap(hm, (0.299, 0.587, 0.114), MIN_HEIGHT, MAX_HEIGHT)
            del hm
        gen_s = time.perf_counter() - t0
        ms, frames = [], []
        for i, n in enumerate([frame_ids[0]] * warmup + frame_ids):
            c = camera(wl, n)
            fr = O.make_frame(projection=wl["projection"], width=W, height=H, grid_width=GRID_WIDTH,
                              step_dist=wl["step_dist"], min_height=MIN_HEIGHT, max_height=MAX_HEIGHT, **c)
            t0 = time.perf_counter()
            if room:
                fb, _, _ = O.render(fr, heights, cm, want_steps=False)
            else:
                fb, _, _ = O.render_synth(fr, wl["log2n"], SEED, want_steps=False)
            dt = (time.perf_counter() - t0) * 1e3
            if i >= warmup:
                ms.append(dt)
                frames.append(fb)
        return dict(kind="port", cores=cores, sample=sample, W=W, H=H, ms=ms, ms_as_shipped=None, frames=frames,
                    gen_s=gen_s, binary="oracle/_build/liboracle.so (gcc -O2 -fopenmp), " +
                    ("FP64 height array as the reference holds it" if room else "texels generated on the fly (host too small for the arrays)")
                    + "; the reference itself cannot load a 32768^2 map")

    t0 = time.perf_counter()
    hm, cm = O.synth_maps(wl["log2n"], SEED)
    gen_s = time.perf_counter() - t0
    if O.REF_BIN_O2.exists() and O.REF_BIN.exists():
        hp, cp = workdir / "height.pgm", workdir / "color.tga"
        with open(hp, "wb") as f:
            f.write(b"P5\n%d %d\n255\n" % (hm.shape[1], hm.shape[0]))
            f.write(np.ascontiguousarray(hm[:, :, 0]).tobytes())
        O.write_tga_rgba(cp, cm)
        cams = [camera(wl, n) for n in ([frame_ids[0]] * warmup + frame_ids)]
        kw = dict(width=W, height=H, grid_width=GRID_WIDTH, step_dist=wl["step_dist"], min_height=MIN_HEIGHT,
                  max_height=MAX_HEIGHT, **cams[0])
        cfg = O.config_text(kw, hp, cp)
        script = ["pos %r %r %r hang %r vang %r ortho_width %r" % (*c["pos"], c["hang_deg"], c["vang_deg"], c["ortho_width"])
                  for c in cams]
        out = {}
        for label, binary in (("O2", O.REF_BIN_O2), ("as_shipped", O.REF_BIN)):
            # the as-shipped build (no -O, ~3x slower) is a second data point only: at most 12 frames of it
            lines = script if label == "O2" else script[: warmup + min(len(frame_ids), 12)]
            frames, times = O.run_ref(cfg, wl["projection"], W, H, script=lines, binary=binary, threads=cores,
                                      timeout=3000)
            out[label] = dict(ms=times[warmup:], frames=frames[warmup:])
        return dict(kind="reference", cores=cores, sample=sample, W=W, H=H, ms=out["O2"]["ms"],
                    ms_as_shipped=out["as_shipped"]["ms"], frames=out["O2"]["frames"], gen_s=gen_s,
                    binary="oracle/_ref/hmap_ref_O2 (reference sources + -O2; as shipped = no -O, also timed)")

    # port: the plain-C restatement, OpenMP over all cores
    heights = O.update_heightmap(hm, (0.299, 0.587, 0.114), MIN_HEIGHT, MAX_HEIGHT)
    ms, frames = [], []
    for i, n in enumerate([frame_ids[0]] * warmup + frame_ids):
        c = camera(wl, n)
        fr = O.make_frame(projection=wl["projection"], width=W, height=H, grid_width=GRID_WIDTH,
                          step_dist=wl["step_dist"], min_height=MIN_HEIGHT, max_height=MAX_HEIGHT, **c)
        t0 = time.perf_counter()
        fb, _, _ = O.render(fr, heights, cm, want_steps=False)
        dt = (time.perf_counter() - t0) * 1e3
        if i >= warmup:
            ms.append(dt)
            frames.append(fb)
    return dict(kind="port", cores=cores, sample=sample, W=W, H=H, ms=ms, ms_as_shipped=None, frames=frames,
                gen_s=gen_s, binary="oracle/_build/liboracle.so (gcc -O2 -fopenmp)")


def reference_arm(args, wl) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frame_ids = [(s * args.gpus) % wl["frames"] for s in range(args.steps)]
    with tempfile.TemporaryDirectory(prefix="hmrm_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
        res = run_cpu_reference(wl, frame_ids, args.warmup, Path(td))
    if args.dump_outputs:
        dump_frame(args.dump_outputs, res["frames"][-1])
    rays = res["W"] * res["H"]
    total_ms = sum(res["ms"])
    value = rays * len(res["ms"]) / (total_ms * 1e-3) / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / len(res["ms"]),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "desc": wl["desc"], "sample": res["sample"]},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample"], "binary": res["binary"]},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if res["ms_as_shipped"]:
        line["cpu_baseline"]["value_as_shipped"] = rays * len(res["ms_as_shipped"]) / (sum(res["ms_as_shipped"]) * 1e-3) / 1e6
    emit(line)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
PEER_SYNC_TEXT = {"memops": "waited on and written by stream memory operations (the GPU front end, no SM)",
                  "kernels": "polled and written by one-thread kernels"}


class Job:
    """One workload on this rank: renderer, frames, output buffers."""

    def __init__(self, hmrm, binding, MG, torch, dist, wl, args, rank, world, local, stream):
        self.hmrm, self.binding, self.MG, self.torch, self.dist = hmrm, binding, MG, torch, dist
        self.wl, self.args, self.rank, self.world, self.local, self.stream = wl, args, rank, world, local, stream
        self.W, self.H = wl["W"], wl["H"]
        self.bands = wl.get("mode") == "bands"
        self.traversal = {"auto": 0, "brute": 1, "skip": 2}[args.traversal]
        self.rgb = args.pixels == "rgb8"
        self.channels = 3 if self.rgb else 4
        self.fmt = hmrm.PIXEL_RGB8 if self.rgb else hmrm.PIXEL_RGBA8
        self.r = hmrm.Renderer(local)
        self.r.min_height, self.r.max_height = MIN_HEIGHT, MAX_HEIGHT
        self.r.synth_maps(wl["log2n"], SEED)
        self.d_out = torch.zeros((MG.padded_height(self.H), self.W, 4), dtype=torch.uint8, device=f"cuda:{local}")
        self.peer = None
        self.band_i = 0
        if args.exchange == "auto":
            # measured (DESIGN.md section 6): the kernel's own peer stores win with one writer into the root (N = 2); with
            # more writers their 24- / 32-byte row pieces saturate the root's NVLink ingress and the copy engine wins
            args.exchange = "peer" if world <= 2 else "peer-copy"
        if self.bands and world > 1 and args.exchange in ("peer", "peer-copy", "peer-allreduce"):
            self.peer = MG.PeerFrame(self.r, self.H, self.W, rank, world, local, channels=self.channels,
                                     buffers=max(2, min(6, args.bands_inflight)),
                                     completion="allreduce" if args.exchange == "peer-allreduce" else "device",
                                     exchange="copy" if args.exchange == "peer-copy" else "stores")

    def frame_of(self, n: int, flags: int = 0, w: int = 0, h: int = 0, whole: bool = False, fmt=None):
        w, h = w or self.W, h or self.H
        c = camera(self.wl, n)
        split = self.bands and not whole and w == self.W
        return self.r.frame(projection=self.wl["projection"], screen_width=w, screen_height=h, cam_pos=c["pos"],
                            hang=self.hmrm.deg2rad(c["hang_deg"]), vang=self.hmrm.deg2rad(c["vang_deg"]),
                            hfov=self.hmrm.deg2rad(c["hfov_deg"]), ortho_width=c["ortho_width"], grid_width=GRID_WIDTH,
                            step_dist=self.wl["step_dist"], traversal=self.traversal, flags=flags,
                            pixel_format=self.fmt if fmt is None else fmt,
                            band_count=self.world if split else 0, band_index=self.rank if split else 0)

    def render_step(self, n: int, flags: int = 0, stream=None, frame=None, out=None, want_tensor=False):
        """One step of the workload on this rank: a whole frame, or this rank's bands of the frame everybody works
        on.  Bands land in rank 0's frame by peer stores from the render kernel itself (default; completion on the
        device or by an all-reduce) or by pack + NCCL gather + unpack (--exchange gather)."""
        s = stream if stream is not None else self.stream
        if frame is None:
            frame = self.frame_of(n, flags=flags)
        if self.peer is not None:
            i = self.band_i
            self.band_i += 1
            self.peer.render(frame, i, s.cuda_stream)
            if self.peer.completion == "device":
                self.peer.complete(i, s.cuda_stream)
            else:
                with self.torch.cuda.stream(s):
                    self.peer.complete(i, s.cuda_stream)
            self.peer.release(i, s.cuda_stream)          # nothing reads the frame in the device-resident timing
            return self.peer.tensor(i) if want_tensor else None
        self.r.render_device(frame, self.d_out if out is None else out, s.cuda_stream)
        if self.bands and self.world > 1 and self.args.exchange != "none":
            view = self.d_out.view(-1)[: self.MG.padded_height(self.H) * self.W * self.channels].view(
                self.MG.padded_height(self.H), self.W, self.channels)
            return self.MG.gather_interleaved_bands(view, self.H, self.rank, self.world)
        return self.d_out

    def close(self):
        if self.peer is not None:
            self.peer.check()
            self.peer.close()
        self.r.close()


def measure(job: Job, steps: int, warmup: int, sampler, want_cpu: bool, dump_dir: str | None = None) -> dict | None:
    """Runs `steps` timed steps of job's workload (after `warmup`): device-resident value, e2e through the C ABI,
    statistics, roofline inputs.  Returns the record on rank 0, None elsewhere.  With `dump_dir`, rank 0's frame of
    the last device-resident timed step goes there (dump_frame)."""
    import numpy as np

    torch, dist, hmrm, binding, MG = job.torch, job.dist, job.hmrm, job.binding, job.MG
    wl, args, rank, world, local, stream = job.wl, job.args, job.rank, job.world, job.local, job.stream
    W, H, bands, r = job.W, job.H, job.bands, job.r
    frames_n = wl["frames"]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if bands:
        # every rank works on the SAME frame: its interleaved tile rows; rank 0 ends up with the whole frame
        my_frames = [s % frames_n for s in range(steps)]
        warm_frames = [(steps + s) % frames_n for s in range(warmup)]
    else:
        my_frames = [(s * world + rank) % frames_n for s in range(steps)]
        warm_frames = [((steps + s) * world + rank) % frames_n for s in range(warmup)]

    # ---- untimed statistics pass over the timed frames: reference-equivalent steps S, hits, fetches ----
    S = hits = fetches = 0
    for n in my_frames:
        job.render_step(n, flags=hmrm.FLAG_STATS)
        st = r.stats()
        S += st.steps
        hits += st.surf_hits
        fetches += st.fetches
        if st.status:
            raise SystemExit(f"frame {n}: kernel reported status {st.status}")

    # ---- value: K frames, device-resident, CUDA events on the launching stream ----
    for n in warm_frames:
        job.render_step(n)

    def keep_busy(seconds: float) -> None:
        """Same kernel, same frames, back to back (untimed): the timed region is short against nvidia-smi's
        sampling period, so the clocks are sampled over this load window that brackets it."""
        t_end = time.perf_counter() + seconds
        while time.perf_counter() < t_end:
            for n in my_frames[:32]:
                r.render_device(job.frame_of(n, whole=True), job.d_out, stream.cuda_stream)
            stream.synchronize()
            if dist is not None:
                break       # collectives must stay in lock step across ranks: one pass only

    t_wall0 = time.perf_counter()
    keep_busy(0.5)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Two frames in flight: frames alternate between two streams (and two output buffers) so that the next frame's
    # CTAs fill the SMs that the previous frame's tail leaves idle.  The timed region starts on `stream` with both
    # streams idle and ends on `stream` after it has joined the others.
    n_flight = max(1, min(6 if bands else 4, args.bands_inflight if bands else args.inflight))
    if bands and job.peer is None and not (world > 1 and args.exchange == "none"):
        n_flight = 1                         # the NCCL gather path works on one buffer
    if job.peer is not None:
        n_flight = min(n_flight, len(job.peer.ptrs))     # one stream per rotating buffer
    streams = [stream] + [torch.cuda.Stream(device=local) for _ in range(n_flight - 1)]
    outs = [job.d_out] + [torch.zeros_like(job.d_out) for _ in range(n_flight - 1)]
    timed_frames = [job.frame_of(n) for n in my_frames]     # host-side frame descriptions, built outside the timed region
    for s2 in streams[1:]:
        s2.wait_stream(stream)
    ev0.record(stream)
    for s2 in streams[1:]:
        s2.wait_event(ev0)
    t_host0 = time.perf_counter()
    for i, n in enumerate(my_frames):
        if bands:
            job.render_step(n, stream=streams[i % n_flight], frame=timed_frames[i], out=outs[i % n_flight])
        else:
            r.render_device(timed_frames[i], outs[i % n_flight], streams[i % n_flight].cuda_stream)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3      # the host's share: how long the K enqueues took
    for s2 in streams[1:]:
        stream.wait_stream(s2)
    ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    dev_ms_own = dev_ms
    last_frame = None
    if dump_dir is not None and rank == 0:
        # copied before keep_busy / the roofline pass render into outs[0] again
        last = outs[(steps - 1) % n_flight]
        last_frame = last.view(-1)[: H * W * job.channels].view(H, W, job.channels).cpu().numpy()
    keep_busy(0.4)

    # ---- e2e: the user's call — host output buffer, D2H inside the timed region ----
    E2E_DEPTH = 3                               # frames that may stay in flight behind the newest one
    host_bufs = [binding.pinned_empty((H, W, job.channels)) for _ in range(E2E_DEPTH + 1)]

    # bands at N > 1: the host frames live in POSIX shared memory, page-locked by every rank; each rank copies its own
    # tile rows out over its own PCIe link (hmrm_render_async with band_count > 1).  Two frames rotate: while frame i is
    # rendered and copied, the ranks agree (all-reduce, host-synchronised) that frame i - 1 is complete in host memory.
    shared = shared_np = None
    if bands and world > 1:
        from multiprocessing import shared_memory

        frame_bytes = H * W * job.channels
        name = [None]
        if rank == 0:
            shared = shared_memory.SharedMemory(create=True, size=2 * frame_bytes)
            name[0] = shared.name
        dist.broadcast_object_list(name, src=0)
        if rank != 0:
            shared = shared_memory.SharedMemory(name=name[0])
            from multiprocessing import resource_tracker

            resource_tracker.unregister(shared._name, "shared_memory")     # rank 0 owns (and unlinks) the segment
        shared_np = np.ndarray((2, H, W, job.channels), dtype=np.uint8, buffer=shared.buf)
        if binding.load_library().hmrm_host_register(shared_np.ctypes.data, 2 * frame_bytes) != 0:
            raise SystemExit("hmrm_host_register failed")
        e2e_token = torch.zeros(1, device=f"cuda:{local}")

    def frame_complete_everywhere() -> None:
        dist.all_reduce(e2e_token)
        e2e_token.cpu()                        # host-synchronised: every rank's copy of that frame has landed

    def e2e_step(i: int, n: int) -> None:
        if bands and world > 1:
            r.render_async(job.frame_of(n), shared_np[i % 2])
            r.wait_pending(1)                  # this rank's part of frame i - 1 is in host memory
            if i > 0:
                frame_complete_everywhere()    # ... and everybody else's: frame i - 1 is whole
        else:
            # the library's streaming call: the newest frames render while an older one is still being copied to the
            # host; after wait_pending(d) frame i-d is complete in its host buffer (d + 1 buffers rotate)
            r.render_async(job.frame_of(n, whole=True), host_bufs[i % (E2E_DEPTH + 1)])
            r.wait_pending(E2E_DEPTH)

    def e2e_drain() -> None:
        r.wait()
        if bands and world > 1:
            frame_complete_everywhere()

    for i, n in enumerate(warm_frames):
        e2e_step(i, n)
    e2e_drain()
    barrier()
    t0 = time.perf_counter()
    for i, n in enumerate(my_frames):
        e2e_step(i, n)
    e2e_drain()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    clocks = None
    if sampler is not None and rank == 0:
        clocks = sampler.stop(t_wall0, time.perf_counter())
        clocks["window"] = "0.9 s of the timed kernel running back to back around the timed region, plus the timed regions"

    # ---- bands: the gathered frame must be byte-identical to the same frame rendered whole on one GPU ----
    bands_ok = None
    single_ms = None
    if bands and world > 1:
        gathered = job.render_step(my_frames[0], want_tensor=True)
        stream.synchronize()
        if rank == 0:
            whole = torch.zeros_like(job.d_out)
            r.render_device(job.frame_of(my_frames[0], whole=True), whole, stream.cuda_stream)
            stream.synchronize()
            want = whole.view(-1)[: MG.padded_height(H) * W * job.channels].view(MG.padded_height(H), W, job.channels)[:H]
            # (--exchange none is a diagnostic: the bands stay on their GPUs, there is no gathered frame to compare)
            bands_ok = bool(torch.equal(gathered, want)) if args.exchange != "none" else None
            # the same frames rendered whole by this one GPU, same build, same two-in-flight pipeline: the strong-scaling base
            k1 = min(len(my_frames), 24)
            outs1 = [whole, torch.zeros_like(whole)]
            st2 = torch.cuda.Stream(device=local)
            for rep in range(2):
                st2.wait_stream(stream)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                st2.wait_event(e0)
                for i, n in enumerate(my_frames[:k1]):
                    r.render_device(job.frame_of(n, whole=True), outs1[i % 2], (stream if i % 2 == 0 else st2).cuda_stream)
                stream.wait_stream(st2)
                e1.record(stream)
                stream.synchronize()
                single_ms = e0.elapsed_time(e1) / k1
        barrier()

    # ---- per-kernel duration for the roofline: CUDA events around K2 inside the library, one frame at a time ----
    kernel_ms = []
    for n in my_frames[:64]:
        r.render_device(job.frame_of(n), job.d_out, stream.cuda_stream)
        kernel_ms.append(r.stats().kernel_ms)
    k_ms_mean = sum(kernel_ms) / len(kernel_ms)

    vals = torch.tensor([dev_ms, e2e_ms, float(S), float(hits), float(fetches), k_ms_mean], dtype=torch.float64,
                        device=f"cuda:{local}")
    per_rank = None
    if dist is not None:
        mine = torch.tensor([dev_ms_own, host_enqueue_ms, k_ms_mean], dtype=torch.float64, device=f"cuda:{local}")
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        per_rank = [[float(x) for x in t.tolist()] for t in every]
        mx = vals.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = vals.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms = float(mx[0]), float(mx[1])
        S, hits, fetches = float(sm[2]), float(sm[3]), float(sm[4])
        k_ms = float(sm[5]) / world
    else:
        k_ms = k_ms_mean

    rec = None
    if rank == 0:
        # frames: every rank renders its own frames (weak); bands: all ranks share each frame (strong)
        rays_total = W * H * steps * (1 if bands else world)
        frames_total = steps * (1 if bands else world)
        value = rays_total / (dev_ms * 1e-3) / 1e6
        e2e_value = rays_total / (e2e_ms * 1e-3) / 1e6
        launches = steps * world             # render-kernel launches (the roofline's "per launch")
        # every kernel of ours inside the timed region: the render kernel, plus — only when the peer-frame protocol
        # runs as one-thread kernels (HMRM_PEER_SYNC=kernels; the default are stream memory operations, no kernels) —
        # per frame: every rank waits for the buffer's release and signals arrival, the root waits for all and releases
        all_launches = launches
        if bands and world > 1 and args.exchange in ("peer", "peer-copy") and r.peer_sync_mode() == "kernels":
            all_launches += steps * (2 * world + 2)
        # algorithmic bytes (SURVEY.md §8d): 8 B per reference step + 4 B colormap per hit + 4 B store per pixel
        # (3 B in RGB8), per launch = per rank and frame
        px_bytes = job.channels
        alg_bytes = (8 * S + 4 * hits + px_bytes * rays_total) / launches
        # bytes the kernel as implemented has to move: one 2 B pyramid texel per fetch, the colour per hit, the pixel
        useful_bytes = (2 * fetches + 4 * hits + px_bytes * rays_total) / launches
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        prof = traffic_profile(args_workload_key(job), bands, world)
        traffic = prof.get("dram_bytes")
        warp_inst = prof.get("warp_inst")
        sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        issue_frac = None
        if warp_inst and (world == 1 or bands):
            issue_frac = warp_inst / (SM_COUNT_FALLBACK * 4 * sm_mhz * 1e6 * (k_ms * 1e-3))
        rec = {
            "value": value, "ms_per_step": dev_ms / steps, "steps": steps,
            "scaling": "strong" if bands else "weak",
            "config": {"workload": job.args.workload if not getattr(job, "sub", False) else job.sub_name, "desc": wl["desc"],
                       "traversal": args.traversal, "precision": "fp64_exact",
                       "pyramid_layout": {0: "rowmajor", 1: "tile4", 2: "zorder"}.get(r.get_layout()),
                       "pixel_format": args.pixels,
                       "in_flight": f"{n_flight} frame(s) on as many streams (the tail of frame n overlaps the head of frame n+1)",
                       "sharding": (f"each frame split into interleaved 4-row tile bands over {world} GPU(s), maps replicated; "
                                    + {"peer": "every rank's kernel stores its bands straight into rank 0's frame (CUDA IPC peer "
                                               "memory over NVLink); completion and buffer release through words in rank 0's "
                                               "memory, " + PEER_SYNC_TEXT[r.peer_sync_mode()] + " (no collective)",
                                       "peer-copy": "every rank renders its bands into a staging frame on its own device and pushes "
                                                    "its tile rows into rank 0's frame with one strided device-to-device copy "
                                                    "(CUDA IPC peer memory over NVLink, copy engine); completion and buffer "
                                                    "release through words in rank 0's memory, "
                                                    + PEER_SYNC_TEXT[r.peer_sync_mode()] + " (no collective)",
                                       "peer-allreduce": "every rank's kernel stores its bands straight into rank 0's frame; "
                                                         "one-element NCCL all-reduce as the completion barrier",
                                       "gather": "bands packed, gathered to rank 0 (NCCL), unpacked",
                                       "none": "DIAGNOSTIC: no exchange, the bands stay on the GPUs that rendered them"}[args.exchange]
                                    if world > 1 else "one GPU renders the whole frame") if bands else
                                   f"frames round-robin over {world} GPU(s), maps replicated, no collective",
                       "l2": "inputs larger than L2 (the height pyramid's level 0 alone is >= 128 MiB; the camera moves "
                             "every frame)" if wl["log2n"] >= 13 else "inputs may fit L2; no flush: the camera moves every frame"
                             if wl.get("camera") != "sample" else "inputs fit L2 and the camera is fixed (the reference's "
                             "own CPU-runnable case): an L2-resident figure"},
            "march_steps_per_s": S / (dev_ms * 1e-3),
            "ref_steps_per_frame": S / frames_total,
            "fetches_per_frame": fetches / frames_total,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak,
                         "peak_source": "measured" if "hbm_gbs" in peaks else "fallback", "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "kernel": "k2_render_lin", "kernel_ms": k_ms,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "useful_bytes": useful_bytes,
                         "traffic_ratio": (traffic / useful_bytes) if traffic else None,
                         "dram_gbs": (traffic / (k_ms * 1e-3) / 1e9) if traffic else None,
                         "dram_frac": (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "warp_inst_per_launch": warp_inst,
                         "issue_frac": issue_frac,
                         "limiter": "instruction issue + latency of the dependent mip fetch (ncu: profiles/), not any memory level",
                         "note": "frac follows SURVEY.md 8(d): algorithmic bytes 8*S + 4*hits + pixel bytes (S = reference-"
                                 "equivalent steps) over the kernel time against the measured HBM peak; the skip traversal "
                                 "issues F << S fetches, so frac > 1 is expected and is NOT a utilisation figure. "
                                 "useful_bytes = 2*F + 4*hits + pixel bytes is what this kernel must move; traffic (ncu dram "
                                 "read+write of one launch of this workload, profiles/traffic.json) / useful_bytes is the "
                                 "re-read factor; issue_frac = warp instructions / (SMs*4*f*t) is the kernel's own ceiling"},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_ms / steps,
                    "h2d_bytes_per_step": 1024, "d2h_bytes_per_step": W * H * job.channels,
                    "d2h_gbs": W * H * job.channels * frames_total / (e2e_ms * 1e-3) / 1e9,
                    "api": ("hmrm_render_async with band_count = N into a host frame in shared memory, page-locked by every "
                            "rank: each rank copies its own tile rows out over its own PCIe link; two host frames rotate and "
                            "an all-reduce per frame tells every rank that the previous frame is whole")
                    if (bands and world > 1) else "hmrm_render_async + hmrm_wait_pending(3): every frame lands in pinned host memory; the "
                           "copy-out of frame n overlaps the kernels of the next frames (four device + four host "
                           "buffers)"},
            "gpu_launches": all_launches,
            "render_kernel_launches": launches,
            "host_enqueue_ms_per_step": host_enqueue_ms / steps,
            "clocks": clocks,
        }
        if bands_ok is not None:
            rec["config"]["gathered_frame_equals_single_gpu_frame"] = bands_ok
            rec["single_gpu_ms_per_step"] = single_ms
            rec["strong_scaling_efficiency"] = (single_ms / (dev_ms / steps)) / world if single_ms else None
            rec["kernel_ms_per_rank"] = k_ms
            if per_rank is not None:
                rec["per_rank"] = {"timed_region_ms_per_step": [x[0] / steps for x in per_rank],
                                   "host_enqueue_ms_per_step": [x[1] / steps for x in per_rank],
                                   "render_kernel_alone_ms": [x[2] for x in per_rank]}
        if want_cpu:
            with tempfile.TemporaryDirectory(prefix="hmrm_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
                res = run_cpu_reference(wl, my_frames[:args.cpu_frames], 1, Path(td))
            cpu_rays = res["W"] * res["H"] * len(res["ms"])
            cb = {"value": cpu_rays / (sum(res["ms"]) * 1e-3) / 1e6, "unit": "Mrays/s", "cores": res["cores"],
                  "kind": res["kind"], "sample": res["sample"], "binary": res["binary"]}
            if res["ms_as_shipped"]:
                cb["value_as_shipped"] = cpu_rays / (sum(res["ms_as_shipped"]) * 1e-3) / 1e6
            # parity of the sampled frames: GPU render at the sample resolution == CPU frame, bit for bit
            ok = True
            for n, want in zip(my_frames[:args.cpu_frames], res["frames"]):
                got = r.render(job.frame_of(n, w=res["W"], h=res["H"], whole=True, fmt=hmrm.PIXEL_RGBA8))
                ok = ok and bool(np.array_equal(got, want))
            cb["parity_of_sample"] = "bit-exact" if ok else "MISMATCH"
            rec["cpu_baseline"] = cb

    if shared is not None:
        ok_host = True
        if rank == 0:
            # the host frame of the last e2e step must be the frame itself
            ok_host = bool(np.array_equal(shared_np[(len(my_frames) - 1) % 2], r.render(job.frame_of(my_frames[-1], whole=True))))
        binding.load_library().hmrm_host_unregister(shared_np.ctypes.data)
        del shared_np
        dist.barrier()
        shared.close()
        if rank == 0:
            shared.unlink()
            if not ok_host:
                raise SystemExit("bands e2e: the shared host frame differs from the frame rendered whole")
    if last_frame is not None:
        dump_frame(dump_dir, last_frame)
    return rec


def traffic_profile(workload: str, bands: bool, world: int) -> dict:
    """ncu counters of ONE render-kernel launch of this workload (profiles/traffic.json, tools/make_traffic_json.py).
    A band launch at N > 1 has its own capture (`<workload>x<N>`: rank 0's band of an N-way split) or none."""
    try:
        table = json.loads((ROOT / "profiles" / "traffic.json").read_text())
    except (OSError, ValueError):
        return {}
    prof = table.get(f"{workload}x{world}" if (bands and world > 1) else workload, {})
    return prof if isinstance(prof, dict) else {"dram_bytes": prof}


def args_workload_key(job: Job) -> str:
    return job.sub_name if getattr(job, "sub", False) else job.args.workload


def ours_arm(args, wl) -> None:
    import torch

    import hmrm_pkg

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if args.dump_outputs and wl.get("mode") == "bands" and world > 1:
        raise SystemExit("--dump-outputs: a band-split frame is assembled across the ranks; run it with --gpus 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    hmrm = hmrm_pkg.load()
    from heightmap_ray_marcher_b200 import binding
    from heightmap_ray_marcher_b200 import multi_gpu as MG

    stream = torch.cuda.Stream(device=local)       # a real (non-default) stream: kernels and events share it
    torch.cuda.set_stream(stream)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    job = Job(hmrm, binding, MG, torch, dist, wl, args, rank, world, local, stream)
    rec = measure(job, args.steps, args.warmup, sampler, want_cpu=(world == 1 and not args.no_cpu_baseline),
                  dump_dir=args.dump_outputs)
    job.close()

    # ---- N > 1, default workload: BASELINE configs[4] (row bands of one 8K frame over the N GPUs) as a sub-record ----
    sub = None
    if world > 1 and args.workload == "flythrough4k" and not args.no_bands:
        sub_wl = WORKLOADS[args.bands_workload]
        job2 = Job(hmrm, binding, MG, torch, dist, sub_wl, args, rank, world, local, stream)
        job2.sub, job2.sub_name = True, args.bands_workload
        sub = measure(job2, max(args.bands_steps, 60 if args.bands_workload == "bands8k" else 1), max(args.warmup, 3), None, want_cpu=False)
        job2.close()

    if rank == 0:
        line = {
            "metric": "Mrays/s", "value": rec["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
            "scaling": rec["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        }
        for k in ("config", "march_steps_per_s", "ref_steps_per_frame", "fetches_per_frame", "roofline", "e2e", "gpu_launches",
                  "render_kernel_launches", "host_enqueue_ms_per_step", "clocks", "single_gpu_ms_per_step", "strong_scaling_efficiency",
                  "kernel_ms_per_rank", "per_rank", "cpu_baseline"):
            if k in rec:
                line[k] = rec[k]
        if sub is not None:
            sub.pop("clocks", None)
            line["bands8k"] = sub
            line["gpu_launches"] += sub["gpu_launches"]
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


_JSON_FD = None


def claim_stdout() -> None:
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner there) must not add
    lines: keep the real stdout for emit() and point fd 1 at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main() -> None:
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240,
                    help="timed steps (frames per GPU); the default is the workload's whole 240-frame camera orbit")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="flythrough4k")
    ap.add_argument("--traversal", choices=["auto", "brute", "skip"], default="auto")
    ap.add_argument("--pixels", choices=["rgb8", "rgba8"], default="rgb8",
                    help="frame format: rgb8 = the reference's pixels without the constant alpha byte (default), "
                         "rgba8 = the reference's framebuf layout")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", choices=["auto", "peer", "peer-copy", "peer-allreduce", "gather", "none"], default="auto",
                    help="bands workloads at N > 1: how the bands reach rank 0 (none: a diagnostic, the bands stay where "
                         "they were rendered: the render kernels' own floor)")
    ap.add_argument("--no-bands", action="store_true", help="N > 1: skip the bands8k sub-record")
    ap.add_argument("--bands-workload", choices=["bands8k", "smokebands"], default="bands8k")
    ap.add_argument("--bands-steps", type=int, default=96)
    ap.add_argument("--cpu-frames", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR/frame.npy + DIR/pixel_index.npy (see above)")
    ap.add_argument("--inflight", type=int, default=2, help="frames in flight in the device-resident timing (1..4)")
    ap.add_argument("--bands-inflight", type=int, default=4,
                    help="bands workloads: frames in flight (1..6; one stream and one peer buffer each); measured per 8K frame: "
                         "N = 4: 0.442 ms with 2, 0.411 ms with 3; N = 8: 0.2395 / 0.2268 / 0.2215 ms with 2 / 3 / 4")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        reference_arm(args, wl)
    else:
        ours_arm(args, wl)


if __name__ == "__main__":
    main()
