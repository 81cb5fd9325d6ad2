"""Many small views of one terrain: a loop of hmrm_render_device (one view per call) against one hmrm_render_views_device
batch, on the bench's flythrough4k map (16384^2 fBm, seed 1234), one GPU.

    python tools/views_probe.py [--reps 3] [--rays 64e6] [--out FILE]      (writes profiles/r13_views_probe.txt)

Cameras: the bench's orbit cameras (frame j % 240), with vang spread over 31 values from 100 to 115 degrees so that the
batch has many distinct row schedules.  Sizes 64^2, 128^2, 256^2, 640x360, 1280x720 perspective and 256^2 spherical;
n views per batch so that one batch has >= --rays rays.  Two more rows at 64^2 give every view its own vang (one row
schedule per view, the host's worst case), at that n and at the largest n, 65536.  In one process, alternating --reps
times:
  (a) loop: n hmrm_render_device calls, view j into byte j * W * H * 4 of one device buffer;
  (b) batch: one hmrm_render_views_device, rank-major schedule (the default);
  (c) batch with the view-major schedule (HMRM_VIEWS_VIEW_MAJOR, a second context over the same map).
All on one caller stream.  device ms: CUDA events around the whole loop / batch; wall ms: host clock from the first
enqueue to a stream synchronise; set-up ms: host time of the hmrm_render_views_device call alone (validation, records,
schedule, spherical tables; the launch slots' buffers have grown in the warm-up).  (a), (b) and (c) must be
byte-identical in every repetition.
"""
import argparse
import json
import math
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402
import hmrm_pkg  # noqa: E402
from png_probe import card  # noqa: E402

# (W, H, projection, n (None: from --rays), every view its own vang)
SIZES = [(64, 64, 1, None, False), (128, 128, 1, None, False), (256, 256, 1, None, False), (640, 360, 1, None, False),
         (1280, 720, 1, None, False), (256, 256, 2, None, False), (64, 64, 1, None, True), (64, 64, 1, 65536, True)]


def cameras(hmrm, wl, n, distinct):
    out = []
    for j in range(n):
        c = bench.camera(wl, j)
        vang = 100.0 + 15.0 * j / n if distinct else 100.0 + 0.5 * (j % 31)
        out.append((c["pos"], hmrm.deg2rad(c["hang_deg"]), hmrm.deg2rad(vang)))
    return out


def make_renderer(hmrm, wl):
    r = hmrm.Renderer(0)
    r.min_height, r.max_height = bench.MIN_HEIGHT, bench.MAX_HEIGHT
    r.synth_maps(wl["log2n"], bench.SEED)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rays", type=float, default=64e6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    hmrm = hmrm_pkg.load()
    wl = bench.WORKLOADS["flythrough4k"]
    r = make_renderer(hmrm, wl)
    os.environ["HMRM_VIEWS_VIEW_MAJOR"] = "1"          # read once, when the context is created
    rv = make_renderer(hmrm, wl)
    del os.environ["HMRM_VIEWS_VIEW_MAJOR"]
    st = torch.cuda.Stream()
    c0 = bench.camera(wl, 0)
    lines, results = [], []
    info = card()
    lines.append(f"card: {info}")
    lines.append("size        proj  n      rays(M)  kind   device_ms  views/s     Grays/s  wall_ms   setup_ms  vang")
    for W, H, proj, n, distinct in SIZES:
        n = n or min(65536, math.ceil(args.rays / (W * H)))
        cams = cameras(hmrm, wl, n, distinct)
        f = r.frame(projection=proj, screen_width=W, screen_height=H, cam_pos=c0["pos"], hfov=hmrm.deg2rad(90.0),
                    grid_width=bench.GRID_WIDTH, step_dist=wl["step_dist"], ortho_width=c0["ortho_width"])
        frames = []
        for pos, hang, vang in cams:
            g = type(f).from_buffer_copy(f)
            g.cam_pos[:] = list(pos)
            g.hang, g.vang = hang, vang
            frames.append(g)
        # the batch takes the cameras as an [n, 5] array: a list of n tuples costs the binding ~1 us per camera in
        # Python, which would otherwise be counted as the library's set-up
        cam_rows = np.array([(*pos, hang, vang) for pos, hang, vang in cams], dtype=np.float64)
        view = W * H * 4
        bufs = {k: torch.empty(n * view, dtype=torch.uint8, device="cuda:0") for k in "abc"}

        def run(kind):
            buf = bufs[kind]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(st)
            setup = 0.0
            if kind == "a":
                base = buf.data_ptr()
                for j, g in enumerate(frames):
                    r.render_device(g, base + j * view, st.cuda_stream)
            else:
                s0 = time.perf_counter()
                (r if kind == "b" else rv).render_views_device(f, cam_rows, buf, st.cuda_stream)
                setup = (time.perf_counter() - s0) * 1e3
            e1.record(st)
            st.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            return e0.elapsed_time(e1), wall, setup

        # warm-up of every shape; the batches once per launch slot, so that no timed batch grows a slot's buffers
        run("a")
        for _ in range(8):
            run("b")
            run("c")
        per = {k: [] for k in "abc"}
        for rep in range(args.reps):
            for kind in ("abc" if rep % 2 == 0 else "cba"):
                per[kind].append(run(kind))
            assert torch.equal(bufs["a"], bufs["b"]) and torch.equal(bufs["a"], bufs["c"]), f"{W}x{H}: outputs differ"
        for kind in "abc":
            dev = sorted(v[0] for v in per[kind])[len(per[kind]) // 2]
            wall = sorted(v[1] for v in per[kind])[len(per[kind]) // 2]
            setup = sorted(v[2] for v in per[kind])[len(per[kind]) // 2]
            rays = n * W * H
            res = dict(W=W, H=H, projection=proj, n=n, distinct_vang=distinct,
                       kind={"a": "loop", "b": "batch", "c": "batch_view_major"}[kind],
                       device_ms=[round(v[0], 3) for v in per[kind]], wall_ms=[round(v[1], 3) for v in per[kind]],
                       setup_ms=[round(v[2], 3) for v in per[kind]], views_per_s=n / dev * 1e3,
                       grays_per_s=rays / dev / 1e6)
            results.append(res)
            lines.append(f"{W}x{H:<6} {'persp' if proj == 1 else 'spher'} {n:<6} {rays / 1e6:7.1f}  {res['kind'][:6]:6} "
                         f"{dev:9.2f}  {res['views_per_s']:10.0f}  {res['grays_per_s']:6.2f}  {wall:8.2f}  {setup:8.2f}  "
                         f"{'per view' if distinct else '31 values'}")
        a = results[-3:]
        lines.append(f"  speed-up of the batch over the loop (median device ms): {a[1]['views_per_s'] / a[0]['views_per_s']:.2f}x,"
                     f" view-major schedule {a[2]['views_per_s'] / a[0]['views_per_s']:.2f}x; outputs byte-identical")
        print("\n".join(lines[-4:]), flush=True)
        del bufs
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n" + json.dumps(dict(card=info, results=results)) + "\n"
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text)
    print(json.dumps(dict(card=info, reps=args.reps)))
    r.close()
    rv.close()


if __name__ == "__main__":
    main()
