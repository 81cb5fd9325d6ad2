"""GPU: bench.py --dump-outputs writes the frame of the last timed step, and that frame is the oracle's frame."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def test_dump_outputs_is_the_last_timed_frame(hmrm, oracle, tmp_path):
    steps = 5
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "smoke", "--steps", str(steps),
                          "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert res.returncode == 0, res.stderr[-2000:]

    # the dump must be the frame of camera steps - 1: the evidence that --steps sets the number of timed steps
    import bench

    wl = bench.WORKLOADS["smoke"]
    hm, cm = oracle.synth_maps(wl["log2n"], bench.SEED)
    heights = oracle.update_heightmap(hm, (0.299, 0.587, 0.114), bench.MIN_HEIGHT, bench.MAX_HEIGHT)
    fr = oracle.make_frame(projection=wl["projection"], width=wl["W"], height=wl["H"], grid_width=bench.GRID_WIDTH,
                           step_dist=wl["step_dist"], min_height=bench.MIN_HEIGHT, max_height=bench.MAX_HEIGHT,
                           **bench.camera(wl, steps - 1))
    want, _, _ = oracle.render(fr, heights, cm, want_steps=False)

    frame, idx = np.load(tmp_path / "frame.npy"), np.load(tmp_path / "pixel_index.npy")
    assert frame.dtype == np.float32 and idx.dtype == np.float64
    assert np.array_equal(idx, np.arange(wl["W"] * wl["H"]))           # a frame this small is dumped whole
    # default pixel format RGB8: the reference's pixels without the alpha byte
    assert np.array_equal(frame, want[:, :, :3].reshape(-1, 3).astype(np.float32))
