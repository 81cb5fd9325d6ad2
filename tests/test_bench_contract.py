"""CPU: bench.py's reference arm runs here (no GPU needed) and prints one JSON line with the contract's keys."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_contract_line(oracle):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "smoke",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["config"]["workload"] == "smoke"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dump_outputs(oracle, tmp_path):
    """--dump-outputs: the last timed frame (160x90 RGBA8 at the reference arm's sample resolution), every pixel."""
    import numpy as np

    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "smoke",
                          "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert res.returncode == 0, res.stderr[-2000:]
    frame, idx = np.load(tmp_path / "frame.npy"), np.load(tmp_path / "pixel_index.npy")
    assert frame.dtype == np.float32 and frame.shape == (160 * 90, 4) and frame.max() <= 255 and frame[:, 3].any()
    assert idx.dtype == np.float64 and np.array_equal(idx, np.arange(160 * 90))


def test_reference_arm_on_other_ranks_is_silent(oracle):
    import os

    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "smoke", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=str(ROOT), env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_orbit_camera_stays_outside_the_box():
    """Every camera of every workload must be outside the terrain AABB, else the frame is all sky (SURVEY.md D-3)."""
    sys.path.insert(0, str(ROOT))
    import bench

    for name, wl in bench.WORKLOADS.items():
        extent = (1 << wl["log2n"]) * bench.GRID_WIDTH
        for n in range(0, wl["frames"], 7):
            c = bench.camera(wl, n)
            x, y, z = c["pos"]
            inside = 0.0 <= x <= extent and -extent <= y <= 0.0 and bench.MIN_HEIGHT <= z <= bench.MAX_HEIGHT
            assert not inside, (name, n, c)
            # (sample720 is the reference's own default camera: beside the map at z = 0, main/hmap.cpp:75)
            assert z > bench.MAX_HEIGHT or wl.get("camera") == "sample"


def test_traffic_profile_lookup():
    """roofline.traffic comes from profiles/traffic.json: whole-frame launches by workload, band launches of an N-way
    split by `<workload>x<N>`; a split that was never captured has no traffic figure rather than a wrong one."""
    import bench

    whole = bench.traffic_profile("bands8k", True, 1)
    assert whole["dram_bytes"] > 0 and whole["warp_inst"] > 0
    assert bench.traffic_profile("flythrough4k", False, 8) == bench.traffic_profile("flythrough4k", False, 1)
    band = bench.traffic_profile("bands8k", True, 8)
    assert 0 < band["warp_inst"] < whole["warp_inst"] / 7 and band["dram_bytes"] < whole["dram_bytes"]
    assert bench.traffic_profile("bands8k", True, 3) == {}
    assert bench.traffic_profile("no_such_workload", False, 1) == {}
