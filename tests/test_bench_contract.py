"""bench.py contract: the reference arm runs without a GPU on a tiny workload and prints exactly one JSON line with the
keys a caller reads; on a GPU, --dump-outputs writes what the timed path returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--scan-points", "3000", "--map-points", "30000"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout          # the ikd-Tree's own printf()s must not reach stdout
    o = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in o, k
    assert o["impl"] == "reference" and o["value"] > 0 and o["higher_is_better"] is True and o["vs_baseline"] is None
    assert o["cpu_baseline"]["kind"] in ("reference", "port") and o["cpu_baseline"]["cores"] >= 1
    assert o["e2e"]["h2d_bytes_per_step"] == 0 and o["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in o["config"] and "model" not in o["config"]


@pytest.mark.gpu
def test_dump_outputs_is_the_timed_pass(tmp_path, gpu_lib):
    """--dump-outputs writes what the last timed search pass returned: the same pass run directly on the same seeded workload."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--scan-points", "3000",
                        "--map-points", "30000", "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 3
    d = {k: np.load(tmp_path / f"{k}.npy") for k in ("HtH", "Htr", "selected_points", "residual_sum")}
    assert all(a.dtype == np.float64 for a in d.values()) and d["HtH"].shape == (12, 12) and d["Htr"].shape == (12,)
    import bench
    c = bench.make_workload("C2", 1, 3000, 30000)
    p = c["pose_init"]
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=int(30000 * 1.2) + 1000, max_scan_points=3016)   # bench.py's sizes
    g.set_reseed(False)
    g.map_build(c["map_xyz"])
    g.scan_upload(c["body_xyz"])
    H, b, m, rs = g.icp_iterate(p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True)
    g.close()
    assert int(d["selected_points"]) == m > 0
    for got, want in ((d["HtH"], H), (d["Htr"], b), (d["residual_sum"], rs)):
        assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()


def test_dump_outputs_rejected_for_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


def test_nonzero_rank_of_reference_arm_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
