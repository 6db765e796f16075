"""bench.py contract checks that need no GPU: the reference arm (CPU oracle on the host cores) prints ONE JSON line
with the keys the driver reads, and the synthetic workload has the shape BASELINE.json names."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def test_workload_shape_is_baseline_config_2():
    txy, toff, rxy, roff, cen, U, n = bench.make_units(20261018, n_pairs=1)
    assert U == 398 and n == 520                       # 2 pullbacks x 199 frame pairs, 500 lumen + 20 catheter points
    assert bench.N_PAIRS == 8                          # the bench batch: the same 8 pullback pairs at every --gpus N
    assert txy.shape == (U * n, 2) and rxy.shape == (U * n, 2) and toff[-1] == U * n
    # units are centred on the frame (lumen) centroid, like align_within_many builds them
    assert abs(txy[:500].mean(axis=0)).max() < 1e-12
    assert bench.flops_per_eval(520, 520) == 10 * 520 * 520 + 6 * 520


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "36000" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == bench.WORKLOAD and d["scaling"] == "strong"
    # the reference arm's config is the GPU arm's (the driver compares them): the bounded sample lives in cpu_baseline
    assert d["config"]["units"] == 398 * bench.N_PAIRS and d["config"]["candidates_per_unit"] == 36000
    assert "sample" not in d["config"] and "1 of the 3184" in d["cpu_baseline"]["sample"]
    # ... key for key: both arms build it with the same function for the same N
    assert d["config"] == bench.base_config(398 * bench.N_PAIRS, 36000, bench.N_POINTS + bench.N_CATH, 1)
    assert "host threads" in d["cpu_baseline"]["parallelism"]
    # --dump-outputs: what the last timed step computed, unit 0 of the committed 1-GPU result
    g = np.load(bench.GOLDEN)
    idx, dist = np.load(tmp_path / "out" / "best_idx.npy"), np.load(tmp_path / "out" / "best_dist.npy")
    assert idx.dtype == dist.dtype == np.float64 and idx.shape == dist.shape == (1,)
    assert idx[0] == g["best_idx"][0] and dist[0] == g["best_dist"][0]
