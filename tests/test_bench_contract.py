"""bench.py's CPU arm (`--impl reference`) prints the contract's JSON line without a GPU; with a
GPU, `--dump-outputs` writes the state the timed steps computed."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "particle-steps/s" and line["unit"] == "particle-steps/s"
    assert line["higher_is_better"] is True and line["dtype"] == "f64" and line["vs_baseline"] is None
    assert line["value"] > 0 and line["steps"] >= 2
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "particles" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "particle-steps/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    import os
    env = dict(os.environ, RANK="3", WORLD_SIZE="8", LOCAL_RANK="3")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "8"],
                       capture_output=True, text=True, timeout=120, cwd=str(ROOT), env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_hold_the_state_after_the_timed_steps(gpu, tmp_path):
    """--dump-outputs on the 1 M workload: a sample of the particle state after warmup + steps
    steps, in global index order, equal to the CPU oracle stepped as often from the same lattice"""
    from sph_mountain_waves_b200 import cases
    from util import field_err, load_oracle
    warmup, steps = 1, 3
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "bell_hill_3d_1M",
                        "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline", "--no-e2e",
                        "--no-strict", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    files = sorted(tmp_path.glob("*.npy"))
    assert {f.stem for f in files} == {"index", "h", "x", "m", "v", "rho_p", "rho", "type"}
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    got = {f.stem: np.load(f) for f in files}
    assert all(a.dtype == np.float64 for a in got.values())
    idx = got.pop("index").astype(np.int64)
    case = cases.bell_hill_3d(480, 38, 48, lean=True)     # bench.py's WORKLOADS["bell_hill_3d_1M"]
    assert 0 < len(idx) < case.n and np.all(np.diff(idx) > 0)
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", warmup + steps)
    for f, a in got.items():
        assert len(a) == len(idx)
        assert field_err(case, f, a, o.field(f)[idx], nsteps=warmup + steps) <= 1e-10, f
