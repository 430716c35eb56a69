"""bench.py's CPU legs (not gpu): the reference arm prints the contract's JSON line, in both kinds, on the GPU arm's
config / metric / unit; the join queries' CPU samples run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


@pytest.mark.parametrize("force_port", [False, True])
def test_reference_arm_line(force_port):
    import bench
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libexec_ref.so"))
    line = _run({"CBGPU_BENCH_CPU": "port"} if force_port else {})
    assert line["impl"] == "reference"
    assert line["metric"] == "TPC-H SF100 Q1 rows/sec" and line["unit"] == "rows/s" and line["higher_is_better"] is True
    assert line["config"]["workload"] == bench.workload_name(100.0, 1)
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["value"] > 1e5
    cb = line["cpu_baseline"]
    assert cb["kind"] == ("reference" if have_ref and not force_port else "port")
    assert cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs(tmp_path):
    """result rows -> DIR/<query>.npy: float64, rows sorted, numeric text as its value, NULL as NaN (sorted last)"""
    import bench
    import numpy as np
    bench.dump_outputs(str(tmp_path), {"q1": [[82, 70, "3774200.00", None], [65, 70, "-0.05", 7], [65, 70, "-0.05", None]],
                                       "empty": []})
    q1 = np.load(tmp_path / "q1.npy")
    assert q1.dtype == np.float64
    np.testing.assert_array_equal(q1, [[65, 70, -0.05, 7], [65, 70, -0.05, np.nan], [82, 70, 3774200.0, np.nan]])
    assert np.load(tmp_path / "empty.npy").shape == (0, 0)


def test_join_cpu_samples():
    import bench
    out = bench.cpu_join_samples(sf=0.1)
    assert set(out) == {"q3", "q5"}
    for b in out.values():
        assert b["kind"] == "port" and b["cores"] == 1 and b["value"] > 1e5
