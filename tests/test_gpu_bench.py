"""bench.py on the device (-m gpu): --steps sets how many timed Q1 steps run (their kernel launches scale with it), and
--dump-outputs writes what the timed queries returned - the same arrays on every run with the same arguments, Q1's equal
to the independent numpy answers in tests/golden/bench_golden.json."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from cloudberry_b200 import bench_golden as BG

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SF = 10


def _bench(out, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--sf", str(SF), "--steps", str(steps),
                        "--warmup", "3", "--no-e2e", "--no-cpu", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


def test_steps_and_dumped_outputs(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    line = _bench(a, 2)
    assert line["result_check"] == "ok"
    assert line["steps"] == 2 and line["q3"]["steps"] == 2 and line["q5"]["steps"] == 2 and line["ssb"]["steps"] == 2
    names = sorted(os.listdir(a))
    assert names == sorted(["q1.npy", "q3.npy", "q5.npy", "ssb_q4_1.npy", "ssb_q4_2.npy", "ssb_q4_3.npy"])
    q1 = np.load(a / "q1.npy")
    want = [[ord(r[0]), ord(r[1])] + [float(x) for x in r[2:]] for r in BG.q1_rows(BG.load()[BG.key("q1", SF)], 1)]
    assert q1.dtype == np.float64 and np.array_equal(q1, np.array(want))
    assert np.load(a / "q3.npy").shape == (10, 4) and np.load(a / "q5.npy").shape == (5, 2)
    line3 = _bench(b, 3)
    # the launches counted over the timed Q1 loop: the same number per step, so 3 steps launch 3/2 as many as 2 steps
    assert line["gpu_launches"] > 0 and 2 * line3["gpu_launches"] == 3 * line["gpu_launches"]
    assert sorted(os.listdir(b)) == names
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == np.float64 and x.size and np.array_equal(x, y, equal_nan=True), n
