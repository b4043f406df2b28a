"""bench.py end to end at the tiny workload: --steps sets the number of timed solves and --dump-outputs writes the
last one's result.  Every step restores the same seeded start, so runs with 1 and 2 timed steps must write the same
solution (up to the summation order of the device reductions)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", str(steps), "--warmup", "1",
           "--e2e-steps", "1", "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, cwd=out_dir.parent, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_bench_dumps_the_last_timed_step(tmp_path):
    l1, d1 = _bench(tmp_path / "one", 1)
    l2, d2 = _bench(tmp_path / "two", 2)
    assert l1["steps"] == 1 and l2["steps"] == 2
    C, P = 200, 20_000
    shapes = {"quat": (C, 4), "trans": (C, 3), "points": (P, 3), "intr_params": (1, 12), "cost": (2,)}
    for d in (d1, d2):
        assert {k: v.shape for k, v in d.items()} == shapes
        assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in d.values())
    assert d1["cost"].tolist() == l1["config"]["cost"] and d2["cost"].tolist() == l2["config"]["cost"]
    assert d1["cost"][1] < d1["cost"][0]
    assert d1["cost"][0] == d2["cost"][0]                                   # identical seeded start
    assert abs(d1["cost"][1] - d2["cost"][1]) <= 1e-9 * d1["cost"][1]
    for k in ("quat", "trans", "points", "intr_params"):
        assert np.abs(d1[k] - d2[k]).max() < 1e-7, k
