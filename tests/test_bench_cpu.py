"""Host logic of bench.py that does not need a GPU: the clock sampler's handling of nvidia-smi rows (the timed region of
the default run is ~150 ms, shorter than nvidia-smi's start-up, so the rows carry timestamps and are filtered to it) and
its graceful behaviour without NVML / nvidia-smi; the --dump-outputs writer and the argument checks."""
import datetime
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    sys.modules["bench_under_test"] = m
    spec.loader.exec_module(m)
    return m


def test_smi_rows_are_filtered_to_the_timed_region():
    B = _bench()
    rows = ["2026/09/23 05:00:00.100, 1965, 1965, 600.1, Not Active, Not Active, Not Active, Active",
            "2026/09/23 05:00:00.150, 1920, 1965, 900.1, Not Active, Not Active, Not Active, Not Active",
            "2026/09/23 05:00:00.210, 1410, 1965, 990.0, Active, Not Active, Not Active, Not Active",
            "[N/A], x, y", "garbage"]
    t0 = datetime.datetime(2026, 9, 23, 5, 0, 0, 120000)
    t1 = datetime.datetime(2026, 9, 23, 5, 0, 0, 200000)
    sm, mx, reasons = B.ClockSampler.parse_smi(rows, t0, t1)
    assert sm == [1920.0] and mx == [1965.0] and reasons == set()
    sm, mx, reasons = B.ClockSampler.parse_smi(rows, None, None)
    assert sm == [1965.0, 1920.0, 1410.0] and reasons == {"sw_power_cap", "hw_slowdown"}


def test_sampler_without_a_gpu_reports_no_samples_instead_of_failing():
    B = _bench()
    s = B.ClockSampler(0)
    s.start()
    s.mark_begin()
    out = s.stop()
    assert out["samples"] == 0 or out["sm_mhz"] is not None
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"}


def test_dump_outputs_writes_float64_and_refuses_more_than_the_limit(tmp_path):
    B = _bench()
    B.dump_outputs(str(tmp_path / "out"), {"points": np.arange(6, dtype=np.float32).reshape(2, 3), "cost": [2.0, 1.0]})
    pts, cost = np.load(tmp_path / "out" / "points.npy"), np.load(tmp_path / "out" / "cost.npy")
    assert pts.dtype == np.float64 and pts.shape == (2, 3) and pts[1, 2] == 5.0
    assert cost.dtype == np.float64 and cost.tolist() == [2.0, 1.0]
    with pytest.raises(SystemExit):
        B.dump_outputs(str(tmp_path / "big"), {"points": np.zeros(B.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not (tmp_path / "big").exists()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 2 and "error" in r.stderr, r.stderr
    assert not (tmp_path / "x").exists()
