"""GPU: bench.py prints ONE JSON line with the keys the driver reads (small fleets, a few steps)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _run(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().split("\n") if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"}


def test_tick_line_has_the_contract_keys():
    d = _run("--cars", "8192", "--steps", "3", "--warmup", "3", "--settle", "5")
    assert BASE <= set(d) and "cpu_baseline" in d
    assert d["metric"] == "car-steps/s" and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 1e5
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"]) and d["roofline"]["bound"] == "hbm"
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-12
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] >= 3 * 4 and "workload" in d["config"] and "model" not in d["config"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])


@pytest.mark.parametrize("wl,cars", [("lidar", "4096"), ("episode", "16384"), ("race", "8192")])
def test_other_workloads_print_a_line(wl, cars):
    d = _run("--workload", wl, "--cars", cars, "--steps", "3", "--warmup", "3", "--settle", "5", "--no-cpu-baseline")
    assert BASE <= set(d) and d["value"] > 0 and d["e2e"]["value"] > 0
    if wl in ("episode", "race"):
        assert d["scaling"] == "strong" and d["episode"]["stats_rows"] == int(cars)


@pytest.mark.parametrize("cars", [40960, 4096])
def test_dump_outputs_of_the_last_timed_tick(tmp_path, cars):
    """--dump-outputs writes the fleet arrays of the last timed tick (40,960 cars: a seeded sample of 32,768 of them; 4,096
    cars: all of them, the tick replayed as a CUDA graph), identical from run to run; 3 timed ticks after 5 settle ticks
    end where 1 timed tick after 7 settle ticks ends."""
    common = ("--cars", str(cars), "--warmup", "2", "--no-cpu-baseline", "--dump-outputs")
    d = _run("--steps", "3", "--settle", "5", *common, str(tmp_path / "a"))
    _run("--steps", "3", "--settle", "5", *common, str(tmp_path / "b"))
    _run("--steps", "1", "--settle", "7", *common, str(tmp_path / "c"))
    assert d["steps"] == 3
    names = {"qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "winners", "status"}
    assert set(os.listdir(tmp_path / "a")) == {n + ".npy" for n in names}
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    for n in names:
        a, b, c = (np.load(tmp_path / r / (n + ".npy")) for r in "abc")
        assert a.dtype == (np.float32 if n == "ranges" else np.float64) and len(a) == min(cars, 32768), n
        assert np.array_equal(a, b) and np.array_equal(a, c), n
    assert np.isfinite(np.load(tmp_path / "a" / "qpos.npy")).all()


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
