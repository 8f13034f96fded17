"""GPU: per-car driver parameter rows in drivers_kernel and the fused tick (ftgp_drivers_params, ftgp_tick_params,
Fleet.set_driver_params).  The kernel equals the reference restatement on random rows; the reference rows are bit-identical to no rows,
at kernel level and through every tick; with random rows every way of issuing the tick agrees; rows rewritten in place
take effect on the next replayed tick; the sweep tool's smoke mode is deterministic."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from test_driver_params_host import _random_rows, _random_scans, driver_params_ref

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STATE = ("qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "status", "winners")
RACE_STATE = ("race_tally", "race_start")


@pytest.fixture(scope="module")
def ft():
    import ft_grandprix_b200 as ft
    return ft


def _poses(t, n, seed):
    from conftest import random_poses
    p = random_poses(t.path, n, seed=seed, level=True)
    return p[:, :2].copy(), 2 * np.arctan2(p[:, 6], p[:, 3])


def _kind_rows(ft, kinds):
    from ft_grandprix_b200.fleet import default_driver_params
    return np.array([default_driver_params(min(int(k), 1)) for k in kinds])


def _drive_rows(ft, rows):
    """Rows a car can race with: the reference rows jittered by up to 30 % in the tunable fields."""
    from ft_grandprix_b200.fleet import DRV
    rng = np.random.default_rng(len(rows))
    out = rows.copy()
    for name in ("car_width", "safety_percentage", "difference_threshold", "speed", "speed_divisor", "boost_speed"):
        out[:, DRV[name]] *= rng.uniform(0.7, 1.3, len(rows))
    return out


def test_kernel_matches_the_reference_with_random_rows(ft):
    """4,096 seeded fp32 scans + the golden scans, one random row per car, kinds nidc / fast / lobotomy mixed, every 7th
    car finished: lobotomy and finished cars drive (0, 0), the others equal driver_params_ref; a car that raises keeps
    its pre-filled ctrl of 99."""
    scans = np.concatenate([np.load(os.path.join(GOLDEN, "drivers.npz"))["scans"], _random_scans(4096, 21)])
    scans32 = scans.astype(np.float32)
    n = len(scans32)
    rows = _random_rows(n, 22)
    rows[::97, ft.fleet.DRV["car_width"]] = np.nan                   # some cars raise at their first disparity
    kinds = np.arange(n) % 3
    t = ft.Track.bundled("small-circle")
    f = ft.Fleet(t, n)
    f.set_driver_kinds(kinds.tolist())
    f.set_driver_params(rows)
    finished = np.arange(n) % 7 == 3
    f.lap[:, ft.fleet.LAP["finished"]] = torch.as_tensor(finished.astype(np.int32), device=f.device)
    f.ranges.copy_(torch.from_numpy(scans32))
    f.ctrl.fill_(99.0)
    torch.cuda.synchronize()
    f.drive(); f.sync()
    got = f.ctrl.cpu().numpy()
    raised = 0
    for i in range(n):
        if finished[i] or kinds[i] == 2:
            want = (0.0, 0.0)
        else:
            want = driver_params_ref(rows[i], scans32[i].astype(np.float64))
            if want is None:
                want, raised = (99.0, 99.0), raised + 1
        np.testing.assert_allclose(got[i], want, rtol=0, atol=1e-12, err_msg=str(i))
    assert raised > 0


def test_reference_rows_equal_no_rows_at_kernel_level(ft):
    """65,536 seeded fp32 scans, nidc / fast mixed: the reference row of each car's kind is bit-identical to no rows."""
    n = 65536
    scans32 = _random_scans(n, 23).astype(np.float32)
    kinds = np.arange(n) % 2
    t = ft.Track.bundled("small-circle")
    out = []
    for rows in (None, _kind_rows(ft, kinds)):
        f = ft.Fleet(t, n)
        f.set_driver_kinds(kinds.tolist())
        f.set_driver_params(rows)
        f.ranges.copy_(torch.from_numpy(scans32))
        f.ctrl.fill_(99.0)
        torch.cuda.synchronize()
        f.drive(); f.sync()
        out.append(f.ctrl.clone())
    assert torch.equal(out[0], out[1])


@pytest.mark.parametrize("n,cpw", [(4096, 1), (4096, 8), (20480, 1), (20480, 8)])
def test_reference_rows_equal_no_rows_through_the_tick(ft, n, cpw):
    """300 fused ticks (graph-replayed at 4,096 cars, eager at 20,480) with reload_finished and race_ticks 120, nidc /
    fast mixed: every state tensor is bit-identical with the reference rows and without rows."""
    t = ft.Track.bundled("small-circle")
    kinds = np.arange(n) % 2
    fleets = []
    for rows in (None, _kind_rows(ft, kinds)):
        f = ft.Fleet(t, n, cars_per_world=cpw, lap_target=1, reload_finished=True, race_ticks=120)
        if cpw == 1:
            f.reset(*_poses(t, n, 61))
        else:
            f.reset_grid()
        f.set_driver_kinds(kinds.tolist())
        f.set_driver_params(rows)
        fleets.append(f)
    for _ in range(300):
        for f in fleets:
            f.tick(1)
    A, B = fleets
    A.sync(); B.sync()
    for k in STATE + RACE_STATE:
        assert torch.equal(getattr(A, k), getattr(B, k)), k
    assert (A.race_tally[:, ft.fleet.RACE["races"]] >= 2).all()


@pytest.mark.parametrize("cpw", [1, 8])
def test_every_way_of_issuing_the_tick_agrees_with_random_rows(ft, cpw):
    """64 cars, random drivable rows, reload_finished with race_ticks 80: tick(1) replayed, tick(200), eager, tick_readback
    and the separate calls reload -> lap_update -> drive -> lidar -> step are bit-identical after 200 ticks."""
    t = ft.Track.bundled("small-circle")
    n = 64
    kinds = np.arange(n) % 2
    rows = _drive_rows(ft, _kind_rows(ft, kinds))
    ranges_h = torch.empty(n, 90, dtype=torch.float32).pin_memory()
    lap_h = torch.empty(n, len(ft.fleet.LAP), dtype=torch.int32).pin_memory()

    def run(kind):
        f = ft.Fleet(t, n, cars_per_world=cpw, reload_finished=True, race_ticks=80)
        if cpw == 1:
            f.reset(*_poses(t, n, 62))
        else:
            f.reset_grid()
        f.set_driver_params(rows)
        if kind == "graph":
            for _ in range(200):
                f.tick(1)
        elif kind == "tick200":
            f.tick(200)
        elif kind == "eager":
            prev = f.lib.ftgp_tick_use_graphs(0)
            try:
                for _ in range(200):
                    f.tick(1)
            finally:
                f.lib.ftgp_tick_use_graphs(prev)
        elif kind == "readback":
            for _ in range(200):
                f.tick_readback(ranges_h, lap_h)
            f.sync_readback()
        else:
            for _ in range(200):
                f.reload(); f.lap_update(); f.drive(); f.lidar(); f.step(1)
        f.sync()
        return {k: getattr(f, k).clone() for k in STATE + RACE_STATE}

    ref = run("graph")
    for kind in ("tick200", "eager", "readback", "separate"):
        got = run(kind)
        for k in ref:
            assert torch.equal(ref[k], got[k]), (kind, k)
    # the rows drive differently from the reference constants
    f = ft.Fleet(t, n, cars_per_world=cpw, reload_finished=True, race_ticks=80)
    f.reset(*_poses(t, n, 62)) if cpw == 1 else f.reset_grid()
    f.set_driver_kinds(kinds.tolist())
    f.tick(200); f.sync()
    assert not torch.equal(f.qpos, ref["qpos"])


@pytest.mark.parametrize("cpw", [1, 8])
def test_rows_rewritten_in_place_take_effect_on_the_next_replayed_tick(ft, cpw):
    """Rows R1 for 100 replayed ticks, then R2 written into fleet.driver_params (same storage) and 100 more: equal to a
    fleet loaded from the tick-100 state_dict with R2.  set_driver_params(None) at tick 100 equals a fleet that never
    had rows."""
    t = ft.Track.bundled("small-circle")
    n = 64
    kinds = np.arange(n) % 2
    r1 = _drive_rows(ft, _kind_rows(ft, kinds))
    r2 = _drive_rows(ft, _kind_rows(ft, kinds[::-1].copy()))

    def fleet():
        f = ft.Fleet(t, n, cars_per_world=cpw, reload_finished=True, race_ticks=80)
        f.reset(*_poses(t, n, 63)) if cpw == 1 else f.reset_grid()
        f.set_driver_kinds(kinds.tolist())
        return f

    for new in (r2, None):
        A = fleet()
        A.set_driver_params(r1)
        ptr = A.driver_params.data_ptr()
        for _ in range(100):
            A.tick(1)
        sd = A.state_dict()
        assert torch.equal(sd["driver_params"], torch.from_numpy(r1))
        if new is None:
            A.set_driver_params(None)
            del sd["driver_params"]
        else:
            with torch.cuda.stream(A.stream):          # in place, in stream order
                A.driver_params.copy_(torch.from_numpy(new).to(A.device))
            assert A.driver_params.data_ptr() == ptr
            sd["driver_params"] = torch.from_numpy(new)
        for _ in range(100):
            A.tick(1)
        B = fleet()
        B.load_state_dict(sd)
        assert (B.driver_params is None) == (new is None)
        for _ in range(100):
            B.tick(1)
        A.sync(); B.sync()
        for k in STATE + RACE_STATE:
            assert torch.equal(getattr(A, k), getattr(B, k)), (k, new is None)


def test_sweep_tool_smoke_is_deterministic(tmp_path):
    """tools/driver_sweep.py --smoke (1,024 cars, 8 variants) twice: identical tallies, and the variants differ."""
    outs = []
    for k in range(2):
        out = tmp_path / f"sweep{k}.json"
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "driver_sweep.py"), "--smoke", "--out", str(out)],
                       check=True, cwd=str(tmp_path), timeout=900)
        lines = [json.loads(x) for x in out.read_text().splitlines()]
        gens = [d for d in lines if d["measure"] == "generation"]
        assert len(gens) == 1 and gens[0]["cars"] == 1024 and "nvidia_smi" in gens[0]
        outs.append(np.array(gens[0]["tally_by_variant"]))
    assert np.array_equal(outs[0], outs[1])
    from ft_grandprix_b200.fleet import RACE
    assert outs[0][:, RACE["races"]].min() >= 1
    assert len({tuple(r) for r in outs[0].tolist()}) > 1
