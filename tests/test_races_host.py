"""CPU: the race-after-race entry points (ftgp_reload / ftgp_tick_reload) are exported, reject bad arguments before any
CUDA call, and the tally rules of include/ftgp.h stated in numpy (used by tests/test_gpu_races.py as the replay) agree
with a hand-built race."""
import ctypes as C

import numpy as np
import pytest


def tally_np(lap, times, tally):
    """Add the race that ends now to tally (int32 [n, RACE_FIELDS]) for every car of lap / times (host copies taken at
    the head of the tick that reloads the world), as reload_kernel does."""
    from ft_grandprix_b200._lib import MAX_LAPTIMES
    from ft_grandprix_b200.fleet import LAP, RACE
    for i in range(len(lap)):
        s, t = lap[i], tally[i]
        stored = [int(v) for v in times[i, :min(int(s[LAP["ntimes"]]), MAX_LAPTIMES)]]
        t[RACE["races"]] += 1
        t[RACE["finished"]] += s[LAP["finished"]]
        t[RACE["wins"]] += int(s[LAP["rank"]] == 1)
        t[RACE["rank_sum"]] += s[LAP["rank"]]
        t[RACE["laps_sum"]] += s[LAP["laps"]]
        if s[LAP["finished"]]:
            t[RACE["time_sum"]] += sum(stored)
        best = [v for v in stored + [int(t[RACE["best_lap"]])] if v > 0]
        t[RACE["best_lap"]] = min(best) if best else 0
        t[RACE["offtrack_ticks"]] += s[LAP["offtrack_ticks"]]
        t[RACE["contact_ticks"]] += s[LAP["contact_ticks"]]
    return tally


def test_library_exports_the_reload_entry_points():
    from ft_grandprix_b200 import _lib
    lib = C.CDLL(_lib.LIB_PATH)
    assert hasattr(lib, "ftgp_reload") and hasattr(lib, "ftgp_tick_reload")
    assert _lib.load().ftgp_abi_version() == 3
    assert len(_lib.RACE_FIELDS) == 9 and _lib.RACE_FIELDS[0] == "races" and _lib.RACE_FIELDS[-1] == "contact_ticks"
    assert C.sizeof(_lib.ReloadArgs) == 5 * 8 + 2 * 4


def _args():
    """Tick arguments whose pointers are non-NULL but point nowhere: only the argument checks may look at them."""
    from ft_grandprix_b200 import _lib
    a = _lib.TickArgs()
    for name in ("geom", "qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "winners", "status"):
        setattr(a, name, 0x1000)
    a.ncars, a.cars_per_world = 8, 1
    r = _lib.ReloadArgs()
    r.start_xy, r.start_yaw, r.start_offset, r.race_start, r.tally = 0x1000, 0x1000, 0x1000, 0x1000, 0x1000
    r.race_ticks = 100
    return a, r


@pytest.mark.parametrize("bad", ["no_args", "qpos", "start_xy", "start_yaw", "start_offset", "negative_race_ticks",
                                 "tally_without_race_start", "race_ticks_without_race_start"])
def test_bad_reload_arguments_raise_before_any_cuda_call(bad):
    from ft_grandprix_b200 import _lib
    lib = _lib.load()
    a, r = _args()
    if bad == "qpos":
        a.qpos = None
    elif bad in ("start_xy", "start_yaw", "start_offset"):
        setattr(r, bad, None)
    elif bad == "negative_race_ticks":
        r.race_ticks = -1
    elif bad == "tally_without_race_start":
        r.race_start, r.race_ticks = None, 0
    elif bad == "race_ticks_without_race_start":
        r.race_start, r.tally = None, None
    rp = None if bad == "no_args" else C.byref(r)
    # FTGP_ERR_ARG (1), not FTGP_ERR_CUDA (2): nothing reached the device
    assert lib.ftgp_reload(C.byref(a), rp, None) == 1
    with pytest.raises(_lib.FtgpError, match="bad"):
        _lib.check(lib.ftgp_reload(C.byref(a), rp, None), "ftgp_reload")
    if bad != "no_args":                       # (r == NULL is a plain ftgp_tick)
        assert lib.ftgp_tick_reload(C.byref(a), rp, 1, None) == 1
        with pytest.raises(_lib.FtgpError, match="bad"):
            _lib.check(lib.ftgp_tick_reload(C.byref(a), rp, 1, None), "ftgp_tick_reload")


def test_tally_rules_on_a_hand_built_race():
    from ft_grandprix_b200._lib import LAP_FIELDS, MAX_LAPTIMES, RACE_FIELDS
    from ft_grandprix_b200.fleet import LAP, RACE
    lap = np.zeros((4, len(LAP_FIELDS)), dtype=np.int32)
    times = np.zeros((4, MAX_LAPTIMES), dtype=np.int32)
    # car 0: won with laps of 900 and 800 steps; car 1: 2nd, 20 laps (only 16 times are stored); car 2: did not finish,
    # one lap stored; car 3: did not finish, no lap, a lap time left past ntimes (a lap undone by reversing)
    lap[0, [LAP["finished"], LAP["rank"], LAP["laps"], LAP["ntimes"], LAP["offtrack_ticks"], LAP["contact_ticks"]]] = 1, 1, 2, 2, 5, 7
    times[0, :2] = 900, 800
    lap[1, [LAP["finished"], LAP["rank"], LAP["laps"], LAP["ntimes"]]] = 1, 2, 20, 20
    times[1] = np.arange(100, 100 + MAX_LAPTIMES)
    lap[2, [LAP["laps"], LAP["ntimes"], LAP["offtrack_ticks"]]] = 1, 1, 40
    times[2, 0] = 950
    lap[3, [LAP["laps"], LAP["ntimes"], LAP["contact_ticks"]]] = -1, 0, 3
    times[3, 0] = 10
    tally = np.zeros((4, len(RACE_FIELDS)), dtype=np.int32)
    tally[0, RACE["best_lap"]] = 700                  # from an earlier race
    tally[2, RACE["best_lap"]] = 1000
    tally_np(lap, times, tally)
    want = np.zeros_like(tally)
    want[:, RACE["races"]] = 1
    want[:, RACE["finished"]] = 1, 1, 0, 0
    want[:, RACE["wins"]] = 1, 0, 0, 0
    want[:, RACE["rank_sum"]] = 1, 2, 0, 0
    want[:, RACE["laps_sum"]] = 2, 20, 1, -1
    want[:, RACE["time_sum"]] = 1700, sum(range(100, 116)), 0, 0
    want[:, RACE["best_lap"]] = 700, 100, 950, 0
    want[:, RACE["offtrack_ticks"]] = 5, 0, 40, 0
    want[:, RACE["contact_ticks"]] = 7, 0, 0, 3
    np.testing.assert_array_equal(tally, want)
    tally_np(lap, times, tally)                       # a second, identical race
    np.testing.assert_array_equal(tally[:, RACE["races"]], 2)
    np.testing.assert_array_equal(tally[:, RACE["time_sum"]], 2 * want[:, RACE["time_sum"]])
    np.testing.assert_array_equal(tally[:, RACE["best_lap"]], want[:, RACE["best_lap"]])
