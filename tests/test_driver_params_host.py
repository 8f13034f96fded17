"""CPU: per-car driver parameter rows (include/ftgp.h FTGP_DRV_*).  A statement-by-statement restatement of the reference
drivers with the constants taken from a row (driver_params_ref, also the GPU tests' reference) reproduces the reference
classes and fto_driver with the reference rows; the torch twin (BatchedNidcDriver(params=...)) equals it on random and
out-of-range rows, a hand-checkable gap moves the chosen beam by the covered count, and the new entry points
are exported and reject bad arguments before any CUDA call."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from conftest import GOLDEN

torch = pytest.importorskip("torch")
RPP = (2 * math.pi) / 90


def _golden_scans():
    return np.load(os.path.join(GOLDEN, "drivers.npz"))["scans"]


def _random_scans(n, seed):
    """Seeded scans with misses (-1), zeros, ties (a beam copied from its neighbour) and NaN."""
    rng = np.random.default_rng(seed)
    s = rng.uniform(0.05, 6.0, (n, 90))
    s[rng.random((n, 90)) < 0.05] = -1.0
    s[rng.random((n, 90)) < 0.03] = 0.0
    tie = rng.random((n, 90)) < 0.1
    tie[:, 0] = False
    s[tie] = np.roll(s, 1, axis=1)[tie]
    s[rng.random((n, 90)) < 0.002] = np.nan
    return s


def _random_rows(n, seed):
    from ft_grandprix_b200.fleet import DRV
    rng = np.random.default_rng(seed)
    rows = np.empty((n, len(DRV)))
    rows[:, DRV["car_width"]] = rng.uniform(0.0, 0.5, n)
    rows[:, DRV["safety_percentage"]] = rng.uniform(0.0, 500.0, n)
    rows[:, DRV["difference_threshold"]] = rng.uniform(0.05, 2.0, n)
    rows[:, DRV["speed"]] = rng.uniform(0.1, 2.0, n)
    rows[:, DRV["speed_divisor"]] = rng.uniform(1.0, 5.0, n)
    rows[:, DRV["max_steer"]] = rng.uniform(0.2, 2.0, n)
    rows[:, DRV["boost_speed"]] = rng.uniform(1.0, 10.0, n)
    rows[:, DRV["boost_max_steer"]] = rng.uniform(0.0, 0.5, n)
    rows[:, DRV["boost_min_rear_range"]] = rng.uniform(0.0, 2.0, n)
    rows[:, DRV["speed_cap"]] = np.where(rng.random(n) < 0.25, np.inf, rng.uniform(0.5, 10.0, n))
    return rows


def _edge_rows():
    from ft_grandprix_b200.fleet import DRV, default_driver_params
    base = default_driver_params("fast")
    out = []
    for field, values in (("car_width", (0.0, -0.3, np.nan, 1e300, np.inf)),
                          ("difference_threshold", (-1.0, np.inf)),
                          ("speed_cap", (1.0,))):                   # a cap below the boost speed (7)
        for v in values:
            r = base.copy()
            r[DRV[field]] = v
            out.append(r)
    return np.array(out)


def driver_params_ref(row, scan, margins=None):
    """process_lidar of nidc.py / fast.py with the constants taken from `row` (include/ftgp.h FTGP_DRV_*), statement by
    statement in float64 scalars (numpy's, so that x / 0 gives inf or nan as it does in the reference).  Returns
    (speed, steer), or None where the reference raises (int(np.ceil(nan)), custom.py:1409-1411).  margins: a list that
    receives |angle / rpp - round(angle / rpp)| of every disparity visited."""
    from ft_grandprix_b200.fleet import DRV
    r = {name: np.float64(row[k]) for name, k in DRV.items()}
    proc = [np.float64(v) for v in scan[11:79]]                  # nidc.py:17-18
    m = len(proc)
    with np.errstate(all="ignore"):
        disp = [i for i in range(1, m) if abs(proc[i] - proc[i - 1]) > r["difference_threshold"]]    # nidc.py:26-40
        width = (r["car_width"] / 2) * (1 + r["safety_percentage"] / 100)                             # nidc.py:93
        for i in disp:                                                                                 # nidc.py:94-104
            a, b = proc[i - 1], proc[i]
            amin = 0 if np.isnan(a) else (1 if np.isnan(b) else int(b < a))
            amax = 0 if np.isnan(a) else (1 if np.isnan(b) else int(b > a))
            close, far = i - 1 + amin, i - 1 + amax
            dist = proc[close]
            q = 2 * np.float64(math.atan(width / (2 * dist))) / RPP                                   # nidc.py:57
            if margins is not None and not np.isnan(q):
                margins.append(abs(q - np.round(q)))
            try:
                num = int(math.ceil(q))                                                                # nidc.py:58
            except ValueError:
                return None
            cover = range(close + 1, min(close + 1 + num, m)) if close < far else range(close - 1, max(close - 1 - num, -1), -1)
            for j in cover:                                                                            # nidc.py:71-84
                if proc[j] > dist:
                    proc[j] = dist
        best = 0                                                  # np.argmax: first maximum, first NaN wins
        if not np.isnan(proc[0]):
            for j in range(1, m):
                if np.isnan(proc[j]):
                    best = j
                    break
                if proc[j] > proc[best]:
                    best = j
        ang = (best - m / 2.0) * RPP                                                                   # nidc.py:112
        lim = r["max_steer"]                                                                           # nidc.py:113
        st = -lim if ang < -lim else (lim if ang > lim else np.float64(ang))
        if abs(st) < r["boost_max_steer"] and np.float64(scan[0]) > r["boost_min_rear_range"]:        # fast.py:135-136
            return float(r["boost_speed"]), float(st)
        sp = r["speed"] * 5 * (1 - abs(st) / r["speed_divisor"])                                       # nidc.py:130, fast.py:138
        return float(sp if sp < r["speed_cap"] else r["speed_cap"]), float(st)


def _ref(row, scan):
    got = driver_params_ref(row, scan)
    return (np.nan, np.nan, True) if got is None else (got[0], got[1], False)


def _twin(rows, scans):
    from ft_grandprix_b200 import BatchedNidcDriver
    d = BatchedNidcDriver(params=torch.from_numpy(np.ascontiguousarray(rows)))
    sp, st = d.process_lidar(torch.from_numpy(np.ascontiguousarray(scans)))
    raised = d.raised.numpy()
    return np.where(raised, np.nan, sp.numpy()), np.where(raised, np.nan, st.numpy()), raised


def _ceil_margin(row, scan):
    margins = []
    driver_params_ref(row, scan, margins)
    return min(margins, default=np.inf)


def _compare(rows, scans, capsys, what):
    """Reference == twin for every (row, scan); a difference must sit on a ceil knife edge."""
    R = np.repeat(rows, len(scans), axis=0)
    S = np.tile(scans, (len(rows), 1))
    tsp, tst, traised = _twin(R, S)
    want = np.array([_ref(r, s) for r, s in zip(R, S)])
    osp, ost, oraised = want[:, 0], want[:, 1], want[:, 2].astype(bool)
    diff = (oraised != traised) | ~((osp == tsp) | (np.isnan(osp) & np.isnan(tsp))) | \
        ~((ost == tst) | (np.isnan(ost) & np.isnan(tst)))
    for k in np.nonzero(diff)[0]:
        assert _ceil_margin(R[k], S[k]) < 1e-12, (what, k, R[k], osp[k], tsp[k], ost[k], tst[k])
    with capsys.disabled():
        print(f"\n[report] {what}: {len(R)} (row, scan) pairs, {int(oraised.sum())} raised, "
              f"{int(diff.sum())} differ (all on a ceil knife edge)")
    return diff.sum()


def test_default_rows_reproduce_the_reference_classes_and_fto_driver(oracle):
    """The reference rows give the answers of ft_grandprix.nidc / fast on the 403 golden scans, and of fto_driver, bit for
    bit: the formula with a row is the two drivers."""
    from ft_grandprix_b200.fleet import default_driver_params
    z = np.load(os.path.join(GOLDEN, "drivers.npz"))
    for kind, name in ((0, "nidc"), (1, "fast")):
        row = default_driver_params(name)
        for s, want in zip(z["scans"], z[name]):
            got = driver_params_ref(row, s)
            assert got == (want[0], want[1]) == oracle.driver(kind, s), (name, got, want)


def test_default_rows_are_the_reference_constants():
    from ft_grandprix_b200.fleet import DRV, default_driver_params
    nidc, fast = default_driver_params("nidc"), default_driver_params("fast")
    assert nidc[DRV["car_width"]] == 0.12 and fast[DRV["car_width"]] == 0.06
    assert nidc[DRV["speed_divisor"]] == 1.57 * 2 and fast[DRV["speed_divisor"]] == 3.141592653589793
    assert nidc[DRV["max_steer"]] == fast[DRV["max_steer"]] == 90.0 * (3.141592653589793 / 180.0)
    assert nidc[DRV["boost_max_steer"]] == 0 and fast[DRV["boost_max_steer"]] == 0.1
    assert nidc[DRV["speed_cap"]] == np.inf and fast[DRV["speed_cap"]] == 2
    with pytest.raises(ValueError):
        default_driver_params("lobotomy")


def test_twin_equals_reference_on_random_rows(capsys):
    scans = np.concatenate([_golden_scans(), _random_scans(2000, 5)])
    _compare(_random_rows(64, 11), scans, capsys, "64 random rows x (403 golden + 2,000 seeded scans)")


def test_twin_equals_reference_on_edge_rows(capsys):
    from ft_grandprix_b200.fleet import DRV
    scans = np.concatenate([_golden_scans(), _random_scans(500, 6)])
    rows = _edge_rows()
    _compare(rows, scans, capsys, f"{len(rows)} edge rows x {len(scans)} scans")
    # what the header promises: a NaN width raises at the first disparity; width 0 or negative covers nothing (the
    # steering is the plain argmax); a negative threshold makes every index a disparity; inf none
    s = np.full(90, 2.0); s[50:60] = 6.0
    row = _edge_rows()[2]
    assert np.isnan(row[DRV["car_width"]]) and driver_params_ref(row, s) is None
    for row in _edge_rows()[:2]:
        assert driver_params_ref(row, s)[1] == (50 - 11 - 34) * RPP
    inf_thr = _edge_rows()[6]
    assert inf_thr[DRV["difference_threshold"]] == np.inf and driver_params_ref(inf_thr, s)[1] == (50 - 11 - 34) * RPP
    cap = _edge_rows()[7]
    sp, st = driver_params_ref(cap, np.full(90, 2.0))
    assert abs(st) >= 0.1 and sp == 1.0                              # the cap applies to the law, not to the boost
    z = np.full(90, 2.0); z[11 + 33:11 + 42] = 6.0                      # a gap straight ahead
    sp, st = driver_params_ref(cap, z)
    assert abs(st) < 0.1 and sp == 7.0


@pytest.mark.parametrize("car_width", [0.05, 0.1, 0.2, 0.4, 1.0, 1.6])
def test_one_gap_moves_the_chosen_beam_by_the_covered_count(car_width):
    """proc = 1 m up to index 39, 5 m from 40: the disparity at 40 covers ceil(2 atan(w / 2) / rpp) beams right of 39,
    so the first 5 m beam -- the one argmax picks -- is 40 + that count (safety 0: w = car_width / 2, no clipping)."""
    from ft_grandprix_b200.fleet import DRV, default_driver_params
    row = default_driver_params("nidc")
    row[DRV["car_width"]], row[DRV["safety_percentage"]], row[DRV["max_steer"]] = car_width, 0.0, 10.0
    scan = np.full(90, 1.0); scan[11 + 40:] = 5.0
    num = math.ceil(2 * math.atan((car_width / 2) / 2) / RPP)
    assert 1 <= num <= 20
    want = (40 + num - 34) * RPP
    assert driver_params_ref(row, scan)[1] == want
    _, st, raised = _twin(row[None], scan[None])
    assert not raised[0] and st[0] == want


def test_library_exports_the_parameter_entry_points():
    from ft_grandprix_b200 import _lib
    lib = C.CDLL(_lib.LIB_PATH)
    assert hasattr(lib, "ftgp_drivers_params") and hasattr(lib, "ftgp_tick_params")
    assert _lib.load().ftgp_abi_version() == 3
    assert len(_lib.DRV_FIELDS) == 10 and _lib.DRV_FIELDS[0] == "car_width" and _lib.DRV_FIELDS[-1] == "speed_cap"


@pytest.mark.parametrize("bad", ["ranges", "ctrl", "ncars", "kind_low", "kind_high"])
def test_bad_driver_arguments_raise_before_any_cuda_call(bad):
    from ft_grandprix_b200 import _lib
    lib = _lib.load()
    ranges, ctrl, params, ncars, kind = 0x1000, 0x1000, 0x1000, 8, 0
    if bad == "ranges":
        ranges = None
    elif bad == "ctrl":
        ctrl = None
    elif bad == "ncars":
        ncars = -1
    else:
        kind = -1 if bad == "kind_low" else 3
    rc = lib.ftgp_drivers_params(ranges, None, kind, params, None, ctrl, ncars, None)
    assert rc == 1                                   # FTGP_ERR_ARG, not FTGP_ERR_CUDA: nothing reached the device
    with pytest.raises(_lib.FtgpError, match="bad"):
        _lib.check(rc, "ftgp_drivers_params")


@pytest.mark.parametrize("bad", ["no_args", "qpos", "ncars", "start_xy", "negative_race_ticks", "nticks"])
def test_bad_tick_arguments_raise_before_any_cuda_call(bad):
    from ft_grandprix_b200 import _lib
    from test_races_host import _args
    lib = _lib.load()
    a, r = _args()
    nticks = 1
    if bad == "qpos":
        a.qpos = None
    elif bad == "ncars":
        a.ncars = -1
    elif bad == "start_xy":
        r.start_xy = None
    elif bad == "negative_race_ticks":
        r.race_ticks = -1
    elif bad == "nticks":
        nticks = -1
    ap = None if bad == "no_args" else C.byref(a)
    rc = lib.ftgp_tick_params(ap, C.byref(r), 0x1000, nticks, None)
    assert rc == 1
    with pytest.raises(_lib.FtgpError, match="bad"):
        _lib.check(rc, "ftgp_tick_params")
