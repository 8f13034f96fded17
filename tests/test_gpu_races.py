"""GPU: race after race on the device (Fleet(reload_finished=True), ftgp_tick_reload / ftgp_reload).  A reloaded world
is bit-identical to a freshly reset fleet (lap START taken relative to the world's race_start), worlds that are not due
are never written, every way of issuing the tick agrees, and the race tallies equal a numpy replay."""
import numpy as np
import pytest

from test_races_host import tally_np

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STATE = ("qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "status", "winners")


@pytest.fixture(scope="module")
def ft():
    import ft_grandprix_b200 as ft
    return ft


def _poses(t, n, seed):
    from conftest import random_poses
    p = random_poses(t.path, n, seed=seed, level=True)
    return p[:, :2].copy(), 2 * np.arctan2(p[:, 6], p[:, 3])


def _lap_rel(f, L):
    """The lap state with START counted from the world's race start (the only lap field a reload leaves absolute)."""
    lap = f.lap.clone()
    if f.reload_finished:
        lap[:, L["start"]] -= f.race_start.repeat_interleave(f.cars_per_world)
    return lap


def _assert_same(a, b, L, what):
    for k in STATE:
        x, y = (_lap_rel(a, L), _lap_rel(b, L)) if k == "lap" else (getattr(a, k), getattr(b, k))
        assert torch.equal(x, y), (k, what)


def _series_against_fresh(ft, t, n, cpw, starts, race_ticks, reset):
    """Fleet A races len(starts) races of race_ticks ticks back to back (the cap ends them); before each race a fresh
    fleet F is reset to that race's start, and after every tick A's state equals F's."""
    L, R = ft.fleet.LAP, ft.fleet.RACE
    A = ft.Fleet(t, n, cars_per_world=cpw, reload_finished=True, race_ticks=race_ticks)
    F = ft.Fleet(t, n, cars_per_world=cpw)
    contact_ticks = 0
    for race, start in enumerate(starts):
        if race == 0:
            reset(A, start)
        elif start is not None:                    # (None: the default next start, the poses of the last reset)
            A.set_next_start(*start)               # read by the reload at the head of A's next tick
        reset(F, start)
        for k in range(1, race_ticks + 1):
            A.tick(1); F.tick(1)
            A.sync(); F.sync()
            _assert_same(A, F, L, (race, k))
            contact_ticks += int(((A.status >> 9) & 1).any())
        assert (A.race_start == race * race_ticks).all()
    assert A.steps == len(starts) * race_ticks
    assert (A.race_tally[:, R["races"]] == len(starts) - 1).all()
    return A, contact_ticks


def test_reload_on_the_race_cap_equals_a_fresh_race(ft):
    """256 one-car worlds on track.png, race_ticks = 150, 450 ticks: at every tick 150 + k and 300 + k every car equals a
    fresh fleet reset to the same starts after k ticks, bit for bit (the second race starts from other poses)."""
    t = ft.Track.bundled("track")
    n = 256
    p1, p2 = _poses(t, n, 31), _poses(t, n, 32)
    A, _ = _series_against_fresh(ft, t, n, 1, [p1, p2, p1], 150, lambda f, s: f.reset(*s))
    assert (A.race_tally[:, ft.fleet.RACE["finished"]] == 0).all()


def test_reload_of_coupled_worlds_equals_a_fresh_race(ft, capsys):
    """4 worlds of 8 cars from the start grid (cars that touch are solved together), race_ticks = 150, 450 ticks."""
    t = ft.Track.bundled("track")
    A, contact_ticks = _series_against_fresh(ft, t, 32, 8, [None, None, None], 150, lambda f, s: f.reset_grid())
    with capsys.disabled():
        print(f"\n[report] 4 x 8 cars from the grid, 3 races of 150 ticks: {contact_ticks} of 450 ticks had car-car "
              "contacts (status bit 9)")


def _near_finish(ft, t, n, **kw):
    """As test_gpu_step.py: car i at path[k_i] two centreline points before its finish line (offset k_i + 2,
    completion 98), so it finishes within a few hundred ticks."""
    fleet = ft.Fleet(t, n, **kw)
    ks = (np.arange(n) * 4) % 100
    xy = t.path[ks]
    nxt = (ks + 1) % 100
    yaw = np.arctan2(t.path[nxt, 1] - xy[:, 1], t.path[nxt, 0] - xy[:, 0])
    fleet.reset(xy, yaw)
    L = ft.fleet.LAP
    fleet.lap[:, L["offset"]] = torch.as_tensor((ks + 2) % 100, dtype=torch.int32, device=fleet.device)
    fleet.lap[:, L["completion"]] = 98
    torch.cuda.synchronize()
    return fleet, ks


def _elsewhere(t, ks, shift=50, togo=10):
    """Next starts at path[k + shift] with the finish line `togo` centreline points ahead."""
    k2 = (ks + shift) % 100
    xy = t.path[k2]
    nxt = (k2 + 1) % 100
    yaw = np.arctan2(t.path[nxt, 1] - xy[:, 1], t.path[nxt, 0] - xy[:, 0])
    return xy, yaw, (k2 - (100 - togo)) % 100


def test_finished_worlds_reload_on_the_next_tick_with_the_replayed_tally(ft, capsys):
    """One-car worlds near their finish line, lap_target 1, no cap: each world reloads at the head of the tick after its
    car finished, from the next starts elsewhere on the track, and race_tally equals the numpy replay of the host
    copies of lap / times taken before each tick, integer for integer."""
    L, R = ft.fleet.LAP, ft.fleet.RACE
    t = ft.Track.bundled("small-circle")
    n = 25
    A, ks = _near_finish(ft, t, n, lap_target=1, reload_finished=True)
    xy2, yaw2, off2 = _elsewhere(t, ks)
    A.set_next_start(xy2, yaw2, off2)
    tally = np.zeros((n, len(R)), dtype=np.int32)
    races = np.zeros(n, dtype=np.int64)
    for step in range(1400):
        lap0, times0 = A.lap.cpu().numpy(), A.times.cpu().numpy()
        rs0 = A.race_start.cpu().numpy()
        due = lap0[:, L["finished"]] == 1
        A.tick(1); A.sync()
        idx = np.nonzero(due)[0]
        sub = tally[idx]
        tally_np(lap0[idx], times0[idx], sub)
        tally[idx] = sub
        races += due
        np.testing.assert_array_equal(A.race_start.cpu().numpy(), np.where(due, step, rs0))
        np.testing.assert_array_equal(A.race_tally.cpu().numpy(), tally, err_msg=f"tick {step}")
        if due.any():
            lap = A.lap.cpu().numpy()
            assert (lap[due, L["start"]] == step).all() and (lap[due, L["offset"]] == off2[due]).all()
            assert (lap[due, L["finished"]] == 0).all() and (A.winners.cpu().numpy()[due] == 0).all()
    assert (races >= 1).sum() >= n // 3, races
    assert tally[:, R["wins"]].sum() == tally[:, R["finished"]].sum() > 0      # one-car worlds: every finisher won
    with capsys.disabled():
        print(f"\n[report] {n} one-car worlds near the finish, 1400 ticks: races ended per world {np.bincount(races).tolist()} "
              f"(index = races); best laps {sorted(set(tally[:, R['best_lap']].tolist()))}")


def test_worlds_of_8_with_some_cars_finished_are_untouched(ft):
    """8-car worlds where half the cars finish and the others are far from their line: no world is due, and every array
    is bit-identical to the same fleet with the option off."""
    L = ft.fleet.LAP
    t = ft.Track.bundled("small-circle")
    n, cpw = 32, 8
    slot = np.arange(n) % cpw
    ks = ((np.arange(n) // cpw) * 3 + slot * 12) % 100
    nxt = (ks + 1) % 100
    xy = t.path[ks]
    yaw = np.arctan2(t.path[nxt, 1] - xy[:, 1], t.path[nxt, 0] - xy[:, 0])
    near = slot < 4
    off = np.where(near, (ks + 2) % 100, (ks - 40) % 100)
    comp = np.where(near, 98, 40)
    fleets = []
    for on in (True, False):
        f = ft.Fleet(t, n, cars_per_world=cpw, lap_target=1, reload_finished=on)
        f.reset(xy, yaw)
        f.lap[:, L["offset"]] = torch.as_tensor(off, dtype=torch.int32, device=f.device)
        f.lap[:, L["completion"]] = torch.as_tensor(comp, dtype=torch.int32, device=f.device)
        torch.cuda.synchronize()
        fleets.append(f)
    A, B = fleets
    for chunk in range(6):
        for _ in range(100):
            A.tick(1); B.tick(1)
        A.sync(); B.sync()
        for k in STATE:
            assert torch.equal(getattr(A, k), getattr(B, k)), (k, chunk)
    assert A.lap[:, L["finished"]].sum().item() > 0
    assert not (A.lap[:, L["finished"]] != 0).view(-1, cpw).all(1).any()
    assert (A.race_start == 0).all() and (A.race_tally == 0).all()


@pytest.mark.parametrize("n,cpw,ticks", [(256, 1, 200), (24576, 8, 40)])
def test_nothing_due_leaves_the_fleet_as_with_the_option_off(ft, n, cpw, ticks):
    """A cap no race reaches: graph-replayed (256 cars) and eager (24,576 cars in 8-car worlds) ticks are bit-identical to
    the plain tick."""
    t = ft.Track.bundled("track")
    xy, yaw = _poses(t, n, 41)
    A = ft.Fleet(t, n, cars_per_world=cpw, reload_finished=True, race_ticks=10_000)
    B = ft.Fleet(t, n, cars_per_world=cpw)
    A.reset(xy, yaw); B.reset(xy, yaw)
    A.tick(ticks); B.tick(ticks)
    A.sync(); B.sync()
    for k in STATE:
        assert torch.equal(getattr(A, k), getattr(B, k)), k
    assert (A.race_tally == 0).all() and (A.race_start == 0).all()


def test_every_way_of_issuing_the_tick_agrees_across_reloads(ft):
    """64 one-car worlds near their finish line, lap_target 1 and race_ticks 150 (both triggers: the first finishes come
    after about 120 ticks), next starts rewritten after 200 ticks: the graph-replayed tick, the eager tick, tick(50),
    tick_readback and the separate calls reload -> lap_update -> drive -> lidar -> step are bit-identical after every 50
    ticks."""
    L, R = ft.fleet.LAP, ft.fleet.RACE
    t = ft.Track.bundled("small-circle")
    n = 64
    keys = STATE + ("race_tally", "race_start", "start_xy", "start_yaw", "start_offset")
    ranges_h = torch.empty(n, 90, dtype=torch.float32).pin_memory()
    lap_h = torch.empty(n, len(L), dtype=torch.int32).pin_memory()

    def run(kind):
        f, ks = _near_finish(ft, t, n, lap_target=1, reload_finished=True, race_ticks=150)
        snaps = []
        for chunk in range(8):
            if chunk == 4:
                f.set_next_start(*_elsewhere(t, ks, shift=30, togo=6))
            if kind == "graph":
                for _ in range(50):
                    f.tick(1)
            elif kind == "eager":
                prev = f.lib.ftgp_tick_use_graphs(0)
                try:
                    for _ in range(50):
                        f.tick(1)
                finally:
                    f.lib.ftgp_tick_use_graphs(prev)
            elif kind == "tick50":
                f.tick(50)
            elif kind == "readback":
                for _ in range(50):
                    f.tick_readback(ranges_h, lap_h)
                f.sync_readback()
                assert torch.equal(lap_h, f.lap.cpu())
            else:
                for _ in range(50):
                    f.reload(); f.lap_update(); f.drive(); f.lidar(); f.step(1)
            f.sync()
            snaps.append({k: getattr(f, k).clone() for k in keys})
        assert f.steps == 400
        return snaps

    ref = run("graph")
    for kind in ("eager", "tick50", "readback", "separate"):
        got = run(kind)
        for chunk, (a, b) in enumerate(zip(ref, got)):
            for k in keys:
                assert torch.equal(a[k], b[k]), (kind, chunk, k)
    tally = ref[-1]["race_tally"]
    assert (tally[:, R["races"]] >= 2).all()                       # the cap ends a race every 150 ticks at the latest
    assert tally[:, R["finished"]].sum().item() > 0               # ... and some cars finished first


def test_full_size_series(ft):
    """65,536 one-car worlds, race_ticks = 40, 100 ticks: every row equals a fresh fleet's after 20 ticks."""
    R = ft.fleet.RACE
    t = ft.Track.bundled("track")
    n = 65536
    xy, yaw = _poses(t, n, 51)
    A = ft.Fleet(t, n, reload_finished=True, race_ticks=40)
    A.reset(xy, yaw)
    A.tick(100)
    F = ft.Fleet(t, n)
    F.reset(xy, yaw)
    F.tick(20)
    A.sync(); F.sync()
    _assert_same(A, F, ft.fleet.LAP, "full size")
    assert (A.race_tally[:, R["races"]] == 2).all() and (A.race_start == 80).all()
