"""GPU: neural-network drivers in the device drivers and the fused tick (ftgp_drivers_policy, ftgp_tick_policy,
Fleet.set_policies).  policy_kernel equals the fp64 restatement policy_ref; how cars are grouped changes no bit; a bank
beside nidc / fast cars changes nothing for them; with policies driving, every way of issuing the tick agrees; a bank
rewritten in place takes effect on the next replayed tick; the sweep tool's smoke mode is deterministic."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_policy_host import _golden_states, policy_ref, random_net, random_states

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STATE = ("qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "status", "winners")
RACE_STATE = ("race_tally", "race_start")


@pytest.fixture(scope="module")
def ft():
    import ft_grandprix_b200 as ft
    return ft


def _bank(seeds, gains=None):
    gains = gains or [1.0] * len(seeds)
    nets = [random_net(s, g) for s, g in zip(seeds, gains)]
    return nets, torch.stack([n.pack() for n in nets])


def _load(f, states):
    s, qpos, qvel, ctrl = states
    f.ranges.copy_(torch.from_numpy(np.ascontiguousarray(s)))
    f.qpos.copy_(torch.from_numpy(np.ascontiguousarray(qpos)))
    f.qvel.copy_(torch.from_numpy(np.ascontiguousarray(qvel)))
    f.ctrl.copy_(torch.from_numpy(np.ascontiguousarray(ctrl)))
    torch.cuda.synchronize()


def _drive(f, states):
    _load(f, states)
    f.drive(); f.sync()
    return f.ctrl.cpu().numpy()


def test_kernel_matches_the_reference(ft):
    """The 403 golden scans plus 4,096 seeded ones with random states and ctrl; 8 policies, three of them with weights
    large enough to saturate most tanh units; kinds nidc / fast / lobotomy / policy mixed, every 7th car finished, some
    ids out of range.  POLICY cars are within 1e-4 x scale of policy_ref; finished, lobotomy and out-of-range cars write
    exactly (0, 0); nidc and fast cars are bit-identical to the same call without a bank."""
    g, r = _golden_states(31), random_states(4096, 32)
    states = tuple(np.concatenate([a, b]) for a, b in zip(g, r))
    n = len(states[0])
    nets, bank = _bank(list(range(40, 48)), [1.0, 1.0, 12.0, 1.0, 12.0, 1.0, 12.0, 1.0])
    rng = np.random.default_rng(33)
    kinds = rng.integers(0, 4, n)
    kinds[:403] = 3                                    # every golden scan goes through a policy
    ids = rng.integers(0, 8, n)
    ids[rng.random(n) < 0.05] = -1
    ids[rng.random(n) < 0.05] = 8
    finished = np.arange(n) % 7 == 3
    t = ft.Track.bundled("small-circle")
    f = ft.Fleet(t, n)
    f.set_driver_kinds(kinds.tolist())
    f.lap[:, ft.fleet.LAP["finished"]] = torch.as_tensor(finished.astype(np.int32), device=f.device)
    plain = _drive(f, states)
    f.set_policies(bank, ids)
    got = _drive(f, states)
    checked = 0
    for i in range(n):
        if finished[i] or kinds[i] == 2 or (kinds[i] == 3 and not 0 <= ids[i] < 8):
            assert got[i, 0] == 0.0 and got[i, 1] == 0.0, i
        elif kinds[i] == 3:
            net = nets[ids[i]]
            want = policy_ref(bank[ids[i]].numpy(), states[0][i], states[1][i], states[2][i], states[3][i])
            err = np.abs(got[i] - want) / np.array([net.speed_scale, net.steer_scale])
            assert err.max() <= 1e-4, (i, got[i], want)
            checked += 1
        else:
            assert got[i, 0] == plain[i, 0] and got[i, 1] == plain[i, 1], i
    assert checked > 1000
    # without a bank a POLICY car is inert
    f.set_policies(None)
    got = _drive(f, states)
    assert (got[kinds == 3] == 0).all()


def _pairs(n, P, seed):
    """n (policy, state) pairs: policy c // (n / P) for pair c"""
    return np.arange(n) // (n // P), random_states(n, seed)


def _run_layout(ft, t, perm, pol, states, bank, one_per_car=False):
    """Fleet position k holds pair perm[k]; returns the ctrl of pair c at row c."""
    n = len(perm)
    f = ft.Fleet(t, n, driver="policy")
    sub = tuple(a[perm] for a in states)
    if one_per_car:
        f.set_policies(bank[torch.from_numpy(pol[perm])], np.arange(n))
    else:
        f.set_policies(bank, pol[perm])
    out = np.empty((n, 2))
    out[perm] = _drive(f, sub)
    f.close()
    return out


def test_grouping_does_not_change_a_bit(ft):
    """4,096 (policy, state) pairs on 64 policies, laid out contiguously, at random, 8-interleaved (neighbours on different
    policies) and with one policy per car: bit-identical ctrl.  One car alone equals the same car in a 65,536-car fleet."""
    n, P = 4096, 64
    pol, states = _pairs(n, P, 34)
    _, bank = _bank(list(range(100, 100 + P)), [12.0 if k % 4 == 0 else 1.0 for k in range(P)])
    t = ft.Track.bundled("small-circle")
    rng = np.random.default_rng(35)
    ref = _run_layout(ft, t, np.arange(n), pol, states, bank)
    inter = np.argsort(np.arange(n) % (n // P), kind="stable")       # position k: pair of policy k % 64
    assert len(set(pol[inter[:8]])) == 8
    for name, perm, one in (("random", rng.permutation(n), False), ("interleaved", inter, False),
                            ("one_per_car", rng.permutation(n), True)):
        got = _run_layout(ft, t, perm, pol, states, bank, one)
        assert np.array_equal(got, ref), name
    # one car alone, then the same car at position 12,345 of a 65,536-car fleet on random ids
    big = random_states(65536, 36)
    ids = rng.integers(0, P, 65536)
    for c in (0, 777, 4095):
        one = ft.Fleet(t, 1, driver="policy")
        one.set_policies(bank[int(pol[c])])
        alone = _drive(one, tuple(a[c:c + 1] for a in states))[0]
        f = ft.Fleet(t, 65536, driver="policy")
        for a, b in zip(big, states):
            a[12345] = b[c]
        ids[12345] = pol[c]
        f.set_policies(bank, ids)
        inside = _drive(f, big)[12345]
        assert np.array_equal(alone, inside), c
        assert np.array_equal(alone, ref[c]), c
        one.close(); f.close()


def _poses(t, n, seed):
    from conftest import random_poses
    p = random_poses(t.path, n, seed=seed, level=True)
    return p[:, :2].copy(), 2 * np.arctan2(p[:, 6], p[:, 3])


def _fleet(ft, t, n, cpw, seed, **kw):
    f = ft.Fleet(t, n, cars_per_world=cpw, lap_target=1, reload_finished=True, **kw)
    if cpw == 1:
        f.reset(*_poses(t, n, seed))
    else:
        f.reset_grid()
    return f


@pytest.mark.parametrize("n,cpw", [(4096, 1), (20480, 8)])
def test_a_bank_beside_nidc_and_fast_changes_nothing(ft, n, cpw):
    """Every car nidc or fast: 300 fused ticks (graph-replayed at 4,096 cars, eager at 20,480) are bit-identical with a
    bank set and without.  The old entry point launches as many kernels per tick as the new one without a bank; a bank
    adds the policy kernels' four launches."""
    import ctypes as C
    t = ft.Track.bundled("small-circle")
    kinds = np.arange(n) % 2
    _, bank = _bank([50, 51, 52])
    fleets = {}
    for name in ("new", "bank", "old"):
        f = _fleet(ft, t, n, cpw, 64, race_ticks=120)
        f.set_driver_kinds(kinds.tolist())
        if name == "bank":
            f.set_policies(bank, np.arange(n) % 3)
        fleets[name] = f
    lib = fleets["new"].lib

    def old_tick(f, k):                                # the entry point that predates the bank
        a, r = f.tick_args(), f.reload_args()
        assert lib.ftgp_tick_params(C.byref(a), C.byref(r), None, k, f._s) == 0
        f.steps += k

    per_tick = {}
    for name, f in fleets.items():
        tick = (lambda k, f=f: old_tick(f, k)) if name == "old" else f.tick
        tick(2)                                        # the first tick of a new argument set runs eagerly
        f.sync()
        c0 = lib.ftgp_launch_count()
        tick(10)
        f.sync()
        per_tick[name] = (lib.ftgp_launch_count() - c0) / 10
    assert per_tick["old"] == per_tick["new"] and per_tick["bank"] == per_tick["new"] + 4, per_tick
    for _ in range(300):
        for name, f in fleets.items():
            old_tick(f, 1) if name == "old" else f.tick(1)
    for f in fleets.values():
        f.sync()
    for k in STATE + RACE_STATE:
        assert torch.equal(getattr(fleets["new"], k), getattr(fleets["bank"], k)), k
        assert torch.equal(getattr(fleets["new"], k), getattr(fleets["old"], k)), k


def _mixed(n, seed):
    """kinds: policy on half the cars, nidc / fast on the rest; ids over 6 policies with one out of range"""
    rng = np.random.default_rng(seed)
    kinds = np.where(np.arange(n) % 2 == 0, 3, rng.integers(0, 2, n))
    return kinds, rng.integers(-1, 6, n)


def _drivable_bank():
    """Policies that drive forward: random nets whose speed output is pushed positive, with small steering."""
    nets, _ = _bank(list(range(60, 66)))
    with torch.no_grad():
        for k, net in enumerate(nets):
            net.l3.bias[0] += 1.5
            net.l3.weight[1] *= 0.3
            net.speed_scale = 1.0 + 0.2 * k
            net.steer_scale = 0.6
    return torch.stack([n.pack() for n in nets])


@pytest.mark.parametrize("n,cpw", [(64, 1), (64, 8), (4096, 1), (20480, 8)])
def test_every_way_of_issuing_the_tick_agrees_with_policies(ft, n, cpw):
    """Policies driving half the cars, reload_finished with race_ticks 80: tick(1) (graph-replayed up to 16,384 cars,
    eager above), tick(50) x 4, graphs off, tick_readback and the separate calls reload -> lap_update -> drive -> lidar
    -> step are bit-identical after 200 ticks."""
    t = ft.Track.bundled("small-circle")
    kinds, ids = _mixed(n, 70)
    bank = _drivable_bank()
    ranges_h = torch.empty(n, 90, dtype=torch.float32).pin_memory()
    lap_h = torch.empty(n, len(ft.fleet.LAP), dtype=torch.int32).pin_memory()

    def run(kind):
        f = _fleet(ft, t, n, cpw, 71, race_ticks=80)
        f.set_driver_kinds(kinds.tolist())
        f.set_policies(bank, ids)
        if kind == "tick1":
            for _ in range(200):
                f.tick(1)
        elif kind == "tick50":
            for _ in range(4):
                f.tick(50)
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
        out = {k: getattr(f, k).clone() for k in STATE + RACE_STATE}
        f.close()
        return out

    ref = run("tick1")
    for kind in ("tick50", "eager", "readback", "separate"):
        got = run(kind)
        for k in ref:
            assert torch.equal(ref[k], got[k]), (kind, k)
    # the policies drive: without the bank their cars stay inert and the race goes otherwise
    f = _fleet(ft, t, n, cpw, 71, race_ticks=80)
    f.set_driver_kinds(kinds.tolist())
    f.tick(200); f.sync()
    assert not torch.equal(f.qpos, ref["qpos"])


@pytest.mark.parametrize("cpw", [1, 8])
def test_bank_rewritten_in_place_takes_effect_on_the_next_replayed_tick(ft, cpw):
    """Bank B1 for 100 replayed ticks, then B2 written into fleet.policy_bank (same storage) on fleet.stream and 100 more:
    equal to a fleet loaded from the tick-100 state_dict with B2."""
    t = ft.Track.bundled("small-circle")
    n = 64
    kinds, ids = _mixed(n, 72)
    b1 = _drivable_bank()
    b2 = b1.flip(0).contiguous()

    def fleet():
        f = _fleet(ft, t, n, cpw, 73, race_ticks=80)
        f.set_driver_kinds(kinds.tolist())
        return f

    A = fleet()
    A.set_policies(b1, ids)
    ptr = A.policy_bank.data_ptr()
    for _ in range(100):
        A.tick(1)
    sd = A.state_dict()
    assert torch.equal(sd["policy_bank"], b1) and torch.equal(sd["policy_id"], torch.from_numpy(ids.astype(np.int32)))
    with torch.cuda.stream(A.stream):
        A.policy_bank.copy_(b2.to(A.device))
    assert A.policy_bank.data_ptr() == ptr
    sd["policy_bank"] = b2
    for _ in range(100):
        A.tick(1)
    B = fleet()
    B.load_state_dict(sd)
    for _ in range(100):
        B.tick(1)
    A.sync(); B.sync()
    for k in STATE + RACE_STATE:
        assert torch.equal(getattr(A, k), getattr(B, k)), k
    # and B2 drives differently from B1
    C_ = fleet()
    C_.load_state_dict(sd | {"policy_bank": b1})
    for _ in range(100):
        C_.tick(1)
    C_.sync()
    assert not torch.equal(C_.qpos, A.qpos)


def test_sweep_tool_smoke_is_deterministic(tmp_path):
    """tools/policy_sweep.py --smoke twice: identical clone, identical tallies, and the variants differ."""
    outs = []
    for k in range(2):
        out = tmp_path / f"sweep{k}.json"
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "policy_sweep.py"), "--smoke", "--out", str(out)],
                       check=True, cwd=str(tmp_path), timeout=900)
        lines = [json.loads(x) for x in out.read_text().splitlines()]
        gens = [d for d in lines if d["measure"] == "generation"]
        clone = [d for d in lines if d["measure"] == "clone_race"]
        assert len(gens) == 1 and len(clone) == 1 and "nvidia_smi" in gens[0]
        outs.append((np.array(gens[0]["tally_by_variant"]), clone[0]["tally_by_driver"], clone[0]["final_loss"]))
    assert np.array_equal(outs[0][0], outs[1][0])
    assert outs[0][1:] == outs[1][1:]
    from ft_grandprix_b200.fleet import RACE
    assert outs[0][0][:, RACE["races"]].min() >= 1
    assert len({tuple(r) for r in outs[0][0].tolist()}) > 1
