"""CPU: neural-network drivers (include/ftgp.h FTGP_DRIVER_POLICY, ft_grandprix_b200/policy.py).  policy_ref, a
statement-by-statement numpy fp64 restatement of the header's function read from the packed layout (also the GPU
tests' reference), equals PolicyNet run in float64; the fp32 twin agrees within the tolerance the kernel is held to;
pack / unpack round-trip; the input rules hold on hand-checkable cases; the constants match the header; the new entry
points reject bad arguments before any CUDA call."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

torch = pytest.importorskip("torch")

# the layout table of include/ftgp.h, restated here rather than imported
FLOATS, NIN, HID = 10504, 96, 64
OFF = {"scalars": 0, "W1": 4, "b1": 6148, "W2": 6212, "b2": 10308, "W3": 10372, "b3": 10500}


def policy_ref(row, ranges, qpos, qvel, ctrl):
    """(speed, steering) of one car under the packed policy `row`, as include/ftgp.h states it: the inputs in fp32 (the
    speeds in fp64, rounded), the network in fp64 from the fp32 weights."""
    row = np.asarray(row, dtype=np.float32)
    clip = row[OFF["scalars"]]
    x = np.zeros(NIN, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        for j in range(90):
            r = np.float32(ranges[j])
            x[j] = np.float32(r / clip) if (r >= 0 and r < clip) else 1.0
    w, qx, qy, qz = (float(v) for v in qpos[3:7])
    yaw = math.atan2(2 * (w * qz + qx * qy), 1 - 2 * (qy * qy + qz * qz))
    vx, vy = float(qvel[0]), float(qvel[1])
    x[90] = np.float32(vx * math.cos(yaw) + vy * math.sin(yaw))
    x[91] = np.float32(-vx * math.sin(yaw) + vy * math.cos(yaw))
    x[92] = np.float32(qvel[5])
    x[93] = np.float32(ctrl[0])
    x[94] = np.float32(ctrl[1])
    x[95] = 0.0
    r64 = row.astype(np.float64)
    W1 = r64[OFF["W1"]:OFF["W1"] + NIN * HID].reshape(NIN, HID)
    b1 = r64[OFF["b1"]:OFF["b1"] + HID]
    W2 = r64[OFF["W2"]:OFF["W2"] + HID * HID].reshape(HID, HID)
    b2 = r64[OFF["b2"]:OFF["b2"] + HID]
    W3 = r64[OFF["W3"]:OFF["W3"] + HID * 2].reshape(HID, 2)
    b3 = r64[OFF["b3"]:OFF["b3"] + 2]
    h1 = np.array([math.tanh(b1[j] + sum(W1[i, j] * x[i] for i in range(NIN))) for j in range(HID)])
    h2 = np.array([math.tanh(b2[j] + sum(W2[i, j] * h1[i] for i in range(HID))) for j in range(HID)])
    z = [b3[o] + sum(W3[i, o] * h2[i] for i in range(HID)) for o in range(2)]
    return r64[1] * math.tanh(z[0]), r64[2] * math.tanh(z[1])


def random_net(seed, gain=1.0):
    """A seeded PolicyNet; gain > 1 scales every weight and bias (at gain 12 about half the hidden units sit within 1e-3 of +-1)."""
    from ft_grandprix_b200.policy import PolicyNet
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    net = PolicyNet(range_clip=rng.uniform(2.0, 12.0), speed_scale=rng.uniform(1.0, 8.0), steer_scale=rng.uniform(0.3, 1.6))
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(gain)
    return net


def random_states(n, seed):
    """Scans with misses, zeros, long ranges and NaN; unit quaternions of any heading with a little pitch and roll;
    velocities and ctrl of a racing car."""
    rng = np.random.default_rng(seed)
    s = rng.uniform(0.05, 14.0, (n, 90))
    s[rng.random((n, 90)) < 0.05] = -1.0
    s[rng.random((n, 90)) < 0.03] = 0.0
    s[rng.random((n, 90)) < 0.002] = np.nan
    qpos = np.zeros((n, 34))
    qpos[:, :2] = rng.uniform(-5, 5, (n, 2))
    q = np.concatenate([rng.normal(0, 1, (n, 1)), rng.normal(0, 0.05, (n, 2)), rng.normal(0, 1, (n, 1))], axis=1)
    qpos[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    qvel = rng.normal(0, 1.5, (n, 29))
    ctrl = np.stack([rng.uniform(0, 7, n), rng.uniform(-1.6, 1.6, n)], axis=1)
    return s.astype(np.float32), qpos, qvel, ctrl


def _golden_states(seed):
    scans = np.load(os.path.join(GOLDEN, "drivers.npz"))["scans"].astype(np.float32)
    _, qpos, qvel, ctrl = random_states(len(scans), seed)
    return scans, qpos, qvel, ctrl


def _twin(net, states, dtype):
    from ft_grandprix_b200.policy import policy_inputs
    s, qpos, qvel, ctrl = states
    x = policy_inputs(torch.from_numpy(s), torch.from_numpy(qpos), torch.from_numpy(qvel), torch.from_numpy(ctrl), net.range_clip)
    with torch.no_grad():
        return net.to(dtype)(x.to(dtype)).double().numpy()


def _refs(row, states, idx):
    s, qpos, qvel, ctrl = states
    return np.array([policy_ref(row, s[i], qpos[i], qvel[i], ctrl[i]) for i in idx])


@pytest.mark.parametrize("seed,gain", [(1, 1.0), (2, 1.0), (3, 12.0)])
def test_reference_equals_the_twin_in_float64(seed, gain):
    net = random_net(seed, gain)
    row = net.pack().numpy()
    states = _golden_states(seed) if seed == 1 else random_states(300, seed)
    idx = range(len(states[0]))
    want = _refs(row, states, idx)
    got = _twin(net, states, torch.float64)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)


@pytest.mark.parametrize("seed,gain", [(4, 1.0), (5, 12.0)])
def test_fp32_twin_within_the_kernel_tolerance(seed, gain):
    """The fp32 twin sums in another order than the kernel: both are held to 1e-4 x scale of the fp64 reference."""
    net = random_net(seed, gain)
    row = net.pack().numpy()
    states = random_states(400, seed)
    want = _refs(row, states, range(400))
    got = _twin(net, states, torch.float32)
    scale = np.array([net.speed_scale, net.steer_scale])
    err = np.abs(got - want) / scale
    assert err.max() <= 1e-4, err.max()
    if gain > 1:                                    # the large weights saturate most hidden units
        from ft_grandprix_b200.policy import policy_inputs
        x = policy_inputs(*(torch.from_numpy(a) for a in states), net.range_clip)
        with torch.no_grad():
            h1 = torch.tanh(net.float().l1(x))
        assert (h1.abs() > 0.999).float().mean() > 0.4


def test_pack_unpack_round_trip():
    from ft_grandprix_b200.policy import PolicyNet
    net = random_net(7, 2.0)
    row = net.pack()
    assert row.dtype == torch.float32 and row.shape == (FLOATS,)
    back = PolicyNet.unpack(row)
    assert torch.equal(back.pack(), row)
    for a, b in zip(net.parameters(), back.parameters()):
        assert torch.equal(a.detach(), b.detach())
    assert (back.range_clip, back.speed_scale, back.steer_scale) == (net.range_clip, net.speed_scale, net.steer_scale)
    assert row[3] == 0 and (row[OFF["b3"] + 2:] == 0).all()
    # input-major: W1[i * 64 + j] multiplies x[i] into unit j
    assert row[OFF["W1"] + 5 * HID + 7] == net.l1.weight[7, 5]
    assert row[OFF["W3"] + 9 * 2 + 1] == net.l3.weight[1, 9]
    with pytest.raises(ValueError):
        PolicyNet.unpack(row[:-1])


def _inputs(ranges, qpos=None, qvel=None, ctrl=(0.0, 0.0), clip=5.0):
    from ft_grandprix_b200.policy import policy_inputs
    q = np.zeros((1, 34)); q[0, 3] = 1.0
    if qpos is not None:
        q[0, 3:7] = qpos
    v = np.zeros((1, 29))
    if qvel is not None:
        v[0, :len(qvel)] = qvel
    return policy_inputs(torch.tensor([ranges], dtype=torch.float32), torch.from_numpy(q), torch.from_numpy(v),
                         torch.tensor([ctrl], dtype=torch.float64), clip)[0].numpy()


def test_input_rules_on_hand_checkable_cases():
    r = np.full(90, 2.5, dtype=np.float32)
    r[0], r[1], r[2], r[3], r[4], r[5] = -1.0, 5.0, 7.0, np.nan, 0.0, 4.999
    x = _inputs(r)
    assert x[0] == 1 and x[1] == 1 and x[2] == 1 and x[3] == 1          # a miss, at the clip, above it, NaN
    assert x[4] == 0 and x[5] == np.float32(np.float32(4.999) / np.float32(5.0)) and x[6] == 0.5
    assert (_inputs(np.zeros(90, dtype=np.float32))[:90] == 0).all()    # the first tick after a reset
    # heading +y (yaw pi/2) at 1 m/s along +y: forward 1, lateral 0; the yaw rate and the previous ctrl pass through
    h = math.pi / 4
    x = _inputs(r, qpos=(math.cos(h), 0, 0, math.sin(h)), qvel=(0.0, 1.0, 0, 0, 0, 0.75), ctrl=(2.25, -0.5))
    assert abs(x[90] - 1) < 1e-7 and abs(x[91]) < 1e-7
    assert x[92] == np.float32(0.75) and x[93] == np.float32(2.25) and x[94] == np.float32(-0.5) and x[95] == 0
    # heading +x, moving +y: all lateral
    x = _inputs(r, qvel=(0.0, 1.0))
    assert x[90] == 0 and x[91] == 1
    want = policy_ref(random_net(8).pack().numpy(), r, np.r_[0, 0, 0, 1.0, 0, 0, 0], np.zeros(29), (0.0, 0.0))
    assert all(np.isfinite(want))


def test_constants_and_offsets_match_the_header():
    from ft_grandprix_b200 import _lib, policy
    src = open(os.path.join(ROOT, "include", "ftgp.h")).read()
    vals = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(FTGP_POLICY_[A-Z0-9_]+)\s*=\s*(\d+)", src)}
    assert vals["FTGP_POLICY_FLOATS"] == policy.POLICY_FLOATS == FLOATS
    assert vals["FTGP_POLICY_NIN"] == policy.POLICY_NIN == NIN and vals["FTGP_POLICY_HIDDEN"] == policy.POLICY_HIDDEN == HID
    for name, off in OFF.items():
        key = {"scalars": "SCALARS"}.get(name, name.upper())
        assert vals["FTGP_POLICY_" + key] == getattr(policy, "POLICY_" + key) == off, name
        assert off % 4 == 0
    assert re.search(r"FTGP_DRIVER_POLICY\s*=\s*3", src) and _lib.DRIVER_POLICY == 3
    assert OFF["b3"] + 4 == FLOATS and FLOATS * 4 == 42016
    assert C.sizeof(_lib.PolicyArgs) == 2 * 8 + 2 * 4
    lib = C.CDLL(_lib.LIB_PATH)
    assert hasattr(lib, "ftgp_drivers_policy") and hasattr(lib, "ftgp_tick_policy")
    from ft_grandprix_b200.fleet import DRIVER_KINDS
    assert DRIVER_KINDS["policy"] == 3


def _policy(weights=0x1000, npolicies=4):
    from ft_grandprix_b200 import _lib
    p = _lib.PolicyArgs()
    p.weights, p.policy_id, p.npolicies = weights, 0x1000, npolicies
    return p


@pytest.mark.parametrize("bad", ["weights", "npolicies", "default_policy_without_bank", "kind_high", "kind_low",
                                 "qpos", "qvel"])
def test_bad_policy_driver_arguments_raise_before_any_cuda_call(bad):
    from ft_grandprix_b200 import _lib
    lib = _lib.load()
    p, kind, qpos, qvel = _policy(), 3, 0x1000, 0x1000
    if bad == "weights":
        p = _policy(weights=None)
    elif bad == "npolicies":
        p = _policy(npolicies=0)
    elif bad == "default_policy_without_bank":
        p = None
    elif bad == "kind_high":
        kind = 4
    elif bad == "kind_low":
        kind = -1
    elif bad == "qpos":
        qpos = None
    else:
        qvel = None
    rc = lib.ftgp_drivers_policy(0x1000, None, kind, None, None if p is None else C.byref(p), qpos, qvel, None, 0x1000, 8,
                                 None)
    assert rc == 1                                   # FTGP_ERR_ARG, not FTGP_ERR_CUDA: nothing reached the device
    with pytest.raises(_lib.FtgpError, match="bad"):
        _lib.check(rc, "ftgp_drivers_policy")


@pytest.mark.parametrize("bad", ["weights", "npolicies", "default_policy_without_bank", "kind_high", "qpos"])
def test_bad_policy_tick_arguments_raise_before_any_cuda_call(bad):
    from ft_grandprix_b200 import _lib
    from test_races_host import _args
    lib = _lib.load()
    a, r = _args()
    p = _policy()
    a.default_driver = 3
    if bad == "weights":
        p = _policy(weights=None)
    elif bad == "npolicies":
        p = _policy(npolicies=-1)
    elif bad == "default_policy_without_bank":
        p = None
    elif bad == "kind_high":
        a.default_driver = 4
    else:
        a.qpos = None
    rc = lib.ftgp_tick_policy(C.byref(a), C.byref(r), None, None if p is None else C.byref(p), 1, None)
    assert rc == 1
    with pytest.raises(_lib.FtgpError, match="bad"):
        _lib.check(rc, "ftgp_tick_policy")
