#!/usr/bin/env python
"""GPU box: learn a driver and race it on the device, one policy of a bank per car (Fleet.set_policies, include/ftgp.h
FTGP_DRIVER_POLICY, ft_grandprix_b200/policy.py).

    python tools/policy_sweep.py [--out FILE.json] [--overhead] [--no-search] [--cars 65536] [--variants 64]
                                 [--generations 5] [--cars-per-world 1|8] [--race-ticks 3000] [--seed 0] [--smoke]

1. --overhead: what the bank costs.  65,536 cars on track.png at random on-track poses, four cases:
     (a) every car nidc, no bank (one-car worlds);
     (b) every car on a policy, 64 policies in contiguous blocks;
     (c) 8-car worlds, 8 different policies per world out of 64 (driver_sweep.assign), beside (a) in 8-car worlds;
     (d) 65,536 distinct policies (a 2.75 GB bank).
   policy_kernel, the grouping kernels and drivers_kernel are timed with torch.profiler (CUDA activities) over drive()
   calls on the same fleets, and the fused tick in alternated windows of 50 ticks after a 100-tick warm-up.  The
   policies are the clone of part 2 with Gaussian weight noise.
2. cloning: a nidc fleet on small-circle.png (one-car worlds, seeded random starts, reload_finished) is run through the
   separate calls reload -> lap_update -> [record policy_inputs and, after drive(), the nidc ctrl] -> lidar -> step.
   A PolicyNet is fitted to the records with Adam on the GPU (seeded, torch.use_deterministic_algorithms), packed and
   raced against the nidc and fast drivers in one fleet: a third of the cars each.
3. the search: a seeded evolution as in driver_sweep.py.  Variants 0 and 1 are the nidc and fast drivers, variants
   2.. are policies: generation 0 is the clone and its mutants (Gaussian noise on every weight); the top quarter of the
   policies are the parents of the rest.  Fitness comes from race_tally (driver_sweep.fitness).
One JSON line per measurement, each with the card's name and power limit; --out collects them.  --smoke: 1,024 cars,
8 variants, a short recording and fit, one generation (the GPU test runs it twice and compares).
"""
import argparse
import json
import os
import sys
import time

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")    # deterministic cuBLAS for the seeded fit
import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ft_grandprix_b200 as ft  # noqa: E402
from driver_sweep import assign, card, fitness, starts, window_ms  # noqa: E402
from ft_grandprix_b200.fleet import LAP, RACE  # noqa: E402
from ft_grandprix_b200.policy import POLICY_FLOATS, PolicyNet, policy_inputs  # noqa: E402

KERNELS = ("policy_kernel", "policy_count_kernel", "policy_scan_kernel", "policy_scatter_kernel", "drivers_kernel")


def mutate(bank, rng, sigma):
    """Gaussian noise on every weight and bias of packed policies [k, POLICY_FLOATS]; the scalars are kept."""
    noise = torch.from_numpy(rng.normal(0, sigma, (bank.shape[0], POLICY_FLOATS)).astype(np.float32))
    noise[:, :4] = 0
    noise[:, -2:] = 0
    return bank + noise


# ------------------------------------------------------------------ 2. cloning
def record(n, ticks, every, seed, clip):
    """(x [m, 96], y [m, 2]): the policy inputs of nidc cars and the ctrl the nidc driver wrote from them."""
    track = ft.Track.bundled("small-circle")
    rng = np.random.default_rng(seed)
    f = ft.Fleet(track, n, driver="nidc", lap_target=1, reload_finished=True, race_ticks=1500)
    xy, yaw, off = starts(track, n, 1, 20, rng)
    f.reset(xy, yaw)
    f.set_next_start(xy, yaw, off)
    xs, ys = [], []
    for t in range(ticks):
        f.reload(); f.lap_update()
        if t % every == 0:
            with torch.cuda.stream(f.stream):
                xs.append(policy_inputs(f.ranges, f.qpos, f.qvel, f.ctrl, clip))
        f.drive()
        if t % every == 0:
            with torch.cuda.stream(f.stream):
                ys.append(f.ctrl.to(torch.float32))
        f.lidar(); f.step(1)
    f.sync()
    f.close()
    return torch.cat(xs), torch.cat(ys)


def fit(x, y, steps, seed, batch=4096):
    torch.manual_seed(seed)
    torch.use_deterministic_algorithms(True)
    net = PolicyNet(range_clip=10.0, speed_scale=3.0, steer_scale=1.6).to(x.device)
    opt = torch.optim.Adam(net.parameters(), lr=2e-3)
    scale = torch.tensor([net.speed_scale, net.steer_scale], device=x.device)
    g = torch.Generator(device=x.device)
    g.manual_seed(seed)
    loss = None
    for _ in range(steps):
        idx = torch.randint(0, x.shape[0], (batch,), device=x.device, generator=g)
        loss = (((net(x[idx]) - y[idx]) / scale) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    torch.use_deterministic_algorithms(False)
    return net.cpu(), float(loss)


def race_groups(f, groups, names):
    """per driver: races, finish rate, mean lap (ticks) and the summed tally"""
    tally = f.race_tally.cpu().numpy()
    out = {}
    for g, name in enumerate(names):
        t = tally[groups == g].sum(0)
        fin = int(t[RACE["finished"]])
        out[name] = {"races": int(t[RACE["races"]]), "finish_rate": fin / max(int(t[RACE["races"]]), 1),
                     "mean_lap_ticks": float(t[RACE["time_sum"]] / fin) if fin else None, "tally": t.tolist()}
    return out


def clone(emit, n_rec, rec_ticks, every, steps, n_race, race_ticks, seed):
    t0 = time.perf_counter()
    x, y = record(n_rec, rec_ticks, every, seed, 10.0)
    net, loss = fit(x, y, steps, seed)
    secs = time.perf_counter() - t0
    track = ft.Track.bundled("small-circle")
    rng = np.random.default_rng(seed + 1)
    groups = np.arange(n_race) % 3                  # nidc, fast, clone
    f = ft.Fleet(track, n_race, lap_target=1, reload_finished=True, race_ticks=race_ticks)
    xy, yaw, off = starts(track, n_race, 1, 20, rng)
    f.reset(xy, yaw)
    f.set_next_start(xy, yaw, off)
    with torch.cuda.stream(f.stream):
        f.lap[:, LAP["offset"]] = torch.as_tensor(off, dtype=torch.int32, device=f.device)
    f.set_driver_kinds(np.where(groups == 2, 3, groups).tolist())
    f.set_policies(net.pack())
    f.tick(2 * race_ticks)
    f.sync()
    res = race_groups(f, groups, ("nidc", "fast", "clone"))
    f.close()
    emit({"measure": "clone_race", "samples": int(x.shape[0]), "fit_steps": steps, "final_loss": loss,
          "record_and_fit_seconds": secs, "cars": n_race, "race_ticks": race_ticks, "ticks": 2 * race_ticks,
          "track": "small-circle", "seed": seed, "result": {k: {kk: vv for kk, vv in v.items() if kk != "tally"} for k, v in res.items()},
          "tally_by_driver": {k: v["tally"] for k, v in res.items()}})
    return net


# ------------------------------------------------------------------ 1. overhead
def kernel_us(f, calls=20):
    from torch.profiler import ProfilerActivity, profile
    f.drive(); f.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            f.drive()
        f.sync()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k + "(" in e.key or e.key.endswith(k) or ("::" + k) in e.key:
                total = getattr(e, "device_time_total", None)
                if total is None:
                    total = e.cuda_time_total
                out[k] = total / calls
    return out


def overhead(emit, base, n=65536, rounds=10, window=50, warmup=100):
    track = ft.Track.bundled("track")
    rng = np.random.default_rng(1)
    idx = rng.integers(0, 100, n)
    nxt = (idx + 1) % 100
    yaw = np.arctan2(track.path[nxt, 1] - track.path[idx, 1], track.path[nxt, 0] - track.path[idx, 0])
    xy, yaw = track.path[idx] + rng.normal(0, 0.1, (n, 2)), yaw + rng.normal(0, 0.3, n)
    bank64 = mutate(base.pack()[None].repeat(64, 1), rng, 0.01)
    cases = {}

    def fleet(cpw, name):
        f = ft.Fleet(track, n, cars_per_world=cpw, driver="nidc" if name.startswith("a") else "policy")
        if cpw == 1:
            f.reset(xy, yaw)
        else:
            f.reset_grid()
        return f

    f = fleet(1, "a"); cases["a_nidc_no_bank"] = f
    f = fleet(1, "b"); f.set_policies(bank64, np.arange(n) // (n // 64)); cases["b_64_contiguous"] = f
    f = fleet(8, "a8"); cases["a8_nidc_no_bank_8car_worlds"] = f
    f = fleet(8, "c"); f.set_policies(bank64, assign(n, 8, 64, rng)); cases["c_64_8_per_world"] = f
    big = torch.empty(n, POLICY_FLOATS, dtype=torch.float32, device="cuda")
    for k in range(0, n, 4096):                      # the clone plus fresh noise per policy, built on the device
        big[k:k + 4096] = base.pack().cuda() + 0.01 * torch.randn(4096, POLICY_FLOATS, device="cuda",
                                                                  generator=torch.Generator("cuda").manual_seed(k))
    big[:, :4] = base.pack()[:4].cuda()
    f = fleet(1, "d"); f.set_policies(big, np.arange(n)); cases["d_65536_distinct"] = f
    del big
    torch.cuda.synchronize()
    for f in cases.values():
        f.tick(warmup); f.sync()
    ms = {k: [] for k in cases}
    for _ in range(rounds):
        for k, f in cases.items():
            ms[k].append(window_ms(f, window))
    tick = {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))} for k, v in ms.items()}
    emit({"measure": "tick_ms", "workload": f"{n:,} cars, track.png, random on-track poses (8-car worlds: start grid)",
          "cars": n, "ticks_per_window": window, "windows": rounds, "result": tick,
          "note": "policy-driven cars drive differently, so the step's cost differs: the tick comparison is not the kernel's cost"})
    kern = {k: kernel_us(f) for k, f in cases.items()}
    bank_bytes = n * POLICY_FLOATS * 4
    emit({"measure": "kernel_us", "cars": n, "result": kern, "timing": "torch.profiler, mean device time per drive() call",
          "case_d_bank_bytes": bank_bytes,
          "case_d_bound_us_at_7.7TBps_datasheet": bank_bytes / 7.7e12 * 1e6,
          "case_d_achieved_GBps": bank_bytes / (kern["d_65536_distinct"].get("policy_kernel", float("nan")) * 1e-6) / 1e9})
    for f in cases.values():
        f.close()


# ------------------------------------------------------------------ 3. the search
def search(emit, base, n, K, gens, cpw, race_ticks, togo, seed, sigma=0.02):
    assert n % K == 0 and (cpw == 1 or K % cpw == 0) and K >= 4
    track = ft.Track.bundled("small-circle")
    rng = np.random.default_rng(seed)
    P = K - 2                                      # variants 0, 1: nidc, fast; variant v >= 2: policy v - 2
    bank = torch.cat([base.pack()[None], mutate(base.pack()[None].repeat(P - 1, 1), rng, sigma)])
    f = ft.Fleet(track, n, cars_per_world=cpw, lap_target=1, reload_finished=True, race_ticks=race_ticks)
    ticks = 2 * race_ticks
    for gen in range(gens):
        variant = assign(n, cpw, K, rng)
        xy, yaw, off = starts(track, n, cpw, togo, rng)
        f.reset(xy, yaw)
        f.set_next_start(xy, yaw, off)
        with torch.cuda.stream(f.stream):
            f.lap[:, LAP["offset"]] = torch.as_tensor(off, dtype=torch.int32, device=f.device)
        f.set_driver_kinds(np.where(variant < 2, variant, 3).tolist())
        f.set_policies(bank, np.maximum(variant - 2, 0))
        f.sync()
        t0 = time.perf_counter()
        f.tick(ticks)
        f.sync()
        secs = time.perf_counter() - t0
        tally = f.race_tally.cpu().numpy()
        fit_ = fitness(tally, variant, K, cpw)
        order = sorted(range(K), key=lambda v: fit_[v][0])
        best = next(v for v in order if v > 1)
        emit({"measure": "generation", "generation": gen, "cars": n, "cars_per_world": cpw, "variants": K,
              "race_ticks": race_ticks, "ticks": ticks, "togo_points": togo, "seed": seed, "seconds": secs,
              "car_steps_per_s": n * ticks / secs, "races_per_s": float(tally[:, RACE["races"]].sum() / secs),
              "rank_nidc": order.index(0) + 1, "rank_fast": order.index(1) + 1, "rank_best_policy": order.index(best) + 1,
              "best_policy": best - 2, "nidc": fit_[0][1] | {"tally": None}, "fast": fit_[1][1] | {"tally": None},
              "best": fit_[best][1] | {"tally": None},
              "tally_by_variant": [fit_[v][1]["tally"] for v in range(K)],
              "timing": "host clock around tick(ticks), ending in a device synchronise"})
        parents = [v - 2 for v in order if v > 1][:max(1, P // 4)]
        for p in range(P):
            if p not in parents:
                bank[p] = mutate(bank[parents[rng.integers(len(parents))]][None], rng, sigma)[0]
    f.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--overhead", action="store_true")
    ap.add_argument("--no-search", action="store_true")
    ap.add_argument("--cars", type=int, default=65536)
    ap.add_argument("--variants", type=int, default=64)
    ap.add_argument("--generations", type=int, default=5)
    ap.add_argument("--cars-per-world", type=int, default=1, choices=(1, 8))
    ap.add_argument("--race-ticks", type=int, default=3000)
    ap.add_argument("--togo", type=int, default=20, help="centreline points from the start to the finish line (>= 10)")
    ap.add_argument("--record-cars", type=int, default=4096)
    ap.add_argument("--record-ticks", type=int, default=3000)
    ap.add_argument("--fit-steps", type=int, default=4000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--smoke", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "policy_sweep.py runs on the GPU; there is nothing to run without one"
    if args.smoke:
        args.cars, args.variants, args.generations, args.race_ticks, args.togo = 1024, 8, 1, 1000, 10
        args.record_cars, args.record_ticks, args.fit_steps = 256, 400, 200
    info = card()
    lines = []

    def emit(d):
        d = d | info
        lines.append(d)
        print(json.dumps(d), flush=True)

    base = clone(emit, args.record_cars, args.record_ticks, 10, args.fit_steps, args.cars if args.smoke else 3 * 4096,
                 args.race_ticks, args.seed)
    if args.overhead:
        overhead(emit, base)
    if not args.no_search:
        search(emit, base, args.cars, args.variants, args.generations, args.cars_per_world, args.race_ticks, args.togo,
               args.seed)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
