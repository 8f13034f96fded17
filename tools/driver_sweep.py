#!/usr/bin/env python
"""GPU box: tune the bundled disparity extender race after race on the device, with one driver parameter row per car
(Fleet.set_driver_params, include/ftgp.h FTGP_DRV_*).

    python tools/driver_sweep.py [--out FILE.json] [--overhead] [--cars 65536] [--variants 64] [--generations 5]
                                 [--cars-per-world 1|8] [--race-ticks 3000] [--seed 0] [--smoke]

1. --overhead: what the rows cost.  The fused tick of 65,536 one-car worlds on track.png (random on-track poses) with
   every car's row set to the nidc reference row against the same fleet without rows, timed alternately in windows of
   50 ticks after a 100-tick warm-up (CUDA events on the fleets' streams), and drivers_kernel's own device time in both
   (torch.profiler, CUDA activities).
2. the search: a seeded evolution of K variants on small-circle.png, lap_target 1, Fleet(reload_finished=True) with a
   race_ticks cap.  Every car starts at a seeded random centreline point (jittered 0.05 m, 0.05 rad) with its finish
   line --togo points ahead; in 8-car worlds the cars of a world start 2 points apart from one such point, and every
   world holds 8 different variants (a fresh seeded assignment each generation).  A generation resets the fleet and runs
   2 x race_ticks ticks; a variant's fitness comes from the race_tally rows of its cars: finish rate, then mean lap time
   (one-car worlds), or wins per race first (8-car worlds).  Variants 0 and 1 are the nidc and fast reference rows and
   are never mutated, so every generation says where they rank; the top quarter are the parents of the rest
   (log-normal jitter of the tunable fields).
One JSON line per measurement, each with the card's name and power limit; --out collects them.  --smoke: 1,024 cars,
8 variants, race_ticks 1000, togo 10, one generation (the GPU test runs it twice and compares the tallies).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ft_grandprix_b200 as ft  # noqa: E402
from ft_grandprix_b200.fleet import DRV, LAP, RACE, default_driver_params  # noqa: E402

TUNABLE = ("car_width", "safety_percentage", "difference_threshold", "speed", "speed_divisor", "boost_speed",
           "boost_max_steer", "speed_cap")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out[0] if out else "unavailable"}


# ------------------------------------------------------------------ 1. overhead
def window_ms(f, nticks):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(f.stream)
    f.tick(nticks)
    e1.record(f.stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / nticks


def drivers_kernel_us(f, calls=20):
    from torch.profiler import ProfilerActivity, profile
    f.drive(); f.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            f.drive()
        f.sync()
    for e in prof.key_averages():
        if "drivers_kernel" in e.key:
            total = getattr(e, "device_time_total", None)
            if total is None:
                total = e.cuda_time_total
            return total / e.count
    raise RuntimeError("drivers_kernel not found in the profile")


def overhead(emit, n=65536, rounds=10, window=50, warmup=100):
    track = ft.Track.bundled("track")
    rng = np.random.default_rng(1)
    idx = rng.integers(0, 100, n)
    nxt = (idx + 1) % 100
    yaw = np.arctan2(track.path[nxt, 1] - track.path[idx, 1], track.path[nxt, 0] - track.path[idx, 0])
    xy, yaw = track.path[idx] + rng.normal(0, 0.1, (n, 2)), yaw + rng.normal(0, 0.3, n)
    fleets = {}
    for name in ("no_rows", "default_rows"):
        f = ft.Fleet(track, n, driver="nidc")
        f.reset(xy, yaw)
        if name == "default_rows":
            f.set_driver_params(default_driver_params("nidc"))
        fleets[name] = f
    for f in fleets.values():
        f.tick(warmup); f.sync()
    ms = {k: [] for k in fleets}
    for _ in range(rounds):
        for k, f in fleets.items():
            ms[k].append(window_ms(f, window))
    A, B = fleets["no_rows"], fleets["default_rows"]
    same = all(torch.equal(getattr(A, k), getattr(B, k)) for k in ("qpos", "qvel", "ctrl", "ranges", "lap"))
    r = {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))} for k, v in ms.items()}
    emit({"measure": "tick_ms", "workload": f"{n:,} one-car worlds, track.png, random on-track poses", "cars": n,
          "ticks_per_window": window, "windows": rounds, "result": r, "bit_identical": same,
          "overhead_pct": 100 * (r["default_rows"]["median_ms"] / r["no_rows"]["median_ms"] - 1)})
    emit({"measure": "drivers_kernel_us", "cars": n, "no_rows": drivers_kernel_us(A), "default_rows": drivers_kernel_us(B)})
    for f in fleets.values():
        f.close()


# ------------------------------------------------------------------ 2. the search
def starts(track, n, cpw, togo, rng):
    """Start poses and lap offsets: a random centreline point per world, cars 2 points apart, each car's finish line
    `togo` points ahead of its start."""
    k0 = np.repeat(rng.integers(0, 100, n // cpw), cpw)
    k = (k0 + 2 * (np.arange(n) % cpw)) % 100
    nxt = (k + 1) % 100
    yaw = np.arctan2(track.path[nxt, 1] - track.path[k, 1], track.path[nxt, 0] - track.path[k, 0])
    xy = track.path[k] + rng.normal(0, 0.05, (n, 2))
    return xy, yaw + rng.normal(0, 0.05, n), (k - (100 - togo)) % 100


def assign(n, cpw, K, rng):
    """variant of every car: n / K cars each; in worlds of 8 every world holds 8 different variants"""
    if cpw == 1:
        return rng.permutation(np.arange(n) % K)
    return np.concatenate([rng.permutation(K) for _ in range(n // K)])


def mutate(row, rng, sigma=0.15):
    out = row.copy()
    for name in TUNABLE:
        v = out[DRV[name]]
        if np.isfinite(v) and v != 0:
            out[DRV[name]] = v * np.exp(rng.normal(0, sigma))
        elif name == "boost_max_steer":
            out[DRV[name]] = abs(rng.normal(0, 0.05))
    return out


def fitness(tally, variant, K, cpw):
    """per variant: (sort key, summary); lower key = better"""
    out = []
    for v in range(K):
        t = tally[variant == v].sum(0)
        races, fin = max(int(t[RACE["races"]]), 1), int(t[RACE["finished"]])
        rate = fin / races
        mean_lap = t[RACE["time_sum"]] / fin if fin else float("inf")
        wins = t[RACE["wins"]] / races
        key = (-wins, -rate, mean_lap) if cpw > 1 else (-rate, mean_lap)
        out.append((key, {"races": int(t[RACE["races"]]), "finish_rate": rate, "mean_lap_ticks": mean_lap,
                          "win_rate": wins, "tally": t.tolist()}))
    return out


def search(emit, n, K, gens, cpw, race_ticks, togo, seed):
    assert n % K == 0 and (cpw == 1 or K % cpw == 0)
    track = ft.Track.bundled("small-circle")
    rng = np.random.default_rng(seed)
    refs = [default_driver_params("nidc"), default_driver_params("fast")]
    rows = np.array(refs + [mutate(refs[i % 2], rng, 0.3) for i in range(K - 2)])
    f = ft.Fleet(track, n, cars_per_world=cpw, driver="nidc", lap_target=1, reload_finished=True, race_ticks=race_ticks)
    ticks = 2 * race_ticks
    for gen in range(gens):
        variant = assign(n, cpw, K, rng)
        xy, yaw, off = starts(track, n, cpw, togo, rng)
        f.reset(xy, yaw)
        f.set_next_start(xy, yaw, off)
        with torch.cuda.stream(f.stream):
            f.lap[:, LAP["offset"]] = torch.as_tensor(off, dtype=torch.int32, device=f.device)
        f.set_driver_params(rows[variant])
        f.sync()
        t0 = time.perf_counter()
        f.tick(ticks)
        f.sync()
        secs = time.perf_counter() - t0
        tally = f.race_tally.cpu().numpy()
        fit = fitness(tally, variant, K, cpw)
        order = sorted(range(K), key=lambda v: fit[v][0])
        emit({"measure": "generation", "generation": gen, "cars": n, "cars_per_world": cpw, "variants": K,
              "race_ticks": race_ticks, "ticks": ticks, "togo_points": togo, "seed": seed, "seconds": secs,
              "car_steps_per_s": n * ticks / secs, "races_per_s": float(tally[:, RACE["races"]].sum() / secs),
              "rank_nidc": order.index(0) + 1, "rank_fast": order.index(1) + 1,
              "top": [{"variant": v, "row": dict(zip(DRV, rows[v].tolist())), **{k: x for k, x in fit[v][1].items() if k != "tally"}}
                      for v in order[:5]],
              "tally_by_variant": [fit[v][1]["tally"] for v in range(K)],
              "timing": "host clock around tick(ticks), ending in a device synchronise"})
        parents = [v for v in order if v > 1][:max(1, K // 4)]
        keep = set(parents) | {0, 1}
        for v in range(2, K):
            if v not in keep:
                rows[v] = mutate(rows[parents[rng.integers(len(parents))]], rng)
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
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--smoke", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "driver_sweep.py runs on the GPU; there is nothing to run without one"
    if args.smoke:
        args.cars, args.variants, args.generations, args.race_ticks, args.togo = 1024, 8, 1, 1000, 10
    info = card()
    lines = []

    def emit(d):
        d = d | info
        lines.append(d)
        print(json.dumps(d), flush=True)

    if args.overhead:
        overhead(emit)
    if not args.no_search:
        search(emit, args.cars, args.variants, args.generations, args.cars_per_world, args.race_ticks, args.togo, args.seed)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
