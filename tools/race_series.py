#!/usr/bin/env python
"""GPU box: what race after race on the device (Fleet(reload_finished=True)) costs, CUDA events on the fleets' streams.

    python tools/race_series.py [--out FILE.json] [--series-ticks 20000]

1. overhead: the plain tick (ftgp_tick) against the reload tick with no world due (a race cap no race reaches), two
   fleets with the same poses, timed alternately in windows of 50 ticks after a 100-tick warm-up: 65,536 one-car worlds
   on track.png (random on-track poses) and 32,768 worlds of 8 cars on the start grid.  The state is ~1.5 KB per car
   plus ~6 KB of step scratch, so the working set (>= 0.5 GB) does not fit the 126 MB L2 and is not flushed in between.
2. every world due: the reload tick with race_ticks = 1 (each world is reloaded at the head of every tick) against the
   plain tick, alternated in the same way, and the reload kernel's own device time (torch.profiler) with every world
   due and with none due.
3. a continuous series: 65,536 cars on circle / small-circle, lap_target 1, race_ticks 25,000, starts = the grid pose +
   seeded jitter (0.1 m, 0.1 rad), rewritten between calls of tick(1000): car-steps/s and completed races per second.
One JSON line per measurement, each with the card's name and power limit; --out collects them.
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
from ft_grandprix_b200.fleet import RACE  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out[0] if out else "unavailable"}


def poses(track, n, seed):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 100, n)
    nxt = (idx + 1) % 100
    yaw = np.arctan2(track.path[nxt, 1] - track.path[idx, 1], track.path[nxt, 0] - track.path[idx, 0])
    return track.path[idx] + rng.normal(0, 0.1, (n, 2)), yaw + rng.normal(0, 0.3, n)


def make(track, n, cpw, grid, **kw):
    f = ft.Fleet(track, n, cars_per_world=cpw, driver="nidc", **kw)
    if grid:
        f.reset_grid()
    else:
        f.reset(*poses(track, n, 1))
    return f


def window_ms(f, nticks):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(f.stream)
    f.tick(nticks)
    e1.record(f.stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / nticks


def ab(fleets, rounds=10, window=50, warmup=100):
    """Per-tick milliseconds of each fleet: median over `rounds` windows, the fleets alternating window by window."""
    for f in fleets.values():
        f.tick(warmup)
        f.sync()
    ms = {k: [] for k in fleets}
    for _ in range(rounds):
        for k, f in fleets.items():
            ms[k].append(window_ms(f, window))
    return {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))} for k, v in ms.items()}


def reload_kernel_us(f, calls=20):
    """Device time of reload_kernel per call (torch.profiler, CUDA activities), with f.steps advanced by one per call
    so that a race_ticks = 1 fleet has every world due at every call."""
    from torch.profiler import ProfilerActivity, profile
    f.reload(); f.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            f.steps += 1
            f.reload()
        f.sync()
    for e in prof.key_averages():
        if "reload_kernel" in e.key:
            total = getattr(e, "device_time_total", None)
            if total is None:
                total = e.cuda_time_total
            return total / e.count
    raise RuntimeError("reload_kernel not found in the profile")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--series-ticks", type=int, default=20000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "race_series.py measures on the GPU; there is nothing to measure without one"
    info = card()
    lines = []

    def emit(d):
        d = d | info
        lines.append(d)
        print(json.dumps(d), flush=True)

    track = ft.Track.bundled("track")
    for n, cpw, grid, label in ((65536, 1, False, "65,536 one-car worlds, track.png, random on-track poses"),
                                (262144, 8, True, "32,768 worlds x 8 cars, track.png, start grid")):
        fleets = {"plain": make(track, n, cpw, grid),
                  "reload_none_due": make(track, n, cpw, grid, reload_finished=True, race_ticks=1 << 30),
                  "reload_all_due": make(track, n, cpw, grid, reload_finished=True, race_ticks=1)}
        r = ab(fleets)
        plain = r["plain"]["median_ms"]
        emit({"measure": "tick_ms", "workload": label, "cars": n, "cars_per_world": cpw, "ticks_per_window": 50,
              "windows": 10, "result": r,
              "overhead_none_due_pct": 100 * (r["reload_none_due"]["median_ms"] / plain - 1),
              "overhead_all_due_pct": 100 * (r["reload_all_due"]["median_ms"] / plain - 1)})
        emit({"measure": "reload_kernel_us", "workload": label, "cars": n, "cars_per_world": cpw,
              "none_due": reload_kernel_us(fleets["reload_none_due"]),
              "all_due": reload_kernel_us(fleets["reload_all_due"])})
        for f in fleets.values():
            f.close()
        del fleets
        torch.cuda.empty_cache()

    n, window = 65536, 1000
    for name in ("circle", "small-circle"):
        t = ft.Track.bundled(name)
        f = ft.Fleet(t, n, driver="nidc", lap_target=1, reload_finished=True, race_ticks=25000)
        x, y, yw = t.start_pose(0)
        rng = np.random.default_rng(7)

        def jitter():
            return (np.array([x, y]) + rng.normal(0, 0.1, (n, 2)), yw + rng.normal(0, 0.1, n))
        f.reset(*jitter())
        f.tick(100); f.sync()                          # warm-up (graphs are not used at this size), then a new series
        f.reset(*jitter())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.series_ticks // window):
            f.set_next_start(*jitter())
            f.tick(window)
        f.sync()
        secs = time.perf_counter() - t0
        tally = f.race_tally.cpu().numpy()
        best = tally[:, RACE["best_lap"]]
        ticks = (args.series_ticks // window) * window
        emit({"measure": "series", "track": f"{name}.png", "cars": n, "lap_target": 1, "race_ticks": 25000,
              "ticks": ticks, "ticks_per_call": window, "seconds": secs, "car_steps_per_s": n * ticks / secs,
              "races_completed": int(tally[:, RACE["races"]].sum()), "races_per_s": float(tally[:, RACE["races"]].sum() / secs),
              "finishes": int(tally[:, RACE["finished"]].sum()),
              "best_lap_ticks": int(best[best > 0].min()) if (best > 0).any() else None,
              "timing": "host clock around the loop (start rewrites included), ending in a device synchronise"})
        f.close()
        del f
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
