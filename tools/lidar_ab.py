#!/usr/bin/env python
"""GPU box: time lidar_kernel of every variant library under variants/ (tools/build_variant.py) and of the shipped one, and
check that every variant returns the shipped ranges bit for bit (scheduling must not change a single ray).  Two cases:
`settled`, N cars (argv[1], default 65,536) after 300 ticks of driving, and `config2`, 4,096 cars at the random poses of
`bench.py --workload lidar`.  L2 flushed between launches.

A variant built with -DFTGP_AB_LANESTATS=1 also reports, for one launch, the rounds and the lanes that entered each block
(ray set-up, walk, sweep), the iterations of the loops inside them with the lanes active in each, and the launch shape
(shared memory per CTA, CTAs per SM, track staged in shared memory, cars per warp batch)."""
import ctypes as C, glob, json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ft_grandprix_b200 as ft
from ft_grandprix_b200 import _lib
from bench import make_poses
track = ft.Track.bundled("track")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
STATS = ("setup", "walk", "sweep", "walk_hop", "sweep_line", "cell_test")     # LS_* pairs of lidar.cu, in order
libs = [("shipped", _lib.LIB_PATH)] + [(os.path.basename(p)[8:-3], p) for p in sorted(glob.glob(os.path.join(ROOT, "variants", "libftgp_*.so")))]
flush = None; state = {}; ref = {}


def lane_stats(lib):
    out = (C.c_ulonglong * (2 * len(STATS) + 4))()
    assert lib.ftgp_lidar_lanestats(out) == 0
    v = list(out)
    s = {k: {"rounds": v[2 * i], "lanes_per_round": v[2 * i + 1] / max(v[2 * i], 1)} for i, k in enumerate(STATS)}
    s["launch"] = {"smem_bytes": v[-4], "ctas_per_sm": v[-3], "track_staged": v[-2], "cars_per_batch": v[-1]}
    return s


for case in ("settled", "config2"):
    cars = n if case == "settled" else 4096
    for name, path in libs:
        lib = C.CDLL(path)
        for fn, (res, args) in _lib.SIGNATURES.items():
            f = getattr(lib, fn); f.restype, f.argtypes = res, args
        _lib._lib = lib                                       # (tools only: the package itself always loads libftgp.so)
        fleet = ft.Fleet(track, cars, driver="nidc")
        fleet.lib = lib
        if case == "settled":
            xy, yaw, _ = make_poses(track.path, cars, seed=1, level=True)
            fleet.reset(xy, yaw)
            if case not in state:
                fleet.tick(300); fleet.sync(); state[case] = fleet.qpos.clone()
        else:
            xy, yaw, poses = make_poses(track.path, cars, seed=0, level=False)
            fleet.reset(xy, yaw)
            fleet.qpos[:, :7] = torch.from_numpy(poses).to(fleet.device)
            state[case] = fleet.qpos.clone()
        if flush is None:
            flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=fleet.device)
        fleet.qpos.copy_(state[case]); torch.cuda.synchronize()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(20)]
        with torch.cuda.stream(fleet.stream):
            for _ in range(3): fleet.lidar()
            for e in ev:
                flush.fill_(1)
                e[0].record(fleet.stream); r = fleet.lidar(); e[1].record(fleet.stream)
        fleet.sync()
        got = r.clone()
        if case not in ref: ref[case] = got
        line = {"case": case, "cars": cars, "variant": name,
                "lidar_ms": float(np.mean([e[0].elapsed_time(e[1]) for e in ev])),
                "bit_identical": bool(torch.equal(got.view(torch.int32), ref[case].view(torch.int32)))}
        if hasattr(lib, "ftgp_lidar_lanestats"):
            lib.ftgp_lidar_lanestats.argtypes = [C.POINTER(C.c_ulonglong)]
            lane_stats(lib)                                   # zero the counters, then count one launch
            fleet.lidar(); fleet.sync()
            line["lanes"] = lane_stats(lib)
        print(json.dumps(line), flush=True)
        fleet.close(); del fleet
