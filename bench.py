#!/usr/bin/env python
"""bench.py -- throughput of the ft_grandprix hot path on B200 (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload tick|lidar|step] [--cars C]
    python bench.py ... --dump-outputs DIR      # also write the last timed step's arrays as DIR/<name>.npy
    python bench.py --impl reference ...        # the CPU arm (oracle port, all host threads)

One "step" = one pass of the hot path over the whole fleet:
  workload tick  (default; BASELINE config 3): lap update + batched nidc driver + 90-beam lidar +
                 vehicle step for 65,536 cars per GPU on track.png  -> metric car-steps/s
                 (rays/s = 90 x car-steps/s is reported beside it)
  workload lidar (BASELINE config 2): 90-beam scan of 4,096 cars at random poses -> rays/s
  workload step  : vehicle step only, 65,536 cars
  workload episode (BASELINE config 4): 1,048,576 cars IN TOTAL over the N ranks (strong scaling) on circle /
                 small-circle alternating by world index, full tick, lap statistics gathered once at the end
  workload race  (BASELINE config 5): 32,768 worlds x 8 cars IN TOTAL on track.png's start grid; the cars of a world see
                 each other (lidar cylinder, chassis mesh, wheels), collide with each other (worlds whose cars touch are
                 advanced as one coupled Newton problem) and are ranked per world
Cars are sharded over the N ranks with no collective on the step path (weak scaling: the per-GPU
fleet is fixed); only the final timing / stats are gathered.

CPU arms (`--impl reference`, and the `cpu_baseline` key of the GPU line): at run time the script PROBES for a real
MuJoCo (`import mujoco`, also with baseline/_ref on sys.path).  If it imports, the arm is the reference's own loop
(custom.py:1337-1426: driver on last step's sensordata, ctrl write, mj_step) on the world this repo's emitter writes
(ft_grandprix_b200/mjcf.py), single thread per model as the reference steps, kind "reference".  Otherwise it is the C
restatement under oracle/ (kind "port").  The CPU arms never import the product package.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES = {  # algorithmic bytes per unit (SURVEY §8 d, DESIGN.md)
    "tick": 2328.0,    # per car-tick, unfused sum: step 1488 + scan 416 + driver 376 + lap 48
    "step": 1488.0,    # per car-step: qpos/qvel/warm in+out + ctrl
    "lidar": 416.0,    # per scan of 90 rays: pose 56 B + ranges 360 B
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)        # a run that fails before stop() must not leave nvidia-smi polling
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 6 for k in range(4) if r[2 + k].startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_poses(path, n, seed, level):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 100, n)
    nxt = (idx + 1) % 100
    heading = np.arctan2(path[nxt, 1] - path[idx, 1], path[nxt, 0] - path[idx, 0])
    xy = path[idx] + rng.normal(0, 0.10, (n, 2))
    yaw = heading + rng.normal(0, 0.3, n)
    if level:
        return xy, yaw, None
    z = 0.0156 + rng.uniform(-0.002, 0.002, n)
    roll, pitch = rng.normal(0, 0.01, n), rng.normal(0, 0.01, n)
    cy, sy, cp, sp, cr, sr = np.cos(yaw / 2), np.sin(yaw / 2), np.cos(pitch / 2), np.sin(pitch / 2), np.cos(roll / 2), np.sin(roll / 2)
    q = np.stack([cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                  cr * cp * sy - sr * sp * cy], 1)
    return xy, yaw, np.concatenate([xy, z[:, None], q], 1)


def workload_name(wl, cars):
    return {"tick": f"full tick (lap + nidc + 90-beam lidar + vehicle step), {cars} cars/GPU on track.png (BASELINE config 3)",
            "lidar": f"lidar-only, {cars} cars/GPU at random poses on track.png, 90 beams, no cutoff (BASELINE config 2)",
            "step": f"vehicle step only, {cars} cars/GPU on track.png"}[wl]


# what one call of the timed path hands back: the fleet arrays it writes
TIMED_OUTPUTS = {"lidar": ("ranges",), "step": ("qpos", "qvel", "warm", "status")}
TICK_OUTPUTS = ("qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "winners", "status")
DUMP_ROWS = 32768      # rows (cars, or worlds for `winners`) per array over all ranks: <= 45 MB of .npy files in all


def dump_outputs(out_dir, fleet, wl, rank, world):
    """--dump-outputs: the fleet arrays the timed path wrote in its last step, as out_dir/<name>.npy (float32 stays
    float32, the integer arrays are widened to float64).  An array of more rows than its share of DUMP_ROWS is cut to a
    fixed, seeded sample of rows, so that two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name in TIMED_OUTPUTS.get(wl, TICK_OUTPUTS):
        a = getattr(fleet, name).cpu().numpy()
        if len(a) > DUMP_ROWS // world:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), DUMP_ROWS // world, replace=False))]
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


# ----------------------------------------------------------------------------- CPU arms
def bundled_track(name="track"):
    """(wall mask, SVG path data) of a bundled track, read straight from the data files (no product import)."""
    z = np.load(os.path.join(ROOT, "ft_grandprix_b200", "assets", "tracks.npz"))
    key = name.replace("-", "_")
    shape = tuple(int(v) for v in z[key + "__shape"])
    wall = np.unpackbits(z[key + "__bits"])[: shape[0] * shape[1]].reshape(shape)
    d = json.load(open(os.path.join(ROOT, "ft_grandprix_b200", "assets", "paths.json")))[name]
    return wall, d


def probe_mujoco():
    """The real reference engine, if this box has it (it does not in the build image: no wheel, no network)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref) and ref not in sys.path:
        sys.path.append(ref)
    try:
        import mujoco
        return mujoco
    except Exception:
        return None


def mujoco_units_per_s(mj, wl, ncars_model, ticks, seed=1):
    """The reference's own loop on real MuJoCo, headless (no DearPyGui, no renderer, no physics_fps sleep): ONE model
    with ncars_model cars, single thread, exactly as custom.py:1337-1426 steps it.  The world comes from this repo's
    emitter, loaded by file path so that the product library is not touched."""
    import importlib.util
    import tempfile
    from oracle import pyoracle
    spec = importlib.util.spec_from_file_location("ftgp_mjcf", os.path.join(ROOT, "ft_grandprix_b200", "mjcf.py"))
    mjcf = importlib.util.module_from_spec(spec); spec.loader.exec_module(mjcf)
    wall, d_attr = bundled_track("track")
    ot = pyoracle.Track(wall)
    path = ot.centreline(d_attr)
    cars = [{"driver": "ft_grandprix.nidc", "name": f"car {i}", "primary": "red", "secondary": "pink", "icon": "white.png"}
            for i in range(ncars_model)]
    with tempfile.TemporaryDirectory() as tmp:
        meta = mjcf.write_chunks(wall, os.path.join(tmp, "chunks"), name="track", scale=2.0)
        mjcf.produce_mjcf(cars, meta, tmp, rangefinders=90)
        m = mj.MjModel.from_xml_path(os.path.join(tmp, "car.xml"))
    dat = mj.MjData(m)
    mj.mj_resetData(m, dat)
    sens = [np.array([mj.mj_name2id(m, mj.mjtObj.mjOBJ_SENSOR, f"rangefinder #{i}.#{j}") for j in range(90)]) for i in range(ncars_model)]
    qadr = [int(m.jnt_qposadr[mj.mj_name2id(m, mj.mjtObj.mjOBJ_JOINT, f"car #{i}")]) for i in range(ncars_model)]
    turn = [mj.mj_name2id(m, mj.mjtObj.mjOBJ_ACTUATOR, f"turn #{i}") for i in range(ncars_model)]
    fwd = [mj.mj_name2id(m, mj.mjtObj.mjOBJ_ACTUATOR, f"forward #{i}") for i in range(ncars_model)]
    for i in range(ncars_model):                                   # position_vehicles (custom.py:1232-1245)
        k = (i % 40 + 5) * 2
        dlt = path[k + 1] - path[k]
        yaw = float(np.arctan2(dlt[1], dlt[0]))
        dat.qpos[qadr[i]:qadr[i] + 2] = path[k]
        dat.qpos[qadr[i] + 3:qadr[i] + 7] = (np.cos(yaw / 2), 0, 0, np.sin(yaw / 2))
    laps = [pyoracle.Lap(offset=(i % 40 + 5) * 2) for i in range(ncars_model)]
    t0 = time.perf_counter()
    for k in range(ticks):
        if wl == "tick":
            for i in range(ncars_model):
                laps[i].update(path, np.array(dat.qpos[qadr[i]:qadr[i] + 2]), k, 10, 0)
                r = pyoracle.driver(0, np.array(dat.sensordata[sens[i]]))
                if r is not None:
                    dat.ctrl[fwd[i]] = r[0]; dat.ctrl[turn[i]] = r[1]
        mj.mj_step(m, dat)                                          # (rangefinders are evaluated inside, like the reference)
    dt = time.perf_counter() - t0
    return ncars_model * ticks * (90 if wl == "lidar" else 1) / dt, dt


def cpu_units_per_s(wl, sample_cars, ticks, threads, seed=1):
    """Times the oracle (oracle/*.c, a C restatement: kind 'port') on a bounded sample of the workload."""
    from concurrent.futures import ThreadPoolExecutor
    # the oracle library as build() left it: it is not re-made when oracle/*.c is newer (build() always runs make -B), and
    # pyoracle.lib() makes it only if it is missing
    from oracle import pyoracle
    wall, d_attr = bundled_track("track")
    ot = pyoracle.Track(wall)
    tpath = ot.centreline(d_attr)
    xy, yaw, poses = make_poses(tpath, sample_cars, seed, level=(wl != "lidar"))
    chunks = np.array_split(np.arange(sample_cars), threads)
    if wl == "lidar":
        def work(ix):
            return ot.scan(poses[ix], threads=1)
        t0 = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(work, chunks))
        dt = time.perf_counter() - t0
        return sample_cars * 90 / dt, dt
    model = pyoracle.Model()
    state = [model.reset(xy[i, 0], xy[i, 1], yaw[i]) for i in range(sample_cars)]
    qpos = np.stack([s[0] for s in state]); qvel = np.stack([s[1] for s in state]); warm = np.stack([s[2] for s in state])
    ctrl = np.zeros((sample_cars, 2)); ranges = np.zeros((sample_cars, 90))
    laps = [pyoracle.Lap(offset=10) for _ in range(sample_cars)]
    # the sample is driven into the running regime first (untimed), like the GPU arm's --settle
    def work(ix, nt):
        lo, hi = int(ix[0]), int(ix[-1]) + 1
        for k in range(nt):
            if wl == "tick":
                for i in range(lo, hi):
                    laps[i].update(tpath, qpos[i, :2], k, 10, 0)
                    r = pyoracle.driver(0, ranges[i])
                    if r is not None:
                        ctrl[i] = r
                ranges[lo:hi] = ot.scan(qpos[lo:hi, :7], threads=1)
            model.step_n(ot, qpos[lo:hi], qvel[lo:hi], warm[lo:hi], ctrl[lo:hi], nthreads=1)
    live = [c for c in chunks if len(c)]
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda c: work(c, CPU_SETTLE_TICKS), live))
        t0 = time.perf_counter()
        list(ex.map(lambda c: work(c, ticks), live))
        dt = time.perf_counter() - t0
    return sample_cars * ticks / dt, dt


CPU_SETTLE_TICKS = 50


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload if args.workload in ("lidar", "step") else "tick"      # episode / race: the CPU arm is the full tick
    threads = os.cpu_count() or 1
    mj = probe_mujoco()
    bound = {"lidar": 64 * threads, "tick": 16 * threads, "step": 16 * threads}[wl]
    sample_cars = max(1, min(args.cars, bound))                    # a bounded sample of the arm's --cars
    ticks = 1 if wl == "lidar" else 10
    vals, dts = [], []
    if mj is not None and wl != "lidar":
        # the real thing: one MuJoCo model, single thread, 3 cars (template/cars/cars.json's size) per model
        ncm, ticks = 3, 400
        for _ in range(args.warmup):
            mujoco_units_per_s(mj, wl, ncm, 50)
        for _ in range(args.steps):
            v, dt = mujoco_units_per_s(mj, wl, ncm, ticks)
            vals.append(v); dts.append(dt)
        kind, cores = "reference", 1
        sample = f"MuJoCo {mj.__version__}, one model of {ncm} cars x {ticks} ticks on track.png, headless custom.py:1337-1426 loop, 1 thread"
        note = "reference = the reference's own MuJoCo loop (single process, single thread, as the reference steps)"
    else:
        for _ in range(args.warmup):
            cpu_units_per_s(wl, max(threads, sample_cars // 8), 1 if wl == "lidar" else 2, threads)
        for _ in range(args.steps):
            v, dt = cpu_units_per_s(wl, sample_cars, ticks, threads)
            vals.append(v); dts.append(dt)
        kind, cores = "port", threads
        sample = (f"{sample_cars} of {args.cars} cars x {ticks} tick(s) per step on track.png after {CPU_SETTLE_TICKS} settle ticks, "
                  f"C oracle (oracle/*.c), {threads} threads")
        note = ("reference = MuJoCo-on-CPU loop; `import mujoco` failed on this box (probed, also baseline/_ref), so the arm "
                "times the C restatement of that loop (oracle/), not MuJoCo itself")
    value = float(np.mean(vals))
    metric, unit = ("lidar rays/s", "rays/s") if wl == "lidar" else ("car-steps/s", "car-steps/s")
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(dts) * 1e3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(wl, args.cars), "sample": sample},
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "sample": sample,
                             "host_cores_available": threads},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "mujoco_probe": ("found " + mj.__version__) if mj is not None else "import mujoco failed",
            "note": note}
    if wl != "lidar":
        line["rays_per_s"] = value * 90 if wl == "tick" else 0.0
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import ft_grandprix_b200 as ft

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl, cars = args.workload, args.cars
    lib = ft._lib.load()
    track = ft.Track.bundled("track")
    fleet = ft.Fleet(track, cars, device=local, driver="nidc")
    xy, yaw, poses = make_poses(track.path, cars, seed=(0 if wl == "lidar" else 1) + 1000 * rank, level=(wl != "lidar"))
    fleet.reset(xy, yaw)
    if wl == "lidar":
        fleet.qpos[:, :7] = torch.from_numpy(poses).to(fleet.device)
    torch.cuda.synchronize()
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=fleet.device)   # > 126 MB L2

    def one_step(kev=None):
        """One pass of the hot path.  The tick is issued as its four kernels in the order of ftgp_tick / custom.py:1337-1426
        (lap update, driver, rangefinders from the pre-step pose, mj_step) so that the two heavy kernels can be bracketed
        by their own CUDA events (kev = [lidar0, lidar1, step0, step1]) on the launching stream."""
        if wl == "lidar":
            if kev: kev[0].record(stream)
            fleet.lidar()
            if kev: kev[1].record(stream)
        elif wl == "step":
            if kev: kev[2].record(stream)
            fleet.step(1)
            if kev: kev[3].record(stream)
        else:
            fleet.lap_update()
            fleet.drive()
            if kev: kev[0].record(stream)
            fleet.lidar()
            if kev: kev[1].record(stream); kev[2].record(stream)
            fleet.step(1)
            if kev: kev[3].record(stream)

    def timed_step():
        if wl == "tick":
            fleet.tick(1)                # the product's fused entry point (ftgp_tick): same kernels, one C call
        else:
            one_step()

    stream = fleet.stream
    if wl == "tick" and args.fused_check:
        # the fused C entry point and the four separate calls are the same kernels in the same order
        sd = fleet.state_dict()
        fleet.tick(3); fleet.sync()
        a = {k: v.clone() for k, v in fleet.state_dict().items() if hasattr(v, "clone")}
        fleet.load_state_dict(sd); torch.cuda.synchronize()
        for _ in range(3):
            one_step()
        fleet.sync()
        b = fleet.state_dict()
        assert all(torch.equal(a[k], b[k]) for k in a), "ftgp_tick differs from the four separate calls"
        fleet.load_state_dict(sd); torch.cuda.synchronize()
    # clocks / throttle reasons are sampled from the warm-up on (nvidia-smi needs a few hundred ms to start reporting;
    # settle + warm-up + timed steps are the same load)
    sampler = ClockSampler(local)
    sampler.start()
    with torch.cuda.stream(stream):
        settle = args.settle if wl != "lidar" else 0
        for k in range(settle):          # drive the fleet into its running regime (untimed)
            one_step()
        for _ in range(args.warmup):     # warms the call that is timed: the first fused tick sets up its side stream and
            flush.fill_(1)               # scratch, and small fleets capture their CUDA graph on the second one
            timed_step()
    stream.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: K steps, each bracketed by CUDA events on the launching stream, L2 flushed between
    launches0 = lib.ftgp_launch_count()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kevs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    with torch.cuda.stream(stream):
        for a, b in ev:
            flush.fill_(1)
            a.record(stream)
            timed_step()
            b.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = lib.ftgp_launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fleet, wl, rank, world)
    # second pass, same regime: the two heavy kernels bracketed by their own CUDA events on the launching stream
    with torch.cuda.stream(stream):
        for kev in kevs:
            flush.fill_(1)
            one_step(kev)
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    lidar_ms = np.mean([k[0].elapsed_time(k[1]) for k in kevs]) if wl != "step" else None
    step_ms = np.mean([k[2].elapsed_time(k[3]) for k in kevs]) if wl != "lidar" else None

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D + kernels + D2H inside the timed region
    e2e_steps = max(3, min(args.steps, 20))
    h2d = d2h = 0
    if wl == "lidar":
        import ctypes as C
        qpos_h = torch.empty(cars, 34, dtype=torch.float64).pin_memory(); qpos_h.copy_(fleet.qpos.cpu())
        out_h = torch.empty(cars, 90, dtype=torch.float32).pin_memory()
        def e2e_step():
            ft._lib.check(lib.ftgp_lidar_host(fleet.geom._ptr, C.c_void_p(qpos_h.data_ptr()), 34, None, cars,
                                              C.c_void_p(out_h.data_ptr())), "ftgp_lidar_host")
        h2d, d2h = cars * 7 * 8, cars * 90 * 4
    else:
        ctrl_h = torch.zeros(cars, 2, dtype=torch.float64).pin_memory()
        ranges_h = torch.empty(cars, 90, dtype=torch.float32).pin_memory()
        lap_h = torch.empty_like(fleet.lap, device="cpu").pin_memory()
        def e2e_step():
            if wl == "tick":
                # the public per-tick call with host delivery: copies overlap the kernels that do not touch the arrays;
                # the host waits for THIS tick's ranges and lap state before the next tick is issued
                fleet.tick_readback(ranges_h, lap_h)
                fleet.sync_readback()
                return
            with torch.cuda.stream(stream):
                fleet.ctrl.copy_(ctrl_h, non_blocking=True)
                one_step()
                ranges_h.copy_(fleet.ranges, non_blocking=True)
                lap_h.copy_(fleet.lap, non_blocking=True)
            stream.synchronize()
        h2d = cars * 16 if wl == "step" else 0
        d2h = cars * 90 * 4 + fleet.lap.numel() * 4
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- reduce over ranks (max time), rank 0 prints
    tt = torch.tensor([dev_ms, e2e_s * 1e3, float(launches)], dtype=torch.float64, device=fleet.device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, launches = float(tt[0]), float(tt[1]), int(tt[2])
    units_per_step = cars * world * (90 if wl == "lidar" else 1)
    value = units_per_step * args.steps / (dev_ms * 1e-3)
    e2e_value = units_per_step * e2e_steps / (e2e_ms * 1e-3)
    peak, peak_src = peaks()
    # roofline of the dominant kernel (step_kernel in the tick, else the only kernel): algorithmic bytes of ONE launch
    # (SURVEY 8d: 1,488 B per car-step, 416 B per 90-ray scan) / its own CUDA-event duration in this timed region
    STEP_KERNEL = "step_quad_kernel"
    dom_is_lidar = wl == "lidar" or (wl == "tick" and lidar_ms > step_ms)
    dom = "lidar_kernel" if dom_is_lidar else STEP_KERNEL
    dom_ms = lidar_ms if dom_is_lidar else step_ms
    per_unit = (BYTES["lidar"] if dom_is_lidar else BYTES["step"])
    achieved = cars * per_unit / (dom_ms * 1e-3) / 1e9
    traffic, prof = None, {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        prof = json.load(open(tp))
        if cars == int(prof.get("cars", 65536)):            # the ncu capture is of ONE fleet size; no figure for others
            traffic = prof.get(dom)
    # FP64 pipe: the step is bound by FP64 issue + latency, not by HBM (SURVEY 8d asks for flop/s beside the HBM line).
    # flop per launch = 2 x DFMA + DADD + DMUL thread-instructions of one step at this fleet size, from the committed
    # ncu capture; peak = 148 SMs x 64 FP64 FMA/clk x 2 x SM clock (the public 37 TFLOP/s HGX B200 figure at 1.965 GHz)
    fp64 = None
    if step_ms is not None and cars == int(prof.get("cars", 65536)) and prof.get("step_fp64_flop"):
        clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
        peak_tf = 148 * 64 * 2 * clk / 1e12
        ach_tf = prof["step_fp64_flop"] / (step_ms * 1e-3) / 1e12
        fp64 = {"flop_per_step_launch": prof["step_fp64_flop"], "flop_per_car_step": prof["step_fp64_flop"] / cars,
                "achieved_tflops": ach_tf, "peak_tflops": peak_tf, "frac": ach_tf / peak_tf,
                "pipe_busy_pct_ncu": prof.get("step_fp64_pipe_pct"), "source": "profiles/traffic.json (ncu sass op counts)"}
    kernels = {}
    if lidar_ms is not None:
        kernels["lidar_kernel"] = {"ms": float(lidar_ms), "rays_per_s": cars * 90 / (lidar_ms * 1e-3), "ns_per_ray": lidar_ms * 1e6 / (cars * 90),
                                   "algorithmic_GBps": cars * BYTES["lidar"] / (lidar_ms * 1e-3) / 1e9}
    if step_ms is not None:
        kernels[STEP_KERNEL] = {"ms": float(step_ms), "car_steps_per_s": cars / (step_ms * 1e-3),
                                "algorithmic_GBps": cars * BYTES["step"] / (step_ms * 1e-3) / 1e9,
                                "includes": "the two counting-sort launches that group cars by Newton iteration count"}
    metric, unit = ("lidar rays/s", "rays/s") if wl == "lidar" else ("car-steps/s", "car-steps/s")
    line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64" if wl != "lidar" else "f32 traversal / f64 pose",
            "data": "synthetic",
            "config": {"workload": workload_name(wl, cars), "cars_per_gpu": cars, "beams": 90, "track": "track.png",
                       "driver": "nidc (device)", "l2": "flushed (512 MiB write) between timed steps",
                       "timing": "CUDA events on the launching stream per step, summed; max over ranks; per-kernel times from a second pass",
                       "sharding": f"{world} x {cars} cars, no collective on the step path"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": dom, "kernel_ms": float(dom_ms),
                         "algorithmic_bytes_per_launch": cars * per_unit, "algorithmic_bytes_per_unit": per_unit,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/)" if traffic else None,
                         "note": "latency/issue-bound path: algorithmic HBM traffic is far below peak by construction (SURVEY §8 d)"},
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "how": "public API with pinned host buffers, wall clock around H2D + kernels + D2H; the host waits for every tick's ranges and lap state"},
            "gpu_launches": launches, "clocks": clocks, "kernels": kernels, "fp64": fp64}
    line["config"]["settle_ticks"] = settle
    if wl != "lidar":
        line["rays_per_s"] = value * 90 if wl == "tick" else 0.0
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            mj = probe_mujoco()
            if mj is not None and wl != "lidar":
                v, dt = mujoco_units_per_s(mj, wl, 3, 1500)
                line["cpu_baseline"] = {"value": v, "unit": unit, "cores": 1, "kind": "reference", "host_cores_available": os.cpu_count(),
                                        "sample": f"MuJoCo {mj.__version__}: one model of 3 cars x 1500 ticks, headless reference loop ({dt:.1f} s)"}
            else:
                threads = 1
                sc = {"lidar": 4096, "tick": 128, "step": 128}[wl]          # ~10-20 s of single-thread CPU work
                nt = 1 if wl == "lidar" else 60
                v, dt = cpu_units_per_s(wl, sc, nt, threads)
                line["cpu_baseline"] = {"value": v, "unit": unit, "cores": threads, "kind": "port",
                                        "host_cores_available": os.cpu_count(), "mujoco_probe": "import mujoco failed",
                                        "sample": (f"{sc} cars x 90 rays at the bench poses, C oracle single thread ({dt:.1f} s)" if wl == "lidar" else
                                                   f"{sc} cars x {nt} tick(s) after {CPU_SETTLE_TICKS} settle ticks, C oracle single thread ({dt:.1f} s)")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- BASELINE config 4: one sharded episode
def run_episode(args, kind="episode"):
    """1,048,576 independent cars (total, strong scaling) on circle / small-circle alternating by GLOBAL world index,
    contiguous blocks of worlds per rank, no collective on the step path; the episode's lap statistics are gathered
    once at the end (NCCL all_gather, ft_grandprix_b200.sharding)."""
    import torch
    import torch.distributed as dist
    import ft_grandprix_b200 as ft
    from ft_grandprix_b200.sharding import STAT_FIELDS, ShardedRace
    from ft_grandprix_b200.track import Geometry

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = ft._lib.load()
    if kind == "race":
        # BASELINE config 5: worlds of 8 cars on the reference start grid of track.png (custom.py:1232-1245), drivers
        # alternating nidc / fast as in template/cars/cars.json; the cars see and hit each other and are ranked per world
        cpw, tracks = 8, [ft.Track.bundled("track")]
        nworlds = args.cars // cpw
        race = ShardedRace(nworlds, cpw, 1, lambda n, tid, first: ft.Fleet(Geometry(tracks, device=local), n, cars_per_world=cpw,
                                                                           device=local, driver="nidc"))
        fleet = race.fleet
        n = fleet.ncars
        grid = np.array([tracks[0].start_pose(c) for c in range(cpw)])
        rng = np.random.default_rng(3 + 1000 * rank)
        xy = np.tile(grid[:, :2], (n // cpw, 1)) + rng.normal(0, 0.01, (n, 2))
        yaw = np.tile(grid[:, 2], n // cpw) + rng.normal(0, 0.02, n)
        fleet.set_driver_kinds(["nidc" if c % 2 == 0 else "fast" for c in range(cpw)] * (n // cpw))
    else:
        cpw, tracks = 1, [ft.Track.bundled("circle"), ft.Track.bundled("small-circle")]
        nworlds = args.cars
        race = ShardedRace(nworlds, 1, 2, lambda n, tid, first: ft.Fleet(Geometry(tracks, device=local), n, device=local, track_id=tid, driver="nidc",
                                                                         lap_target=args.lap_target))
        fleet = race.fleet
        n = fleet.ncars
        xy = np.zeros((n, 2)); yaw = np.zeros(n)
        for t in range(2):
            sel = np.nonzero(race.track_id == t)[0]
            a, b, _ = make_poses(tracks[t].path, len(sel), seed=2 + 1000 * rank + t, level=True)
            xy[sel] = a; yaw[sel] = b
    fleet.reset(xy, yaw)
    xy0 = fleet.qpos[:, :2].clone()
    ncars_total = nworlds * cpw
    stream = fleet.stream
    sampler = ClockSampler(local); sampler.start()
    full = bool(args.full_episode) and kind == "episode"
    if not full:
        with torch.cuda.stream(stream):
            for _ in range(args.settle):
                fleet.tick(1)
            for _ in range(args.warmup):
                fleet.tick(1)
    else:                                                    # an episode starts at the reset: warm the code paths on a scratch copy
        sd = fleet.state_dict()
        fleet.tick(args.warmup); fleet.sync()
        fleet.load_state_dict(sd); torch.cuda.synchronize()
    stream.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = lib.ftgp_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ticks_done = 0
    with torch.cuda.stream(stream):
        e0.record(stream)
        if not full:
            for _ in range(args.steps):
                fleet.tick(1)
            ticks_done = args.steps
        else:
            # SURVEY 8d config 4: "until all finished lap_target laps or 25 000 ticks (100 s)".  Each rank runs its own shard
            # to the end (no collective on the step path); the finished count is read back every 250 ticks.
            FIN = ft.fleet.LAP["finished"]
            while ticks_done < 25000:
                fleet.tick(250); ticks_done += 250
                if int((fleet.lap[:, FIN] == 0).sum().item()) == 0:
                    break
        e1.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = lib.ftgp_launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fleet, kind, rank, world)
    dev_ms = e0.elapsed_time(e1)
    car_steps = float(n) * ticks_done
    t0 = time.perf_counter()
    stats = race.episode_stats()                     # the only collective of the episode
    torch.cuda.synchronize()
    gather_ms = (time.perf_counter() - t0) * 1e3
    # e2e: ticks through the public API with the episode statistics read back to the host every step
    lap_h = torch.empty_like(fleet.lap, device="cpu").pin_memory()
    ranges_h = torch.empty(n, 90, dtype=torch.float32).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fleet.tick_readback(ranges_h, lap_h)         # per-tick host delivery, copies overlapped with the kernels
        fleet.sync_readback()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    # the same with the lap state only (what an episode's consumer reads per tick; the ranges stay on the device for the drivers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fleet.tick_readback(None, lap_h)
        fleet.sync_readback()
    barrier()
    e2e_lap_ms = (time.perf_counter() - t0) * 1e3
    tt = torch.tensor([dev_ms, e2e_ms, float(launches), gather_ms, float(ticks_done), e2e_lap_ms], dtype=torch.float64, device=fleet.device)
    cs = torch.tensor([car_steps], dtype=torch.float64, device=fleet.device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
    dev_ms, e2e_ms, launches, gather_ms, ticks_max, e2e_lap_ms = float(tt[0]), float(tt[1]), int(tt[2]), float(tt[3]), int(tt[4]), float(tt[5])
    value = float(cs[0]) / (dev_ms * 1e-3)
    peak, peak_src = peaks()
    achieved = value * BYTES["tick"] / 1e9
    laps = stats[:, STAT_FIELDS.index("laps")]
    line = {"metric": "car-steps/s", "value": value, "unit": "car-steps/s", "n_gpus": world, "steps": ticks_max, "warmup": args.warmup,
            "ms_per_step": dev_ms / ticks_max, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": (f"sharded episode, {nworlds} cars in total on circle/small-circle alternating by world index, "
                                    f"full tick, stats gathered once (BASELINE config 4)") if kind == "episode" else
                                   (f"race worlds, {nworlds} worlds x 8 cars in total on track.png, start grid, nidc/fast alternating, cars see "
                                    f"and hit each other (coupled world solve for touching cars), per-world ranking (BASELINE config 5)"),
                       "cars_total": ncars_total,
                       "cars_per_gpu": n, "beams": 90, "driver": "nidc (device)",
                       "l2": "fleet state per GPU (>= 190 MB at 8 GPUs) exceeds the 126 MB L2", "timing": "CUDA events around the K ticks; max over ranks",
                       "sharding": f"{world} contiguous blocks of worlds, no collective on the step path"},
            "roofline": {"bound": "hbm", "achieved": achieved / world, "peak": peak, "unit": "GB/s", "frac": achieved / world / peak,
                         "traffic": None, "peak_source": peak_src, "kernel": "whole tick (per GPU)",
                         "algorithmic_bytes_per_unit": BYTES["tick"],
                         "note": "latency/issue-bound path: algorithmic HBM traffic is far below peak by construction (SURVEY 8d)"},
            "e2e": {"value": ncars_total * e2e_steps / (e2e_ms * 1e-3), "unit": "car-steps/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": n * 90 * 4 + fleet.lap.numel() * 4, "steps": e2e_steps,
                    "how": "Fleet.tick_readback: ranges and lap state to pinned host memory every tick (host waits for them), wall clock",
                    "lap_state_only": {"value": ncars_total * e2e_steps / (e2e_lap_ms * 1e-3), "d2h_bytes_per_step": fleet.lap.numel() * 4,
                                       "how": "Fleet.tick_readback(None, lap_host): only the lap state crosses PCIe"}},
            "gpu_launches": launches, "clocks": clocks, "rays_per_s": value * 90,
            "episode": {"gather_ms": gather_ms, "stats_rows": int(stats.shape[0]), "stats_bytes": int(stats.numel() * 4),
                        "laps_max": int(laps.max()), "ticks": ticks_max, "to_completion": full, "lap_target": args.lap_target,
                        "finished_cars": int(stats[:, STAT_FIELDS.index("finished")].sum()) if "finished" in STAT_FIELDS else None,
                        "cars_moved_5cm_this_rank": int(((fleet.qpos[:, :2] - xy0).norm(dim=1) > 0.05).sum()),
                        "cars_in_coupled_worlds_last_tick_this_rank": int(((fleet.status >> 9) & 1).sum())}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5,
                    help="untimed steps through the same call as the timed ones; fleets of up to 16,384 cars capture the tick's "
                         "CUDA graph on its second call, so fewer than 2 leave that capture in the first timed step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("FTGP_WORKLOAD", "tick"), choices=["tick", "lidar", "step", "episode", "race"])
    ap.add_argument("--cars", type=int, default=None)
    ap.add_argument("--settle", type=int, default=1000, help="untimed ticks before timing (SURVEY 8d config 3: 1 000 warm ticks)")
    ap.add_argument("--full-episode", action="store_true",
                    help="episode workload: run until every car of the rank has finished --lap-target laps or 25 000 ticks (SURVEY 8d config 4)")
    ap.add_argument("--lap-target", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fused-check", action="store_true", help="assert that ftgp_tick == the four separate calls, bit for bit")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the timed path computed in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has no such outputs")
    if args.cars is None:
        args.cars = {"lidar": 4096, "episode": 1048576, "race": 262144}.get(args.workload, 65536)
    if args.workload in ("episode", "race") and args.impl != "reference":
        return run_episode(args, args.workload)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
