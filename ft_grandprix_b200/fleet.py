"""Fleet: the device-resident replacement for the reference's MjData + per-car VehicleState.

Mirrors what `Mujoco.physics_thread` touches every tick (ft_grandprix/custom.py:1337-1426):

    reference                                         here
    ------------------------------------------------  ---------------------------------------
    data.joint("car #i").qpos / .qvel                 fleet.qpos[i], fleet.qvel[i]   (fp64 rows)
    data.sensordata[vehicle_state.sensors]            fleet.ranges[i]                (fp32[90])
    data.ctrl[forward #i], data.ctrl[turn #i]         fleet.ctrl[i] = (speed, steering)
    vehicle_state.{laps,completion,finished,...}      fleet.lap[i]  (int32 fields, LAP_FIELDS)
    vehicle_state.times                               fleet.times[i] (lap durations in steps)
    self.winners                                      fleet.lap[:, rank] / fleet.winners[world]
    mujoco.mj_step(model, data)                       fleet.step()
    driver.process_lidar(ranges)                      fleet.drive() (device) / fleet.drive_host()
    the drivers' constants (nidc.py:5-10, fast.py:4-9) fleet.set_driver_params(rows): one row per car (DRV fields)
    reload() after every car has finished             Fleet(reload_finished=True): inside fleet.tick(), per world,
                                                      race results summed in fleet.race_tally (RACE_FIELDS)

All arithmetic runs in libftgp.so (hand-written sm_100a CUDA behind include/ftgp.h); torch only
owns the device memory and the stream.  There is no CPU fallback: constructing a Fleet without a
CUDA device raises.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import (DRIVER_FAST, DRIVER_LOBOTOMY, DRIVER_NIDC, DRV_FIELDS, LAP_FIELDS, MAX_LAPTIMES, NBEAMS, NQ, NU, NV,
                   RACE_FIELDS)
from .drivers import BatchedFastDriver, BatchedNidcDriver
from .track import Geometry, Track
from .vehicle import VehicleStateSnapshot

TIMESTEP = 0.004                      # template/mushr.em.xml:30
LAP = {name: k for k, name in enumerate(LAP_FIELDS)}
RACE = {name: k for k, name in enumerate(RACE_FIELDS)}
DRV = {name: k for k, name in enumerate(DRV_FIELDS)}
DRIVER_KINDS = {"nidc": DRIVER_NIDC, "fast": DRIVER_FAST, "lobotomy": DRIVER_LOBOTOMY,
                "ft_grandprix.nidc": DRIVER_NIDC, "ft_grandprix.fast": DRIVER_FAST,
                "ft_grandprix.lobotomy": DRIVER_LOBOTOMY}

def default_driver_params(kind):
    """The reference parameter row (DRV fields, include/ftgp.h FTGP_DRV_*) of a bundled driver: 'nidc' or 'fast' (or
    DRIVER_NIDC / DRIVER_FAST), as a float64 numpy array [10]."""
    k = DRIVER_KINDS[kind] if isinstance(kind, str) else int(kind)
    if k not in (DRIVER_NIDC, DRIVER_FAST):
        raise ValueError("only the nidc and fast drivers have a parameter row")
    return np.array((BatchedNidcDriver if k == DRIVER_NIDC else BatchedFastDriver).default_row(), dtype=np.float64)

def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None

class Fleet:
    def __init__(self, tracks, ncars, cars_per_world=1, device=0, track_id=None, driver="nidc",
                 lap_target=10, naive_flatten=False, bubble_wrap=False, reload_finished=False, race_ticks=0):
        """lap_target, naive_flatten, bubble_wrap: the path-relevant options of the reference (custom.py:961,981,970).
        reload_finished: race after race on the device.  At the head of every tick a world whose cars have all finished,
        or whose race has run race_ticks ticks (race_ticks > 0), is reloaded (custom.py:1089-1128) from the next-start
        tensors (set_next_start(); by default the poses of the last reset()), and the race that ended is added to
        race_tally[car] (RACE fields).  The other worlds go on racing."""
        if not torch.cuda.is_available():
            raise _lib.FtgpError("Fleet needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", int(device))
        self.geom = tracks if isinstance(tracks, Geometry) else Geometry(tracks, device=int(device))
        self.ncars, self.cars_per_world = int(ncars), int(cars_per_world)
        if self.ncars % self.cars_per_world:
            raise ValueError("ncars must be a multiple of cars_per_world")
        self.nworlds = self.ncars // self.cars_per_world
        self.lap_target = int(lap_target)
        self.reload_finished = bool(reload_finished)
        self.race_ticks = int(race_ticks)
        if self.race_ticks < 0:
            raise ValueError("race_ticks must be >= 0")
        self.naive_flatten = bool(naive_flatten)
        self.bubble_wrap = bool(bubble_wrap)
        self.default_driver = DRIVER_KINDS[driver] if isinstance(driver, str) else int(driver)
        dev, n = self.device, self.ncars
        with torch.cuda.device(dev):
            self.stream = torch.cuda.Stream(device=dev)
        self.qpos = torch.zeros(n, NQ, dtype=torch.float64, device=dev)
        self.qvel = torch.zeros(n, NV, dtype=torch.float64, device=dev)
        self.warm = torch.zeros(n, NV, dtype=torch.float64, device=dev)
        self.ctrl = torch.zeros(n, NU, dtype=torch.float64, device=dev)
        self.ranges = torch.zeros(n, NBEAMS, dtype=torch.float32, device=dev)   # zeros on the first tick (B.11)
        self.lap = torch.zeros(n, len(LAP_FIELDS), dtype=torch.int32, device=dev)
        self.times = torch.zeros(n, MAX_LAPTIMES, dtype=torch.int32, device=dev)
        self.winners = torch.zeros(self.nworlds, dtype=torch.int32, device=dev)
        self.status = torch.zeros(n, dtype=torch.int32, device=dev)
        self.track_id = None if track_id is None else torch.as_tensor(track_id, dtype=torch.int32).to(dev).contiguous()
        self.driver_kind = None
        self.driver_params = None            # [ncars, len(DRV)] float64 rows (set_driver_params), None = reference constants
        self._driver_params = None           # the rows' storage, allocated once (the tick's graph key holds its address)
        self.steps = 0
        if self.reload_finished:
            self.race_tally = torch.zeros(n, len(RACE_FIELDS), dtype=torch.int32, device=dev)
            self.race_start = torch.zeros(self.nworlds, dtype=torch.int32, device=dev)   # tick at which the world's race began
            self.start_xy = torch.zeros(n, 2, dtype=torch.float64, device=dev)           # the next race's start grid
            self.start_yaw = torch.zeros(n, dtype=torch.float64, device=dev)
            self.start_offset = self._grid_offsets()
        # options manual_control / always_invoke_driver / detach_control of the loop's driver block (custom.py:952-957,1401-1423)
        self.manual_control = False          # the watched car takes (speed, steering) from the operator
        self.always_invoke_driver = True     # ... while the drivers are still invoked (reference default)
        self.detach_control = False          # drivers run, data.ctrl is not written
        self.watching = None                 # car id (custom.py: self.watching)
        self.manual_speed, self.manual_steering = 0.0, 0.0        # self.mv.speed, self.mv.steering_angle
        self.driver_out = None               # [ncars, 2]: vehicle_state.speed / steering_angle of the last tick (only kept with the options on)
        torch.cuda.synchronize(dev)

    @property
    def options(self):
        return (_lib.OPT_NAIVE_FLATTEN if self.naive_flatten else 0) | (_lib.OPT_BUBBLE_WRAP if self.bubble_wrap else 0)

    def close(self):
        """Free the step kernel's per-stream scratch (about 6 KB per car)."""
        if getattr(self, "stream", None) is not None and getattr(self, "lib", None) is not None:
            with torch.cuda.device(self.device):
                self.stream.synchronize()
                self.lib.ftgp_release_scratch(self._s)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    @property
    def _s(self):
        return C.c_void_p(self.stream.cuda_stream)

    def sync(self):
        self.stream.synchronize()

    def set_driver_kinds(self, kinds):
        """Per-car built-in driver: names ('nidc', 'fast', 'lobotomy') or FTGP_DRIVER_* ints."""
        k = [DRIVER_KINDS[x] if isinstance(x, str) else int(x) for x in kinds]
        self.driver_kind = torch.tensor(k, dtype=torch.int32, device=self.device)

    def set_driver_params(self, rows):
        """Per-car constants of the device drivers: rows [ncars, len(DRV)] (or one row [len(DRV)] for every car), float64,
        fields DRV (default_driver_params(kind) gives the reference rows).  With rows, a car's row alone decides its
        disparity extender and speed law; driver kinds then only matter as 'lobotomy', and finished cars are still
        lobotomised.  None returns to the reference constants of each car's kind.  The rows are copied into
        fleet.driver_params in stream order (ticks already issued read the old rows); that tensor keeps its address, so
        a graph-replayed tick reads new rows without a recapture, and writing into it in place on fleet.stream works
        as well."""
        if rows is None:
            self.driver_params = None
            return
        rows = torch.as_tensor(rows, dtype=torch.float64, device=self.device)
        if rows.shape not in ((len(DRV),), (self.ncars, len(DRV))):
            raise ValueError(f"rows must be [ncars, {len(DRV)}] or [{len(DRV)}]")
        if self._driver_params is None:
            self._driver_params = torch.empty(self.ncars, len(DRV), dtype=torch.float64, device=self.device)
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.stream):
            self._driver_params.copy_(rows.expand(self.ncars, -1))
        rows.record_stream(self.stream)
        self.driver_params = self._driver_params

    def _grid_offsets(self):
        """VehicleState(offset=(i+5)*2) of grid slot i (custom.py:96-118)."""
        idx = torch.arange(self.ncars, device=self.device, dtype=torch.int32) % self.cars_per_world
        return (idx + 5) * 2

    # ------------------------------------------------------------------ reset (custom.py:1089-1128,1232-1245)
    def reset(self, xy, yaw):
        xy = torch.as_tensor(np.asarray(xy, dtype=np.float64)).to(self.device).contiguous()
        yaw = torch.as_tensor(np.asarray(yaw, dtype=np.float64)).to(self.device).contiguous()
        if xy.shape != (self.ncars, 2) or yaw.shape != (self.ncars,):
            raise ValueError("xy must be [ncars,2] and yaw [ncars]")
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        _lib.check(self.lib.ftgp_reset(_ptr(self.qpos), _ptr(self.qvel), _ptr(self.warm), _ptr(self.ctrl),
                                       _ptr(xy), _ptr(yaw), self.ncars, self._s), "ftgp_reset")
        with torch.cuda.stream(self.stream):
            self.ranges.zero_(); self.lap.zero_(); self.times.zero_(); self.winners.zero_(); self.status.zero_()
            # VehicleState(offset=(i+5)*2) with good_start=True (custom.py:96-118)
            self.lap[:, LAP["offset"]] = self._grid_offsets()
            self.lap[:, LAP["good_start"]] = 1
            if self.reload_finished:                  # the default next start; a reset begins a new series
                self.start_xy.copy_(xy); self.start_yaw.copy_(yaw)
                self.start_offset.copy_(self.lap[:, LAP["offset"]])
                self.race_start.zero_(); self.race_tally.zero_()
        self.steps = 0
        self.sync()
        self._keep = (xy, yaw)

    def reset_grid(self):
        """The reference start grid: car i of each world at path[(i+5)*2] (custom.py:1232-1245)."""
        slot = np.arange(self.ncars) % self.cars_per_world
        tid = np.zeros(self.ncars, dtype=np.int64) if self.track_id is None else self.track_id.cpu().numpy().astype(np.int64)
        xy = np.zeros((self.ncars, 2)); yaw = np.zeros(self.ncars)
        for k, t in enumerate(self.geom.tracks):
            poses = np.array([t.start_pose(i) for i in range(self.cars_per_world)])      # (x, y, yaw) per grid slot
            sel = tid == k
            xy[sel] = poses[slot[sel], :2]; yaw[sel] = poses[slot[sel], 2]
        self.reset(xy, yaw)

    # ------------------------------------------------------------------ race after race (reload_finished)
    def set_next_start(self, xy, yaw, offset=None):
        """Start poses ([ncars, 2], [ncars]) and lap offsets ([ncars]; default: the grid slot's (slot+5)*2, as reset()
        sets it) of the next race of every world.  They are read when a world is reloaded, so a caller may rewrite them
        between ticks, e.g. grid poses plus seeded jitter: device drivers are deterministic, and a world reloaded from an
        unchanged start runs the same race again."""
        self._need_reload("set_next_start")
        xy = torch.as_tensor(xy, dtype=torch.float64, device=self.device)
        yaw = torch.as_tensor(yaw, dtype=torch.float64, device=self.device)
        off = self._grid_offsets() if offset is None else torch.as_tensor(offset, dtype=torch.int32, device=self.device)
        if xy.shape != (self.ncars, 2) or yaw.shape != (self.ncars,) or off.shape != (self.ncars,):
            raise ValueError("xy must be [ncars,2], yaw and offset [ncars]")
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.stream):            # in stream order: ticks already issued read the old starts
            self.start_xy.copy_(xy); self.start_yaw.copy_(yaw); self.start_offset.copy_(off)
        for t in (xy, yaw, off):
            t.record_stream(self.stream)

    def _need_reload(self, what):
        if not self.reload_finished:
            raise ValueError(f"{what} needs Fleet(..., reload_finished=True)")

    def reload_args(self):
        self._need_reload("reload_args")
        r = _lib.ReloadArgs()
        r.start_xy, r.start_yaw, r.start_offset = (self.start_xy.data_ptr(), self.start_yaw.data_ptr(),
                                                   self.start_offset.data_ptr())
        r.race_start, r.tally = self.race_start.data_ptr(), self.race_tally.data_ptr()
        r.race_ticks = self.race_ticks
        return r

    def reload(self):
        """Reload the worlds whose race is over, now (the piece fleet.tick() runs at the head of every tick, for loops
        that issue the tick's pieces one by one: reload -> lap_update -> drive -> lidar -> step)."""
        a, r = self.tick_args(), self.reload_args()
        _lib.check(self.lib.ftgp_reload(C.byref(a), C.byref(r), self._s), "ftgp_reload")

    # ------------------------------------------------------------------ the per-tick pieces
    def lidar(self, visible=None, min_range=None, shadow_finished=True, qpos=None, stream=None):
        """data.sensordata[vehicle_state.sensors] for every car (custom.py:1395).  Finished cars are shadowed as in
        the reference (stale ranges, invisible to the others) unless shadow_finished is False.  qpos / stream: scan a copy
        of the poses on another stream (tick_readback runs the scan beside the vehicle step that way)."""
        _lib.check(self.lib.ftgp_lidar(self.geom._ptr, _ptr(self.qpos if qpos is None else qpos), NQ, _ptr(self.track_id),
                                       _ptr(visible), _ptr(self.lap) if shadow_finished else None,
                                       self.ncars, self.cars_per_world, _ptr(self.ranges), _ptr(min_range),
                                       self._s if stream is None else C.c_void_p(stream.cuda_stream)), "ftgp_lidar")
        return self.ranges

    def _control_options(self):
        return self.manual_control or self.detach_control

    def set_manual_control(self, on, watching=None, speed=0.0, steering_angle=0.0, always_invoke_driver=True):
        """Options manual_control / always_invoke_driver (custom.py:954-957): the watched car is driven by (speed,
        steering_angle) -- the reference's keyboard state self.mv -- instead of its driver."""
        self.manual_control = bool(on)
        self.watching = None if watching is None else int(watching)
        self.manual_speed, self.manual_steering = float(speed), float(steering_angle)
        self.always_invoke_driver = bool(always_invoke_driver)

    def drive(self):
        """Built-in batched drivers + control write (custom.py:1398-1423), with the options of that block:
        `always_invoke_driver or not manual_control` decides whether the drivers run at all (else (0, 0)); under
        manual_control the watched car takes the operator's (speed, steering), and a released throttle decays
        (speed = ctrl * 0.99 while ctrl > 0, custom.py:1413-1416); under detach_control the result goes to
        vehicle_state.speed / steering_angle (driver_out) only and data.ctrl keeps its values (custom.py:1421-1423)."""
        special = self._control_options()
        if special:
            with torch.cuda.stream(self.stream):
                prev = self.ctrl.clone()
        if self.always_invoke_driver or not self.manual_control:
            _lib.check(self.lib.ftgp_drivers_params(_ptr(self.ranges), _ptr(self.driver_kind), self.default_driver,
                                                    _ptr(self.driver_params), _ptr(self.lap), _ptr(self.ctrl), self.ncars,
                                                    self._s), "ftgp_drivers_params")
        else:
            with torch.cuda.stream(self.stream):
                self.ctrl.zero_()
        if special:
            with torch.cuda.stream(self.stream):
                if self.manual_control and self.watching is not None:
                    w = self.watching
                    if self.manual_speed == 0.0:
                        sp = torch.where(prev[w, 0] > 0.0, prev[w, 0] * 0.99, torch.zeros_like(prev[w, 0]))
                    else:
                        sp = torch.full_like(prev[w, 0], self.manual_speed)
                    self.ctrl[w, 0] = sp
                    self.ctrl[w, 1] = self.manual_steering
                self.driver_out = self.ctrl.clone()
                if self.detach_control:
                    self.ctrl.copy_(prev)
        return self.ctrl

    def drive_host(self, drivers):
        """Slow path for unmodified reference-style drivers (SURVEY §8 B1): one Python object per car
        with process_lidar(ranges) or process_lidar(ranges, state); exceptions are printed and leave
        that car's ctrl unchanged (custom.py:1403-1411).  fleet.driver_params is ignored: host drivers carry their
        own constants."""
        import inspect
        self.sync()
        ranges = self.ranges.cpu().numpy().astype(np.float64)
        ctrl = self.ctrl.cpu().numpy()
        finished = self.lap[:, LAP["finished"]].cpu().numpy()
        snaps = None
        prev = ctrl.copy()
        invoke = self.always_invoke_driver or not self.manual_control        # custom.py:1403
        for i, d in enumerate(drivers):
            if finished[i] or not invoke:            # shadow() swapped in LobotomyDriver (custom.py:1437) / nobody is asked
                ctrl[i] = (0.0, 0.0)
                continue
            try:
                if len(inspect.signature(d.process_lidar).parameters) >= 2:   # v2 driver (custom.py:103)
                    if snaps is None:
                        snaps = self.snapshots()
                    sp, st = d.process_lidar(ranges[i].copy(), snaps[i])
                else:
                    sp, st = d.process_lidar(ranges[i].copy())
                ctrl[i] = (float(sp), float(st))
            except Exception as e:                                          # custom.py:1409-1411
                print(f"Error in vehicle `{i}`: `{e}`")
        if self.manual_control and self.watching is not None:               # custom.py:1413-1416
            w = self.watching
            sp = self.manual_speed
            if sp == 0.0 and prev[w, 0] > 0.0:
                sp = prev[w, 0] * 0.99
            ctrl[w] = (sp, self.manual_steering)
        if self._control_options():
            self.driver_out = torch.from_numpy(ctrl.copy()).to(self.device)
        if self.detach_control:                                             # custom.py:1421-1423
            ctrl = prev
        self.ctrl.copy_(torch.from_numpy(ctrl))
        return self.ctrl

    def step(self, nsteps=1, shadow_finished=True):
        """mujoco.mj_step(model, data) (custom.py:1425).  Finished cars are shadow()ed as in the reference
        (custom.py:1455-1464: they pass through walls) unless shadow_finished is False."""
        _lib.check(self.lib.ftgp_step(self.geom._ptr, _ptr(self.qpos), _ptr(self.qvel), _ptr(self.warm),
                                      _ptr(self.ctrl), _ptr(self.track_id),
                                      _ptr(self.lap) if shadow_finished else None, self.ncars, self.cars_per_world,
                                      int(nsteps), _ptr(self.status), self.options, self._s), "ftgp_step")
        self.steps += int(nsteps)

    def flatten(self):
        """Option naive_flatten (custom.py:1338-1339): keep the chassis' yaw, zero its pitch and roll."""
        _lib.check(self.lib.ftgp_naive_flatten(_ptr(self.qpos), NQ, self.ncars, self._s), "ftgp_naive_flatten")

    def lap_update(self):
        """Progress / lap state machine (custom.py:1340-1372); with the option naive_flatten the flattening that precedes it
        in the reference's loop body (custom.py:1338-1339)."""
        if self.naive_flatten:
            self.flatten()
        _lib.check(self.lib.ftgp_lap_update(self.geom._ptr, _ptr(self.qpos), NQ, _ptr(self.track_id),
                                            _ptr(self.lap), _ptr(self.times), _ptr(self.winners),
                                            _ptr(self.status), self.ncars, self.cars_per_world, self.steps,
                                            self.lap_target, self._s), "ftgp_lap_update")

    def tick_args(self):
        a = _lib.TickArgs()
        a.geom = self.geom._ptr
        a.qpos, a.qvel, a.warm, a.ctrl = (self.qpos.data_ptr(), self.qvel.data_ptr(), self.warm.data_ptr(),
                                          self.ctrl.data_ptr())
        a.ranges = self.ranges.data_ptr()
        a.track_id = None if self.track_id is None else self.track_id.data_ptr()
        a.driver_kind = None if self.driver_kind is None else self.driver_kind.data_ptr()
        a.lap, a.times, a.winners, a.status = (self.lap.data_ptr(), self.times.data_ptr(),
                                               self.winners.data_ptr(), self.status.data_ptr())
        a.ncars = self.ncars
        a.cars_per_world, a.default_driver = self.cars_per_world, self.default_driver
        a.lap_target, a.steps = self.lap_target, self.steps
        a.options = self.options
        return a

    def tick(self, nticks=1):
        """nticks iterations of the physics loop (custom.py:1337-1426), all on device."""
        if self._control_options():                   # operator options: the driver block needs the host's say every tick
            for _ in range(int(nticks)):
                if self.reload_finished:
                    self.reload()
                self.lap_update(); self.drive(); self.lidar(); self.step(1)
            return
        a = self.tick_args()
        r = C.byref(self.reload_args()) if self.reload_finished else None
        _lib.check(self.lib.ftgp_tick_params(C.byref(a), r, _ptr(self.driver_params), int(nticks), self._s),
                   "ftgp_tick_params")
        self.steps += int(nticks)

    def tick_readback(self, ranges_host, lap_host, cars=None):
        """One iteration of the physics loop with this tick's ranges and lap state delivered to pinned host buffers
        (ranges_host = None: lap state only; cars = (lo, hi): only that slice of the fleet's ranges, e.g. the cars a host
        driver or a viewer is interested in -- at 1 M cars the full ranges tensor is 94 % of the per-tick PCIe traffic),
        the copies overlapped with the kernels that do not touch those arrays: the lap state leaves right after the
        lap kernel, the ranges right after the lidar kernel (the vehicle step runs meanwhile), and only the NEXT
        tick's lidar / lap kernels wait for the copies.  Call sync_readback() before reading the host buffers."""
        if not hasattr(self, "_copy_stream"):
            with torch.cuda.device(self.device):
                self._copy_stream = torch.cuda.Stream(device=self.device)
                self._scan_stream = torch.cuda.Stream(device=self.device)
            self._ev = [torch.cuda.Event() for _ in range(5)]      # lap ready, ranges ready, lap copied, ranges copied, poses copied
            self._ev[2].record(self._copy_stream); self._ev[3].record(self._copy_stream)
            self._qpos_scan = torch.empty_like(self.qpos)
        s, c, l = self.stream, self._copy_stream, self._scan_stream
        lap_ready, ranges_ready, lap_copied, ranges_copied, poses_copied = self._ev
        with torch.cuda.stream(s):
            s.wait_event(lap_copied)                 # the previous copy of the lap state has left
            if self.reload_finished:
                s.wait_event(ranges_copied)          # ... and of the ranges: a reload writes both
                self.reload()
            self.lap_update()
            lap_ready.record(s)
            self.drive()
            # the rangefinders see the pre-step pose (custom.py:1425): they scan a copy of it on their own stream while
            # the vehicle step advances the state on this one (as ftgp_tick does, DESIGN.md 3.3b)
            self._qpos_scan.copy_(self.qpos, non_blocking=True)
            poses_copied.record(s)
        with torch.cuda.stream(l):
            l.wait_event(poses_copied)
            if ranges_host is not None:
                l.wait_event(ranges_copied)          # ... and the previous copy of the ranges
            self.lidar(qpos=self._qpos_scan, stream=l)
            ranges_ready.record(l)
        with torch.cuda.stream(s):
            self.step(1)
            s.wait_event(ranges_ready)               # join: the next tick's drivers read these ranges
        with torch.cuda.stream(c):
            c.wait_event(lap_ready)
            lap_host.copy_(self.lap, non_blocking=True)
            lap_copied.record(c)
            if ranges_host is not None:
                c.wait_event(ranges_ready)
                src = self.ranges if cars is None else self.ranges[cars[0]:cars[1]]
                ranges_host.copy_(src, non_blocking=True)
                ranges_copied.record(c)

    def sync_readback(self):
        self.stream.synchronize()
        if hasattr(self, "_copy_stream"):
            self._scan_stream.synchronize()
            self._copy_stream.synchronize()

    # ------------------------------------------------------------------ v2 driver input (custom.py:149-160)
    def snapshots(self):
        self.sync()
        qpos = self.qpos.cpu().numpy(); qvel = self.qvel.cpu().numpy(); lap = self.lap.cpu().numpy()
        out = []
        for i in range(self.ncars):
            w, x, y, z = qpos[i, 3:7]
            # quaternion_to_euler (custom.py:62-76)
            roll = math.atan2(2 * (w * x + y * z), 1 - 2 * (x * x + y * y))
            t2 = max(-1.0, min(1.0, 2 * (w * y - z * x)))
            pitch = math.asin(t2)
            yaw = math.atan2(2 * (w * z + x * y), 1 - 2 * (y * y + z * z))
            comp = int(lap[i, LAP["completion"]])
            lap_completion = comp if lap[i, LAP["good_start"]] else comp - 100      # custom.py:132-140
            laps = int(lap[i, LAP["laps"]])
            out.append(VehicleStateSnapshot(laps=laps, velocity=qvel[i, 0:3], yaw=yaw, pitch=pitch, roll=roll,
                                            lap_completion=lap_completion,
                                            absolute_completion=laps * 100 + lap_completion,
                                            time=self.steps / TIMESTEP))          # custom.py:1397 (sic)
        return out

    def snapshot_tensors(self):
        """The fields of VehicleStateSnapshot (ft_grandprix/vehicle.py:3-12, custom.py:132-160) for the whole fleet as
        device tensors, for batched v2 drivers `process_lidar(ranges, state)`: nothing leaves the GPU.  `velocity`
        aliases fleet.qvel like the reference's view of `joint.qvel[0:3]`."""
        with torch.cuda.stream(self.stream):
            w, x, y, z = (self.qpos[:, 3], self.qpos[:, 4], self.qpos[:, 5], self.qpos[:, 6])
            # quaternion_to_euler (custom.py:62-76): ZYX, asin clamped to +-1
            roll = torch.atan2(2 * (w * x + y * z), 1 - 2 * (x * x + y * y))
            pitch = torch.asin(torch.clamp(2 * (w * y - z * x), -1.0, 1.0))
            yaw = torch.atan2(2 * (w * z + x * y), 1 - 2 * (y * y + z * z))
            comp = self.lap[:, LAP["completion"]]
            lap_completion = torch.where(self.lap[:, LAP["good_start"]] != 0, comp, comp - 100)   # custom.py:132-140
            laps = self.lap[:, LAP["laps"]]
            return {"laps": laps, "velocity": self.qvel[:, 0:3], "yaw": yaw, "pitch": pitch, "roll": roll,
                    "lap_completion": lap_completion, "absolute_completion": laps * 100 + lap_completion,
                    "time": self.steps / TIMESTEP}                                            # custom.py:1397 (sic)

    def _state_keys(self):
        keys = ("qpos", "qvel", "warm", "ctrl", "ranges", "lap", "times", "winners", "status")
        if self.reload_finished:
            keys += ("race_tally", "race_start", "start_xy", "start_yaw", "start_offset")
        return keys

    def state_dict(self):
        """The fleet's arrays on the host, with driver_params when rows are set."""
        self.sync()
        sd = {k: getattr(self, k).cpu() for k in self._state_keys()} | {"steps": self.steps}
        if self.driver_params is not None:
            sd["driver_params"] = self.driver_params.cpu()
        return sd

    def load_state_dict(self, sd):
        for k in self._state_keys():
            getattr(self, k).copy_(sd[k])
        self.set_driver_params(sd.get("driver_params"))
        self.steps = int(sd["steps"])
