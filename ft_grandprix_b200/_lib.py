"""ctypes loader for libftgp.so (C ABI declared in include/ftgp.h).

There is no CPU fallback: if the shared object is missing this raises, and every device
entry point fails with FTGP_ERR_CUDA on a machine without a GPU.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libftgp.so")

NBEAMS, NQ, NV, NU, NPATH = 90, 34, 29, 2, 100
MAX_TRACKS, MAX_LAPTIMES = 4, 16
LAP_FIELDS = ("offset", "completion", "laps", "start", "good_start", "finished", "ntimes",
              "off_track", "rank", "delta", "offtrack_ticks", "contact_ticks")
RACE_FIELDS = ("races", "finished", "wins", "rank_sum", "laps_sum", "time_sum", "best_lap", "offtrack_ticks",
               "contact_ticks")
DRIVER_NIDC, DRIVER_FAST, DRIVER_LOBOTOMY = 0, 1, 2
DRV_FIELDS = ("car_width", "safety_percentage", "difference_threshold", "speed", "speed_divisor", "max_steer",
              "boost_speed", "boost_max_steer", "boost_min_rear_range", "speed_cap")
OPT_NAIVE_FLATTEN, OPT_BUBBLE_WRAP = 1, 2

class FtgpError(RuntimeError):
    pass

class TickArgs(C.Structure):
    _fields_ = [("geom", C.c_void_p),
                ("qpos", C.c_void_p), ("qvel", C.c_void_p), ("warm", C.c_void_p), ("ctrl", C.c_void_p),
                ("ranges", C.c_void_p), ("track_id", C.c_void_p), ("driver_kind", C.c_void_p),
                ("lap", C.c_void_p), ("times", C.c_void_p), ("winners", C.c_void_p), ("status", C.c_void_p),
                ("ncars", C.c_int64),
                ("cars_per_world", C.c_int32), ("default_driver", C.c_int32),
                ("lap_target", C.c_int32), ("steps", C.c_int32), ("options", C.c_int32), ("reserved", C.c_int32)]

class ReloadArgs(C.Structure):
    _fields_ = [("start_xy", C.c_void_p), ("start_yaw", C.c_void_p), ("start_offset", C.c_void_p),
                ("race_start", C.c_void_p), ("tally", C.c_void_p), ("race_ticks", C.c_int32), ("reserved", C.c_int32)]

_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
# name -> (restype, argtypes); mirrors include/ftgp.h one to one
SIGNATURES = {
    "ftgp_last_error": (C.c_char_p, []),
    "ftgp_abi_version": (_i, []),
    "ftgp_launch_count": (_i64, []),
    "ftgp_track_create": (_vp, [_vp, _i, _i, _i, _d, _i]),
    "ftgp_track_destroy": (None, [_vp]),
    "ftgp_track_meta": (_i, [_vp, _vp, _vp]),
    "ftgp_track_chunks": (_i, [_vp, _vp, _vp]),
    "ftgp_centreline": (_i, [C.c_char_p, _i, _i, _i, _i, _i, _d, _vp]),
    "ftgp_geom_create": (_vp, [_vp, _vp, _i, _i]),
    "ftgp_geom_destroy": (None, [_vp]),
    "ftgp_geom_blob": (_i64, [_vp, _vp, _i, _vp, _i64]),
    "ftgp_blob_track_view": (_i, [_vp, _i, _vp, _vp]),
    "ftgp_geom_device": (_i, [_vp]),
    "ftgp_geom_bytes": (_i64, [_vp]),
    "ftgp_lidar": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _i, _vp, _vp, _vp]),
    "ftgp_lidar_host": (_i, [_vp, _vp, _i64, _vp, _i64, _vp]),
    "ftgp_reset": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ftgp_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _i, _vp]),
    "ftgp_release_scratch": (_i, [_vp]),
    "ftgp_naive_flatten": (_i, [_vp, _i64, _i64, _vp]),
    "ftgp_drivers": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _vp]),
    "ftgp_drivers_params": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i64, _vp]),
    "ftgp_lap_update": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _i, C.c_int32, C.c_int32, _vp]),
    "ftgp_tick": (_i, [C.POINTER(TickArgs), _i, _vp]),
    "ftgp_release_graphs": (_i, []),
    "ftgp_tick_use_graphs": (_i, [_i]),
    "ftgp_reload": (_i, [C.POINTER(TickArgs), C.POINTER(ReloadArgs), _vp]),
    "ftgp_tick_reload": (_i, [C.POINTER(TickArgs), C.POINTER(ReloadArgs), _i, _vp]),
    "ftgp_tick_params": (_i, [C.POINTER(TickArgs), C.POINTER(ReloadArgs), _vp, _i, _vp]),
}

_lib = None

def load():
    """Load libftgp.so or raise -- never falls back to another implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FtgpError(f"{LIB_PATH} is missing: build it with `python ft_grandprix_b200/build.py` "
                        "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib

def check(rc, what=""):
    if rc != 0:
        msg = load().ftgp_last_error()
        raise FtgpError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")

def last_error():
    msg = load().ftgp_last_error()
    return msg.decode() if msg else ""
