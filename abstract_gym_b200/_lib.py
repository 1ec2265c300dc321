"""ctypes binding of the C ABI declared in include/abstract_gym_b200.h.

There is no CPU implementation behind this module: if the CUDA extension is missing and cannot be
built, importing it raises; if no CUDA device is present, the device entry points return a CUDA
error which `check` turns into an exception.
"""
import ctypes as C
import os

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))

ABI_VERSION = 9
ENGINE_EXACT, ENGINE_FAST, ENGINE_BRUTE = 0, 1, 2
ENGINES = {"exact": ENGINE_EXACT, "fast": ENGINE_FAST, "brute": ENGINE_BRUTE}
FLAG_COLLISION, FLAG_DONE = 1, 2
ST_EPISODES, ST_COLLISIONS, ST_SUCCESSES, ST_ENV_STEPS, ST_EP_LEN_SUM, ST_RETURN_MILLI, \
    ST_STUCK_RESETS, ST_AXIS_ALIGNED, ST_COUNT = range(9)
DIAG_NAMES = ("exact_steps", "cold_calls", "warp_exits")
STAT_NAMES = ("episodes", "collisions", "successes", "env_steps", "ep_len_sum", "return_milli",
              "stuck_resets", "axis_aligned")


class AgError(RuntimeError):
    def __init__(self, status, what):
        self.status = status
        super().__init__("%s failed: status %d (%s)" % (what, status, status_string(status)))


class Params(C.Structure):
    """ag_params: the literals of scenario/scene_0.py, collision_checker.py:81, two_joint_robot.py:12-13."""
    _fields_ = [("link_1", C.c_double), ("link_2", C.c_double),
                ("target_x", C.c_double), ("target_y", C.c_double),
                ("target_j1", C.c_double), ("target_j2", C.c_double),
                ("reach_eps", C.c_double), ("section_eps", C.c_double),
                ("reward_collision", C.c_double), ("reward_reach", C.c_double),
                ("action_scale", C.c_double),
                ("choose_j_tar", C.c_int32), ("max_reset_tries", C.c_int32)]


class Grid(C.Structure):
    """ag_grid"""
    _fields_ = [("bits", C.c_void_p), ("min_x", C.c_void_p), ("min_y", C.c_void_p),
                ("side", C.c_double), ("env_size", C.c_double),
                ("S", C.c_int32), ("words_per_row", C.c_int32), ("n_grids", C.c_int32), ("max_occupied", C.c_int32),
                ("grid_stride_words", C.c_int64), ("envs_per_grid", C.c_int64), ("bits_t", C.c_void_p),
                ("hier", C.c_void_p)]


class RolloutArgs(C.Structure):
    """ag_rollout_args"""
    _fields_ = [("n", C.c_int64), ("env_id0", C.c_int64), ("K", C.c_int32), ("engine", C.c_int32),
                ("seed", C.c_uint64), ("actions", C.c_void_p), ("reset_u", C.c_void_p),
                ("R", C.c_int32), ("reserved", C.c_int32),
                ("j1", C.c_void_p), ("j2", C.c_void_p), ("reward", C.c_void_p), ("flags", C.c_void_p),
                ("step_ctr", C.c_void_p), ("reset_ctr", C.c_void_p), ("ep_len", C.c_void_p),
                ("rec_j1", C.c_void_p), ("rec_j2", C.c_void_p), ("rec_reward", C.c_void_p),
                ("rec_flags", C.c_void_p), ("stats", C.c_void_p), ("diag", C.c_void_p), ("targets", C.c_void_p),
                ("events", C.c_void_p), ("event_count", C.c_void_p), ("event_capacity", C.c_int64),
                ("event_step0", C.c_int32), ("reserved2", C.c_int32)]


# every symbol include/abstract_gym_b200.h declares: (restype, argtypes)
_vp, _i32, _i64, _u64, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
SYMBOLS = {
    "ag_abi_version": (_i32, []),
    "ag_status_string": (C.c_char_p, [_i32]),
    "ag_default_params": (None, [C.POINTER(Params)]),
    "ag_grid_words_per_row": (_i32, [_i32]),
    "ag_grid_stride_words": (_i64, [_i32]),
    "ag_grid_pack_host": (_i32, [_vp, _i32, _i32, _vp]),
    "ag_grid_tables_host": (_i32, [_i32, _dbl, _vp, _vp, C.POINTER(_dbl)]),
    "ag_grid_pack": (_i32, [_vp, _i32, _i32, _vp, _i64, _vp]),
    "ag_segment_square": (_i32, [_vp, _vp, _dbl, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ag_forward_kinematics": (_i32, [C.POINTER(Params), _vp, _vp, _vp, _i64, _vp]),
    "ag_inverse_kinematics": (_i32, [C.POINTER(Params), _vp, _vp, _vp, _i32, _i64, _vp]),
    "ag_move_to_joint_pose": (_i32, [_vp, _vp, _vp, _i32, _i64, _vp]),
    "ag_collision_check": (_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp]),
    "ag_check_motion": (_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp]),
    "ag_cspace_occupancy": (_i32, [C.POINTER(Params), C.POINTER(Grid), _dbl, _dbl, _i32, _dbl, _dbl, _i32, _vp, _vp, _i32, _vp]),
    "ag_cspace_components": (_i32, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp]),
    "ag_cspace_distance": (_i32, [_vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp]),
    "ag_cspace_descend": (_i32, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "ag_step":(_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                       _i64, _i64, _i32, _vp]),
    "ag_reset": (_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _u64, _i32,
                        _vp, _i64, _i64, _i32, _vp]),
    "ag_step_obs": (_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                           _vp, _vp, _i32, _vp, _u64, _i32, _i64, _i64, _i32, _vp]),
    "ag_rollout": (_i32, [C.POINTER(Params), C.POINTER(Grid), C.POINTER(RolloutArgs), _vp]),
    "ag_launch_count": (_i64, []),
    "ag_grid_hier_bytes": (_i64, [_i32]),
    "ag_grid_pack_hier": (_i32, [_vp, _i32, _i32, _i64, _vp, _vp]),
    "ag_cspace_map_words": (_i64, [C.POINTER(_i32), C.POINTER(_i32)]),
    "ag_cspace_map": (_i32, [C.POINTER(Params), C.POINTER(Grid), _vp, _vp]),
    "ag_pipeline_create": (_i32, [C.POINTER(_vp), _i32, _i64, _i32, _i64, _i32, _i32, _i64]),
    "ag_pipeline_destroy": (None, [_vp]),
    "ag_rollout_host": (_i32, [_vp, C.POINTER(Params), C.POINTER(Grid), C.POINTER(RolloutArgs), _vp]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building in-tree if needed) libabstract_gym_b200.so.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path) or _build.needs_build():
        try:
            _build.build()
        except Exception as e:  # never run a stale binary silently: the sources are newer than the library
            raise ImportError("abstract_gym_b200: the CUDA extension %s is %s and could not be built (%s). "
                              "There is no CPU fallback." % (path, "stale" if os.path.exists(path) else "missing", e)) from e
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:   # an older build of the library: never run it
            raise ImportError("abstract_gym_b200: %s does not export %s (include/abstract_gym_b200.h declares it): the "
                              "library is older than the package; rebuild it with `python abstract_gym_b200/build.py "
                              "--force`" % (path, name)) from e
        fn.restype, fn.argtypes = res, args
    if lib.ag_abi_version() != ABI_VERSION:
        raise ImportError("abstract_gym_b200: ABI version mismatch")
    _lib = lib
    return lib


def status_string(status: int) -> str:
    return load().ag_status_string(status).decode()


def check(status: int, what: str):
    if status != 0:
        raise AgError(status, what)


def default_params() -> Params:
    p = Params()
    load().ag_default_params(C.byref(p))
    return p


def launch_count() -> int:
    return int(load().ag_launch_count())
