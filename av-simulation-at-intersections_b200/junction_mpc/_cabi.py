"""ctypes binding of libjmpc.so (include/jmpc.h).  No fallback: a missing library is an ImportError-grade failure."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JMPC_LIB", os.path.join(_HERE, "libjmpc.so"))

ABI_VERSION = 2
JMPC_MAX_T = 31
RECORD_LEN = 8
STATUS_OPTIMAL, STATUS_MAX_ITER, STATUS_INFEASIBLE, STATUS_INDEX_RULE = 0, 1, 2, 3
# enum jmpc_done: why an episode stopped
DONE_RUNNING, DONE_GOAL, DONE_INDEX_RULE, DONE_NO_COURSE, DONE_MATE_NO_COURSE = 0, 1, 2, 3, 4
# enum jmpc_right_of_way_rule
ROW_FIXED, ROW_FIRST_COME = 1, 2

c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)


class Options(C.Structure):
    _fields_ = [("max_solver_iters", C.c_int32), ("linearisation_iters", C.c_int32), ("mu_tol", C.c_double),
                ("warps_per_sm", C.c_int32), ("du_th", C.c_double)]


# name -> (restype, argtypes); the exported-symbol test walks this table against include/jmpc.h
SIGNATURES = {
    "jmpc_abi_version": (C.c_int32, []),
    "jmpc_nparam": (C.c_int32, []),
    "jmpc_last_error": (C.c_char_p, []),
    "jmpc_create": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                C.POINTER(Options), C.POINTER(C.c_void_p)]),
    "jmpc_destroy": (C.c_int32, [C.c_void_p]),
    "jmpc_set_default_params": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "jmpc_set_courses": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "jmpc_set_course_speed": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "jmpc_set_car_geometry": (C.c_int32, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "jmpc_step": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 17 + [C.c_void_p]),
    "jmpc_debug_cycles": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32]),
    "jmpc_set_schedule": (C.c_int32, [C.c_void_p, C.c_int32]),
    "jmpc_reset_schedule_hints": (C.c_int32, [C.c_void_p]),
    "jmpc_set_skip_mask": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "jmpc_set_record_peers": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]),
    "jmpc_set_record_flags": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_uint64]),
    "jmpc_gather_wait": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p]),
    "jmpc_gather_timed_out": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32)]),
    "jmpc_set_host_transfer": (C.c_int32, [C.c_void_p, C.c_int32]),
    "jmpc_step_host": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 17),
    "jmpc_step_host_io": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 20),
    "jmpc_host_alloc": (C.c_int32, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "jmpc_host_free": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "jmpc_collision": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "jmpc_collision_planned": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_void_p]
                               + [C.c_int32] * 4 + [C.c_double] + [C.c_void_p] * 4),
    "jmpc_collision_host": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "jmpc_plant_step": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "jmpc_episode_pre": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 7 + [C.c_double, C.c_double, C.c_void_p]),
    "jmpc_episode_post": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 10 + [C.c_double, C.c_void_p]),
    "jmpc_episode_post_dev": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 10 + [C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_double, C.c_void_p]),
    "jmpc_counter_add": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "jmpc_episode_outcomes": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
                              + [C.c_void_p] * 6 + [C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "jmpc_scene_exchange": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 9),
    "jmpc_scene_plans": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 6
                         + [C.c_int32, C.c_void_p, C.c_void_p]),
    "jmpc_scene_init": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "jmpc_right_of_way_init": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_void_p, C.c_void_p]),
    "jmpc_right_of_way": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 7),
    "jmpc_collision_masked": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_void_p]
                              + [C.c_int32] * 2 + [C.c_void_p] + [C.c_int32] * 2 + [C.c_double] + [C.c_void_p] * 4),
    "jmpc_obstacle_step": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "jmpc_scripted_obstacle_step": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_int32, C.c_void_p]),
    "jmpc_plan_host": (C.c_int32, [C.c_int32] * 5 + [C.c_void_p] * 3 + [C.c_int32] * 2 + [C.c_void_p] * 9 + [C.c_int32] * 3
                       + [C.c_void_p] * 10),
    "jmpc_planner_create": (C.c_int32, [C.c_int32] * 5 + [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.POINTER(C.c_void_p)]),
    "jmpc_planner_destroy": (C.c_int32, [C.c_void_p]),
    "jmpc_planner_set_scenes": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "jmpc_plan": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 16),
    "jmpc_set_courses_device": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 6),
    "jmpc_get_courses": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 4),
    "jmpc_get_arc_tables": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "jmpc_episode_init_from_courses": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_void_p] * 7),
    "jmpc_launch_count": (C.c_int64, [C.c_void_p]),
    "jmpc_measure_fma_peak": (C.c_int32, [C.c_void_p, c_f64p, c_f64p]),
    "jmpc_debug_linalg": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "jmpc_debug_linalg_g": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
}

_lib = None


class JmpcError(RuntimeError):
    pass


def load():
    """Load libjmpc.so once.  Raises if it has not been built (python __graft_entry__.py / build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise JmpcError(f"{LIB_PATH} not found: build it first (python -c 'import __graft_entry__ as g; g.build()'). "
                        "junction_mpc has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.jmpc_abi_version() != ABI_VERSION:
        raise JmpcError("libjmpc.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().jmpc_last_error()
        raise JmpcError(f"{what}: {msg.decode() if msg else 'error'} (rc={rc})")
