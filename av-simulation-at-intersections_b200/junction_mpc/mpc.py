"""Drop-in replacement of the reference's `lib.mpc` module (main/lib/mpc.py), backed by libjmpc.so.

Everything a scenario runner touches keeps its name, signature and types (SURVEY.md section 8b):

    from lib.mpc import MPC, MAX_ACCEL                                   mpc_intersection.py:20
    mpc = MPC(cx=..., cy=..., cyaw=..., dl=..., dt=DT, car_dimensions=..., speed=30/3.6)     mpc.py:246-247
    mpc.set_trajectory_fromarray(tmp_trajectory)                          mpc.py:279-282
    delta, acceleration = mpc.step(state)                                 mpc.py:284-303
    mpc.get_current_xref_deviation(); mpc.is_goal(state)                  mpc.py:305-330
    mpc.ox, mpc.oy, mpc.xref, mpc.di                                      mpc_intersection.py:301-306

A single ego is a batch of one: `step` runs the same CUDA kernel as `BatchedMPC` through `jmpc_step_host_io`.
`install()` registers this module as `lib.mpc` (and the sensitivity / speed-profile flavours as
`lib.mpc_sensitivity` / `lib.mpc_with_speed`) so the
reference's scenario scripts run unmodified; see INTEGRATION.md.
"""
from __future__ import annotations

import math
import os
import sys
import types
from typing import List, Optional, Tuple

import numpy as np

from . import _cabi
from .batched import BatchedMPC
from .config import MPCConfig, SIM_MAX_SPEED

# ---- module-level configuration, as main/lib/mpc.py:14-39 exposes it --------------------------------------
_config_path = os.environ.get("JMPC_CONFIG")
_cfg = MPCConfig.from_json(_config_path) if _config_path else MPCConfig.default()

NX, NU, T = _cfg.nx, _cfg.nu, _cfg.T
w_perp, w_para = _cfg.w_perp, _cfg.w_para
R, Rd = np.diag(_cfg.R), np.diag(_cfg.Rd)
Q_v_yaw = np.diag(_cfg.Q_v_yaw)
Qf = np.diag(_cfg.Qf_raw) * T
GOAL_DIS, STOP_SPEED, MAX_TIME = _cfg.goal_dis, _cfg.stop_speed, _cfg.max_time
MAX_ITER, DU_TH = _cfg.max_iter, _cfg.du_th
MAX_DSTEER = _cfg.max_dsteer
MAX_ACCEL, MAX_DECEL = _cfg.max_accel, _cfg.max_decel


class MPCSolutionNotFoundException(Exception):
    pass


def smooth_yaw(yaw):
    """In-place yaw unwrapping (mpc.py:46-58); returns its argument."""
    for k in range(len(yaw) - 1):
        while yaw[k + 1] - yaw[k] >= math.pi / 2.0:
            yaw[k + 1] -= math.pi * 2.0
        while yaw[k + 1] - yaw[k] <= -math.pi / 2.0:
            yaw[k + 1] += math.pi * 2.0
    return yaw


class MPC:
    """Stateful single-ego controller with the reference's interface."""

    _reload_config_each_step = False      # the sensitivity flavour re-reads its JSON in every solve
    _config = _cfg
    # The reference left the DU_TH exit of the linearisation loop commented out (mpc.py:236-240), so it is off here
    # too; setting this to True on the class (or an instance, before the first step) applies DU_TH of the JSON.
    enable_du_th_exit = False

    def __init__(self, cx: np.ndarray, cy: np.ndarray, cyaw: np.ndarray, dl: float, car_dimensions,
                 speed: float = 30 / 3.6, dt: float = 0.2):
        self.cx = cx
        self.cy = cy
        cyaw = smooth_yaw(cyaw)           # in place, on the caller's view of trajectory_full[:, 2] (mpc.py:260)
        self.cyaw = cyaw
        self.dl = dl
        self.dt = dt
        self.car_dimensions = car_dimensions
        self.speed = speed
        self.goal: Tuple[float, float] = cx[-1], cy[-1]
        self.target_ind: int = 0
        self.odelta: Optional[List[float]] = None
        self.oa: Optional[List[float]] = None
        self.ox = self.oy = self.oyaw = self.ov = self.xref = None
        self.di: float = 0.0
        self.ai: float = 0.0
        self.status: int = _cabi.STATUS_OPTIMAL
        self.iterations: int = 0
        self.cost: float = float("nan")
        self._full = np.stack([np.asarray(cx, float), np.asarray(cy, float), np.asarray(cyaw, float)], axis=1)
        self._engine = self._make_engine(self._config)

    # ---- engine plumbing ------------------------------------------------------------------------------------
    def _make_engine(self, cfg: MPCConfig) -> BatchedMPC:
        L = float(self.car_dimensions.distance_back_to_front_wheel)
        self._cfg_used = cfg
        return BatchedMPC([self._full], dl=float(self.dl), T=cfg.T, config=cfg, dt=float(self.dt), L=L,
                          speed=float(self.speed), max_batch=1, max_T=_cabi.JMPC_MAX_T,
                          du_th=float(cfg.du_th) if self.enable_du_th_exit else 0.0)

    def _effective_length(self) -> int:
        """`set_trajectory_fromarray(trajectory_full[:k])` always passes a prefix of the course given to the
        constructor (mpc_intersection.py:138); it is expressed as an effective length on the uploaded table.
        Anything else is uploaded afresh.  "Is a prefix" is decided on all of the data (three vectorised compares of
        at most a few hundred doubles), never on samples: a different course must not run on the old table."""
        n = len(self.cx)
        full = self._full
        if 1 <= n <= len(full) and np.array_equal(self.cx, full[:n, 0]) and np.array_equal(self.cy, full[:n, 1]) \
                and np.array_equal(self.cyaw, full[:n, 2]):
            return n
        self._full = np.stack([np.asarray(self.cx, float), np.asarray(self.cy, float), np.asarray(self.cyaw, float)],
                              axis=1)
        self._engine.close()
        self._engine = self._make_engine(self._cfg_used)
        self._course_changed()
        return n

    def _course_changed(self):
        """Hook for flavours that keep per-course device tables besides x / y / yaw."""

    def _instance_params(self):
        return None                        # handle defaults; flavours with per-step parameters override this

    # ---- reference interface --------------------------------------------------------------------------------
    def set_trajectory_fromarray(self, trajectory: np.ndarray):
        self.cx = trajectory[:, 0]
        self.cy = trajectory[:, 1]
        self.cyaw = trajectory[:, 2]

    def step(self, state) -> Tuple[float, float]:
        if self._reload_config_each_step:
            cfg = type(self)._load_config()
            if cfg != self._cfg_used:
                self._engine.close()
                self._engine = self._make_engine(cfg)
                self._course_changed()
        n = self._effective_length()
        Th = self._cfg_used.T
        warm = self.oa is not None and self.odelta is not None
        x0 = np.array([[state.x, state.y, state.v, state.yaw]], dtype=np.float64)
        out = self._engine.step_host(
            x0, np.array([self.target_ind], np.int32),
            oa=np.asarray(self.oa, float).reshape(1, Th) if warm else np.zeros((1, Th)),
            od=np.asarray(self.odelta, float).reshape(1, Th) if warm else np.zeros((1, Th)),
            course_len=np.array([n], np.int32), warm=np.array([1 if warm else 0], np.int32),
            params=self._instance_params())
        self.status = int(out.status[0])
        self.iterations = int(out.iters[0])
        if self.status == _cabi.STATUS_INDEX_RULE:
            raise Exception("something wrong")                     # trajectories.py:120
        self.target_ind = int(out.target_ind[0])
        self.xref = out.xref[0]
        if self.status != _cabi.STATUS_OPTIMAL:
            # infeasible, or the solver gave up (iteration cap without even the reduced tolerances): the reference
            # accepts only OPTIMAL / OPTIMAL_INACCURATE (mpc.py:199); otherwise it prints, returns None for all
            # outputs, keeps di and brakes with MAX_DECEL (mpc.py:207-209, 298-301)
            print("Error: Cannot solve mpc...", file=sys.stderr)
            self.oa = self.odelta = self.ox = self.oy = self.oyaw = self.ov = None
            self.ai = self._cfg_used.max_decel
            return self.di, self.ai
        self.oa, self.odelta = out.oa[0], out.od[0]
        self.ox, self.oy, self.ov, self.oyaw = out.ox[0], out.oy[0], out.ov[0], out.oyaw[0]
        self.cost = float(out.cost[0])
        self.di, self.ai = float(self.odelta[0]), float(self.oa[0])
        return self.di, self.ai

    def get_current_xref_deviation(self):
        ref_point = np.array([self.cx[self.target_ind], self.cy[self.target_ind]])
        true_point = np.array([self.ox[0], self.oy[0]])
        ref_yaw_perp = self.cyaw[self.target_ind] + np.pi / 2
        diff = ref_point - true_point
        return np.linalg.norm(np.array([np.cos(ref_yaw_perp) * diff[0], np.sin(ref_yaw_perp) * diff[1]]))

    def is_goal(self, state) -> bool:
        d = math.hypot(state.x - self.goal[0], state.y - self.goal[1])
        isgoal = d <= self._cfg_used.goal_dis
        if abs(self.target_ind - len(self.cx)) >= 5:
            isgoal = False
        isstop = abs(state.v) <= self._cfg_used.stop_speed
        return bool(isgoal and isstop)


# ---- the sensitivity flavour (main/lib/mpc_sensitivity.py) ---------------------------------------------------
class _SensitivityMPC(MPC):
    """`lib.mpc_sensitivity.MPC`: no `speed` argument (Simulation.MAX_SPEED is the cap, mpc_sensitivity.py:207)
    and the JSON is re-read inside every solve (mpc_sensitivity.py:153-166), which is how the sweep script changes
    weights between runs."""
    _reload_config_each_step = True
    _config_file: Optional[str] = None

    def __init__(self, cx, cy, cyaw, dl, car_dimensions, dt: float = 0.2):
        type(self)._config = type(self)._load_config()
        super().__init__(cx, cy, cyaw, dl, car_dimensions, speed=SIM_MAX_SPEED, dt=dt)

    @classmethod
    def _load_config(cls) -> MPCConfig:
        path = cls._config_file or os.environ.get("JMPC_CONFIG_SENSITIVITY")
        return MPCConfig.from_json(path) if path else MPCConfig.default()


# ---- the speed-profile flavour (main/lib/mpc_with_speed.py) --------------------------------------------------
_WITH_SPEED_CONFIG = MPCConfig.from_dict({
    # constants hard-coded at mpc_with_speed.py:16-36 and :161,165 (xy weights 10 / 1)
    "NX": 4, "NU": 2, "T": 13, "w_perp": 10.0, "w_para": 1.0, "R": [0.01, 0.01], "Rd": [0.01, 1.0],
    "Q_v_yaw": [20, 0.5], "Qf": [1.0, 1.0, 0.0, 0.5], "GOAL_DIS": 1.5, "STOP_SPEED": 0.5 / 3.6, "MAX_TIME": 13.0,
    "MAX_ITER": 1, "DU_TH": 0.1, "MAX_DSTEER": 30.0, "MAX_ACCEL": 2.0, "MAX_DECEL": -5})
WITH_SPEED_MAX_SPEED = 25 / 3.6                     # mpc_with_speed.py:36


class _WithSpeedMPC(MPC):
    """`lib.mpc_with_speed.MPC(cx, cy, cv, cyaw, dl, car_dimensions, dt)`: the reference speed profile `cv` enters
    xref[2] (mpc_with_speed.py:104) and is tracked with Q_v = 20; `set_trajectory_fromarray(trajectory, cutoff_idx)`
    rebuilds it as MAX_SPEED before `cutoff_idx` and 0 from there on (:276-282).  The speed cap of the QP is
    Simulation.MAX_SPEED (:187)."""
    _config = _WITH_SPEED_CONFIG

    def __init__(self, cx, cy, cv, cyaw, dl, car_dimensions, dt: float = 0.2):
        self._cv_uploaded = None
        super().__init__(cx, cy, cyaw, dl, car_dimensions, speed=SIM_MAX_SPEED, dt=dt)
        self.cv = cv
        self._v_ref, self._v_cut = 0.0, 1e9

    def set_trajectory_fromarray(self, trajectory: np.ndarray, cutoff_idx: int = 999):
        super().set_trajectory_fromarray(trajectory)
        self.cv = np.full_like(self.cyaw, WITH_SPEED_MAX_SPEED)
        if cutoff_idx != 999:
            self.cv[cutoff_idx:] = 0

    def _course_changed(self):
        self._cv_uploaded = None             # a fresh engine has no speed table

    def _instance_params(self):
        """`cv` is an attribute the reference reads at every step (mpc_with_speed.py:104).  A two-level profile
        (constant, or constant up to an index and 0 from there on: what set_trajectory_fromarray builds) travels as
        the two per-instance parameters v_ref / v_ref_cut; anything else is uploaded as a per-course table."""
        from .config import PARAM_INDEX
        n = len(self.cx)
        cv = np.asarray(self.cv, float)
        if cv.ndim != 1 or len(cv) < n:
            raise ValueError("cv must hold one reference speed per course point")
        cv = cv[:n]
        v_ref, v_cut, table = float(cv[0]), 1e9, None
        changes = np.nonzero(cv != cv[0])[0]
        if changes.size:
            if np.all(cv[changes[0]:] == 0.0):
                v_cut = float(changes[0])
            else:
                table = np.zeros(len(self._full))
                table[:n] = cv
        if table is None:
            if self._cv_uploaded is not None:
                self._engine.set_course_speed(None)
                self._cv_uploaded = None
        elif self._cv_uploaded is None or not np.array_equal(self._cv_uploaded, table):
            self._engine.set_course_speed([table])
            self._cv_uploaded = table
        self._v_ref, self._v_cut = v_ref, v_cut
        p = self._engine.default_params.copy()
        p[PARAM_INDEX["v_ref"]] = v_ref
        p[PARAM_INDEX["v_ref_cut"]] = v_cut
        return p[None, :]


def _module_from(cls, cfg: MPCConfig, name: str) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__doc__ = f"junction_mpc drop-in for the reference module {name}"
    m.MPC = cls
    m.MPCSolutionNotFoundException = MPCSolutionNotFoundException
    m.smooth_yaw = smooth_yaw
    m.NX, m.NU, m.T = cfg.nx, cfg.nu, cfg.T
    m.w_perp, m.w_para = cfg.w_perp, cfg.w_para
    m.R, m.Rd, m.Q_v_yaw = np.diag(cfg.R), np.diag(cfg.Rd), np.diag(cfg.Q_v_yaw)
    m.Qf = np.diag(cfg.Qf_raw) * cfg.T
    m.GOAL_DIS, m.STOP_SPEED, m.MAX_TIME = cfg.goal_dis, cfg.stop_speed, cfg.max_time
    m.MAX_ITER, m.DU_TH = cfg.max_iter, cfg.du_th
    m.MAX_DSTEER, m.MAX_ACCEL, m.MAX_DECEL = cfg.max_dsteer, cfg.max_accel, cfg.max_decel
    return m


def install(reference_main: Optional[str] = None) -> None:
    """Make `from lib.mpc import MPC, MAX_ACCEL` and `from lib.mpc_sensitivity import MPC, MAX_ACCEL` resolve to
    this implementation.  `reference_main` is the reference's `main/` directory: its `config/mpc_config.json` and
    `config/mpc_config_sensitivity.json` are read unchanged, and it is put on sys.path so the rest of `lib`
    (simulation, collision_avoidance, ...) is still the reference's own code."""
    global _cfg
    cfg, sens_cfg_path = _cfg, None
    if reference_main:
        if reference_main not in sys.path:
            sys.path.insert(0, reference_main)
        p = os.path.join(reference_main, "config", "mpc_config.json")
        if os.path.exists(p):
            cfg = MPCConfig.from_json(p)
        p = os.path.join(reference_main, "config", "mpc_config_sensitivity.json")
        if os.path.exists(p):
            sens_cfg_path = p

    class _MPC(MPC):
        _config = cfg
    _MPC.__name__ = _MPC.__qualname__ = "MPC"

    class _SMPC(_SensitivityMPC):
        _config_file = sens_cfg_path
    _SMPC.__name__ = _SMPC.__qualname__ = "MPC"

    sys.modules["lib.mpc"] = _module_from(_MPC, cfg, "lib.mpc")
    sens_cfg = MPCConfig.from_json(sens_cfg_path) if sens_cfg_path else cfg
    sys.modules["lib.mpc_sensitivity"] = _module_from(_SMPC, sens_cfg, "lib.mpc_sensitivity")
    ws = _module_from(_WithSpeedMPC, _WITH_SPEED_CONFIG, "lib.mpc_with_speed")
    ws.MAX_SPEED = WITH_SPEED_MAX_SPEED
    ws.MPC = type("MPC", (_WithSpeedMPC,), {})
    sys.modules["lib.mpc_with_speed"] = ws
    from . import planner as _planner          # the planner drop-in (SURVEY.md 8f row f4)
    pl = types.ModuleType("lib.mp_search_ww_generic")
    pl.__doc__ = "junction_mpc drop-in for the reference module lib.mp_search_ww_generic"
    pl.MotionPrimitiveSearch = _planner.MotionPrimitiveSearch
    sys.modules["lib.mp_search_ww_generic"] = pl
    try:                                   # `import lib.mpc` also needs the attribute on the package
        import lib                         # the reference's package, when reference_main is on sys.path
        lib.mpc = sys.modules["lib.mpc"]
        lib.mpc_sensitivity = sys.modules["lib.mpc_sensitivity"]
        lib.mpc_with_speed = ws
        lib.mp_search_ww_generic = pl
    except ImportError:
        pkg = types.ModuleType("lib")
        pkg.__path__ = []
        pkg.mpc, pkg.mpc_sensitivity, pkg.mpc_with_speed = sys.modules["lib.mpc"], sys.modules["lib.mpc_sensitivity"], ws
        pkg.mp_search_ww_generic = pl
        sys.modules["lib"] = pkg
