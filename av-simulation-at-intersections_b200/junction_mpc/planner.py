"""Batched motion-primitive A* planner on the GPU, and a drop-in for the reference's `MotionPrimitiveSearch`.

    from lib.mp_search_ww_generic import MotionPrimitiveSearch           main/scenarios/mpc_intersection.py:23
    search = MotionPrimitiveSearch(scenario, car_dimensions, mps, margin=car_dimensions.radius)   :62
    cost, path, trajectory_full = search.run(debug=False)                mp_search_ww_generic.py:136-140

`BatchedPlanner.plan` runs many (start, goal, weights, scene) searches in one kernel launch (one warp per search,
csrc/jmpc_planner.cuh) through `jmpc_plan_host`; `MotionPrimitiveSearch` is the same call for a batch of one with the
reference's constructor and return values.  The planned courses go straight into `BatchedMPC(courses=...)`.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _cabi

MAX_HP = 8
WEIGHT_KEYS = ("wh_dist", "wh_theta", "wh_steering", "wh_obstacle", "wh_center", "wc_dist", "wc_steering", "wc_obstacle",
               "wc_center")
DEFAULT_WEIGHTS = dict(wh_dist=1.0, wh_theta=2.7, wh_steering=15.0, wh_obstacle=0.0, wh_center=0.0, wc_dist=1.0,
                       wc_steering=5.0, wc_obstacle=0.1, wc_center=0.0)            # mp_search_ww_generic.py:27-31
STATUS_FOUND, STATUS_NO_SOLUTION, STATUS_LIMIT = 0, 1, 2
_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "motion_primitives_bicycle_model.npz")


def load_motion_primitives() -> Tuple[List[str], np.ndarray, np.ndarray]:
    """The reference's bicycle-model primitive set (main/data/motion_primitives_bicycle_model/*.pkl) as arrays:
    names (sorted), points [n_mp, n_pts, 3] relative to the start pose, total_length [n_mp]."""
    with np.load(_DATA) as z:
        return [str(n) for n in z["names"]], np.array(z["points"], float), np.array(z["total_length"], float)


def box_halfplanes(xy_width, xy_center, margin: float = 0.0) -> np.ndarray:
    """BoxObstacle.to_convex (obstacles.py:83-95)."""
    (wx, wy), (cx, cy) = xy_width, xy_center
    x1, y1, x2, y2 = cx - wx / 2, cy - wy / 2, cx + wx / 2, cy + wy / 2
    return np.array([[1, 0, -(x2 + margin)], [-1, 0, x1 - margin], [0, 1, -(y2 + margin)], [0, -1, y1 - margin]], float)


def circle_halfplanes(radius: float, xy_center, margin: float = 0.0) -> np.ndarray:
    """CircleObstacle.to_convex (obstacles.py:135-150): the circumscribed octagon."""
    cx, cy = xy_center
    r, q = radius, radius * np.sqrt(2)
    return np.array([[1, 0, -(cx + r + margin)], [-1, 0, cx - r - margin], [0, 1, -(cy + r + margin)], [0, -1, cy - r - margin],
                     [-1, 1, cx - cy - q - 2 * margin], [1, -1, -cx + cy - q - 2 * margin],
                     [-1, -1, cx + cy - q - 2 * margin], [1, 1, -cx - cy - q - 2 * margin]], float)


def collision_check_points(mp_points: np.ndarray, radius: float, circle_centers: np.ndarray) -> np.ndarray:
    """Check points of one primitive (mp_search_ww_generic.py:121-138): keep a point whenever the arc length passes
    another multiple of the car radius (first and last always), then the centre of every collision circle at each
    kept pose.  Returns [n_circles * n_kept, 2], circle by circle.  Host side, once per primitive set."""
    pts = np.asarray(mp_points, float)
    seg = np.hypot(np.diff(pts[:, 0]), np.diff(pts[:, 1]))
    bucket = np.floor(np.concatenate([[0.0], seg]).cumsum() / radius).astype(np.int64)
    keep = np.concatenate([[True], np.diff(bucket) >= 1])
    keep[-1] = True
    kept = pts[keep]
    c, s = np.cos(kept[:, 2]), np.sin(kept[:, 2])
    out = [np.stack([c * ox - s * oy + kept[:, 0], s * ox + c * oy + kept[:, 1]], axis=1) for ox, oy in circle_centers]
    return np.concatenate(out, axis=0)


def pack_plan_inputs(start, goal_point, goal_area, allowed_dtheta, scenes, scene_id=None, weights=None):
    """The arguments of `BatchedPlanner.plan` in the C ABI's layout: (start, goal_point, goal_area, allowed, weights,
    scene_id or None, (n_scenes, max_obs, hp, hp_n, n_obs))."""
    f = lambda a, shape: np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), shape))   # noqa: E731
    start = np.ascontiguousarray(np.asarray(start, np.float64).reshape(-1, 3))
    B = len(start)
    goal_point, goal_area = f(goal_point, (B, 3)), f(goal_area, (B, 4))
    allowed = f(allowed_dtheta, (B,))
    if weights is None or isinstance(weights, dict):
        w = dict(DEFAULT_WEIGHTS, **(weights or {}))
        weights = [w[k] for k in WEIGHT_KEYS]
    weights = f(weights, (B, 9))
    n_scenes = len(scenes)
    max_obs = max(1, max(len(s) for s in scenes))
    hp = np.zeros((n_scenes, max_obs, MAX_HP, 3))
    hp_n = np.zeros((n_scenes, max_obs), np.int32)
    n_obs = np.array([len(s) for s in scenes], np.int32)
    for i, s in enumerate(scenes):
        for k, rows in enumerate(s):
            rows = np.asarray(rows, float).reshape(-1, 3)
            if not 1 <= len(rows) <= MAX_HP:
                raise ValueError(f"an obstacle needs 1..{MAX_HP} half-planes")
            hp[i, k, :len(rows)] = rows
            hp_n[i, k] = len(rows)
    sid = None if scene_id is None else np.ascontiguousarray(scene_id, dtype=np.int32)
    return start, goal_point, goal_area, allowed, weights, sid, (n_scenes, max_obs, hp, hp_n, n_obs)


@dataclass
class DevicePlanBatch:
    """What `BatchedPlanner.plan_device` returns: the fields of `PlanBatch` as torch CUDA tensors (same shapes), still
    being computed on the stream they were enqueued on.  Feed it to `BatchedMPC.from_plans` to drive the courses
    without a host round trip."""
    cost: object
    status: object
    n_path: object
    path: object
    path_mp: object
    n_traj: object
    traj: object                # [B, max_traj, 3] x, y, raw yaw
    expansions: object
    log: object = None

    def __len__(self) -> int:
        return int(self.cost.shape[0])

    def to_host(self) -> PlanBatch:
        """Synchronising copy into a `PlanBatch` (kernel_ms = NaN: the launch was not timed)."""
        c = lambda t: None if t is None else t.cpu().numpy()            # noqa: E731
        return PlanBatch(cost=c(self.cost), status=c(self.status), n_path=c(self.n_path), path=c(self.path),
                         path_mp=c(self.path_mp), n_traj=c(self.n_traj), traj=c(self.traj),
                         expansions=c(self.expansions), log=c(self.log), kernel_ms=float("nan"))


@dataclass
class PlanBatch:
    cost: np.ndarray            # [B]
    status: np.ndarray          # [B] 0 found, 1 no solution (the reference raises), 2 limit reached
    n_path: np.ndarray          # [B]
    path: np.ndarray            # [B, max_path, 3]
    path_mp: np.ndarray         # [B, max_path]
    n_traj: np.ndarray          # [B]
    traj: np.ndarray            # [B, max_traj, 3]
    expansions: np.ndarray      # [B]
    log: Optional[np.ndarray]   # [B, max_log, 5] g, h, x, y, theta in expansion order
    kernel_ms: float

    def trajectory(self, b: int) -> np.ndarray:
        """trajectory_full of search b (path_to_full_trajectory, mp_search_ww_generic.py:245-256)."""
        return self.traj[b, :self.n_traj[b]].copy()

    def courses(self) -> List[np.ndarray]:
        """The planned courses of all successful searches, ready for BatchedMPC(courses=...) (yaw still raw: the
        controller smooths it, mpc.py:260)."""
        return [self.trajectory(b) for b in range(len(self.cost)) if self.status[b] == STATUS_FOUND]


class BatchedPlanner:
    def __init__(self, mp_points: Optional[np.ndarray] = None, mp_total_length: Optional[np.ndarray] = None,
                 car_radius: float = 2.0 / 2 ** 0.5, circle_centers=((2.18, 0.0), (0.68, 0.0)), device: int = 0,
                 max_batch: int = 4096):
        """Defaults: the reference's bicycle-model primitives and BicycleModelDimensions (car_dimensions.py:62-90:
        width 2, length 3.5, circle centres at L/2 +- (length - width)/2 ahead of the rear axle: 2.18 and 0.68).
        `max_batch`: searches per launch of `plan_device`, whose persistent workspace is allocated for that many
        (about 2 MB per search at max_expansions = 4096); larger batches run in chunks."""
        self._lib = _cabi.load()
        if mp_points is None:
            _, mp_points, mp_total_length = load_motion_primitives()
        self.mp_points = np.ascontiguousarray(mp_points, dtype=np.float64)
        self.mp_len = np.ascontiguousarray(mp_total_length, dtype=np.float64)
        if self.mp_points.ndim != 3 or self.mp_points.shape[2] != 3 or len(self.mp_len) != len(self.mp_points):
            raise ValueError("mp_points must be [n_mp, n_pts, 3] with one total_length each")
        cc = [collision_check_points(p, float(car_radius), np.asarray(circle_centers, float)) for p in self.mp_points]
        if len({len(c) for c in cc}) != 1:
            raise ValueError("primitives with different numbers of collision-check points are not supported")
        self.mp_cc = np.ascontiguousarray(np.stack(cc), dtype=np.float64)
        self.device = int(device)
        if int(max_batch) < 1:
            raise ValueError("max_batch must be positive")
        self.max_batch = int(max_batch)
        self._handle, self._handle_key = None, None         # jmpc_planner of plan_device, created on first use

    def plan(self, start, goal_point, goal_area, allowed_dtheta, scenes: Sequence[Sequence[np.ndarray]], scene_id=None,
             weights=None, max_expansions: int = 4096, max_path: int = 48, log: bool = False) -> PlanBatch:
        """start, goal_point [B, 3]; goal_area [B, 4] = x1, y1, x2, y2; allowed_dtheta [B] or scalar;
        scenes: list of scenes, each a list of half-plane arrays [m, 3] (one per obstacle, m <= 8); scene_id [B];
        weights [B, 9] in WEIGHT_KEYS order, a dict, or None for the reference defaults."""
        start, goal_point, goal_area, allowed, weights, sid, (n_scenes, max_obs, hp, hp_n, n_obs) = pack_plan_inputs(
            start, goal_point, goal_area, allowed_dtheta, scenes, scene_id, weights)
        B = len(start)
        n_mp, n_pts = self.mp_points.shape[:2]
        n_cc = self.mp_cc.shape[1]
        max_traj = (max_path - 1) * (n_pts - 1)
        max_log = int(max_expansions) if log else 0
        out = PlanBatch(cost=np.zeros(B), status=np.zeros(B, np.int32), n_path=np.zeros(B, np.int32),
                        path=np.zeros((B, max_path, 3)), path_mp=np.zeros((B, max_path), np.int32),
                        n_traj=np.zeros(B, np.int32), traj=np.zeros((B, max_traj, 3)), expansions=np.zeros(B, np.int32),
                        log=np.zeros((B, max_log, 5)) if log else None, kernel_ms=0.0)
        ms = C.c_double(0.0)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)      # noqa: E731
        _cabi.check(self._lib.jmpc_plan_host(
            self.device, B, n_mp, n_pts, n_cc, p(self.mp_points), p(self.mp_len), p(self.mp_cc), n_scenes, max_obs, p(hp),
            p(hp_n), p(n_obs), p(sid), p(start), p(goal_point), p(goal_area), p(allowed), p(weights), int(max_expansions),
            int(max_path), max_log, p(out.cost), p(out.status), p(out.n_path), p(out.path), p(out.path_mp), p(out.n_traj),
            p(out.traj), p(out.expansions), p(out.log), C.cast(C.byref(ms), C.c_void_p)), "jmpc_plan_host")
        out.kernel_ms = float(ms.value)
        return out

    def plan_device(self, start, goal_point, goal_area, allowed_dtheta, scenes: Sequence[Sequence[np.ndarray]],
                    scene_id=None, weights=None, max_expansions: int = 4096, max_path: int = 48,
                    log: bool = False) -> DevicePlanBatch:
        """`plan` with the results left on the device: the same arguments, the same kernel and bit-identical
        results, as torch CUDA tensors enqueued on torch's current stream (nothing is synchronised).  The workspace
        is this planner's persistent `jmpc_planner`, created on first use for `max_batch` searches (re-created when
        max_expansions / max_path / log change); batches larger than `max_batch` run in chunks on the same stream."""
        import torch
        start, goal_point, goal_area, allowed, weights, sid, (n_scenes, max_obs, hp, hp_n, n_obs) = pack_plan_inputs(
            start, goal_point, goal_area, allowed_dtheta, scenes, scene_id, weights)
        B = len(start)
        if sid is not None and (sid.shape != (B,) or (B and (sid.min() < 0 or sid.max() >= n_scenes))):
            raise ValueError("scene_id must be [B] with values in [0, len(scenes))")
        max_expansions, max_path = int(max_expansions), int(max_path)
        max_log = max_expansions if log else 0
        p = self._planner_handle(max_expansions, max_path, max_log)
        _cabi.check(self._lib.jmpc_planner_set_scenes(p, n_scenes, max_obs, hp.ctypes.data_as(C.c_void_p),
                                                      hp_n.ctypes.data_as(C.c_void_p), n_obs.ctypes.data_as(C.c_void_p)),
                    "jmpc_planner_set_scenes")
        dev = torch.device("cuda", self.device)
        f64, i32 = torch.float64, torch.int32
        # np.array copies: the packed inputs can be read-only broadcast views, which torch does not wrap
        up = lambda a, dt: None if a is None else torch.as_tensor(np.array(a), dtype=dt).to(dev)      # noqa: E731
        d_start, d_goal, d_area, d_allowed, d_w, d_sid = (up(start, f64), up(goal_point, f64), up(goal_area, f64),
                                                          up(allowed, f64), up(weights, f64), up(sid, i32))
        max_traj = (max_path - 1) * (self.mp_points.shape[1] - 1)
        out = DevicePlanBatch(cost=torch.empty(B, dtype=f64, device=dev), status=torch.empty(B, dtype=i32, device=dev),
                              n_path=torch.empty(B, dtype=i32, device=dev),
                              path=torch.empty(B, max_path, 3, dtype=f64, device=dev),
                              path_mp=torch.empty(B, max_path, dtype=i32, device=dev),
                              n_traj=torch.empty(B, dtype=i32, device=dev),
                              traj=torch.empty(B, max_traj, 3, dtype=f64, device=dev),
                              expansions=torch.empty(B, dtype=i32, device=dev),
                              log=torch.empty(B, max_log, 5, dtype=f64, device=dev) if log else None)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        q = lambda t, lo: None if t is None else C.c_void_p(t[lo:].data_ptr())           # noqa: E731
        for lo in range(0, B, self.max_batch):
            n = min(self.max_batch, B - lo)
            _cabi.check(self._lib.jmpc_plan(
                p, n, q(d_sid, lo), q(d_start, lo), q(d_goal, lo), q(d_area, lo), q(d_allowed, lo), q(d_w, lo),
                q(out.cost, lo), q(out.status, lo), q(out.n_path, lo), q(out.path, lo), q(out.path_mp, lo),
                q(out.n_traj, lo), q(out.traj, lo), q(out.expansions, lo), q(out.log, lo), stream), "jmpc_plan")
        return out

    def _planner_handle(self, max_expansions: int, max_path: int, max_log: int):
        key = (max_expansions, max_path, max_log)
        if self._handle is not None and self._handle_key == key:
            return self._handle
        self.close()
        n_mp, n_pts = self.mp_points.shape[:2]
        h = C.c_void_p()
        p = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
        _cabi.check(self._lib.jmpc_planner_create(self.device, self.max_batch, n_mp, n_pts, self.mp_cc.shape[1],
                                                  p(self.mp_points), p(self.mp_len), p(self.mp_cc), max_expansions,
                                                  max_path, max_log, C.byref(h)), "jmpc_planner_create")
        self._handle, self._handle_key = h, key
        return h

    def close(self):
        """Free the persistent workspace of `plan_device` (waits for the device first)."""
        if getattr(self, "_handle", None) is not None:
            import torch
            torch.cuda.synchronize(self.device)
            self._lib.jmpc_planner_destroy(self._handle)
            self._handle, self._handle_key = None, None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MotionPrimitiveSearch:
    """Drop-in for `lib.mp_search_ww_generic.MotionPrimitiveSearch` (same constructor, `run` returns the same triple):
    one search = a batch of one through `BatchedPlanner`."""

    def __init__(self, scenario, car_dimensions, mps: Dict[str, object], margin: float, wh_dist: float = 1.0,
                 wh_theta: float = 2.7, wh_steering: float = 15.0, wh_obstacle: float = 0.0, wh_center: float = 0.0,
                 wc_dist: float = 1.0, wc_steering: float = 5.0, wc_obstacle: float = 0.1, wc_center: float = 0.0):
        self._names = list(mps)                                   # the dict's own order, as the reference iterates it
        self._planner = BatchedPlanner(np.stack([np.asarray(mps[n].points, float) for n in self._names]),
                                       np.array([mps[n].total_length for n in self._names], float),
                                       car_radius=float(car_dimensions.radius),
                                       circle_centers=np.asarray(car_dimensions.circle_centers, float))
        self._scenario = scenario
        self._scene = [np.asarray(o.to_convex(margin=margin), float) for o in scenario.obstacles]
        self._weights = dict(wh_dist=wh_dist, wh_theta=wh_theta, wh_steering=wh_steering, wh_obstacle=wh_obstacle,
                             wh_center=wh_center, wc_dist=wc_dist, wc_steering=wc_steering, wc_obstacle=wc_obstacle,
                             wc_center=wc_center)
        self.debug_data = []
        self.last: Optional[PlanBatch] = None

    def run(self, debug: bool = False):
        sc = self._scenario
        area = [*sc.goal_area.xy1, *sc.goal_area.xy2]
        r = self._planner.plan([sc.start], [sc.goal_point], [area], sc.allowed_goal_theta_difference, [self._scene],
                               weights=self._weights, max_expansions=16384, max_path=64, log=debug)
        self.last = r
        if debug:
            self.debug_data = [tuple(row) for row in r.log[0, :r.expansions[0]]]
        if r.status[0] == STATUS_NO_SOLUTION:
            raise Exception("No solution found.")                 # a_star.py:78
        if r.status[0] != STATUS_FOUND:
            raise RuntimeError("motion-primitive search: expansion / path limit reached")
        path = [tuple(float(v) for v in node) for node in r.path[0, :r.n_path[0]]]
        return float(r.cost[0]), path, r.trajectory(0)
