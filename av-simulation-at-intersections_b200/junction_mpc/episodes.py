"""BatchedEpisodes: B closed-loop episodes of the reference's scenario loop, device resident.

One iteration = the body of `for i in itertools.count()` in main/scenarios/mpc_intersection.py:99-163:
goal test -> ego index on the full course -> collision flag / cut -> MPC step -> plant step + history.
Everything runs in libjmpc.so kernels on torch-owned device tensors; the host only sequences launches and looks
at the `done` flags every few iterations.  Obstacles are the reference's scripted vehicles stepped on the device
(`obstacle_program`, see `scripted_obstacles`), constant-input vehicles advanced on the device (`obstacles`), or a
per-step recording (`obstacle_script`).  With `outcomes=True` every episode also keeps a compact outcome record on
the device (contact, clearance, comfort; enum jmpc_outcome in include/jmpc.h), so that a study needs no History.
With `agents_per_scene=k` every k consecutive episodes form a scene whose MPC-driven vehicles see each other as moving
obstacles (jmpc_scene_exchange); with `share_plans=True` they predict each other along their MPC plans
(jmpc_scene_plans, jmpc_collision_planned); with `right_of_way` a rule decides which mates each vehicle yields to
(jmpc_right_of_way, jmpc_collision_masked); with `depart` / `on_goal="leave"` every vehicle has a lifetime in its scene:
it enters at its departure iteration and may leave at its goal (jmpc_scene_enter, jmpc_scene_presence); with
`from_trips` the scenes' slots are fed from a stream of timed trips (jmpc_scene_trips), and `run()` returns one row per
trip; with `signals` a fixed-time signal plan cuts the courses of vehicles facing red at their stop line (jmpc_signals).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np

from . import _cabi
from .batched import BatchedMPC
from .config import NPARAM, PARAM_INDEX


OBS_KINDS = {"constant": 0, "t_intersection": 1, "roundabout": 2, "arterial": 3}

# public columns of the outcome record, in the order of enum jmpc_outcome (include/jmpc.h)
OUTCOME_NAMES = ("min_clearance", "min_clearance_eval", "min_clearance_obs", "first_contact_eval", "first_contact_obs",
                 "contact_evals", "cut_steps", "limit_steps", "failed_solves", "max_abs_accel", "max_abs_jerk",
                 "max_abs_steer_rate", "max_abs_lat_accel", "max_xref_dev", "sum_xref_dev", "distance")
OUTCOME_INT = frozenset(OUTCOME_NAMES[1:9])          # evaluation / obstacle indices and counts
OUTCOME_LEN = 22                                     # JMPC_OUTCOME_LEN: the public columns, then private running state
MAX_OBSTACLES = 8                                    # kMaxObstacles of the collision and outcome kernels


def outcome_setup(outcomes: bool, record_obstacles: bool, n_obs: int) -> bool:
    """Host-side checks of the outcome options of `BatchedEpisodes`: returns whether the outcome kernel runs.
    The obstacle tracks are written by the outcome kernel, so `record_obstacles` needs `outcomes`."""
    if record_obstacles and not outcomes:
        raise ValueError("record_obstacles=True needs outcomes=True")
    if outcomes and not 0 <= n_obs <= MAX_OBSTACLES:
        raise ValueError(f"outcomes support at most {MAX_OBSTACLES} obstacles per episode, got {n_obs}")
    return bool(outcomes)


def scene_setup(B: int, agents_per_scene: int, n_extra: int, has_script: bool) -> int:
    """Host-side checks of the scene option of `BatchedEpisodes`: returns the obstacle slots per episode,
    (agents_per_scene - 1) scene mates + n_extra own obstacles (enum jmpc_done / jmpc_scene_exchange in include/jmpc.h)."""
    k = agents_per_scene
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 1:
        raise ValueError(f"agents_per_scene must be an integer >= 1, got {k!r}")
    k = int(k)
    if B % k:
        raise ValueError(f"the batch of {B} episodes is not a whole number of scenes of {k} vehicles")
    if k > 1 and has_script:
        raise ValueError("obstacle_script cannot be combined with agents_per_scene > 1: a recording cannot react to the "
                         "scene's vehicles; give obstacles or obstacle_program for the scripted traffic")
    n_obs = (k - 1) + int(n_extra)
    if n_obs > MAX_OBSTACLES:
        raise ValueError(f"{k - 1} scene mates + {n_extra} obstacles exceed the {MAX_OBSTACLES} obstacle slots of an "
                         "episode")
    return n_obs


def plan_share_setup(share_plans: bool, k: int, params) -> bool:
    """Host-side checks of the shared-plans option of `BatchedEpisodes`: returns whether the plans are exchanged.
    A mate's plan is in its own steps and the predictor runs at the evaluating vehicle's dt, so every vehicle of a scene
    needs the same dt (params [B, NPARAM] rows; None = the engine's defaults for all)."""
    if not share_plans:
        return False
    if k < 2:
        raise ValueError("share_plans=True needs agents_per_scene > 1: there are no scene mates to share plans with")
    if params is not None:
        dt = np.asarray(params, np.float64)[:, PARAM_INDEX["dt"]].reshape(-1, k)
        bad = np.flatnonzero((dt != dt[:, :1]).any(axis=1))
        if len(bad):
            raise ValueError(f"share_plans=True needs one dt per scene: scene {int(bad[0])} has dt {dt[bad[0]].tolist()}")
    return True


RIGHT_OF_WAY_RULES = {"fixed": _cabi.ROW_FIXED, "first_come": _cabi.ROW_FIRST_COME}


def right_of_way_setup(right_of_way, k: int, B: int, priority=None, junction=None):
    """Host-side checks of the right-of-way option of `BatchedEpisodes`.  Returns None without a rule, else
    (rule code of enum jmpc_right_of_way_rule, priority float64 [B] or None, junction float64 [1 or B / k, 3] or None).
    "fixed" takes priority [B] (finite; default: each episode's position j in its scene) and no junction; "first_come"
    takes junction = (x, y, r), once for all scenes or [B / k, 3], finite with r > 0, and no priority."""
    if right_of_way is None:
        if priority is not None or junction is not None:
            raise ValueError("priority / junction are arguments of a right-of-way rule: give right_of_way too")
        return None
    if right_of_way not in RIGHT_OF_WAY_RULES:
        raise ValueError(f"right_of_way must be None, 'fixed' or 'first_come', got {right_of_way!r}")
    if k < 2:
        raise ValueError("a right-of-way rule needs agents_per_scene > 1: there are no scene mates to yield to")
    if right_of_way == "fixed":
        if junction is not None:
            raise ValueError("the fixed rule takes no junction")
        if priority is None:
            return _cabi.ROW_FIXED, (np.arange(B) % k).astype(np.float64), None
        prio = np.asarray(priority, np.float64)
        if prio.shape != (B,):
            raise ValueError(f"priority must be [{B}] (one key per episode), got shape {prio.shape}")
        if not np.isfinite(prio).all():
            raise ValueError("priority must be finite")
        return _cabi.ROW_FIXED, np.ascontiguousarray(prio), None
    if priority is not None:
        raise ValueError("the first_come rule takes no priority: its keys come from the junction zone")
    if junction is None:
        raise ValueError("the first_come rule needs junction = (x, y, r)")
    junc = np.asarray(junction, np.float64)
    if junc.shape == (3,):
        junc = junc[None, :]
    if junc.shape not in ((1, 3), (B // k, 3)):
        raise ValueError(f"junction must be (x, y, r) or [{B // k}, 3] (one per scene), got shape {np.shape(junction)}")
    if not np.isfinite(junc).all() or not (junc[:, 2] > 0).all():
        raise ValueError("junction must be finite with r > 0")
    return _cabi.ROW_FIRST_COME, None, np.ascontiguousarray(junc)


ON_GOAL = ("park", "leave")


def lifetime_setup(depart, on_goal: str, k: int, B: int):
    """Host-side checks of the lifetime options of `BatchedEpisodes`.  Returns None when every vehicle is present from
    evaluation 0 and parks at its goal (depart None or all zero, on_goal "park": the run without lifetimes), else
    (depart int32 [B], leave).  depart: integer array [B] >= 0, the loop iteration of each vehicle's first step;
    on_goal "park" | "leave" (leave needs agents_per_scene > 1)."""
    if on_goal not in ON_GOAL:
        raise ValueError(f"on_goal must be 'park' or 'leave', got {on_goal!r}")
    leave = on_goal == "leave"
    if leave and k < 2:
        raise ValueError("on_goal='leave' needs agents_per_scene > 1: there are no scene mates to leave")
    if depart is None:
        dep = np.zeros(B, np.int32)
    else:
        dep = np.asarray(depart)
        if not np.issubdtype(dep.dtype, np.integer):
            raise ValueError(f"depart must be an integer array, got dtype {dep.dtype}")
        if dep.shape != (B,):
            raise ValueError(f"depart must be [{B}] (one entry iteration per episode), got shape {dep.shape}")
        if (dep < 0).any():
            raise ValueError("depart must be >= 0")
        if (dep > np.iinfo(np.int32).max).any():
            raise ValueError("depart must fit in int32")
    if not leave and not dep.any():
        return None
    return np.ascontiguousarray(dep, dtype=np.int32), leave


def _int_array(a, name: str, n: Optional[int] = None) -> np.ndarray:
    arr = np.asarray(a)
    if arr.ndim != 1 or not np.issubdtype(arr.dtype, np.integer):
        raise ValueError(f"{name} must be a 1-D integer array")
    if n is not None and len(arr) != n:
        raise ValueError(f"{name} must be [{n}] (one entry per trip), got shape {arr.shape}")
    return arr.astype(np.int64)


class Trips:
    """Validated trip arrays for `BatchedEpisodes.from_trips`.  Trip t: scene[t] (its scene), arrival[t] (integer >= 0,
    the earliest loop iteration of its first step), course_id[t] (a course id, or a plan index with `plans`),
    state[t] (x, y, v, yaw start state; omitted with plans, whose start states come from the planned courses),
    params[t] (NPARAM row; default the engine's defaults), priority[t] (the fixed rule's key; default the trip's
    rank in its scene's order) and group[t] (its signal group with `signals`, -1 = unsignalised)."""

    def __init__(self, scene, arrival, course_id, state=None, params=None, priority=None, group=None):
        self.scene = _int_array(scene, "scene")
        n = self.n = len(self.scene)
        if n < 1:
            raise ValueError("Trips needs at least one trip")
        self.arrival = _int_array(arrival, "arrival", n)
        if (self.arrival < 0).any():
            raise ValueError("arrival must be >= 0")
        if (self.arrival > np.iinfo(np.int32).max).any():
            raise ValueError("arrival must fit in int32")
        self.course_id = _int_array(course_id, "course_id", n)
        self.state = None if state is None else np.asarray(state, np.float64)
        if self.state is not None and self.state.shape != (n, 4):
            raise ValueError(f"state must be [{n}, 4], got shape {self.state.shape}")
        self.params = None if params is None else np.asarray(params, np.float64)
        if self.params is not None and self.params.shape != (n, NPARAM):
            raise ValueError(f"params must be [{n}, {NPARAM}], got shape {self.params.shape}")
        self.priority = None if priority is None else np.asarray(priority, np.float64)
        if self.priority is not None:
            if self.priority.shape != (n,):
                raise ValueError(f"priority must be [{n}] (one key per trip), got shape {self.priority.shape}")
            if not np.isfinite(self.priority).all():
                raise ValueError("priority must be finite")
        self.group = None if group is None else _int_array(group, "group", n)
        if self.group is not None and (self.group < -1).any():
            raise ValueError("group must be >= -1 (-1: unsignalised)")


def poisson_trips(n_scenes: int, routes, rate_per_hour: float, dt: float, n_iterations: int, entry_speed: float = 0.0,
                  seed: int = 0, groups=None) -> Trips:
    """Seeded Poisson demand: in every scene each approach (route group) of `routes` sends vehicles at rate_per_hour,
    with exponential gaps in seconds; a vehicle arriving at time a enters no earlier than iteration floor(a / dt), and
    arrivals from n_iterations on are dropped.  Each vehicle takes a route of its approach uniformly at random.
    routes[g] is a list of (course_id, (x, y, yaw)) pairs: the trip starts at that pose at entry_speed.  With
    (course_id, None) pairs (plan indices) the trips carry no state, for `from_trips(plans=...)`.  groups (one integer
    >= -1 per approach, or None) gives each trip the signal group of its approach (Trips.group); the draws do not
    depend on it."""
    if rate_per_hour < 0 or dt <= 0 or n_iterations < 0 or n_scenes < 1:
        raise ValueError("poisson_trips needs rate_per_hour >= 0, dt > 0, n_iterations >= 0 and n_scenes >= 1")
    if groups is not None:
        groups = np.asarray(groups)
        if groups.shape != (len(routes),) or not np.issubdtype(groups.dtype, np.integer) or (groups < -1).any():
            raise ValueError(f"groups must be {len(routes)} integers >= -1 (one signal group per approach)")
    rng = np.random.default_rng(seed)
    rate = rate_per_hour / 3600.0
    horizon = n_iterations * dt
    planned = all(pose is None for group in routes for _, pose in group)
    scene, arrival, cid, state, approach = [], [], [], [], []
    for s in range(n_scenes):
        for g, group in enumerate(routes):
            t = 0.0
            while rate > 0:
                t += rng.exponential(1.0 / rate)
                it = int(math.floor(t / dt))
                if t >= horizon or it >= n_iterations:
                    break
                course, pose = group[int(rng.integers(len(group)))]
                scene.append(s), arrival.append(it), cid.append(int(course)), approach.append(g)
                if not planned:
                    state.append([pose[0], pose[1], entry_speed, pose[2]])
    order = np.lexsort((np.arange(len(scene)), arrival, scene))
    take = lambda a: np.asarray(a)[order] if len(a) else np.zeros(0, np.int64)   # noqa: E731
    return Trips(take(scene), take(arrival), take(cid),
                 None if planned else np.asarray(state, np.float64).reshape(-1, 4)[order],
                 group=None if groups is None else groups[take(approach)])


def trips_setup(trips: Trips, n_scenes: int, k, n_courses: int, planned: bool, n_extra: int, right_of_way,
                share_plans: bool, params_default, depart=None, on_goal=None, obstacle_script=None, signals=None):
    """Host-side checks of `BatchedEpisodes.from_trips`.  Returns (order, params [N, NPARAM], priority or None): order
    sorts the trips by (scene, arrival, trip index), the layout the trips pass walks."""
    if depart is not None or on_goal is not None:
        raise ValueError("depart / on_goal do not apply to trips: a trip enters at its arrival and leaves at its goal")
    if obstacle_script is not None:
        raise ValueError("obstacle_script cannot be combined with trips: give obstacles or obstacle_program")
    if not isinstance(trips, Trips):
        raise ValueError("trips must be a Trips object")
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 2 <= k <= MAX_OBSTACLES + 1:
        raise ValueError(f"trips need agents_per_scene in [2, {MAX_OBSTACLES + 1}], got {k!r}")
    if (k - 1) + n_extra > MAX_OBSTACLES:
        raise ValueError(f"{k - 1} scene mates + {n_extra} obstacles exceed the {MAX_OBSTACLES} obstacle slots of an "
                         "episode")
    if isinstance(n_scenes, bool) or not isinstance(n_scenes, (int, np.integer)) or n_scenes < 1:
        raise ValueError(f"n_scenes must be an integer >= 1, got {n_scenes!r}")
    if trips.scene.min() < 0 or trips.scene.max() >= n_scenes:
        raise ValueError(f"trip scene out of range [0, {n_scenes})")
    if trips.course_id.min() < 0 or trips.course_id.max() >= n_courses:
        raise ValueError(f"trip course_id out of range [0, {n_courses})")
    if planned and trips.state is not None:
        raise ValueError("with plans the start states come from the planned courses: give no state")
    if not planned and trips.state is None:
        raise ValueError("trips need state [N, 4] unless plans are given")
    if trips.priority is not None and right_of_way != "fixed":
        raise ValueError("priority is an argument of the fixed right-of-way rule")
    if signals is None and trips.group is not None:
        raise ValueError("group is an argument of signals: give signals too")
    if signals is not None:
        signal_plan_check(signals, int(n_scenes))
        if trips.group is None:
            raise ValueError("signals need Trips.group (one signal group per trip, -1 = unsignalised)")
        signal_groups(trips.group, signals, "Trips.group")
    order = np.lexsort((np.arange(trips.n), trips.arrival, trips.scene))
    params = (np.repeat(np.asarray(params_default, np.float64)[None, :], trips.n, axis=0) if trips.params is None
              else trips.params)[order]
    if share_plans:
        dt = params[:, PARAM_INDEX["dt"]]
        scene = trips.scene[order]
        first = np.r_[True, scene[1:] != scene[:-1]]
        ref = dt[np.flatnonzero(first)[np.cumsum(first) - 1]]
        bad = np.flatnonzero(dt != ref)
        if len(bad):
            raise ValueError(f"share_plans=True needs one dt per scene: scene {int(scene[bad[0]])} has trips with dt "
                             f"{float(ref[bad[0]])} and {float(dt[bad[0]])}")
    priority = None
    if right_of_way == "fixed":
        if trips.priority is not None:
            priority = trips.priority[order]
        else:
            scene = trips.scene[order]
            start = np.searchsorted(scene, scene, side="left")
            priority = (np.arange(trips.n) - start).astype(np.float64)
    return order, np.ascontiguousarray(params), priority


class SignalPlan:
    """A fixed-time signal plan for `BatchedEpisodes(signals=...)` (jmpc_signals in include/jmpc.h).
    cycle: C >= 1 loop iterations.  green: one (start, length) window per signal group, 1 to 8 groups, start in [0, C),
    length in [0, C]; group g is green in loop iteration i of scene s iff ((i + offset[s] - start) mod C) < length, red
    otherwise (no amber state: the clearance time is the gap between windows).  junction: (x, y, r), r > 0; a
    vehicle's stop line is the first point of its course within r of (x, y), its zone entry e.  margin: course points
    between the cut and the stop line, L = e - margin (None: the run's collision margin).  stop_decel: the deceleration
    (m/s^2, finite, > 0) of the stopping test that decides, once per red phase, whether a vehicle holds at L or goes.
    offset: one integer per scene (None: 0), shifting each scene's cycle."""

    def __init__(self, cycle, green, junction, margin=None, stop_decel: float = 3.0, offset=None):
        i32 = np.iinfo(np.int32).max
        if isinstance(cycle, bool) or not isinstance(cycle, (int, np.integer)) or not 1 <= cycle <= i32:
            raise ValueError(f"cycle must be an integer >= 1, got {cycle!r}")
        self.cycle = int(cycle)
        win = np.asarray(green)
        if win.ndim != 2 or win.shape[1] != 2 or not 1 <= len(win) <= _cabi.SIGNAL_MAX_GROUPS:
            raise ValueError(f"green must be 1 to {_cabi.SIGNAL_MAX_GROUPS} (start, length) pairs, one per signal group")
        if not np.issubdtype(win.dtype, np.integer):
            raise ValueError("green windows must be integers (loop iterations)")
        if ((win[:, 0] < 0) | (win[:, 0] >= cycle)).any():
            raise ValueError(f"green start must be in [0, {cycle})")
        if ((win[:, 1] < 0) | (win[:, 1] > cycle)).any():
            raise ValueError(f"green length must be in [0, {cycle}]")
        self.green = win.astype(np.int64)
        junc = np.asarray(junction, np.float64)
        if junc.shape != (3,) or not np.isfinite(junc).all() or not junc[2] > 0:
            raise ValueError("junction must be (x, y, r), finite with r > 0")
        self.junction = junc
        if margin is not None and (isinstance(margin, bool) or not isinstance(margin, (int, np.integer))
                                   or not 0 <= margin <= i32):
            raise ValueError(f"margin must be None or an integer >= 0, got {margin!r}")
        self.margin = None if margin is None else int(margin)
        stop_decel = float(stop_decel)
        if not math.isfinite(stop_decel) or stop_decel <= 0:
            raise ValueError("stop_decel must be finite and > 0")
        self.stop_decel = stop_decel
        self.offset = None
        if offset is not None:
            off = np.asarray(offset)
            if off.ndim != 1 or not np.issubdtype(off.dtype, np.integer):
                raise ValueError("offset must be a 1-D integer array (one per scene)")
            if (np.abs(off.astype(np.int64)) > 2 ** 30).any():
                raise ValueError("offset must be within +-2**30")
            self.offset = off.astype(np.int32)

    @property
    def n_groups(self) -> int:
        return len(self.green)

    def struct(self, margin: int):
        """struct jmpc_signal_plan, with the run's `margin` where the plan has none."""
        p = _cabi.SignalPlan(cycle=self.cycle, n_groups=self.n_groups,
                             margin=int(margin if self.margin is None else self.margin), stop_decel=self.stop_decel)
        for g, (start, length) in enumerate(self.green):
            p.green_start[g], p.green_len[g] = int(start), int(length)
        return p


def signal_groups(group, signals: SignalPlan, name: str, n: Optional[int] = None) -> np.ndarray:
    """Checks per-vehicle (or per-trip) signal groups against the plan: integers in [-1, G).  Returns int32."""
    grp = np.asarray(group)
    if grp.ndim != 1 or not np.issubdtype(grp.dtype, np.integer):
        raise ValueError(f"{name} must be a 1-D integer array")
    if n is not None and len(grp) != n:
        raise ValueError(f"{name} must be [{n}] (one signal group per episode), got shape {grp.shape}")
    if ((grp < -1) | (grp >= signals.n_groups)).any():
        raise ValueError(f"{name} must be in [-1, {signals.n_groups}) (-1: unsignalised)")
    return np.ascontiguousarray(grp, dtype=np.int32)


def signal_plan_check(signals, n_scenes: int) -> None:
    """The plan against the run: a SignalPlan whose offset, if any, has one entry per scene.  The pass reads
    offset[b / k] on the device, where its length cannot be checked."""
    if not isinstance(signals, SignalPlan):
        raise ValueError("signals must be a SignalPlan")
    if signals.offset is not None and signals.offset.shape != (n_scenes,):
        raise ValueError(f"the plan's offset must be [{n_scenes}] (one per scene), got shape {signals.offset.shape}")


def signal_setup(signals, signal_group, B: int, k: int):
    """Host-side checks of the signals option of `BatchedEpisodes`.  Returns None without signals, else
    (group int32 [B], offset int32 [B / k] or None)."""
    if signals is None:
        if signal_group is not None:
            raise ValueError("signal_group is an argument of signals: give signals too")
        return None
    signal_plan_check(signals, B // k)
    if signal_group is None:
        raise ValueError("signals need signal_group [B] (one signal group per episode, -1 = unsignalised)")
    return signal_groups(signal_group, signals, "signal_group", B), signals.offset


TRIP_STATE = ("slot", "entry", "exit", "steps", "done", "blocked_waits")


def trip_holding(slot, entry, exit, k: int, obs, evaluation) -> np.ndarray:
    """The trip that held mate slot `obs` of trip t's slot at evaluation `evaluation` [N] (trip table columns slot,
    entry, exit [N]; a trip is in its slot at evaluations entry .. exit).  -1 where obs is -1 or an extra (>= k - 1)."""
    slot, entry, exit, obs, evaluation = (np.asarray(a, np.int64) for a in (slot, entry, exit, obs, evaluation))
    out = np.full(len(slot), -1, np.int64)
    held = np.flatnonzero(slot >= 0)
    q = np.flatnonzero((obs >= 0) & (obs < k - 1) & (slot >= 0))
    if not len(held) or not len(q):
        return out
    span = int(max(entry.max(), exit.max(), evaluation.max())) + 2
    key = slot[held] * span + entry[held]
    by = np.argsort(key, kind="stable")
    key, held = key[by], held[by]
    j = slot[q] % k
    mate = slot[q] - j + np.where(obs[q] < j, obs[q], obs[q] + 1)          # jmpc_scene_exchange's mate order
    pos = np.searchsorted(key, mate * span + evaluation[q], side="right") - 1
    u = held[np.maximum(pos, 0)]
    hit = (pos >= 0) & (slot[u] == mate) & (entry[u] <= evaluation[q]) & (evaluation[q] <= exit[u])
    out[q[hit]] = u[hit]
    return out


def outcome_columns(record) -> dict:
    """[B, >= len(OUTCOME_NAMES)] float64 outcome records -> dict of [B] arrays keyed by OUTCOME_NAMES (the index and
    count columns as int64)."""
    record = np.asarray(record, dtype=np.float64)
    if record.ndim != 2 or record.shape[1] < len(OUTCOME_NAMES):
        raise ValueError(f"outcome records must be [B, >= {len(OUTCOME_NAMES)}]")
    return {n: (record[:, k].astype(np.int64) if n in OUTCOME_INT else record[:, k].copy())
            for k, n in enumerate(OUTCOME_NAMES)}


def scripted_obstacles(specs, L: float = 2.86):
    """Device-side description of the reference's scripted obstacles (main/lib/moving_obstacles.py).

    specs: nested list [B][n_obs] of dicts with the constructor arguments of the reference classes:
      kind = "t_intersection" | "roundabout" | "arterial", direction, turning, speed, offset, dt, and for the arterial
      x_init, y_init, initial_speed.
    Returns (script [B, n_obs, 8], model [B, n_obs, 4]) float64 arrays for `BatchedEpisodes(obstacle_program=...)`:
    the constant script rows (enum jmpc_obs_script in include/jmpc.h) and the initial Bicycle state + step counter
    (start poses of moving_obstacles.py:52-61, 134-137, 190-199)."""
    B, n = len(specs), len(specs[0])
    script, model = np.zeros((B, n, 8)), np.zeros((B, n, 4))
    for b, row in enumerate(specs):
        if len(row) != n:
            raise ValueError("every episode needs the same number of obstacles")
        for k, s in enumerate(row):
            kind = OBS_KINDS[s["kind"]]
            direction = 1.0 if s.get("direction", 1) >= 0 else -1.0
            dt = float(s.get("dt", 0.2))
            offset = s.get("offset")
            aux = float(np.arctan((1 / 5) * 2.86)) if kind == 2 else float(s.get("initial_speed", 0.0))
            script[b, k] = [kind, direction, 1.0 if s.get("turning", False) else 0.0, float(s.get("speed", 25 / 3.6)),
                            -1.0 if (offset is None or offset <= 0) else float(offset), dt, 0.2 if kind == 2 else dt, aux]
            if kind == 3:
                model[b, k] = [float(s["x_init"]), float(s["y_init"]), np.pi / 2, 0.0]
            elif direction > 0:
                model[b, k] = [-30.0, -3.0, 0.0, 0.0]
            else:
                model[b, k] = [30.0, 3.0, np.pi, 0.0]
    return script, model


def plan_episode_setup(course_ok, course_dl, plan_id, n_plans: int, car_radius: float):
    """Host-side checks of `BatchedEpisodes.from_plans`: returns (plan_id as int32 [B], margin).
    plan_id None -> one episode per plan.  The margin is EXTRA_CUTOFF_MARGIN = 4 * ceil(radius / dl)
    (mpc_intersection.py:87-88) over the usable courses the episodes drive; it is one scalar for the batch, so courses
    that disagree on it are an error (0 when no episode has a usable course)."""
    course_ok, course_dl = np.asarray(course_ok), np.asarray(course_dl, np.float64)
    if course_ok.shape != (n_plans,) or course_dl.shape != (n_plans,):
        raise ValueError(f"course_ok / course_dl must be [{n_plans}]")
    pid = np.arange(n_plans, dtype=np.int64) if plan_id is None else np.asarray(plan_id)
    if pid.ndim != 1 or len(pid) < 1 or not np.issubdtype(pid.dtype, np.integer):
        raise ValueError("plan_id must be a non-empty 1-D integer array")
    if pid.min() < 0 or pid.max() >= n_plans:
        raise ValueError(f"plan_id out of range [0, {n_plans})")
    used = np.unique(pid[course_ok[pid] != 0])
    margins = {4 * int(math.ceil(car_radius / float(course_dl[c]))) for c in used}
    if len(margins) > 1:
        raise ValueError(f"the planned courses disagree on the cut-off margin 4 * ceil(radius / dl): {sorted(margins)}")
    return np.ascontiguousarray(pid, dtype=np.int32), (margins.pop() if margins else 0)


class BatchedEpisodes:
    @classmethod
    def from_plans(cls, engine: BatchedMPC, plans, plan_id=None, params=None, obstacle_program=None, obstacles=None,
                   frame_window: int = 10, max_steps: int = 256, record_history: bool = True, horizon_s: float = 7.0,
                   obstacle_script=None, outcomes: bool = False, record_obstacles: bool = False,
                   agents_per_scene: int = 1, share_plans: bool = False, right_of_way=None, priority=None,
                   junction=None, depart=None, on_goal: str = "park", signals=None,
                   signal_group=None) -> "BatchedEpisodes":
        """Episodes on the planned courses of `engine` (filled by `BatchedMPC.from_plans(plans)` /
        `set_courses_from_plans(plans)`), the second half of main/scenarios/mpc_intersection.py:63-163 for a batch:
        episode b drives plan `plan_id[b]` (default: one episode per plan; zeros = one course, many controllers).
        Its start state (the course's first pose at v = 0), its params row `dl` and done = 3 for a plan without a usable
        course are written on the device (jmpc_episode_init_from_courses); such episodes are never stepped.
        `params` [B, NPARAM] (default: the engine's defaults) supplies every other parameter row.  `run()` adds
        plan_status, plan_cost and expansions per episode.  `outcomes` / `record_obstacles` / `agents_per_scene` /
        `share_plans` / `right_of_way` / `priority` / `junction` / `depart` / `on_goal` / `signals` / `signal_group` as
        in `__init__`; evaluation 0 of the outcome record sees the planned start states; the junction zones and stop
        lines are found on the planned courses, and first_come distances and the signals' stopping test use
        each course's dl.  With agents_per_scene > 1 a scene with a done = 3 vehicle is not driven: its other vehicles get
        done = 4 (jmpc_scene_init); such vehicles never wait either: the waiting code is set after this pass."""
        if engine.course_ok is None or len(engine.course_ok) != len(plans):
            raise ValueError("the engine's courses do not come from these plans (BatchedMPC.from_plans)")
        import torch
        pid, margin = plan_episode_setup(engine._ok_host, engine._dl_host, plan_id, len(plans), engine.car_radius)
        B = len(pid)
        if params is None:
            params = np.repeat(engine.default_params[None, :], B, axis=0)
        elif np.shape(params) != (B, NPARAM):
            raise ValueError(f"params must be [{B}, {NPARAM}]")
        ep = cls(engine, np.zeros((B, 4)), course_id=pid, obstacles=obstacles, obstacle_script=obstacle_script,
                 frame_window=frame_window, margin=margin, params=params, max_steps=max_steps,
                 record_history=record_history, horizon_s=horizon_s, obstacle_program=obstacle_program,
                 outcomes=outcomes, record_obstacles=record_obstacles, agents_per_scene=agents_per_scene,
                 share_plans=share_plans, right_of_way=right_of_way, priority=priority, junction=junction,
                 depart=depart, on_goal=on_goal, signals=signals, signal_group=signal_group)
        stream = C.c_void_p(torch.cuda.current_stream(engine.device).cuda_stream)
        _cabi.check(engine._lib.jmpc_episode_init_from_courses(
            engine._h, B, ep._p(ep.course_id), ep._p(engine.course_ok), ep._p(engine.course_dl), ep._p(ep.state),
            ep._p(ep.params), ep._p(ep.done), stream), "jmpc_episode_init_from_courses")
        if ep.k > 1:
            _cabi.check(engine._lib.jmpc_scene_init(engine._h, B, ep.k, ep._p(ep.done), stream), "jmpc_scene_init")
        ep._plans = (plans, ep.course_id.long())
        return ep

    @classmethod
    def from_trips(cls, engine: BatchedMPC, trips: Trips, n_scenes: int, agents_per_scene: int = 4, plans=None,
                   entry_gap: float = 2.0, obstacles=None, obstacle_program=None, frame_window: int = 10,
                   margin: int = 72, max_steps: int = 256, record_history: bool = True, horizon_s: float = 7.0,
                   outcomes: bool = False, record_obstacles: bool = False, share_plans: bool = False,
                   right_of_way=None, junction=None, depart=None, on_goal=None,
                   obstacle_script=None, signals=None) -> "BatchedEpisodes":
        """Scenes fed from a stream of timed trips (jmpc_scene_trips / jmpc_scene_trips_finish in include/jmpc.h).
        The batch is n_scenes x k slots (episode b = s * k + j is slot j of scene s, k in [2, 9]); a slot holds at most
        one trip at a time and starts empty.  An empty slot is handled as a vehicle that has not entered under lifetimes:
        not stepped, absent for its mates, NaN obstacle_history rows, its extras keep the loop's clock.  Once before
        evaluation 0 and then in every loop iteration i (after the extras advance, before the exchange) the trips pass
        closes the trips whose goal test fired (they always leave at the goal; a done = 2 vehicle keeps its slot), then
        admits the scene's due trips (arrival <= i + 1) in (arrival, trip index) order into the lowest empty slot, when
        their start pose has a clearance >= entry_gap metres to every vehicle in the scene and to every earlier trip
        still pending (first-in, first-out per approach).  A trip whose planned course is unusable is closed with
        done = 3.  An admitted slot is a fresh vehicle on the trip's course, params row and start state, entering at
        evaluation i + 1 (entry).  run() stops when no slot is driving and no trip is pending, and adds `trips`.

        trips: a `Trips` object; with `plans` (a planner result whose courses `engine` holds, as for from_plans) its
        course_id are plan indices and the start states, dl and usability come from the planned courses.  The other
        options are those of `__init__`: obstacles / obstacle_program are per-slot extras; share_plans needs one dt per
        scene across its trips; right_of_way "fixed" takes the trips' priority (default: rank in the scene's order),
        "first_come" a junction (once or per scene); signals takes each trip's group from Trips.group (the latch,
        hold_steps and go belong to the trip; run() also gives the per-slot counts).  depart, on_goal and
        obstacle_script do not apply to trips."""
        import torch
        n_extra = 0
        if obstacles is not None:
            n_extra = int(np.shape(obstacles)[1])
        elif obstacle_program is not None:
            n_extra = int(np.shape(obstacle_program[0])[1])
        planned = plans is not None
        if planned and (engine.course_ok is None or len(engine.course_ok) != len(plans)):
            raise ValueError("the engine's courses do not come from these plans (BatchedMPC.from_plans)")
        n_courses = len(plans) if planned else len(engine.course_len)
        k = agents_per_scene
        order, params, priority = trips_setup(trips, n_scenes, k, n_courses, planned, n_extra, right_of_way,
                                              share_plans, engine.default_params, depart, on_goal, obstacle_script,
                                              signals)
        entry_gap = float(entry_gap)
        if not math.isfinite(entry_gap) or entry_gap < 0:
            raise ValueError("entry_gap must be finite and >= 0")
        if planned:
            _, margin = plan_episode_setup(engine._ok_host, engine._dl_host, trips.course_id, len(plans),
                                           engine.car_radius)
        k, B, N = int(k), int(n_scenes) * int(k), trips.n
        if B > engine.max_batch:
            raise ValueError(f"n_scenes * k = {B} exceeds the engine's max_batch {engine.max_batch}")
        row = right_of_way_setup(right_of_way, k, B, None, junction)
        ep = cls(engine, np.zeros((B, 4)), course_id=np.zeros(B, np.int32), obstacles=obstacles,
                 obstacle_program=obstacle_program, frame_window=frame_window, margin=margin,
                 params=np.repeat(engine.default_params[None, :], B, axis=0), max_steps=max_steps,
                 record_history=record_history, horizon_s=horizon_s, outcomes=outcomes,
                 record_obstacles=record_obstacles, agents_per_scene=k, share_plans=share_plans, on_goal="leave")
        dev, i32, f64 = ep.dev, torch.int32, torch.float64
        t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)   # noqa: E731
        lib, h = engine._lib, engine._h
        stream = C.c_void_p(torch.cuda.current_stream(engine.device).cuda_stream)
        scene = trips.scene[order]
        T = dict(scene_start=t(np.searchsorted(scene, np.arange(n_scenes + 1)), i32), arrival=t(trips.arrival[order], i32),
                 course_id=t(trips.course_id[order], i32), params=t(params, f64))
        T["course_len"] = torch.as_tensor(engine.course_len, dtype=i32, device=dev)[T["course_id"].long()].contiguous()
        usable = torch.zeros(N, dtype=i32, device=dev)          # jmpc_episode_init_from_courses writes 3 where unusable
        T["start"] = t(np.zeros((N, 4)) if planned else trips.state[order], f64)
        if planned:
            for a in range(0, N, engine.max_batch):
                n = min(engine.max_batch, N - a)
                _cabi.check(lib.jmpc_episode_init_from_courses(
                    h, n, ep._p(T["course_id"][a:]), ep._p(engine.course_ok), ep._p(engine.course_dl),
                    ep._p(T["start"][a:]), ep._p(T["params"][a:]), ep._p(usable[a:]), stream),
                    "jmpc_episode_init_from_courses")
        T["usable"] = (usable == 0).to(i32)
        bad = np.where(T["usable"].cpu().numpy() == 0, np.arange(N), N)     # the first unusable trip at or after t
        T["next_unusable"] = t(np.minimum.accumulate(bad[::-1])[::-1], i32)
        T["zone"] = T["priority"] = None
        if row is not None:
            ep.row_rule, _, junc = row
            ep.consider = torch.full((B,), -1, dtype=i32, device=dev)
            ep._collision_mask = ep.consider
            if junc is not None:
                ep.junction = t(junc, f64)
                ep.zone = torch.full((B, 2), -1, dtype=i32, device=dev)
                per_trip = t(junc[scene] if len(junc) > 1 else np.repeat(junc, N, axis=0), f64)
                T["zone"] = torch.empty(N, 2, dtype=i32, device=dev)
                for a in range(0, N, engine.max_batch):
                    n = min(engine.max_batch, N - a)
                    _cabi.check(lib.jmpc_right_of_way_init(
                        h, n, 1, ep._p(T["course_id"][a:]), ep._p(per_trip[a:]), n, ep._p(T["zone"][a:]), stream),
                        "jmpc_right_of_way_init")
            else:
                ep.priority = torch.zeros(B, dtype=f64, device=dev)
                T["priority"] = t(priority, f64)
        z = lambda v: torch.full((N,), v, dtype=i32, device=dev)   # noqa: E731
        T.update(cursor=T["scene_start"][:-1].clone(), pending=t(np.bincount(scene, minlength=n_scenes), i32),
                 phase=z(0), slot_trip=torch.full((B,), -1, dtype=i32, device=dev), slot=z(-1), entry=z(-1),
                 exit=z(-1), steps=z(0), done=z(_cabi.WAITING), blocked_waits=z(0),
                 outcomes=(torch.full((N, len(OUTCOME_NAMES)), 0.0, dtype=f64, device=dev) if ep.outcomes is not None
                           else None))
        if T["outcomes"] is not None:                          # the empty record, for trips that never drive
            T["outcomes"][:, OUTCOME_NAMES.index("min_clearance")] = math.inf
            for c in ("min_clearance_eval", "min_clearance_obs", "first_contact_eval", "first_contact_obs"):
                T["outcomes"][:, OUTCOME_NAMES.index(c)] = -1.0
        ep.done.fill_(_cabi.WAITING)
        if signals is not None:                                # per trip: its group and stop line; owner = slot_trip
            same = T["zone"] is not None and bool((junc == signals.junction).all())
            zone = T["zone"] if same else ep._zones(T["course_id"], signals.junction)   # first_come's zones if equal
            ep._signals_init(signals, t(trips.group[order], i32), zone, N, owner=T["slot_trip"])
        ep._trips = T
        ep._trip_order = order
        ep._trips_struct = _cabi.Trips(
            n_scenes=int(n_scenes), k=k, n_trips=N, T=ep.T, entry_gap=entry_gap,
            **{n: T[n].data_ptr() if T[n] is not None else None for n in (
                "scene_start", "arrival", "course_id", "course_len", "usable", "next_unusable", "start", "params",
                "zone", "priority", "cursor", "pending", "phase", "slot_trip", "slot", "entry", "exit", "steps", "done",
                "blocked_waits", "outcomes")},
            state=ep.state.data_ptr(), ep_course_id=ep.course_id.data_ptr(), ep_params=ep.params.data_ptr(),
            ep_course_len=ep.course_len.data_ptr(), target_ind=ep.target_ind.data_ptr(),
            agent_idx=ep.agent_idx.data_ptr(), ep_steps=ep.steps.data_ptr(), warm=ep.warm.data_ptr(),
            flag=ep.flag.data_ptr(), di=ep.di.data_ptr(), oa=ep.oa.data_ptr(), od=ep.od.data_ptr(),
            ep_zone=None if ep.zone is None else ep.zone.data_ptr(),
            ep_priority=None if T["priority"] is None else ep.priority.data_ptr(), depart=ep.depart.data_ptr(),
            ep_done=ep.done.data_ptr(), ep_outcomes=None if ep.outcomes is None else ep.outcomes.data_ptr())
        return ep

    def _trips_pass(self, initial: int):
        e = self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(e._lib.jmpc_scene_trips(e._h, C.byref(self._trips_struct), self._p(self.iter_dev), int(initial),
                                            stream), "jmpc_scene_trips")

    def _trip_table(self) -> dict:
        """The trip table in the caller's trip order (jmpc_scene_trips_finish first)."""
        e, T = self.e, self._trips
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(e._lib.jmpc_scene_trips_finish(e._h, C.byref(self._trips_struct), self.iteration, stream),
                    "jmpc_scene_trips_finish")
        order = self._trip_order
        N = len(order)

        def back(a):
            out = np.empty((N,) + a.shape[1:], a.dtype)
            out[order] = a
            return out
        scene_sorted = np.repeat(np.arange(len(T["scene_start"]) - 1), np.diff(T["scene_start"].cpu().numpy()))
        res = dict(scene=back(scene_sorted.astype(np.int64)), arrival=back(T["arrival"].cpu().numpy().astype(np.int64)))
        for n in TRIP_STATE:
            res[n] = back(T[n].cpu().numpy().astype(np.int64))
        # every pass in which a trip is due and pending waits for a slot or is blocked: the passes of entries
        # arrival .. entry - 1, or arrival .. self.iteration for a trip still pending
        due = np.where(res["entry"] >= 0, res["entry"] - res["arrival"],
                       np.where(res["done"] == _cabi.WAITING, np.maximum(self.iteration + 1 - res["arrival"], 0), 0))
        res["slot_waits"] = due - res["blocked_waits"]
        res["entry_delay"] = np.where(res["entry"] >= 0, res["entry"] - res["arrival"], -1)
        res["travel"] = np.where((res["entry"] >= 0) & (res["exit"] >= 0), res["exit"] - res["entry"], -1)
        if self.signals is not None:
            res["signal_hold_steps"] = back(self.signal_hold.cpu().numpy().astype(np.int64))
            res["signal_go"] = back(self.signal_go.cpu().numpy().astype(np.int64))
        if T["outcomes"] is not None:
            res.update(outcome_columns(back(T["outcomes"].cpu().numpy())))
            for col in ("min_clearance", "first_contact"):
                res[f"{col}_trip"] = trip_holding(res["slot"], res["entry"], res["exit"], self.k,
                                                  res[f"{col}_obs"], res[f"{col}_eval"])
        return res

    def __init__(self, engine: BatchedMPC, state0, course_id=None, obstacles=None, obstacle_script=None,
                 frame_window: int = 10, margin: int = 72, params=None, max_steps: int = 256,
                 record_history: bool = True, horizon_s: float = 7.0, obstacle_program=None, outcomes: bool = False,
                 record_obstacles: bool = False, agents_per_scene: int = 1, share_plans: bool = False,
                 right_of_way=None, priority=None, junction=None, depart=None, on_goal: str = "park",
                 signals=None, signal_group=None):
        """outcomes: keep one outcome record per episode on the device (jmpc_episode_outcomes): contact and clearance
        against the obstacles, cut / limit steps, failed solves, comfort and tracking columns; `run()` returns it as
        `outcomes`.  It observes only: the episodes are exactly those of outcomes=False.  record_obstacles (needs
        outcomes): also keep the obstacle poses of every evaluation, `run()`'s `obstacle_history`
        [iterations + 1, B, n_obs, 6], whose row i + 1 is simultaneous with History row i.

        agents_per_scene = k > 1: k consecutive episodes form a scene of MPC-driven vehicles that see each other as
        moving obstacles (jmpc_scene_exchange in include/jmpc.h).  Each episode's obstacle slots are its k - 1 scene mates
        in episode order (itself skipped), then its own `obstacles` / `obstacle_program` (n_extra of them), at most 8
        in all; the outcome record's *_obs columns index these slots.  A mate's row is its state and the (a, clamped
        steer) it last applied; a finished mate stays parked at its last pose with v = a = steer = 0.  All vehicles move
        simultaneously: the rows iteration i + 1 reads are those after iteration i.  k = 1 is the single-vehicle loop,
        with nothing launched or allocated for scenes.

        share_plans (needs k > 1 and one dt per scene): each vehicle predicts its mates along their MPC plans instead of
        holding their last applied (a, steer) for the whole horizon (jmpc_scene_plans / jmpc_collision_planned in
        include/jmpc.h).  The mate rows, the outcome record and obstacle_history are unchanged; only the prediction of
        the mate slots changes.  A mate's plan is the rest of its last solve, oa / od[1:], its last input held past the
        end; a mate that is done, or has no usable warm start (before its first step, after a failed solve), is
        predicted from its row as without the option.  Extras keep their constant-input prediction.

        right_of_way = "fixed" | "first_come" (needs k > 1; None: every mate is considered, as before): a rule that
        decides which moving mates a vehicle yields to (jmpc_right_of_way / jmpc_collision_masked in include/jmpc.h).
        Every iteration, after the goal test, each vehicle gets a consider mask (`consider` [B] int32, bit s = obstacle
        slot s takes part in its collision cut).  Extras and parked mates (done != 0) are always considered; a moving
        mate only if its key (class, key, episode index) is smaller than the vehicle's own, so no cycle of waiting can
        form.  The rule changes nothing else: the mate rows, obstacle_history and the outcome record are unchanged, and
        contacts with ignored mates are still measured.
          "fixed": class 0, key priority[b] (float64 [B], finite; default: the position j of b in its scene).
          "first_come": junction = (x, y, r), for all scenes or [B / k, 3].  entry / exit are the first and last points
          of b's course within r of the centre (jmpc_right_of_way_init, `zone` [B, 2]; -1 when it never enters), a its
          course index, dl its params' dl: committed (a >= entry) class 0, key (exit - a) dl; approaching class 1,
          key (entry - a) dl; a course that never enters the zone class 2 (it yields to every moving mate).

        depart (integer [B] >= 0; None = all zeros) and on_goal = "park" | "leave": each vehicle's lifetime in its scene
        (jmpc_scene_depart_init / jmpc_scene_enter / jmpc_scene_presence / jmpc_episode_outcomes_scene in
        include/jmpc.h).  Vehicle b takes its first step in loop iteration depart[b]; until then it waits at its start
        state with done = WAITING (5): not stepped, not goal-tested, no History row, absent for its mates.  It enters
        between iteration depart[b] - 1 and evaluation depart[b] with its start state, speed kept.  Its extras follow the
        loop's clock while it waits, so at entry it sees what a depart = 0 vehicle sees then.  With "leave" (needs k > 1)
        a vehicle whose goal test fires at the top of iteration g is present in evaluation g and absent from iteration
        g's collision check on; done = 2 (index rule) stays parked under both.  Absent mates take no part in the
        collision cut (with a rule: the rule's mask AND presence, written into `consider`), and add no clearance or
        contact to the outcome record, whose obstacle_history rows for them are NaN.  A vehicle's outcome record starts
        at evaluation depart[b]; the *_eval columns stay global evaluation indices, and `steps` counts its own steps.
        A vehicle that has not entered when the run ends keeps done = WAITING.  depart all zero with "park" is the run
        without lifetimes, with nothing launched or allocated for them.

        signals (a `SignalPlan`) and signal_group (integer [B] in [-1, G), -1 = unsignalised): fixed-time traffic
        signals (jmpc_signals in include/jmpc.h).  Vehicle b's stop line is e, the first point of its course within the
        plan's junction (jmpc_right_of_way_init; a course that never enters it is unsignalised), and its cut point is
        L = e - margin.  Every iteration, after the collision check and before the step, a vehicle whose group is red
        decides once per red phase: it holds iff a < L and v * v <= 2 stop_decel (L - 1 - a) dl (a its course index,
        v its speed, dl its params' dl), else it goes.  A held vehicle's course is cut at max(a + 1, L) as a collision
        cut is, until it sees green; a vehicle that goes is left alone, and one that goes with a < L (it could not
        stop) counts a GO pass.  run() adds `signal_hold_steps` and `signal_go` per episode.  The collision flag,
        History, the outcome record and the masks are unchanged: a signal stop is not a cut step.  signals=None
        launches and allocates nothing for signals."""
        import torch
        self.torch = torch
        self.e = engine
        self.dev = torch.device("cuda", engine.device)
        f64, i32 = torch.float64, torch.int32
        t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=self.dev)  # noqa: E731
        self.state = t(state0, f64)
        self.B = B = self.state.shape[0]
        self.T = engine.T
        self.course_id = t(course_id, i32)
        self.params = t(params, f64)
        self.obstacles = t(obstacles, f64)                       # [B, n_obs, 6], advanced on the device
        self.script = t(obstacle_script, f64)                    # [S, B, n_obs, 6], read per step
        self.program = None
        if obstacle_program is not None:                         # the reference's scripted obstacles, stepped on the device
            if obstacles is not None or obstacle_script is not None:
                raise ValueError("give one of obstacles / obstacle_script / obstacle_program")
            self.program = (t(obstacle_program[0], f64), t(obstacle_program[1], f64))
            self.obstacles = torch.zeros(B, self.program[0].shape[1], 6, dtype=f64, device=self.dev)
        if self.obstacles is not None and self.script is not None:
            raise ValueError("give either constant-input obstacles or a script")
        self.frame_window, self.margin, self.horizon_s = int(frame_window), int(margin), float(horizon_s)
        self.max_steps = int(max_steps)
        full = torch.as_tensor(engine.course_len, dtype=i32, device=self.dev)
        self.full_len = full[self.course_id.long()] if self.course_id is not None else full[0].expand(B).contiguous()
        self.course_len = self.full_len.clone()
        z = lambda: torch.zeros(B, dtype=i32, device=self.dev)   # noqa: E731
        self.agent_idx, self.target_ind, self.done, self.steps, self.warm, self.flag = z(), z(), z(), z(), z(), z()
        self.di = torch.zeros(B, dtype=f64, device=self.dev)
        self.v = torch.zeros(B, dtype=f64, device=self.dev)
        self.oa = torch.zeros(B, self.T, dtype=f64, device=self.dev)
        self.od = torch.zeros(B, self.T, dtype=f64, device=self.dev)
        self.out = engine.alloc_outputs(B)
        self.history = torch.full((self.max_steps, B, 8), float("nan"), dtype=f64, device=self.dev) if record_history else None
        self.flags = torch.zeros(self.max_steps, B, dtype=i32, device=self.dev) if record_history else None
        self.iteration = 0
        self.iter_dev = torch.zeros(1, dtype=i32, device=self.dev)     # the same counter on the device (graph replay)
        self._plans = None                                           # (DevicePlanBatch, plan index per episode): from_plans
        n_obs = 0
        if self.obstacles is not None:
            n_obs = int(self.obstacles.shape[1])
        elif self.script is not None:
            n_obs = int(self.script.shape[2])
        n_obs = scene_setup(B, agents_per_scene, n_obs, self.script is not None)
        self.k = int(agents_per_scene)
        # k > 1: the obstacle rows every kernel reads, written by jmpc_scene_exchange from the vehicles and the extras
        self.scene_obs = torch.empty(B, n_obs, 6, dtype=f64, device=self.dev) if self.k > 1 else None
        # share_plans: the mates' remaining plans [B, k - 1, T - 1, 2], written by jmpc_scene_plans after every exchange
        self.scene_plans = (torch.empty(B, self.k - 1, self.T - 1, 2, dtype=f64, device=self.dev)
                            if plan_share_setup(share_plans, self.k, params) else None)
        self.n_obs = n_obs
        # right_of_way: the per-episode consider mask (jmpc_right_of_way, every iteration) and the rule's constant inputs
        self.consider = self.zone = self.priority = self.junction = None
        row = right_of_way_setup(right_of_way, self.k, B, priority, junction)
        if row is not None:
            self.row_rule, prio, junc = row
            self.consider = torch.full((B,), -1, dtype=i32, device=self.dev)
            self.priority = t(prio, f64)
            if junc is not None:
                # the course ids are final here (from_plans passes its plan ids): the zones are found once
                self.junction = t(junc, f64)
                self.zone = torch.empty(B, 2, dtype=i32, device=self.dev)
                stream = C.c_void_p(torch.cuda.current_stream(engine.device).cuda_stream)
                _cabi.check(engine._lib.jmpc_right_of_way_init(
                    engine._h, B, self.k, self._p(self.course_id), self._p(self.junction), int(junc.shape[0]),
                    self._p(self.zone), stream), "jmpc_right_of_way_init")
        # signals: per-episode group and stop line, the latch and the counters (jmpc_signals, every iteration)
        self.signals = None
        sig = signal_setup(signals, signal_group, B, self.k)
        if sig is not None:
            self._signals_init(signals, t(sig[0], i32), self._zones(self.course_id, signals.junction), B)
        # lifetimes: depart [B] int32; the collision mask (a rule's `consider` ANDed with presence, or presence alone)
        # and the evaluation mask `presence` [B], both written by jmpc_scene_presence every iteration (k > 1)
        self.depart = self.presence = None
        self._collision_mask = self.consider
        self._leave = self._entering = False
        life = lifetime_setup(depart, on_goal, self.k, B)
        if life is not None:
            dep, self._leave = life
            self.depart = t(dep, i32)
            self._entering = bool(dep.any())
            if self.k > 1:
                self.presence = torch.full((B,), -1, dtype=i32, device=self.dev)
                if self._collision_mask is None:
                    self._collision_mask = torch.full((B,), -1, dtype=i32, device=self.dev)
        self.outcomes = self.obstacle_history = None
        if outcome_setup(outcomes, record_obstacles, n_obs):
            self.outcomes = torch.empty(B, OUTCOME_LEN, dtype=f64, device=self.dev)     # evaluation 0 fills it
            if record_obstacles:
                self.obstacle_history = torch.full((self.max_steps + 1, B, n_obs, 6), float("nan"), dtype=f64,
                                                   device=self.dev)
        self._trips = None                                            # from_trips: the trip arrays and table
        self._started = False
        if self.program is not None:                                 # get() before the first iteration
            self._scripted_step(advance=0)

    def _zones(self, course_id, junction):
        """(entry, exit) [n, 2] int32 of every course in course_id [n] (None: course 0 for all B episodes) in the zone
        junction = (x, y, r) (jmpc_right_of_way_init, in launches of at most max_batch)."""
        torch, e = self.torch, self.e
        stream = C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)
        n = self.B if course_id is None else int(course_id.shape[0])
        junc = torch.as_tensor(np.asarray(junction, np.float64)[None, :], device=self.dev)
        zone = torch.empty(n, 2, dtype=torch.int32, device=self.dev)
        for a in range(0, n, e.max_batch):
            m = min(e.max_batch, n - a)
            _cabi.check(e._lib.jmpc_right_of_way_init(
                e._h, m, 1, None if course_id is None else self._p(course_id[a:]), self._p(junc), 1,
                self._p(zone[a:]), stream), "jmpc_right_of_way_init")
        return zone

    def _signals_init(self, signals: "SignalPlan", group, zone, n_owner: int, owner=None):
        """The signal pass's arrays: group and zone [n_owner], the latch [B, 2] = (-1, 0), the counters per owner and,
        with an owner array (trips), per slot."""
        torch, i32 = self.torch, self.torch.int32
        self._signal_plan = signals.struct(self.margin)
        if not 0 <= self._signal_plan.margin <= self.e.max_N:
            raise ValueError(f"the signal margin must be in [0, {self.e.max_N}] (the engine's max_N), got "
                             f"{self._signal_plan.margin}")
        self.signals = signals
        self.signal_offset = (None if signals.offset is None
                              else torch.as_tensor(signals.offset, dtype=i32, device=self.dev))
        self.signal_group, self.signal_zone, self.signal_owner = group, zone, owner
        self.signal_latch = torch.zeros(self.B, 2, dtype=i32, device=self.dev)
        self.signal_latch[:, 0] = -1
        self.signal_hold = torch.zeros(n_owner, dtype=i32, device=self.dev)
        self.signal_go = torch.zeros(n_owner, dtype=i32, device=self.dev)
        self.signal_slot_hold = self.signal_slot_go = None
        if owner is not None:
            self.signal_slot_hold = torch.zeros(self.B, dtype=i32, device=self.dev)
            self.signal_slot_go = torch.zeros(self.B, dtype=i32, device=self.dev)

    def _signal_pass(self, checked: bool):
        e = self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(e._lib.jmpc_signals(
            e._h, self.B, self.k, C.byref(self._signal_plan), self._p(self.signal_offset), self._p(self.signal_owner),
            self._p(self.signal_group), self._p(self.signal_zone), self._p(self.course_id), self._p(self.agent_idx),
            self._p(self.state), self._p(self.params), self._p(self.done), int(checked), self._p(self.course_len),
            self._p(self.signal_latch), self._p(self.signal_hold), self._p(self.signal_go),
            self._p(self.signal_slot_hold), self._p(self.signal_slot_go), self._p(self.iter_dev), stream),
            "jmpc_signals")

    def _scripted_step(self, advance: int):
        e = self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(e._lib.jmpc_scripted_obstacle_step(
            e._h, self.B, int(self.program[0].shape[1]), self._p(self.program[0]), self._p(self.program[1]),
            self._p(self.obstacles), self._p(self.done), int(advance), stream), "jmpc_scripted_obstacle_step")

    def _outcome_eval(self, obs, initial: int):
        """Evaluation 0 (initial) or i + 1 of the outcome record; obs: the obstacle poses of that instant."""
        e, torch = self.e, self.torch
        stream = C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)
        has_obs = obs is not None and self.n_obs > 0
        if self.depart is not None:
            _cabi.check(e._lib.jmpc_episode_outcomes_scene(
                e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(obs) if has_obs else None,
                self.n_obs if has_obs else 0, self._p(self.out.record), self._p(self.di),
                self._p(self.flag) if has_obs else None, self._p(self.params), self._p(self.done),
                self._p(self.presence), self._p(self.depart), self._p(self.iter_dev), int(initial),
                self._p(self.outcomes), self._p(self.obstacle_history), self.max_steps, stream),
                "jmpc_episode_outcomes_scene")
            return
        _cabi.check(e._lib.jmpc_episode_outcomes(
            e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(obs) if has_obs else None,
            self.n_obs if has_obs else 0, self._p(self.out.record), self._p(self.di),
            self._p(self.flag) if has_obs else None, self._p(self.params), self._p(self.done), self._p(self.iter_dev),
            int(initial), self._p(self.outcomes), self._p(self.obstacle_history), self.max_steps, stream),
            "jmpc_episode_outcomes")

    def _scene_exchange(self):
        """The obstacle rows of every episode from its scene mates' states and its own extras (jmpc_scene_exchange), and
        with share_plans the mates' plans (jmpc_scene_plans)."""
        e = self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        n_extra = 0 if self.obstacles is None else int(self.obstacles.shape[1])
        _cabi.check(e._lib.jmpc_scene_exchange(
            e._h, self.B, self.k, n_extra, self._p(self.state), self._p(self.out.record), self._p(self.di),
            self._p(self.params), self._p(self.done), self._p(self.steps), self._p(self.obstacles) if n_extra else None,
            self._p(self.scene_obs), stream), "jmpc_scene_exchange")
        if self.scene_plans is not None:
            _cabi.check(e._lib.jmpc_scene_plans(
                e._h, self.B, self.k, self.T, self._p(self.oa), self._p(self.od), self._p(self.warm), self._p(self.done),
                self._p(self.params), self._p(self.scene_obs), self.n_obs, self._p(self.scene_plans), stream),
                "jmpc_scene_plans")

    def _presence(self, mask, combine: int):
        """Clears the bits of absent mates in mask (jmpc_scene_presence); combine = 0 starts from -1."""
        e = self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(e._lib.jmpc_scene_presence(e._h, self.B, self.k, int(self._leave), self._p(self.done), self._p(mask),
                                               int(combine), stream), "jmpc_scene_presence")

    def _current_obstacles(self, frame: int):
        """The obstacle rows that loop iteration `frame`'s collision check reads (evaluation `frame`)."""
        if self.scene_obs is not None:
            return self.scene_obs
        return self.obstacles if self.script is None else self.script[min(frame, self.script.shape[0] - 1)]

    def _start(self):
        """Launched once before the first iteration, after __init__ / from_plans wrote the start states and done codes:
        the waiting codes, the scene's first exchange, then evaluation 0 of the outcome record."""
        if self._started:
            return
        if self._trips is not None:
            self._trips_pass(initial=1)
        if self._entering:
            e = self.e
            stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
            _cabi.check(e._lib.jmpc_scene_depart_init(e._h, self.B, self._p(self.depart), self._p(self.done), stream),
                        "jmpc_scene_depart_init")
        if self.scene_obs is not None:
            self._scene_exchange()
        if self.presence is not None and self.outcomes is not None:
            self._presence(self.presence, 0)
        if self.outcomes is not None:
            self._outcome_eval(self._current_obstacles(0), initial=1)
        self._started = True

    def _p(self, ten):
        return None if ten is None else C.c_void_p(ten.data_ptr())

    def iterate(self):
        """One loop iteration for every episode that is not done.  The engine-wide skip mask (finished episodes cost
        nothing in the step / collision kernels) is installed for the duration of the launches only: the engine never
        keeps a pointer into this object's tensors between calls."""
        self._start()
        self.e.set_skip_mask(self.done)
        try:
            self._iterate()
        finally:
            self.e.set_skip_mask(None)

    def _iterate(self):
        e, lib, torch = self.e, self.e._lib, self.torch
        stream = C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)
        i = self.iteration
        cfg = e.config
        _cabi.check(lib.jmpc_episode_pre(e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(self.course_len),
                                         self._p(self.target_ind), self._p(self.steps), self._p(self.agent_idx),
                                         self._p(self.done), float(cfg.goal_dis), float(cfg.stop_speed), stream),
                    "jmpc_episode_pre")
        if self.consider is not None:          # this iteration's agent_idx and done: who yields to whom
            _cabi.check(lib.jmpc_right_of_way(
                e._h, self.B, self.k, self.row_rule, self._p(self.agent_idx), self._p(self.done), self._p(self.params),
                self._p(self.zone), self._p(self.priority), self._p(self.consider), stream), "jmpc_right_of_way")
        if self.presence is not None:          # the same done codes: who is in the scene
            self._presence(self._collision_mask, int(self.consider is not None))
        obs = self._current_obstacles(i)
        if obs is not None and obs.shape[1] > 0:
            self.v.copy_(self.state[:, 2])
            e.collision(self.agent_idx, self.v, obs, self.frame_window, self.margin, self.flag, self.course_len,
                        course_id=self.course_id, params=self.params, horizon_s=self.horizon_s, plans=self.scene_plans,
                        n_planned=self.k - 1, consider=self._collision_mask)
            has_flags = True
        else:
            has_flags = False
        if self.signals is not None:           # the red-light cut: after the collision check, before the step
            self._signal_pass(has_flags)
        e.step(self.state, self.target_ind, self.oa, self.od, self.out, course_id=self.course_id,
               course_len=self.course_len, warm=self.warm, params=self.params)
        # history row, flag copy and time stamp are indexed by the device-side iteration counter: nothing in the loop
        # body depends on a host value that changes from one iteration to the next (except a script's frame)
        _cabi.check(lib.jmpc_episode_post_dev(
            e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(self.out.record), self._p(self.params),
            self._p(self.target_ind), self._p(self.steps), self._p(self.done), self._p(self.di), self._p(self.warm),
            self._p(self.history), self.max_steps, self._p(self.flags) if has_flags else None, self._p(self.flag),
            self._p(self.iter_dev), float(e.dt), stream), "jmpc_episode_post_dev")
        if self.program is not None:
            self._scripted_step(advance=1)
        elif self.obstacles is not None and self.obstacles.shape[1] > 0:
            _cabi.check(lib.jmpc_obstacle_step(e._h, self.B, int(self.obstacles.shape[1]), self._p(self.obstacles),
                                               self._p(self.done), float(e.dt), stream), "jmpc_obstacle_step")
        if self._trips is not None:            # close finished trips, admit the trips whose first step is i + 1
            self._trips_pass(initial=0)
        if self._entering:                     # the vehicles whose first step is iteration i + 1
            _cabi.check(lib.jmpc_scene_enter(e._h, self.B, self._p(self.depart), self._p(self.iter_dev),
                                             self._p(self.done), stream), "jmpc_scene_enter")
        if self.scene_obs is not None:         # all vehicles have moved: the scene's rows of evaluation i + 1
            self._scene_exchange()
        if self.presence is not None and self.outcomes is not None:
            self._presence(self.presence, 0)
        if self.outcomes is not None:          # the obstacle poses that iteration i + 1's collision check reads
            self._outcome_eval(self._current_obstacles(i + 1), initial=0)
        _cabi.check(lib.jmpc_counter_add(e._h, self._p(self.iter_dev), 1, stream), "jmpc_counter_add")
        self.iteration += 1

    def _finished(self) -> bool:
        """No episode is running (done = 0) or waiting to enter (done = WAITING; with trips: no trip is pending)."""
        if self._trips is not None:
            return not bool(((self.done == 0).any() | (self._trips["pending"] != 0).any()).item())
        if self._entering:
            return bool(((self.done != 0) & (self.done != _cabi.WAITING)).all().item())
        return bool((self.done != 0).all().item())

    def run(self, max_steps: Optional[int] = None, check_every: int = 8, use_graph: bool = False):
        """Iterate until every episode reached its goal (or max_steps).  Returns a dict of numpy results; with
        outcomes=True also `outcomes` (dict of [B] arrays keyed by OUTCOME_NAMES, enum jmpc_outcome in include/jmpc.h)
        and with record_obstacles=True `obstacle_history` [min(iterations, max_steps) + 1, B, n_obs, 6].

        With constant-input obstacles the loop body takes no per-iteration host argument, so with `use_graph`
        `check_every` iterations are captured once as a CUDA graph and replayed (one launch per 8 iterations instead
        of ~50 driver calls).  Measured on 4096 episodes (T = 13, ~290 iterations, 0.164 s): the capture costs more
        than the replays save (0.167-0.183 s), the loop is not launch bound at this size, so it is off by default;
        it pays for long runs of small batches."""
        torch = self.torch
        max_steps = int(max_steps or self.max_steps)
        self._start()
        graph = None
        if use_graph and self.script is None and max_steps - self.iteration > 2 * check_every:
            self.iterate()                                    # eager once: scratch allocations, kernel attributes
            torch.cuda.synchronize(self.e.device)
            it0 = self.iteration
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, capture_error_mode="relaxed"):
                    for _ in range(check_every):
                        self.iterate()
                self.iteration = it0                          # capturing executed nothing
            except Exception:                                 # capture refused: plain launches
                graph = None
                self.iteration = it0
                torch.cuda.synchronize(self.e.device)
        while self.iteration < max_steps:
            if graph is not None and max_steps - self.iteration >= check_every:
                graph.replay()
                self.iteration += check_every
                if self._finished():
                    break
                continue
            self.iterate()
            if self.iteration % check_every == 0 and self._finished():
                break
        # the reference tests the goal at the top of the next iteration
        lib, e = self.e._lib, self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(lib.jmpc_episode_pre(e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(self.course_len),
                                         self._p(self.target_ind), self._p(self.steps), self._p(self.agent_idx),
                                         self._p(self.done), float(e.config.goal_dis), float(e.config.stop_speed), stream),
                    "jmpc_episode_pre")
        trips = self._trip_table() if self._trips is not None else None
        self.torch.cuda.synchronize(e.device)
        res = dict(steps=self.steps.cpu().numpy(), done=self.done.cpu().numpy(), state=self.state.cpu().numpy(),
                   iterations=self.iteration)
        if self.history is not None:
            n = min(self.iteration, self.max_steps)
            # [steps, B, 8]: x, y, yaw, v, t, delta, a, xref_dev; row i is what History.store appends after step i
            # (t = (i + 2) dt: HistorySimulation stores the initial state first, at t = dt; simulation.py:53-61)
            res["history"] = self.history[:n].cpu().numpy()
            res["flags"] = self.flags[:n].cpu().numpy()
        if self.outcomes is not None:
            res["outcomes"] = outcome_columns(self.outcomes.cpu().numpy())
            if self.obstacle_history is not None:
                res["obstacle_history"] = self.obstacle_history[:min(self.iteration, self.max_steps) + 1].cpu().numpy()
        if self.signals is not None:
            per_slot = self.signal_owner is not None
            res["signal_hold_steps"] = (self.signal_slot_hold if per_slot else self.signal_hold).cpu().numpy()
            res["signal_go"] = (self.signal_slot_go if per_slot else self.signal_go).cpu().numpy()
        if trips is not None:
            res["trips"] = trips
        if self._plans is not None:
            plans, pid = self._plans
            res.update(plan_status=plans.status[pid].cpu().numpy(), plan_cost=plans.cost[pid].cpu().numpy(),
                       expansions=plans.expansions[pid].cpu().numpy())
        return res
