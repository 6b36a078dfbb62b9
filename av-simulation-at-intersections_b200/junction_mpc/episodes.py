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
(jmpc_right_of_way, jmpc_collision_masked).
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
                   junction=None) -> "BatchedEpisodes":
        """Episodes on the planned courses of `engine` (filled by `BatchedMPC.from_plans(plans)` /
        `set_courses_from_plans(plans)`), the second half of main/scenarios/mpc_intersection.py:63-163 for a batch:
        episode b drives plan `plan_id[b]` (default: one episode per plan; zeros = one course, many controllers).
        Its start state (the course's first pose at v = 0), its params row `dl` and done = 3 for a plan without a usable
        course are written on the device (jmpc_episode_init_from_courses); such episodes are never stepped.
        `params` [B, NPARAM] (default: the engine's defaults) supplies every other parameter row.  `run()` adds
        plan_status, plan_cost and expansions per episode.  `outcomes` / `record_obstacles` / `agents_per_scene` /
        `share_plans` / `right_of_way` / `priority` / `junction` as in `__init__`; evaluation 0 of the outcome record sees
        the planned start states; the junction zones are found on the planned courses, and first_come distances use
        each course's dl.  With agents_per_scene > 1 a scene with a done = 3 vehicle is not driven: its other vehicles get
        done = 4 (jmpc_scene_init)."""
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
                 share_plans=share_plans, right_of_way=right_of_way, priority=priority, junction=junction)
        stream = C.c_void_p(torch.cuda.current_stream(engine.device).cuda_stream)
        _cabi.check(engine._lib.jmpc_episode_init_from_courses(
            engine._h, B, ep._p(ep.course_id), ep._p(engine.course_ok), ep._p(engine.course_dl), ep._p(ep.state),
            ep._p(ep.params), ep._p(ep.done), stream), "jmpc_episode_init_from_courses")
        if ep.k > 1:
            _cabi.check(engine._lib.jmpc_scene_init(engine._h, B, ep.k, ep._p(ep.done), stream), "jmpc_scene_init")
        ep._plans = (plans, ep.course_id.long())
        return ep

    def __init__(self, engine: BatchedMPC, state0, course_id=None, obstacles=None, obstacle_script=None,
                 frame_window: int = 10, margin: int = 72, params=None, max_steps: int = 256,
                 record_history: bool = True, horizon_s: float = 7.0, obstacle_program=None, outcomes: bool = False,
                 record_obstacles: bool = False, agents_per_scene: int = 1, share_plans: bool = False,
                 right_of_way=None, priority=None, junction=None):
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
          key (entry - a) dl; a course that never enters the zone class 2 (it yields to every moving mate)."""
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
        self.outcomes = self.obstacle_history = None
        if outcome_setup(outcomes, record_obstacles, n_obs):
            self.outcomes = torch.empty(B, OUTCOME_LEN, dtype=f64, device=self.dev)     # evaluation 0 fills it
            if record_obstacles:
                self.obstacle_history = torch.full((self.max_steps + 1, B, n_obs, 6), float("nan"), dtype=f64,
                                                   device=self.dev)
        self._started = False
        if self.program is not None:                                 # get() before the first iteration
            self._scripted_step(advance=0)

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

    def _current_obstacles(self, frame: int):
        """The obstacle rows that loop iteration `frame`'s collision check reads (evaluation `frame`)."""
        if self.scene_obs is not None:
            return self.scene_obs
        return self.obstacles if self.script is None else self.script[min(frame, self.script.shape[0] - 1)]

    def _start(self):
        """Launched once before the first iteration, after __init__ / from_plans wrote the start states: the scene's
        first exchange, then evaluation 0 of the outcome record."""
        if self._started:
            return
        if self.scene_obs is not None:
            self._scene_exchange()
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
        obs = self._current_obstacles(i)
        if obs is not None and obs.shape[1] > 0:
            self.v.copy_(self.state[:, 2])
            e.collision(self.agent_idx, self.v, obs, self.frame_window, self.margin, self.flag, self.course_len,
                        course_id=self.course_id, params=self.params, horizon_s=self.horizon_s, plans=self.scene_plans,
                        n_planned=self.k - 1, consider=self.consider)
            has_flags = True
        else:
            has_flags = False
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
        if self.scene_obs is not None:         # all vehicles have moved: the scene's rows of evaluation i + 1
            self._scene_exchange()
        if self.outcomes is not None:          # the obstacle poses that iteration i + 1's collision check reads
            self._outcome_eval(self._current_obstacles(i + 1), initial=0)
        _cabi.check(lib.jmpc_counter_add(e._h, self._p(self.iter_dev), 1, stream), "jmpc_counter_add")
        self.iteration += 1

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
                if bool((self.done != 0).all().item()):
                    break
                continue
            self.iterate()
            if self.iteration % check_every == 0 and bool((self.done != 0).all().item()):
                break
        # the reference tests the goal at the top of the next iteration
        lib, e = self.e._lib, self.e
        stream = C.c_void_p(self.torch.cuda.current_stream(e.device).cuda_stream)
        _cabi.check(lib.jmpc_episode_pre(e._h, self.B, self._p(self.state), self._p(self.course_id), self._p(self.course_len),
                                         self._p(self.target_ind), self._p(self.steps), self._p(self.agent_idx),
                                         self._p(self.done), float(e.config.goal_dis), float(e.config.stop_speed), stream),
                    "jmpc_episode_pre")
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
        if self._plans is not None:
            plans, pid = self._plans
            res.update(plan_status=plans.status[pid].cpu().numpy(), plan_cost=plans.cost[pid].cpu().numpy(),
                       expansions=plans.expansions[pid].cpu().numpy())
        return res
