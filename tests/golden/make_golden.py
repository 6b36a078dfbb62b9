#!/usr/bin/env python
"""Generate the committed golden fixtures by running the UNMODIFIED reference in this container.

Run from the repo root (only in the build container, where /root/reference exists):

    python tests/golden/make_golden.py

What it does (recipe of SURVEY.md Appendix B):
  * stubs `matplotlib*` and `cvxpy` in sys.modules and registers a `lib.motion_primitive` stand-in
    (the reference's dataclass default breaks on Python >= 3.11), then imports the reference's own
    modules from /root/reference/main without touching them;
  * runs the reference planner for the three scenario families -> `courses.npz`;
  * calls the reference's numpy functions on seeded random inputs -> `functions.npz`
    (nearest index, reference sampling, rollout, Jacobians, projector, smooth_yaw, resample_curve,
    obstacle prediction, collision check, cut lookup);
  * runs four runs of the sensitivity sweep (`mpc_sensitivity_analysis_comulative.py`, `lib.mpc_sensitivity.MPC`)
    -> `sensitivity_runs.npz` (full History tables);
  * runs the `mpc_intersection_new_ref.py` loop with `lib.mpc_with_speed.MPC` -> `episode_new_ref.npz`;
  * runs the literal `mpc_intersection.py` / `mpc_roundabout.py` loops with
    `lib.mpc._linear_mpc_control` monkey-patched to the oracle QP solve (cvxpy+ECOS cannot be installed
    here; that one function is the only non-reference arithmetic in the loop) and records every step
    -> `episode_intersection.npz`, `episode_roundabout.npz`.

The fixtures pin the oracle (tests/test_oracle_golden.py) and, through it, the CUDA path.
"""
import glob
import math
import os
import pickle
import sys
import types
from dataclasses import dataclass, field

import numpy as np

REF = "/root/reference/main"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)


class _Swallow(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Swallow(self.__name__ + "." + name)

    def __call__(self, *a, **k):
        return _Swallow(self.__name__ + "()")


def install_shims():
    for name in ["matplotlib", "matplotlib.pyplot", "matplotlib.colors", "matplotlib.lines",
                 "matplotlib.animation", "matplotlib.patches", "matplotlib.ticker", "matplotlib.collections",
                 "matplotlib.transforms", "cvxpy", "tqdm"]:
        sys.modules.setdefault(name, _Swallow(name))
    sys.path.insert(0, REF)
    mp_mod = types.ModuleType("lib.motion_primitive")

    @dataclass
    class MotionPrimitive:
        name: str
        forward_speed: float
        steering_angle: float
        n_seconds: float
        total_length: float = 0.
        points: np.ndarray = field(default_factory=lambda: np.array([]))

    MotionPrimitive.__module__ = "lib.motion_primitive"

    def load_motion_primitives(version="prius"):
        d = os.path.join(REF, "data", "motion_primitives_" + version)
        out = {}
        for fn in sorted(glob.glob(os.path.join(d, "*.pkl"))):
            with open(fn, "rb") as f:
                m = pickle.load(f)
            out[m.name] = m
        return out

    mp_mod.MotionPrimitive = MotionPrimitive
    mp_mod.load_motion_primitives = load_motion_primitives
    import lib  # noqa: F401  (reference package)
    sys.modules["lib.motion_primitive"] = mp_mod


def plan_courses():
    from lib.car_dimensions import BicycleModelDimensions
    from lib.motion_primitive import load_motion_primitives
    from lib.mp_search_ww_generic import MotionPrimitiveSearch
    from envs.intersection import intersection
    from envs.roundabout import roundabout
    from envs.intersection_multi_lanes import intersection as intersection_ml

    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    mps = load_motion_primitives(version="bicycle_model")
    out = {}
    for name, scen in [
        ("intersection", intersection(start_pos=1, turn_indicator=1)),
        ("roundabout", roundabout(start_pos=1, turn_indicator=4, size="big")),
        ("multilane", intersection_ml(start_pos=1, turn_indicator=1, start_lane=1, goal_lane=1, number_of_lanes=2)),
    ]:
        search = MotionPrimitiveSearch(scen, cd, mps, margin=cd.radius)
        _, _, traj = search.run(debug=False)
        out[name] = np.ascontiguousarray(traj[:, :3], dtype=np.float64)
        print(f"course {name}: {out[name].shape}")
    return out


def function_vectors(courses, rng):
    """Reference functions evaluated on seeded random inputs."""
    import lib.mpc as M
    from lib.car_dimensions import BicycleModelDimensions
    from lib.simulation import State, Simulation
    from lib.trajectories import calc_nearest_index_in_direction, resample_curve
    from lib.collision_avoidance import check_collision_moving_cars, get_cutoff_curve_by_position_idx
    from lib.moving_obstacles_prediction import MovingObstaclesPrediction

    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    out = {}
    T = M.T
    # --- smooth_yaw on raw planner yaw
    for name, c in courses.items():
        raw = c[:, 2].copy()
        out[f"smooth_{name}_in"] = raw.copy()
        out[f"smooth_{name}_out"] = M.smooth_yaw(raw.copy())
    wrapped = rng.uniform(-math.pi, math.pi, 64).cumsum() % (2 * math.pi) - math.pi
    out["smooth_rand_in"] = wrapped.copy()
    out["smooth_rand_out"] = M.smooth_yaw(wrapped.copy())

    course = courses["intersection"].copy()
    M.smooth_yaw(course[:, 2])
    cx, cy, cyaw = course[:, 0], course[:, 1], course[:, 2]
    N = len(cx)
    dl = float(np.linalg.norm(course[0, :2] - course[1, :2]))
    n = 200
    rec = {k: [] for k in ["state", "start", "ncourse", "oa", "od", "near", "target", "xref", "reach", "xbar",
                           "A", "B", "C", "ok"]}
    for k in range(n):
        s = int(rng.integers(0, N - 60))
        ncourse = N if rng.random() < 0.6 else int(rng.integers(s + 2, min(N, s + 300)))
        if k % 25 == 0:
            ncourse = min(N, s + int(rng.integers(1, 4)))     # exercises the len<=3 branches
        st = State(x=cx[s] + rng.uniform(-.5, .5), y=cy[s] + rng.uniform(-.5, .5),
                   yaw=cyaw[s] + rng.uniform(-.1, .1), v=rng.uniform(0, 30 / 3.6))
        start = max(s - 3, 0)
        oa = rng.uniform(-1, 2, T)
        od = np.clip(np.cumsum(rng.uniform(-.05, .05, T)), -.7, .7)
        ok = 1
        try:
            near = calc_nearest_index_in_direction(st, cx[:ncourse], cy[:ncourse], start_index=start, forward=True)
            xref, target, dref, reach = M._calc_ref_trajectory(st, cx[:ncourse], cy[:ncourse], cyaw[:ncourse], dl, 0.2,
                                                               start, None)
        except Exception:
            ok, near, target = 0, -1, -1
            xref, reach = np.zeros((4, T + 1)), np.zeros(T + 1, bool)
        x0 = [st.x, st.y, st.v, st.yaw]
        xbar = M._predict_motion(x0, oa, od, xref, cd, 0.2)
        Ab, Bb, Cb = zip(*[M._get_linear_model_matrix(xbar[2, t], xbar[3, t], 0.0, 0.2, cd.distance_back_to_front_wheel)
                           for t in range(T)])
        for key, val in [("state", x0), ("start", start), ("ncourse", ncourse), ("oa", oa), ("od", od), ("near", near),
                         ("target", target), ("xref", xref), ("reach", reach), ("xbar", xbar), ("A", np.array(Ab)),
                         ("B", np.array(Bb)), ("C", np.array(Cb)), ("ok", ok)]:
            rec[key].append(val)
    for k, v in rec.items():
        out["step_" + k] = np.array(v)
    out["step_dl"] = np.array(dl)
    ang = rng.uniform(-4, 4, 32)
    out["proj_angle"] = ang
    out["proj_out"] = np.array([M._get_xy_cost_mtx_for_orientation(a) for a in ang])

    # --- collision flag producer on random obstacles (roundabout course, both frame windows)
    for cname, fw in [("intersection", 10), ("roundabout", 20)]:
        path = courses[cname].copy()
        M.smooth_yaw(path[:, 2])
        dlc = float(np.linalg.norm(path[0, :2] - path[1, :2]))
        margin = 4 * int(math.ceil(cd.radius / dlc))
        R = {k: [] for k in ["idx", "v", "obs", "flag", "cut", "k", "nres", "pred0"]}
        for _ in range(60):
            idx = int(rng.integers(0, len(path) - 80))
            v = float(rng.uniform(0, 30 / 3.6)) if rng.random() < 0.9 else 30 / 3.6
            centre = path[min(idx + int(rng.integers(0, 250)), len(path) - 1), :2]
            obs = []
            for _o in range(2):
                far = rng.random() < 0.4
                pos = rng.uniform(-35, 35, 2) if far else centre + rng.uniform(-12, 12, 2)
                obs.append([pos[0], pos[1], rng.uniform(0, 30 / 3.6), rng.uniform(-math.pi, math.pi), 0.0,
                            rng.uniform(-.4, .4)])
            trajectory = path[idx:]
            if v < Simulation.MAX_SPEED:
                rdl = np.zeros((trajectory.shape[0],)) + M.MAX_ACCEL
                rdl = np.cumsum(rdl) + v
                rdl = 0.2 * np.minimum(rdl, Simulation.MAX_SPEED)
                tres = resample_curve(trajectory, dl=rdl)
            else:
                tres = resample_curve(trajectory, dl=0.2 * Simulation.MAX_SPEED)
            preds = [np.vstack(MovingObstaclesPrediction(*o, sample_time=0.2, car_dimensions=cd).state_prediction(7.)).T
                     for o in obs]
            hit = check_collision_moving_cars(cd, tres, trajectory, preds, frame_window=fw)
            if hit is None:
                flag, cut, k = 0, len(path), -1
            else:
                k = int(hit[2])
                cut = max(idx + 1, int(get_cutoff_curve_by_position_idx(path, hit[0], hit[1])) - margin)
                flag = 1
            for key, val in [("idx", idx), ("v", v), ("obs", obs), ("flag", flag), ("cut", cut), ("k", k),
                             ("nres", len(tres)), ("pred0", preds[0])]:
                R[key].append(val)
        for k, v in R.items():
            out[f"coll_{cname}_{k}"] = np.array(v)
        out[f"coll_{cname}_fw"] = np.array(fw)
        out[f"coll_{cname}_margin"] = np.array(margin)
    return out


def run_episode(kind, courses, max_steps=400):
    """The literal scenario loop (mpc_intersection.py:75-163 / mpc_roundabout.py) with recording."""
    import lib.mpc as M
    from lib.car_dimensions import BicycleModelDimensions
    from lib.simulation import State, Simulation, HistorySimulation
    from lib.trajectories import calc_nearest_index_in_direction, resample_curve
    from lib.collision_avoidance import check_collision_moving_cars, get_cutoff_curve_by_position_idx
    from lib.moving_obstacles import MovingObstacleTIntersection, MovingObstacleRoundabout
    from lib.moving_obstacles_prediction import MovingObstaclesPrediction
    from oracle import mpc_oracle as O

    DT = 0.2
    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    trajectory_full = courses[kind].copy()
    if kind == "intersection":
        obstacles = [MovingObstacleTIntersection(cd, direction=1, offset=2., turning=False, speed=25 / 3.6, dt=DT),
                     MovingObstacleTIntersection(cd, direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=DT)]
        FRAME_WINDOW = 10
    else:
        obstacles = [MovingObstacleRoundabout(cd, direction=1, offset=1., turning=True, speed=25 / 3.6, dt=DT),
                     MovingObstacleRoundabout(cd, direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=DT)]
        FRAME_WINDOW = 20
    dl = np.linalg.norm(trajectory_full[0, :2] - trajectory_full[1, :2])
    params = O.Params.from_json(os.path.join(REF, "config", "mpc_config.json"), dl=float(dl), dt=DT,
                                L=cd.distance_back_to_front_wheel, speed=30 / 3.6)

    log = {k: [] for k in ["state", "target_in", "warm", "oa_in", "od_in", "agent_idx", "obs", "flag", "ncourse",
                           "target_out", "xref", "reach", "xbar", "oa", "od", "ox", "oy", "ov", "oyaw", "cost",
                           "dev", "kkt", "di", "ai"]}
    cur = {}

    def qp_patch(xref, xbar, x0, dref, reaches_end, dt, car_dimensions, speed):
        assert speed == params.speed and dt == params.dt
        status, oa, od, ox, oy, oyaw, ov, cost, res = O.linear_mpc_control(params, xref, xbar, x0, reaches_end)
        assert status == O.STATUS_OPTIMAL, (status, res.kkt if res else None)
        cur.update(xref=xref.copy(), reach=np.array(reaches_end), xbar=xbar.copy(), cost=cost,
                   kkt=max(res.kkt.values()))
        return oa, od, ox, oy, oyaw, ov

    M._linear_mpc_control = qp_patch
    mpc = M.MPC(cx=trajectory_full[:, 0], cy=trajectory_full[:, 1], cyaw=trajectory_full[:, 2], dl=dl, dt=DT,
                car_dimensions=cd, speed=30 / 3.6)
    state = State(x=trajectory_full[0, 0], y=trajectory_full[0, 1], yaw=trajectory_full[0, 2], v=0.0)
    simulation = HistorySimulation(car_dimensions=cd, sample_time=DT, initial_state=state)
    EXTRA_CUTOFF_MARGIN = 4 * int(math.ceil(cd.radius / dl))
    traj_agent_idx = 0
    tmp_trajectory = None
    for i in range(max_steps):
        if mpc.is_goal(state):
            break
        if tmp_trajectory is None or np.any(tmp_trajectory[traj_agent_idx, :] != tmp_trajectory[-1, :]):
            traj_agent_idx = calc_nearest_index_in_direction(state, trajectory_full[:, 0], trajectory_full[:, 1],
                                                             start_index=traj_agent_idx, forward=True)
        trajectory_res = trajectory = trajectory_full[traj_agent_idx:]
        if state.v < Simulation.MAX_SPEED:
            resample_dl = np.zeros((trajectory_res.shape[0],)) + M.MAX_ACCEL
            resample_dl = np.cumsum(resample_dl) + state.v
            resample_dl = DT * np.minimum(resample_dl, Simulation.MAX_SPEED)
            trajectory_res = resample_curve(trajectory_res, dl=resample_dl)
        else:
            trajectory_res = resample_curve(trajectory_res, dl=DT * Simulation.MAX_SPEED)
        obs_now = [list(o.get()) for o in obstacles]
        trajs = [np.vstack(MovingObstaclesPrediction(*o, sample_time=DT, car_dimensions=cd).state_prediction(7.)).T
                 for o in obs_now]
        collision_xy = check_collision_moving_cars(cd, trajectory_res, trajectory, trajs, frame_window=FRAME_WINDOW)
        if collision_xy is not None:
            cutoff_idx = get_cutoff_curve_by_position_idx(trajectory_full, collision_xy[0],
                                                          collision_xy[1]) - EXTRA_CUTOFF_MARGIN
            cutoff_idx = max(traj_agent_idx + 1, cutoff_idx)
            tmp_trajectory = trajectory_full[:cutoff_idx]
        else:
            tmp_trajectory = trajectory_full
        mpc.set_trajectory_fromarray(tmp_trajectory)
        log["state"].append([state.x, state.y, state.v, state.yaw])
        log["target_in"].append(mpc.target_ind)
        log["warm"].append(0 if mpc.oa is None else 1)
        log["oa_in"].append(np.zeros(M.T) if mpc.oa is None else np.array(mpc.oa))
        log["od_in"].append(np.zeros(M.T) if mpc.odelta is None else np.array(mpc.odelta))
        log["agent_idx"].append(traj_agent_idx)
        log["obs"].append(obs_now)
        log["flag"].append(0 if collision_xy is None else 1)
        log["ncourse"].append(len(tmp_trajectory))
        delta, acceleration = mpc.step(state)
        for k in ["xref", "reach", "xbar", "cost", "kkt"]:
            log[k].append(cur[k])
        log["target_out"].append(mpc.target_ind)
        for k, v in [("oa", mpc.oa), ("od", mpc.odelta), ("ox", mpc.ox), ("oy", mpc.oy), ("ov", mpc.ov),
                     ("oyaw", mpc.oyaw)]:
            log[k].append(np.array(v))
        log["di"].append(delta)
        log["ai"].append(acceleration)
        dev = mpc.get_current_xref_deviation()
        log["dev"].append(dev)
        for o in obstacles:
            o.step()
        state = simulation.step(a=acceleration, delta=delta, xref_deviation=dev)
    out = {k: np.array(v) for k, v in log.items()}
    out["final_state"] = np.array([state.x, state.y, state.v, state.yaw])
    out["frame_window"] = np.array(FRAME_WINDOW)
    out["margin"] = np.array(EXTRA_CUTOFF_MARGIN)
    out["dl"] = np.array(dl)
    out["course_smoothed"] = trajectory_full          # MPC.__init__ smoothed column 2 in place
    print(f"episode {kind}: {len(out['state'])} steps, collision flag on {int(out['flag'].sum())}, "
          f"cut range {out['ncourse'][out['flag'] == 1].min() if out['flag'].any() else '-'}"
          f"..{out['ncourse'][out['flag'] == 1].max() if out['flag'].any() else '-'}, worst kkt {out['kkt'].max():.2e}")
    return out


def run_sensitivity_runs(courses):
    """mpc_sensitivity_analysis_comulative.py:178-266 for a few parameter values: `lib.mpc_sensitivity.MPC` (no
    `speed` argument), no obstacles, History recorded by HistorySimulation.  The JSON the reference re-reads in every
    solve lives in the read-only reference tree, so the values of `reset_config` (:32-51) plus the one parameter
    under study are handed to the patched QP solve directly."""
    import lib.mpc_sensitivity as MS
    from lib.car_dimensions import BicycleModelDimensions
    from lib.simulation import State, HistorySimulation
    from lib.trajectories import calc_nearest_index_in_direction
    from oracle import mpc_oracle as O

    DT = 0.2
    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    base = {"NX": 4, "NU": 2, "T": 13, "w_perp": 20.0, "w_para": 1.0, "R": [0.1, 0.01], "Rd": [10, 1.0],
            "Q_v_yaw": [0.0, 0.5], "Qf": [1.0, 1.0, 0.0, 0.5], "GOAL_DIS": 1.5, "STOP_SPEED": 0.1389, "MAX_TIME": 13.0,
            "MAX_ITER": 1, "DU_TH": 0.1, "MAX_DSTEER": 30.0, "MAX_ACCEL": 2.0, "MAX_DECEL": -10}
    out = {}
    for tag, override in [("default", {}), ("w_para_0p1", {"w_para": 0.1}), ("R_acc_10", {"R": [10, 0.01]}),
                          ("Rd_steer_0", {"Rd": [10, 0]})]:
        cfg = dict(base)
        cfg.update(override)
        trajectory_full = courses["intersection"].copy()
        dl = np.linalg.norm(trajectory_full[0, :2] - trajectory_full[1, :2])
        params = O.Params.from_config(cfg, dl=float(dl), dt=DT, L=cd.distance_back_to_front_wheel, speed=30 / 3.6)

        def qp_patch(xref, xbar, x0, dref, reaches_end, dt, car_dimensions):
            status, oa, od, ox, oy, oyaw, ov, cost, res = O.linear_mpc_control(params, xref, xbar, x0, reaches_end)
            assert status == O.STATUS_OPTIMAL
            return oa, od, ox, oy, oyaw, ov

        MS._linear_mpc_control = qp_patch
        mpc = MS.MPC(cx=trajectory_full[:, 0], cy=trajectory_full[:, 1], cyaw=trajectory_full[:, 2], dl=dl, dt=DT,
                     car_dimensions=cd)
        state = State(x=trajectory_full[0, 0], y=trajectory_full[0, 1], yaw=trajectory_full[0, 2], v=0.0)
        simulation = HistorySimulation(car_dimensions=cd, sample_time=DT, initial_state=state)
        traj_agent_idx, tmp_trajectory = 0, None
        for i in range(600):
            if mpc.is_goal(state):
                break
            if tmp_trajectory is None or np.any(tmp_trajectory[traj_agent_idx, :] != tmp_trajectory[-1, :]):
                traj_agent_idx = calc_nearest_index_in_direction(state, trajectory_full[:, 0], trajectory_full[:, 1],
                                                                 start_index=traj_agent_idx, forward=True)
            tmp_trajectory = trajectory_full            # no obstacles: check_collision_moving_cars returns None
            mpc.set_trajectory_fromarray(tmp_trajectory)
            delta, acceleration = mpc.step(state)
            state = simulation.step(a=acceleration, delta=delta, xref_deviation=mpc.get_current_xref_deviation())
        h = simulation.history
        out[tag] = np.array([h.x, h.y, h.yaw, h.v, h.t, h.delta, h.a, h.xref_deviation]).T
        print(f"sensitivity run {tag}: {len(h.x) - 1} steps, sim time {h.t[-1]:.1f} s")
    out["config_R"] = np.array(base["R"])
    out["config_Rd"] = np.array(base["Rd"])
    return out


def run_new_ref_episode(courses, max_steps=400):
    """main/scenarios/mpc_intersection_new_ref.py:62-160 with `lib.mpc_with_speed.MPC` (speed profile cv in xref[2],
    Q_v_yaw = diag(20, .5), w = 10 / 1, MAX_DECEL = -5): the course is never truncated, the cut index only zeroes
    the speed profile behind it."""
    import lib.mpc_with_speed as MW
    from lib.car_dimensions import BicycleModelDimensions
    from lib.simulation import State, Simulation, HistorySimulation
    from lib.trajectories import calc_nearest_index_in_direction, resample_curve
    from lib.collision_avoidance import check_collision_moving_cars, get_cutoff_curve_by_position_idx
    from lib.moving_obstacles import MovingObstacleTIntersection
    from lib.moving_obstacles_prediction import MovingObstaclesPrediction
    from oracle import mpc_oracle as O

    DT = 0.2
    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    trajectory_full = courses["intersection"].copy()
    obstacles = [MovingObstacleTIntersection(cd, direction=1, offset=1., turning=False, speed=25 / 3.6, dt=DT),
                 MovingObstacleTIntersection(cd, direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=DT)]
    dl = np.linalg.norm(trajectory_full[0, :2] - trajectory_full[1, :2])
    params = O.Params(T=MW.T, dt=DT, dl=float(dl), L=cd.distance_back_to_front_wheel, speed=Simulation.MAX_SPEED,
                      w_perp=10.0, w_para=1.0, R=(0.01, 0.01), Rd=(0.01, 1.0), Q_v_yaw=(20.0, 0.5),
                      Qf=(1.0 * MW.T, 1.0 * MW.T, 0.0, 0.5 * MW.T), max_decel=float(MW.MAX_DECEL),
                      max_accel=float(MW.MAX_ACCEL), max_dsteer=float(MW.MAX_DSTEER))
    log = {k: [] for k in ["state", "target_in", "warm", "oa_in", "od_in", "agent_idx", "obs", "flag", "cutoff",
                           "target_out", "xref", "oa", "od", "ox", "oy", "ov", "oyaw", "cost", "di", "ai", "dev"]}
    cur = {}

    def qp_patch(xref, xbar, x0, dref, reaches_end, dt, car_dimensions):
        status, oa, od, ox, oy, oyaw, ov, cost, res = O.linear_mpc_control(params, xref, xbar, x0, reaches_end)
        assert status == O.STATUS_OPTIMAL
        cur.update(xref=xref.copy(), cost=cost)
        return oa, od, ox, oy, oyaw, ov

    MW._linear_mpc_control = qp_patch
    cv = np.full(trajectory_full[:, 1].shape, 30 / 3.6)
    mpc = MW.MPC(cx=trajectory_full[:, 0], cy=trajectory_full[:, 1], cv=cv, cyaw=trajectory_full[:, 2], dl=dl, dt=DT,
                 car_dimensions=cd)
    state = State(x=trajectory_full[0, 0], y=trajectory_full[0, 1], yaw=trajectory_full[0, 2], v=0.0)
    simulation = HistorySimulation(car_dimensions=cd, sample_time=DT, initial_state=state)
    FRAME_WINDOW = 20
    EXTRA_CUTOFF_MARGIN = 4 * int(math.ceil(cd.radius / dl))
    traj_agent_idx, tmp_trajectory = 0, None
    for i in range(max_steps):
        if mpc.is_goal(state):
            break
        if tmp_trajectory is None or np.any(tmp_trajectory[traj_agent_idx, :] != tmp_trajectory[-1, :]):
            traj_agent_idx = calc_nearest_index_in_direction(state, trajectory_full[:, 0], trajectory_full[:, 1],
                                                             start_index=traj_agent_idx, forward=True)
        trajectory_res = trajectory = trajectory_full[traj_agent_idx:]
        if state.v < Simulation.MAX_SPEED:
            resample_dl = np.zeros((trajectory_res.shape[0],)) + MW.MAX_ACCEL
            resample_dl = np.cumsum(resample_dl) + state.v
            resample_dl = DT * np.minimum(resample_dl, Simulation.MAX_SPEED)
            trajectory_res = resample_curve(trajectory_res, dl=resample_dl)
        else:
            trajectory_res = resample_curve(trajectory_res, dl=DT * Simulation.MAX_SPEED)
        obs_now = [list(o.get()) for o in obstacles]
        trajs = [np.vstack(MovingObstaclesPrediction(*o, sample_time=DT, car_dimensions=cd).state_prediction(7.)).T
                 for o in obs_now]
        collision_xy = check_collision_moving_cars(cd, trajectory_res, trajectory, trajs, frame_window=FRAME_WINDOW)
        cutoff_idx = 999
        if collision_xy is not None:
            cutoff_idx = get_cutoff_curve_by_position_idx(trajectory_full, collision_xy[0],
                                                          collision_xy[1]) - EXTRA_CUTOFF_MARGIN
            cutoff_idx = max(traj_agent_idx + 1, cutoff_idx)
        tmp_trajectory = trajectory_full
        mpc.set_trajectory_fromarray(tmp_trajectory, cutoff_idx=cutoff_idx)
        log["state"].append([state.x, state.y, state.v, state.yaw])
        log["target_in"].append(mpc.target_ind)
        log["warm"].append(0 if mpc.oa is None else 1)
        log["oa_in"].append(np.zeros(MW.T) if mpc.oa is None else np.array(mpc.oa))
        log["od_in"].append(np.zeros(MW.T) if mpc.odelta is None else np.array(mpc.odelta))
        log["agent_idx"].append(traj_agent_idx)
        log["obs"].append(obs_now)
        log["flag"].append(0 if collision_xy is None else 1)
        log["cutoff"].append(cutoff_idx)
        delta, acceleration = mpc.step(state)
        log["xref"].append(cur["xref"])
        log["cost"].append(cur["cost"])
        log["target_out"].append(mpc.target_ind)
        for k, v in [("oa", mpc.oa), ("od", mpc.odelta), ("ox", mpc.ox), ("oy", mpc.oy), ("ov", mpc.ov),
                     ("oyaw", mpc.oyaw)]:
            log[k].append(np.array(v))
        log["di"].append(delta)
        log["ai"].append(acceleration)
        dev = mpc.get_current_xref_deviation()
        log["dev"].append(dev)
        for o in obstacles:
            o.step()
        state = simulation.step(a=acceleration, delta=delta, xref_deviation=dev)
    out = {k: np.array(v) for k, v in log.items()}
    out["final_state"] = np.array([state.x, state.y, state.v, state.yaw])
    out["dl"] = np.array(dl)
    out["margin"] = np.array(EXTRA_CUTOFF_MARGIN)
    out["frame_window"] = np.array(FRAME_WINDOW)
    out["v_profile"] = np.array(MW.MAX_SPEED)
    out["course_smoothed"] = trajectory_full
    print(f"episode new_ref (mpc_with_speed): {len(out['state'])} steps, collision flag on {int(out['flag'].sum())}, "
          f"max speed {out['state'][:, 2].max():.3f}")
    return out


def record_scripted_obstacles(steps=160):
    """The reference's scripted obstacles (main/lib/moving_obstacles.py) stepped as the scenario loops step them:
    `get()` (whose steering property has side effects on the roundabout model) then `step()`.  One row per spec:
    [kind, direction, turning, speed, offset (-1 = None), dt, x_init, y_init, initial_speed]."""
    import contextlib
    import io
    from lib.car_dimensions import BicycleModelDimensions
    from lib.moving_obstacles import MovingObstacleArterial, MovingObstacleRoundabout, MovingObstacleTIntersection
    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    specs, tracks = [], []
    for kind, cls in [(1, MovingObstacleTIntersection), (2, MovingObstacleRoundabout)]:
        for direction in (1, -1):
            for turning in (False, True):
                for speed, offset, dt in [(25 / 3.6, 2.0, 0.2), (25 / 3.6, 4.0, 0.2), (30 / 3.6, None, 0.2),
                                          (20 / 3.6, 3.0, 0.2), (15 / 3.6, 0.0, 0.1), (25 / 3.6, 1.0, 0.2)]:
                    o = cls(cd, direction=direction, turning=turning, speed=speed, offset=offset, dt=dt)
                    rows = []
                    with contextlib.redirect_stdout(io.StringIO()):         # the roundabout property prints
                        for _ in range(steps):
                            rows.append(list(o.get()))
                            o.step()
                    specs.append([kind, direction, float(turning), speed, -1.0 if offset is None else offset, dt, 0, 0, 0])
                    tracks.append(rows)
    for x0, y0, speed, v_init, offset in [(3.0, -20.0, 25 / 3.6, 5 / 3.6, 2.0), (-3.0, -35.0, 30 / 3.6, 0.0, None),
                                          (1.5, -10.0, 20 / 3.6, 10 / 3.6, 5.0)]:
        o = MovingObstacleArterial(cd, x_init=x0, y_init=y0, speed=speed, initial_speed=v_init, offset=offset, dt=0.2)
        rows = []
        for _ in range(steps):
            rows.append(list(o.get()))
            o.step()
        specs.append([3, 1, 0.0, speed, -1.0 if offset is None else offset, 0.2, x0, y0, v_init])
        tracks.append(rows)
    print(f"scripted obstacles: {len(specs)} specs x {steps} steps")
    return dict(specs=np.array(specs, float), tracks=np.array(tracks, float))


def record_planner(max_seconds=20):
    """The reference's motion-primitive A* (main/lib/mp_search_ww_generic.py + a_star.py) on scenario / weight
    variants: inputs as plain arrays (start, goal, goal area, obstacle half-planes, weights) and what the search
    returned (cost, node path, primitive per edge, full trajectory, the order in which nodes were expanded)."""
    import signal
    from lib.car_dimensions import BicycleModelDimensions
    from lib.motion_primitive import load_motion_primitives
    from lib.mp_search_ww_generic import MotionPrimitiveSearch
    from envs.intersection import intersection
    from envs.roundabout import roundabout
    from envs.intersection_multi_lanes import intersection as intersection_ml
    from envs.t_intersection import t_intersection

    cd = BicycleModelDimensions(skip_back_circle_collision_checking=False)
    mps = load_motion_primitives(version="bicycle_model")
    names = sorted(mps)
    out = {"mp_names": np.array(names), "mp_points": np.stack([mps[n].points for n in names]),
           "mp_total_length": np.array([mps[n].total_length for n in names]),
           "car_radius": np.array(cd.radius), "car_circle_centers": np.array(cd.circle_centers)}
    variants = []
    for sp in (1, 2, 3, 4):
        for ti in (1, 2, 3):
            variants.append((f"intersection_{sp}_{ti}", lambda sp=sp, ti=ti: intersection(start_pos=sp, turn_indicator=ti), {}))
    for sp in (1, 2, 3, 4):
        for ti in (1, 2, 3, 4):
            variants.append((f"roundabout_{sp}_{ti}_big", lambda sp=sp, ti=ti: roundabout(start_pos=sp, turn_indicator=ti, size="big"), {}))
    for sp, ti in [(1, 1), (1, 2), (2, 3), (3, 1)]:
        variants.append((f"roundabout_{sp}_{ti}_normal", lambda sp=sp, ti=ti: roundabout(start_pos=sp, turn_indicator=ti), {}))
    for sp, ti, sl, gl in [(1, 1, 1, 1), (1, 1, 2, 2), (1, 2, 1, 2), (2, 3, 2, 1), (3, 1, 1, 2), (4, 2, 2, 2)]:
        variants.append((f"multilane_{sp}_{ti}_{sl}_{gl}",
                         lambda sp=sp, ti=ti, sl=sl, gl=gl: intersection_ml(start_pos=sp, turn_indicator=ti, start_lane=sl,
                                                                          goal_lane=gl, number_of_lanes=2), {}))
    for sp, ti in [(1, 1), (1, 3), (2, 2), (2, 3)]:
        variants.append((f"t_intersection_{sp}_{ti}", lambda sp=sp, ti=ti: t_intersection(start_pos=sp, turn_indicator=ti), {}))
    # weight variants of the reference's default scene (the knobs of mp_search_ww_generic.py:27-31)
    for k, w in enumerate([dict(wh_theta=1.0), dict(wh_steering=5.0), dict(wc_steering=1.0), dict(wh_dist=1.5, wc_dist=0.8),
                           dict(wh_obstacle=0.2, wc_obstacle=0.5), dict(wh_center=0.1, wc_center=0.1),
                           dict(wh_theta=4.0, wh_steering=25.0), dict(wc_obstacle=1.0, wh_obstacle=0.05)]):
        variants.append((f"intersection_1_1_w{k}", lambda: intersection(start_pos=1, turn_indicator=1), w))
        variants.append((f"roundabout_1_4_big_w{k}", lambda: roundabout(start_pos=1, turn_indicator=4, size="big"), w))

    class _Timeout(Exception):
        pass

    def _alarm(*_):
        raise _Timeout()
    signal.signal(signal.SIGALRM, _alarm)
    wkeys = ["wh_dist", "wh_theta", "wh_steering", "wh_obstacle", "wh_center", "wc_dist", "wc_steering", "wc_obstacle", "wc_center"]
    defaults = dict(wh_dist=1.0, wh_theta=2.7, wh_steering=15.0, wh_obstacle=0.0, wh_center=0.0, wc_dist=1.0, wc_steering=5.0,
                    wc_obstacle=0.1, wc_center=0.0)
    kept = []
    for name, make, w in variants:
        try:
            scen = make()
        except Exception as exc:          # noqa: BLE001  (some start / turn combinations do not exist in an env)
            print(f"planner variant {name}: scenario not available ({type(exc).__name__})")
            continue
        search = MotionPrimitiveSearch(scen, cd, mps, margin=cd.radius, **w)
        signal.alarm(max_seconds)
        try:
            cost, path, traj = search.run(debug=True)
        except _Timeout:
            print(f"planner variant {name}: more than {max_seconds} s, skipped")
            continue
        except Exception as exc:          # noqa: BLE001
            if "No solution" not in str(exc) or name not in ("roundabout_2_3_big", "roundabout_4_4_big"):
                print(f"planner variant {name}: {exc}")
                continue
            cost, path, traj = float("nan"), [], np.zeros((0, 3))      # the open list ran empty (a_star.py:78)
        finally:
            signal.alarm(0)
        hp = search._obstacles_hp
        hp_tab = np.zeros((len(hp), 8, 3))
        hp_n = np.array([len(h) for h in hp])
        for k, h in enumerate(hp):
            hp_tab[k, :len(h)] = h
        ww = dict(defaults, **w)
        mp_idx = [names.index(search._points_to_mp_names[a, b]) for a, b in zip(path[:-1], path[1:])]
        pre = f"{name}/"
        out.update({pre + "start": np.array(scen.start, float), pre + "goal_point": np.array(scen.goal_point, float),
                    pre + "goal_area": np.array([*scen.goal_area.xy1, *scen.goal_area.xy2], float),
                    pre + "allowed_dtheta": np.array(scen.allowed_goal_theta_difference), pre + "hp": hp_tab, pre + "hp_n": hp_n,
                    pre + "weights": np.array([ww[k] for k in wkeys]), pre + "cost": np.array(cost),
                    pre + "path": np.array(path, float).reshape(-1, 3), pre + "mp_idx": np.array(mp_idx), pre + "trajectory": traj,
                    pre + "expanded": np.array([[d.g, d.h, *d.node] for d in search.debug_data], float)})
        kept.append(name)
        print(f"planner variant {name}: cost {cost:.6f}, {len(path)} nodes, {len(search.debug_data)} expansions, traj {traj.shape}")
    out["variants"] = np.array(kept)
    # the collision-check points the reference derives per primitive (mp_search_ww_generic.py:121-138), for the
    # host-side restatement of that derivation
    out["mp_collision_points"] = np.stack([search._mp_collision_points[n] for n in names])
    return out


def savez_planner(path, arrays):
    """np.savez_compressed with every trajectory that equals an earlier variant's stored once, which keeps
    planner.npz under 1 MB: the rows (name, stored name) of `aliases` restore it (tests/helpers.py
    load_planner_golden)."""
    arrays, stored, aliases = dict(arrays), {}, []
    for name in list(arrays):
        if name.endswith("/trajectory"):
            a = np.asarray(arrays[name])
            key = (a.dtype.str, a.shape, a.tobytes())
            if key in stored:
                aliases.append((name, stored[key]))
                del arrays[name]
            else:
                stored[key] = name
    np.savez_compressed(path, aliases=np.array(aliases, dtype=str).reshape(-1, 2), **arrays)


def main():
    install_shims()
    if "--planner" in sys.argv:
        savez_planner(os.path.join(HERE, "planner.npz"), record_planner())
        return
    if "--obstacles" in sys.argv:
        np.savez_compressed(os.path.join(HERE, "scripted_obstacles.npz"), **record_scripted_obstacles())
        return
    rng = np.random.default_rng(20261018)
    courses = plan_courses()
    np.savez_compressed(os.path.join(HERE, "courses.npz"), **courses)
    np.savez_compressed(os.path.join(HERE, "functions.npz"), **function_vectors(courses, rng))
    for kind in ["intersection", "roundabout"]:
        np.savez_compressed(os.path.join(HERE, f"episode_{kind}.npz"), **run_episode(kind, courses))
    np.savez_compressed(os.path.join(HERE, "sensitivity_runs.npz"), **run_sensitivity_runs(courses))
    np.savez_compressed(os.path.join(HERE, "episode_new_ref.npz"), **run_new_ref_episode(courses))
    np.savez_compressed(os.path.join(HERE, "scripted_obstacles.npz"), **record_scripted_obstacles())


if __name__ == "__main__":
    main()
