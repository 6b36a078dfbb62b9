"""Planner -> controller on the device: planned courses feed closed-loop episodes without a host round trip
(jmpc_planner / jmpc_plan, jmpc_set_courses_device, jmpc_episode_init_from_courses).

Gates: the two recorded reference episodes are reproduced from nothing but their planner inputs and obstacle
scripts; everywhere else the device pipeline is compared bit for bit with the host pipeline it replaces
(BatchedPlanner.plan -> synth.smooth_yaw_inplace -> BatchedMPC(courses) -> BatchedEpisodes)."""
import math
import os

import numpy as np
import pytest

from helpers import load_planner_golden

pytestmark = pytest.mark.gpu

# the scripted obstacles of the two reference scenarios (mpc_intersection.py:46-49, mpc_roundabout.py:48-51)
SCENARIO_OBSTACLES = {
    "intersection": [dict(kind="t_intersection", direction=1, offset=2., turning=False, speed=25 / 3.6, dt=0.2),
                     dict(kind="t_intersection", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)],
    "roundabout": [dict(kind="roundabout", direction=1, offset=1., turning=True, speed=25 / 3.6, dt=0.2),
                   dict(kind="roundabout", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)],
}
PLAN_FIELDS = ("cost", "status", "n_path", "path", "path_mp", "n_traj", "traj", "expansions")


@pytest.fixture(scope="module")
def fx(golden_dir):
    import __graft_entry__ as g
    g.build()
    from junction_mpc import planner as P
    z = load_planner_golden(golden_dir)
    return z, P


def _planner(z, P, max_batch=64):
    return P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"],
                            max_batch=max_batch)


def _inputs(z, names):
    g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
    scenes = [[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in names]
    return dict(start=np.stack([g(n, "start") for n in names]), goal_point=np.stack([g(n, "goal_point") for n in names]),
                goal_area=np.stack([g(n, "goal_area") for n in names]),
                allowed_dtheta=np.array([float(g(n, "allowed_dtheta")) for n in names]), scenes=scenes,
                scene_id=np.arange(len(names)), weights=np.stack([g(n, "weights") for n in names]))


def _assert_plans_equal(a, b, log=False):
    for f in PLAN_FIELDS + (("log",) if log else ()):
        assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), f


def _fake_plans(trajs):
    """A DevicePlanBatch holding hand-made trajectories (all 'found')."""
    import torch
    from junction_mpc.planner import DevicePlanBatch
    n, stride = len(trajs), max(len(t) for t in trajs)
    traj = np.zeros((n, stride, 3))
    for k, t in enumerate(trajs):
        traj[k, :len(t)] = t
    d = lambda a, dt: torch.as_tensor(a, dtype=dt, device="cuda")      # noqa: E731
    i = lambda: d(np.zeros(n), torch.int32)                             # noqa: E731
    return DevicePlanBatch(cost=d(np.zeros(n), torch.float64), status=i(), n_path=i(), path=d(np.zeros((n, 2, 3)), torch.float64),
                           path_mp=d(np.zeros((n, 2)), torch.int32), n_traj=d([len(t) for t in trajs], torch.int32),
                           traj=d(traj, torch.float64), expansions=i())


@pytest.mark.parametrize("name,variant", [("intersection", "intersection_1_1"), ("roundabout", "roundabout_1_4_big")])
def test_reference_scenario_from_scene_to_goal(fx, golden_dir, name, variant):
    """Only the planner inputs of the recorded search and the reference's obstacle scripts go in; planning, course
    ingestion and the closed loop run on the device.  Gates of test_replay_of_reference_episode."""
    z, P = fx
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes, scripted_obstacles
    e = np.load(os.path.join(golden_dir, f"episode_{name}.npz"))
    n = len(e["state"])
    plans = _planner(z, P, 4).plan_device(**_inputs(z, [variant]), max_expansions=8192)
    engine = BatchedMPC.from_plans(plans, T=13, max_batch=8)
    course = engine.get_courses(0, 1)[0]
    assert course.shape == e["course_smoothed"].shape
    np.testing.assert_allclose(course, e["course_smoothed"], rtol=0, atol=1e-9)
    ep = BatchedEpisodes.from_plans(engine, plans, obstacle_program=scripted_obstacles([SCENARIO_OBSTACLES[name]]),
                                    frame_window=int(e["frame_window"]), max_steps=160)
    assert ep.margin == int(e["margin"])
    res = ep.run(check_every=4)
    assert res["plan_status"][0] == P.STATUS_FOUND and res["expansions"][0] == len(z[f"{variant}/expanded"])
    assert res["done"][0] == 1
    assert res["steps"][0] == n                                        # 91 / 116 iterations, as the reference
    h = res["history"][:n, 0]
    states_after = np.vstack([e["state"][1:], e["final_state"][None]])
    np.testing.assert_allclose(h[:, [0, 1, 3, 2]], states_after, rtol=0, atol=1e-5)
    np.testing.assert_allclose(h[:, 5], e["di"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(h[:, 6], e["ai"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(h[:, 7], e["dev"], rtol=0, atol=1e-5)
    assert np.array_equal(res["flags"][:n, 0], e["flag"])
    np.testing.assert_allclose(res["state"][0], e["final_state"], rtol=0, atol=1e-5)
    engine.close()


def test_run_planned_scenarios(fx, golden_dir):
    """The scenario-level function: both reference scenarios in one call (one frame window for the batch, so only the
    intersection, whose FRAME_WINDOW is 10, is held to its recorded step count), plus a search that finds nothing."""
    z, P = fx
    from junction_mpc.scenarios import run_planned_scenarios
    names = ["intersection_1_1", "roundabout_1_4_big", "roundabout_2_3_big"]
    obs = [SCENARIO_OBSTACLES["intersection"], SCENARIO_OBSTACLES["roundabout"], SCENARIO_OBSTACLES["roundabout"]]
    res = run_planned_scenarios(**_inputs(z, names), obstacles=obs, frame_window=10, T=13, max_steps=160,
                                max_expansions=8192, planner=_planner(z, P, 4))
    e = np.load(os.path.join(golden_dir, "episode_intersection.npz"))
    assert res["margin"] == 72 and res["done"].tolist()[::2] == [1, 3] and res["steps"][0] == len(e["state"])
    assert res["plan_status"].tolist() == [P.STATUS_FOUND, P.STATUS_FOUND, P.STATUS_NO_SOLUTION]
    np.testing.assert_allclose(res["state"][0], e["final_state"], rtol=0, atol=1e-5)


def _constant_obstacles(courses, seed):
    rng = np.random.default_rng(seed)
    obst = np.zeros((len(courses), 2, 6))
    for b, c in enumerate(courses):
        if c is None:
            continue
        k = rng.integers(len(c) // 4, 3 * len(c) // 4, 2)
        ang = rng.uniform(-np.pi, np.pi, 2)
        obst[b, :, 0] = c[k, 0] - 25 * np.cos(ang)
        obst[b, :, 1] = c[k, 1] - 25 * np.sin(ang)
        obst[b, :, 2] = rng.uniform(3, 8, 2)
        obst[b, :, 3] = ang
        obst[b, :, 5] = rng.uniform(-.05, .05, 2)
    return obst


def test_device_pipeline_equals_host_pipeline(fx):
    """All recorded searches (the failed ones included) in one batch: the ingested courses equal the host-smoothed
    trajectories, and ~60 closed-loop steps against constant-input obstacles equal the host pipeline's, bit for bit."""
    z, P = fx
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    from junction_mpc.episodes import BatchedEpisodes
    names = [str(n) for n in z["variants"]]
    inp = _inputs(z, names)
    planner = _planner(z, P)
    plans = planner.plan_device(**inp, max_expansions=8192, max_path=32)
    hp = planner.plan(**inp, max_expansions=8192, max_path=32)
    _assert_plans_equal(plans.to_host(), hp)
    engine = BatchedMPC.from_plans(plans, T=13, max_batch=len(names))
    ok = engine.course_ok.cpu().numpy().astype(bool)
    dl = engine.course_dl.cpu().numpy()
    assert np.array_equal(ok, hp.status == P.STATUS_FOUND) and (~ok).sum() >= 2
    host_courses = [None] * len(names)
    for b in np.flatnonzero(ok):
        c = hp.trajectory(b)
        synth.smooth_yaw_inplace(c[:, 2])
        host_courses[b] = c
        assert dl[b] == math.sqrt((c[0, 0] - c[1, 0]) ** 2 + (c[0, 1] - c[1, 1]) ** 2)
    assert np.isnan(dl[~ok]).all()
    got = engine.get_courses()
    for b in np.flatnonzero(ok):
        assert np.array_equal(got[b], host_courses[b]), names[b]
    assert all(len(got[b]) == 1 for b in np.flatnonzero(~ok))

    obst = _constant_obstacles(host_courses, 11)
    steps = 60
    ep = BatchedEpisodes.from_plans(engine, plans, obstacles=obst.copy(), frame_window=10, max_steps=steps)
    dev = ep.run(max_steps=steps)
    idx = np.flatnonzero(ok)
    courses = [host_courses[b] for b in idx]
    host = BatchedMPC(courses, dl=float(dl[idx[0]]), T=13, max_batch=len(idx))
    params = np.repeat(host.default_params[None, :], len(idx), axis=0)
    params[:, PARAM_INDEX["dl"]] = dl[idx]
    state0 = np.array([[c[0, 0], c[0, 1], 0.0, c[0, 2]] for c in courses])
    hep = BatchedEpisodes(host, state0, course_id=np.arange(len(idx)), obstacles=obst[idx].copy(), frame_window=10,
                          margin=ep.margin, params=params, max_steps=steps)
    ref = hep.run(max_steps=steps)
    assert np.array_equal(dev["done"][idx], ref["done"]) and np.array_equal(dev["steps"][idx], ref["steps"])
    assert np.array_equal(dev["state"][idx], ref["state"])
    n = min(len(dev["history"]), len(ref["history"]))
    assert n >= 50
    assert np.array_equal(dev["history"][:n][:, idx], ref["history"][:n], equal_nan=True)
    assert np.array_equal(dev["flags"][:n][:, idx], ref["flags"][:n])
    assert dev["flags"][:n][:, idx].any()                              # the obstacles do interfere
    bad = np.flatnonzero(~ok)
    assert (dev["done"][bad] == 3).all() and (dev["steps"][bad] == 0).all()
    assert np.isnan(dev["history"][:, bad]).all()
    assert np.array_equal(dev["plan_status"], hp.status)
    host.close()
    engine.close()


def test_yaw_smoothing_kernel_edge_cases(fx):
    """Hand-made yaw sequences through the ingestion kernel give exactly what smooth_yaw_inplace gives."""
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    h = math.pi / 2
    yaws = [
        [0.0, 4 * math.pi + 0.1, -6 * math.pi + 0.2, 0.3, 10 * math.pi, -10 * math.pi - 0.4, 2.0, 2.0 + 14 * math.pi],
        [0.0, h, 0.0, -h, -h - h, 1.0, 1.0 + h, 1.0 + h - h, 3 * h, -3 * h, 5 * h, h, -h, 0.0],
        [0.25, 0.25 - h],
        list(np.random.default_rng(5).uniform(-40, 40, 200)),
    ]
    trajs = [np.stack([np.arange(len(y)) * 0.3, np.arange(len(y)) * -0.1, np.asarray(y, float)], axis=1) for y in yaws]
    engine = BatchedMPC.from_plans(_fake_plans(trajs), T=13, max_batch=4)
    assert engine.course_ok.cpu().numpy().tolist() == [1, 1, 1, 1]
    dl = engine.course_dl.cpu().numpy()
    for k, (t, c) in enumerate(zip(trajs, engine.get_courses())):
        want = t.copy()
        synth.smooth_yaw_inplace(want[:, 2])
        assert np.array_equal(c, want), k
        assert dl[k] == math.sqrt((t[0, 0] - t[1, 0]) ** 2 + (t[0, 1] - t[1, 1]) ** 2)
    engine.close()


def test_failed_plans_do_not_drive(fx):
    """A NO_SOLUTION search, a LIMIT search and a course longer than max_N get done = 3, no steps and NaN history;
    the usable episodes are bit-identical to a batch that holds only them."""
    import torch
    z, P = fx
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes, scripted_obstacles
    from junction_mpc.planner import DevicePlanBatch
    planner = _planner(z, P, 8)
    names = ["intersection_1_3", "intersection_1_1", "roundabout_2_3_big", "multilane_2_3_2_1"]   # 600, 720, -, 480 points
    a = planner.plan_device(**_inputs(z, names), max_expansions=8192, max_path=32)
    lim = planner.plan_device(**_inputs(z, ["multilane_1_1_2_2"]), max_expansions=50, max_path=32)
    plans = DevicePlanBatch(**{f: torch.cat([getattr(a, f), getattr(lim, f)]) for f in PLAN_FIELDS})
    status = plans.status.cpu().numpy()
    assert status.tolist() == [P.STATUS_FOUND, P.STATUS_FOUND, P.STATUS_NO_SOLUTION, P.STATUS_FOUND, P.STATUS_LIMIT]
    max_N, steps = 700, 120
    engine = BatchedMPC.from_plans(plans, T=13, max_N=max_N, max_batch=8)
    assert engine.course_ok.cpu().numpy().tolist() == [1, 0, 0, 1, 0]
    start = plans.traj[1, 0].cpu().numpy()
    assert np.array_equal(engine.get_courses(1, 1)[0], start[None])          # placeholder: the start pose
    obs = [SCENARIO_OBSTACLES["intersection"]]
    ep = BatchedEpisodes.from_plans(engine, plans, obstacle_program=scripted_obstacles(obs * 5), max_steps=steps)
    res = ep.run(max_steps=steps)
    bad, good = [1, 2, 4], [0, 3]
    assert (res["done"][bad] == 3).all() and (res["steps"][bad] == 0).all()
    assert np.isnan(res["history"][:, bad]).all()
    assert res["plan_status"].tolist() == status.tolist() and np.isnan(res["plan_cost"][[2, 4]]).all()
    only = planner.plan_device(**_inputs(z, [names[0], names[3]]), max_expansions=8192, max_path=32)
    engine2 = BatchedMPC.from_plans(only, T=13, max_N=max_N, max_batch=8)
    ref = BatchedEpisodes.from_plans(engine2, only, obstacle_program=scripted_obstacles(obs * 2), max_steps=steps).run(max_steps=steps)
    assert (res["steps"][good] > 0).all()
    assert np.array_equal(res["steps"][good], ref["steps"]) and np.array_equal(res["done"][good], ref["done"])
    assert np.array_equal(res["state"][good], ref["state"])
    n = min(len(res["history"]), len(ref["history"]))
    assert np.array_equal(res["history"][:n][:, good], ref["history"][:n], equal_nan=True)
    assert np.array_equal(res["flags"][:n][:, good], ref["flags"][:n])
    engine.close()
    engine2.close()


def test_planner_handle(fx):
    """jmpc_plan on the persistent handle equals jmpc_plan_host bit for bit, whatever the handle ran before, and a
    batch larger than max_batch is chunked with the same results."""
    z, P = fx
    names = [str(n) for n in z["variants"]]
    planner = _planner(z, P)
    kw = dict(max_expansions=8192, max_path=32, log=True)
    ref = planner.plan(**_inputs(z, names), **kw)
    _assert_plans_equal(planner.plan_device(**_inputs(z, names), **kw).to_host(), ref, log=True)
    other = names[::-1][:20] + names[:7]                              # a different, reordered batch on the same handle
    _assert_plans_equal(planner.plan_device(**_inputs(z, other), **kw).to_host(), planner.plan(**_inputs(z, other), **kw),
                        log=True)
    small = _planner(z, P, max_batch=7)
    _assert_plans_equal(small.plan_device(**_inputs(z, names), **kw).to_host(), ref, log=True)
    planner.close()
    small.close()


def test_plan_once_sweep_the_controller(fx):
    """One planned course, the 30 runs of the reference's sensitivity studies driving it (plan_id = 0 for all), with
    the params rows sweep.run_sensitivity_studies builds: histories equal BatchedEpisodes on the host-smoothed course."""
    z, P = fx
    from junction_mpc import sweep, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import MPCConfig, PARAM_INDEX, SIM_MAX_SPEED
    from junction_mpc.episodes import BatchedEpisodes
    planner = _planner(z, P, 4)
    plans = planner.plan_device(**_inputs(z, ["intersection_1_1"]), max_expansions=8192)
    cfg = MPCConfig.from_dict(sweep.SENSITIVITY_DEFAULTS)
    kw = dict(T=cfg.T, config=cfg, dt=0.2, L=2.86, speed=SIM_MAX_SPEED, max_batch=32)
    engine = BatchedMPC.from_plans(plans, **kw)
    dl = float(engine.course_dl.cpu().numpy()[0])
    base = cfg.param_vector(dl=dl, dt=0.2, L=2.86, speed=SIM_MAX_SPEED)
    rows = []
    for key, values in sweep.REFERENCE_STUDIES.values():
        for val in values:
            p = base.copy()
            p[PARAM_INDEX[key]] = float(val)
            rows.append(p)
    params = np.array(rows)
    assert len(params) == 30
    steps = 400
    dev = BatchedEpisodes.from_plans(engine, plans, plan_id=np.zeros(30, np.int64), params=params,
                                     max_steps=steps).run(max_steps=steps)
    course = plans.to_host().trajectory(0)
    synth.smooth_yaw_inplace(course[:, 2])
    host = BatchedMPC([course], dl=dl, **kw)
    state0 = np.repeat(np.array([[course[0, 0], course[0, 1], 0.0, course[0, 2]]]), 30, axis=0)
    ref = BatchedEpisodes(host, state0, params=params, max_steps=steps).run(max_steps=steps)
    assert np.array_equal(dev["steps"], ref["steps"]) and np.array_equal(dev["done"], ref["done"])
    assert (dev["done"] == 1).any()
    assert np.array_equal(dev["state"], ref["state"])
    assert np.array_equal(dev["history"], ref["history"], equal_nan=True)
    engine.close()
    host.close()
