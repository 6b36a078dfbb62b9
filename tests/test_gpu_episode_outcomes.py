"""Per-episode outcome record (jmpc_episode_outcomes, BatchedEpisodes(outcomes=True)) against the recorded reference
episodes and against the numpy oracle (oracle/episode_outcomes.py) fed by the run's History and by obstacle tracks
generated independently of the device.

Integer columns match exactly, MIN_CLEARANCE to 1e-12 m, the other float columns to 1e-12 relative (1e-12 absolute
where the value is 0).  Wherever a contact decision is compared, no (ego, obstacle) clearance of the fixture lies
within 1e-9 of 0, so that a last-ulp difference of cos / sin cannot flip it."""
import math
import os

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import episode_outcomes as EO
from oracle import obstacle_oracle as OO

pytestmark = pytest.mark.gpu

SCENARIO_OBSTACLES = {
    "intersection": [dict(kind="t_intersection", direction=1, offset=2., turning=False, speed=25 / 3.6, dt=0.2),
                     dict(kind="t_intersection", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)],
    "roundabout": [dict(kind="roundabout", direction=1, offset=1., turning=True, speed=25 / 3.6, dt=0.2),
                   dict(kind="roundabout", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)],
}
KINDS = {"t_intersection": OO.KIND_TINTERSECTION, "roundabout": OO.KIND_ROUNDABOUT}
GEO = C.CarGeometry()
FAST = slice(0, None, 256)
R2 = 2 * GEO.radius


@pytest.fixture(scope="module")
def jm():
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    from junction_mpc.episodes import OUTCOME_INT, OUTCOME_NAMES, BatchedEpisodes
    return synth, BatchedMPC, BatchedEpisodes, PARAM_INDEX, OUTCOME_NAMES, OUTCOME_INT


def _prm(engine, PI):
    p = engine.default_params
    return dict(dt=float(p[PI["dt"]]), L=float(p[PI["L"]]), max_steer=float(p[PI["max_steer"]]))


def _assert_outcome(got: dict, b: int, want: dict, names, ints, what=""):
    for n in names:
        g, w = got[n][b], want[n]
        if n in ints:
            assert int(g) == int(w), (what, b, n, g, w)
        elif n == "min_clearance":
            assert (g == w) if math.isinf(w) else abs(g - w) <= 1e-12, (what, b, n, g, w)
        elif w == 0.0:
            assert abs(g) <= 1e-12, (what, b, n, g, w)
        else:
            assert abs(g - w) <= 1e-12 * abs(w), (what, b, n, g, w)


def _assert_no_boundary(state0, history, track):
    """No (ego, obstacle) clearance within 1e-9 of 0: contact decisions cannot depend on the last ulp."""
    if track.shape[1] == 0:
        return
    poses = np.vstack([[[state0[0], state0[1], state0[3]]], history[:, :3]])
    clear, _ = EO.clearance_and_contact(poses, track, GEO)
    assert (np.abs(clear) > 1e-9).all(), np.abs(clear).min()


def _oracle(res, b, state0, track, prm):
    n = int(res["steps"][b])
    h, f = res["history"][:n, b], res["flags"][:n, b]
    _assert_no_boundary(state0, h, track[:n + 1])
    return EO.episode_outcomes(state0, h, f, track[:n + 1], **prm)


def _scripted_tracks(specs, n):
    """[n + 1, n_obs, 6]: the get() tuples of oracle/obstacle_oracle.py's obstacles before the first step and after
    each of n steps."""
    obs = [OO.ScriptedObstacle(KINDS[s["kind"]], s["direction"], s["turning"], s["speed"], s["offset"], s["dt"])
           for s in specs]
    out = []
    for e in range(n + 1):
        if e:
            for o in obs:
                o.step()
        out.append([o.get() for o in obs])
    return np.array(out, dtype=np.float64)


def _constant_tracks(obst, n, dt, L=2.86):
    """[n + 1, B, n_obs, 6]: the constant-input update of the obstacles' predictor, as _cpu_episode of
    test_gpu_episodes.py runs it, vectorised over the batch."""
    o = obst.copy()
    out = np.empty((n + 1,) + o.shape)
    out[0] = o
    for e in range(1, n + 1):
        o[..., 0] += o[..., 2] * np.cos(o[..., 3]) * dt
        o[..., 1] += o[..., 2] * np.sin(o[..., 3]) * dt
        o[..., 2] += o[..., 4] * dt
        o[..., 3] += (o[..., 2] / L) * np.tan(o[..., 5]) * dt
        out[e] = o
    return out


def _bench_workload(course, B, seed=11):
    """tests/tools/bench_episodes.py's batch: start on the course at 0-3 m/s, two constant-input obstacles crossing."""
    rng = np.random.default_rng(seed)
    state0 = np.repeat(np.array([[course[0, 0], course[0, 1], 0.0, course[0, 2]]]), B, axis=0)
    state0[:, 2] = rng.uniform(0, 3, B)
    obst = np.zeros((B, 2, 6))
    k = rng.integers(150, 400, (B, 2))
    ang = rng.uniform(-np.pi, np.pi, (B, 2))
    obst[:, :, 0] = course[k, 0] - 25 * np.cos(ang)
    obst[:, :, 1] = course[k, 1] - 25 * np.sin(ang)
    obst[:, :, 2] = rng.uniform(3, 8, (B, 2))
    obst[:, :, 3] = ang
    obst[:, :, 5] = rng.uniform(-.05, .05, (B, 2))
    return state0, obst


def _intersection(jm, B):
    synth, BatchedMPC = jm[0], jm[1]
    course = synth.load_course("intersection")
    dl = float(np.linalg.norm(course[0, :2] - course[1, :2]))
    return course, dl, BatchedMPC([course], dl=dl, T=13, max_batch=B)


@pytest.mark.parametrize("name", ["intersection", "roundabout"])
def test_reference_episodes(jm, golden_dir, name):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    from junction_mpc.episodes import scripted_obstacles
    e = np.load(os.path.join(golden_dir, f"episode_{name}.npz"))
    n = len(e["state"])
    engine = BatchedMPC([e["course_smoothed"]], dl=float(e["dl"]), T=13, max_batch=8)
    state0 = e["state"][:1]
    ep = BatchedEpisodes(engine, state0, frame_window=int(e["frame_window"]), margin=int(e["margin"]), max_steps=160,
                         obstacle_program=scripted_obstacles([SCENARIO_OBSTACLES[name]]), outcomes=True,
                         record_obstacles=True)
    res = ep.run(check_every=4)
    assert res["steps"][0] == n and res["done"][0] == 1
    out, track_dev = res["outcomes"], res["obstacle_history"]
    assert track_dev.shape == (res["iterations"] + 1, 1, 2, 6)

    # 1. clearance and contact per evaluation 0 .. n-1 from the reference's own poses, against the device's poses
    m = min(n, len(e["obs"]))
    ref_poses = e["state"][:m][:, [0, 1, 3]]
    ref_clear, ref_hit = EO.clearance_and_contact(ref_poses, e["obs"][:m], GEO)
    dev_poses = np.vstack([state0[:, [0, 1, 3]], res["history"][:m - 1, 0, :3]])
    dev_clear, dev_hit = EO.clearance_and_contact(dev_poses, track_dev[:m, 0], GEO)
    np.testing.assert_allclose(dev_clear, ref_clear, rtol=0, atol=1e-5)
    sure = np.abs(ref_clear) > 1e-5
    assert np.array_equal(dev_hit[sure], ref_hit[sure])
    if out["min_clearance_eval"][0] < m:
        assert abs(out["min_clearance"][0] - ref_clear.min()) <= 1e-5

    # 2. every column against the oracle fed by the History and by independently generated obstacle tracks
    track = _scripted_tracks(SCENARIO_OBSTACLES[name], n)
    want = _oracle(res, 0, state0[0], track, _prm(engine, PI))
    _assert_outcome(out, 0, want, names, ints, name)
    assert out["min_clearance"][0] > 0 and out["first_contact_eval"][0] == -1     # the reference drives through

    # 3. the recorded obstacle poses are those tracks (rows after the episode ended stay NaN)
    np.testing.assert_allclose(track_dev[:n + 1, 0], track, rtol=0, atol=1e-9)
    assert np.isnan(track_dev[n + 1:]).all()
    engine.close()


def test_forced_contact_at_a_known_evaluation(jm):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    course, dl, engine = _intersection(jm, 8)
    margin = C.cutoff_margin(GEO, dl)
    steps = 40
    state0 = np.array([[course[0, 0], course[0, 1], 2.0, course[0, 2]]])
    free = BatchedEpisodes(engine, state0, max_steps=steps, margin=margin).run(max_steps=steps)
    assert free["steps"][0] == steps
    hist = free["history"][:, 0]
    k, k2 = 20, 12
    far = [course[0, 0] + 1000.0, course[0, 1], 0.0, 0.0, 0.0, 0.0]

    def beside(row, d):            # same heading, displaced sideways by d: the nearest circle pairs are d apart
        x, y, yaw = row[0], row[1], row[2]
        return [x - d * math.sin(yaw), y + d * math.cos(yaw), 0.0, yaw, 0.0, 0.0]

    # episode 0: obstacle 0 on the ego's pose of row k - 1 at evaluation k; episodes 1 / 2: obstacle 1 beside the ego
    # of row k2 - 1 at 2r - 1e-6 / 2r + 1e-6 at evaluation k2; far away at every other frame
    S = steps + 1
    script = np.empty((S, 3, 2, 6))
    script[:] = far
    script[k, 0, 0] = [hist[k - 1, 0], hist[k - 1, 1], 0.0, hist[k - 1, 2], 0.0, 0.0]
    script[k2, 1, 1] = beside(hist[k2 - 1], R2 - 1e-6)
    script[k2, 2, 1] = beside(hist[k2 - 1], R2 + 1e-6)
    ep = BatchedEpisodes(engine, np.repeat(state0, 3, axis=0), obstacle_script=script, max_steps=steps, margin=margin,
                         outcomes=True, record_obstacles=True)
    res = ep.run(max_steps=steps)
    out = res["outcomes"]
    assert np.array_equal(res["history"][:k, 0], hist[:k])               # the ego path before k is unchanged
    assert np.array_equal(res["history"][:k2, 1], hist[:k2]) and np.array_equal(res["history"][:k2, 2], hist[:k2])
    assert out["first_contact_eval"][0] == k and out["first_contact_obs"][0] == 0
    assert out["min_clearance"][0] == -R2
    assert out["min_clearance_eval"][0] == k and out["min_clearance_obs"][0] == 0
    assert out["first_contact_eval"][1] == k2 and out["first_contact_obs"][1] == 1 and out["contact_evals"][1] == 1
    assert abs(out["min_clearance"][1] + 1e-6) < 1e-9 and out["min_clearance_eval"][1] == k2
    assert out["first_contact_eval"][2] == -1 and out["contact_evals"][2] == 0
    assert abs(out["min_clearance"][2] - 1e-6) < 1e-9 and out["min_clearance_eval"][2] == k2
    # the recorded poses are the script's frames, and all columns match the oracle
    prm = _prm(engine, PI)
    for b in range(3):
        n = int(res["steps"][b])
        track = script[np.minimum(np.arange(n + 1), S - 1), b]
        assert np.array_equal(res["obstacle_history"][:n + 1, b], track)
        _assert_outcome(out, b, _oracle(res, b, state0[0], track, prm), names, ints, "forced")
    engine.close()


@pytest.fixture(scope="module")
def synthetic_batch(jm):
    course, dl, engine = _intersection(jm, 4096)
    state0, obst = _bench_workload(course, 4096)
    # no seed of this workload has a failed solve (seeds 0-8 and 11 tried), so 16 episodes start above the QP's speed
    # cap, which the solver reports as infeasible: the ego brakes with MAX_DECEL until it is back under the cap
    state0[FAST, 2] = 9.0
    margin = C.cutoff_margin(GEO, dl)
    BatchedEpisodes = jm[2]
    runs = {}
    for outcomes in (True, False):
        ep = BatchedEpisodes(engine, state0, obstacles=obst.copy(), frame_window=10, margin=margin, max_steps=400,
                             outcomes=outcomes)
        runs[outcomes] = ep.run(max_steps=400)
    yield engine, state0, obst, runs
    engine.close()


def test_synthetic_batch_at_scale(jm, synthetic_batch):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    engine, state0, obst, runs = synthetic_batch
    res = runs[True]
    out = res["outcomes"]
    B = len(state0)
    n_max = int(res["steps"].max())
    tracks = _constant_tracks(obst, n_max, engine.dt)
    prm = _prm(engine, PI)
    for b in range(B):
        n = int(res["steps"][b])
        _assert_outcome(out, b, _oracle(res, b, state0[b], tracks[:n + 1, b], prm), names, ints, "synthetic")
    # the batch covers the interesting cases
    contact = out["first_contact_eval"] >= 0
    assert contact.any() and (~contact).any()
    assert (out["cut_steps"] > 0).any()
    assert (out["failed_solves"][FAST] > 0).all()
    assert (out["limit_steps"] == 0).all()
    assert np.array_equal(out["cut_steps"], (res["flags"] == 1).sum(axis=0))


def test_outcomes_do_not_change_the_episodes(jm, synthetic_batch):
    engine, state0, obst, runs = synthetic_batch
    a, b = runs[True], runs[False]
    assert "outcomes" not in b and "obstacle_history" not in a
    for key in ("steps", "done", "state"):
        assert np.array_equal(a[key], b[key]), key
    assert a["iterations"] == b["iterations"]
    assert np.array_equal(a["history"], b["history"], equal_nan=True)
    assert np.array_equal(a["flags"], b["flags"])


def test_limit_flags_are_counted(jm):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    course, dl, engine = _intersection(jm, 64)
    state0, obst = _bench_workload(course, 64, seed=5)
    steps = 60
    # 15 s at dt = 0.2 is 75 obstacle prediction steps, more than the kernel's 71: every check reports flag = -1
    ep = BatchedEpisodes(engine, state0, obstacles=obst.copy(), frame_window=10, margin=C.cutoff_margin(GEO, dl),
                         max_steps=steps, horizon_s=15.0, outcomes=True)
    res = ep.run(max_steps=steps)
    out = res["outcomes"]
    assert (res["steps"] > 0).all()
    assert np.array_equal(out["limit_steps"], res["steps"]) and (out["cut_steps"] == 0).all()
    tracks = _constant_tracks(obst, steps, engine.dt)
    prm = _prm(engine, PI)
    for b in range(64):
        n = int(res["steps"][b])
        _assert_outcome(out, b, _oracle(res, b, state0[b], tracks[:n + 1, b], prm), names, ints, "limit")
    engine.close()


def test_graph_replay_gives_the_same_outcomes(jm):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    course = synth.load_course("intersection")
    dl = float(np.linalg.norm(course[0, :2] - course[1, :2]))
    state0, obst = _bench_workload(course, 96, seed=3)
    margin = C.cutoff_margin(GEO, dl)
    got = []
    for use_graph in (False, True):
        engine = BatchedMPC([course], dl=dl, T=13, max_batch=96)
        ep = BatchedEpisodes(engine, state0, obstacles=obst.copy(), frame_window=10, margin=margin, max_steps=400,
                             outcomes=True, record_obstacles=True)
        got.append(ep.run(max_steps=400, use_graph=use_graph))
        engine.close()
    a, b = got
    assert np.array_equal(a["steps"], b["steps"]) and np.array_equal(a["done"], b["done"])
    for n in names:
        assert np.array_equal(a["outcomes"][n], b["outcomes"][n]), n
    # the graph loop stops on an 8-iteration boundary after one eager iteration: the row counts may differ, the rows
    # past the last executed step are NaN in both
    rows = int(a["steps"].max()) + 1
    assert np.array_equal(a["obstacle_history"][:rows], b["obstacle_history"][:rows], equal_nan=True)
    assert np.isnan(a["obstacle_history"][rows:]).all() and np.isnan(b["obstacle_history"][rows:]).all()


def test_planned_scenarios(jm, golden_dir):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    from junction_mpc import planner as P
    from junction_mpc.scenarios import run_planned_scenarios
    z = load_planner_golden(golden_dir)
    variants = [str(n) for n in z["variants"]]
    g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
    inp = dict(start=np.stack([g(n, "start") for n in variants]),
               goal_point=np.stack([g(n, "goal_point") for n in variants]),
               goal_area=np.stack([g(n, "goal_area") for n in variants]),
               allowed_dtheta=np.array([float(g(n, "allowed_dtheta")) for n in variants]),
               scenes=[[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in variants],
               scene_id=np.arange(len(variants)), weights=np.stack([g(n, "weights") for n in variants]))
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"],
                               max_batch=64)
    specs = SCENARIO_OBSTACLES["intersection"]
    kw = dict(obstacles=[specs] * len(variants), frame_window=10, T=13, max_steps=160, max_expansions=8192, max_path=32,
              planner=planner, outcomes=True)
    lean = run_planned_scenarios(**inp, record_history=False, **kw)
    full = run_planned_scenarios(**inp, record_history=True, **kw)
    assert "history" not in lean and "flags" not in lean
    for key in ("steps", "done", "state", "plan_status"):
        assert np.array_equal(lean[key], full[key]), key
    for n in names:
        assert np.array_equal(lean["outcomes"][n], full["outcomes"][n]), n
    out = full["outcomes"]
    failed = np.flatnonzero(full["done"] == 3)
    assert len(failed) >= 2
    empty = dict(min_clearance=math.inf, min_clearance_eval=-1, min_clearance_obs=-1, first_contact_eval=-1,
                 first_contact_obs=-1)
    for b in failed:
        for n in names:
            assert out[n][b] == empty.get(n, 0), (b, n)
    plans = planner.plan(**inp, max_expansions=8192, max_path=32)
    track = _scripted_tracks(specs, int(full["steps"].max()))
    from junction_mpc.config import MPCConfig
    p = MPCConfig.default().param_vector(dl=0.083)
    prm = dict(dt=float(p[PI["dt"]]), L=float(p[PI["L"]]), max_steer=float(p[PI["max_steer"]]))
    driven = np.flatnonzero(full["done"] != 3)
    assert len(driven) >= 10
    for b in driven:
        t0 = plans.trajectory(b)[0]
        state0 = np.array([t0[0], t0[1], 0.0, t0[2]])
        n = int(full["steps"][b])
        _assert_outcome(out, b, _oracle(full, b, state0, track[:n + 1], prm), names, ints, variants[b])


def test_no_obstacles(jm):
    synth, BatchedMPC, BatchedEpisodes, PI, names, ints = jm
    course, dl, engine = _intersection(jm, 16)
    state0, _ = _bench_workload(course, 16, seed=9)
    steps = 80
    ep = BatchedEpisodes(engine, state0, max_steps=steps, margin=C.cutoff_margin(GEO, dl), outcomes=True,
                         record_obstacles=True)
    res = ep.run(max_steps=steps)
    out = res["outcomes"]
    assert np.isinf(out["min_clearance"]).all() and (out["min_clearance"] > 0).all()
    for n in ("min_clearance_eval", "min_clearance_obs", "first_contact_eval", "first_contact_obs"):
        assert (out[n] == -1).all(), n
    assert (out["contact_evals"] == 0).all() and (out["cut_steps"] == 0).all() and (out["limit_steps"] == 0).all()
    assert res["obstacle_history"].shape == (res["iterations"] + 1, 16, 0, 6)
    prm = _prm(engine, PI)
    for b in range(16):
        n = int(res["steps"][b])
        _assert_outcome(out, b, _oracle(res, b, state0[b], np.zeros((n + 1, 0, 6)), prm), names, ints, "free")
    assert (out["distance"] > 0).all() and (out["max_abs_accel"] > 0).all()
    engine.close()
