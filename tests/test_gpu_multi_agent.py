"""Scenes of several MPC-driven vehicles that see each other as moving obstacles (jmpc_scene_exchange,
BatchedEpisodes(agents_per_scene=k)).

The scenes are built from the recorded planner courses of the intersection's four approaches
(tests/golden/planner.npz: intersection_{1..4}_{1..3}), one vehicle per approach, starts staggered along the courses
so that the paths meet in the junction.  Gates:
  * replay: the scene run equals driving every vehicle alone against its recorded obstacle rows
    (obstacle_script = obstacle_history[:, b]), bit for bit -- History, flags, steps, done, state and outcome record;
  * the recorded mate rows equal oracle/scene_exchange.py applied to the run's own History, bit for bit;
  * the reductions (k = 1, outcomes on / off, graph replay, mates plus extras) and planned scenes with a failed search.
"""
import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import scene_exchange as SX

pytestmark = pytest.mark.gpu

K = 4
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
GEO = C.CarGeometry()
STEPS = 200
SCENARIO_OBSTACLES = [dict(kind="t_intersection", direction=1, offset=2., turning=False, speed=25 / 3.6, dt=0.2),
                      dict(kind="t_intersection", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)]


@pytest.fixture(scope="module")
def jm(golden_dir):
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    from junction_mpc.episodes import OUTCOME_NAMES, BatchedEpisodes
    z = load_planner_golden(golden_dir)
    courses = []
    for row in ROUTES:
        for name in row:
            c = np.array(z[f"{name}/trajectory"], dtype=np.float64)
            synth.smooth_yaw_inplace(c[:, 2])
            courses.append(c)
    # a course that doubles back 0.05 m beside itself, far from the junction: the index rule raises once the ego
    # reaches the second leg (done = 2 mid-run)
    xs = np.concatenate([np.linspace(0, 20, 201), np.linspace(20, 10, 101)]) + 1000.0
    ys = np.concatenate([np.zeros(201), np.full(101, 0.05)]) + 1000.0
    courses.append(np.stack([xs, ys, np.zeros(302)], axis=1))
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    return dict(z=z, synth=synth, BatchedMPC=BatchedMPC, BatchedEpisodes=BatchedEpisodes, PI=PARAM_INDEX,
                names=OUTCOME_NAMES, courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl))


def _scenes(jm, n_scenes, seed=7, forced=True):
    """Start states, course ids and params rows of n_scenes x K vehicles: vehicle j of a scene comes from approach j on
    a random route, 0-8 m along it at 2-5 m/s.  forced: scene 0's last vehicle drives the doubling-back course, and
    every 16th scene's first vehicle starts above the QP's speed cap (failed solves until it has braked below it)."""
    rng = np.random.default_rng(seed)
    courses, PI = jm["courses"], jm["PI"]
    B = n_scenes * K
    cid = (np.arange(B) % K) * 3 + rng.integers(0, 3, B)
    off = rng.integers(0, 96, B)
    state0 = np.empty((B, 4))
    for b in range(B):
        c = courses[cid[b]]
        state0[b] = [c[off[b], 0], c[off[b], 1], 0.0, c[off[b], 2]]
    state0[:, 2] = rng.uniform(2, 5, B)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=max(B, 64))
    params = np.repeat(engine.default_params[None, :], B, axis=0)
    if forced:
        hp = len(courses) - 1
        cid[K - 1] = hp
        state0[K - 1] = [courses[hp][0, 0], courses[hp][0, 1], 3.0, 0.0]
        params[K - 1, PI["dl"]] = 0.1
        state0[0::16 * K, 2] = 9.0
    return engine, state0, cid, params


def _assert_same_episodes(a, b, names, history=True):
    for key in ("steps", "done", "state"):
        assert np.array_equal(a[key], b[key]), key
    if history:
        n = min(len(a["history"]), len(b["history"]))
        assert np.array_equal(a["history"][:n], b["history"][:n], equal_nan=True)
        assert np.array_equal(a["flags"][:n], b["flags"][:n])
    if "outcomes" in a and "outcomes" in b:
        for n in names:
            assert np.array_equal(a["outcomes"][n], b["outcomes"][n]), n


def _replay_and_oracle(jm, engine, state0, cid, params, res, k, n_extra=0):
    """The scene run `res` (record_history, outcomes, record_obstacles) against (1) every vehicle driven alone on its
    recorded rows and (2) the oracle's mate rows.  Returns the oracle rows."""
    oh = res["obstacle_history"]
    solo = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                                 max_steps=STEPS, obstacle_script=oh, outcomes=True, record_obstacles=True)
    ref = solo.run(max_steps=STEPS)
    assert ref["iterations"] == res["iterations"]
    _assert_same_episodes(res, ref, jm["names"])
    assert np.array_equal(res["obstacle_history"], ref["obstacle_history"], equal_nan=True)

    B = len(state0)
    max_steer = params[:, jm["PI"]["max_steer"]]
    rows = SX.mate_rows(state0, res["history"], res["steps"], res["done"], max_steer, k, len(oh))
    e = np.arange(len(oh))[:, None]
    active = (e <= res["steps"][None, :]) & ~np.isin(res["done"], SX.NEVER_STEPPED)[None, :]    # rows the run recorded
    assert np.array_equal(oh[:, :, :k - 1][active], rows[active])
    assert np.isnan(oh[~active]).all()
    assert oh.shape == (len(oh), B, k - 1 + n_extra, 6)
    return rows, active


@pytest.fixture(scope="module")
def big(jm):
    """4 096 scenes x 4 vehicles, History, outcomes and obstacle rows on."""
    engine, state0, cid, params = _scenes(jm, 4096)
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=K, outcomes=True, record_obstacles=True)
    res = ep.run(max_steps=STEPS)
    yield engine, state0, cid, params, res
    engine.close()


def test_replay_equals_solo_driving_and_mate_rows_equal_the_oracle_at_scale(jm, big):
    engine, state0, cid, params, res = big
    rows, active = _replay_and_oracle(jm, engine, state0, cid, params, res, K)
    done, out = res["done"], res["outcomes"]
    # the forced cases occur: done = 2 mid-run, goals, failed solves, and mates seen parked by vehicles still driving
    assert done[K - 1] == 2 and res["steps"][K - 1] > 0
    assert (done == 1).any()
    assert (out["failed_solves"][0::16 * K] > 0).all()
    parked = active[:, :, None] & (rows[..., 2] == 0) & (rows[..., 4] == 0) & (rows[..., 5] == 0)
    assert parked[1:, 0:K - 1].any()                       # scene 0's vehicles see the done = 2 vehicle parked
    finished_mates = 0
    for s in range(0, 4096, 97):
        for j in range(K):
            b = s * K + j
            finished_mates += int(parked[int(res["steps"][b]), b].sum())
    assert finished_mates > 0
    print(f"\n[multi-agent scale] {len(done)} vehicles: done codes {np.bincount(done).tolist()}, "
          f"{res['iterations']} iterations, {int(res['steps'].sum())} control steps")


def test_the_interaction_is_real(jm, big):
    engine, state0, cid, params, res = big
    out = res["outcomes"]
    B = len(state0)
    cut = out["cut_steps"] > 0
    close = out["min_clearance"] < 3.0
    touch = out["first_contact_eval"] >= 0
    print(f"\n[multi-agent interaction] {B} vehicles, no scripted obstacles: {int(cut.sum())} with cut steps "
          f"({cut.mean():.1%}), {int(close.sum())} came within 3 m of a mate's circles, {int(touch.sum())} touched one")
    assert cut.mean() >= 0.05
    assert close.sum() >= 10


class _Calls:
    """The engine's library with every call's name recorded."""
    def __init__(self, lib):
        self.lib, self.names = lib, []

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.startswith("jmpc_"):
            return fn

        def call(*a):
            self.names.append(name)
            return fn(*a)
        return call


def test_one_vehicle_per_scene_is_todays_run(jm):
    engine, state0, cid, params = _scenes(jm, 16, seed=3, forced=False)
    obst = np.zeros((len(state0), 2, 6))
    obst[:, :, :2] = state0[:, None, :2] + [[20.0, 0.0], [0.0, 20.0]]
    obst[:, :, 2] = 2.0
    obst[:, 0, 3], obst[:, 1, 3] = np.pi, -np.pi / 2
    got, names, launches = [], [], []
    for kw in (dict(), dict(agents_per_scene=1)):
        lib = engine._lib
        engine._lib = _Calls(lib)
        try:
            l0 = engine.launch_count
            ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, obstacles=obst.copy(),
                                       frame_window=10, margin=jm["margin"], max_steps=STEPS, outcomes=True, **kw)
            got.append(ep.run(max_steps=STEPS))
            launches.append(engine.launch_count - l0)
            names.append(engine._lib.names)
            assert ep.scene_obs is None
        finally:
            engine._lib = lib
    _assert_same_episodes(got[0], got[1], jm["names"])
    assert launches[0] == launches[1] and names[0] == names[1]
    assert not any(n.startswith("jmpc_scene") for n in names[1])
    # with scenes: one exchange before the loop and one per iteration, nothing else added
    engine._lib = _Calls(engine._lib)
    try:
        ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                                   max_steps=STEPS, agents_per_scene=K)
        r = ep.run(max_steps=STEPS)
        assert engine._lib.names.count("jmpc_scene_exchange") == r["iterations"] + 1
        assert "jmpc_scene_init" not in engine._lib.names                 # only from_plans runs the scene pass
    finally:
        engine._lib = engine._lib.lib
    engine.close()


def test_outcomes_on_and_off_and_graph_replay_give_the_same_episodes(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=5)
    runs = {}
    for key, kw in (("plain", dict()), ("outcomes", dict(outcomes=True, record_obstacles=True)),
                    ("graph", dict(outcomes=True, record_obstacles=True))):
        ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                                   max_steps=STEPS, agents_per_scene=K, **kw)
        runs[key] = ep.run(max_steps=STEPS, use_graph=key == "graph")
    _assert_same_episodes(runs["plain"], runs["outcomes"], jm["names"])
    assert (runs["plain"]["flags"] == 1).any()
    _replay_and_oracle(jm, engine, state0, cid, params, runs["outcomes"], K)
    # the graph loop stops on an 8-iteration boundary: History / obstacle rows past the last executed step are NaN
    a, g = runs["outcomes"], runs["graph"]
    _assert_same_episodes(a, g, jm["names"])
    rows = int(a["steps"].max()) + 1
    assert np.array_equal(a["obstacle_history"][:rows], g["obstacle_history"][:rows], equal_nan=True)
    engine.close()


def test_mates_plus_extras(jm):
    engine, state0, cid, params = _scenes(jm, 32, seed=9)
    B = len(state0)
    rng = np.random.default_rng(1)
    obst = np.zeros((B, 2, 6))
    ang = rng.uniform(-np.pi, np.pi, (B, 2))
    obst[:, :, 0] = rng.uniform(-15, 15, (B, 2)) - 20 * np.cos(ang)
    obst[:, :, 1] = rng.uniform(-15, 15, (B, 2)) - 20 * np.sin(ang)
    obst[:, :, 2] = rng.uniform(2, 6, (B, 2))
    obst[:, :, 3] = ang
    obst[:, :, 5] = rng.uniform(-.05, .05, (B, 2))
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, obstacles=obst.copy(), frame_window=10,
                               margin=jm["margin"], max_steps=STEPS, agents_per_scene=K, outcomes=True,
                               record_obstacles=True)
    res = ep.run(max_steps=STEPS)
    assert ep.n_obs == K - 1 + 2
    rows, active = _replay_and_oracle(jm, engine, state0, cid, params, res, K, n_extra=2)
    # the extras advance with constant inputs as for a single vehicle
    o, L, dt = obst.copy(), 2.86, engine.dt
    oh = res["obstacle_history"]
    for e in range(len(oh)):
        if e:
            o[..., 0] += o[..., 2] * np.cos(o[..., 3]) * dt
            o[..., 1] += o[..., 2] * np.sin(o[..., 3]) * dt
            o[..., 2] += o[..., 4] * dt
            o[..., 3] += (o[..., 2] / L) * np.tan(o[..., 5]) * dt
        np.testing.assert_allclose(oh[e, active[e], K - 1:], o[active[e]], rtol=0, atol=1e-9)
    assert (res["outcomes"]["min_clearance_obs"] >= K - 1).any() and (res["outcomes"]["min_clearance_obs"] < K - 1).any()
    engine.close()


def test_planned_scenes_with_a_failed_search(jm):
    z = jm["z"]
    from junction_mpc import planner as P
    from junction_mpc.scenarios import run_planned_scenarios
    scenes = [[r[0] for r in ROUTES], [r[1] for r in ROUTES[:3]] + ["roundabout_2_3_big"], [r[2] for r in ROUTES]]

    def inputs(names):
        g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
        return dict(start=np.stack([g(n, "start") for n in names]),
                    goal_point=np.stack([g(n, "goal_point") for n in names]),
                    goal_area=np.stack([g(n, "goal_area") for n in names]),
                    allowed_dtheta=np.array([float(g(n, "allowed_dtheta")) for n in names]),
                    scenes=[[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in names],
                    scene_id=np.arange(len(names)), weights=np.stack([g(n, "weights") for n in names]))
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"],
                               max_batch=16)
    kw = dict(frame_window=10, T=13, max_steps=160, max_expansions=8192, max_path=32, planner=planner, outcomes=True,
              agents_per_scene=K)
    names = [n for s in scenes for n in s]
    res = run_planned_scenarios(**inputs(names), obstacles=[SCENARIO_OBSTACLES] * 3, **kw)
    assert res["plan_status"][7] != P.STATUS_FOUND
    assert res["done"][4:8].tolist() == [4, 4, 4, 3] and (res["steps"][4:8] == 0).all()
    assert np.isnan(res["history"][:, 4:8]).all()
    assert (res["steps"][[0, 1, 2, 3, 8, 9, 10, 11]] > 0).all()
    # the other scenes are unaffected: the same two scenes planned and driven without it
    names2 = scenes[0] + scenes[2]
    ref = run_planned_scenarios(**inputs(names2), obstacles=[SCENARIO_OBSTACLES] * 2, **kw)
    keep = [0, 1, 2, 3, 8, 9, 10, 11]
    for key in ("steps", "done", "state"):
        assert np.array_equal(res[key][keep], ref[key]), key
    n = min(len(res["history"]), len(ref["history"]))
    assert np.array_equal(res["history"][:n][:, keep], ref["history"][:n], equal_nan=True)
    for name in jm["names"]:
        assert np.array_equal(res["outcomes"][name][keep], ref["outcomes"][name]), name
    with pytest.raises(ValueError, match="one list per scene"):
        run_planned_scenarios(**inputs(names), obstacles=[SCENARIO_OBSTACLES] * 12, **kw)
    planner.close()


def test_argument_errors_on_the_device_path(jm):
    engine, state0, cid, params = _scenes(jm, 2, forced=False)
    BE = jm["BatchedEpisodes"]
    with pytest.raises(ValueError, match="whole number of scenes"):
        BE(engine, state0[:7], course_id=cid[:7], agents_per_scene=K)
    with pytest.raises(ValueError, match="obstacle_script cannot be combined"):
        BE(engine, state0, course_id=cid, obstacle_script=np.zeros((2, 8, 1, 6)), agents_per_scene=2)
    with pytest.raises(ValueError, match="exceed the 8 obstacle slots"):
        BE(engine, state0, course_id=cid, obstacles=np.zeros((8, 6, 6)), agents_per_scene=K)
    with pytest.raises(ValueError, match="needs outcomes"):
        BE(engine, state0, course_id=cid, agents_per_scene=K, record_obstacles=True)
    from junction_mpc import _cabi
    lib = engine._lib
    with pytest.raises(_cabi.JmpcError, match="multiple of k"):
        _cabi.check(lib.jmpc_scene_exchange(engine._h, 6, 4, 0, *([None] * 8), None), "jmpc_scene_exchange")
    with pytest.raises(_cabi.JmpcError, match=r"\[0, 8\]"):
        _cabi.check(lib.jmpc_scene_exchange(engine._h, 8, 4, 6, *([None] * 8), None), "jmpc_scene_exchange")
    engine.close()
