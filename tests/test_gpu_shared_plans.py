"""Scene mates predicted along their shared MPC plans (jmpc_collision_planned, jmpc_scene_plans,
BatchedEpisodes(share_plans=True)).

Gates:
  * constant plans are today's kernel: jmpc_collision_planned with every plan entry equal to the row's (a, steer) gives
    jmpc_collision's flags and cut lengths bit for bit on the synthetic config-3 / config-4 workloads;
  * real plans against the collision oracle (oracle/shared_plans.collision_cut(..., plans=...)), exactly;
  * scenes stepped with iterate(): every evaluation's plans equal oracle/shared_plans.mate_plans of a snapshot, a
    sample of the flags equals the oracle on that evaluation's rows and plans, and the mate rows are unchanged;
  * the reductions: share_plans=False is today's run, iteration 0 is identical in both modes, graph replay, outcomes
    on / off, mates plus extras, planned scenes with a failed search.
"""
import ctypes

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import scene_exchange as SX
from oracle import shared_plans as SP

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
    import torch
    from junction_mpc import _cabi, synth
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
    # a course that doubles back 0.05 m beside itself, far from the junction: the index rule raises (done = 2 mid-run)
    xs = np.concatenate([np.linspace(0, 20, 201), np.linspace(20, 10, 101)]) + 1000.0
    ys = np.concatenate([np.zeros(201), np.full(101, 0.05)]) + 1000.0
    courses.append(np.stack([xs, ys, np.zeros(302)], axis=1))
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    return dict(z=z, torch=torch, cabi=_cabi, synth=synth, BatchedMPC=BatchedMPC, BatchedEpisodes=BatchedEpisodes,
                PI=PARAM_INDEX, names=OUTCOME_NAMES, courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl))


def _scenes(jm, n_scenes, seed=7, forced=True):
    """n_scenes x K vehicles, vehicle j of a scene from approach j on a random route, 0-8 m along it at 2-5 m/s.
    forced: scene 0's last vehicle drives the doubling-back course (done = 2), every 16th scene's first vehicle starts
    above the QP's speed cap (failed solves, warm = 0, until it has braked below it)."""
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


def _same_episodes(a, b, names, history=True):
    for key in ("steps", "done", "state"):
        assert np.array_equal(a[key], b[key]), key
    if history:
        n = min(len(a["history"]), len(b["history"]))
        assert np.array_equal(a["history"][:n], b["history"][:n], equal_nan=True)
        assert np.array_equal(a["flags"][:n], b["flags"][:n])
    if "outcomes" in a and "outcomes" in b:
        for n in names:
            assert np.array_equal(a["outcomes"][n], b["outcomes"][n]), n


def _device_collision(jm, engine, agent_idx, v, obst, fw, margin, plans=None, n_planned=0):
    torch = jm["torch"]
    dev = torch.device("cuda", engine.device)
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)   # noqa: E731
    B = len(agent_idx)
    flag, clen = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    engine.collision(t(agent_idx, torch.int32), t(v, torch.float64), t(obst, torch.float64), fw, margin, flag, clen,
                     plans=None if plans is None else t(plans, torch.float64), n_planned=n_planned)
    torch.cuda.synchronize(dev)
    return flag.cpu().numpy(), clen.cpu().numpy()


def _near_workload(jm, config, B, seed=99):
    w = jm["synth"].make_workload(config, B=B)
    course = w["courses"][0]
    rng = np.random.default_rng(seed)
    near = rng.random(B) < 0.5                          # half of the first obstacles next to the path
    k = np.minimum(w["agent_idx"] + rng.integers(0, 200, B), len(course) - 1)
    w["obstacles"][near, 0, 0] = course[k[near], 0] + rng.uniform(-8, 8, near.sum())
    w["obstacles"][near, 0, 1] = course[k[near], 1] + rng.uniform(-8, 8, near.sum())
    return w


@pytest.mark.parametrize("config", [3, 4])
def test_constant_plans_are_todays_kernel(jm, config):
    B = 4096
    w = _near_workload(jm, config, B)
    course, obst = w["courses"][0], w["obstacles"]
    n_obs = obst.shape[1]
    margin = C.cutoff_margin(GEO, w["dl"])
    engine = jm["BatchedMPC"]([course], dl=w["dl"], T=13, max_batch=B)
    v = w["state"][:, 2].copy()
    v[::17] = 30 / 3.6
    ref = _device_collision(jm, engine, w["agent_idx"], v, obst, w["frame_window"], margin)
    assert 0.05 < ref[0].mean() < 0.95
    for n_planned in sorted({1, n_obs}):
        for plan_len in (1, 12, 40):
            plans = np.repeat(obst[:, :n_planned, None, 4:6], plan_len, axis=2)
            got = _device_collision(jm, engine, w["agent_idx"], v, obst, w["frame_window"], margin, plans, n_planned)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), (n_planned, plan_len)
    engine.close()


def test_real_plans_match_the_oracle(jm):
    w = jm["synth"].make_workload(3, B=64)
    course = w["courses"][0]
    margin = C.cutoff_margin(GEO, w["dl"])
    engine = jm["BatchedMPC"]([course], dl=w["dl"], T=13, max_batch=128)
    p = engine.default_params
    PI = jm["PI"]
    lo, hi, ms = p[PI["max_decel"]], p[PI["max_accel"]], p[PI["max_steer"]]
    rng = np.random.default_rng(5)
    n, fw = 72, 20
    # (plan_len, n_obs, n_planned): plans shorter than, equal to and longer than the 35 predictor frames
    cases = [(1, 1, 1), (5, 3, 2), (12, 8, 5), (34, 2, 1), (35, 4, 4), (36, 6, 3), (40, 8, 8), (20, 5, 0)]
    total = changed = flagged = 0
    for plan_len, n_obs, n_planned in cases:
        a_idx = rng.integers(0, len(course) - 300, n)
        v = rng.uniform(0, 8, n)
        obst = np.zeros((n, n_obs, 6))
        k = np.minimum(a_idx[:, None] + rng.integers(20, 250, (n, n_obs)), len(course) - 1)
        ang = rng.uniform(-np.pi, np.pi, (n, n_obs))
        obst[..., 0] = course[k, 0] - 12 * np.cos(ang) + rng.uniform(-3, 3, (n, n_obs))
        obst[..., 1] = course[k, 1] - 12 * np.sin(ang) + rng.uniform(-3, 3, (n, n_obs))
        obst[..., 2] = rng.uniform(0, 8, (n, n_obs))
        obst[..., 3] = ang
        obst[..., 4] = rng.uniform(lo, hi, (n, n_obs))
        obst[..., 5] = rng.uniform(-ms, ms, (n, n_obs))
        plans = np.stack([rng.uniform(lo, hi, (n, n_planned, plan_len)), rng.uniform(-ms, ms, (n, n_planned, plan_len))],
                         axis=-1)
        flag, clen = _device_collision(jm, engine, a_idx, v, obst, fw, margin, plans, n_planned)
        const = _device_collision(jm, engine, a_idx, v, obst, fw, margin)
        for i in range(n):
            pl = [plans[i, s] for s in range(n_planned)] + [None] * (n_obs - n_planned)
            f, cl = SP.collision_cut(GEO, course, int(a_idx[i]), float(v[i]), obst[i], dt=0.2, frame_window=fw,
                                    max_accel=hi, max_speed=p[PI["sim_max_speed"]], margin=margin, plans=pl)
            assert (int(f), cl) == (int(flag[i]), int(clen[i])), (plan_len, n_obs, n_planned, i)
        total += n
        flagged += int(flag.sum())
        changed += int(((flag != const[0]) | (clen != const[1])).sum())
    print(f"\n[shared plans] {total} instances against the oracle, {flagged} flagged; the plans changed the flag or "
          f"cut of {changed} against constant inputs")
    assert changed > 0 and 0 < flagged < total
    # argument errors of the new entry points
    cabi, lib, h = jm["cabi"], engine._lib, engine._h
    args = lambda n_obs, plans, n_planned, plan_len: (h, 0, None, None, None, None, n_obs, plans, n_planned,  # noqa: E731
                                                       plan_len, 10, 8, 7.0, None, None, None, None)
    dummy = ctypes.c_void_p(1)             # never dereferenced: every call below fails its checks first
    with pytest.raises(cabi.JmpcError, match=r"n_planned must be in \[0, n_obs\]"):
        cabi.check(lib.jmpc_collision_planned(*args(2, dummy, 3, 4)), "jmpc_collision_planned")
    with pytest.raises(cabi.JmpcError, match=r"n_planned must be in \[0, n_obs\]"):
        cabi.check(lib.jmpc_collision_planned(*args(2, dummy, -1, 4)), "jmpc_collision_planned")
    with pytest.raises(cabi.JmpcError, match="plan_len must be >= 1"):
        cabi.check(lib.jmpc_collision_planned(*args(2, dummy, 1, 0)), "jmpc_collision_planned")
    with pytest.raises(cabi.JmpcError, match="plans is NULL"):
        cabi.check(lib.jmpc_collision_planned(*args(2, None, 1, 4)), "jmpc_collision_planned")
    with pytest.raises(cabi.JmpcError, match="jmpc_collision_planned: NULL array"):
        cabi.check(lib.jmpc_collision_planned(*args(2, dummy, 1, 4)), "jmpc_collision_planned")
    with pytest.raises(cabi.JmpcError, match="T must be >= 2"):
        cabi.check(lib.jmpc_scene_plans(h, 8, 4, 1, *([dummy] * 6), 3, dummy, None), "jmpc_scene_plans")
    with pytest.raises(cabi.JmpcError, match="multiple of k"):
        cabi.check(lib.jmpc_scene_plans(h, 6, 4, 13, *([dummy] * 6), 3, dummy, None), "jmpc_scene_plans")
    with pytest.raises(cabi.JmpcError, match=r"n_obs must be in \[k - 1, 8\]"):
        cabi.check(lib.jmpc_scene_plans(h, 8, 4, 13, *([dummy] * 6), 2, dummy, None), "jmpc_scene_plans")
    engine.close()


def _snap(ep):
    c = lambda t: t.cpu().numpy().copy()      # noqa: E731
    return dict(oa=c(ep.oa), od=c(ep.od), warm=c(ep.warm), done=c(ep.done), steps=c(ep.steps), rows=c(ep.scene_obs),
                plans=c(ep.scene_plans))


def _step_and_check(jm, ep, engine, cid, params, sample=3, seed=0):
    """Steps `ep` with iterate() to the end, checking every evaluation's plans against mate_plans and a sample of the
    vehicles stepped in each iteration against the collision oracle.  Returns run()'s result and counters."""
    PI, courses = jm["PI"], jm["courses"]
    max_steer = params[:, PI["max_steer"]]
    rng = np.random.default_rng(seed)
    ep._start()
    prev = _snap(ep)
    n_valid = n_fallback = checked = 0
    n_extra = ep.n_obs - (K - 1)
    while ep.iteration < STEPS:
        ref = SP.mate_plans(prev["oa"], prev["od"], prev["warm"], prev["done"], prev["rows"], max_steer, K)
        assert np.array_equal(prev["plans"], ref), ep.iteration
        ep.iterate()
        now = _snap(ep)
        stepped = np.flatnonzero(now["steps"] > prev["steps"])
        flag, clen = ep.flag.cpu().numpy(), ep.course_len.cpu().numpy()
        a_idx, v = ep.agent_idx.cpu().numpy(), ep.v.cpu().numpy()
        for b in rng.choice(stepped, min(sample, len(stepped)), replace=False):
            pr = params[b]
            pl = [prev["plans"][b, s] for s in range(K - 1)] + [None] * n_extra
            f, cl = SP.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]), prev["rows"][b], dt=pr[PI["dt"]],
                                    frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                                    max_speed=pr[PI["sim_max_speed"]], margin=ep.margin, plans=pl)
            assert (int(f), cl) == (int(flag[b]), int(clen[b])), (ep.iteration, b)
            checked += 1
        mate_ok = (prev["done"] == 0) & (prev["warm"] != 0)
        n_valid += int(mate_ok.sum())
        n_fallback += int((~mate_ok).sum())
        prev = now
        if (now["done"] != 0).all():
            break
    ref = SP.mate_plans(prev["oa"], prev["od"], prev["warm"], prev["done"], prev["rows"], max_steer, K)
    assert np.array_equal(prev["plans"], ref)
    return ep.run(max_steps=ep.iteration), dict(valid=n_valid, fallback=n_fallback, checked=checked)


def test_scene_plans_and_flags_against_the_oracle(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=7)
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=K, share_plans=True, outcomes=True,
                               record_obstacles=True)
    assert tuple(ep.scene_plans.shape) == (len(state0), K - 1, 12, 2)
    res, n = _step_and_check(jm, ep, engine, cid, params)
    print(f"\n[shared plans scenes] {res['iterations']} iterations, vehicle-evaluations with a plan {n['valid']}, "
          f"without (row repeated) {n['fallback']}, flags checked against the oracle {n['checked']}; "
          f"done codes {np.bincount(res['done']).tolist()}")
    assert n["valid"] > 0 and n["fallback"] > 0 and n["checked"] > 100
    # the forced cases occur: done = 2 mid-run, goals, failed solves
    assert res["done"][K - 1] == 2 and (res["done"] == 1).any()
    assert (res["outcomes"]["failed_solves"][0::16 * K] > 0).all()
    # the mate rows are those of the exchange, as without shared plans
    oh = res["obstacle_history"]
    rows = SX.mate_rows(state0, res["history"], res["steps"], res["done"], params[:, jm["PI"]["max_steer"]], K, len(oh))
    e = np.arange(len(oh))[:, None]
    active = (e <= res["steps"][None, :]) & ~np.isin(res["done"], SX.NEVER_STEPPED)[None, :]
    assert np.array_equal(oh[:, :, :K - 1][active], rows[active])
    engine.close()


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


def test_reductions(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=5)
    BE = jm["BatchedEpisodes"]
    kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS, agents_per_scene=K)
    runs, names = {}, {}
    for key, extra in (("before", dict()), ("off", dict(share_plans=False)), ("on", dict(share_plans=True)),
                       ("on_outcomes", dict(share_plans=True, outcomes=True, record_obstacles=True)),
                       ("off_outcomes", dict(outcomes=True, record_obstacles=True))):
        lib = engine._lib
        engine._lib = _Calls(lib)
        try:
            ep = BE(engine, state0, **kw, **extra)
            runs[key] = ep.run(max_steps=STEPS)
            names[key] = engine._lib.names
        finally:
            engine._lib = lib
        assert (ep.scene_plans is None) == (not extra.get("share_plans", False))
    # share_plans=False: the same library calls in the same order as without the option, and the same episodes
    assert names["off"] == names["before"]
    assert not any(n in ("jmpc_scene_plans", "jmpc_collision_planned") for n in names["off"])
    _same_episodes(runs["before"], runs["off"], jm["names"])
    # on: one plan exchange after every scene exchange, every collision call planned
    on = names["on"]
    assert on.count("jmpc_scene_plans") == on.count("jmpc_scene_exchange") == runs["on"]["iterations"] + 1
    assert all(on[i + 1] == "jmpc_scene_plans" for i, n in enumerate(on) if n == "jmpc_scene_exchange")
    assert "jmpc_collision" not in on and on.count("jmpc_collision_planned") == runs["on"]["iterations"]
    # outcomes observe only
    _same_episodes(runs["on"], runs["on_outcomes"], jm["names"])
    # iteration 0 is identical in both modes (no mate has a plan yet); then the runs differ
    a, b = runs["off"], runs["on"]
    assert np.array_equal(a["history"][0], b["history"][0], equal_nan=True)
    assert np.array_equal(a["flags"][0], b["flags"][0])
    n = min(len(a["history"]), len(b["history"]))
    differ = ~np.all((a["history"][:n] == b["history"][:n]) | (np.isnan(a["history"][:n]) & np.isnan(b["history"][:n])),
                     axis=(0, 2))
    flags_differ = (a["flags"][:n] != b["flags"][:n]).any(axis=0)
    print(f"\n[shared plans reductions] {len(state0)} vehicles: {int(differ.sum())} drive differently with shared plans, "
          f"{int(flags_differ.sum())} see different flags; outcome contacts off / on "
          f"{int((runs['off_outcomes']['outcomes']['first_contact_eval'] >= 0).sum())} / "
          f"{int((runs['on_outcomes']['outcomes']['first_contact_eval'] >= 0).sum())}")
    assert differ.sum() > 0
    # the mate rows and the outcome record's evaluation 0 are the same in both modes
    assert np.array_equal(runs["off_outcomes"]["obstacle_history"][0], runs["on_outcomes"]["obstacle_history"][0])
    # graph replay equals eager iteration
    ep = BE(engine, state0, **kw, share_plans=True, outcomes=True, record_obstacles=True)
    g = ep.run(max_steps=STEPS, use_graph=True)
    e = runs["on_outcomes"]
    _same_episodes(e, g, jm["names"])
    rows = int(e["steps"].max()) + 1
    assert np.array_equal(e["obstacle_history"][:rows], g["obstacle_history"][:rows], equal_nan=True)
    # argument checks on the device path
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        BE(engine, state0, course_id=cid, share_plans=True)
    bad = params.copy()
    bad[6, jm["PI"]["dt"]] = 0.1
    with pytest.raises(ValueError, match="one dt per scene: scene 1"):
        BE(engine, state0, course_id=cid, params=bad, agents_per_scene=K, share_plans=True)
    engine.close()


def test_mates_plus_extras(jm):
    engine, state0, cid, params = _scenes(jm, 16, seed=9)
    B = len(state0)
    rng = np.random.default_rng(1)
    obst = np.zeros((B, 2, 6))
    ang = rng.uniform(-np.pi, np.pi, (B, 2))
    obst[:, :, 0] = rng.uniform(-15, 15, (B, 2)) - 20 * np.cos(ang)
    obst[:, :, 1] = rng.uniform(-15, 15, (B, 2)) - 20 * np.sin(ang)
    obst[:, :, 2] = rng.uniform(2, 6, (B, 2))
    obst[:, :, 3] = ang
    obst[:, :, 4] = rng.uniform(-1, 1, (B, 2))
    obst[:, :, 5] = rng.uniform(-.05, .05, (B, 2))
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, obstacles=obst.copy(), frame_window=10,
                               margin=jm["margin"], max_steps=STEPS, agents_per_scene=K, share_plans=True,
                               outcomes=True, record_obstacles=True)
    assert ep.n_obs == K - 1 + 2 and tuple(ep.scene_plans.shape) == (B, K - 1, 12, 2)
    res, n = _step_and_check(jm, ep, engine, cid, params, sample=4, seed=1)
    assert n["checked"] > 50
    assert (res["outcomes"]["min_clearance_obs"] >= K - 1).any()
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
              agents_per_scene=K, share_plans=True)
    names = [n for s in scenes for n in s]
    res = run_planned_scenarios(**inputs(names), obstacles=[SCENARIO_OBSTACLES] * 3, **kw)
    assert res["plan_status"][7] != P.STATUS_FOUND
    assert res["done"][4:8].tolist() == [4, 4, 4, 3] and (res["steps"][4:8] == 0).all()
    assert (res["steps"][[0, 1, 2, 3, 8, 9, 10, 11]] > 0).all()
    names2 = scenes[0] + scenes[2]
    ref = run_planned_scenarios(**inputs(names2), obstacles=[SCENARIO_OBSTACLES] * 2, **kw)
    keep = [0, 1, 2, 3, 8, 9, 10, 11]
    for key in ("steps", "done", "state"):
        assert np.array_equal(res[key][keep], ref[key]), key
    n = min(len(res["history"]), len(ref["history"]))
    assert np.array_equal(res["history"][:n][:, keep], ref["history"][:n], equal_nan=True)
    for name in jm["names"]:
        assert np.array_equal(res["outcomes"][name][keep], ref["outcomes"][name]), name
    planner.close()
