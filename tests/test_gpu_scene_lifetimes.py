"""Lifetimes of scene vehicles: entry iterations and leaving the scene at the goal (BatchedEpisodes(depart=...,
on_goal=...), jmpc_scene_depart_init, jmpc_scene_enter, jmpc_scene_presence, jmpc_episode_outcomes_scene).

Gates:
  * the defaults are today's run: the same library calls in the same order and bit-identical results, for scenes of 4
    with a rule and for single vehicles;
  * one departure iteration d for a whole scene (no extras) is the depart = 0 scene shifted by d iterations, bit for
    bit;
  * scenes with mixed departures, first_come and "leave", stepped with iterate(): every collision mask equals the rule's
    oracle mask AND oracle presence on a snapshot of done, sampled flags equal collision_oracle on the present and
    considered rows, and obstacle_history and the outcome records equal the extended oracles;
  * a waiting vehicle's scripted obstacles keep to the loop's clock;
  * graph replay equals eager iteration;
  * leaving at the goal unblocks the exit lanes: far fewer vehicles still driving than when parking there.
"""
import math

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import episode_outcomes as EO
from oracle import right_of_way as RW
from oracle import scene_exchange as SX
from oracle import scene_lifetimes as SL

pytestmark = pytest.mark.gpu

K = 4
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
GEO = C.CarGeometry()
STEPS = 200
JUNCTION = (0.0, 0.0, 10.0)
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
    from junction_mpc.episodes import OUTCOME_INT, OUTCOME_NAMES, BatchedEpisodes
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
    return dict(torch=torch, cabi=_cabi, BatchedMPC=BatchedMPC, BatchedEpisodes=BatchedEpisodes, PI=PARAM_INDEX,
                names=OUTCOME_NAMES, ints=OUTCOME_INT, courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl))


def _scenes(jm, n_scenes, seed=7, forced=True):
    """n_scenes x K vehicles, vehicle j of a scene from approach j on a random route, 0-8 m along it at 2-5 m/s.
    forced: scene 0's last vehicle drives the doubling-back course (done = 2), every 16th scene's first vehicle starts
    above the QP's speed cap (failed solves)."""
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


class _Calls:
    """The engine's library with every call's name recorded; `before` / `after` hooks run around a named call."""
    def __init__(self, lib, hooks=None):
        self.lib, self.names, self.hooks = lib, [], hooks or {}

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.startswith("jmpc_"):
            return fn

        def call(*a):
            self.names.append(name)
            before, after = self.hooks.get(name, (None, None))
            if before:
                before()
            rc = fn(*a)
            if after:
                after()
            return rc
        return call


def _run_logged(engine, make, **run_kw):
    lib = engine._lib
    engine._lib = _Calls(lib)
    try:
        ep = make()
        res = ep.run(**run_kw)
        return ep, res, engine._lib.names
    finally:
        engine._lib = lib


def _same(a, b, names, history=True):
    for key in ("steps", "done", "state"):
        assert np.array_equal(a[key], b[key]), key
    if history:
        assert np.array_equal(a["history"], b["history"], equal_nan=True)
        assert np.array_equal(a["flags"], b["flags"])
    if "outcomes" in a:
        for n in names:
            assert np.array_equal(a["outcomes"][n], b["outcomes"][n]), n
    if "obstacle_history" in a:
        assert np.array_equal(a["obstacle_history"], b["obstacle_history"], equal_nan=True)


# ---- reductions ------------------------------------------------------------------------------------------------------

def test_defaults_are_todays_run(jm):
    from junction_mpc.episodes import scripted_obstacles
    engine, state0, cid, params = _scenes(jm, 64, seed=5)
    BE = jm["BatchedEpisodes"]
    B = len(state0)
    for k, extra in ((K, dict(right_of_way="first_come", junction=JUNCTION)), (1, dict())):
        kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS,
                  agents_per_scene=k, outcomes=True, record_obstacles=True, **extra)
        if k == 1:
            kw["obstacle_program"] = scripted_obstacles([SCENARIO_OBSTACLES] * B)
        runs = {}
        for key, life in (("before", dict()), ("none", dict(depart=None, on_goal="park")),
                          ("zeros", dict(depart=np.zeros(B, np.int64), on_goal="park"))):
            ep, res, names = _run_logged(engine, lambda: BE(engine, state0, **kw, **life), max_steps=STEPS)
            assert ep.depart is None and ep.presence is None
            runs[key] = (res, names)
        for key in ("none", "zeros"):
            assert runs[key][1] == runs["before"][1], (k, key)
            _same(runs["before"][0], runs[key][0], jm["names"])
        nm = runs["before"][1]
        assert not any(n.startswith("jmpc_scene_depart") or n in ("jmpc_scene_enter", "jmpc_scene_presence",
                                                                  "jmpc_episode_outcomes_scene") for n in nm)
    engine.close()


def test_one_departure_per_scene_shifts_the_scene(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=5)
    BE = jm["BatchedEpisodes"]
    B = len(state0)
    d_scene = np.random.default_rng(3).integers(0, 9, B // K)
    d_scene[:4] = [0, 3, 8, 1]
    depart = np.repeat(d_scene, K)
    dt = float(engine.default_params[jm["PI"]["dt"]])
    shifted = 0
    for on_goal, extra in (("park", dict()), ("leave", dict(right_of_way="first_come", junction=JUNCTION))):
        kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], agents_per_scene=K, outcomes=True,
                  on_goal=on_goal, **extra)
        ref = BE(engine, state0, max_steps=STEPS, **kw).run(max_steps=STEPS)
        got = BE(engine, state0, max_steps=STEPS + 8, depart=depart, **kw).run(max_steps=STEPS + 8)
        still = ref["done"] == 0                                   # cut off by max_steps: compare their first rows only
        for s in range(B // K):
            d, idx = int(d_scene[s]), slice(s * K, (s + 1) * K)
            h_ref, h_got = ref["history"][:, idx], got["history"][d:d + STEPS, idx]
            assert np.isnan(got["history"][:d, idx]).all()
            n = min(len(h_ref), len(h_got))
            keep = [c for c in range(8) if c != 4]
            assert np.array_equal(h_ref[:n][..., keep], h_got[:n][..., keep], equal_nan=True), (on_goal, s)
            np.testing.assert_allclose(h_got[:n][..., 4], h_ref[:n][..., 4] + d * dt, rtol=0, atol=1e-9)
            if still[idx].any():
                continue
            for key in ("steps", "done", "state"):
                assert np.array_equal(ref[key][idx], got[key][idx]), (on_goal, s, key)
            for name in jm["names"]:
                r, g = ref["outcomes"][name][idx], got["outcomes"][name][idx]
                if name.endswith("_eval"):
                    r = np.where(r >= 0, r + d, r)
                assert np.array_equal(r, g), (on_goal, s, name)
            shifted += d > 0
    print(f"\n[lifetimes: shift] {B // K} scenes, departures {np.bincount(d_scene).tolist()}: {shifted} shifted scenes "
          "equal their depart = 0 runs")
    assert shifted > 20
    engine.close()


# ---- stepped scenes against the oracle --------------------------------------------------------------------------------

def _assert_outcome(got, b, want, names, ints):
    for n in names:
        g, w = got[n][b], want[n]
        if n in ints:
            assert int(g) == int(w), (b, n, g, w)
        elif n == "min_clearance":
            assert (g == w) if math.isinf(w) else abs(g - w) <= 1e-12, (b, n, g, w)
        elif w == 0.0:
            assert abs(g) <= 1e-12, (b, n, g, w)
        else:
            assert abs(g - w) <= 1e-12 * abs(w), (b, n, g, w)


def test_stepped_scenes_with_lifetimes_against_the_oracle(jm):
    torch, PI, courses, WAITING = jm["torch"], jm["PI"], jm["courses"], jm["cabi"].WAITING
    engine, state0, cid, params = _scenes(jm, 1024, seed=7)
    B = len(state0)
    rng = np.random.default_rng(0)
    depart = np.where(rng.random(B) < 0.5, 0, rng.integers(1, 40, B))
    depart[:K] = [0, 0, 5, 0]                        # scene 0: its done = 2 vehicle stays parked for its mates
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=K, right_of_way="first_come", junction=JUNCTION,
                               depart=depart, on_goal="leave", outcomes=True, record_obstacles=True)
    dl = params[:, PI["dl"]]
    zone = ep.zone.cpu().numpy()
    snap = {}
    calls = {"n": 0}

    def before_row():
        torch.cuda.synchronize()
        snap.update(a=ep.agent_idx.cpu().numpy().copy(), done=ep.done.cpu().numpy().copy())

    def after_presence():
        calls["n"] += 1
        if calls["n"] % 2 == 1:                      # the first of the iteration: the collision mask
            torch.cuda.synchronize()
            snap["mask"] = ep.consider.cpu().numpy().copy()

    n = dict(waiting=0, entered=0, left=0, parked2=0, checked=0, absent_cut=0)
    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_right_of_way": (before_row, None), "jmpc_scene_presence": (None, after_presence)})
    try:
        ep._start()
        calls["n"] = 0                               # _start's evaluation mask
        rows = ep.scene_obs.cpu().numpy().copy()
        prev_done = ep.done.cpu().numpy().copy()
        assert ((prev_done == WAITING) == (depart > 0)).all()
        while ep.iteration < STEPS:
            i = ep.iteration
            prev_steps = ep.steps.cpu().numpy().copy()
            ep.iterate()
            a, done, mask = snap["a"], snap["done"], snap["mask"]
            # waiting exactly until the departure iteration; presence from the done codes of this instant
            assert np.array_equal(done == WAITING, depart > i), i
            present = (done != WAITING) & (done != 1)
            ref = (RW.consider_masks("first_come", K, a, done, dl, zone) & SL.presence_masks(present, K)).astype(np.int32)
            assert np.array_equal(mask, ref), i
            n["waiting"] += int((done == WAITING).sum())
            n["parked2"] += int(((done.reshape(-1, K) == 2).any(axis=1) & (done.reshape(-1, K) == 0).any(axis=1)).sum())
            n["left"] += int(((done.reshape(-1, K) == 1).any(axis=1) & (done.reshape(-1, K) == 0).any(axis=1)).sum())
            done_now = ep.done.cpu().numpy()
            n["entered"] += int(((prev_done == WAITING) & (done_now == 0)).sum())
            prev_done = done_now.copy()
            stepped = np.flatnonzero(ep.steps.cpu().numpy() > prev_steps)
            assert (depart[stepped] <= i).all()
            flag, clen = ep.flag.cpu().numpy(), ep.course_len.cpu().numpy()
            a_idx, v = ep.agent_idx.cpu().numpy(), ep.v.cpu().numpy()
            full = (1 << (K - 1)) - 1
            pres = SL.presence_masks(present, K)
            part = stepped[(pres[stepped] & full) != full]         # prefer vehicles with an absent mate
            pool = part if len(part) >= 3 else stepped
            for b in rng.choice(pool, min(3, len(pool)), replace=False):
                pr = params[b]
                kw = dict(dt=pr[PI["dt"]], frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                          max_speed=pr[PI["sim_max_speed"]], margin=ep.margin)
                f, cl = C.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]),
                                        RW.considered_rows(rows[b], mask[b]), **kw)
                assert (int(f), cl) == (int(flag[b]), int(clen[b])), (i, b)
                n["checked"] += 1
                rule_only = RW.consider_masks("first_come", K, a, done, dl, zone)[b]
                n["absent_cut"] += int(C.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]),
                                                       RW.considered_rows(rows[b], rule_only), **kw) != (f, cl))
            rows = ep.scene_obs.cpu().numpy().copy()
            if not ((done_now == 0) | (done_now == WAITING)).any():
                break
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)

    # obstacle_history: the oracle's mate rows where the mate is present, NaN where absent or outside b's lifetime
    oh, steps, done = res["obstacle_history"], res["steps"], res["done"]
    n_eval = len(oh)
    max_steer = params[:, PI["max_steer"]]
    mates = SL.mate_rows(state0, res["history"], steps, done, max_steer, K, n_eval, depart)
    pres = SL.presence(depart, steps, done, "leave", n_eval)
    slot_present = np.empty((n_eval, B, K - 1), bool)
    for b in range(B):
        s, j = divmod(b, K)
        slot_present[:, b] = pres[:, [s * K + m for m in range(K) if m != j]]
    e = np.arange(n_eval)[:, None]
    alive = (e >= depart[None, :]) & (e <= (depart + steps)[None, :]) & ~np.isin(done, SX.NEVER_STEPPED)[None, :]
    want = np.where((alive[..., None] & slot_present)[..., None], mates, np.nan)
    assert np.array_equal(oh, want, equal_nan=True)
    # the outcome records: the extended oracle on each vehicle's own evaluations
    dt, L = float(engine.default_params[PI["dt"]]), float(engine.default_params[PI["L"]])
    boundary = 0
    for b in range(B):
        if np.isin(done[b], SX.NEVER_STEPPED):
            continue
        d, m = int(depart[b]), int(steps[b])
        if done[b] == WAITING:
            assert m == 0 and d >= res["iterations"]
            continue
        track = oh[d:d + m + 1, b]
        h, f = res["history"][d:d + m, b], res["flags"][d:d + m, b]
        poses = np.vstack([[[state0[b, 0], state0[b, 1], state0[b, 3]]], h[:, :3]])
        clear, _ = EO.clearance_and_contact(poses, np.nan_to_num(track, nan=1e6), GEO)
        if (np.abs(clear) <= 1e-9).any():
            boundary += 1
            continue
        ref = SL.episode_outcomes(state0[b], h, f, track, dt=dt, L=L, max_steer=float(max_steer[b]), geo=GEO, first=d)
        _assert_outcome(res["outcomes"], b, ref, jm["names"], jm["ints"])
    print(f"\n[lifetimes: stepped] {B} vehicles, {ep.iteration} iterations: vehicle-iterations waiting {n['waiting']}, "
          f"entered {n['entered']}, scene-iterations with a mate gone {n['left']} / parked at done = 2 {n['parked2']}; "
          f"flags checked {n['checked']}, of which absence changed {n['absent_cut']}; outcome records on the boundary "
          f"{boundary}; done codes {np.bincount(done).tolist()}")
    assert n["waiting"] > 0 and n["entered"] == int((depart[:] > 0).sum() - (done == WAITING).sum())
    assert n["entered"] > 1000 and n["left"] > 0 and n["parked2"] > 0 and n["checked"] > 200
    assert n["absent_cut"] > 0 and boundary < B // 100
    assert done[K - 1] == 2 and (done == 1).any()
    engine.close()


# ---- extras keep the loop's clock --------------------------------------------------------------------------------------

def test_scripted_obstacles_of_a_waiting_vehicle_keep_the_clock(jm):
    from junction_mpc.episodes import scripted_obstacles
    engine, state0, cid, params = _scenes(jm, 16, seed=2, forced=False)
    B = len(state0)
    program = scripted_obstacles([SCENARIO_OBSTACLES] * B)
    kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS,
              obstacle_program=program, outcomes=True, record_obstacles=True)
    d = 12
    ref = jm["BatchedEpisodes"](engine, state0, **kw)
    got = jm["BatchedEpisodes"](engine, state0, depart=np.full(B, d), **kw)
    for _ in range(d):
        ref.iterate()
        got.iterate()
    assert np.array_equal(ref.obstacles.cpu().numpy(), got.obstacles.cpu().numpy())
    assert (got.steps.cpu().numpy() == 0).all() and (got.done.cpu().numpy() == 0).all()
    r, g = ref.run(max_steps=STEPS), got.run(max_steps=STEPS)
    # evaluation d: the entering vehicle sees what the depart = 0 vehicle sees then; before it nothing was recorded
    assert np.array_equal(g["obstacle_history"][d], r["obstacle_history"][d])
    assert np.isnan(g["obstacle_history"][:d]).all()
    assert (g["outcomes"]["min_clearance_eval"] >= d).all()
    engine.close()


# ---- graph replay -----------------------------------------------------------------------------------------------------

def test_graph_replay_equals_eager_iteration(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=9)
    B = len(state0)
    depart = np.random.default_rng(5).integers(0, 30, B)
    kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS, agents_per_scene=K,
              right_of_way="first_come", junction=JUNCTION, depart=depart, on_goal="leave", outcomes=True,
              record_obstacles=True)
    e = jm["BatchedEpisodes"](engine, state0, **kw).run(max_steps=STEPS)
    g = jm["BatchedEpisodes"](engine, state0, **kw).run(max_steps=STEPS, use_graph=True)
    n = min(e["iterations"], g["iterations"])
    for key in ("steps", "done", "state"):
        assert np.array_equal(e[key], g[key]), key
    assert np.array_equal(e["history"][:n], g["history"][:n], equal_nan=True)
    assert np.array_equal(e["obstacle_history"][:n + 1], g["obstacle_history"][:n + 1], equal_nan=True)
    for name in jm["names"]:
        assert np.array_equal(e["outcomes"][name], g["outcomes"][name]), name
    # no rule: presence alone is the collision mask
    kw.pop("right_of_way"), kw.pop("junction")
    e = jm["BatchedEpisodes"](engine, state0, **kw).run(max_steps=STEPS)
    g = jm["BatchedEpisodes"](engine, state0, **kw).run(max_steps=STEPS, use_graph=True)
    for key in ("steps", "done", "state"):
        assert np.array_equal(e[key], g[key]), key
    # the keyword checks on the device path
    BE = jm["BatchedEpisodes"]
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        BE(engine, state0, course_id=cid, on_goal="leave")
    with pytest.raises(ValueError, match=r"depart must be \["):
        BE(engine, state0, course_id=cid, agents_per_scene=K, depart=np.zeros(3, np.int32))
    engine.close()


# ---- leaving unblocks the exit lanes -----------------------------------------------------------------------------------

def test_leaving_at_the_goal_leaves_fewer_vehicles_driving(jm):
    engine, state0, cid, _ = _scenes(jm, 1024, seed=11, forced=False)
    still = {}
    for on_goal in ("park", "leave"):
        ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, frame_window=10, margin=jm["margin"], max_steps=400,
                                   record_history=False, outcomes=True, agents_per_scene=K, right_of_way="first_come",
                                   junction=JUNCTION, on_goal=on_goal)
        res = ep.run(max_steps=400)
        o = res["outcomes"]
        still[on_goal] = int((res["done"] == 0).sum())
        print(f"\n[lifetimes first_come + {on_goal}] {len(state0)} vehicles, 400 steps: still driving {still[on_goal]}, "
              f"contact {int((o['first_contact_eval'] >= 0).sum())}, within 3 m {int((o['min_clearance'] < 3.0).sum())}, "
              f"median steps to goal {float(np.median(res['steps'][res['done'] == 1]))}")
    assert still["leave"] * 10 <= still["park"]
    engine.close()
