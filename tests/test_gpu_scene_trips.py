"""Trips through scene slots (BatchedEpisodes.from_trips, jmpc_scene_trips, jmpc_scene_trips_finish).

Gates:
  * static reduction: one trip per slot, arriving at a departure iteration, is the lifetimes run with that depart and
    on_goal="leave", bit for bit (History, flags, steps, states, outcome records, obstacle_history), with and without
    first_come, with shared plans and with constant-input extras;
  * chain reduction: trips of k = 2 scenes that never overlap reuse slot 0, and each equals a fresh single-vehicle
    run of its course from its start state, bit for bit -- anything a slot keeps from its previous trip breaks this;
  * a dynamic Poisson run against the oracle: every pass's decisions against oracle.scene_trips.trips_pass on a
    snapshot taken where the pass runs, every collision mask against the rule oracle AND the presence reconstructed
    from the trip table, sampled flags against collision_oracle, and every trip's outcome record at the end;
  * graph replay equals eager iteration;
  * a trip whose planned course is unusable is closed with done = 3 and changes nothing for the others;
  * demand above capacity leaves trips pending with entry = -1 / WAITING and counts their waits;
  * runs without trips launch nothing new.
"""
import math

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import right_of_way as RW
from oracle import scene_lifetimes as SL
from oracle import scene_trips as ST

pytestmark = pytest.mark.gpu

K = 4
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
GEO = C.CarGeometry()
JUNCTION = (0.0, 0.0, 10.0)


@pytest.fixture(scope="module")
def jm(golden_dir):
    import __graft_entry__ as g
    g.build()
    import torch
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    from junction_mpc import episodes as E
    z = load_planner_golden(golden_dir)
    courses = []
    for row in ROUTES:
        for name in row:
            c = np.array(z[f"{name}/trajectory"], dtype=np.float64)
            synth.smooth_yaw_inplace(c[:, 2])
            courses.append(c)
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    return dict(torch=torch, cabi=_cabi, BatchedMPC=BatchedMPC, E=E, BE=E.BatchedEpisodes, PI=PARAM_INDEX,
                courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl))


def _routes(jm, speed=4.0):
    """poisson_trips routes: approach g, route r starts at course point 0."""
    cs = jm["courses"]
    return [[(3 * g + r, tuple(cs[3 * g + r][0, :3])) for r in range(3)] for g in range(4)], speed


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


# ---- reductions ------------------------------------------------------------------------------------------------------

def _static(jm, n_scenes, seed):
    """n_scenes x K vehicles, vehicle j of a scene from approach j on a random route, 0-8 m along it at 2-5 m/s, with
    departures in [0, 8) that do not decrease with j (so trips fill the slots in order)."""
    rng = np.random.default_rng(seed)
    courses = jm["courses"]
    B = n_scenes * K
    cid = (np.arange(B) % K) * 3 + rng.integers(0, 3, B)
    off = rng.integers(0, 96, B)
    state0 = np.array([[courses[c][o, 0], courses[c][o, 1], 0.0, courses[c][o, 2]] for c, o in zip(cid, off)])
    state0[:, 2] = rng.uniform(2, 5, B)
    depart = np.sort(rng.integers(0, 8, (n_scenes, K)), axis=1).reshape(-1)
    return state0, cid, depart


@pytest.mark.parametrize("variant", ["none", "first_come", "shared_plans", "extras"])
def test_one_trip_per_slot_is_the_lifetimes_run(jm, variant):
    n_scenes, steps = 128, 160
    state0, cid, depart = _static(jm, n_scenes, seed=3)
    B = len(state0)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=B)
    kw = dict(frame_window=10, margin=jm["margin"], max_steps=steps, agents_per_scene=K, outcomes=True,
              record_obstacles=True)
    if variant == "first_come":
        kw.update(right_of_way="first_come", junction=JUNCTION)
    if variant == "shared_plans":
        kw.update(share_plans=True, right_of_way="first_come", junction=JUNCTION)
    if variant == "extras":
        rng = np.random.default_rng(1)
        kw["obstacles"] = np.concatenate([rng.uniform(-30, 30, (B, 2, 2)), rng.uniform(0, 5, (B, 2, 1)),
                                          rng.uniform(-3, 3, (B, 2, 1)), np.zeros((B, 2, 2))], axis=2)
    ref = jm["BE"](engine, state0, course_id=cid, depart=depart, on_goal="leave", **kw).run(max_steps=steps)
    trips = jm["E"].Trips(np.arange(B) // K, depart, cid, state0)
    got = jm["BE"].from_trips(engine, trips, n_scenes, **kw).run(max_steps=steps)
    tab = got["trips"]
    assert np.array_equal(tab["entry"], depart) and np.array_equal(tab["slot"], np.arange(B))
    assert got["iterations"] == ref["iterations"]
    for key in ("steps", "state"):
        assert np.array_equal(got[key], ref[key]), key
    assert np.array_equal(tab["steps"], ref["steps"]) and np.array_equal(tab["done"], ref["done"])
    closed = (ref["done"] == 1) & (got["done"] == jm["cabi"].WAITING)
    assert np.array_equal(np.where(closed, 1, got["done"]), ref["done"])
    assert np.array_equal(got["history"], ref["history"], equal_nan=True)
    assert np.array_equal(got["flags"], ref["flags"])
    assert np.array_equal(got["obstacle_history"], ref["obstacle_history"], equal_nan=True)
    for n in jm["E"].OUTCOME_NAMES:
        assert np.array_equal(got["outcomes"][n], ref["outcomes"][n]), n
        assert np.array_equal(tab[n], ref["outcomes"][n]), n
    goal = tab["done"] == 1
    assert goal.sum() > B // 2 and np.array_equal(tab["exit"][goal], (tab["entry"] + tab["steps"])[goal])
    engine.close()


def test_a_slot_reused_by_a_chain_of_trips_is_a_fresh_vehicle_each_time(jm):
    n_scenes, per, gap = 64, 3, 250
    rng = np.random.default_rng(5)
    courses = jm["courses"]
    N = n_scenes * per
    cid = rng.integers(0, 12, N)
    off = rng.integers(0, 96, N)
    state0 = np.array([[courses[c][o, 0], courses[c][o, 1], 0.0, courses[c][o, 2]] for c, o in zip(cid, off)])
    state0[:, 2] = rng.uniform(2, 5, N)
    scene = np.repeat(np.arange(n_scenes), per)
    arrival = np.tile(np.arange(per) * gap, n_scenes) + rng.integers(0, 20, N)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=max(N, 2 * n_scenes))
    steps = per * gap + 40
    kw = dict(frame_window=10, margin=jm["margin"], max_steps=steps, outcomes=True, record_obstacles=True)
    got = jm["BE"].from_trips(engine, jm["E"].Trips(scene, arrival, cid, state0), n_scenes, agents_per_scene=2,
                              **kw).run(max_steps=steps)
    tab = got["trips"]
    assert (tab["done"] == 1).all()
    nxt = arrival.reshape(n_scenes, per)[:, 1:].reshape(-1)
    assert (tab["exit"].reshape(n_scenes, per)[:, :-1].reshape(-1) < nxt).all()     # never two trips at once
    assert np.array_equal(tab["slot"], 2 * scene) and np.array_equal(tab["entry"], arrival)
    ref = jm["BE"](engine, state0, course_id=cid, **{**kw, "record_obstacles": False}).run(max_steps=steps)
    dt = float(engine.default_params[jm["PI"]["dt"]])
    keep = [c for c in range(8) if c != 4]
    for t in range(N):
        e, n, b = int(tab["entry"][t]), int(tab["steps"][t]), int(tab["slot"][t])
        assert n == ref["steps"][t] and ref["done"][t] == 1, t
        h, r = got["history"][e:e + n, b], ref["history"][:n, t]
        assert np.array_equal(h[:, keep], r[:, keep], equal_nan=True), t
        np.testing.assert_allclose(h[:, 4], r[:, 4] + e * dt, rtol=0, atol=1e-9)
        assert np.array_equal(got["flags"][e:e + n, b], ref["flags"][:n, t]), t
        for name in jm["E"].OUTCOME_NAMES:
            w = ref["outcomes"][name][t]
            if name.endswith("_eval") and w >= 0:
                w = w + e
            assert tab[name][t] == w, (t, name)
    engine.close()


# ---- a dynamic run against the oracle ------------------------------------------------------------------------------

def _assert_outcome(got, t, want, names, ints):
    for n in names:
        g, w = got[n][t], want[n]
        if n in ints:
            assert int(g) == int(w), (t, n, g, w)
        elif n == "min_clearance":
            assert (g == w) if math.isinf(w) else abs(g - w) <= 1e-12, (t, n, g, w)
        elif w == 0.0:
            assert abs(g) <= 1e-12, (t, n, g, w)
        else:
            assert abs(g - w) <= 1e-12 * abs(w), (t, n, g, w)


def test_poisson_demand_against_the_oracle(jm):
    torch, PI, courses, E = jm["torch"], jm["PI"], jm["courses"], jm["E"]
    n_scenes, steps = 1024, 240
    routes, speed = _routes(jm)
    trips = E.poisson_trips(n_scenes, routes, 900.0, 0.2, steps - 40, speed, seed=2)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=n_scenes * K)
    B = n_scenes * K
    ep = jm["BE"].from_trips(engine, trips, n_scenes, agents_per_scene=K, frame_window=10, margin=jm["margin"],
                             max_steps=steps, right_of_way="first_come", junction=JUNCTION, outcomes=True,
                             record_obstacles=True)
    T = ep._trips
    order = ep._trip_order
    scene_start, arrival = T["scene_start"].cpu().numpy(), T["arrival"].cpu().numpy()
    usable, start = T["usable"].cpu().numpy(), T["start"].cpu().numpy()
    snap, masks = {}, []
    slot_waits = np.zeros(trips.n, np.int64)                  # the oracle's, in the scene-sorted layout
    calls = {"presence": 0}
    cnt = dict(pass_checks=0, admitted=0, blocked=0, slot_waits=0, flags=0)
    g = lambda x: x.cpu().numpy().copy()                                          # noqa: E731

    def before_pass():
        torch.cuda.synchronize()
        snap.update(done=g(ep.done), state=g(ep.state), slot_trip=g(T["slot_trip"]), phase=g(T["phase"]),
                    bw=g(T["blocked_waits"]), it=ep.iteration)

    def after_pass():
        torch.cuda.synchronize()
        initial = not ep._started
        want = ST.trips_pass(snap["done"], snap["state"], snap["slot_trip"], snap["phase"], scene_start, arrival,
                             usable, start, K, snap["it"], initial=initial, entry_gap=2.0, geo=GEO)
        assert np.array_equal(g(ep.done), want["done"]), snap["it"]
        assert np.array_equal(g(T["slot_trip"]), want["slot_trip"]), snap["it"]
        assert np.array_equal(g(T["phase"]), want["phase"]), snap["it"]
        bw = g(T["blocked_waits"]) - snap["bw"]
        assert sorted(np.flatnonzero(bw)) == want["blocked_waits"], snap["it"]
        slot_waits[want["slot_waits"]] += 1
        entry = g(T["entry"])
        for t, b in want["admitted"]:
            assert entry[t] == want["entry"] and g(T["slot"])[t] == b
        cnt["pass_checks"] += 1
        cnt["admitted"] += len(want["admitted"])
        cnt["blocked"] += len(want["blocked_waits"])
        cnt["slot_waits"] += len(want["slot_waits"])

    def before_row():
        torch.cuda.synchronize()
        snap.update(a=g(ep.agent_idx), rdone=g(ep.done), zone=g(ep.zone), dl=g(ep.params)[:, PI["dl"]],
                    cid=g(ep.course_id), rows=g(ep.scene_obs))

    def after_presence():
        if not ep._started:                          # _start's evaluation mask
            return
        calls["presence"] += 1
        if calls["presence"] % 2 == 1:               # the first of the iteration: the collision mask
            torch.cuda.synchronize()
            masks.append((snap["a"], snap["rdone"], snap["zone"], snap["dl"], g(ep.consider)))

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_scene_trips": (before_pass, after_pass), "jmpc_right_of_way": (before_row, None),
                               "jmpc_scene_presence": (None, after_presence)})
    rng = np.random.default_rng(0)
    try:
        snap["it"] = 0
        ep._start()
        while ep.iteration < steps and not ep._finished():
            prev = g(ep.steps)
            ep.iterate()
            stepped = np.flatnonzero(g(ep.steps) > prev)
            flag, clen, a_idx, v = g(ep.flag), g(ep.course_len), g(ep.agent_idx), g(ep.v)
            params = g(ep.params)
            for b in rng.choice(stepped, min(3, len(stepped)), replace=False):
                pr = params[b]
                kw = dict(dt=pr[PI["dt"]], frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                          max_speed=pr[PI["sim_max_speed"]], margin=ep.margin)
                f, cl = C.collision_cut(GEO, courses[snap["cid"][b]], int(a_idx[b]), float(v[b]),
                                        RW.considered_rows(snap["rows"][b], masks[-1][4][b]), **kw)
                assert (int(f), cl) == (int(flag[b]), int(clen[b])), (ep.iteration, b)
                cnt["flags"] += 1
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)
    tab = res["trips"]
    n_it = res["iterations"]
    # the collision masks: the rule's mask AND the presence the trip table gives for that iteration
    slot_s, entry_s, exit_s = (tab[n][order] for n in ("slot", "entry", "exit"))
    pres = ST.presence(slot_s, entry_s, exit_s, B, n_it, collision=True)
    for i, (a, done, zone, dl, mask) in enumerate(masks):
        ref = RW.consider_masks("first_come", K, a, done, dl, zone) & SL.presence_masks(pres[i], K)
        assert np.array_equal(mask, ref.astype(np.int32)), i
    back = np.empty_like(slot_waits)
    back[order] = slot_waits
    assert np.array_equal(tab["slot_waits"], back)
    # every trip's outcome record, and exit = entry + steps for the goal trips
    dt, L = float(engine.default_params[PI["dt"]]), float(engine.default_params[PI["L"]])
    max_steer = float(engine.default_params[PI["max_steer"]])
    goal = tab["done"] == 1
    assert np.array_equal(tab["exit"][goal], (tab["entry"] + tab["steps"])[goal])
    for t in np.flatnonzero(tab["entry"] >= 0):
        want = ST.trip_outcomes(trips.state[t], res["history"], res["flags"], res["obstacle_history"],
                                int(tab["slot"][t]), int(tab["entry"][t]), int(tab["steps"][t]), dt, L, max_steer, GEO)
        _assert_outcome(tab, t, want, E.OUTCOME_NAMES, E.OUTCOME_INT)
    print(f"\n[trips: poisson] {trips.n} trips in {n_scenes} scenes x {K}, {n_it} iterations: passes checked "
          f"{cnt['pass_checks']}, admitted {cnt['admitted']}, blocked waits {cnt['blocked']}, slot waits "
          f"{cnt['slot_waits']}, flags checked {cnt['flags']}; done codes {np.bincount(tab['done']).tolist()}")
    assert cnt["admitted"] > 2000 and cnt["blocked"] > 100 and cnt["slot_waits"] > 100 and cnt["flags"] > 200
    engine.close()


# ---- graph replay, overload, runs without trips ------------------------------------------------------------------------

def test_graph_replay_equals_eager_iteration(jm):
    E = jm["E"]
    routes, speed = _routes(jm)
    trips = E.poisson_trips(64, routes, 600.0, 0.2, 200, speed, seed=4)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=64 * K)
    kw = dict(agents_per_scene=K, frame_window=10, margin=jm["margin"], max_steps=240, right_of_way="first_come",
              junction=JUNCTION, outcomes=True, record_obstacles=True)
    e = jm["BE"].from_trips(engine, trips, 64, **kw).run(max_steps=240)
    g = jm["BE"].from_trips(engine, trips, 64, **kw).run(max_steps=240, use_graph=True)
    n = min(e["iterations"], g["iterations"])
    assert np.array_equal(e["history"][:n], g["history"][:n], equal_nan=True)
    assert np.array_equal(e["obstacle_history"][:n + 1], g["obstacle_history"][:n + 1], equal_nan=True)
    if e["iterations"] == g["iterations"]:
        for key in ("steps", "done", "state"):
            assert np.array_equal(e[key], g[key]), key
        for key, v in e["trips"].items():
            assert np.array_equal(v, g["trips"][key]), key
    engine.close()


def test_a_failed_plan_is_closed_without_a_slot(jm):
    import torch
    from junction_mpc.planner import DevicePlanBatch
    E, courses = jm["E"], jm["courses"]
    # the 12 recorded courses as found plans, and a 900-point course longer than max_N: course_ok = 0
    long = np.stack([np.arange(900) * 0.1, np.zeros(900), np.zeros(900)], axis=1)
    trajs = courses + [long]
    n, stride = len(trajs), max(len(t) for t in trajs)
    traj = np.zeros((n, stride, 3))
    for k, t in enumerate(trajs):
        traj[k, :len(t)] = t
    d = lambda a, dt: torch.as_tensor(a, dtype=dt, device="cuda")      # noqa: E731
    i = lambda: d(np.zeros(n), torch.int32)                             # noqa: E731
    plans = DevicePlanBatch(cost=d(np.zeros(n), torch.float64), status=i(), n_path=i(),
                            path=d(np.zeros((n, 2, 3)), torch.float64), path_mp=d(np.zeros((n, 2)), torch.int32),
                            n_traj=d([len(t) for t in trajs], torch.int32), traj=d(traj, torch.float64), expansions=i())
    engine = jm["BatchedMPC"].from_plans(plans, T=13, max_N=850, max_batch=64 * K)
    assert engine.course_ok.cpu().numpy().tolist() == [1] * 12 + [0]
    base = E.poisson_trips(64, [[(3 * g + r, None) for r in range(3)] for g in range(4)], 600.0, 0.2, 120, seed=8)
    bad_scene = np.array([0, 1, 5])
    with_bad = E.Trips(np.r_[base.scene, bad_scene], np.r_[base.arrival, [0, 3, 40]], np.r_[base.course_id, [12] * 3])
    kw = dict(agents_per_scene=K, plans=plans, frame_window=10, max_steps=160, right_of_way="first_come",
              junction=JUNCTION, outcomes=True)
    ref = jm["BE"].from_trips(engine, base, 64, **kw).run(max_steps=160)
    got = jm["BE"].from_trips(engine, with_bad, 64, **kw).run(max_steps=160)
    tg, tr = got["trips"], ref["trips"]
    assert (tg["done"][base.n:] == 3).all() and (tg["entry"][base.n:] == -1).all() and (tg["slot"][base.n:] == -1).all()
    for key, v in tr.items():
        assert np.array_equal(tg[key][:base.n], v, equal_nan=True), key
    for key in ("steps", "done", "state", "history", "flags"):
        assert np.array_equal(got[key], ref[key], equal_nan=True), key
    assert (tg["entry"][:base.n] >= 0).sum() > 500
    engine.close()


def test_demand_above_capacity_leaves_trips_pending(jm):
    E, WAITING = jm["E"], jm["cabi"].WAITING
    routes, speed = _routes(jm)
    steps = 120
    trips = E.poisson_trips(64, routes, 3600.0, 0.2, steps, speed, seed=6)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=64 * 2)
    res = jm["BE"].from_trips(engine, trips, 64, agents_per_scene=2, frame_window=10, margin=jm["margin"],
                              max_steps=steps, record_history=False, outcomes=True).run(max_steps=steps)
    tab = res["trips"]
    pending = tab["entry"] < 0
    assert res["iterations"] == steps and pending.sum() > trips.n // 4
    assert (tab["done"][pending] == WAITING).all() and (tab["slot"][pending] == -1).all()
    assert (tab["exit"][pending] == -1).all() and (tab["entry_delay"][pending] == -1).all()
    waits = tab["slot_waits"] + tab["blocked_waits"]
    # a trip arriving at a is due in the passes that admit entries a, a + 1, ..., steps (one per pass); it waits in
    # every one of them until the one that admits it
    assert np.array_equal(waits[pending], steps + 1 - trips.arrival[pending])
    admitted = ~pending & (tab["done"] != 3)
    assert np.array_equal(waits[admitted], tab["entry_delay"][admitted])
    assert (tab["slot_waits"] > 0).any() and (tab["blocked_waits"] > 0).any()
    engine.close()


def test_runs_without_trips_launch_nothing_new(jm):
    state0, cid, depart = _static(jm, 32, seed=1)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=len(state0))
    lib = engine._lib
    for extra in (dict(), dict(right_of_way="first_come", junction=JUNCTION, depart=depart, on_goal="leave")):
        engine._lib = _Calls(lib)
        try:
            ep = jm["BE"](engine, state0, course_id=cid, agents_per_scene=K, frame_window=10, margin=jm["margin"],
                          max_steps=60, outcomes=True, **extra)
            res = ep.run(max_steps=60)
            names = engine._lib.names
        finally:
            engine._lib = lib
        assert ep._trips is None and "trips" not in res
        assert not any(n.startswith("jmpc_scene_trips") for n in names)
    engine.close()
