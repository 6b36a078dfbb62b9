"""Fixed-time traffic signals (BatchedEpisodes(signals=...), jmpc_signals).

Gates:
  * reduction: a plan whose groups are always green is the run without signals, bit for bit -- k = 1 with scripted
    traffic, k = 4 with first_come and shared plans, and a trips run;
  * signals=None launches nothing new, and a plan adds exactly one launch per iteration;
  * a Poisson trips run (1 024 scenes x 4 slots, two-phase plan, first_come, mixed offsets) against
    oracle.signals.signal_pass at every iteration: course_len, latch and counters exactly, on a snapshot taken where
    the pass runs; no held vehicle reaches its zone entry while its group is red; the per-trip hold steps and GO passes
    add up to the per-slot counts;
  * a single vehicle under an always-red group stops before its stop line with course_len = max(a + 1, L) throughout;
  * graph replay equals eager iteration;
  * k = 1 without traffic (no collision check: the pass restores the full course itself) against the oracle at every
    iteration, through red and green phases;
  * plans the pass cannot run (a margin outside [0, max_N], an offset that is not one per scene) are refused.
"""
import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import signals as S

pytestmark = pytest.mark.gpu

K = 4
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
JUNCTION = (0.0, 0.0, 10.0)
PHASES = [0, 1, 0, 1]                  # approaches 1 and 3 (south, north) form group 0, approaches 2 and 4 group 1


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
                courses=courses, dl=dl, margin=C.cutoff_margin(C.CarGeometry(), dl))


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


def _routes(jm, speed=4.0):
    cs = jm["courses"]
    return [[(3 * g + r, tuple(cs[3 * g + r][0, :3])) for r in range(3)] for g in range(4)], speed


def _static(jm, B, seed, per_approach=True):
    """B vehicles, vehicle b from approach b % 4 (or any) on a random route, 0-8 m along it at 2-5 m/s."""
    rng = np.random.default_rng(seed)
    courses = jm["courses"]
    cid = ((np.arange(B) % K) * 3 + rng.integers(0, 3, B)) if per_approach else rng.integers(0, 12, B)
    off = rng.integers(0, 96, B)
    state0 = np.array([[courses[c][o, 0], courses[c][o, 1], 0.0, courses[c][o, 2]] for c, o in zip(cid, off)])
    state0[:, 2] = rng.uniform(2, 5, B)
    return state0, cid


def _same(got, ref, keys):
    for key in keys:
        if isinstance(ref[key], dict):
            for n, v in ref[key].items():
                assert np.array_equal(got[key][n], v, equal_nan=True), (key, n)
        else:
            assert np.array_equal(got[key], ref[key], equal_nan=True), key


# ---- reductions ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("variant", ["k1_scripted", "k4_first_come_shared", "trips"])
def test_always_green_is_the_run_without_signals(jm, variant):
    E, BE = jm["E"], jm["BE"]
    steps = 160
    rng = np.random.default_rng(11)
    green = E.SignalPlan(37, [(0, 37), (5, 37), (36, 37)], JUNCTION)
    kw = dict(frame_window=10, margin=jm["margin"], max_steps=steps, outcomes=True)
    if variant == "trips":
        n_scenes = 128
        routes, speed = _routes(jm)
        trips = E.poisson_trips(n_scenes, routes, 600.0, 0.2, steps - 20, speed, seed=9, groups=[0, 1, 2, -1])
        engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=n_scenes * K)
        kw.update(agents_per_scene=K, right_of_way="first_come", junction=JUNCTION, record_obstacles=True)
        plan = E.SignalPlan(37, [(0, 37), (5, 37), (36, 37)], JUNCTION, offset=rng.integers(-50, 50, n_scenes))
        ref = BE.from_trips(engine, E.Trips(trips.scene, trips.arrival, trips.course_id, trips.state), n_scenes,
                            **kw).run(max_steps=steps)
        got = BE.from_trips(engine, trips, n_scenes, signals=plan, **kw).run(max_steps=steps)
        for key, v in ref["trips"].items():
            assert np.array_equal(got["trips"][key], v, equal_nan=True), key
        assert (got["trips"]["signal_hold_steps"] == 0).all() and (got["trips"]["signal_go"] == 0).all()
        assert (got["trips"]["entry"] >= 0).sum() > 500
    else:
        B = 256
        if variant == "k1_scripted":
            state0, cid = _static(jm, B, seed=2, per_approach=False)
            specs = [[dict(kind="t_intersection", direction=1 if b % 2 else -1, turning=bool(b % 3 == 0),
                           speed=4.0 + (b % 5), offset=float(b % 7), dt=0.2)] for b in range(B)]
            kw.update(obstacle_program=E.scripted_obstacles(specs))
        else:
            state0, cid = _static(jm, B, seed=4)
            kw.update(agents_per_scene=K, share_plans=True, right_of_way="first_come", junction=JUNCTION,
                      record_obstacles=True)
            green = E.SignalPlan(37, [(0, 37), (5, 37), (36, 37)], JUNCTION, offset=rng.integers(-9, 9, B // K))
        engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=B)
        group = rng.integers(-1, 3, B)
        ref = BE(engine, state0, course_id=cid, **kw).run(max_steps=steps)
        got = BE(engine, state0, course_id=cid, signals=green, signal_group=group, **kw).run(max_steps=steps)
        assert (got["signal_hold_steps"] == 0).all() and (got["signal_go"] == 0).all()
    assert got["iterations"] == ref["iterations"]
    _same(got, ref, [k for k in ref if k not in ("trips",)])
    engine.close()


def test_launches_with_and_without_signals(jm):
    E, BE = jm["E"], jm["BE"]
    B = 128
    state0, cid = _static(jm, B, seed=1)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=B)
    lib = engine._lib
    kw = dict(course_id=cid, agents_per_scene=K, frame_window=10, margin=jm["margin"], max_steps=40, outcomes=True,
              right_of_way="first_come", junction=JUNCTION)
    per_iteration, names = {}, {}
    for name, extra in (("none", {}), ("plan", dict(signals=E.SignalPlan(30, [(0, 15), (15, 15)], JUNCTION),
                                                     signal_group=np.arange(B) % 2))):
        engine._lib = _Calls(lib)
        try:
            ep = BE(engine, state0, **kw, **extra)
            ep.iterate()
            n0 = engine.launch_count
            for _ in range(5):
                ep.iterate()
            per_iteration[name] = (engine.launch_count - n0) / 5
            names[name] = engine._lib.names
        finally:
            engine._lib = lib
    assert "jmpc_signals" not in names["none"] and ep.signals is not None
    assert per_iteration["plan"] == per_iteration["none"] + 1, per_iteration
    assert names["plan"].count("jmpc_signals") == 6
    engine.close()


# ---- a dynamic run against the oracle ------------------------------------------------------------------------------

def test_poisson_signals_against_the_oracle(jm):
    torch, PI, E = jm["torch"], jm["PI"], jm["E"]
    n_scenes, steps = 1024, 240
    routes, speed = _routes(jm)
    trips = E.poisson_trips(n_scenes, routes, 600.0, 0.2, steps - 40, speed, seed=5, groups=PHASES)
    rng = np.random.default_rng(3)
    plan = E.SignalPlan(60, [(0, 25), (30, 25)], JUNCTION, offset=rng.integers(-200, 200, n_scenes))
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=n_scenes * K)
    ep = jm["BE"].from_trips(engine, trips, n_scenes, agents_per_scene=K, frame_window=10, margin=jm["margin"],
                             max_steps=steps, right_of_way="first_come", junction=JUNCTION, signals=plan,
                             record_history=False, outcomes=True)
    course_n = np.asarray(engine.course_len)
    group, zone = ep.signal_group.cpu().numpy(), ep.signal_zone.cpu().numpy()
    g = lambda x: x.cpu().numpy().copy()                                          # noqa: E731
    snap = {}
    cnt = dict(passes=0, held=0, decided_hold=0, go=0)

    def before():
        torch.cuda.synchronize()
        snap.update(iteration=ep.iteration, cycle=plan.cycle, green_start=plan.green[:, 0], green_len=plan.green[:, 1],
                    margin=ep._signal_plan.margin, stop_decel=plan.stop_decel, k=K, offset=plan.offset,
                    owner=g(ep.signal_owner), group=group, zone=zone, course_id=g(ep.course_id), course_n=course_n,
                    agent_idx=g(ep.agent_idx), state=g(ep.state), dl=g(ep.params)[:, PI["dl"]], done=g(ep.done),
                    checked=True, course_len=g(ep.course_len), latch=g(ep.signal_latch), hold_steps=g(ep.signal_hold),
                    go=g(ep.signal_go), slot_hold=g(ep.signal_slot_hold), slot_go=g(ep.signal_slot_go))

    def after():
        torch.cuda.synchronize()
        it = snap["iteration"]
        course_len, latch, hold, go = S.signal_pass(snap)
        assert np.array_equal(g(ep.course_len), course_len), it
        assert np.array_equal(g(ep.signal_latch), latch), it
        assert np.array_equal(g(ep.signal_hold), hold), it
        assert np.array_equal(g(ep.signal_go), go), it
        run = snap["done"] == 0
        o = np.where(run, snap["owner"], 0)
        assert np.array_equal(g(ep.signal_slot_hold) - snap["slot_hold"],
                              np.where(run, (hold - snap["hold_steps"])[o], 0)), it
        assert np.array_equal(g(ep.signal_slot_go) - snap["slot_go"], np.where(run, (go - snap["go"])[o], 0)), it
        # a held vehicle (latch HOLD after the pass: its group is red now) has not reached its stop line
        held = run & (latch[:, 0] == o) & (latch[:, 1] == 1)
        assert (snap["agent_idx"][held] < zone[o[held], 0]).all(), it
        cnt["passes"] += 1
        cnt["held"] += int(held.sum())
        cnt["decided_hold"] += int((held & (snap["latch"][:, 0] != o)).sum())
        cnt["go"] += int((go - snap["go"]).sum())

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_signals": (before, after)})
    try:
        ep._start()
        while ep.iteration < steps and not ep._finished():
            ep.iterate()
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)
    tab = res["trips"]
    # the per-trip counts add up to the per-slot counts
    held_in = tab["slot"] >= 0
    B = n_scenes * K
    for col in ("signal_hold_steps", "signal_go"):
        per_slot = np.bincount(tab["slot"][held_in], weights=tab[col][held_in], minlength=B).astype(np.int64)
        assert np.array_equal(per_slot, res[col]), col
        assert (tab[col][~held_in] == 0).all(), col
    print(f"\n[signals: poisson] {trips.n} trips in {n_scenes} scenes x {K}, {res['iterations']} iterations: passes "
          f"checked {cnt['passes']}, held vehicle-steps {cnt['held']}, hold decisions {cnt['decided_hold']}, GO passes "
          f"{cnt['go']}, completed {(tab['done'] == 1).sum()}, contacts "
          f"{(tab['first_contact_eval'][tab['entry'] >= 0] >= 0).sum()}")
    assert cnt["passes"] == res["iterations"] and cnt["held"] > 10000 and cnt["decided_hold"] > 500
    assert cnt["go"] > 0
    engine.close()


def test_a_single_vehicle_stops_before_an_always_red_line(jm):
    torch, E, courses = jm["torch"], jm["E"], jm["courses"]
    B, steps = 12, 300
    state0 = np.array([[c[0, 0], c[0, 1], 4.0, c[0, 2]] for c in courses])
    plan = E.SignalPlan(10, [(0, 0)], JUNCTION)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=B)
    ep = jm["BE"](engine, state0, course_id=np.arange(B), frame_window=10, margin=jm["margin"], max_steps=steps,
                  outcomes=True, signals=plan, signal_group=np.zeros(B, np.int64))
    e = ep.signal_zone.cpu().numpy()[:, 0]
    L = e - jm["margin"]
    assert (e > 200).all() and (L > 0).all()
    seen = {"steps": 0}

    def after():
        torch.cuda.synchronize()
        run = ep.done.cpu().numpy() == 0
        a, cl = ep.agent_idx.cpu().numpy(), ep.course_len.cpu().numpy()
        assert np.array_equal(cl[run], np.maximum(a + 1, L)[run]), ep.iteration
        seen["steps"] += int(run.sum())

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_signals": (None, after)})
    try:
        res = ep.run(max_steps=steps)
    finally:
        engine._lib = lib
    a = ep.agent_idx.cpu().numpy()
    v = res["state"][:, 2]
    print(f"\n[signals: always red] final course index {a.tolist()} (stop lines {e.tolist()}, L {L.tolist()}), "
          f"speeds {np.round(v, 4).tolist()}, failed solves {res['outcomes']['failed_solves'].tolist()}, hold steps "
          f"{res['signal_hold_steps'].tolist()}, GO passes {res['signal_go'].tolist()}")
    assert seen["steps"] == B * steps and (res["done"] == 0).all()
    assert (a < e).all() and (np.abs(v) < 0.1).all()
    assert (res["signal_hold_steps"] == steps).all() and (res["signal_go"] == 0).all()
    engine.close()


def test_graph_replay_equals_eager_iteration(jm):
    E = jm["E"]
    routes, speed = _routes(jm)
    trips = E.poisson_trips(64, routes, 600.0, 0.2, 200, speed, seed=4, groups=PHASES)
    engine = jm["BatchedMPC"](jm["courses"], dl=jm["dl"], T=13, max_batch=64 * K)
    plan = E.SignalPlan(60, [(0, 25), (30, 25)], JUNCTION, offset=np.arange(64) * 7 - 100)
    kw = dict(agents_per_scene=K, frame_window=10, margin=jm["margin"], max_steps=240, right_of_way="first_come",
              junction=JUNCTION, outcomes=True, signals=plan)
    e = jm["BE"].from_trips(engine, trips, 64, **kw).run(max_steps=240)
    g = jm["BE"].from_trips(engine, trips, 64, **kw).run(max_steps=240, use_graph=True)
    n = min(e["iterations"], g["iterations"])
    assert np.array_equal(e["history"][:n], g["history"][:n], equal_nan=True)
    if e["iterations"] == g["iterations"]:
        for key in ("steps", "done", "state", "signal_hold_steps", "signal_go"):
            assert np.array_equal(e[key], g[key]), key
        for key, v in e["trips"].items():
            assert np.array_equal(v, g["trips"][key], equal_nan=True), key
    assert e["trips"]["signal_hold_steps"].sum() > 0
    engine.close()


def test_without_traffic_the_pass_restores_the_course_against_the_oracle(jm):
    # k = 1 and no obstacles: no collision check runs, so the pass itself writes the full course length every
    # iteration (checked = 0) before it cuts for red; green phases must give held vehicles their whole course back
    torch, E, PI, courses = jm["torch"], jm["E"], jm["PI"], jm["courses"]
    B, steps = 96, 200
    cid = np.arange(B) % 12
    state0 = np.array([[courses[c][0, 0], courses[c][0, 1], 4.0, courses[c][0, 2]] for c in cid])
    plan = E.SignalPlan(40, [(0, 15), (20, 15)], JUNCTION)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=B)
    ep = jm["BE"](engine, state0, course_id=cid, frame_window=10, margin=jm["margin"], max_steps=steps,
                  params=np.repeat(engine.default_params[None, :], B, axis=0), record_history=False,
                  signals=plan, signal_group=np.arange(B) % 3 - 1)
    course_n = np.asarray(engine.course_len)
    group, zone = ep.signal_group.cpu().numpy(), ep.signal_zone.cpu().numpy()
    g = lambda x: x.cpu().numpy().copy()                                          # noqa: E731
    snap, cnt = {}, dict(passes=0, restored=0, held=0)

    def before():
        torch.cuda.synchronize()
        snap.update(iteration=ep.iteration, cycle=plan.cycle, green_start=plan.green[:, 0], green_len=plan.green[:, 1],
                    margin=ep._signal_plan.margin, stop_decel=plan.stop_decel, k=1, offset=None, owner=None,
                    group=group, zone=zone, course_id=cid, course_n=course_n, agent_idx=g(ep.agent_idx),
                    state=g(ep.state), dl=g(ep.params)[:, PI["dl"]], done=g(ep.done), checked=False,
                    course_len=g(ep.course_len), latch=g(ep.signal_latch), hold_steps=g(ep.signal_hold),
                    go=g(ep.signal_go))

    def after():
        torch.cuda.synchronize()
        it = snap["iteration"]
        course_len, latch, hold, go = S.signal_pass(snap)
        assert np.array_equal(g(ep.course_len), course_len), it
        assert np.array_equal(g(ep.signal_latch), latch), it
        assert np.array_equal(g(ep.signal_hold), hold), it
        assert np.array_equal(g(ep.signal_go), go), it
        full = course_n[cid]
        cnt["passes"] += 1
        cnt["restored"] += int(((snap["course_len"] < full) & (course_len == full) & (snap["done"] == 0)).sum())
        cnt["held"] += int((hold - snap["hold_steps"]).sum())

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_signals": (before, after)})
    try:
        res = ep.run(max_steps=steps)
    finally:
        engine._lib = lib
    print(f"\n[signals: no traffic] {cnt['passes']} passes, {cnt['held']} held vehicle-steps, {cnt['restored']} "
          f"courses given back in full on green, done codes {np.bincount(res['done']).tolist()}")
    assert cnt["passes"] == res["iterations"] and cnt["held"] > 500 and cnt["restored"] >= 32
    engine.close()


def test_plans_the_pass_cannot_run_are_refused(jm):
    E, BE, courses = jm["E"], jm["BE"], jm["courses"]
    B = 8
    state0, cid = _static(jm, B, seed=0)
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=B)
    group = np.zeros(B, np.int64)
    with pytest.raises(ValueError, match="signal margin must be in"):
        BE(engine, state0, course_id=cid, signals=E.SignalPlan(30, [(0, 15)], JUNCTION, margin=engine.max_N + 1),
           signal_group=group)
    # from_trips: the pass reads offset[scene], so the offset must have one entry per scene
    trips = E.Trips([0, 1], [0, 0], [0, 3], state0[:2], group=[0, 0])
    with pytest.raises(ValueError, match=r"offset must be \[2\]"):
        BE.from_trips(engine, trips, 2, agents_per_scene=4, signals=E.SignalPlan(30, [(0, 15)], JUNCTION, offset=[0]))
    with pytest.raises(ValueError, match="signals must be a SignalPlan"):
        BE.from_trips(engine, trips, 2, agents_per_scene=4, signals=(30, [(0, 15)]))
    # the C entry point refuses a margin outside [0, max_N] with a message, before any launch
    ep = BE(engine, state0, course_id=cid, margin=jm["margin"], signals=E.SignalPlan(30, [(0, 15)], JUNCTION),
            signal_group=group)
    for m in (-1, engine.max_N + 1):
        ep._signal_plan.margin = m
        with pytest.raises(jm["cabi"].JmpcError, match=r"margin must be in \[0, max_N\]"):
            ep._signal_pass(True)
    engine.close()
