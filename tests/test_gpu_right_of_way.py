"""Right-of-way rules in scenes of MPC-driven vehicles (jmpc_collision_masked, jmpc_right_of_way_init,
jmpc_right_of_way, BatchedEpisodes(right_of_way=...)).

Gates:
  * the masked check is the unmasked one on the considered rows: jmpc_collision_masked equals jmpc_collision (and
    jmpc_collision_planned) run on the compacted rows and plans, bit for bit, on the synthetic config-3 / config-4
    workloads with random, all-zero and all-ones masks; the all-ones mask is the unmasked call; the skip mask holds;
    at the table limit (flag = -1 exit) a mask without a considered slot gives 0, any other mask -1;
  * the zone indices equal oracle/right_of_way.zone_indices on the recorded and on planned courses, -1 included;
  * scenes stepped with iterate() under both rules: every evaluation's mask equals oracle/right_of_way.consider_masks of
    a snapshot taken when the rule runs, and a sample of the flags equals collision_oracle on the considered rows;
  * the reductions: right_of_way=None is today's run, graph replay, outcomes on / off, shared plans, extras, planned
    scenes with a failed search;
  * the rule does its job: fewer vehicles still driving after 400 steps than without a rule.
"""
import ctypes

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import right_of_way as RW
from oracle import shared_plans as SP

pytestmark = pytest.mark.gpu

K = 4
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
GEO = C.CarGeometry()
STEPS = 200
JUNCTION = (0.0, 0.0, 10.0)            # every recorded intersection course enters it (right turns come within 7.24 m)
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
    # a course that doubles back 0.05 m beside itself, far from the junction: the index rule raises (done = 2 mid-run),
    # and it never enters the zone (entry = exit = -1)
    xs = np.concatenate([np.linspace(0, 20, 201), np.linspace(20, 10, 101)]) + 1000.0
    ys = np.concatenate([np.zeros(201), np.full(101, 0.05)]) + 1000.0
    courses.append(np.stack([xs, ys, np.zeros(302)], axis=1))
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    return dict(z=z, torch=torch, cabi=_cabi, synth=synth, BatchedMPC=BatchedMPC, BatchedEpisodes=BatchedEpisodes,
                PI=PARAM_INDEX, names=OUTCOME_NAMES, courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl))


def _scenes(jm, n_scenes, seed=7, forced=True):
    """tests/test_gpu_multi_agent.py's scenes: n_scenes x K vehicles, vehicle j of a scene from approach j on a random
    route, 0-8 m along it at 2-5 m/s.  forced: scene 0's last vehicle drives the doubling-back course (done = 2, never in
    the zone), every 16th scene's first vehicle starts above the QP's speed cap (failed solves)."""
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


# ---- the masked check ----------------------------------------------------------------------------------------------

def _device_collision(jm, engine, agent_idx, v, obst, fw, margin, plans=None, n_planned=0, consider=None, skip=None,
                      horizon_s=7.0):
    torch = jm["torch"]
    dev = torch.device("cuda", engine.device)
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)   # noqa: E731
    B = len(agent_idx)
    flag = torch.full((B,), -7, dtype=torch.int32, device=dev)
    clen = torch.full((B,), -7, dtype=torch.int32, device=dev)
    if skip is not None:
        skip = t(skip, torch.int32)
        engine.set_skip_mask(skip)
    try:
        engine.collision(t(agent_idx, torch.int32), t(v, torch.float64), t(obst, torch.float64), fw, margin, flag, clen,
                         plans=None if plans is None else t(plans, torch.float64), n_planned=n_planned,
                         consider=None if consider is None else t(consider, torch.int32), horizon_s=horizon_s)
        torch.cuda.synchronize(dev)
    finally:
        if skip is not None:
            engine.set_skip_mask(None)
    return flag.cpu().numpy(), clen.cpu().numpy()


def _near_workload(jm, config, B, seed=99, n_obs=None):
    """The synthetic workload with half of every obstacle slot moved next to the path, so that several slots cut.
    n_obs: that many obstacle slots (synth.make_obstacles) instead of the config's."""
    w = jm["synth"].make_workload(config, B=B)
    course = w["courses"][0]
    rng = np.random.default_rng(seed)
    if n_obs is not None:
        w["obstacles"] = jm["synth"].make_obstacles(rng, B, n_obs)
    for s in range(w["obstacles"].shape[1]):
        near = rng.random(B) < 0.5
        k = np.minimum(w["agent_idx"] + rng.integers(0, 200, B), len(course) - 1)
        w["obstacles"][near, s, 0] = course[k[near], 0] + rng.uniform(-8, 8, near.sum())
        w["obstacles"][near, s, 1] = course[k[near], 1] + rng.uniform(-8, 8, near.sum())
    return w


@pytest.mark.parametrize("config,n_slots", [(3, None), (4, None), (4, 8)], ids=["3", "4", "4-8slots"])
def test_masked_check_is_the_check_on_the_considered_rows(jm, config, n_slots):
    """n_slots = 8: every obstacle slot a scene can have, so that bit 7 and the (1 << n_obs) - 1 limit are used, with
    n_planned 4 and 8."""
    B = 4096
    w = _near_workload(jm, config, B, n_obs=n_slots)
    course, obst = w["courses"][0], w["obstacles"]
    n_obs = obst.shape[1]
    margin = C.cutoff_margin(GEO, w["dl"])
    fw = w["frame_window"]
    engine = jm["BatchedMPC"]([course], dl=w["dl"], T=13, max_batch=B)
    p, PI = engine.default_params, jm["PI"]
    rng = np.random.default_rng(config)
    v = w["state"][:, 2].copy()
    v[::17] = 30 / 3.6
    a_idx = w["agent_idx"]
    # random masks over the slots, random bits above them (never read), and the all-zero / all-ones masks
    mask = rng.integers(0, 1 << n_obs, B) | (rng.integers(0, 2, B) << n_obs) * rng.integers(1, 1 << 20, B)
    mask[::7] = 0
    mask[1::7] = -1
    mask = mask.astype(np.int32)
    # n_planned: the lower half of the slots, and with 8 slots also every slot
    planned = [max(1, n_obs // 2)] + ([n_obs] if n_obs == 8 else [])
    plans = np.stack([rng.uniform(p[PI["max_decel"]], p[PI["max_accel"]], (B, planned[-1], 12)),
                      rng.uniform(-p[PI["max_steer"]], p[PI["max_steer"]], (B, planned[-1], 12))], axis=-1)
    full = _device_collision(jm, engine, a_idx, v, obst, fw, margin)
    got = _device_collision(jm, engine, a_idx, v, obst, fw, margin, consider=mask)
    low = mask.astype(np.int64) & ((1 << n_obs) - 1)
    assert ((low >> (n_obs - 1)) & 1).any() and ((low >> (n_obs - 1)) & 1 == 0).any()
    changed = 0
    for n_planned in planned:
        pn = plans[:, :n_planned]
        full_planned = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pn, n_planned)
        got_planned = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pn, n_planned, consider=mask)
        for m in np.unique(low):
            idx = np.flatnonzero(low == m)
            keep = [s for s in range(n_obs) if (m >> s) & 1]
            if not keep:                                   # no considered slot: the n_obs = 0 result
                for g in (got, got_planned):
                    assert (g[0][idx] == 0).all() and (g[1][idx] == len(course)).all()
                continue
            ref = _device_collision(jm, engine, a_idx[idx], v[idx], obst[idx][:, keep], fw, margin)
            kp = [s for s in keep if s < n_planned]
            ref_p = _device_collision(jm, engine, a_idx[idx], v[idx], obst[idx][:, keep], fw, margin,
                                      plans[idx][:, kp] if kp else None, len(kp))
            for g, r in ((got, ref), (got_planned, ref_p)):
                assert np.array_equal(g[0][idx], r[0]) and np.array_equal(g[1][idx], r[1]), (config, m)
            changed += int(((got[0][idx] != full[0][idx]) | (got[1][idx] != full[1][idx])).sum())
        # the all-ones mask (and any mask with every slot's bit) is the unmasked call
        every = low == (1 << n_obs) - 1
        for g, r in ((got, full), (got_planned, full_planned)):
            assert np.array_equal(g[0][every], r[0][every]) and np.array_equal(g[1][every], r[1][every])
        all_ones = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pn, n_planned, consider=np.full(B, -1))
        assert np.array_equal(all_ones[0], full_planned[0]) and np.array_equal(all_ones[1], full_planned[1])
        # a spot check against the oracle on the considered rows
        for i in rng.choice(B, 24, replace=False):
            keep = [s for s in range(n_obs) if (int(mask[i]) >> s) & 1]
            f, cl = C.collision_cut(GEO, course, int(a_idx[i]), float(v[i]), RW.considered_rows(obst[i], mask[i]),
                                    dt=0.2, frame_window=fw, max_accel=p[PI["max_accel"]],
                                    max_speed=p[PI["sim_max_speed"]], margin=margin)
            assert (int(f), cl) == (int(got[0][i]), int(got[1][i])), i
            pl = [plans[i, s] if s < n_planned else None for s in keep]
            f, cl = SP.collision_cut(GEO, course, int(a_idx[i]), float(v[i]), RW.considered_rows(obst[i], mask[i]),
                                     dt=0.2, frame_window=fw, max_accel=p[PI["max_accel"]],
                                     max_speed=p[PI["sim_max_speed"]], margin=margin, plans=pl)
            assert (int(f), cl) == (int(got_planned[0][i]), int(got_planned[1][i])), i
        # the skip mask: skipped instances are left untouched
        skip = (rng.random(B) < 0.3).astype(np.int32)
        sk = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pn, n_planned, consider=mask, skip=skip)
        assert (sk[0][skip != 0] == -7).all() and (sk[1][skip != 0] == -7).all()
        assert np.array_equal(sk[0][skip == 0], got_planned[0][skip == 0])
        assert np.array_equal(sk[1][skip == 0], got_planned[1][skip == 0])
    print(f"\n[masked check] config {config}, n_obs {n_obs}, n_planned {planned}: {B} instances, "
          f"{len(np.unique(low))} distinct masks, the mask changed the flag or cut of {changed}; flagged unmasked / "
          f"masked {int((full[0] == 1).sum())} / {int((got[0] == 1).sum())}")
    assert changed > 0
    # argument errors of the new entry points
    cabi, lib, h = jm["cabi"], engine._lib, engine._h
    dummy = ctypes.c_void_p(1)             # never dereferenced: every call below fails its checks first
    args = lambda plans, n_planned, plan_len, consider: (h, 0, None, None, None, None, 2, plans, n_planned,  # noqa: E731
                                                         plan_len, consider, 10, 8, 7.0, None, None, None, None)
    for a, msg in ((args(dummy, 3, 4, dummy), r"n_planned must be in \[0, n_obs\]"),
                   (args(dummy, 1, 0, dummy), "plan_len must be >= 1"), (args(None, 1, 4, dummy), "plans is NULL"),
                   (args(None, 0, 1, None), "consider is NULL"),
                   (args(None, 0, 1, dummy), "jmpc_collision_masked: NULL array")):
        with pytest.raises(cabi.JmpcError, match=msg):
            cabi.check(lib.jmpc_collision_masked(*a), "jmpc_collision_masked")
    with pytest.raises(cabi.JmpcError, match=r"k in \[2, 9\]"):
        cabi.check(lib.jmpc_right_of_way(h, 8, 1, 1, *([dummy] * 7)), "jmpc_right_of_way")
    with pytest.raises(cabi.JmpcError, match=r"k in \[2, 9\]"):
        cabi.check(lib.jmpc_right_of_way(h, 20, 10, 1, *([dummy] * 7)), "jmpc_right_of_way")
    with pytest.raises(cabi.JmpcError, match="unknown rule"):
        cabi.check(lib.jmpc_right_of_way(h, 8, 4, 0, *([dummy] * 7)), "jmpc_right_of_way")
    with pytest.raises(cabi.JmpcError, match="needs priority"):
        cabi.check(lib.jmpc_right_of_way(h, 8, 4, 1, dummy, dummy, None, dummy, None, dummy, None), "jmpc_right_of_way")
    with pytest.raises(cabi.JmpcError, match="needs zone"):
        cabi.check(lib.jmpc_right_of_way(h, 8, 4, 2, dummy, dummy, None, None, dummy, dummy, None), "jmpc_right_of_way")
    with pytest.raises(cabi.JmpcError, match="n_junction must be 1 or B / k"):
        cabi.check(lib.jmpc_right_of_way_init(h, 8, 4, None, dummy, 3, dummy, None), "jmpc_right_of_way_init")
    engine.close()


@pytest.mark.parametrize("config", [3, 4])
def test_masked_check_at_the_table_limit(jm, config):
    """A horizon beyond the kernel's obstacle-prediction table (more than kMaxObsFrames - 1 = 71 steps of dt = 0.2)
    takes the flag = -1 exit.  There a mask without a considered slot must still give the n_obs = 0 result (flag 0,
    full length), and any other mask the unmasked -1."""
    B = 256
    w = _near_workload(jm, config, B)
    course, obst = w["courses"][0], w["obstacles"]
    n_obs = obst.shape[1]
    margin = C.cutoff_margin(GEO, w["dl"])
    engine = jm["BatchedMPC"]([course], dl=w["dl"], T=13, max_batch=B)
    p, PI = engine.default_params, jm["PI"]
    assert 15.0 > 71 * p[PI["dt"]]
    rng = np.random.default_rng(config + 10)
    # zero, one slot, all but one slot, all ones; zero low bits with high bits set (never read)
    kinds = np.array([0, 1, (1 << n_obs) - 2, -1, 1 << n_obs])
    mask = kinds[np.arange(B) % len(kinds)].astype(np.int32)
    plans = np.stack([np.zeros((B, 1, 12)), rng.uniform(-0.3, 0.3, (B, 1, 12))], axis=-1)
    a_idx, v = w["agent_idx"], w["state"][:, 2]
    fw = w["frame_window"]
    none = (mask.astype(np.int64) & ((1 << n_obs) - 1)) == 0
    for pl, npl in ((None, 0), (plans, 1)):
        ref = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pl, npl, horizon_s=15.0)
        assert (ref[0] == -1).all() and (ref[1] == len(course)).all()
        got = _device_collision(jm, engine, a_idx, v, obst, fw, margin, pl, npl, consider=mask, horizon_s=15.0)
        assert (got[0][none] == 0).all() and (got[0][~none] == -1).all(), np.unique(got[0])
        assert (got[1] == len(course)).all()
    assert none.sum() > 0 and (~none).sum() > 0
    engine.close()


# ---- zone indices ----------------------------------------------------------------------------------------------------

def test_zone_indices_on_the_recorded_courses(jm):
    courses = jm["courses"]
    torch = jm["torch"]
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=64)
    n = len(courses)
    cid = np.tile(np.arange(n), 4)[:4 * n]                  # 4 * 13 episodes = 13 scenes of 4
    B = len(cid)
    state0 = np.zeros((B, 4))
    # one zone for all scenes, and one per scene (centres and radii that some courses miss: -1)
    rng = np.random.default_rng(2)
    per_scene = np.stack([rng.uniform(-6, 6, B // K), rng.uniform(-6, 6, B // K), rng.uniform(0.5, 12, B // K)], axis=1)
    got_none = 0
    for junction in (JUNCTION, per_scene):
        ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, agents_per_scene=K, right_of_way="first_come",
                                   junction=junction, record_history=False)
        torch.cuda.synchronize()
        zone = ep.zone.cpu().numpy()
        J = np.broadcast_to(np.asarray(junction, np.float64).reshape(-1, 3), (B // K, 3))
        for b in range(B):
            assert tuple(zone[b]) == RW.zone_indices(courses[cid[b]], J[b // K]), (b, cid[b])
        got_none += int((zone[:, 0] < 0).sum())
        if junction is JUNCTION:
            # every intersection course enters r = 10 m; the doubling-back course does not
            assert (zone[cid < n - 1, 0] >= 0).all() and (zone[cid == n - 1] == -1).all()
    assert got_none > B // n
    engine.close()


# ---- stepped scenes against the oracle ------------------------------------------------------------------------------

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


def _step_and_check(jm, ep, engine, cid, params, rule, steps=STEPS, sample=3, seed=0):
    """Steps `ep` with iterate(), checking every evaluation's consider mask against the oracle on a snapshot of
    agent_idx / done taken when jmpc_right_of_way runs, and a sample of the stepped vehicles' flags against
    collision_oracle on the considered rows.  Returns run()'s result and counters of the cases met."""
    torch, PI, courses = jm["torch"], jm["PI"], jm["courses"]
    rng = np.random.default_rng(seed)
    dl = params[:, PI["dl"]]
    zone = None if ep.zone is None else ep.zone.cpu().numpy()
    prio = None if ep.priority is None else ep.priority.cpu().numpy()
    snap = {}
    n = dict(evals=0, parked=0, ignored=0, committed=0, approaching=0, outside=0, ties=0, checked=0, cut_ignored=0)
    B = ep.B

    def before():
        torch.cuda.synchronize()
        snap.update(a=ep.agent_idx.cpu().numpy().copy(), done=ep.done.cpu().numpy().copy())

    def after():
        torch.cuda.synchronize()
        snap["mask"] = ep.consider.cpu().numpy().copy()

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_right_of_way": (before, after)})
    try:
        ep._start()
        rows = ep.scene_obs.cpu().numpy().copy()
        while ep.iteration < steps:
            prev_steps = ep.steps.cpu().numpy().copy()
            ep.iterate()
            a, done, mask = snap["a"], snap["done"], snap["mask"]
            ref = RW.consider_masks(rule, K, a, done, dl, zone, prio)
            assert np.array_equal(mask, ref), ep.iteration
            n["evals"] += 1
            moving = done == 0
            cls, key = RW.scene_keys(rule, a, dl, zone, prio)
            n["committed"] += int((moving & (cls == 0)).sum())
            n["approaching"] += int((moving & (cls == 1)).sum())
            n["outside"] += int((moving & (cls == 2)).sum())
            d = done.reshape(-1, K)
            n["parked"] += int(((d != 0).any(axis=1) & (d == 0).any(axis=1)).sum())
            n["ignored"] += int((moving & ((mask & ((1 << (K - 1)) - 1)) != (1 << (K - 1)) - 1)).sum())
            c, kk = cls.reshape(-1, K), key.reshape(-1, K)
            mv = moving.reshape(-1, K)
            for i in range(K):
                for j in range(i + 1, K):
                    n["ties"] += int((mv[:, i] & mv[:, j] & (c[:, i] == c[:, j]) & (kk[:, i] == kk[:, j])).sum())
            steps_now = ep.steps.cpu().numpy()
            stepped = np.flatnonzero(steps_now > prev_steps)
            flag, clen = ep.flag.cpu().numpy(), ep.course_len.cpu().numpy()
            a_idx, v = ep.agent_idx.cpu().numpy(), ep.v.cpu().numpy()
            # prefer vehicles that ignore a mate, so that the masked slots are exercised
            part = stepped[(mask[stepped] & ((1 << (K - 1)) - 1)) != (1 << (K - 1)) - 1]
            pool = part if len(part) >= sample else stepped
            for b in rng.choice(pool, min(sample, len(pool)), replace=False):
                pr = params[b]
                f, cl = C.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]),
                                        RW.considered_rows(rows[b], mask[b]), dt=pr[PI["dt"]],
                                        frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                                        max_speed=pr[PI["sim_max_speed"]], margin=ep.margin)
                assert (int(f), cl) == (int(flag[b]), int(clen[b])), (ep.iteration, b)
                full = C.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]), rows[b], dt=pr[PI["dt"]],
                                       frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                                       max_speed=pr[PI["sim_max_speed"]], margin=ep.margin)
                n["cut_ignored"] += int(full != (f, cl))
                n["checked"] += 1
            rows = ep.scene_obs.cpu().numpy().copy()
            if (ep.done.cpu().numpy() != 0).all():
                break
    finally:
        engine._lib = lib
    return ep.run(max_steps=ep.iteration), n


@pytest.mark.parametrize("rule", ["first_come", "fixed"])
def test_stepped_scenes_against_the_oracle(jm, rule):
    engine, state0, cid, params = _scenes(jm, 4096, seed=7)
    B = len(state0)
    kw = dict(junction=JUNCTION) if rule == "first_come" else \
        dict(priority=np.random.default_rng(4).integers(0, 3, B).astype(np.float64))     # many ties
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=K, right_of_way=rule, record_history=False,
                               outcomes=True, **kw)
    res, n = _step_and_check(jm, ep, engine, cid, params, rule, steps=120)
    print(f"\n[right of way {rule}] {B} vehicles, {n['evals']} evaluations: scene-evaluations with a parked mate "
          f"{n['parked']}, vehicle-evaluations committed / approaching / outside the zone {n['committed']} / "
          f"{n['approaching']} / {n['outside']}, ignoring a mate {n['ignored']}, ties {n['ties']}; flags checked "
          f"{n['checked']}, of which the mask changed {n['cut_ignored']}; done codes {np.bincount(res['done']).tolist()}")
    assert n["parked"] > 0 and n["ignored"] > 0 and n["ties"] > 0 and n["checked"] > 200 and n["cut_ignored"] > 0
    if rule == "first_come":
        assert n["committed"] > 0 and n["approaching"] > 0 and n["outside"] > 0
    assert res["done"][K - 1] == 2 and (res["done"] == 1).any()
    engine.close()


# ---- reductions ------------------------------------------------------------------------------------------------------

def test_reductions(jm):
    engine, state0, cid, params = _scenes(jm, 64, seed=5)
    BE = jm["BatchedEpisodes"]
    kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS, agents_per_scene=K)
    runs, names = {}, {}
    for key, extra in (("before", dict()), ("none", dict(right_of_way=None)),
                       ("fc", dict(right_of_way="first_come", junction=JUNCTION)),
                       ("fc_outcomes", dict(right_of_way="first_come", junction=JUNCTION, outcomes=True,
                                            record_obstacles=True)),
                       ("fixed", dict(right_of_way="fixed"))):
        lib = engine._lib
        engine._lib = _Calls(lib)
        try:
            ep = BE(engine, state0, **kw, **extra)
            runs[key] = ep.run(max_steps=STEPS)
            names[key] = engine._lib.names
        finally:
            engine._lib = lib
        assert (ep.consider is None) == ("right_of_way" not in extra or extra["right_of_way"] is None)
    # right_of_way=None: the same library calls in the same order as without the option, and the same episodes
    assert names["none"] == names["before"]
    assert not any(n.startswith("jmpc_right_of_way") or n == "jmpc_collision_masked" for n in names["none"])
    _same_episodes(runs["before"], runs["none"], jm["names"])
    # a rule: the zones once (first_come only), then per iteration the rule right after the goal test and before the
    # masked check, which replaces jmpc_collision
    for key in ("fc", "fixed"):
        nm, it = names[key], runs[key]["iterations"]
        assert nm.count("jmpc_right_of_way_init") == (1 if key == "fc" else 0)
        assert nm.count("jmpc_right_of_way") == nm.count("jmpc_collision_masked") == it
        assert "jmpc_collision" not in nm
        pre = [i for i, n in enumerate(nm) if n == "jmpc_episode_pre"]
        for i, n in enumerate(nm):
            if n == "jmpc_right_of_way":
                assert nm[i - 1] == "jmpc_episode_pre" and nm[i + 1] == "jmpc_collision_masked"
        assert len(pre) == it + 1
    _same_episodes(runs["fc"], runs["fc_outcomes"], jm["names"])
    # the rule changes the runs
    a, b = runs["none"], runs["fc"]
    n = min(len(a["history"]), len(b["history"]))
    differ = ~np.all((a["history"][:n] == b["history"][:n]) | (np.isnan(a["history"][:n]) & np.isnan(b["history"][:n])),
                     axis=(0, 2))
    print(f"\n[right of way reductions] {len(state0)} vehicles: {int(differ.sum())} drive differently with first_come; "
          f"still driving none / first_come / fixed {int((a['done'] == 0).sum())} / {int((b['done'] == 0).sum())} / "
          f"{int((runs['fixed']['done'] == 0).sum())}")
    assert differ.sum() > 0
    # graph replay equals eager iteration
    g = BE(engine, state0, **kw, right_of_way="first_come", junction=JUNCTION, outcomes=True,
           record_obstacles=True).run(max_steps=STEPS, use_graph=True)
    e = runs["fc_outcomes"]
    _same_episodes(e, g, jm["names"])
    rows = int(e["steps"].max()) + 1
    assert np.array_equal(e["obstacle_history"][:rows], g["obstacle_history"][:rows], equal_nan=True)
    _same_episodes(runs["fixed"], BE(engine, state0, **kw, right_of_way="fixed").run(max_steps=STEPS, use_graph=True),
                   jm["names"])
    # the keyword checks on the device path
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        BE(engine, state0, course_id=cid, right_of_way="fixed")
    with pytest.raises(ValueError, match="needs junction"):
        BE(engine, state0, course_id=cid, agents_per_scene=K, right_of_way="first_come")
    with pytest.raises(ValueError, match=r"priority must be \["):
        BE(engine, state0, course_id=cid, agents_per_scene=K, right_of_way="fixed", priority=np.zeros(3))
    engine.close()


def test_with_shared_plans_and_extras(jm):
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
    torch, PI = jm["torch"], jm["PI"]
    # shared plans: the mask checked against the oracle each iteration, sampled flags against the planned oracle
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, obstacles=obst.copy(), frame_window=10,
                               margin=jm["margin"], max_steps=STEPS, agents_per_scene=K, share_plans=True,
                               right_of_way="first_come", junction=JUNCTION, outcomes=True, record_obstacles=True)
    assert ep.n_obs == K - 1 + 2
    dl = params[:, PI["dl"]]
    zone = ep.zone.cpu().numpy()
    snap = {}

    def before():
        torch.cuda.synchronize()
        snap.update(a=ep.agent_idx.cpu().numpy().copy(), done=ep.done.cpu().numpy().copy())

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_right_of_way": (before, None)})
    checked = ignored = 0
    try:
        ep._start()
        rows, plans = ep.scene_obs.cpu().numpy().copy(), ep.scene_plans.cpu().numpy().copy()
        while ep.iteration < STEPS:
            prev_steps = ep.steps.cpu().numpy().copy()
            ep.iterate()
            mask = ep.consider.cpu().numpy()
            assert np.array_equal(mask, RW.consider_masks("first_come", K, snap["a"], snap["done"], dl, zone))
            # the extras' bits are always set
            assert (((mask.astype(np.int64) >> (K - 1)) & 3) == 3).all()
            ignored += int(((mask & 7) != 7).sum())
            stepped = np.flatnonzero(ep.steps.cpu().numpy() > prev_steps)
            flag, clen = ep.flag.cpu().numpy(), ep.course_len.cpu().numpy()
            a_idx, v = ep.agent_idx.cpu().numpy(), ep.v.cpu().numpy()
            for b in rng.choice(stepped, min(3, len(stepped)), replace=False):
                keep = [s for s in range(ep.n_obs) if (int(mask[b]) >> s) & 1]
                pr = params[b]
                pl = [plans[b, s] if s < K - 1 else None for s in keep]
                f, cl = SP.collision_cut(GEO, jm["courses"][cid[b]], int(a_idx[b]), float(v[b]), rows[b][keep],
                                         dt=pr[PI["dt"]], frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                                         max_speed=pr[PI["sim_max_speed"]], margin=ep.margin, plans=pl)
                assert (int(f), cl) == (int(flag[b]), int(clen[b])), (ep.iteration, b)
                checked += 1
            rows, plans = ep.scene_obs.cpu().numpy().copy(), ep.scene_plans.cpu().numpy().copy()
            if (ep.done.cpu().numpy() != 0).all():
                break
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)
    print(f"\n[right of way + shared plans + extras] {checked} flags checked, {ignored} vehicle-evaluations ignore a mate; "
          f"done codes {np.bincount(res['done']).tolist()}")
    assert checked > 50 and ignored > 0
    assert (res["outcomes"]["min_clearance_obs"] >= K - 1).any()
    engine.close()


def test_planned_scenes_with_a_failed_search(jm):
    z = jm["z"]
    torch = jm["torch"]
    from junction_mpc import planner as P
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
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
    names = [n for s in scenes for n in s]
    # the zone indices on the planned courses, with a zone per scene that one course misses
    junction = np.array([JUNCTION, JUNCTION, (500.0, 500.0, 2.0)])
    plans = planner.plan_device(**inputs(names), max_expansions=8192, max_path=32)
    engine = BatchedMPC.from_plans(plans, T=13, max_batch=16)
    ep = BatchedEpisodes.from_plans(engine, plans, frame_window=10, agents_per_scene=K, right_of_way="first_come",
                                    junction=junction)
    torch.cuda.synchronize()
    zone, done = ep.zone.cpu().numpy(), ep.done.cpu().numpy()
    courses = engine.get_courses()
    for b in range(len(names)):
        if done[b] != 3:
            assert tuple(zone[b]) == RW.zone_indices(courses[b], junction[b // K]), b
    assert (zone[8:] == -1).all() and (zone[:4, 0] >= 0).all()
    engine.close()
    for rule, extra in (("first_come", dict(junction=JUNCTION)), ("fixed", dict())):
        kw = dict(frame_window=10, T=13, max_steps=160, max_expansions=8192, max_path=32, planner=planner, outcomes=True,
                  agents_per_scene=K, share_plans=True, right_of_way=rule, **extra)
        res = run_planned_scenarios(**inputs(names), obstacles=[SCENARIO_OBSTACLES] * 3, **kw)
        assert res["plan_status"][7] != P.STATUS_FOUND
        assert res["done"][4:8].tolist() == [4, 4, 4, 3] and (res["steps"][4:8] == 0).all()
        assert (res["steps"][[0, 1, 2, 3, 8, 9, 10, 11]] > 0).all()
        names2 = scenes[0] + scenes[2]
        ref = run_planned_scenarios(**inputs(names2), obstacles=[SCENARIO_OBSTACLES] * 2, **kw)
        keep = [0, 1, 2, 3, 8, 9, 10, 11]
        for key in ("steps", "done", "state"):
            assert np.array_equal(res[key][keep], ref[key]), (rule, key)
        n = min(len(res["history"]), len(ref["history"]))
        assert np.array_equal(res["history"][:n][:, keep], ref["history"][:n], equal_nan=True)
        for name in jm["names"]:
            assert np.array_equal(res["outcomes"][name][keep], ref["outcomes"][name]), (rule, name)
    planner.close()


# ---- the rule does its job -------------------------------------------------------------------------------------------

def test_rules_leave_fewer_vehicles_waiting(jm):
    engine, state0, cid, _ = _scenes(jm, 1024, seed=11, forced=False)
    still = {}
    for rule, kw in ((None, {}), ("first_come", dict(junction=JUNCTION)), ("fixed", {})):
        ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, frame_window=10, margin=jm["margin"], max_steps=400,
                                   record_history=False, outcomes=True, agents_per_scene=K, right_of_way=rule, **kw)
        res = ep.run(max_steps=400)
        o = res["outcomes"]
        still[rule] = int((res["done"] == 0).sum())
        print(f"\n[right of way {rule}] {len(state0)} vehicles, 400 steps: still driving {still[rule]}, contact "
              f"{int((o['first_contact_eval'] >= 0).sum())}, within 3 m {int((o['min_clearance'] < 3.0).sum())}, "
              f"median steps to goal {float(np.median(res['steps'][res['done'] == 1]))}")
    assert still["first_come"] < still[None] and still["fixed"] < still[None]
    engine.close()
