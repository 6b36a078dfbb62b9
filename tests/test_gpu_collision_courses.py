"""Collision kernel on many courses against the oracle, on both of its arc-length paths.

A course gets an arc-length table while the handle's 256 MB budget lasts; for the others the kernel sums the arc
lengths on the fly.  Here the course set is larger than the budget, instances are spread over every course by
course_id, parameters come per instance, and the kernel's shape limits are hit at their edges.  Flags and cut
lengths are integers defined bit for bit by oracle/collision_oracle.py, so every check is exact.  The same course
set then feeds a multi-course step against the step oracle, and planned courses in three copies (most of the third
without a table) feed closed-loop episodes against the loop run on the CPU."""
import math
import os
from multiprocessing import get_context

import numpy as np
import pytest

from helpers import compare_step, load_planner_golden, oracle_batch, params_from_vector
from oracle import collision_oracle as C
from oracle import mpc_oracle as O

pytestmark = pytest.mark.gpu

GEO = C.CarGeometry()
DS = 0.083                                  # point spacing of the planned courses
MARGIN = C.cutoff_margin(GEO, DS)           # 72
MAX_EGO, MAX_OBS_STEPS = 160, 71            # flag = -1 beyond these (include/jmpc.h)
ARC_CAP = (256 << 20) // 8                  # doubles of arc-length tables per handle
SHORT = (1, 2, 31, 32, 33, 64, 65)          # ballot-loop edges


def _procs():
    return min(32, os.cpu_count() or 1)


def _need(n):
    return n * (n + 1) // 2


def _long_course(n, seed, x0=0.0, y0=0.0):
    """Straights and arcs (radius >= 12 m) with a continuous yaw.  The spacing swings between 0.6 and 1.4 DS along the
    course: on the planned courses every segment is DS long, so an arc-length sum over the wrong segments would go
    unnoticed there."""
    rng = np.random.default_rng(seed)
    curv = np.zeros(n)
    k = 0
    while k < n:
        seg = int(rng.integers(150, 600))
        curv[k:k + seg] = 0.0 if rng.random() < 0.4 else rng.uniform(-1 / 12, 1 / 12)
        k += seg
    ds = DS * (1.0 + 0.4 * np.sin(2 * np.pi * np.arange(n) / rng.uniform(60, 240) + rng.uniform(0, 2 * np.pi)))
    yaw = rng.uniform(-np.pi, np.pi) + np.concatenate([[0.0], np.cumsum(curv[1:] * ds[1:])])
    x = x0 + np.concatenate([[0.0], np.cumsum(ds[1:] * np.cos(yaw[:-1]))])
    y = y0 + np.concatenate([[0.0], np.cumsum(ds[1:] * np.sin(yaw[:-1]))])
    return np.stack([x, y, yaw], axis=1)


def _shifted(c, k):
    d = c.copy()
    d[:, 0] += 100.0 * k
    d[:, 1] -= 50.0 * k
    return d


# ---- oracle in a fork pool -------------------------------------------------------------------------------
_COURSES = None


def _expect_one(job):
    """(flag, course length) the kernel must report: the oracle's, or (-1, N) past the kernel's table sizes."""
    cid, a0, v, obs, dt, fw, max_accel, max_speed, margin, horizon = job
    course = _COURSES[cid]
    if (len(C.ego_prediction(course[a0:], v, dt, max_accel, max_speed)) > MAX_EGO
            or len(np.arange(0, horizon, dt)) > MAX_OBS_STEPS):
        return -1, len(course)
    f, n = C.collision_cut(GEO, course, a0, v, obs, dt=dt, frame_window=fw, max_accel=max_accel, max_speed=max_speed,
                           margin=margin, horizon=horizon)
    return int(f), int(n)


def _expect(courses, jobs):
    global _COURSES
    _COURSES = courses
    if len(jobs) < 16 or _procs() == 1:
        return np.array([_expect_one(j) for j in jobs]).reshape(-1, 2)
    with get_context("fork").Pool(_procs()) as pool:
        return np.array(pool.map(_expect_one, jobs, chunksize=max(1, len(jobs) // (4 * _procs())))).reshape(-1, 2)


def _cpu_episode_job(job):
    return _cpu_episode(*job)


def _obstacles(rng, courses, cid, a0, n_obs, near):
    """Obstacles scattered around the ego; where `near`, the first one sits next to the path ahead."""
    B = len(cid)
    obs = np.zeros((B, n_obs, 6))
    for b in range(B):
        c = courses[cid[b]]
        obs[b, :, :2] = c[a0[b], :2] + rng.uniform(-35, 35, (n_obs, 2))
        if near[b]:
            k = min(a0[b] + int(rng.integers(0, 200)), len(c) - 1)
            obs[b, 0, :2] = c[k, :2] + rng.uniform(-8, 8, 2)
    obs[:, :, 2] = rng.uniform(0, 30 / 3.6, (B, n_obs))
    obs[:, :, 3] = rng.uniform(-np.pi, np.pi, (B, n_obs))
    obs[:, :, 5] = rng.uniform(-0.4, 0.4, (B, n_obs))
    return obs


def _jobs(cid, a0, v, obs, params, fw, margin, horizon, PI):
    return [(int(cid[b]), int(a0[b]), float(v[b]), obs[b], float(params[b, PI["dt"]]), fw, float(params[b, PI["max_accel"]]),
             float(params[b, PI["sim_max_speed"]]), margin, horizon) for b in range(len(cid))]


# ---- fixtures --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def jm():
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    return synth, BatchedMPC, PARAM_INDEX


@pytest.fixture(scope="module")
def recorded(jm, golden_dir):
    synth = jm[0]
    z = load_planner_golden(golden_dir)
    out = []
    for n in z["variants"]:
        t = np.array(z[f"{n}/trajectory"], dtype=np.float64)
        if len(t):
            synth.smooth_yaw_inplace(t[:, 2])
            out.append(t)
    assert len(out) == 51
    return out


@pytest.fixture(scope="module")
def course_set(jm, recorded):
    """Short courses, one long course, the recorded and synthetic courses and translated copies of them, then two
    more long courses, placed in this order: about 1.5x the arc-table budget."""
    synth, BatchedMPC, PI = jm
    base = recorded + [synth.load_course(n) for n in ("intersection", "roundabout", "multilane")]
    longs = [_long_course(n, 40 + k, 500.0 * k, -300.0 * k) for k, n in enumerate((3300, 2500, 4000))]
    bend = _long_course(200, 7, -900.0, 900.0)
    shorts = [bend[20:20 + n].copy() for n in SHORT]
    courses = shorts + longs[:1] + list(base)
    k = 1
    while sum(_need(len(c)) for c in courses + longs[1:] + base) <= 1.6 * ARC_CAP:
        courses += [_shifted(c, k) for c in base]
        k += 1
    courses += longs[1:]
    kind = (["short"] * len(shorts) + ["long"] + ["planned"] * len(base) + ["copy"] * (len(courses) - len(shorts) - 3 - len(base))
            + ["long"] * 2)
    mpc = BatchedMPC(courses, dl=DS, T=13, max_batch=8192)
    has = mpc.arc_table_flags()
    assert has.shape == (len(courses),)
    assert has.any() and not has.all()
    return dict(courses=courses, kind=np.array(kind), has=has, mpc=mpc)


@pytest.fixture(scope="module")
def many(jm, course_set):
    """4096 instances over every course, half of them on courses without a table; device results (host entry point) and
    the oracle's, for every instance."""
    synth, BatchedMPC, PI = jm
    courses, mpc, has = course_set["courses"], course_set["mpc"], course_set["has"]
    rng = np.random.default_rng(2024)
    B = 4096
    rest = B - len(courses)
    cid = np.concatenate([np.arange(len(courses)), rng.choice(np.flatnonzero(has), rest // 2),
                          rng.choice(np.flatnonzero(~has), rest - rest // 2)]).astype(np.int32)
    a0 = np.array([rng.integers(0, len(courses[c])) for c in cid], dtype=np.int32)
    v = rng.uniform(0, 30 / 3.6, B)
    v[::13] = 30 / 3.6
    obs = _obstacles(rng, courses, cid, a0, 2, rng.random(B) < 0.5)
    params = np.repeat(mpc.default_params[None, :], B, axis=0)
    flag, clen = mpc.collision_host(a0, v, obs, frame_window=20, margin=MARGIN, course_id=cid, params=params)
    want = _expect(courses, _jobs(cid, a0, v, obs, params, 20, MARGIN, 7.0, PI))
    return dict(cid=cid, a0=a0, v=v, obs=obs, params=params, flag=flag, clen=clen, want=want)


# ---- 1. many courses, both arc paths ---------------------------------------------------------------------
def test_many_courses_both_arc_paths_match_oracle(course_set, many):
    has = course_set["has"][many["cid"]]
    bad = np.flatnonzero((many["flag"] != many["want"][:, 0]) | (many["clen"] != many["want"][:, 1]))
    assert len(bad) == 0, [(int(b), int(many["cid"][b]), bool(has[b]), many["flag"][b], many["clen"][b],
                            tuple(many["want"][b])) for b in bad[:10]]
    for group in (has, ~has):
        assert group.sum() >= 500
        hit = many["flag"][group] == 1
        assert 0.05 < hit.mean() < 0.95
    assert len(np.unique(many["cid"])) == len(course_set["courses"])


# ---- 2. table path and on-the-fly path give identical bits ------------------------------------------------
def test_table_and_on_the_fly_arc_paths_agree(jm, recorded):
    synth, BatchedMPC, PI = jm
    smallest = min(_need(len(c)) for c in recorded)
    fillers, left = [], ARC_CAP
    while left >= smallest:
        n = min(4000, int((math.sqrt(8 * left + 1) - 1) / 2))
        fillers.append(_long_course(n, 100 + len(fillers)))
        left -= _need(n)
    a = BatchedMPC(recorded, dl=DS, T=13, max_batch=4096)
    b = BatchedMPC(fillers + recorded, dl=DS, T=13, max_batch=4096)
    assert a.arc_table_flags().all()
    hb = b.arc_table_flags()
    assert hb[:len(fillers)].all() and not hb[len(fillers):].any()
    rng = np.random.default_rng(5)
    B = 4096
    cid = rng.integers(0, len(recorded), B).astype(np.int32)
    a0 = np.array([rng.integers(0, len(recorded[c])) for c in cid], dtype=np.int32)
    v = rng.uniform(0, 30 / 3.6, B)
    v[::11] = 30 / 3.6
    obs = _obstacles(rng, recorded, cid, a0, 3, rng.random(B) < 0.6)
    fa, la = a.collision_host(a0, v, obs, frame_window=20, margin=MARGIN, course_id=cid)
    fb, lb = b.collision_host(a0, v, obs, frame_window=20, margin=MARGIN, course_id=cid + len(fillers))
    assert np.array_equal(fa, fb) and np.array_equal(la, lb)
    assert 0.05 < (fa == 1).mean() < 0.95
    a.close()
    b.close()


# ---- 3. parameter and shape grid -------------------------------------------------------------------------
@pytest.mark.parametrize("n_obs", [1, 3, 8])
def test_parameter_and_shape_grid(jm, course_set, n_obs):
    synth, BatchedMPC, PI = jm
    courses, mpc, kind = course_set["courses"], course_set["mpc"], course_set["kind"]
    pool = np.flatnonzero((kind == "planned") | (kind == "copy"))
    rng = np.random.default_rng(300 + n_obs)
    base = mpc.default_params
    ms0 = float(base[PI["sim_max_speed"]])
    rows, vs = [], []
    for dt in (0.1, 0.2, 0.25):
        for acc in (2.0, 1.0, 0.35):                    # 0.35: the sequential cumsum branch
            for ms in (ms0, 5.0):
                for v in (0.0, np.nextafter(ms, 0.0), ms, ms + 1.0):
                    p = base.copy()
                    p[PI["dt"]], p[PI["max_accel"]], p[PI["sim_max_speed"]] = dt, acc, ms
                    rows.append(p)
                    vs.append(v)
    params, v = np.array(rows), np.array(vs)
    B = len(v)
    checked = 0
    for fw in (0, 1, 15, 16, 32):
        for horizon in (3.5, 7.0):
            cid = rng.choice(pool, B).astype(np.int32)
            a0 = np.array([rng.integers(0, len(courses[c]) - 1) for c in cid], dtype=np.int32)
            obs = _obstacles(rng, courses, cid, a0, n_obs, rng.random(B) < 0.7)
            flag, clen = mpc.collision_host(a0, v, obs, frame_window=fw, margin=MARGIN, course_id=cid, params=params,
                                            horizon_s=horizon)
            want = _expect(courses, _jobs(cid, a0, v, obs, params, fw, MARGIN, horizon, PI))
            assert np.array_equal(flag, want[:, 0]), (fw, horizon, np.flatnonzero(flag != want[:, 0])[:10])
            assert np.array_equal(clen, want[:, 1]), (fw, horizon, np.flatnonzero(clen != want[:, 1])[:10])
            checked += (flag == 1).sum()
    assert checked > 0


# ---- 4. the documented limits, at their edges ------------------------------------------------------------
def test_table_limits_at_their_edges(jm, course_set):
    synth, BatchedMPC, PI = jm
    courses, mpc, kind, has = course_set["courses"], course_set["mpc"], course_set["kind"], course_set["has"]
    base = mpc.default_params
    ms = float(base[PI["sim_max_speed"]])
    cases = []                                          # (course, agent_idx, v, dt) keeping 159 .. 162 ego points
    for c in np.flatnonzero(kind == "long"):
        path = courses[c]
        for dt in (0.1, 0.2):
            for v in (0.0, ms):
                # from the last point back, starting where ~140 points are kept
                rest = np.cumsum(np.hypot(*np.diff(path[::-1, :2], axis=0).T))
                for a in range(len(path) - 1 - int(np.searchsorted(rest, 140 * dt * ms)), -1, -1):
                    n = len(C.ego_prediction(path[a:], v, dt, 2.0, ms))
                    if 159 <= n <= 162 and sum(k[2:] == (v, dt, n) for k in cases if k[0] == c) < 3:
                        cases.append((c, a, v, dt, n))
                    if n > 162:
                        break
    counts = {n for *_, n in cases}
    assert {160, 161} <= counts
    assert {bool(has[c]) for c, *_ in cases} == {True, False}
    cid = np.array([k[0] for k in cases], np.int32)
    a0 = np.array([k[1] for k in cases], np.int32)
    v = np.array([k[2] for k in cases])
    params = np.repeat(base[None, :], len(cases), axis=0)
    params[:, PI["dt"]] = [k[3] for k in cases]
    n_ego = np.array([k[4] for k in cases])
    rng = np.random.default_rng(4)
    obs = _obstacles(rng, courses, cid, a0, 2, np.ones(len(cases), bool))
    seen = set()
    for horizon in (7.0, 7.1, 7.2, 14.2, 14.4):        # dt 0.1: 70 / 71 / 72 obstacle steps; dt 0.2: 71 / 72
        flag, clen = mpc.collision_host(a0, v, obs, frame_window=10, margin=MARGIN, course_id=cid, params=params,
                                        horizon_s=horizon)
        want = _expect(courses, _jobs(cid, a0, v, obs, params, 10, MARGIN, horizon, PI))
        assert np.array_equal(flag, want[:, 0]) and np.array_equal(clen, want[:, 1]), horizon
        steps = np.array([len(np.arange(0, horizon, dt)) for dt in params[:, PI["dt"]]])
        over = (n_ego > MAX_EGO) | (steps > MAX_OBS_STEPS)
        assert np.array_equal(flag == -1, over)
        assert (clen[over] == [len(courses[c]) for c in cid[over]]).all()
        seen |= {(int(e), int(s), bool(f)) for e, s, f in zip(n_ego, steps, over)}
    assert (160, 71, False) in seen and (161, 71, True) in seen and (160, 72, True) in seen


# ---- 5. index edges --------------------------------------------------------------------------------------
@pytest.mark.parametrize("margin", [0, MARGIN])
def test_index_edges_on_short_courses(jm, course_set, margin):
    synth, BatchedMPC, PI = jm
    courses, mpc, kind = course_set["courses"], course_set["mpc"], course_set["kind"]
    rows = []
    for c in np.flatnonzero(kind == "short"):
        N = len(courses[c])
        for a in sorted({0, max(N - 2, 0), N - 1}):
            rows.append((c, a))
    cid = np.array([r[0] for r in rows] * 3, np.int32)
    a0 = np.array([r[1] for r in rows] * 3, np.int32)
    B = len(cid)
    n = len(rows)
    rng = np.random.default_rng(11 + margin)
    v = np.concatenate([np.zeros(n), rng.uniform(0, 8, n), np.full(n, 30 / 3.6)])
    obs = _obstacles(rng, courses, cid, a0, 2, np.ones(B, bool))
    on_top = np.arange(B) < n
    for b in np.flatnonzero(on_top):                    # a standing car on the ego's pose
        x, y, yaw = courses[cid[b]][a0[b]]
        obs[b, 0] = (x, y, 0.0, yaw, 0.0, 0.0)
    params = np.repeat(mpc.default_params[None, :], B, axis=0)
    flag, clen = mpc.collision_host(a0, v, obs, frame_window=10, margin=margin, course_id=cid, params=params)
    want = _expect(courses, _jobs(cid, a0, v, obs, params, 10, margin, 7.0, PI))
    assert np.array_equal(flag, want[:, 0]) and np.array_equal(clen, want[:, 1])
    assert (flag[on_top] == 1).all() and (clen[on_top] == a0[on_top] + 1).all()


# ---- 6. skip mask on the device entry point -----------------------------------------------------------------
def test_skip_mask_on_device_entry_point(course_set, many):
    import torch
    mpc = course_set["mpc"]
    B = len(many["cid"])
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")     # noqa: E731
    skip = (np.random.default_rng(6).random(B) < 0.3).astype(np.int32)
    d_skip = t(skip, torch.int32)
    flag = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    clen = torch.full((B,), -9, dtype=torch.int32, device="cuda")
    mpc.set_skip_mask(d_skip)
    try:
        mpc.collision(t(many["a0"], torch.int32), t(many["v"], torch.float64), t(many["obs"], torch.float64), 20, MARGIN,
                      flag, clen, course_id=t(many["cid"], torch.int32), params=t(many["params"], torch.float64))
        torch.cuda.synchronize()
    finally:
        mpc.set_skip_mask(None)
    f, n = flag.cpu().numpy(), clen.cpu().numpy()
    s = skip != 0
    assert (f[s] == -7).all() and (n[s] == -9).all()
    assert np.array_equal(f[~s], many["flag"][~s]) and np.array_equal(n[~s], many["clen"][~s])


# ---- long courses: warps per block ------------------------------------------------------------------------
@pytest.mark.parametrize("N,n_courses,n_obs", [(6000, 2, 2), (6000, 2, 8), (20000, 1, 8)])
def test_long_courses_without_table_match_oracle(jm, N, n_courses, n_obs):
    """Courses too long for 4 warps per block of the on-the-fly arc scan (2 warps at 6 000 points, 1 at 20 000)."""
    synth, BatchedMPC, PI = jm
    first = _long_course(N, 60 + n_obs)
    courses = [first, _shifted(first, 3)][:n_courses]
    mpc = BatchedMPC(courses, dl=DS, T=13, max_batch=1024)
    assert mpc.arc_table_flags().tolist() == ([True, False] if N == 6000 else [False])
    rng = np.random.default_rng(N + n_obs)
    B = 192
    cid = rng.integers(0, n_courses, B).astype(np.int32)
    a0 = np.where(rng.random(B) < 0.85, rng.integers(N - 3000, N, B), rng.integers(0, N, B)).astype(np.int32)
    v = rng.uniform(0, 30 / 3.6, B)
    obs = _obstacles(rng, courses, cid, a0, n_obs, rng.random(B) < 0.6)
    params = np.repeat(mpc.default_params[None, :], B, axis=0)
    flag, clen = mpc.collision_host(a0, v, obs, frame_window=20, margin=MARGIN, course_id=cid, params=params)
    want = _expect(courses, _jobs(cid, a0, v, obs, params, 20, MARGIN, 7.0, PI))
    assert np.array_equal(flag, want[:, 0]) and np.array_equal(clen, want[:, 1])
    assert (flag == 1).any() and (flag == 0).any()
    mpc.close()


def test_course_too_long_for_one_warp_is_an_error(jm):
    synth, BatchedMPC, PI = jm
    from junction_mpc._cabi import JmpcError
    N = 30000                                           # one warp would need 242 880 bytes at one obstacle
    mpc = BatchedMPC([_long_course(N, 3)], dl=DS, T=13, max_batch=64)
    assert not mpc.arc_table_flags()[0]
    before = mpc.launch_count
    flag, clen = np.full(4, -7, np.int32), np.full(4, -9, np.int32)
    with pytest.raises(JmpcError, match="too long for the shared-memory arc scan"):
        mpc.collision_host(np.full(4, N - 100, np.int32), np.ones(4), np.zeros((4, 1, 6)), frame_window=10, margin=MARGIN,
                           out=(flag, clen))
    assert mpc.launch_count == before
    assert (flag == -7).all() and (clen == -9).all()
    mpc.close()


# ---- multi-course step against the oracle -------------------------------------------------------------------
def test_multi_course_step_matches_oracle(jm, course_set, many):
    synth, BatchedMPC, PI = jm
    courses, mpc, kind = course_set["courses"], course_set["mpc"], course_set["kind"]
    rng = np.random.default_rng(21)
    usable = np.isin(kind[many["cid"]], ["planned", "copy"]) & (many["a0"] < np.array([len(courses[c]) for c in many["cid"]]) - 5)
    idx = rng.choice(np.flatnonzero(usable), 320, replace=False)
    cid, a0 = many["cid"][idx], many["a0"][idx]
    assert len(np.unique(cid)) >= 40 and (kind[cid] == "copy").any()
    B, T = len(idx), 13
    pts = np.array([courses[c][a] for c, a in zip(cid, a0)])
    state = np.stack([pts[:, 0] + rng.uniform(-0.5, 0.5, B), pts[:, 1] + rng.uniform(-0.5, 0.5, B), many["v"][idx],
                      pts[:, 2] + rng.uniform(-0.1, 0.1, B)], axis=1)
    oa = rng.uniform(-1.0, 2.0, (B, T))
    od = np.clip(np.cumsum(rng.uniform(-0.05, 0.05, (B, T)), axis=1), -0.7, 0.7)
    params = np.repeat(mpc.default_params[None, :], B, axis=0)
    params[:, PI["dl"]] = [math.hypot(*(courses[c][0, :2] - courses[c][1, :2])) for c in cid]
    w = dict(T=T, courses=courses, course_id=cid, state=state, oa=oa, od=od, target_ind=np.maximum(a0 - 3, 0).astype(np.int32),
             course_len=many["clen"][idx], params=params, dl=DS)
    assert (w["course_len"] < [len(courses[c]) for c in cid]).any()
    out = mpc.step_host(w["state"], w["target_ind"], oa, od, course_id=cid, course_len=w["course_len"], params=params)
    refs = oracle_batch(w, range(B))
    worst = compare_step(out, refs, range(B))
    assert worst <= 1.0
    assert (out.status == O.STATUS_OPTIMAL).sum() >= B // 2


# ---- multi-course closed-loop episodes against the CPU loop -------------------------------------------------
def _cpu_episode(course, p, state0, obstacles, fw, margin, max_steps):
    """The scenario loop with constant-input obstacles, on the CPU with the oracle's functions (test_gpu_episodes.py),
    for one episode with its own course and Params."""
    st = tuple(state0)
    obs = [list(o) for o in obstacles]
    agent, tmp_len, target, oa, od, di = 0, None, 0, None, None, 0.0
    n_full = len(course)
    log = []
    for i in range(max_steps):
        d = np.hypot(st[0] - course[-1, 0], st[1] - course[-1, 1])
        cur_len = n_full if tmp_len is None else tmp_len
        if d <= p.goal_dis and abs(target - cur_len) < 5 and abs(st[2]) <= p.stop_speed:
            break
        if tmp_len is None or np.any(course[min(agent, tmp_len - 1)] != course[tmp_len - 1]):
            agent = O.nearest_index_forward(st[0], st[1], course[:, 0], course[:, 1], agent)
        flag, cut = C.collision_cut(GEO, course, agent, st[2], obs, dt=p.dt, frame_window=fw, max_accel=p.max_accel,
                                    max_speed=p.sim_max_speed, margin=margin)
        tmp_len = cut
        r = O.mpc_step(p, st, oa, od, course[:cut, 0], course[:cut, 1], course[:cut, 2], target)
        target = r.target_ind
        if r.oa is not None:
            oa, od, di, ai = r.oa, r.od, float(r.od[0]), float(r.oa[0])
        else:
            oa = od = None
            ai = p.max_decel
        st = O.plant_step(p, st, ai, di)
        log.append(st + (int(flag),))
        for o in obs:        # constant-input motion, as their predictor does it
            o[0] += o[2] * np.cos(o[3]) * p.dt
            o[1] += o[2] * np.sin(o[3]) * p.dt
            o[2] += o[4] * p.dt
            o[3] += (o[2] / p.L) * np.tan(o[5]) * p.dt
    return np.array(log)


def _episode_obstacles(courses, seed):
    """Two constant-input cars crossing each course (as _constant_obstacles in test_gpu_plan_and_drive.py)."""
    rng = np.random.default_rng(seed)
    obst = np.zeros((len(courses), 2, 6))
    for b, c in enumerate(courses):
        if len(c) < 8:
            continue
        k = rng.integers(len(c) // 4, 3 * len(c) // 4, 2)
        ang = rng.uniform(-np.pi, np.pi, 2)
        obst[b, :, 0] = c[k, 0] - 25 * np.cos(ang)
        obst[b, :, 1] = c[k, 1] - 25 * np.sin(ang)
        obst[b, :, 2] = rng.uniform(3, 8, 2)
        obst[b, :, 3] = ang
        obst[b, :, 5] = rng.uniform(-.05, .05, 2)
    return obst


def test_planned_courses_in_three_copies_match_cpu_loop(jm, golden_dir):
    """The recorded planner variants three times: the third copy mostly gets no arc-length table.  The failed searches
    come first, so course 0 is a one-point placeholder: a kernel that read course 0's length or tables for another
    course's episode would not reproduce the CPU loop."""
    synth, BatchedMPC, PI = jm
    from junction_mpc import planner as P
    from junction_mpc.episodes import BatchedEpisodes
    z = load_planner_golden(golden_dir)
    names = sorted((str(n) for n in z["variants"]), key=lambda n: not np.isnan(z[f"{n}/cost"]))
    V = len(names)
    g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
    rep = names * 3
    inp = dict(start=np.stack([g(n, "start") for n in rep]), goal_point=np.stack([g(n, "goal_point") for n in rep]),
               goal_area=np.stack([g(n, "goal_area") for n in rep]),
               allowed_dtheta=np.array([float(g(n, "allowed_dtheta")) for n in rep]),
               scenes=[[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in names],
               scene_id=np.tile(np.arange(V), 3), weights=np.stack([g(n, "weights") for n in rep]))
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"],
                               max_batch=64)
    plans = planner.plan_device(**inp, max_expansions=8192, max_path=32)
    engine = BatchedMPC.from_plans(plans, T=13, max_batch=len(rep))
    ok = engine.course_ok.cpu().numpy().astype(bool)
    assert not ok[0] and ok[:V].sum() >= 45 and np.array_equal(np.tile(ok[:V], 3), ok)
    has = engine.arc_table_flags()
    assert (ok & ~has).sum() >= 30 and (ok & has).sum() >= 51
    courses = engine.get_courses()
    obst = np.tile(_episode_obstacles(courses[:V], 11), (3, 1, 1))
    steps, fw = 60, 10
    ep = BatchedEpisodes.from_plans(engine, plans, obstacles=obst.copy(), frame_window=fw, max_steps=steps)
    params = ep.params.cpu().numpy()
    res = ep.run(max_steps=steps)
    assert (res["done"][~ok] == 3).all() and (res["steps"][~ok] == 0).all()
    hist, flags = res["history"], res["flags"]
    assert len(hist) == steps
    for p in range(V):                                  # the copies of a plan drive identically, table or not
        for k in (1, 2):
            assert np.array_equal(hist[:, p], hist[:, k * V + p], equal_nan=True), names[p]
            assert np.array_equal(flags[:, p], flags[:, k * V + p]), names[p]
            assert np.array_equal(res["steps"][p], res["steps"][k * V + p])
    # against the CPU loop: copy p % 3 of every usable plan, so both arc paths are compared
    eps = [(p % 3) * V + p for p in range(V) if ok[p]]
    assert not has[eps].all() and has[eps].any()
    jobs = [(courses[e], params_from_vector(params[e], 13), (courses[e][0, 0], courses[e][0, 1], 0.0, courses[e][0, 2]),
             obst[e], fw, ep.margin, steps) for e in eps]
    with get_context("fork").Pool(_procs()) as pool:
        refs = pool.map(_cpu_episode_job, jobs, chunksize=1)
    raised = {True: 0, False: 0}
    for e, ref in zip(eps, refs):
        assert res["steps"][e] == len(ref)
        np.testing.assert_allclose(hist[:len(ref), e][:, [0, 1, 3, 2]], ref[:, :4], rtol=0, atol=1e-5)
        assert np.array_equal(flags[:len(ref), e], ref[:, 4].astype(np.int32)), e
        raised[bool(has[e])] += int(ref[:, 4].sum())
    assert raised[True] > 0 and raised[False] > 0
    planner.close()
    engine.close()
