"""The scene kernels at every scene size the C ABI allows: k in [1, 9] ([2, 9] for right of way and trips) and up to
n_obs = (k - 1) + n_extra = 8 obstacle slots (include/jmpc.h).

The K = 4 scene tests cannot tell `b % k` from `b & 3` or `b / k` from `b >> 2`, and never clear a mask bit above 2.
Here:
  * kernel grid: every scene entry point called directly through the engine's library on synthetic device arrays of
    B = 2520 episodes (the least common multiple of 1 .. 9, so every layout runs on the same data), with distinct
    values per episode, against its numpy oracle, bit for bit.  Every case also evaluates the oracle under a wrong
    layout (k - 1 or k + 1) on the host and asserts that it disagrees with the kernel: a case that passed under two
    layouts would not be testing the layout;
  * closed-loop scenes at other sizes, under the gates of the K = 4 files: the replay gate and the mate-row oracle at
    k = 2, 3, 5 (with 4 extras: 8 slots), 6 and 9; right of way with shared plans at k = 3 and 9; lifetimes with
    on_goal="leave" at k = 9; trips with a signal plan at k = 9.  Vehicle j of a scene drives approach j % 4 at queue
    position j // 4; the forced cases (doubling-back course, start above the speed cap) sit in slot k - 1.
"""
import ctypes

import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import collision_oracle as C
from oracle import right_of_way as RW
from oracle import scene_exchange as SX
from oracle import scene_lifetimes as SL
from oracle import scene_trips as ST
from oracle import shared_plans as SP
from oracle import signals as SG
from test_gpu_multi_agent import _replay_and_oracle

pytestmark = pytest.mark.gpu

B = 2520                                   # every k in 1 .. 9 divides it
ROUTES = [[f"intersection_{i}_{j}" for j in (1, 2, 3)] for i in (1, 2, 3, 4)]     # [approach][route]
GEO = C.CarGeometry()
STEPS = 200
JUNCTION = (0.0, 0.0, 10.0)


@pytest.fixture(scope="module")
def jm(golden_dir):
    import __graft_entry__ as g
    g.build()
    import torch
    from junction_mpc import _cabi, synth
    from junction_mpc import episodes as E
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    z = load_planner_golden(golden_dir)
    courses = []
    for row in ROUTES:
        for name in row:
            c = np.array(z[f"{name}/trajectory"], dtype=np.float64)
            synth.smooth_yaw_inplace(c[:, 2])
            courses.append(c)
    # a course that doubles back 0.05 m beside itself, far from the junction: the index rule raises once the ego
    # reaches the second leg (done = 2 mid-run), and it never enters the zone
    xs = np.concatenate([np.linspace(0, 20, 201), np.linspace(20, 10, 101)]) + 1000.0
    ys = np.concatenate([np.zeros(201), np.full(101, 0.05)]) + 1000.0
    courses.append(np.stack([xs, ys, np.zeros(302)], axis=1))
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=B)
    yield dict(torch=torch, cabi=_cabi, E=E, BatchedMPC=BatchedMPC, BatchedEpisodes=E.BatchedEpisodes, PI=PARAM_INDEX,
               names=E.OUTCOME_NAMES, courses=courses, dl=dl, margin=C.cutoff_margin(GEO, dl), engine=engine)
    engine.close()


# ---- the kernel grid -------------------------------------------------------------------------------------------------

def _dev(jm, a, dtype):
    torch = jm["torch"]
    dt = {np.float64: torch.float64, np.int32: torch.int32}[dtype]
    return torch.as_tensor(np.ascontiguousarray(a, dtype=dtype), dtype=dt, device="cuda")


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _host(jm, t):
    jm["torch"].cuda.synchronize()
    return t.cpu().numpy()


def _call(jm, name, *args):
    """engine._lib.<name>(handle, *args, default stream); tensors are passed as device pointers and stay referenced
    until the call has returned (a temporary freed earlier could hand its memory to the next argument)."""
    torch = jm["torch"]
    ptrs = [_p(a) if isinstance(a, torch.Tensor) else a for a in args]
    jm["cabi"].check(getattr(jm["engine"]._lib, name)(jm["engine"]._h, *ptrs, None), name)


def _mate_index(n, k):
    """[n, k - 1]: the episodes in the mate slots of every episode, in oracle/scene_lifetimes._mates order."""
    return np.array([m for _, m in SL._mates(n, k)], np.int64).reshape(n, k - 1)


def _params(jm, rng):
    """Default rows with a per-episode MAX_STEER, MAX_DECEL and dl, so that reading another episode's row shows."""
    PI = jm["PI"]
    p = np.repeat(jm["engine"].default_params[None, :], B, axis=0)
    p[:, PI["max_steer"]] = rng.uniform(0.2, 0.9, B)
    p[:, PI["max_decel"]] = -rng.uniform(2.0, 10.0, B)
    p[:, PI["dl"]] = rng.choice([0.05, 0.1, 0.2], B)
    return p


def _disagrees(got, wrong):
    """The kernel's output and the oracle under a wrong layout differ (on their common leading slots)."""
    got, wrong = np.asarray(got), np.asarray(wrong)
    if got.ndim > 1 and got.shape[1] != wrong.shape[1]:
        n = min(got.shape[1], wrong.shape[1])
        got, wrong = got[:, :n], wrong[:, :n]
    return not np.array_equal(got, wrong, equal_nan=True)


def _exchange_rows(state, record, di, done, steps, max_steer, max_decel):
    """[B, 6]: the row every vehicle presents at the instant of an exchange, by oracle/scene_exchange.vehicle_rows.
    The snapshot is one History row (the current pose and the controls its last step applied: the record's (delta, a)
    after an optimal solve, else (di, MAX_DECEL)); a running vehicle that has stepped shows that row (evaluation 1 of
    a one-step History), one that has not its start row (evaluation 0), a finished one its parked row."""
    ok = record[:, 3].astype(np.int64) == 0
    delta = np.where(ok, record[:, 0], di)
    acc = np.where(ok, record[:, 1], max_decel)
    nan = np.full(len(state), np.nan)
    hist = np.stack([state[:, 0], state[:, 1], state[:, 3], state[:, 2], nan, delta, acc, nan], axis=1)[None]
    moving = (done == 0) & (steps > 0)
    rows = SX.vehicle_rows(state, hist, moving.astype(np.int64), done, max_steer, 2)
    return np.where(((done == 0) & (steps == 0))[:, None], rows[0], rows[1])


def _exchange_want(rows, extras, k):
    return np.concatenate([rows[_mate_index(len(rows), k)], extras], axis=1)


@pytest.mark.parametrize("k", range(1, 10))
def test_scene_exchange_at_every_size(jm, k):
    PI = jm["PI"]
    rng = np.random.default_rng(100 + k)
    params = _params(jm, rng)
    state = np.stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B), rng.uniform(0.5, 10, B),
                      rng.uniform(-np.pi, np.pi, B)], axis=1)
    record = rng.uniform(-3, 3, (B, 8))
    record[:, 0] = rng.uniform(-1.5, 1.5, B)                             # delta: often beyond +-MAX_STEER
    record[:, 3] = rng.choice([0, 0, 0, 1, 2], B)                        # failed solves apply (di, MAX_DECEL)
    di = rng.uniform(-1.5, 1.5, B)
    done = rng.choice([0, 0, 0, 0, 1, 2, 3, 4, 5], B).astype(np.int32)
    steps = np.where(rng.random(B) < 0.3, 0, rng.integers(1, 50, B)).astype(np.int32)
    max_steer, max_decel = params[:, PI["max_steer"]], params[:, PI["max_decel"]]
    assert set(np.unique(done)) == {0, 1, 2, 3, 4, 5}
    run = (done == 0) & (steps > 0)
    assert (run & (record[:, 3] != 0)).any() and (run & (record[:, 3] == 0) & (np.abs(record[:, 0]) > max_steer)).any()
    assert (run & (record[:, 3] != 0) & (np.abs(di) > max_steer)).any() and ((done == 0) & (steps == 0)).any()
    rows = _exchange_rows(state, record, di, done, steps, max_steer, max_decel)
    d_state, d_record, d_di = _dev(jm, state, np.float64), _dev(jm, record, np.float64), _dev(jm, di, np.float64)
    d_params, d_done, d_steps = _dev(jm, params, np.float64), _dev(jm, done, np.int32), _dev(jm, steps, np.int32)
    for n_extra in sorted({0, 8 - (k - 1)}):
        n_obs = (k - 1) + n_extra
        extras = rng.uniform(-100, 100, (B, n_extra, 6))
        out = _dev(jm, np.full((B, max(n_obs, 1), 6), np.nan), np.float64)
        _call(jm, "jmpc_scene_exchange", B, k, n_extra, d_state, d_record, d_di, d_params, d_done,
              d_steps, _dev(jm, extras, np.float64) if n_extra else None, out)
        got = _host(jm, out)
        if n_obs == 0:                                  # nothing to lay out: the kernel writes nothing
            assert np.isnan(got).all()
            continue
        want = _exchange_want(rows, extras, k)
        assert np.array_equal(got, want), (k, n_extra)
        assert np.array_equal(got[:, k - 1:], extras)
        for kw in (k - 1, k + 1):
            if kw >= 1 and (kw - 1) + n_extra > 0:           # a layout with slots to compare
                assert _disagrees(got, _exchange_want(rows, extras, kw)), (k, n_extra, kw)
    print(f"\n[scene sizes: exchange] k = {k}, n_extra in {sorted({0, 8 - (k - 1)})}, B = {B}: bit for bit")


@pytest.mark.parametrize("k", range(2, 10))
def test_scene_plans_at_every_size_and_horizon(jm, k):
    PI = jm["PI"]
    rng = np.random.default_rng(200 + k)
    params = _params(jm, rng)
    max_steer = params[:, PI["max_steer"]]
    d_params = _dev(jm, params, np.float64)
    for T in (2, 3, 8, 13, 16, 31):
        n_obs = 8 if T % 2 else k - 1                 # the rows' stride: the full 8 slots, or the mates only
        oa = rng.uniform(-5, 3, (B, T))
        od = rng.uniform(-1.5, 1.5, (B, T))           # often beyond +-MAX_STEER
        warm = rng.integers(0, 2, B).astype(np.int32)
        done = rng.choice([0, 0, 0, 1, 2, 3, 4, 5], B).astype(np.int32)
        assert len({(w, d) for w, d in zip(warm, done)}) == 12          # every combination of warm and done
        obst = rng.uniform(-50, 50, (B, n_obs, 6))
        out = _dev(jm, np.full((B, k - 1, T - 1, 2), np.nan), np.float64)
        _call(jm, "jmpc_scene_plans", B, k, T, _dev(jm, oa, np.float64), _dev(jm, od, np.float64),
              _dev(jm, warm, np.int32), _dev(jm, done, np.int32), d_params, _dev(jm, obst, np.float64),
              n_obs, out)
        got = _host(jm, out)
        want = SP.mate_plans(oa, od, warm, done, obst, max_steer, k)
        assert np.array_equal(got, want), (k, T)
        kw = k - 1 if k >= 3 else k + 1
        rows = np.concatenate([obst, rng.uniform(-50, 50, (B, max(0, kw - 1 - n_obs), 6))], axis=1)
        assert _disagrees(got, SP.mate_plans(oa, od, warm, done, rows, max_steer, kw)), (k, T, kw)
    print(f"\n[scene sizes: plans] k = {k}, T in (2, 3, 8, 13, 16, 31), B = {B}: bit for bit")


@pytest.mark.parametrize("rule", ["first_come", "fixed"])
@pytest.mark.parametrize("k", range(2, 10))
def test_right_of_way_at_every_size(jm, k, rule):
    PI = jm["PI"]
    rng = np.random.default_rng(300 + k)
    params = _params(jm, rng)
    dl = params[:, PI["dl"]]
    agent_idx = rng.integers(0, 40, B).astype(np.int32)
    done = np.where(rng.random(B) < 0.7, 0, rng.choice([1, 2, 3, 4, 5], B)).astype(np.int32)
    entry = rng.choice([-1, 10, 20, 30], B, p=[0.15, 0.3, 0.3, 0.25])   # -1: class 2, never in the zone
    zone = np.stack([entry, np.where(entry < 0, -1, entry + rng.choice([5, 10], B))], axis=1).astype(np.int32)
    priority = rng.integers(0, 3, B).astype(np.float64)                # few keys: many ties
    code = jm["cabi"].ROW_FIRST_COME if rule == "first_come" else jm["cabi"].ROW_FIXED
    out = _dev(jm, np.zeros(B), np.int32)
    _call(jm, "jmpc_right_of_way", B, k, code, _dev(jm, agent_idx, np.int32), _dev(jm, done, np.int32),
          _dev(jm, params, np.float64), _dev(jm, zone, np.int32) if rule == "first_come" else None,
          _dev(jm, priority, np.float64) if rule == "fixed" else None, out)
    got = _host(jm, out)
    want = RW.consider_masks(rule, k, agent_idx, done, dl, zone, priority)
    assert np.array_equal(got, want)
    # the bits at and above k - 1 stay set, every mate slot's bit is cleared somewhere and kept for a parked mate
    # somewhere, and the episode index decides ties
    assert ((got.astype(np.int64) >> (k - 1)) == -1).all()
    mates = _mate_index(B, k)
    run = done == 0
    for s in range(k - 1):
        assert (run & ((got >> s) & 1 == 0)).any(), s
        assert (run & (done[mates[:, s]] != 0)).any(), s
    cls, key = RW.scene_keys(rule, agent_idx, dl, zone, priority)
    tie = run[:, None] & run[mates] & (cls[:, None] == cls[mates]) & (key[:, None] == key[mates])
    assert tie.any()
    if rule == "first_come":
        assert (run & (cls == 2)).any() and (run & (cls == 0)).any() and (run & (cls == 1)).any()
    for kw in (k - 1, k + 1):
        if kw >= 2:
            assert _disagrees(got, RW.consider_masks(rule, kw, agent_idx, done, dl, zone, priority)), kw
    print(f"\n[scene sizes: right of way {rule}] k = {k}: {int(tie.sum())} moving pairs tie on (cls, key)")


@pytest.mark.parametrize("k", range(1, 10))
def test_scene_presence_at_every_size(jm, k):
    rng = np.random.default_rng(400 + k)
    done = rng.choice([0, 0, 1, 2, 3, 4, 5, 5], B).astype(np.int32)
    d_done = _dev(jm, done, np.int32)
    for leave in (0, 1):
        present = ~((done == 5) | (bool(leave) & (done == 1)))
        for combine in (0, 1):
            mask0 = rng.integers(-2 ** 31, 2 ** 31, B).astype(np.int32)        # random high bits with combine = 1
            mask = _dev(jm, mask0, np.int32)
            _call(jm, "jmpc_scene_presence", B, k, leave, d_done, mask, combine)
            got = _host(jm, mask)
            oracle = lambda kk: SL.presence_masks(present, kk) & (mask0 if combine else -1)    # noqa: E731
            assert np.array_equal(got, oracle(k)), (leave, combine)
            for kw in (k - 1, k + 1):
                if kw >= 1:
                    assert _disagrees(got, oracle(kw)), (leave, combine, kw)
            absent = SL.presence_masks(present, k)
            for s in range(k - 1):                  # every mate slot has an absent mate somewhere
                assert ((absent >> s) & 1 == 0).any(), (leave, s)


def _scene_init_oracle(done, k):
    d = np.array(done).reshape(-1, k)
    d[(d == 3).any(axis=1)[:, None] & (d == 0)] = 4
    return d.reshape(-1)


@pytest.mark.parametrize("k", range(1, 10))
def test_scene_init_at_every_size(jm, k):
    rng = np.random.default_rng(500 + k)
    done = np.where(rng.random(B) < 0.9, 0, rng.choice([1, 2, 5], B)).astype(np.int32)
    s = np.arange(B // k)
    planted = s[s % 3 != 2]                           # two scenes in three get a done = 3 ...
    pos = (planted // 3) % k                          # ... in every position j of the scene
    done[planted * k + pos] = 3
    assert len(np.unique(pos)) == k
    d = _dev(jm, done, np.int32)
    _call(jm, "jmpc_scene_init", B, k, d)
    got = _host(jm, d)
    assert np.array_equal(got, _scene_init_oracle(done, k))
    for kw in (k - 1, k + 1):
        if kw >= 1:
            assert _disagrees(got, _scene_init_oracle(done, kw)), kw


@pytest.mark.parametrize("k", [2, 3, 5, 9])
def test_right_of_way_init_with_a_junction_per_scene(jm, k):
    courses = jm["courses"]
    rng = np.random.default_rng(600 + k)
    n_scenes = B // k
    cid = rng.integers(0, len(courses), B).astype(np.int32)
    # every scene's zone shifted: its own centre and radius (some courses miss some zones: -1)
    junction = np.stack([rng.uniform(-6, 6, n_scenes), rng.uniform(-6, 6, n_scenes), rng.uniform(0.5, 12, n_scenes)],
                        axis=1)
    out = _dev(jm, np.full((B, 2), -7), np.int32)
    _call(jm, "jmpc_right_of_way_init", B, k, _dev(jm, cid, np.int32), _dev(jm, junction, np.float64),
          n_scenes, out)
    got = _host(jm, out)
    oracle = lambda kk: np.array([RW.zone_indices(courses[cid[b]], junction[b // kk]) for b in range(B)])   # noqa: E731
    assert np.array_equal(got, oracle(k))
    assert (got[:, 0] < 0).any() and (got[:, 0] >= 0).any()
    assert _disagrees(got, oracle(k + 1))


@pytest.mark.parametrize("owned", [False, True], ids=["owner_null", "owner_array"])
@pytest.mark.parametrize("k", [1, 2, 3, 5, 9])
def test_signals_with_an_offset_per_scene(jm, k, owned):
    PI, cabi = jm["PI"], jm["cabi"]
    rng = np.random.default_rng(700 + k + 50 * owned)
    n_scenes = B // k
    cycle, green = 17, [(0, 6), (6, 5), (11, 0), (3, 17)]               # one always red, one always green
    plan = cabi.SignalPlan(cycle=cycle, n_groups=len(green), margin=3, stop_decel=3.0)
    for g, (a, n) in enumerate(green):
        plan.green_start[g], plan.green_len[g] = a, n
    offset = rng.permutation(np.arange(n_scenes) - n_scenes // 2).astype(np.int32)    # distinct, negatives included
    n_owner = B + 500 if owned else B
    owner = rng.permutation(n_owner)[:B].astype(np.int32) if owned else None
    o_of_b = owner if owned else np.arange(B)
    group = rng.integers(-1, len(green) + 1, n_owner).astype(np.int32)  # -1 and G: unsignalised
    entry = np.where(rng.random(n_owner) < 0.15, -1, rng.integers(5, 200, n_owner))
    zone = np.stack([entry, entry + 20], axis=1).astype(np.int32)
    course_n = np.asarray(jm["engine"].course_len)
    params = _params(jm, rng)
    n = dict(held=0, decided=0, go=0, known=0)
    for it, i in enumerate((0, 9, 40, 123)):
        checked = it % 2
        done = np.where(rng.random(B) < 0.8, 0, rng.choice([1, 2, 5], B)).astype(np.int32)
        agent_idx = rng.integers(0, 220, B).astype(np.int32)
        state = np.stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B), rng.uniform(0, 12, B),
                          rng.uniform(-3, 3, B)], axis=1)
        cid = rng.integers(0, len(course_n), B).astype(np.int32)
        course_len = rng.integers(1, 300, B).astype(np.int32)
        kind = rng.integers(0, 3, B)                  # latch empty, this owner's decision, another owner's
        latch = np.stack([np.where(kind == 0, -1, np.where(kind == 1, o_of_b, (o_of_b + 1) % n_owner)),
                          rng.integers(0, 2, B)], axis=1).astype(np.int32)
        latch[kind == 0, 1] = 0
        hold0, go0 = rng.integers(0, 5, n_owner).astype(np.int32), rng.integers(0, 5, n_owner).astype(np.int32)
        slot0 = [rng.integers(0, 5, B).astype(np.int32) for _ in range(2)] if owned else None
        d = dict(course_len=_dev(jm, course_len, np.int32), latch=_dev(jm, latch, np.int32),
                 hold=_dev(jm, hold0, np.int32), go=_dev(jm, go0, np.int32),
                 slot_hold=_dev(jm, slot0[0], np.int32) if owned else None,
                 slot_go=_dev(jm, slot0[1], np.int32) if owned else None)
        _call(jm, "jmpc_signals", B, k, ctypes.byref(plan), _dev(jm, offset, np.int32),
              _dev(jm, owner, np.int32) if owned else None, _dev(jm, group, np.int32),
              _dev(jm, zone, np.int32), _dev(jm, cid, np.int32), _dev(jm, agent_idx, np.int32),
              _dev(jm, state, np.float64), _dev(jm, params, np.float64), _dev(jm, done, np.int32), checked,
              d["course_len"], d["latch"], d["hold"], d["go"], d["slot_hold"], d["slot_go"],
              _dev(jm, [i], np.int32))
        got = [_host(jm, d[n_]) for n_ in ("course_len", "latch", "hold", "go")]
        snap = dict(iteration=i, cycle=cycle, green_start=[a for a, _ in green], green_len=[n_ for _, n_ in green],
                    margin=3, stop_decel=3.0, k=k, offset=offset, owner=owner, group=group, zone=zone, course_id=cid,
                    course_n=course_n, agent_idx=agent_idx, state=state, dl=params[:, PI["dl"]], done=done,
                    checked=bool(checked), course_len=course_len, latch=latch, hold_steps=hold0, go=go0)
        want = SG.signal_pass(snap)
        for name, g_, w_ in zip(("course_len", "latch", "hold_steps", "go"), got, want):
            assert np.array_equal(g_, w_), (i, name)
        if owned:
            run = done == 0
            o = np.where(run, owner, 0)
            assert np.array_equal(_host(jm, d["slot_hold"]) - slot0[0], np.where(run, (want[2] - hold0)[o], 0)), i
            assert np.array_equal(_host(jm, d["slot_go"]) - slot0[1], np.where(run, (want[3] - go0)[o], 0)), i
        wrong = SG.signal_pass({**snap, "k": k + 1})
        assert any(_disagrees(g_, w_) for g_, w_ in zip(got, wrong)), (i, k + 1)
        o = o_of_b
        held = (done == 0) & (want[1][:, 0] == o) & (want[1][:, 1] == 1)
        n["held"] += int(held.sum())
        n["decided"] += int((held & (latch[:, 0] != o)).sum())
        n["known"] += int((held & (latch[:, 0] == o)).sum())
        n["go"] += int((want[3] - go0).sum())
    print(f"\n[scene sizes: signals] k = {k}, owner {'array' if owned else 'NULL'}: held {n['held']} (decided now "
          f"{n['decided']}, latched {n['known']}), GO passes {n['go']}")
    assert n["decided"] > 0 and n["known"] > 0 and n["go"] > 0


def _trip_snapshot(jm, ep, k, rng, iteration):
    """Writes a random mid-run state into the trips run `ep`: every slot empty or holding one of its scene's trips with
    done 0, 1 (its goal test fired) or 2; one scene in four with every slot held; pending and closed trips, unusable
    ones among them.  Returns the host copies the oracle reads."""
    T = ep._trips
    scene_start = T["scene_start"].cpu().numpy()
    n_scenes, N = len(scene_start) - 1, int(scene_start[-1])
    phase = np.where(rng.random(N) < 0.75, ST.PENDING, ST.CLOSED)
    done = np.full(B, ST.WAITING)
    slot_trip = np.full(B, -1)
    for s in range(n_scenes):
        trips = rng.permutation(np.arange(scene_start[s], scene_start[s + 1]))
        held = np.ones(k, bool) if s % 4 == 0 else rng.random(k) < 0.5
        for j in np.flatnonzero(held)[:len(trips)]:
            b, t = s * k + j, trips[j]
            slot_trip[b], phase[t] = t, ST.IN_SLOT
            done[b] = rng.choice([0, 0, 1, 2])
    state = np.stack([rng.uniform(-25, 25, B), rng.uniform(-25, 25, B), rng.uniform(0, 8, B),
                      rng.uniform(-np.pi, np.pi, B)], axis=1)
    usable = (rng.random(N) >= 0.1).astype(np.int32)
    bad = np.where(usable == 0, np.arange(N), N)
    torch = jm["torch"]
    for name, a in (("phase", phase), ("slot_trip", slot_trip), ("usable", usable),
                    ("next_unusable", np.minimum.accumulate(bad[::-1])[::-1]), ("blocked_waits", np.zeros(N)),
                    ("cursor", scene_start[:-1]), ("pending", np.full(n_scenes, 1000))):
        T[name].copy_(torch.as_tensor(np.asarray(a, np.int32)))
    ep.done.copy_(torch.as_tensor(done.astype(np.int32)))
    ep.state.copy_(torch.as_tensor(state))
    ep.iter_dev.fill_(iteration)
    return dict(done=done, state=state, slot_trip=slot_trip, phase=phase, usable=usable, scene_start=scene_start)


@pytest.mark.parametrize("k", [2, 3, 9])
def test_trips_pass_snapshots(jm, k):
    E, torch = jm["E"], jm["torch"]
    rng = np.random.default_rng(800 + k)
    n_scenes = B // k
    per = rng.integers(k, 2 * k + 5, n_scenes)
    scene = np.repeat(np.arange(n_scenes), per)
    arrival = np.concatenate([np.sort(rng.integers(0, 24, n)) for n in per])
    # starts at four approach poses with a little jitter: trips of one approach block each other (first in, first out)
    approach = np.array([[-20, -2, 0], [20, 2, np.pi], [2, -20, np.pi / 2], [-2, 20, -np.pi / 2]], np.float64)
    g = rng.integers(0, 4, len(scene))
    start = np.stack([approach[g, 0] + rng.uniform(-1, 1, len(g)), approach[g, 1] + rng.uniform(-1, 1, len(g)),
                      rng.uniform(0, 5, len(g)), approach[g, 2]], axis=1)
    cid = rng.integers(0, 12, len(scene))
    ep = jm["BatchedEpisodes"].from_trips(jm["engine"], E.Trips(scene, arrival, cid, start), n_scenes,
                                          agents_per_scene=k, frame_window=10, margin=jm["margin"], max_steps=8,
                                          record_history=False)
    assert np.array_equal(ep._trip_order, np.arange(len(scene)))          # the trips are given in the pass's order
    T = ep._trips
    n = dict(closed=0, admitted=0, no_course=0, blocked=0, slot_waits=0, close_and_admit=0, full=0, above_lowest=0)
    for initial, iteration in ((0, 12), (1, 0)):
        snap = _trip_snapshot(jm, ep, k, rng, iteration)
        torch.cuda.synchronize()
        jm["cabi"].check(jm["engine"]._lib.jmpc_scene_trips(jm["engine"]._h, ctypes.byref(ep._trips_struct),
                                                            _p(ep.iter_dev), initial, None), "jmpc_scene_trips")
        args = (snap["done"], snap["state"], snap["slot_trip"], snap["phase"], snap["scene_start"], arrival,
                snap["usable"], start)
        want = ST.trips_pass(*args, k, iteration, initial=bool(initial), entry_gap=2.0, geo=GEO)
        got_done, got_slot_trip = _host(jm, ep.done), _host(jm, T["slot_trip"])
        assert np.array_equal(got_done, want["done"])
        assert np.array_equal(got_slot_trip, want["slot_trip"])
        assert np.array_equal(_host(jm, T["phase"]), want["phase"])
        assert np.array_equal(_host(jm, ep.state), want["state"])
        assert sorted(np.flatnonzero(_host(jm, T["blocked_waits"]))) == want["blocked_waits"]
        entry, slot, exit_, tdone = (_host(jm, T[x]) for x in ("entry", "slot", "exit", "done"))
        for t, b in want["admitted"]:
            assert entry[t] == want["entry"] and slot[t] == b, t
        for t, b in want["closed"]:
            assert exit_[t] == (-1 if initial else iteration) and tdone[t] == 1, t
        assert (tdone[want["no_course"]] == 3).all()
        settled = np.bincount(np.searchsorted(snap["scene_start"], [t for t, _ in want["admitted"]] + want["no_course"],
                                              side="right") - 1, minlength=n_scenes)
        assert np.array_equal(_host(jm, T["pending"]), 1000 - settled)
        wrong = ST.trips_pass(*args, k - 1, iteration, initial=bool(initial), entry_gap=2.0, geo=GEO)
        assert _disagrees(got_done, wrong["done"]) or _disagrees(got_slot_trip, wrong["slot_trip"])
        closed_s = {b // k for _, b in want["closed"]}
        admitted_s = {b // k for _, b in want["admitted"]}
        n["closed"] += len(want["closed"])
        n["admitted"] += len(want["admitted"])
        n["no_course"] += len(want["no_course"])
        n["blocked"] += len(want["blocked_waits"])
        n["slot_waits"] += len(want["slot_waits"])
        n["close_and_admit"] += len(closed_s & admitted_s)
        n["full"] += int((want["done"].reshape(-1, k) != ST.WAITING).all(axis=1).sum())
        n["above_lowest"] += sum(b % k > 0 for _, b in want["admitted"])
    print(f"\n[scene sizes: trips] k = {k}: {n}")
    assert all(v > 0 for v in n.values()), n


# ---- closed-loop scenes at other sizes -------------------------------------------------------------------------------

def _scenes(jm, n_scenes, k, seed=7, forced=True):
    """Start states, course ids and params rows of n_scenes x k vehicles: vehicle j of a scene drives approach j % 4 on
    a random route, at queue position j // 4, about 7 m behind the vehicle ahead (the leader furthest in), at 2-5 m/s.
    forced: slot k - 1 of scene 0 drives the doubling-back course (done = 2 mid-run), slot k - 1 of every 16th scene
    from scene 16 on starts above the QP's speed cap (failed solves until it has braked below it)."""
    rng = np.random.default_rng(seed)
    courses, PI, dl = jm["courses"], jm["PI"], jm["dl"]
    n = n_scenes * k
    j = np.arange(n) % k
    cid = (j % 4) * 3 + rng.integers(0, 3, n)
    gap = int(round(7.0 / dl))
    queue = (k - 1 - j % 4) // 4 + 1                 # vehicles on the approach of j
    off = rng.integers(0, 40, n_scenes).repeat(k) + (queue - 1 - j // 4) * gap
    state0 = np.array([[courses[c][o, 0], courses[c][o, 1], 0.0, courses[c][o, 2]] for c, o in zip(cid, off)])
    state0[:, 2] = rng.uniform(2, 5, n)
    engine = jm["BatchedMPC"](courses, dl=dl, T=13, max_batch=max(n, 64))
    params = np.repeat(engine.default_params[None, :], n, axis=0)
    if forced:
        state0[16 * k + k - 1::16 * k, 2] = 9.0
        hp = len(courses) - 1
        cid[k - 1] = hp
        state0[k - 1] = [courses[hp][0, 0], courses[hp][0, 1], 3.0, 0.0]
        params[k - 1, PI["dl"]] = 0.1
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


@pytest.mark.parametrize("k,n_extra", [(2, 0), (3, 0), (5, 4), (6, 0), (9, 0)],
                         ids=["k2", "k3", "k5_extras4", "k6", "k9"])
def test_closed_loop_replay_and_mate_rows(jm, k, n_extra):
    n_scenes = 40
    engine, state0, cid, params = _scenes(jm, n_scenes, k, seed=10 + k)
    n = len(state0)
    kw = dict(course_id=cid, params=params, frame_window=10, margin=jm["margin"], max_steps=STEPS, agents_per_scene=k,
              outcomes=True, record_obstacles=True)
    if n_extra:
        rng = np.random.default_rng(1)
        obst = np.zeros((n, n_extra, 6))
        ang = rng.uniform(-np.pi, np.pi, (n, n_extra))
        obst[..., 0] = rng.uniform(-15, 15, (n, n_extra)) - 20 * np.cos(ang)
        obst[..., 1] = rng.uniform(-15, 15, (n, n_extra)) - 20 * np.sin(ang)
        obst[..., 2] = rng.uniform(2, 6, (n, n_extra))
        obst[..., 3] = ang
        obst[..., 5] = rng.uniform(-.05, .05, (n, n_extra))
        kw["obstacles"] = obst
    ep = jm["BatchedEpisodes"](engine, state0, **kw)
    assert ep.n_obs == k - 1 + n_extra
    res = ep.run(max_steps=STEPS)
    rows, active = _replay_and_oracle(jm, engine, state0, cid, params, res, k, n_extra)
    done, out = res["done"], res["outcomes"]
    assert done[k - 1] == 2 and res["steps"][k - 1] > 0
    assert (done == 1).any()
    assert (out["failed_solves"][16 * k + k - 1::16 * k] > 0).all()
    parked = active[:, :, None] & (rows[..., 2] == 0) & (rows[..., 4] == 0) & (rows[..., 5] == 0)
    assert parked[1:, :k - 1].any()                 # scene 0's vehicles see the done = 2 vehicle parked
    if n_extra:
        assert (out["min_clearance_obs"] >= k - 1).any() and (out["min_clearance_obs"] < k - 1).any()
    print(f"\n[scene sizes: replay] k = {k}, n_extra = {n_extra}: {n} vehicles, {res['iterations']} iterations, done "
          f"codes {np.bincount(done).tolist()}, parked mate-slot rows seen {int(parked.sum())}")
    engine.close()


@pytest.mark.parametrize("k", [3, 9])
def test_closed_loop_right_of_way_with_shared_plans(jm, k):
    torch, PI, courses = jm["torch"], jm["PI"], jm["courses"]
    engine, state0, cid, params = _scenes(jm, 32, k, seed=20 + k)
    n = len(state0)
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=k, share_plans=True, right_of_way="first_come",
                               junction=JUNCTION, record_history=False)
    dl, max_steer = params[:, PI["dl"]], params[:, PI["max_steer"]]
    zone = ep.zone.cpu().numpy()
    mates = _mate_index(n, k)
    rng = np.random.default_rng(0)
    snap = {}
    cnt = dict(evals=0, checked=0, ties=0, parked=0, ignored_bits=np.zeros(8, np.int64))

    def before():
        torch.cuda.synchronize()
        snap.update(a=ep.agent_idx.cpu().numpy().copy(), done=ep.done.cpu().numpy().copy())

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_right_of_way": (before, None)})
    try:
        ep._start()
        g = lambda t: t.cpu().numpy().copy()          # noqa: E731
        rows, plans = g(ep.scene_obs), g(ep.scene_plans)
        assert np.array_equal(plans, SP.mate_plans(g(ep.oa), g(ep.od), g(ep.warm), g(ep.done), rows, max_steer, k))
        while ep.iteration < STEPS:
            prev_steps = g(ep.steps)
            ep.iterate()
            a, done, mask = snap["a"], snap["done"], g(ep.consider)
            assert np.array_equal(mask, RW.consider_masks("first_come", k, a, done, dl, zone)), ep.iteration
            run = done == 0
            for s in range(k - 1):
                cnt["ignored_bits"][s] += int((run & ((mask >> s) & 1 == 0)).sum())
            cnt["parked"] += int((run[:, None] & (done[mates] != 0)).sum())
            cls, key = RW.scene_keys("first_come", a, dl, zone)
            cnt["ties"] += int((run[:, None] & run[mates] & (cls[:, None] == cls[mates])
                                & (key[:, None] == key[mates])).sum())
            cnt["evals"] += 1
            stepped = np.flatnonzero(g(ep.steps) > prev_steps)
            flag, clen, a_idx, v = g(ep.flag), g(ep.course_len), g(ep.agent_idx), g(ep.v)
            full = (1 << (k - 1)) - 1
            part = stepped[(mask[stepped] & full) != full]          # prefer vehicles that ignore a mate
            pool = part if len(part) >= 3 else stepped
            for b in rng.choice(pool, min(3, len(pool)), replace=False):
                keep = [s for s in range(ep.n_obs) if (int(mask[b]) >> s) & 1]
                pr = params[b]
                f, cl = SP.collision_cut(GEO, courses[cid[b]], int(a_idx[b]), float(v[b]), rows[b][keep],
                                         dt=pr[PI["dt"]], frame_window=ep.frame_window, max_accel=pr[PI["max_accel"]],
                                         max_speed=pr[PI["sim_max_speed"]], margin=ep.margin,
                                         plans=[plans[b, s] for s in keep])
                assert (int(f), cl) == (int(flag[b]), int(clen[b])), (ep.iteration, b)
                cnt["checked"] += 1
            rows, plans = g(ep.scene_obs), g(ep.scene_plans)
            assert np.array_equal(plans, SP.mate_plans(g(ep.oa), g(ep.od), g(ep.warm), g(ep.done), rows, max_steer,
                                                       k)), ep.iteration
            if (g(ep.done) != 0).all():
                break
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)
    print(f"\n[scene sizes: right of way + shared plans] k = {k}, {n} vehicles, {cnt['evals']} evaluations: mates "
          f"ignored per slot bit {cnt['ignored_bits'][:k - 1].tolist()}, parked mate-slots {cnt['parked']}, ties "
          f"{cnt['ties']}, flags checked {cnt['checked']}; done codes {np.bincount(res['done']).tolist()}")
    assert (cnt["ignored_bits"][:k - 1] > 0).all() and cnt["parked"] > 0 and cnt["ties"] > 0 and cnt["checked"] > 100
    assert res["done"][k - 1] == 2
    engine.close()


def test_closed_loop_lifetimes_leave_at_nine(jm):
    k = 9
    torch, WAITING = jm["torch"], jm["cabi"].WAITING
    engine, state0, cid, params = _scenes(jm, 32, k, seed=31)
    n = len(state0)
    rng = np.random.default_rng(2)
    depart = np.where(rng.random(n) < 0.4, 0, rng.integers(1, 60, n))
    ep = jm["BatchedEpisodes"](engine, state0, course_id=cid, params=params, frame_window=10, margin=jm["margin"],
                               max_steps=STEPS, agents_per_scene=k, depart=depart, on_goal="leave", outcomes=True,
                               record_history=False)
    snap, cnt = {}, dict(checks=0, absent_bits=np.zeros(8, np.int64))
    which = {"n": 0}
    present_at_eval = []

    def before():
        torch.cuda.synchronize()
        snap["done"] = ep.done.cpu().numpy().copy()

    def after():
        # _start writes the evaluation mask; then every iteration the collision mask, then the evaluation mask
        evaluation = not ep._started or which["n"] % 2 == 1
        if ep._started:
            which["n"] += 1
        torch.cuda.synchronize()
        got = (ep.presence if evaluation else ep._collision_mask).cpu().numpy()
        done = snap["done"]
        present = (done != WAITING) & (done != 1)
        assert np.array_equal(got, SL.presence_masks(present, k)), ep.iteration
        if evaluation:
            present_at_eval.append(present)
        for s in range(k - 1):
            cnt["absent_bits"][s] += int(((got >> s) & 1 == 0).sum())
        cnt["checks"] += 1

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_scene_presence": (before, after)})
    try:
        res = ep.run(max_steps=STEPS)
    finally:
        engine._lib = lib
    print(f"\n[scene sizes: lifetimes] k = {k}, {n} vehicles, {res['iterations']} iterations, {cnt['checks']} masks "
          f"checked: absent mates per slot bit {cnt['absent_bits'][:k - 1].tolist()}; done codes "
          f"{np.bincount(res['done']).tolist()}")
    assert cnt["checks"] == 2 * res["iterations"] + 1
    # every evaluation's presence is the oracle's, from the departures and the run's steps and done codes
    want = SL.presence(depart, res["steps"], res["done"], "leave", res["iterations"] + 1)
    assert np.array_equal(np.array(present_at_eval), want)
    assert (cnt["absent_bits"][:k - 1] > 0).all() and (res["done"] == 1).any()
    engine.close()


def test_closed_loop_trips_with_signals_at_nine(jm):
    k = 9
    torch, PI, E, courses = jm["torch"], jm["PI"], jm["E"], jm["courses"]
    n_scenes, steps = 48, 160
    routes = [[(3 * g + r, tuple(courses[3 * g + r][0, :3])) for r in range(3)] for g in range(4)]
    trips = E.poisson_trips(n_scenes, routes, 2400.0, 0.2, steps - 40, 4.0, seed=3, groups=[0, 1, 0, 1])
    rng = np.random.default_rng(4)
    plan = E.SignalPlan(40, [(0, 18), (20, 18)], JUNCTION, offset=rng.integers(-100, 100, n_scenes))
    engine = jm["BatchedMPC"](courses, dl=jm["dl"], T=13, max_batch=n_scenes * k)
    ep = jm["BatchedEpisodes"].from_trips(engine, trips, n_scenes, agents_per_scene=k, frame_window=10,
                                          margin=jm["margin"], max_steps=steps, signals=plan, record_history=False)
    T = ep._trips
    scene_start, arrival = T["scene_start"].cpu().numpy(), T["arrival"].cpu().numpy()
    usable, start = T["usable"].cpu().numpy(), T["start"].cpu().numpy()
    course_n = np.asarray(engine.course_len)
    group, zone = ep.signal_group.cpu().numpy(), ep.signal_zone.cpu().numpy()
    g = lambda x: x.cpu().numpy().copy()                                          # noqa: E731
    snap, sig = {}, {}
    cnt = dict(passes=0, signal_passes=0, admitted=0, full=0, held=0)
    held_offsets = set()

    def before_pass():
        torch.cuda.synchronize()
        snap.update(done=g(ep.done), state=g(ep.state), slot_trip=g(T["slot_trip"]), phase=g(T["phase"]),
                    it=ep.iteration)

    def after_pass():
        torch.cuda.synchronize()
        want = ST.trips_pass(snap["done"], snap["state"], snap["slot_trip"], snap["phase"], scene_start, arrival,
                             usable, start, k, snap["it"], initial=not ep._started, entry_gap=2.0, geo=GEO)
        assert np.array_equal(g(ep.done), want["done"]), snap["it"]
        assert np.array_equal(g(T["slot_trip"]), want["slot_trip"]), snap["it"]
        assert np.array_equal(g(T["phase"]), want["phase"]), snap["it"]
        cnt["passes"] += 1
        cnt["admitted"] += len(want["admitted"])
        cnt["full"] += int((want["done"].reshape(-1, k) != ST.WAITING).all(axis=1).sum())

    def before_signals():
        torch.cuda.synchronize()
        sig.update(iteration=ep.iteration, cycle=plan.cycle, green_start=plan.green[:, 0], green_len=plan.green[:, 1],
                   margin=ep._signal_plan.margin, stop_decel=plan.stop_decel, k=k, offset=plan.offset,
                   owner=g(ep.signal_owner), group=group, zone=zone, course_id=g(ep.course_id), course_n=course_n,
                   agent_idx=g(ep.agent_idx), state=g(ep.state), dl=g(ep.params)[:, PI["dl"]], done=g(ep.done),
                   checked=True, course_len=g(ep.course_len), latch=g(ep.signal_latch), hold_steps=g(ep.signal_hold),
                   go=g(ep.signal_go))

    def after_signals():
        torch.cuda.synchronize()
        course_len, latch, hold, go = SG.signal_pass(sig)
        it = sig["iteration"]
        assert np.array_equal(g(ep.course_len), course_len), it
        assert np.array_equal(g(ep.signal_latch), latch), it
        assert np.array_equal(g(ep.signal_hold), hold), it
        assert np.array_equal(g(ep.signal_go), go), it
        run = sig["done"] == 0
        o = np.where(run, sig["owner"], 0)
        held = run & (latch[:, 0] == o) & (latch[:, 1] == 1)
        held_offsets.update(int(plan.offset[s]) % plan.cycle for s in np.flatnonzero(held) // k)
        cnt["held"] += int(held.sum())
        cnt["signal_passes"] += 1

    lib = engine._lib
    engine._lib = _Calls(lib, {"jmpc_scene_trips": (before_pass, after_pass),
                               "jmpc_signals": (before_signals, after_signals)})
    try:
        snap["it"] = 0
        ep._start()
        while ep.iteration < steps and not ep._finished():
            ep.iterate()
    finally:
        engine._lib = lib
    res = ep.run(max_steps=ep.iteration)
    print(f"\n[scene sizes: trips + signals] k = {k}, {trips.n} trips in {n_scenes} scenes, {res['iterations']} "
          f"iterations: passes checked {cnt['passes']} / signal passes {cnt['signal_passes']}, admitted "
          f"{cnt['admitted']}, scene-passes with all {k} slots held {cnt['full']}, held vehicle-steps {cnt['held']} "
          f"under {len(held_offsets)} distinct scene offsets (mod the cycle)")
    assert cnt["passes"] == res["iterations"] + 1 and cnt["signal_passes"] == res["iterations"]
    assert cnt["full"] > 0 and cnt["held"] > 0 and len(held_offsets) >= 3
    engine.close()
