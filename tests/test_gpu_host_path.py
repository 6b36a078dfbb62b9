"""The host entry points (`jmpc_step_host[_io]`, `jmpc_collision_host`): every transfer mode, pageable and page-locked
callers, and the host-side refusals.  Needs a GPU: `pytest -m gpu`."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ["staged", "zero_copy_results", "zero_copy"]
SKIP_MSG = "a skip mask is set (jmpc_set_skip_mask is for the device entry points)"


@pytest.fixture(scope="module")
def jm():
    import __graft_entry__ as g
    g.build()
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.config import PARAM_INDEX
    return synth, BatchedMPC, PARAM_INDEX, _cabi


@pytest.fixture(scope="module")
def scene(jm):
    """400 collision instances over three courses with per-instance parameters; the first obstacle of most of them sits
    next to the path ahead, so that both flag values occur."""
    synth, BatchedMPC, PI, _ = jm
    courses = [synth.load_course(n) for n in ("intersection", "roundabout", "multilane")]
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    mpc = BatchedMPC(courses, dl=dl, T=13, max_batch=512)
    rng = np.random.default_rng(31)
    B, n_obs = 400, 3
    cid = rng.integers(0, len(courses), B).astype(np.int32)
    a0 = np.array([rng.integers(0, len(courses[c]) - 1) for c in cid], dtype=np.int32)
    v = rng.uniform(0, 30 / 3.6, B)
    v[::9] = 30 / 3.6
    params = np.repeat(mpc.default_params[None, :], B, axis=0)
    params[:, PI["dt"]] = rng.choice([0.1, 0.2], B)
    params[:, PI["max_accel"]] = rng.choice([0.35, 1.0, 2.0], B)
    obs = np.zeros((B, n_obs, 6))
    for b in range(B):
        c = courses[cid[b]]
        obs[b, :, :2] = c[a0[b], :2] + rng.uniform(-35, 35, (n_obs, 2))
        k = min(a0[b] + int(rng.integers(0, 150)), len(c) - 1)
        obs[b, 0, :2] = c[k, :2] + rng.uniform(-6, 6, 2)
    obs[:, :, 2] = rng.uniform(0, 30 / 3.6, (B, n_obs))
    obs[:, :, 3] = rng.uniform(-np.pi, np.pi, (B, n_obs))
    obs[:, :, 5] = rng.uniform(-0.4, 0.4, (B, n_obs))
    inputs = dict(agent_idx=a0, v=v, obstacles=obs, course_id=cid, params=params)
    kw = dict(frame_window=20, margin=40, horizon_s=7.0)
    want = {n: _device_collision(mpc, inputs, obstacles, kw) for n, obstacles in ((n_obs, obs), (0, None))}
    hit = want[n_obs][0] == 1
    assert 0.05 < hit.mean() < 0.95
    assert (want[0][0] == 0).all()
    yield mpc, inputs, kw, want
    mpc.close()


def _device_collision(mpc, inputs, obstacles, kw):
    import torch
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")     # noqa: E731
    B = len(inputs["v"])
    flag = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    clen = torch.full((B,), -9, dtype=torch.int32, device="cuda")
    mpc.collision(t(inputs["agent_idx"], torch.int32), t(inputs["v"], torch.float64),
                  None if obstacles is None else t(obstacles, torch.float64), kw["frame_window"], kw["margin"], flag,
                  clen, course_id=t(inputs["course_id"], torch.int32), params=t(inputs["params"], torch.float64),
                  horizon_s=kw["horizon_s"])
    torch.cuda.synchronize()
    return flag.cpu().numpy(), clen.cpu().numpy()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("pinned_in", [False, True])
@pytest.mark.parametrize("pinned_out", [False, True])
def test_collision_host_equals_device_path(scene, mode, pinned_in, pinned_out):
    mpc, inputs, kw, want = scene
    B = len(inputs["v"])
    if pinned_in:
        arrays = {}
        for k, a in inputs.items():
            arrays[k] = mpc.pinned_empty(a.shape, a.dtype)
            arrays[k][...] = a
    else:
        arrays = inputs
    mpc.set_host_transfer(mode)
    try:
        for n_obs in want:
            obstacles = arrays["obstacles"] if n_obs else np.zeros((B, 0, 6))
            out = None
            if pinned_out:
                out = (mpc.pinned_empty((B,), np.int32), mpc.pinned_empty((B,), np.int32))
                out[0][...], out[1][...] = -5, -5
            flag, clen = mpc.collision_host(arrays["agent_idx"], arrays["v"], obstacles, course_id=arrays["course_id"],
                                            params=arrays["params"], out=out, **kw)
            if pinned_out:
                assert flag is out[0] and clen is out[1]
            assert np.array_equal(flag, want[n_obs][0]), (n_obs, np.flatnonzero(flag != want[n_obs][0])[:10])
            assert np.array_equal(clen, want[n_obs][1]), (n_obs, np.flatnonzero(clen != want[n_obs][1])[:10])
    finally:
        mpc.set_host_transfer("zero_copy_results")
    for k, a in inputs.items():                     # inputs are only read
        assert np.array_equal(arrays[k], a), k


# ---- step -------------------------------------------------------------------------------------------------
KEYS = ["oa", "od", "cost", "status", "iters", "target_ind", "record"]


@pytest.fixture(scope="module")
def step_case(jm):
    synth, BatchedMPC, _, _ = jm
    w = synth.make_workload(2, B=130)
    state = w["state"].copy()
    state[3, 2] = 30.0            # v0 above the speed cap -> infeasible (status 2): in-out values carried over
    mpc = BatchedMPC(w["courses"], dl=w["dl"], T=w["T"], max_batch=256)
    mpc.set_host_transfer("staged")
    ref = mpc.step_host(state, w["target_ind"], w["oa"], w["od"], course_len=w["course_len"])
    mpc.set_host_transfer("zero_copy_results")
    assert ref.status[3] == 2 and np.array_equal(ref.oa[3], w["oa"][3]) and np.array_equal(ref.od[3], w["od"][3])
    yield mpc, w, state, ref
    mpc.close()


def _step_host_c(jm, mpc, w, state, alloc):
    """jmpc_step_host called directly: target_ind / oa / od are read and written in place."""
    _cabi = jm[3]
    B, T = len(state), w["T"]

    def arr(shape, dtype=np.float64, fill=0):
        a = alloc(shape, dtype)
        a[...] = fill
        return a
    tgt, oa, od = arr((B,), np.int32), arr((B, T)), arr((B, T))
    tgt[...], oa[...], od[...] = w["target_ind"], w["oa"], w["od"]
    ox, oy, ov, oyaw = (arr((B, T + 1)) for _ in range(4))
    xref, cost = arr((B, 4, T + 1)), arr((B,), fill=np.nan)
    status, iters, record = arr((B,), np.int32), arr((B,), np.int32), arr((B, _cabi.RECORD_LEN))
    p = lambda a: a.ctypes.data_as(C.c_void_p)     # noqa: E731
    clen = np.ascontiguousarray(w["course_len"], np.int32)
    _cabi.check(mpc._lib.jmpc_step_host(mpc._h, B, T, p(state), None, p(clen), p(tgt), None, p(oa), p(od),
                                        None, p(ox), p(oy), p(ov), p(oyaw), p(xref), p(cost), p(status), p(iters),
                                        p(record)), "jmpc_step_host")
    from junction_mpc.batched import StepOutput
    return StepOutput(oa, od, ox, oy, ov, oyaw, xref, cost, status, iters, tgt, record)


@pytest.mark.parametrize("mode", MODES)
def test_step_host_paths_agree(jm, step_case, mode):
    """`step_host` with fresh results, with `host_outputs`, and the in-place C entry point `jmpc_step_host` on pageable
    and on page-locked arrays give the same arrays; the caller's inputs stay as they were."""
    mpc, w, state, ref = step_case
    solved = ref.status == 0
    inputs = {k: w[k].copy() for k in ("target_ind", "oa", "od")}
    mpc.set_host_transfer(mode)
    try:
        got = {"fresh": mpc.step_host(state, w["target_ind"], w["oa"], w["od"], course_len=w["course_len"]),
               "host_outputs": mpc.step_host(state, w["target_ind"], w["oa"], w["od"], course_len=w["course_len"],
                                             out=mpc.host_outputs(len(state))),
               "c_pageable": _step_host_c(jm, mpc, w, state, lambda s, dt: np.empty(s, dt)),
               "c_pinned": _step_host_c(jm, mpc, w, state, mpc.pinned_empty)}
    finally:
        mpc.set_host_transfer("zero_copy_results")
    for k, a in inputs.items():
        assert np.array_equal(w[k], a), k
    for name, out in got.items():
        for key in KEYS:
            assert np.array_equal(getattr(out, key), getattr(ref, key), equal_nan=True), (name, key)
        for key in ["ox", "oy", "ov", "oyaw"]:           # only defined for solved instances
            assert np.array_equal(getattr(out, key)[solved], getattr(ref, key)[solved]), (name, key)
        assert np.array_equal(out.xref, ref.xref), name


# ---- refusals -----------------------------------------------------------------------------------------------
def test_host_calls_refuse_bad_course_ids_and_a_skip_mask(jm, scene):
    import torch
    JmpcError = jm[3].JmpcError
    mpc, inputs, kw, _ = scene
    B = len(inputs["v"])
    state = np.zeros((B, 4))
    tgt = np.zeros(B, np.int32)

    def step(cid):
        return mpc.step_host(state, tgt, course_id=cid)

    def collide(cid):
        return mpc.collision_host(inputs["agent_idx"], inputs["v"], inputs["obstacles"], course_id=cid, **kw)
    for call, name in ((step, "jmpc_step_host"), (collide, "jmpc_collision_host")):
        for bad in (3, -1):
            cid = inputs["course_id"].copy()
            cid[B // 2] = bad
            with pytest.raises(JmpcError, match=re.escape(f"{name}: course_id out of range")):
                call(cid)
        mask = torch.zeros(B, dtype=torch.int32, device="cuda")
        mpc.set_skip_mask(mask)
        try:
            with pytest.raises(JmpcError, match=re.escape(f"{name}: {SKIP_MSG}")):
                call(inputs["course_id"])
        finally:
            mpc.set_skip_mask(None)
        call(inputs["course_id"])


def test_unknown_transfer_modes_are_refused(jm, scene):
    _cabi = jm[3]
    mpc = scene[0]
    for mode in (3, -1):
        assert mpc._lib.jmpc_set_host_transfer(mpc._h, mode) != 0
        assert _cabi.load().jmpc_last_error().decode() == "jmpc_set_host_transfer: mode must be 0, 1 or 2"
    with pytest.raises(KeyError):
        mpc.set_host_transfer("zero-copy")
    for mode in (0, 2, 1):
        assert mpc._lib.jmpc_set_host_transfer(mpc._h, mode) == 0
