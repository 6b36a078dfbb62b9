"""Shared plans (BatchedEpisodes(share_plans=True)), CPU side: the planned obstacle predictor of oracle/shared_plans.py
against the collision oracle's constant-input one, hand-built cases of the mate-plan oracle (shared_plans.mate_plans), the
argument checks, and the register / spill report of the new kernels from ptxas for sm_100a."""
import math
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import collision_oracle as C
from oracle import shared_plans as SP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "av-simulation-at-intersections_b200", "csrc", "jmpc.cu")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
MS = math.radians(45.0)


@pytest.mark.parametrize("plan_len", [1, 12, 35, 40])
def test_constant_plan_is_the_constant_input_predictor(plan_len):
    rng = np.random.default_rng(plan_len)
    for _ in range(20):
        x, y, v, yaw = rng.uniform(-30, 30), rng.uniform(-30, 30), rng.uniform(0, 10), rng.uniform(-np.pi, np.pi)
        a, steer = rng.uniform(-5, 2), rng.uniform(-MS, MS)
        ref = C.predict_obstacle(x, y, v, yaw, a, steer, dt=0.2, L=2.86)
        got = SP.predict_obstacle_plan(x, y, v, yaw, [(a, steer)] * plan_len, dt=0.2, L=2.86)
        assert ref.shape == (35, 4) and np.array_equal(got, ref)


def test_plan_inputs_per_step_and_last_input_held():
    rng = np.random.default_rng(3)
    plan = np.stack([rng.uniform(-5, 2, 12), rng.uniform(-MS, MS, 12)], axis=1)
    held = np.concatenate([plan, np.repeat(plan[-1:], 23, axis=0)])
    a = SP.predict_obstacle_plan(1.0, 2.0, 4.0, 0.3, plan, dt=0.2, L=2.86)
    assert np.array_equal(a, SP.predict_obstacle_plan(1.0, 2.0, 4.0, 0.3, held, dt=0.2, L=2.86))
    # a longer plan than the 35 frames: the inputs past the horizon are never used
    longer = np.concatenate([held, rng.uniform(-1, 1, (5, 2))])
    assert np.array_equal(a, SP.predict_obstacle_plan(1.0, 2.0, 4.0, 0.3, longer, dt=0.2, L=2.86))
    # step k: the position moves with the old speed / heading, then v += a_k dt, then yaw with the new speed
    x, y, v, yaw = 1.0, 2.0, 4.0, 0.3
    for k in range(3):
        x += v * math.cos(yaw) * 0.2
        y += v * math.sin(yaw) * 0.2
        v += plan[k, 0] * 0.2
        yaw += (v / 2.86) * math.tan(plan[k, 1]) * 0.2
        assert a[k].tolist() == [x, y, yaw, k * 0.2]
    with pytest.raises(ValueError):
        SP.predict_obstacle_plan(0, 0, 1, 0, [], dt=0.2, L=2.86)


def test_collision_cut_with_constant_plans_equals_without():
    path = np.stack([np.linspace(-40, 40, 801), np.zeros(801), np.zeros(801)], axis=1)
    geo = C.CarGeometry()
    obst = [(5.0, -20.0, 4.0, np.pi / 2, 0.5, 0.0), (30.0, 3.0, 2.0, np.pi, -1.0, 0.1)]
    kw = dict(dt=0.2, frame_window=10, max_accel=2.0, max_speed=30 / 3.6, margin=8)
    ref = C.collision_cut(geo, path, 10, 3.0, obst, **kw)
    assert ref[0]
    assert SP.collision_cut(geo, path, 10, 3.0, obst, plans=[[o[4:6]] * 7 for o in obst], **kw) == ref
    assert SP.collision_cut(geo, path, 10, 3.0, obst, plans=[None, [obst[1][4:6]]], **kw) == ref
    # the crossing vehicle plans to stop well before the ego's path: no collision any more
    assert SP.collision_cut(geo, path, 10, 3.0, obst[:1], plans=[[(-5.0, 0.0)] * 12], **kw)[0] is False
    with pytest.raises(ValueError, match="one entry"):
        SP.collision_cut(geo, path, 10, 3.0, obst, plans=[None], **kw)


def _snapshot():
    """3 vehicles of one scene with T = 4: vehicle 0 runs with a plan, vehicle 1 has warm = 0, vehicle 2 is parked."""
    oa = np.array([[1.0, 0.5, -0.5, -1.0], [2.0, 2.0, 2.0, 2.0], [0.3, 0.3, 0.3, 0.3]])
    od = np.array([[0.1, 0.2, 1.5, -0.3], [0.4, 0.4, 0.4, 0.4], [0.2, 0.2, 0.2, 0.2]])
    rows = np.zeros((3, 2, 6))                      # rows[b, slot] = (x, y, v, yaw, a, steer) of b's mates
    row = {0: [0.0, 0.0, 3.0, 0.0, 1.0, 0.1], 1: [10.0, 0.0, 2.0, 1.0, -5.0, -MS], 2: [20.0, 0.0, 0.0, 2.0, 0.0, 0.0]}
    for b in range(3):
        for slot, m in enumerate(q for q in range(3) if q != b):
            rows[b, slot] = row[m]
    return oa, od, rows, row


def test_mate_plans_hand_cases():
    oa, od, rows, row = _snapshot()
    got = SP.mate_plans(oa, od, [1, 0, 1], [0, 0, 1], rows, MS, 3)
    assert got.shape == (3, 2, 3, 2)
    # a valid plan: the rest of it, steer beyond MAX_STEER clamped (od[0, 2] = 1.5)
    assert got[1, 0].tolist() == [[0.5, 0.2], [-0.5, MS], [-1.0, -0.3]]
    assert np.array_equal(got[2, 0], got[1, 0])
    # warm = 0 (a failed solve): the row's (MAX_DECEL, clamped steer) repeated; before the first step the row's (0, 0)
    assert got[0, 0].tolist() == [[-5.0, -MS]] * 3 and got[2, 1].tolist() == [[-5.0, -MS]] * 3
    rows0 = rows.copy()
    rows0[:, :, 4:6] = 0.0
    first = SP.mate_plans(oa, od, [0, 0, 0], [0, 0, 0], rows0, MS, 3)
    assert (first == 0.0).all()
    # parked (done != 0): (0, 0) from its row, whatever its warm flag says
    assert got[0, 1].tolist() == [[0.0, 0.0]] * 3 and got[1, 1].tolist() == [[0.0, 0.0]] * 3
    # the clamp is the mate's own MAX_STEER
    got = SP.mate_plans(oa, od, [1, 0, 1], [0, 0, 1], rows, np.array([1.0, MS, MS]), 3)
    assert got[1, 0, 1].tolist() == [-0.5, 1.0]
    # extras after the mate slots are not read; two scenes are independent
    wide = np.concatenate([rows, np.full((3, 1, 6), np.nan)], axis=1)
    assert np.array_equal(SP.mate_plans(oa, od, [1, 0, 1], [0, 0, 1], wide, MS, 3)[:, :, :, :],
                          SP.mate_plans(oa, od, [1, 0, 1], [0, 0, 1], rows, MS, 3))
    two = SP.mate_plans(np.tile(oa, (2, 1)), np.tile(od, (2, 1)), [1, 0, 1, 1, 1, 1], [0, 0, 1, 0, 0, 0],
                        np.tile(rows, (2, 1, 1)), MS, 3)
    assert np.array_equal(two[:3], SP.mate_plans(oa, od, [1, 0, 1], [0, 0, 1], rows, MS, 3))
    assert two[3, 0].tolist() == [[2.0, 0.4]] * 3


def test_mate_plans_argument_errors():
    oa, od, rows, _ = _snapshot()
    with pytest.raises(ValueError):
        SP.mate_plans(oa, od, [1] * 3, [0] * 3, rows, MS, 1)
    with pytest.raises(ValueError):
        SP.mate_plans(oa[:, :1], od[:, :1], [1] * 3, [0] * 3, rows, MS, 3)
    with pytest.raises(ValueError):
        SP.mate_plans(oa, od, [1] * 3, [0] * 3, rows, MS, 2)


def test_share_plans_argument_checks():
    from junction_mpc.config import NPARAM, PARAM_INDEX
    from junction_mpc.episodes import plan_share_setup
    assert plan_share_setup(False, 1, None) is False
    assert plan_share_setup(False, 4, None) is False
    assert plan_share_setup(True, 4, None) is True
    with pytest.raises(ValueError, match="needs agents_per_scene > 1"):
        plan_share_setup(True, 1, None)
    params = np.zeros((8, NPARAM))
    params[:, PARAM_INDEX["dt"]] = 0.2
    params[:, PARAM_INDEX["dl"]] = np.arange(8)             # other parameters may differ within a scene
    assert plan_share_setup(True, 4, params) is True
    params[5, PARAM_INDEX["dt"]] = 0.1
    with pytest.raises(ValueError, match="one dt per scene: scene 1"):
        plan_share_setup(True, 4, params)
    assert plan_share_setup(True, 2, params[:4]) is True
    assert plan_share_setup(False, 4, params) is False      # without the option a scene may mix dt as before


_PROPS = re.compile(r"Function properties for (\S+)\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                    r"(\d+) bytes spill loads\s*\n[^\n]*Used (\d+) registers")


@pytest.fixture(scope="module")
def resources(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip(f"nvcc not found at {NVCC}")
    out = tmp_path_factory.mktemp("ptxas") / "jmpc.cubin"
    cmd = [NVCC, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xptxas", "-v", "-o", str(out), SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    return {m.group(1): (int(m.group(3)), int(m.group(4)), int(m.group(5))) for m in _PROPS.finditer(res.stderr)}


def _one(resources, pattern):
    hits = [v for k, v in resources.items() if re.fullmatch(pattern, k)]
    assert len(hits) == 1, (pattern, sorted(resources))
    return hits[0]


def test_new_kernels_are_spill_free(resources):
    for pattern in (r"_ZN4jmpc16collision_kernelILb1EEEvNS_13CollisionArgsE", r"_ZN4jmpc18scene_plans_kernel.*"):
        stores, loads, _ = _one(resources, pattern)
        assert (stores, loads) == (0, 0), pattern


def test_constant_input_collision_kernel_unchanged(resources):
    stores, loads, regs = _one(resources, r"_ZN4jmpc16collision_kernelILb0EEEvNS_13CollisionArgsE")
    assert (stores, loads) == (0, 0) and regs <= 64
