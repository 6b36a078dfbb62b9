"""Host-side argument checks of the planned-episode path (no GPU): plan_id range, the one-margin rule, input shapes."""
import math

import numpy as np
import pytest


def test_plan_episode_setup_checks():
    from junction_mpc.episodes import plan_episode_setup
    r = 2.0 / 2 ** 0.5
    ok, dl = np.array([1, 0, 1], np.int32), np.array([0.083, np.nan, 0.083])
    pid, margin = plan_episode_setup(ok, dl, None, 3, r)
    assert pid.dtype == np.int32 and pid.tolist() == [0, 1, 2]
    assert margin == 4 * math.ceil(r / 0.083) == 72                   # mpc_intersection.py:87-88
    pid, margin = plan_episode_setup(ok, dl, np.zeros(30, np.int64), 3, r)
    assert len(pid) == 30 and margin == 72
    assert plan_episode_setup(ok, dl, [1, 1], 3, r)[1] == 0            # no usable course driven: no margin needed
    for bad in ([3], [-1, 0], [], [[0, 1]], [0.5]):
        with pytest.raises(ValueError):
            plan_episode_setup(ok, dl, np.array(bad), 3, r)
    with pytest.raises(ValueError, match="disagree"):
        plan_episode_setup(np.ones(2, np.int32), np.array([0.083, 0.05]), None, 2, r)
    # an unusable course's dl does not take part in the margin
    assert plan_episode_setup(np.array([1, 0]), np.array([0.083, 0.05]), None, 2, r)[1] == 72
    with pytest.raises(ValueError):
        plan_episode_setup(ok[:2], dl, None, 3, r)


def test_plan_input_shapes():
    from junction_mpc.planner import pack_plan_inputs
    box = [np.array([[1, 0, -1], [-1, 0, -1], [0, 1, -1], [0, -1, -1]], float)]
    start, goal, area, allowed, w, sid, (n_scenes, max_obs, hp, hp_n, n_obs) = pack_plan_inputs(
        np.zeros((2, 3)), [0, 10, 0], [-1, 9, 1, 11], 0.5, [box], scene_id=[0, 0])
    assert goal.shape == (2, 3) and area.shape == (2, 4) and allowed.shape == (2,) and w.shape == (2, 9)
    assert sid.dtype == np.int32 and hp.shape == (1, 1, 8, 3) and hp_n.tolist() == [[4]] and n_obs.tolist() == [1]
    with pytest.raises(ValueError):
        pack_plan_inputs(np.zeros((2, 3)), [0, 10, 0], np.zeros((2, 3)), 0.5, [box])          # goal_area is [B, 4]
    with pytest.raises(ValueError):
        pack_plan_inputs(np.zeros((2, 3)), [0, 10, 0], [-1, 9, 1, 11], 0.5, [[np.zeros((9, 3))]])   # <= 8 half-planes
