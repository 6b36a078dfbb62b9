"""Scenes of several MPC-driven vehicles, CPU side: the argument checks of BatchedEpisodes(agents_per_scene=...), the
done codes of include/jmpc.h against Python, and hand-built cases of the numpy scene-exchange oracle
(oracle/scene_exchange.py)."""
import math
import os
import re

import numpy as np
import pytest

from oracle import scene_exchange as SX

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = math.radians(45.0)


def test_done_enum_matches_python():
    from junction_mpc import _cabi
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        header = f.read()
    body = re.sub(r"/\*.*?\*/", "", re.search(r"enum jmpc_done \{(.*?)\};", header, re.S).group(1), flags=re.S)
    codes = dict((n, int(v)) for n, v in re.findall(r"JMPC_DONE_([A-Z_]+)\s*=\s*(\d+)", body))
    assert codes == dict(RUNNING=_cabi.DONE_RUNNING, GOAL=_cabi.DONE_GOAL, INDEX_RULE=_cabi.DONE_INDEX_RULE,
                         NO_COURSE=_cabi.DONE_NO_COURSE, MATE_NO_COURSE=_cabi.DONE_MATE_NO_COURSE)
    assert codes["MATE_NO_COURSE"] == 4
    assert set(SX.NEVER_STEPPED) == {_cabi.DONE_NO_COURSE, _cabi.DONE_MATE_NO_COURSE}


def test_scene_argument_checks():
    from junction_mpc.episodes import outcome_setup, scene_setup
    assert scene_setup(8, 1, 3, False) == 3                  # one vehicle per scene: today's slots
    assert scene_setup(8, 1, 2, True) == 2                   # recordings stay usable without scenes
    assert scene_setup(8, 4, 0, False) == 3 and scene_setup(8, 4, 5, False) == 8
    assert scene_setup(9, 9, 0, False) == 8
    with pytest.raises(ValueError, match="whole number of scenes"):
        scene_setup(10, 4, 0, False)
    with pytest.raises(ValueError, match="exceed the 8 obstacle slots"):
        scene_setup(8, 4, 6, False)
    with pytest.raises(ValueError, match="exceed the 8 obstacle slots"):
        scene_setup(10, 10, 0, False)
    with pytest.raises(ValueError, match="obstacle_script cannot be combined"):
        scene_setup(8, 2, 1, True)
    for bad in (0, -2, 1.5, True, "2"):
        with pytest.raises(ValueError, match="integer >= 1"):
            scene_setup(8, bad, 0, False)
    assert scene_setup(8, np.int64(2), 0, False) == 1
    # the slot count feeds the outcome checks unchanged: record_obstacles still needs outcomes
    with pytest.raises(ValueError, match="needs outcomes"):
        outcome_setup(False, True, scene_setup(8, 4, 0, False))


def _hist(rows):
    """rows [R][B] of (x, y, yaw, v, delta, a) -> History [R, B, 8]."""
    h = np.full((len(rows), len(rows[0]), 8), np.nan)
    for i, row in enumerate(rows):
        for b, r in enumerate(row):
            if r is not None:
                x, y, yaw, v, d, a = r
                h[i, b] = [x, y, yaw, v, 0.2 * (i + 2), d, a, 0.1]
    return h


def test_first_evaluation_reports_start_states_without_controls():
    state0 = np.array([[0.0, 1.0, 2.0, 0.3], [5.0, 6.0, 7.0, -0.4]])
    rows = SX.mate_rows(state0, np.zeros((0, 2, 8)), [0, 0], [0, 0], MS, 2, 1)
    assert rows.shape == (1, 2, 1, 6)
    assert rows[0, 0, 0].tolist() == [5.0, 6.0, 7.0, -0.4, 0.0, 0.0]
    assert rows[0, 1, 0].tolist() == [0.0, 1.0, 2.0, 0.3, 0.0, 0.0]


def test_parked_mate_after_goal_and_failed_solve_and_steer_clamp():
    # vehicle 0: two steps, the second a failed solve (a = MAX_DECEL = -5, delta kept), then done = 1
    # vehicle 1: three steps, the last with delta beyond MAX_STEER; vehicle 2: never stepped (done = 4)
    state0 = np.array([[0.0, 0.0, 1.0, 0.0], [10.0, 0.0, 2.0, 1.0], [20.0, 0.0, 0.0, 2.0]])
    h = _hist([[(0.2, 0.0, 0.01, 1.2, 0.05, 1.0), (11.0, 0.1, 1.1, 2.5, -0.2, 2.0), None],
               [(0.4, 0.0, 0.02, 0.2, 0.05, -5.0), (12.0, 0.2, 1.2, 3.0, 0.1, 2.5), None],
               [None, (13.0, 0.3, 1.3, 3.5, 2.0, -1.0), None]])
    rows = SX.mate_rows(state0, h, steps=[2, 3, 0], done=[1, 0, 4], max_steer=MS, k=3, n_eval=5)
    assert rows.shape == (5, 3, 2, 6)
    v0 = rows[:, 1, 0]                                      # vehicle 0 as vehicle 1 sees it (slot 0)
    assert v0[0].tolist() == [0.0, 0.0, 1.0, 0.0, 0.0, 0.0]
    assert v0[1].tolist() == [0.2, 0.0, 1.2, 0.01, 1.0, 0.05]
    assert v0[2].tolist() == [0.4, 0.0, 0.2, 0.02, -5.0, 0.05]          # failed solve: MAX_DECEL, previous delta
    for e in (3, 4):                                                      # parked at its last pose
        assert v0[e].tolist() == [0.4, 0.0, 0.0, 0.02, 0.0, 0.0]
    v1 = rows[:, 0, 0]                                      # vehicle 1 as vehicle 0 sees it (slot 0)
    assert v1[3].tolist() == [13.0, 0.3, 3.5, 1.3, -1.0, MS]             # steer clamped to +MAX_STEER
    assert v1[4].tolist() == [13.0, 0.3, 0.0, 1.3, 0.0, 0.0]
    assert np.array_equal(rows[:, 2, 1], v1)                # vehicle 2 sees vehicle 1 in slot 1 (itself skipped)
    v2 = rows[:, 0, 1]                                      # the never-stepped vehicle: parked from evaluation 0
    for e in range(5):
        assert v2[e].tolist() == [20.0, 0.0, 0.0, 2.0, 0.0, 0.0]
    # per-vehicle MAX_STEER: the clamp is the mate's own
    rows = SX.mate_rows(state0, h, [2, 3, 0], [1, 0, 4], np.array([MS, 0.5, MS]), 3, 4)
    assert rows[3, 0, 0, 5] == 0.5 and rows[1, 0, 0, 5] == -0.2
    neg = _hist([[(1.0, 0.0, 0.0, 1.0, -3.0, 0.0)]])
    assert SX.vehicle_rows([[0.0, 0.0, 1.0, 0.0]], neg, [1], [0], MS, 2)[1, 0, 5] == -MS


def test_oracle_argument_errors():
    with pytest.raises(ValueError):
        SX.mate_rows(np.zeros((3, 4)), np.zeros((1, 3, 8)), [0, 0, 0], [0, 0, 0], MS, 2, 1)
    with pytest.raises(ValueError):
        SX.vehicle_rows(np.zeros((2, 4)), np.zeros((1, 2, 8)), [2, 0], [0, 0], MS, 1)
