"""Per-episode outcome record, CPU side: the header's column enum against the Python table, hand-built cases of the
numpy oracle (oracle/episode_outcomes.py), and the host-side argument checks of BatchedEpisodes' outcome options."""
import math
import os
import re

import numpy as np
import pytest

from oracle import episode_outcomes as EO
from oracle.collision_oracle import CarGeometry

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEO = CarGeometry()
R2 = 2 * GEO.radius
DT, L, MS = 0.2, 2.86, math.radians(45.0)


def test_outcome_enum_matches_python_table():
    from junction_mpc.episodes import OUTCOME_LEN, OUTCOME_NAMES
    with open(os.path.join(ROOT, "include", "jmpc.h")) as f:
        header = f.read()
    body = re.search(r"enum jmpc_outcome \{(.*?)\};", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"JMPC_(?:O_)?([A-Z_]+)", body)
    assert names[-1] == "NOUTCOME"
    assert [n.lower() for n in names[:-1]] == list(OUTCOME_NAMES)
    assert list(EO.COLUMNS) == list(OUTCOME_NAMES)
    assert int(re.search(r"#define JMPC_OUTCOME_LEN (\d+)", header).group(1)) == OUTCOME_LEN > len(OUTCOME_NAMES)


def _row(x, y, yaw, v, delta=0.0, a=0.0, dev=0.1):
    return [x, y, yaw, v, 0.0, delta, a, dev]


def _parked(x, y, yaw=0.0):
    return [x, y, 0.0, yaw, 0.0, 0.0]


def test_touching_at_exactly_2r_is_contact():
    # ego at the origin heading +x, obstacle beside it heading +x: the circles line up, the nearest pairs are
    # (front, front) and (rear, rear) at dist = sqrt(yo * yo) = yo exactly
    for yo, want in ((R2, True), (np.nextafter(R2, np.inf), False), (np.nextafter(R2, 0.0), True)):
        track = np.array([[_parked(0.0, yo)]])
        out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], np.zeros((0, 8)), [], track, DT, L, MS)
        assert out["contact_evals"] == int(want)
        assert (out["first_contact_eval"], out["first_contact_obs"]) == ((0, 0) if want else (-1, -1))
        assert out["min_clearance"] == yo - R2
        assert out["min_clearance_eval"] == 0 and out["min_clearance_obs"] == 0


def test_tie_for_the_minimum_first_evaluation_and_lowest_obstacle_win():
    # two obstacles at the same pose relative to the ego, at evaluations 1 and 2 (ego does not move)
    hist = np.array([_row(0.0, 0.0, 0.0, 0.0), _row(0.0, 0.0, 0.0, 0.0)])
    far = _parked(1000.0, 0.0)
    near = _parked(10.0, 0.0)
    track = np.array([[far, far], [far, near], [near, near]])
    out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], hist, [0, 0], track, DT, L, MS)
    assert out["min_clearance_eval"] == 1 and out["min_clearance_obs"] == 1
    assert out["first_contact_eval"] == -1 and out["contact_evals"] == 0
    track = np.array([[near, near], [near, near], [near, near]])
    out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], hist, [0, 0], track, DT, L, MS)
    assert out["min_clearance_eval"] == 0 and out["min_clearance_obs"] == 0
    # contact in two evaluations with the second obstacle only, then both
    on = _parked(0.0, 0.0)
    track = np.array([[far, far], [far, on], [on, on]])
    out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], hist, [1, -1], track, DT, L, MS)
    assert out["first_contact_eval"] == 1 and out["first_contact_obs"] == 1 and out["contact_evals"] == 2
    assert out["min_clearance"] == -R2 and out["min_clearance_eval"] == 1 and out["min_clearance_obs"] == 1
    assert out["cut_steps"] == 1 and out["limit_steps"] == 1


def test_one_step_has_no_jerk_or_steer_rate():
    hist = np.array([_row(1.0, 0.0, 0.05, 3.0, delta=2.0, a=-1.5, dev=0.25)])
    out = EO.episode_outcomes([0.0, 0.0, 2.5, 0.0], hist, [0], np.zeros((2, 0, 6)), DT, L, MS)
    assert out["max_abs_jerk"] == 0.0 and out["max_abs_steer_rate"] == 0.0
    assert out["max_abs_accel"] == 1.5 and out["distance"] == 1.0
    assert out["max_abs_lat_accel"] == abs(2.5 * ((2.5 / L) * math.tan(MS)))       # steer clamped, speed BEFORE the step
    assert out["max_xref_dev"] == 0.25 == out["sum_xref_dev"] and out["failed_solves"] == 0
    assert out["min_clearance"] == math.inf and out["min_clearance_eval"] == -1 and out["first_contact_eval"] == -1


def test_failed_solve_is_left_out_of_the_deviation_columns():
    hist = np.array([_row(0.5, 0.0, 0.0, 1.0, delta=0.1, a=1.0, dev=0.3),
                     _row(1.0, 0.0, 0.0, 0.0, delta=0.1, a=-5.0, dev=np.nan),
                     _row(1.5, 0.0, 0.0, 0.5, delta=-0.2, a=2.5, dev=0.2)])
    out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], hist, [0, 0, 0], np.zeros((4, 0, 6)), DT, L, MS)
    assert out["failed_solves"] == 1
    assert out["max_xref_dev"] == 0.3 and out["sum_xref_dev"] == 0.3 + 0.2
    assert out["max_abs_jerk"] == 7.5 / DT and out["max_abs_steer_rate"] == pytest.approx(0.3 / DT, rel=1e-15)
    assert out["distance"] == 1.5 and out["max_abs_accel"] == 5.0


def test_empty_episode():
    out = EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], np.zeros((0, 8)), [], np.zeros((1, 0, 6)), DT, L, MS)
    assert out == dict(min_clearance=math.inf, min_clearance_eval=-1, min_clearance_obs=-1, first_contact_eval=-1,
                       first_contact_obs=-1, contact_evals=0, cut_steps=0, limit_steps=0, failed_solves=0,
                       max_abs_accel=0.0, max_abs_jerk=0.0, max_abs_steer_rate=0.0, max_abs_lat_accel=0.0,
                       max_xref_dev=0.0, sum_xref_dev=0.0, distance=0.0)
    with pytest.raises(ValueError):
        EO.episode_outcomes([0.0, 0.0, 0.0, 0.0], np.zeros((2, 8)), [0, 0], np.zeros((2, 0, 6)), DT, L, MS)


def test_outcome_argument_checks():
    from junction_mpc.episodes import OUTCOME_INT, OUTCOME_LEN, OUTCOME_NAMES, outcome_columns, outcome_setup
    assert outcome_setup(False, False, 3) is False
    assert outcome_setup(True, False, 0) is True and outcome_setup(True, True, 8) is True
    with pytest.raises(ValueError, match="needs outcomes"):
        outcome_setup(False, True, 2)
    with pytest.raises(ValueError, match="at most 8"):
        outcome_setup(True, False, 9)
    rec = np.arange(3 * OUTCOME_LEN, dtype=np.float64).reshape(3, OUTCOME_LEN)
    cols = outcome_columns(rec)
    assert list(cols) == list(OUTCOME_NAMES)
    for k, name in enumerate(OUTCOME_NAMES):
        assert cols[name].shape == (3,) and np.array_equal(cols[name], rec[:, k])
        assert cols[name].dtype == (np.int64 if name in OUTCOME_INT else np.float64)
    assert {"min_clearance_eval", "first_contact_obs", "contact_evals", "failed_solves"} <= OUTCOME_INT
    assert "min_clearance" not in OUTCOME_INT and "distance" not in OUTCOME_INT
    with pytest.raises(ValueError):
        outcome_columns(rec[:, :5])
