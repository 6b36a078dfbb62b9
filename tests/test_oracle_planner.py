"""The planner restatement (oracle/planner_oracle.py) against searches recorded from the reference's own
MotionPrimitiveSearch / AStar (tests/golden/planner.npz, made by tests/golden/make_golden.py --planner)."""
import numpy as np
import pytest

from helpers import load_planner_golden
from oracle import planner_oracle as PO


@pytest.fixture(scope="module")
def fx(golden_dir):
    z = load_planner_golden(golden_dir)
    planner = PO.Planner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
    return z, planner


def test_collision_points_of_the_primitives(fx):
    z, planner = fx
    assert len(z["variants"]) >= 32
    for got, ref in zip(planner.cc, z["mp_collision_points"]):
        assert np.array_equal(got, ref)


def test_every_recorded_search_is_reproduced(fx):
    z, planner = fx
    for name in z["variants"]:
        g = lambda k: z[f"{name}/{k}"]            # noqa: E731
        r = planner.plan(g("start"), g("goal_point"), g("goal_area"), float(g("allowed_dtheta")), g("hp"), g("hp_n"),
                         g("weights"))
        if np.isnan(g("cost")):
            assert r.status == PO.STATUS_NO_SOLUTION, name
        else:
            assert r.status == PO.STATUS_FOUND and abs(r.cost - float(g("cost"))) <= 1e-12 * abs(float(g("cost"))), name
            assert np.array_equal(r.mp_idx, g("mp_idx")), name
            assert np.array_equal(r.path, g("path")), name
            assert np.array_equal(r.trajectory, g("trajectory")), name
        assert np.array_equal(r.expanded, g("expanded")), name        # the node sequence, in expansion order
