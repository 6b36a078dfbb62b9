"""Batched motion-primitive A* on the GPU (SURVEY.md section 8f row f4) against searches recorded from the
reference's own MotionPrimitiveSearch / AStar (tests/golden/planner.npz).

Exact: status, number of expansions, the primitive of every edge (i.e. the node path as a sequence of decisions).
Node coordinates, expansion log and trajectory: 1e-9 (sin / cos come from CUDA's libm, numpy's from the host's);
cost: 1e-12 relative."""
import types

import numpy as np
import pytest

from helpers import load_planner_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fx(golden_dir):
    import __graft_entry__ as g
    g.build()
    from junction_mpc import planner as P
    z = load_planner_golden(golden_dir)
    return z, P


def _inputs(z, names):
    g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
    scenes = [[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in names]
    return dict(start=np.stack([g(n, "start") for n in names]), goal_point=np.stack([g(n, "goal_point") for n in names]),
                goal_area=np.stack([g(n, "goal_area") for n in names]),
                allowed_dtheta=np.array([float(g(n, "allowed_dtheta")) for n in names]), scenes=scenes,
                scene_id=np.arange(len(names)), weights=np.stack([g(n, "weights") for n in names]))


def test_all_recorded_searches_in_one_batch(fx):
    z, P = fx
    names = [str(n) for n in z["variants"]]
    assert len(names) >= 32
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
    r = planner.plan(**_inputs(z, names), max_expansions=8192, max_path=32, log=True)
    for b, n in enumerate(names):
        g = lambda k: z[f"{n}/{k}"]            # noqa: E731
        exp = g("expanded")
        if np.isnan(g("cost")):
            # The open list runs empty after ~3900 expansions (the reference raises "No solution found.").  An
            # exhaustive search meets nodes that two different primitive sequences reach: the reference's dict merges
            # them only when their floats are bit-equal, which depends on the last bits of sin / cos (numpy's here,
            # CUDA's there), so the expansion COUNT of an exhaustive search may differ by a fraction of a percent.
            assert r.status[b] == P.STATUS_NO_SOLUTION and np.isnan(r.cost[b]), n
            assert abs(int(r.expansions[b]) - len(exp)) <= 0.02 * len(exp), (n, r.expansions[b], len(exp))
            np.testing.assert_allclose(r.log[b, :100], exp[:100], rtol=0, atol=1e-9, err_msg=n)
            continue
        assert r.expansions[b] == len(exp), n
        np.testing.assert_allclose(r.log[b, :len(exp)], exp, rtol=0, atol=1e-9, err_msg=n)      # the node sequence
        assert r.status[b] == P.STATUS_FOUND, n
        assert abs(r.cost[b] - float(g("cost"))) <= 1e-12 * abs(float(g("cost"))), n
        k = len(g("path"))
        assert r.n_path[b] == k and np.array_equal(r.path_mp[b, :k - 1], g("mp_idx")), n
        np.testing.assert_allclose(r.path[b, :k], g("path"), rtol=0, atol=1e-9, err_msg=n)
        np.testing.assert_allclose(r.trajectory(b), g("trajectory"), rtol=0, atol=1e-9, err_msg=n)
    assert r.kernel_ms > 0


def test_results_do_not_depend_on_batch_composition(fx):
    z, P = fx
    names = [str(n) for n in z["variants"]][:8]
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
    a = planner.plan(**_inputs(z, names), max_path=32)
    rev = names[::-1] * 5
    b = planner.plan(**_inputs(z, rev), max_path=32)
    for i, n in enumerate(rev):
        j = names.index(n)
        assert a.cost[j] == b.cost[i] and np.array_equal(a.trajectory(j), b.trajectory(i)), n


def test_expansion_limit_is_reported(fx):
    z, P = fx
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
    r = planner.plan(**_inputs(z, ["multilane_1_1_2_2"]), max_expansions=50)
    assert r.status[0] == P.STATUS_LIMIT and r.expansions[0] == 50 and np.isnan(r.cost[0])


def test_drop_in_motion_primitive_search(fx):
    """Same constructor and return triple as lib.mp_search_ww_generic.MotionPrimitiveSearch, fed with stand-ins for
    the reference's Scenario / obstacle / primitive objects."""
    z, P = fx
    n = "intersection_1_1"
    hp, hp_n = z[f"{n}/hp"], z[f"{n}/hp_n"]

    class Obst:
        def __init__(self, rows):
            self.rows = rows

        def to_convex(self, margin=0.0):
            assert margin == float(z["car_radius"])
            return self.rows
    area = z[f"{n}/goal_area"]
    scen = types.SimpleNamespace(start=tuple(z[f"{n}/start"]), goal_point=tuple(z[f"{n}/goal_point"]),
                                 goal_area=types.SimpleNamespace(xy1=(area[0], area[1]), xy2=(area[2], area[3])),
                                 allowed_goal_theta_difference=float(z[f"{n}/allowed_dtheta"]),
                                 obstacles=[Obst(hp[k, :hp_n[k]]) for k in range(len(hp_n))])
    car = types.SimpleNamespace(radius=float(z["car_radius"]), circle_centers=z["car_circle_centers"])
    mps = {str(name): types.SimpleNamespace(points=z["mp_points"][k], total_length=float(z["mp_total_length"][k]))
           for k, name in enumerate(z["mp_names"])}
    search = P.MotionPrimitiveSearch(scen, car, mps, margin=car.radius)
    cost, path, traj = search.run(debug=True)
    assert abs(cost - float(z[f"{n}/cost"])) <= 1e-12 * cost and len(path) == len(z[f"{n}/path"])
    assert isinstance(path[0], tuple) and len(search.debug_data) == len(z[f"{n}/expanded"])
    np.testing.assert_allclose(traj, z[f"{n}/trajectory"], rtol=0, atol=1e-9)
    # the planned course drives the controller: planner -> BatchedMPC, one step against the oracle
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from helpers import params_from_vector
    from oracle import mpc_oracle as O
    course = traj.copy()
    synth.smooth_yaw_inplace(course[:, 2])
    dl = float(np.linalg.norm(course[0, :2] - course[1, :2]))
    mpc = BatchedMPC([course], dl=dl, T=13, max_batch=4)
    st = np.array([[course[40, 0] + 0.1, course[40, 1] - 0.1, 3.0, course[40, 2]]])
    out = mpc.step_host(st, np.array([37], np.int32))
    ref = O.mpc_step(params_from_vector(mpc.default_params, 13), st[0], None, None, course[:, 0], course[:, 1], course[:, 2], 37)
    assert out.status[0] == 0 and out.target_ind[0] == ref.target_ind
    np.testing.assert_allclose(out.oa[0], ref.oa, rtol=1e-3, atol=1e-4)


def test_no_solution_raises_like_the_reference(fx):
    z, P = fx
    planner = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
    r = planner.plan(**_inputs(z, ["roundabout_2_3_big"]), max_expansions=8192)
    assert r.status[0] == P.STATUS_NO_SOLUTION
