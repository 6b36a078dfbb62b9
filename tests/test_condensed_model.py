"""CPU check of the algorithm the CUDA kernel runs: exact condensing of the reference QP and the predictor-corrector
iteration (oracle/condensed_model.py is the numpy model of both) against the sparse-form oracle."""
import dataclasses

import numpy as np
import pytest

from helpers import default_vector, make_pool, params_from_vector, scaled_err
from oracle import condensed_model as CM
from oracle import mpc_oracle as O
from oracle.qp import solve_qp


@pytest.fixture(scope="module")
def cases():
    from junction_mpc import synth
    out = []
    for w in (synth.make_workload(2, B=12), synth.make_sweep(13, states_per_point=1, max_points=12),
              synth.make_sweep(8, states_per_point=1, max_points=6)):
        base = default_vector(w)
        c = w["courses"][0]
        for k in range(w["B"]):
            p = params_from_vector(base if w["params"] is None else w["params"][k], w["T"])
            n = int(w["course_len"][k])
            r = O.mpc_step(p, w["state"][k], w["oa"][k], w["od"][k], c[:n, 0], c[:n, 1], c[:n, 2], int(w["target_ind"][k]))
            assert r.status == O.STATUS_OPTIMAL
            out.append((p, w["state"][k], r))
    return out


def test_condensing_is_exact(cases):
    """Eliminating the states changes nothing: same optimiser, same objective value (constants included)."""
    for p, x0, r in cases:
        cq = CM.condense(p, r.xref, r.xbar, x0, r.reaches_end)
        u_ref = np.concatenate([r.oa, r.od])
        assert abs(CM.objective(cq, u_ref) - r.cost) <= 1e-9 * max(1.0, abs(r.cost))
        X = CM.states_from_controls(cq, u_ref)
        for got, ref in zip(X, [r.ox, r.oy, r.ov, r.oyaw]):
            np.testing.assert_allclose(got, ref, rtol=0, atol=1e-9)
        n = len(cq.q)
        G, h = np.vstack([cq.A, -cq.A]), np.concatenate([cq.hi, -cq.lo])
        res = solve_qp(cq.P, cq.q, np.zeros((0, n)), np.zeros(0), G, h, c0=cq.c0)
        assert res.ok
        np.testing.assert_allclose(res.z, u_ref, rtol=0, atol=1e-8)


def test_structured_normal_matrix(cases):
    """K = P + A' diag(w) A assembled from the stage structure (suffix-sum block + tridiagonal) equals the dense product."""
    rng = np.random.default_rng(0)
    p, x0, r = cases[0]
    cq = CM.condense(p, r.xref, r.xbar, x0, r.reaches_end)
    T = p.T
    w = rng.uniform(0.1, 1e6, (4, T))
    w[2, T - 1] = 0.0
    dense = np.concatenate([w[0], w[1], w[2][:T - 1], w[3]])
    np.testing.assert_allclose(CM._assemble_K(T, cq.P, w), cq.P + cq.A.T @ (dense[:, None] * cq.A), rtol=1e-12)
    t = rng.normal(size=(4, T))
    t[2, T - 1] = 0.0
    td = np.concatenate([t[0], t[1], t[2][:T - 1], t[3]])
    np.testing.assert_allclose(CM._rows_apply_T(T, t), cq.A.T @ td, atol=1e-12)
    u = rng.normal(size=2 * T)
    z = CM._rows_apply(T, u)
    np.testing.assert_allclose(np.concatenate([z[0], z[1], z[2][:T - 1], z[3]]), cq.A @ u, atol=1e-12)


def test_interior_point_model_meets_the_parity_gate(cases):
    iters = []
    for p, x0, r in cases:
        cq = CM.condense(p, r.xref, r.xbar, x0, r.reaches_end)
        u, it, ok = CM.ipm_solve(cq)
        assert ok and it <= 30
        iters.append(it)
        T = p.T
        assert scaled_err(u[:T], r.oa) <= 1.0 and scaled_err(u[T:], r.od) <= 1.0
        assert abs(CM.objective(cq, u) - r.cost) <= 1e-6 * max(1.0, abs(r.cost))
    assert np.mean(iters) < 14


def test_cumulative_acceleration_form(cases):
    """The unknowns of the CUDA kernel are s_k = a_0 + ... + a_k (csrc/jmpc_step.cuh, step_prep): its Hessian and
    linear term, computed from suffix sums as the kernel does, are E' P E and E' q of the a_k formulation."""
    for p, x0, r in cases:
        cq = CM.condense(p, r.xref, r.xbar, x0, r.reaches_end)
        E = CM.cumulative_transform(p.T)
        P, q = CM.condense_cumulative(p, r.xref, r.xbar, x0, r.reaches_end)
        Pt, qt = E.T @ cq.P @ E, E.T @ cq.q
        assert np.abs(P - Pt).max() <= 1e-11 * np.abs(Pt).max()
        assert np.abs(q - qt).max() <= 1e-11 * max(np.abs(qt).max(), 1.0)
        # same optimiser: the solution in s maps onto the controls
        u_ref = np.concatenate([r.oa, r.od])
        s_ref = np.linalg.solve(E, u_ref)
        np.testing.assert_allclose(s_ref[:p.T], np.cumsum(r.oa), rtol=0, atol=1e-12)


def test_interior_point_iterates_do_not_depend_on_the_unknowns(cases):
    """A linear change of unknowns leaves the rows, the slacks and the multipliers alone, so the predictor-corrector
    iteration in [s; delta] takes the same number of iterations and ends in the same controls as in [a; delta]
    (DESIGN.md section 5: the kernel changed unknowns without changing a single iteration count on config 2)."""
    import dataclasses
    for p, x0, r in cases:
        cq = CM.condense(p, r.xref, r.xbar, x0, r.reaches_end)
        u_a, it_a, ok_a = CM.ipm_solve(cq)
        P, q = CM.condense_cumulative(p, r.xref, r.xbar, x0, r.reaches_end)
        u_s, it_s, ok_s = CM.ipm_solve(dataclasses.replace(cq, P=P, q=q), cumulative=True)
        assert ok_a and ok_s
        assert abs(it_a - it_s) <= 1                      # roundoff may move an exit by one iteration
        np.testing.assert_allclose(u_s, u_a, rtol=0, atol=1e-7)
        T = p.T
        assert scaled_err(u_s[:T], r.oa) <= 1.0 and scaled_err(u_s[T:], r.od) <= 1.0


def _model_against_oracle(args):
    pv, T, state, oa, od, course, n, target = args
    p = params_from_vector(pv, T)
    r = O.mpc_step(p, state, oa, od, course[:n, 0], course[:n, 1], course[:n, 2], int(target))
    assert r.status == O.STATUS_OPTIMAL
    cq = CM.condense(p, r.xref, r.xbar, state, r.reaches_end)
    P, q = CM.condense_cumulative(p, r.xref, r.xbar, state, r.reaches_end)
    u, it, ok, kind = CM.ipm_solve_exit(dataclasses.replace(cq, P=P, q=q), cumulative=True)
    u_or = np.concatenate([r.oa, r.od])
    f_star = CM.objective(cq, u_or)
    # multipliers of the rows active at the oracle's optimum (least squares on P u + q + A_act' y = 0)
    z = cq.A @ u_or
    act = np.flatnonzero(np.minimum(cq.hi - z, z - cq.lo) <= 1e-7)
    y = np.linalg.lstsq(cq.A[act].T, -(cq.P @ u_or + cq.q), rcond=None)[0] if len(act) else np.zeros(0)
    return dict(gap=(CM.objective(cq, u) - f_star) / max(1.0, abs(f_star)), du=float(np.abs(u - u_or).max()),
                exit=kind, ok=ok, iters=it, weakest=float(np.abs(y).min()) if len(y) else np.inf)


def test_interior_point_model_is_as_accurate_as_the_certified_oracle():
    """What the kernel's algorithm delivers, measured against the certified oracle (mpc_oracle + qp.solve_qp) on about
    100 instances each of config 2, sweep points at T = 8 and 25 and the degenerate set (T = 13).  The model iterates
    in the kernel's unknowns with the kernel's tolerances and all four of its exits.

      * cost: (f(u_model) - f*) / max(1, |f*|) within 1e-10 (measured: -1.3e-12 .. 1.8e-12);
      * exits: every solve ends at the strict or the complementarity exit, never at reduced tolerances;
      * controls: within 1e-7 of the oracle's where every row active at the optimum carries a multiplier of at least
        1e-3 (measured: at most 9.9e-9; 392 of the 400 instances).  Where an active row's multiplier vanishes (strict
        complementarity fails: on config 2 the speed row of the last stage, which bounds the sum of all accelerations)
        an interior point approaches the optimum along that row only at the rate of sqrt(mu), so at mu <= 1e-13 the
        last acceleration can be off by ~1e-5 (measured: 1.5e-5 on config 2, 5.7e-7 at T = 8) while the cost is
        within 1e-12.  Those instances are held to 1e-4.

    Iterations: 5 to 20 (measured), every exit strict.

    The GPU test of the kernel against this model (tests/test_gpu_solver_accuracy.py) relies on these figures: its tight
    band belongs to the algorithm, not to luck."""
    from junction_mpc import synth
    sets = {"config2": synth.make_workload(2, B=100), "sweep_T8": synth.make_sweep(8, states_per_point=1, max_points=100),
            "sweep_T25": synth.make_sweep(25, states_per_point=1, max_points=100),
            "degenerate_T13": synth.make_degenerate(13, B=100)}
    with make_pool() as pool:
        for name, w in sets.items():
            base = default_vector(w)
            jobs = [(base if w["params"] is None else w["params"][k], w["T"], w["state"][k], w["oa"][k], w["od"][k],
                     w["courses"][0], int(w["course_len"][k]), int(w["target_ind"][k])) for k in range(w["B"])]
            res = pool.map(_model_against_oracle, jobs)
            gap = np.array([r["gap"] for r in res])
            du = np.array([r["du"] for r in res])
            strict_compl = np.array([r["weakest"] >= 1e-3 for r in res])
            assert all(r["ok"] and r["exit"] in ("strict", "complementarity") for r in res), name
            assert np.abs(gap).max() <= 1e-10, (name, gap.min(), gap.max())
            assert du[strict_compl].max() <= 1e-7, (name, np.sort(du[strict_compl])[-3:])
            assert du.max() <= 1e-4, (name, du.max())
            assert strict_compl.mean() >= 0.9, name
