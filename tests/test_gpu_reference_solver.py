"""The CUDA step against cvxpy + ECOS, the reference's own solver (SURVEY.md section 8(c) last row).  Runs where
both packages import; otherwise skips with the probe's reason (this image has neither)."""
import json
import os

import numpy as np
import pytest

from helpers import ABS_TOL, REL_TOL, default_vector, params_from_vector, scaled_err
from oracle import reference_solver as RS

pytestmark = pytest.mark.gpu


def _cost_of(out, k):
    return float(out.cost[k])


def test_gpu_matches_ecos_on_frozen_inputs(golden_dir):
    """Frozen config-2 inputs (first 96 instances) and the recorded config-1 episode, solved by ECOS through the
    reference's formulation.  Gate: the north-star tolerances; where ECOS's own tolerance (1e-8 on a cost that is
    almost flat in some directions) leaves a control outside them, the GPU point must be feasible and at least as
    good in the objective, i.e. the discrepancy must be the reference solver's."""
    r = RS.probe()
    if not r["available"]:
        pytest.skip("cvxpy + ECOS not importable here: " + r["reason"])
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    w = synth.make_workload(2, B=96)
    mpc = BatchedMPC(w["courses"], dl=w["dl"], T=w["T"], max_batch=128)
    out = mpc.step_host(w["state"], w["target_ind"], w["oa"], w["od"], course_len=w["course_len"])
    base = default_vector(w)
    worst, loose = 0.0, 0
    for k in range(96):
        p = params_from_vector(base, w["T"])
        c = w["courses"][0][:int(w["course_len"][k])]
        ref = RS.mpc_step_reference_solver(p, w["state"][k], w["oa"][k], w["od"][k], c[:, 0], c[:, 1], c[:, 2],
                                           int(w["target_ind"][k]))
        assert ref.status == int(out.status[k]) == 0
        assert ref.target_ind == int(out.target_ind[k]) and np.array_equal(ref.xref, out.xref[k])
        assert abs(out.cost[k] - ref.cost) <= 1e-4 * abs(ref.cost)
        e = max(scaled_err(out.oa[k], ref.oa), scaled_err(out.od[k], ref.od), scaled_err(out.ov[k], ref.ov),
                scaled_err(out.ox[k], ref.ox), scaled_err(out.oy[k], ref.oy), scaled_err(out.oyaw[k], ref.oyaw))
        worst = max(worst, e)
        if e > 1.0:
            loose += 1
            assert out.cost[k] <= ref.cost + 1e-9 * abs(ref.cost), (k, e)
    report_dir = os.environ.get("JMPC_REPORT_DIR")          # summary only on request: the source tree is never written
    if report_dir:
        with open(os.path.join(report_dir, "r2_reference_solver_parity.json"), "w") as f:
            json.dump({"probe": r, "instances": 96, "worst_scaled_error": worst, "outside_gate_but_better_objective": loose,
                       "gate": {"abs": ABS_TOL, "rel": REL_TOL}}, f, indent=1)
    assert loose <= 96 // 10
