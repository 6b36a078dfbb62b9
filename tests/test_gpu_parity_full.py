"""Full-size parity of the CUDA step with the CPU oracle, run by the driver with `-m gpu` (VERDICT r1 item 1b):

  * config 2 in full (4096 x T=20);
  * 4096-instance batches of configs 3 and 4 (T=13) with the truncated course lengths coming from the flag kernel
    (`collision_host`), as the scenario loop feeds them, and the flags / cut lengths themselves against the
    collision oracle on a subset;
  * config 5: 1024 sweep points per horizon T in {8, 13, 20, 25} (dt in {0.1, 0.2} and all weight axes);
  * config 5's degenerate side set (zero weights, SURVEY.md section 8d): 1024 per horizon, judged on cost and
    predicted states only.

Gates are the north star's (tests/helpers.py).  A summary of what was compared is written to
$JMPC_REPORT_DIR/r2_parity_validation.json when that variable names a directory (profiles/ holds the one of the final
build); the source tree itself is never written."""
import json
import os
import time

import numpy as np
import pytest

from helpers import compare_step, default_vector, oracle_batch
from oracle import collision_oracle as C
from oracle import mpc_oracle as O

pytestmark = pytest.mark.gpu

SUMMARY = {}


@pytest.fixture(scope="module")
def jm():
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    yield synth, BatchedMPC
    report_dir = os.environ.get("JMPC_REPORT_DIR")
    if SUMMARY and report_dir:
        doc = {"gates": {"controls_states": "|d| <= 1e-4 + 1e-3 |ref|", "cost": "1e-4 relative",
                         "target_ind / xref / status / flags / cut lengths": "exact"},
               "oracle": "oracle/mpc_oracle.py + oracle/qp.py (certified optimum; row 8 is not pinned to cvxpy+ECOS, "
                         "see tests/test_gpu_reference_solver.py)",
               "written_by": "tests/test_gpu_parity_full.py", "cases": SUMMARY,
               "total_instances": int(sum(c["instances"] for c in SUMMARY.values()))}
        with open(os.path.join(report_dir, "r2_parity_validation.json"), "w") as f:
            json.dump(doc, f, indent=1)


def _solve(BatchedMPC, w):
    mpc = BatchedMPC(w["courses"], dl=w["dl"], T=w["T"], max_batch=max(w["B"], 64))
    out = mpc.step_host(w["state"], w["target_ind"], w["oa"], w["od"], course_len=w["course_len"],
                        params=w.get("params"))
    return mpc, out


def _record(name, w, out, worst, t_oracle, **extra):
    st, cnt = np.unique(out.status, return_counts=True)
    SUMMARY[name] = dict(instances=int(w["B"]), T=int(w["T"]), worst_scaled_error=float(worst),
                         status_counts={int(a): int(b) for a, b in zip(st, cnt)},
                         solver_iters_mean=float(out.iters.mean()), solver_iters_max=int(out.iters.max()),
                         oracle_seconds=round(t_oracle, 1), **extra)


def test_config2_full(jm):
    synth, BatchedMPC = jm
    w = synth.make_workload(2)
    mpc, out = _solve(BatchedMPC, w)
    t0 = time.time()
    refs = oracle_batch(w, range(w["B"]))
    worst = compare_step(out, refs, range(w["B"]))
    assert (out.status == 0).all()
    _record("config2_4096xT20", w, out, worst, time.time() - t0)


@pytest.mark.parametrize("config", [3, 4])
def test_configs_3_4_with_cut_lengths_from_the_flag_kernel(jm, config):
    synth, BatchedMPC = jm
    w = synth.make_workload(config, B=4096)
    mpc = BatchedMPC(w["courses"], dl=w["dl"], T=w["T"], max_batch=4096)
    geo = C.CarGeometry()
    margin = C.cutoff_margin(geo, w["dl"])
    flag, clen = mpc.collision_host(w["agent_idx"], w["state"][:, 2], w["obstacles"], frame_window=w["frame_window"],
                                    margin=margin)
    assert 0.05 < flag.mean() < 0.95
    # flags and cut lengths against the collision oracle (row 11), every 16th instance
    course = w["courses"][0]
    for k in range(0, 4096, 16):
        f, cut = C.collision_cut(geo, course, int(w["agent_idx"][k]), float(w["state"][k, 2]), w["obstacles"][k], dt=0.2,
                                 frame_window=w["frame_window"], max_accel=2.0, max_speed=30 / 3.6, margin=margin)
        assert int(f) == flag[k] and int(cut) == clen[k], k
    # the step on the truncated courses, searching from the ego index as mpc.target_ind does in the closed loop
    w["course_len"] = clen
    w["target_ind"] = np.minimum(w["target_ind"], clen - 1).astype(np.int32)
    out = mpc.step_host(w["state"], w["target_ind"], w["oa"], w["od"], course_len=clen)
    t0 = time.time()
    refs = oracle_batch(w, range(4096))
    worst = compare_step(out, refs, range(4096))
    assert (out.status == 0).mean() > 0.99
    _record(f"config{config}_4096xT13_cut_by_flag_kernel", w, out, worst, time.time() - t0,
            flag_rate=float(flag.mean()), flags_checked_against_collision_oracle=256, n_obs=int(w["obstacles"].shape[1]))


@pytest.mark.parametrize("T", [8, 13, 20, 25])
def test_config5_sweep_points(jm, T):
    synth, BatchedMPC = jm
    w = synth.make_sweep(T, states_per_point=1, max_points=1024)
    assert set(np.unique(w["params"][:, 0])) == {0.1, 0.2}            # both sample times are in the draw
    mpc, out = _solve(BatchedMPC, w)
    t0 = time.time()
    refs = oracle_batch(w, range(w["B"]))
    worst = compare_step(out, refs, range(w["B"]))
    assert (out.status == 0).all()
    _record(f"config5_sweep_T{T}", w, out, worst, time.time() - t0)


@pytest.mark.parametrize("T", [8, 13, 20, 25])
def test_config5_degenerate_side_set(jm, T):
    """w_perp = 0, w_para = 0, R_* = 0, Rd_* = 0 (the reference's own sweep lists): cost and predicted states."""
    synth, BatchedMPC = jm
    w = synth.make_degenerate(T, B=1024)
    mpc, out = _solve(BatchedMPC, w)
    t0 = time.time()
    refs = oracle_batch(w, range(w["B"]))
    worst = compare_step(out, refs, range(w["B"]), controls=False)
    assert (out.status == 0).all()
    # where the weight that vanished does not touch uniqueness the controls agree as well: report how many do
    ok_controls = 0
    for k, r in enumerate(refs):
        d = max(np.max(np.abs(out.oa[k] - r.oa) / (1e-4 + 1e-3 * np.abs(r.oa))),
                np.max(np.abs(out.od[k] - r.od) / (1e-4 + 1e-3 * np.abs(r.od))))
        ok_controls += int(d <= 1.0)
    _record(f"config5_degenerate_T{T}", w, out, worst, time.time() - t0, judged="cost and predicted states",
            controls_also_inside_gate=ok_controls)
