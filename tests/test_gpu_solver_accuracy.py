"""Accuracy and iteration counts of the CUDA step's interior-point solve against its numpy model (GPU).

The north-star parity gates (tests/helpers.py: controls within 1e-4 + 1e-3 |ref|, cost within 1e-4 relative, at most
40 iterations) leave three to four orders of magnitude between what they accept and what the kernel's algorithm
delivers.  This module closes that gap.  Per instance it runs the certified oracle (oracle/mpc_oracle.py +
oracle/qp.py), condenses the oracle's QP in both unknowns (CM.condense, CM.condense_cumulative: same xref, xbar and
end flags), and runs `CM.ipm_solve_exit(..., cumulative=True)`, the float64 model of the kernel's Mehrotra iteration with
its start point, centring, fraction-to-the-boundary rule and all four exits.  The kernel runs one linearisation pass.

Per instance, with f the objective of the oracle's condensed QP and f* = f(u_oracle):

  gap    (f(u_kernel) - f*) / max(1, |f*|), so the kernel's own cost arithmetic is not trusted (its reported cost is
         checked against f(u_kernel) separately);
  du     max |u_kernel - u_model| over the controls [a; delta];
  diter  kernel iterations - model iterations.

Gates, per case:

  0. every instance the oracle solves and the model solves, the kernel solves (reports OPTIMAL);
  1. no gap below -1e-9 (the kernel cannot beat the certified optimum unless it is infeasible or the oracle is wrong);
  2. the tight band gap <= 1e-9 and du <= 1e-6: at most N_LOOSE[case] instances outside it;
  3. inside the tight band |diter| <= 1 everywhere, diter == 0 on at least EXACT[case] of the instances;
  4. the kernel's iterations summed over the case exceed the model's by at most 0.5 %;
  5. the degenerate set (zero weights: the optimal controls need not be unique) is judged on gap and iterations only.

N_LOOSE and EXACT are set from the B200 run recorded in profiles/r9_solver_accuracy.json (see the numbers there and
beside the tables below): N_LOOSE is twice the measured count outside the band (at least 4), EXACT the measured
fraction of exact iteration counts minus 0.01.

`test_the_gates_fail_on_a_loose_solver` runs an engine with mu_tol = 1e-9 (a runtime option) on the config 2 batch and
checks that gates 2 and 3 both reject it, so the gates are shown to bite.

When JMPC_REPORT_DIR names a directory the per-case distributions are written to r9_solver_accuracy.json there."""
import dataclasses
import json
import os
import subprocess
import time

import numpy as np
import pytest

from helpers import default_vector, make_pool, params_from_vector
from oracle import collision_oracle as C
from oracle import condensed_model as CM
from oracle import mpc_oracle as O

pytestmark = pytest.mark.gpu

GAP_FLOOR = -1e-9          # gate 1
GAP_TIGHT = 1e-9           # gate 2
DU_TIGHT = 1e-6
ITER_SUM_EXCESS = 0.005    # gate 4
COST_REL = 1e-9            # the kernel's reported cost against f(u_kernel), relative to max(1, |f|)

# Gate 2: instances allowed outside the tight band.  Measured on the B200: none in any case (largest du 2.5e-8 on
# config 2, at most 6.4e-9 elsewhere; largest gap 3.1e-11), so every case gets the floor of 4.
N_LOOSE = {name: 4 for name in (
    "config2_4096xT20", "config3_4096xT13_cut_by_flag_kernel", "config4_4096xT13_cut_by_flag_kernel",
    "config5_sweep_T8", "config5_sweep_T13", "config5_sweep_T20", "config5_sweep_T25",
    "config5_degenerate_T8", "config5_degenerate_T13", "config5_degenerate_T20", "config5_degenerate_T25",
    "generic_T5", "generic_T10", "generic_T31")}
# Gate 3: fraction of the instances inside the band with the model's exact iteration count, the measured fraction
# minus 0.01.  Measured: 4094 / 4096 on config 2 (two solves one iteration shorter), 254 / 256 at T = 31 (one solve one
# iteration longer where the model's factorisation breaks down, one shorter), every instance elsewhere.
EXACT = {name: 0.99 for name in N_LOOSE}
EXACT["config2_4096xT20"] = 0.9895
EXACT["generic_T31"] = 0.9822

SUMMARY = {}


def _device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    import torch
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q}


@pytest.fixture(scope="module")
def jm():
    import __graft_entry__ as g
    g.build()
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    pool = make_pool(min(32, os.cpu_count() or 1))
    yield synth, BatchedMPC, pool
    pool.close()
    pool.join()
    report_dir = os.environ.get("JMPC_REPORT_DIR")
    if SUMMARY and report_dir:
        doc = {"device": _device_info(),
               "written_by": "tests/test_gpu_solver_accuracy.py",
               "reference": "oracle/condensed_model.ipm_solve_exit(cumulative=True) on the condensed QP of the certified oracle "
                            "(oracle/mpc_oracle.py + oracle/qp.py); one linearisation pass",
               "gates": {"gap_floor": GAP_FLOOR, "tight_band": {"gap": GAP_TIGHT, "du": DU_TIGHT},
                         "iteration_sum_excess": ITER_SUM_EXCESS, "cost_rel": COST_REL,
                         "n_loose": N_LOOSE, "exact_iteration_fraction": EXACT},
               "cases": SUMMARY}
        with open(os.path.join(report_dir, "r9_solver_accuracy.json"), "w") as f:
            json.dump(doc, f, indent=1)


def _job(args):
    """Oracle step, condensed QP in both unknowns, the model's solve; f at each set of kernel controls."""
    pv, T, state, oa, od, course, n, target, u_kernels = args
    p = params_from_vector(pv, T)
    r = O.mpc_step(p, state, oa, od, course[:n, 0], course[:n, 1], course[:n, 2], int(target))
    if r.status != O.STATUS_OPTIMAL:
        return None
    cq = CM.condense(p, r.xref, r.xbar, state, r.reaches_end)
    P, q = CM.condense_cumulative(p, r.xref, r.xbar, state, r.reaches_end)
    u, it, ok, kind = CM.ipm_solve_exit(dataclasses.replace(cq, P=P, q=q), cumulative=True)
    u_or = np.concatenate([r.oa, r.od])
    return dict(f_star=CM.objective(cq, u_or), f_model=CM.objective(cq, u), u_model=u, u_oracle=u_or, iters=it,
                ok=ok, exit=kind, f_kernel=[CM.objective(cq, uk) for uk in u_kernels])


def _evaluate(pool, w, outs):
    """Per-instance reference data of workload `w` for the kernel outputs `outs` (one StepOutput per engine)."""
    base = default_vector(w)
    jobs = []
    for k in range(w["B"]):
        pv = base if w.get("params") is None else w["params"][k]
        jobs.append((pv, w["T"], w["state"][k], w["oa"][k], w["od"][k], w["courses"][0], int(w["course_len"][k]),
                     int(w["target_ind"][k]), [np.concatenate([o.oa[k], o.od[k]]) for o in outs]))
    return pool.map(_job, jobs, chunksize=max(1, len(jobs) // (8 * pool._processes)))


def _measure(ev, out, which=0):
    """Arrays over the instances both sides solved: gap, du (kernel - model), diter, cost error, model exits; and the
    instances the model solves but the kernel reports as failed."""
    keep = [k for k, e in enumerate(ev) if e is not None and int(out.status[k]) == 0]
    failed = [k for k, e in enumerate(ev) if e is not None and e["ok"] and int(out.status[k]) != 0]
    f_star = np.array([ev[k]["f_star"] for k in keep])
    f_ker = np.array([ev[k]["f_kernel"][which] for k in keep])
    scale = np.maximum(1.0, np.abs(f_star))
    u_ker = np.array([np.concatenate([out.oa[k], out.od[k]]) for k in keep])
    return dict(
        idx=np.array(keep, int),
        gap=(f_ker - f_star) / scale,
        gap_model=np.array([ev[k]["f_model"] - ev[k]["f_star"] for k in keep]) / scale,
        du=np.abs(u_ker - np.array([ev[k]["u_model"] for k in keep])).max(axis=1),
        du_oracle=np.abs(u_ker - np.array([ev[k]["u_oracle"] for k in keep])).max(axis=1),
        diter=out.iters[keep].astype(int) - np.array([ev[k]["iters"] for k in keep]),
        iters=out.iters[keep].astype(int), model_iters=np.array([ev[k]["iters"] for k in keep]),
        cost_err=np.abs(out.cost[keep] - f_ker) / np.maximum(1.0, np.abs(f_ker)),
        exit=np.array([ev[k]["exit"] for k in keep]),
        not_compared=int(len(ev) - len(keep)), kernel_failed=np.array(failed, int))


def _tight(m, controls):
    return (m["gap"] <= GAP_TIGHT) & ((m["du"] <= DU_TIGHT) if controls else True)


def _quantiles(x):
    qs = (0.0, 0.5, 0.9, 0.99, 0.999, 1.0)
    return {f"q{q:g}": float(np.quantile(x, q)) for q in qs} if len(x) else {}


def _judge(name, w, m, controls=True, seconds=0.0):
    tight = _tight(m, controls)
    inside = m["diter"][tight]
    loose = np.flatnonzero(~tight)
    ex, cnt = np.unique(m["exit"], return_counts=True)
    dv, dc = np.unique(m["diter"], return_counts=True)
    SUMMARY[name] = dict(
        T=int(w["T"]), instances=int(w["B"]), compared=int(len(m["gap"])), not_compared=m["not_compared"],
        kernel_failed_where_model_solves=[int(k) for k in m["kernel_failed"]],
        judged="gap and iterations" if not controls else "gap, controls and iterations",
        gap=_quantiles(m["gap"]), gap_model=_quantiles(m["gap_model"]), du_model=_quantiles(m["du"]),
        du_oracle=_quantiles(m["du_oracle"]), cost_err=_quantiles(m["cost_err"]),
        model_exits={str(a): int(b) for a, b in zip(ex, cnt)},
        diter_histogram={int(a): int(b) for a, b in zip(dv, dc)},
        outside_tight_band=int(len(loose)),
        outside_tight_band_model_exits={str(a): int(b) for a, b in zip(*np.unique(m["exit"][loose], return_counts=True))},
        outside_tight_band_examples=[dict(instance=int(m["idx"][j]), gap=float(m["gap"][j]), du=float(m["du"][j]),
                                          du_oracle=float(m["du_oracle"][j]), iters=int(m["iters"][j]),
                                          model_iters=int(m["model_iters"][j]), model_exit=str(m["exit"][j]))
                                     for j in loose[:8]],
        exact_iteration_fraction=float(np.mean(inside == 0)) if len(inside) else 1.0,
        inside_band_max_abs_diter=int(np.abs(inside).max()) if len(inside) else 0,
        kernel_iterations=int(m["iters"].sum()), model_iterations=int(m["model_iters"].sum()),
        n_loose_gate=N_LOOSE.get(name), exact_fraction_gate=EXACT.get(name), reference_seconds=round(seconds, 1))
    s = SUMMARY[name]
    assert s["compared"] >= 0.98 * s["instances"], s["not_compared"]
    assert not s["kernel_failed_where_model_solves"], f"{name}: the kernel fails solves the model completes"
    assert m["gap"].min() >= GAP_FLOOR, f"{name}: kernel below the certified optimum by {-m['gap'].min():.3g}"
    assert m["cost_err"].max() <= COST_REL, f"{name}: reported cost off f(u_kernel) by {m['cost_err'].max():.3g}"
    assert len(loose) <= N_LOOSE[name], f"{name}: {len(loose)} instances outside the tight band: {s['outside_tight_band_examples']}"
    assert s["inside_band_max_abs_diter"] <= 1, f"{name}: diter histogram {s['diter_histogram']}"
    assert s["exact_iteration_fraction"] >= EXACT[name], f"{name}: exact iteration counts on {s['exact_iteration_fraction']:.4f}"
    assert s["kernel_iterations"] <= (1 + ITER_SUM_EXCESS) * s["model_iterations"], (s["kernel_iterations"],
                                                                                       s["model_iterations"])


def _engine(BatchedMPC, w, **kw):
    return BatchedMPC(w["courses"], dl=w["dl"], T=w["T"], max_batch=max(w["B"], 64), linearisation_iters=1,
                      max_T=max(w["T"], 25), **kw)


def _step(mpc, w):
    return mpc.step_host(w["state"], w["target_ind"], w["oa"], w["od"], course_len=w["course_len"], params=w.get("params"))


@pytest.fixture(scope="module")
def config2(jm):
    """The config 2 batch through the default engine and through one with mu_tol = 1e-9, one reference pass for both."""
    synth, BatchedMPC, pool = jm
    w = synth.make_workload(2)
    out = _step(_engine(BatchedMPC, w), w)
    loose = _step(_engine(BatchedMPC, w, mu_tol=1e-9), w)
    t0 = time.time()
    ev = _evaluate(pool, w, [out, loose])
    return w, out, loose, ev, time.time() - t0


def test_config2_full(config2):
    w, out, _, ev, sec = config2
    _judge("config2_4096xT20", w, _measure(ev, out), seconds=sec)


@pytest.mark.parametrize("config", [3, 4])
def test_configs_3_4_with_cut_lengths_from_the_flag_kernel(jm, config):
    synth, BatchedMPC, pool = jm
    w = synth.make_workload(config, B=4096)
    mpc = _engine(BatchedMPC, w)
    margin = C.cutoff_margin(C.CarGeometry(), w["dl"])
    _, clen = mpc.collision_host(w["agent_idx"], w["state"][:, 2], w["obstacles"], frame_window=w["frame_window"],
                                 margin=margin)
    w["course_len"] = clen
    w["target_ind"] = np.minimum(w["target_ind"], clen - 1).astype(np.int32)
    out = _step(mpc, w)
    t0 = time.time()
    ev = _evaluate(pool, w, [out])
    _judge(f"config{config}_4096xT13_cut_by_flag_kernel", w, _measure(ev, out), seconds=time.time() - t0)


@pytest.mark.parametrize("T", [8, 13, 20, 25])
def test_config5_sweep_points(jm, T):
    synth, BatchedMPC, pool = jm
    w = synth.make_sweep(T, states_per_point=1, max_points=1024)
    out = _step(_engine(BatchedMPC, w), w)
    t0 = time.time()
    ev = _evaluate(pool, w, [out])
    _judge(f"config5_sweep_T{T}", w, _measure(ev, out), seconds=time.time() - t0)


@pytest.mark.parametrize("T", [8, 13, 20, 25])
def test_config5_degenerate_side_set(jm, T):
    synth, BatchedMPC, pool = jm
    w = synth.make_degenerate(T, B=1024)
    out = _step(_engine(BatchedMPC, w), w)
    t0 = time.time()
    ev = _evaluate(pool, w, [out])
    _judge(f"config5_degenerate_T{T}", w, _measure(ev, out), controls=False, seconds=time.time() - t0)


@pytest.mark.parametrize("T", [5, 10, 31])
def test_generic_horizons(jm, T):
    """Horizons without a compile-time specialisation run the generic (runtime-T) kernel."""
    synth, BatchedMPC, pool = jm
    course = synth.load_course("roundabout")
    w = synth.make_states(np.random.default_rng(T), course, 256, T)
    w.update(T=T, courses=[course], params=None, B=256, dl=float(np.linalg.norm(course[0, :2] - course[1, :2])))
    out = _step(BatchedMPC([course], dl=w["dl"], T=T, max_batch=256, max_T=31, linearisation_iters=1), w)
    t0 = time.time()
    ev = _evaluate(pool, w, [out])
    _judge(f"generic_T{T}", w, _measure(ev, out), seconds=time.time() - t0)


def test_the_gates_fail_on_a_loose_solver(config2):
    """mu_tol = 1e-9 stops the kernel one to five iterations early: gate 2 must flag far more instances than it
    allows, and gate 3 must find almost no exact iteration counts inside the band."""
    w, _, loose, ev, _ = config2
    m = _measure(ev, loose, which=1)
    tight = _tight(m, True)
    inside = m["diter"][tight]
    s = SUMMARY["self_check_config2_mu_tol_1e-9"] = dict(
        compared=int(len(m["gap"])), outside_tight_band=int((~tight).sum()),
        exact_iteration_fraction=float(np.mean(inside == 0)) if len(inside) else 1.0,
        du_model=_quantiles(m["du"]), gap=_quantiles(m["gap"]),
        diter_histogram={int(a): int(b) for a, b in zip(*np.unique(m["diter"], return_counts=True))})
    # measured on the B200: 1026 instances outside the band, and none of the 3070 inside it with the model's count
    assert s["outside_tight_band"] > 50 * N_LOOSE["config2_4096xT20"], s
    assert s["exact_iteration_fraction"] < 0.5, s
