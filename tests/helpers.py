"""Shared test helpers: run the CPU oracle over workload instances (in parallel) and compare with a StepOutput."""
import os
import sys
from multiprocessing import get_context

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import mpc_oracle as O  # noqa: E402
from junction_mpc.config import MPCConfig, PARAM_INDEX as PI  # noqa: E402

# parity gates of BASELINE.json's north_star
ABS_TOL, REL_TOL, COST_REL = 1e-4, 1e-3, 1e-4


def params_from_vector(v, T, max_iter=1):
    return O.Params(
        T=T, dt=float(v[PI["dt"]]), dl=float(v[PI["dl"]]), L=float(v[PI["L"]]), speed=float(v[PI["speed"]]),
        w_perp=float(v[PI["w_perp"]]), w_para=float(v[PI["w_para"]]), R=(float(v[PI["R_a"]]), float(v[PI["R_d"]])),
        Rd=(float(v[PI["Rd_a"]]), float(v[PI["Rd_d"]])), Q_v_yaw=(float(v[PI["Q_v"]]), float(v[PI["Q_yaw"]])),
        Qf=(float(v[PI["Qf_x"]]), float(v[PI["Qf_y"]]), float(v[PI["Qf_v"]]), float(v[PI["Qf_yaw"]])),
        R_end=(float(v[PI["Rend_a"]]), float(v[PI["Rend_d"]])), max_dsteer=float(v[PI["max_dsteer"]]),
        max_accel=float(v[PI["max_accel"]]), max_decel=float(v[PI["max_decel"]]), max_steer=float(v[PI["max_steer"]]),
        sim_max_speed=float(v[PI["sim_max_speed"]]), min_speed=float(v[PI["min_speed"]]),
        v_ref_min=float(v[PI["v_ref_min"]]), v_ref=float(v[PI["v_ref"]]), v_ref_cut=float(v[PI["v_ref_cut"]]),
        max_iter=max_iter)


def load_planner_golden(golden_dir):
    """tests/golden/planner.npz as a dict.  A trajectory equal to an earlier variant's is stored once; the rows
    (name, stored name) of `aliases` give it back under every name it was recorded under."""
    with np.load(os.path.join(golden_dir, "planner.npz")) as z:
        d = {k: z[k] for k in z.files}
    for name, stored in d.pop("aliases"):
        d[str(name)] = d[str(stored)]
    return d


def default_vector(w, cfg=None):
    cfg = cfg or MPCConfig.default()
    return cfg.with_T(w["T"]).param_vector(dl=w["dl"])


def _one(args):
    pv, T, state, oa, od, warm, course, n, target, max_iter = args
    p = params_from_vector(pv, T, max_iter)
    r = O.mpc_step(p, state, oa if warm else None, od if warm else None, course[:n, 0], course[:n, 1], course[:n, 2],
                   int(target))
    r.qp = None
    return r


def make_pool(processes=None):
    """A worker pool for oracle_batch(..., pool=...); lets a benchmark keep process start-up out of its timed region."""
    return get_context("fork").Pool(processes or min(8, os.cpu_count() or 1))


def oracle_batch(w, idx, processes=None, max_iter=1, warm=None, pool=None):
    """Oracle results for workload instances `idx` (list of StepResult)."""
    base = default_vector(w)
    jobs = []
    for k in idx:
        pv = base if w.get("params") is None else w["params"][k]
        cid = int(w["course_id"][k]) if w.get("course_id") is not None else 0
        wk = True if warm is None else bool(warm[k])
        jobs.append((pv, w["T"], w["state"][k], w["oa"][k], w["od"][k], wk, w["courses"][cid], int(w["course_len"][k]),
                     int(w["target_ind"][k]), max_iter))
    if pool is not None:
        n = pool._processes
        return pool.map(_one, jobs, chunksize=max(1, len(jobs) // (4 * n)))
    processes = processes or min(32, os.cpu_count() or 1)
    if processes == 1 or len(jobs) < 8:
        return [_one(j) for j in jobs]
    with get_context("fork").Pool(processes) as pool:
        return pool.map(_one, jobs, chunksize=max(1, len(jobs) // (4 * processes)))


def scaled_err(got, ref):
    """max over entries of |got - ref| / (ABS_TOL + REL_TOL |ref|): <= 1 means inside the parity gate."""
    got, ref = np.asarray(got, float), np.asarray(ref, float)
    return float(np.max(np.abs(got - ref) / (ABS_TOL + REL_TOL * np.abs(ref)))) if ref.size else 0.0


def compare_step(out, refs, idx, check_cost=True, controls=True):
    """Assert parity of a StepOutput against oracle results; returns the worst scaled error.  `controls=False` judges
    predicted states and cost only (degenerate parameter points, where the optimal controls need not be unique)."""
    worst = 0.0
    for pos, k in enumerate(idx):
        r = refs[pos]
        assert int(out.status[k]) == r.status, f"instance {k}: status {out.status[k]} vs oracle {r.status}"
        if r.status == O.STATUS_INDEX_RULE:
            continue
        assert int(out.target_ind[k]) == r.target_ind, f"instance {k}: target_ind {out.target_ind[k]} vs {r.target_ind}"
        assert np.array_equal(out.xref[k], r.xref), f"instance {k}: xref differs"
        if r.status != O.STATUS_OPTIMAL:
            continue
        fields = [("ox", out.ox[k], r.ox), ("oy", out.oy[k], r.oy), ("ov", out.ov[k], r.ov), ("oyaw", out.oyaw[k], r.oyaw)]
        if controls:
            fields = [("oa", out.oa[k], r.oa), ("od", out.od[k], r.od)] + fields
        for name, got, ref in fields:
            e = scaled_err(got, ref)
            assert e <= 1.0, f"instance {k}: {name} outside tolerance (scaled err {e:.3g})\n got {got}\n ref {ref}"
            worst = max(worst, e)
        if check_cost:
            ce = abs(out.cost[k] - r.cost) / max(abs(r.cost), 1e-12)
            assert ce <= COST_REL, f"instance {k}: cost {out.cost[k]} vs {r.cost}"
    return worst
