"""Scenes whose vehicles predict each other along their shared MPC plans (BatchedEpisodes(share_plans=True)) against the
constant-input prediction of the mates' last applied controls (share_plans=False).

Workload: bench_multi_agent.workload -- 16 384 scenes x 4 vehicles on the intersection's recorded planner courses,
T = 13, outcome record only, max_steps = 400.
  study    share_plans off and on, alternating, after one warm-up round: wall time of construction + run() (host clock,
           run() ends in a device synchronise), iterations, control steps/s, and the outcome summary of each mode
  kernels  on the final state of the last 'on' run, without a skip mask (every instance evaluated): CUDA events around
           1 000 back-to-back launches each of jmpc_collision, jmpc_collision_planned with the real plans and with
           constant plans (the rows' (a, steer) repeated) on the same rows, and jmpc_scene_plans
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r7_shared_plans.json).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests"),
          os.path.dirname(os.path.abspath(__file__))):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402

from bench_multi_agent import K, workload  # noqa: E402


def summary(res):
    out, done, steps = res["outcomes"], res["done"], res["steps"]
    return dict(iterations=int(res["iterations"]), control_steps=int(steps.sum()), done_codes=np.bincount(done).tolist(),
                still_driving=int((done == 0).sum()), cut=int((out["cut_steps"] > 0).sum()),
                contact=int((out["first_contact_eval"] >= 0).sum()), within_3m=int((out["min_clearance"] < 3.0).sum()),
                median_steps_to_goal=float(np.median(steps[done == 1])) if (done == 1).any() else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_shared_plans.json"))
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_shared_plans needs a CUDA device")
    gpu = dict(name=torch.cuda.get_device_name(0))
    try:
        gpu["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # noqa: BLE001
        gpu["power_limit"] = f"unavailable ({e})"
    z = load_planner_golden(os.path.join(ROOT, "tests", "golden"))
    courses = []
    for i in (1, 2, 3, 4):
        for j in (1, 2, 3):
            c = np.array(z[f"intersection_{i}_{j}/trajectory"], dtype=np.float64)
            synth.smooth_yaw_inplace(c[:, 2])
            courses.append(c)
    dl = float(np.linalg.norm(courses[0][0, :2] - courses[0][1, :2]))
    margin = C.cutoff_margin(C.CarGeometry(), dl)
    state0, cid, _ = workload(courses, a.scenes)
    B = len(state0)
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=B)

    def one(mode):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ep = BatchedEpisodes(engine, state0, course_id=cid, frame_window=10, margin=margin, max_steps=a.steps,
                             record_history=False, outcomes=True, agents_per_scene=K, share_plans=mode == "on")
        res = ep.run(max_steps=a.steps)
        return time.perf_counter() - t0, res, ep

    walls = {"off": [], "on": []}
    last = {}
    for r in range(a.rounds + 1):                # round 0 is the warm-up
        for m in (("on", "off") if r % 2 else ("off", "on")):
            wall, res, ep = one(m)
            if r:
                walls[m].append(wall)
                last[m] = (res, ep)
            print(f"round {r} {m}: {wall * 1e3:.1f} ms, {res['iterations']} iterations", flush=True)

    res, ep = last["on"]
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream().cuda_stream
    n_obs, plan_len = ep.n_obs, ep.T - 1
    flag = torch.zeros(B, dtype=torch.int32, device=ep.dev)
    clen = torch.zeros(B, dtype=torch.int32, device=ep.dev)
    const_plans = ep.scene_obs[:, :K - 1, None, 4:6].expand(B, K - 1, plan_len, 2).contiguous()
    v = ep.state[:, 2].contiguous()
    p = ep._p

    def collision(plans):
        return lambda: engine.collision(ep.agent_idx, v, ep.scene_obs, ep.frame_window, ep.margin, flag, clen,
                                        course_id=ep.course_id, horizon_s=ep.horizon_s, plans=plans, n_planned=K - 1)

    def plans_call():
        _cabi.check(lib.jmpc_scene_plans(h, B, K, ep.T, p(ep.oa), p(ep.od), p(ep.warm), p(ep.done), None,
                                         p(ep.scene_obs), n_obs, p(ep.scene_plans), stream), "jmpc_scene_plans")

    def timed(fn):
        for _ in range(20):
            fn()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(a.launches):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) * 1e3 / a.launches

    kernels = {}
    for rep in range(2):                         # alternating, twice
        for name, fn in (("collision", collision(None)), ("collision_planned", collision(ep.scene_plans)),
                         ("collision_planned_constant", collision(const_plans)), ("scene_plans", plans_call)):
            kernels.setdefault(name, []).append(timed(fn))
    kernels = {k: dict(us_per_launch=v, us_per_launch_min=min(v)) for k, v in kernels.items()}
    ref = kernels["collision"]["us_per_launch_min"]
    for k in ("collision_planned", "collision_planned_constant"):
        kernels[k]["ratio_to_collision"] = kernels[k]["us_per_launch_min"] / ref
    med = {m: statistics.median(walls[m]) for m in walls}
    modes = {}
    for m in walls:
        s = summary(last[m][0])
        s.update(wall_s=walls[m], wall_s_median=med[m], control_steps_per_s=s["control_steps"] / med[m],
                 iteration_us=med[m] * 1e6 / s["iterations"])
        modes[m] = s
    kernels["scene_plans"]["share_of_iteration"] = kernels["scene_plans"]["us_per_launch_min"] / modes["on"]["iteration_us"]
    kernels["scene_plans"]["bytes_written_per_launch"] = B * (K - 1) * plan_len * 16
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes x {K} vehicles (intersection approaches 1-4, recorded planner courses, 0-8 m along "
                 f"at 2-5 m/s), T = 13, outcomes only, max_steps = {a.steps}; wall = construction + run(); kernels: "
                 f"B = {B}, {K - 1} mate slots, plan_len = {plan_len}, no skip mask, final state of the last 'on' run",
        rounds=a.rounds, share_plans_off=modes["off"], share_plans_on=modes["on"], kernels=kernels)
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
