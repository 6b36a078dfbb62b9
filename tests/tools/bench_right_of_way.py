"""Right-of-way rules in scenes of MPC-driven vehicles (BatchedEpisodes(right_of_way=...)): the r6 / r7 intersection
study with no rule, "fixed" and "first_come", each with share_plans off and on.

Workload: bench_multi_agent.workload -- 16 384 scenes x 4 vehicles on the intersection's recorded planner courses,
T = 13, outcome record only, max_steps = 400; first_come with junction = (0, 0, --radius) for every scene (the
right-turn courses come within 7.24 m of the centre and the straight ones within 3.0 m, so every course enters r > 7.24).
  study    the six modes, one warm-up round then --rounds rounds in rotating order: wall time of construction + run()
           (host clock, run() ends in a device synchronise), control steps, and the outcome summary of each mode
  causes   the vehicles still driving at 400 steps of each rule, sorted by what cuts their course at the end:
           a parked mate, a moving mate the rule makes them yield to, or nothing, from jmpc_collision_masked with
           the parked / yielded slots alone; how many of them have a mate parked at its goal on their own exit lane
           (course ends within 5 m: two of the recorded routes end on each exit lane, 0.8-2.4 m apart); their failed
           solves
  kernels  on the state after --mid iterations of a first_come run (share_plans off), without a skip mask: CUDA events
           around --launches back-to-back launches of jmpc_right_of_way (both rules), jmpc_collision,
           jmpc_collision_masked with an all-ones mask and with that state's real masks
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r8_right_of_way.json) and, with --dump, a few scenes with vehicles still driving (record_obstacles).
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
from bench_shared_plans import summary  # noqa: E402

MODES = [(rule, plans) for rule in (None, "fixed", "first_come") for plans in (False, True)]


def mode_name(rule, plans):
    return f"{rule or 'none'}{'_shared_plans' if plans else ''}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--radius", type=float, default=10.0)
    ap.add_argument("--mid", type=int, default=40)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_right_of_way.json"))
    ap.add_argument("--dump", default=None, help="npz path for a few scenes with vehicles still driving")
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_right_of_way needs a CUDA device")
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
    closest = [float(np.hypot(c[:, 0], c[:, 1]).min()) for c in courses]
    if max(closest) >= a.radius:
        raise SystemExit(f"--radius {a.radius} misses a course: closest approaches {closest}")
    junction = (0.0, 0.0, a.radius)
    ends = np.array([c[-1, :2] for c in courses])
    state0, cid, _ = workload(courses, a.scenes)
    B = len(state0)
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=B)

    def make(rule, plans, **kw):
        extra = dict(junction=junction) if rule == "first_come" else {}
        return BatchedEpisodes(engine, state0, course_id=cid, frame_window=10, margin=margin, max_steps=a.steps,
                               record_history=False, outcomes=True, agents_per_scene=K, share_plans=plans,
                               right_of_way=rule, **extra, **kw)

    def one(rule, plans):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ep = make(rule, plans)
        res = ep.run(max_steps=a.steps)
        return time.perf_counter() - t0, res, ep

    walls = {mode_name(*m): [] for m in MODES}
    last = {}
    for r in range(a.rounds + 1):                # round 0 is the warm-up
        order = MODES[r % len(MODES):] + MODES[:r % len(MODES)]
        for m in order:
            wall, res, ep = one(*m)
            name = mode_name(*m)
            if r:
                walls[name].append(wall)
                last[name] = (res, ep)
            print(f"round {r} {name}: {wall * 1e3:.1f} ms, {res['iterations']} iterations, still driving "
                  f"{int((res['done'] == 0).sum())}", flush=True)

    flag = torch.zeros(B, dtype=torch.int32, device=engine.device)
    clen = torch.zeros(B, dtype=torch.int32, device=engine.device)

    def masked(ep, mask):
        engine.collision(ep.agent_idx, ep.state[:, 2].contiguous(), ep.scene_obs, ep.frame_window, ep.margin, flag,
                         clen, course_id=ep.course_id, horizon_s=ep.horizon_s, plans=ep.scene_plans,
                         n_planned=K - 1, consider=torch.as_tensor(mask, dtype=torch.int32, device=ep.dev))
        torch.cuda.synchronize()
        return flag.cpu().numpy().copy()

    causes = {}
    dumps = {}
    for rule in ("fixed", "first_come"):
        for plans in (False, True):
            name = mode_name(rule, plans)
            res, ep = last[name]
            done = res["done"]
            still = np.flatnonzero(done == 0)
            consider = ep.consider.cpu().numpy().astype(np.int64)
            d = done.reshape(-1, K)
            parked_bits = np.zeros(B, np.int64)
            for b in range(B):
                s, j = divmod(b, K)
                for slot, m in enumerate(q for q in range(K) if q != j):
                    if d[s, m]:
                        parked_bits[b] |= 1 << slot
            mate_bits = (1 << (K - 1)) - 1
            # what cuts the course at the last evaluation: a parked mate, then a mate the rule makes it yield to
            by_parked = masked(ep, parked_bits) == 1          # the study has no extras: the mate slots are all
            yielded = consider & mate_bits & ~parked_bits
            by_yield = masked(ep, yielded) == 1
            out = res["outcomes"]
            own_exit = np.zeros(B, bool)                       # a mate parked at its goal on b's exit lane
            for b in still:
                s = b // K
                for m in range(s * K, s * K + K):
                    if m != b and done[m] == 1 and np.hypot(*(ends[cid[m]] - ends[cid[b]])) < 5.0:
                        own_exit[b] = True
            c = dict(still_driving=int(len(still)),
                     blocked_by_parked_mate=int(by_parked[still].sum()),
                     yielding_to_a_moving_mate=int((by_yield & ~by_parked)[still].sum()),
                     not_cut_at_the_end=int((~by_parked & ~by_yield)[still].sum()),
                     mate_parked_on_own_exit_lane=int(own_exit[still].sum()),
                     with_failed_solves=int((out["failed_solves"][still] > 0).sum()),
                     standing=int((np.abs(res["state"][still, 2]) < 0.05).sum()),
                     scenes_with_a_vehicle_still_driving=int((d == 0).any(axis=1).sum()))
            causes[name] = c
            print(name, c, flush=True)
            if a.dump and not plans and len(still):
                dumps[rule] = np.unique(still // K)[:4]

    # a few stuck scenes, re-run alone with record_obstacles
    dump_info = {}
    if a.dump:
        arrays = {}
        for rule, scenes in dumps.items():
            idx = np.concatenate([np.arange(s * K, (s + 1) * K) for s in scenes])
            extra = dict(junction=junction) if rule == "first_come" else {}
            ep = BatchedEpisodes(engine, state0[idx], course_id=cid[idx], frame_window=10, margin=margin,
                                 max_steps=a.steps, record_history=True, outcomes=True, record_obstacles=True,
                                 agents_per_scene=K, right_of_way=rule, **extra)
            res = ep.run(max_steps=a.steps)
            arrays.update({f"{rule}/episodes": idx, f"{rule}/course_id": cid[idx], f"{rule}/done": res["done"],
                           f"{rule}/steps": res["steps"], f"{rule}/history": res["history"],
                           f"{rule}/obstacle_history": res["obstacle_history"]})
            dump_info[rule] = dict(scenes=scenes.tolist(), done=res["done"].tolist(), steps=res["steps"].tolist(),
                                   final_speed=np.round(res["state"][:, 2], 3).tolist(),
                                   final_xy=np.round(res["state"][:, :2], 2).tolist())
        os.makedirs(os.path.dirname(os.path.abspath(a.dump)), exist_ok=True)
        np.savez_compressed(a.dump, **arrays)

    # kernel times on a mid-run state
    ep = make("first_come", False)
    for _ in range(a.mid):
        ep.iterate()
    torch.cuda.synchronize()
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream().cuda_stream
    p = ep._p
    v = ep.state[:, 2].contiguous()
    ones = torch.full((B,), -1, dtype=torch.int32, device=ep.dev)
    real = ep.consider.clone()
    prio = torch.as_tensor(np.arange(B) % K, dtype=torch.float64, device=ep.dev)
    scratch = torch.empty(B, dtype=torch.int32, device=ep.dev)

    def collision(mask):
        return lambda: engine.collision(ep.agent_idx, v, ep.scene_obs, ep.frame_window, ep.margin, flag, clen,
                                        course_id=ep.course_id, horizon_s=ep.horizon_s, consider=mask)

    def rule_call(rule):
        code = _cabi.ROW_FIRST_COME if rule == "first_come" else _cabi.ROW_FIXED
        return lambda: _cabi.check(lib.jmpc_right_of_way(h, B, K, code, p(ep.agent_idx), p(ep.done), None, p(ep.zone),
                                                         p(prio), p(scratch), stream), "jmpc_right_of_way")

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

    real_np = real.cpu().numpy().astype(np.int64)
    kernels = {}
    for rep in range(2):                         # alternating, twice
        for name, fn in (("collision", collision(None)), ("collision_masked_all_ones", collision(ones)),
                         ("collision_masked_real", collision(real)), ("right_of_way_first_come", rule_call("first_come")),
                         ("right_of_way_fixed", rule_call("fixed"))):
            kernels.setdefault(name, []).append(timed(fn))
    kernels = {k: dict(us_per_launch=v, us_per_launch_min=min(v)) for k, v in kernels.items()}
    ref = kernels["collision"]["us_per_launch_min"]
    for k in ("collision_masked_all_ones", "collision_masked_real"):
        kernels[k]["ratio_to_collision"] = kernels[k]["us_per_launch_min"] / ref
    moving = ep.done.cpu().numpy() == 0
    mate_bits = (1 << (K - 1)) - 1
    kernels["collision_masked_real"]["mate_slots_ignored_share"] = float(
        (K - 1 - np.array([bin(int(m) & mate_bits).count("1") for m in real_np[moving]])).sum() / ((K - 1) * moving.sum()))
    modes = {}
    for m in MODES:
        name = mode_name(*m)
        s = summary(last[name][0])
        med = statistics.median(walls[name])
        s.update(wall_s=walls[name], wall_s_median=med, control_steps_per_s=s["control_steps"] / med,
                 iteration_us=med * 1e6 / s["iterations"])
        modes[name] = s
    for k in ("right_of_way_first_come", "right_of_way_fixed"):
        kernels[k]["share_of_iteration"] = kernels[k]["us_per_launch_min"] / modes["first_come"]["iteration_us"]
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes x {K} vehicles (intersection approaches 1-4, recorded planner courses, 0-8 m along "
                 f"at 2-5 m/s), T = 13, outcomes only, max_steps = {a.steps}; first_come junction = (0, 0, {a.radius}) "
                 f"(closest approach of the courses to the centre {max(closest):.2f} m); wall = construction + run(); "
                 f"kernels: B = {B}, {K - 1} mate slots, no skip mask, state after {a.mid} iterations of first_come",
        rounds=a.rounds, modes=modes, still_driving_causes=causes, kernels=kernels)
    if dump_info:
        out["dumped_scenes"] = dump_info
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
