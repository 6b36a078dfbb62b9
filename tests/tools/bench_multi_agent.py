"""Cost of scenes of MPC-driven vehicles that see each other (BatchedEpisodes(agents_per_scene=4)).

Workload: the intersection's four approaches from the recorded planner courses (tests/golden/planner.npz,
intersection_{1..4}_{1..3}), one vehicle per approach and scene on a random route, 0-8 m along it at 2-5 m/s
(tests/test_gpu_multi_agent.py's scenes), T = 13, outcome record only (no History), max_steps = 400.
  study      16 384 scenes x 4 vehicles: wall time of construction + run() (host clock, run() ends in a device
             synchronise) and control steps per second, median over the rounds after one warm-up round
  exchange   jmpc_scene_exchange alone on the study's final state: CUDA events around 1 000 back-to-back launches,
             per launch, and its share of a loop iteration (study wall / iterations)
  single     for reference, the same 65 536 vehicles alone, each with 3 constant-input obstacles crossing its course
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r6_multi_agent.json).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402

K = 4


def workload(courses, n_scenes, seed=7):
    rng = np.random.default_rng(seed)
    B = n_scenes * K
    cid = (np.arange(B) % K) * 3 + rng.integers(0, 3, B)
    off = rng.integers(0, 96, B)
    state0 = np.empty((B, 4))
    for c in range(len(courses)):
        m = cid == c
        state0[m] = np.stack([courses[c][off[m], 0], courses[c][off[m], 1], np.zeros(m.sum()), courses[c][off[m], 2]],
                             axis=1)
    state0[:, 2] = rng.uniform(2, 5, B)
    obst = np.zeros((B, 3, 6))                   # the single-vehicle reference: 3 constant-input vehicles crossing
    ang = rng.uniform(-np.pi, np.pi, (B, 3))
    obst[:, :, 0] = rng.uniform(-10, 10, (B, 3)) - 25 * np.cos(ang)
    obst[:, :, 1] = rng.uniform(-10, 10, (B, 3)) - 25 * np.sin(ang)
    obst[:, :, 2] = rng.uniform(3, 8, (B, 3))
    obst[:, :, 3] = ang
    obst[:, :, 5] = rng.uniform(-.05, .05, (B, 3))
    return state0, cid, obst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_multi_agent.json"))
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_multi_agent needs a CUDA device")
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
    state0, cid, obst = workload(courses, a.scenes)
    B = len(state0)
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=B)

    def one(mode):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        kw = dict(agents_per_scene=K) if mode == "study" else dict(obstacles=obst.copy())
        ep = BatchedEpisodes(engine, state0, course_id=cid, frame_window=10, margin=margin, max_steps=a.steps,
                             record_history=False, outcomes=True, **kw)
        res = ep.run(max_steps=a.steps)
        return time.perf_counter() - t0, res, ep

    walls = {"study": [], "single": []}
    last = {}
    for r in range(a.rounds + 1):                # round 0 is the warm-up
        for m in (("study", "single") if r % 2 else ("single", "study")):
            wall, res, ep = one(m)
            if r:
                walls[m].append(wall)
                last[m] = (res, ep)
            print(f"round {r} {m}: {wall * 1e3:.1f} ms, {res['iterations']} iterations", flush=True)

    res, ep = last["study"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(20):
        ep._scene_exchange()
    ev0.record()
    for _ in range(a.launches):
        ep._scene_exchange()
    ev1.record()
    torch.cuda.synchronize()
    exchange_us = ev0.elapsed_time(ev1) * 1e3 / a.launches
    med = {m: statistics.median(walls[m]) for m in walls}
    it = int(res["iterations"])
    iter_us = med["study"] * 1e6 / it
    steps = {m: int(last[m][0]["steps"].sum()) for m in walls}
    out_s, out_1 = res["outcomes"], last["single"][0]["outcomes"]
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes x {K} vehicles (intersection approaches 1-4, recorded planner courses, 0-8 m along "
                 f"at 2-5 m/s), T = 13, outcomes only, max_steps = {a.steps}; single: the same {B} vehicles alone with 3 "
                 "constant-input obstacles each; wall = construction + run()",
        rounds=a.rounds,
        study=dict(wall_s=walls["study"], wall_s_median=med["study"], iterations=it, control_steps=steps["study"],
                   control_steps_per_s=steps["study"] / med["study"], iteration_us=iter_us,
                   done_codes=np.bincount(res["done"]).tolist(), cut=int((out_s["cut_steps"] > 0).sum()),
                   contact=int((out_s["first_contact_eval"] >= 0).sum()),
                   within_3m=int((out_s["min_clearance"] < 3.0).sum())),
        exchange=dict(launches=a.launches, B=B, n_obs=K - 1, us_per_launch=exchange_us,
                      bytes_written_per_launch=B * (K - 1) * 48, share_of_iteration=exchange_us / iter_us),
        single=dict(wall_s=walls["single"], wall_s_median=med["single"], iterations=int(last["single"][0]["iterations"]),
                    control_steps=steps["single"], control_steps_per_s=steps["single"] / med["single"],
                    done_codes=np.bincount(last["single"][0]["done"]).tolist(),
                    cut=int((out_1["cut_steps"] > 0).sum())))
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
