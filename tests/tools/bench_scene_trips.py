"""Trips through scene slots (BatchedEpisodes.from_trips): junction throughput, entry delay and travel time of the
recorded intersection under Poisson demand, and the cost of the trips pass.

Workload: --scenes scenes on the 12 recorded intersection courses (approaches 1-4 x 3 turns, loaded as
bench_scene_lifetimes does); every trip starts at its course's point 0 at 4 m/s; T = 13; first_come with junction
(0, 0, --radius) and shared plans; outcome record only; --steps iterations (dt = 0.2 s); seeded Poisson arrivals per
approach (poisson_trips, seed 12).
  runs     k = 8 slots at 150 / 300 / 450 / 600 veh/h per approach, and k = 4 at 300 veh/h.  One warm-up run
           (k = 8, 40 iterations), then each run once: wall time of construction + run() (host clock, run() ends in a
           device synchronise), control steps (every trip's executed steps), and per run the trips admitted /
           completed / pending, throughput per junction, mean and p95 entry delay and travel time (iterations),
           slot_waits / blocked_waits and contacts per 1000 admitted trips
  pass     on the state after --mid iterations of the k = 8, 600 veh/h run: CUDA events around --launches
           back-to-back launches of jmpc_scene_trips at that iteration (the first may admit or close trips, the others
           walk the same pending trips and add blocked waits)
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r12_scene_trips.json).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402

RUNS = [("k8_150", 8, 150.0), ("k8_300", 8, 300.0), ("k8_450", 8, 450.0), ("k8_600", 8, 600.0), ("k4_300", 4, 300.0)]


def stats(x):
    x = np.asarray(x, np.float64)
    return dict(mean=float(x.mean()), p95=float(np.percentile(x, 95))) if len(x) else dict(mean=None, p95=None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--radius", type=float, default=10.0)
    ap.add_argument("--mid", type=int, default=300)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_scene_trips.json"))
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes, poisson_trips
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene_trips needs a CUDA device")
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
    routes = [[(3 * g + r, tuple(courses[3 * g + r][0, :3])) for r in range(3)] for g in range(4)]
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=a.scenes * 8)
    dt = float(engine.dt)

    demand = {rate: poisson_trips(a.scenes, routes, rate, dt, a.steps, 4.0, seed=12) for rate in {r[2] for r in RUNS}}

    def make(k, rate, steps):
        trips = demand[rate]
        return BatchedEpisodes.from_trips(engine, trips, a.scenes, agents_per_scene=k, frame_window=10, margin=margin,
                                          max_steps=steps, record_history=False, outcomes=True, share_plans=True,
                                          right_of_way="first_come", junction=(0.0, 0.0, a.radius)), trips

    make(8, 600.0, 40)[0].run(max_steps=40)      # warm-up (the demand is drawn before the timed runs)
    runs = {}
    for name, k, rate in RUNS:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ep, trips = make(k, rate, a.steps)
        t1 = time.perf_counter()
        res = ep.run(max_steps=a.steps)
        wall = time.perf_counter() - t0
        run_s = time.perf_counter() - t1
        tab = res["trips"]
        adm = tab["entry"] >= 0
        done = tab["done"] == 1
        hours = res["iterations"] * dt / 3600.0
        control = int(tab["steps"][adm].sum())
        runs[name] = dict(
            k=k, rate_per_hour_per_approach=rate, trips=int(trips.n), iterations=int(res["iterations"]),
            admitted=int(adm.sum()), completed=int(done.sum()), pending=int((~adm & (tab["done"] != 3)).sum()),
            pending_share=float((~adm).mean()), still_driving=int((tab["done"][adm] == 0).sum()),
            index_rule=int((tab["done"] == 2).sum()),
            throughput_veh_per_hour_per_junction=float(done.sum() / a.scenes / hours),
            entry_delay_iterations=stats(tab["entry_delay"][adm]), travel_iterations=stats(tab["travel"][done]),
            slot_waits=int(tab["slot_waits"].sum()), blocked_waits=int(tab["blocked_waits"].sum()),
            contacts_per_1000_trips=float(1000.0 * (tab["first_contact_eval"][adm] >= 0).sum() / max(adm.sum(), 1)),
            control_steps=control, wall_s=wall, run_s=run_s, control_steps_per_s=control / wall,
            iteration_us=wall * 1e6 / max(res["iterations"], 1))
        print(name, json.dumps(runs[name]), flush=True)

    # the trips pass on a mid-run state
    ep, _ = make(8, 600.0, a.steps)
    for _ in range(a.mid):
        ep.iterate()
    torch.cuda.synchronize()
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream().cuda_stream
    import ctypes as Ct
    done_np = ep.done.cpu().numpy()
    pending = int(ep._trips["pending"].sum().item())

    def one():
        _cabi.check(lib.jmpc_scene_trips(h, Ct.byref(ep._trips_struct), ep._p(ep.iter_dev), 0, stream),
                    "jmpc_scene_trips")
    for _ in range(20):
        one()
    times = []
    for _ in range(2):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(a.launches):
            one()
        ev1.record()
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1) * 1e3 / a.launches)
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes on the 12 recorded intersection courses, trips start at course point 0 at 4 m/s, "
                 f"T = 13, first_come junction = (0, 0, {a.radius}) with shared plans, outcomes only, {a.steps} "
                 f"iterations of dt = {dt} s; Poisson arrivals per approach (4 approaches, seed 12); wall = "
                 "construction + run()",
        runs=runs,
        trips_pass=dict(us_per_launch=times, us_per_launch_min=min(times), scenes=a.scenes, slots=8,
                        state=dict(iteration=a.mid, running=int((done_np == 0).sum()),
                                   empty=int((done_np == _cabi.WAITING).sum()), pending_trips=pending)),
        r11_first_come_park_control_steps_per_s=12.9e6)
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
