"""Fixed-time traffic signals (BatchedEpisodes(signals=...)): the recorded intersection under a two-phase plan against
first_come alone, at four Poisson demand levels, and the cost of the signal pass.

Workload (the r12 workload of bench_scene_trips): --scenes scenes x 8 slots on the 12 recorded intersection courses,
every trip starts at its course's point 0 at 4 m/s; T = 13; first_come with junction (0, 0, 10 m) and shared plans;
outcome record only; --steps iterations (dt = 0.2 s); seeded Poisson arrivals per approach (poisson_trips, seed 12) at
150 / 300 / 450 / 600 veh/h per approach.
  plan     approaches 1 and 3 (south, north) form group 0, approaches 2 and 4 group 1; cycle 300 iterations (60 s),
           greens (0, 130) and (150, 130): 20 iterations (4 s) of clearance after each; stop line = the zone entry of
           the junction (0, 0, 10 m), point 246-247 on all 12 courses; margin = the collision margin; stop_decel 3 m/s^2
  runs     each demand level without and with the plan, in the same process, after one warm-up run of each kind
           (40 iterations): wall time of construction + run() (host clock, run() ends in a device synchronise), control
           steps (every trip's executed steps), throughput per junction, entry delay and travel time (iterations),
           pending trips, contacts per 1000 admitted trips, hold steps and GO passes
  pass     on the state after --mid iterations of the 600 veh/h run with the plan: CUDA events around --launches
           back-to-back launches of jmpc_signals (the first may decide, the rest find their decisions latched and add
           hold steps)
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r13_signals.json).
"""
import argparse
import ctypes as Ct
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402

RATES = (150.0, 300.0, 450.0, 600.0)
GROUPS = [0, 1, 0, 1]


def stats(x):
    x = np.asarray(x, np.float64)
    return dict(mean=float(x.mean()), p95=float(np.percentile(x, 95))) if len(x) else dict(mean=None, p95=None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--mid", type=int, default=300)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_signals.json"))
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import _cabi, synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes, SignalPlan, poisson_trips
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_signals needs a CUDA device")
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
    junction = (0.0, 0.0, 10.0)
    plan = SignalPlan(300, [(0, 130), (150, 130)], junction)
    demand = {rate: poisson_trips(a.scenes, routes, rate, dt, a.steps, 4.0, seed=12, groups=GROUPS) for rate in RATES}

    def make(rate, steps, signals):
        trips = demand[rate]
        if signals is None:                      # the same draws without groups
            trips = type(trips)(trips.scene, trips.arrival, trips.course_id, trips.state)
        return BatchedEpisodes.from_trips(engine, trips, a.scenes, agents_per_scene=8, frame_window=10, margin=margin,
                                          max_steps=steps, record_history=False, outcomes=True, share_plans=True,
                                          right_of_way="first_come", junction=junction, signals=signals), trips

    for signals in (None, plan):                 # warm-up (the demand is drawn before the timed runs)
        make(600.0, 40, signals)[0].run(max_steps=40)
    runs = {}
    for rate in RATES:
        for name, signals in (("first_come", None), ("signals", plan)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ep, trips = make(rate, a.steps, signals)
            res = ep.run(max_steps=a.steps)
            wall = time.perf_counter() - t0
            tab = res["trips"]
            adm = tab["entry"] >= 0
            done = tab["done"] == 1
            hours = res["iterations"] * dt / 3600.0
            control = int(tab["steps"][adm].sum())
            row = dict(
                rate_per_hour_per_approach=rate, trips=int(trips.n), iterations=int(res["iterations"]),
                admitted=int(adm.sum()), completed=int(done.sum()), pending=int((~adm & (tab["done"] != 3)).sum()),
                still_driving=int((tab["done"][adm] == 0).sum()), index_rule=int((tab["done"] == 2).sum()),
                throughput_veh_per_hour_per_junction=float(done.sum() / a.scenes / hours),
                entry_delay_iterations=stats(tab["entry_delay"][adm]), travel_iterations=stats(tab["travel"][done]),
                contacts_per_1000_trips=float(1000.0 * (tab["first_contact_eval"][adm] >= 0).sum() / max(adm.sum(), 1)),
                failed_solves=int(tab["failed_solves"][adm].sum()),
                control_steps=control, wall_s=wall, control_steps_per_s=control / wall)
            if signals is not None:
                row.update(hold_steps=int(tab["signal_hold_steps"].sum()), go_passes=int(tab["signal_go"].sum()),
                           trips_held=int((tab["signal_hold_steps"] > 0).sum()))
            runs[f"{name}_{int(rate)}"] = row
            print(f"{name}_{int(rate)}", json.dumps(row), flush=True)

    # the signal pass on a mid-run state
    ep, _ = make(600.0, a.steps, plan)
    for _ in range(a.mid):
        ep.iterate()
    torch.cuda.synchronize()
    done_np = ep.done.cpu().numpy()
    latch = ep.signal_latch.cpu().numpy()
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream().cuda_stream

    def one():
        _cabi.check(lib.jmpc_signals(
            h, ep.B, ep.k, Ct.byref(ep._signal_plan), ep._p(ep.signal_offset), ep._p(ep.signal_owner),
            ep._p(ep.signal_group), ep._p(ep.signal_zone), ep._p(ep.course_id), ep._p(ep.agent_idx), ep._p(ep.state),
            ep._p(ep.params), ep._p(ep.done), 1, ep._p(ep.course_len), ep._p(ep.signal_latch), ep._p(ep.signal_hold),
            ep._p(ep.signal_go), ep._p(ep.signal_slot_hold), ep._p(ep.signal_slot_go), ep._p(ep.iter_dev), stream),
            "jmpc_signals")
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
    fc, sg = runs["first_come_600"], runs["signals_600"]
    sat = max(RATES, key=lambda r: runs[f"first_come_{int(r)}"]["throughput_veh_per_hour_per_junction"])
    pass_us = min(times)
    estimates = dict(
        pass_at_most_5us=dict(measured_us=pass_us, met=pass_us <= 5.0),
        fewer_contacts_under_the_plan={
            str(int(r)): dict(first_come=runs[f"first_come_{int(r)}"]["contacts_per_1000_trips"],
                              signals=runs[f"signals_{int(r)}"]["contacts_per_1000_trips"],
                              met=runs[f"signals_{int(r)}"]["contacts_per_1000_trips"]
                              < runs[f"first_come_{int(r)}"]["contacts_per_1000_trips"]) for r in (450.0, 600.0)},
        lower_throughput_at_first_come_saturation=dict(
            rate=sat, first_come=runs[f"first_come_{int(sat)}"]["throughput_veh_per_hour_per_junction"],
            signals=runs[f"signals_{int(sat)}"]["throughput_veh_per_hour_per_junction"],
            met=runs[f"signals_{int(sat)}"]["throughput_veh_per_hour_per_junction"]
            < runs[f"first_come_{int(sat)}"]["throughput_veh_per_hour_per_junction"]))
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes x 8 slots on the 12 recorded intersection courses, trips start at course point 0 "
                 f"at 4 m/s, T = 13, first_come junction = (0, 0, 10) with shared plans, outcomes only, {a.steps} "
                 f"iterations of dt = {dt} s; Poisson arrivals per approach (4 approaches, seed 12); wall = "
                 "construction + run()",
        plan=dict(cycle=plan.cycle, green=plan.green.tolist(), groups_by_approach=GROUPS, junction=list(junction),
                  margin=margin, stop_decel=plan.stop_decel),
        runs=runs,
        signal_pass=dict(us_per_launch=times, us_per_launch_min=pass_us, episodes=ep.B,
                         state=dict(iteration=a.mid, running=int((done_np == 0).sum()),
                                    held=int(((latch[:, 0] >= 0) & (latch[:, 1] == 1)).sum()))),
        estimates=estimates)
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
