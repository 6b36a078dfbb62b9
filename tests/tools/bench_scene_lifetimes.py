"""Lifetimes of scene vehicles (BatchedEpisodes(depart=..., on_goal=...)): the r8 intersection study with vehicles that
park at their goal (today's rule) or leave the scene there, without a rule and with first_come, plus one staggered
arrival mode.

Workload: bench_multi_agent.workload -- 16 384 scenes x 4 vehicles on the intersection's recorded planner courses,
T = 13, outcome record only, max_steps = 400; first_come with junction = (0, 0, --radius) for every scene, as r8.
  study    five modes: {no rule, first_come} x {park, leave}, and first_come + leave with a seeded depart uniform in
           [0, --spread) iterations.  One warm-up round, then --rounds rounds in rotating order: wall time of
           construction + run() (host clock, run() ends in a device synchronise), control steps (every vehicle's own
           executed steps), and the r8 outcome summary of each mode
  kernels  on the state after --mid iterations of the staggered mode (vehicles waiting, driving and gone), without a
           skip mask: CUDA events around --launches back-to-back launches of jmpc_scene_presence, jmpc_scene_enter,
           jmpc_episode_outcomes_scene and jmpc_episode_outcomes, alternating twice (scratch outputs: the run's state
           is not changed)
The card's name and power limit are read in the same process.  Writes the JSON to --out (default
profiles/r11_scene_lifetimes.json).
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

MODES = [("none_park", None, "park", False), ("none_leave", None, "leave", False),
         ("first_come_park", "first_come", "park", False), ("first_come_leave", "first_come", "leave", False),
         ("first_come_leave_staggered", "first_come", "leave", True)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--radius", type=float, default=10.0)
    ap.add_argument("--spread", type=int, default=50)
    ap.add_argument("--mid", type=int, default=40)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_scene_lifetimes.json"))
    a = ap.parse_args()
    import torch
    from helpers import load_planner_golden
    from junction_mpc import synth
    from junction_mpc import _cabi
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene_lifetimes needs a CUDA device")
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
    junction = (0.0, 0.0, a.radius)
    state0, cid, _ = workload(courses, a.scenes)
    B = len(state0)
    depart = np.random.default_rng(11).integers(0, a.spread, B)
    engine = BatchedMPC(courses, dl=dl, T=13, max_batch=B)

    def make(rule, on_goal, staggered):
        extra = dict(junction=junction) if rule == "first_come" else {}
        return BatchedEpisodes(engine, state0, course_id=cid, frame_window=10, margin=margin, max_steps=a.steps,
                               record_history=False, outcomes=True, agents_per_scene=K, right_of_way=rule,
                               on_goal=on_goal, depart=depart if staggered else None, **extra)

    walls = {m[0]: [] for m in MODES}
    last = {}
    for r in range(a.rounds + 1):                # round 0 is the warm-up
        order = MODES[r % len(MODES):] + MODES[:r % len(MODES)]
        for name, *m in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = make(*m).run(max_steps=a.steps)
            wall = time.perf_counter() - t0
            if r:
                walls[name].append(wall)
                last[name] = res
            print(f"round {r} {name}: {wall * 1e3:.1f} ms, {res['iterations']} iterations, still driving "
                  f"{int((res['done'] == 0).sum())}, waiting {int((res['done'] == _cabi.WAITING).sum())}", flush=True)

    # kernel times on a mid-run state of the staggered mode
    ep = make("first_come", "leave", True)
    for _ in range(a.mid):
        ep.iterate()
    torch.cuda.synchronize()
    lib, h = engine._lib, engine._h
    stream = torch.cuda.current_stream().cuda_stream
    p = ep._p
    done_np = ep.done.cpu().numpy()
    mask = torch.empty(B, dtype=torch.int32, device=ep.dev)
    done_scratch = ep.done.clone()
    record = ep.outcomes.clone()

    def presence():
        _cabi.check(lib.jmpc_scene_presence(h, B, K, 1, p(ep.done), p(mask), 0, stream), "jmpc_scene_presence")

    def enter():
        _cabi.check(lib.jmpc_scene_enter(h, B, p(ep.depart), p(ep.iter_dev), p(done_scratch), stream), "jmpc_scene_enter")

    def outcomes(scene):
        args = (h, B, p(ep.state), p(ep.course_id), p(ep.scene_obs), ep.n_obs, p(ep.out.record), p(ep.di), p(ep.flag),
                None, p(ep.done))
        tail = (p(ep.iter_dev), 0, p(record), None, 0, stream)
        if scene:
            return lambda: _cabi.check(lib.jmpc_episode_outcomes_scene(*args, p(ep.presence), p(ep.depart), *tail),
                                       "jmpc_episode_outcomes_scene")
        return lambda: _cabi.check(lib.jmpc_episode_outcomes(*args, *tail), "jmpc_episode_outcomes")

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
    for _ in range(2):                           # alternating, twice
        for name, fn in (("scene_presence", presence), ("scene_enter", enter),
                         ("episode_outcomes_scene", outcomes(True)), ("episode_outcomes", outcomes(False))):
            kernels.setdefault(name, []).append(timed(fn))
    kernels = {k: dict(us_per_launch=v, us_per_launch_min=min(v)) for k, v in kernels.items()}
    kernels["episode_outcomes_scene"]["ratio_to_episode_outcomes"] = (
        kernels["episode_outcomes_scene"]["us_per_launch_min"] / kernels["episode_outcomes"]["us_per_launch_min"])
    state = dict(iteration=a.mid, waiting=int((done_np == _cabi.WAITING).sum()), running=int((done_np == 0).sum()),
                 gone=int((done_np == 1).sum()))
    modes = {}
    for name, *_ in MODES:
        s = summary(last[name])
        s["waiting_at_end"] = int((last[name]["done"] == _cabi.WAITING).sum())
        med = statistics.median(walls[name])
        s.update(wall_s=walls[name], wall_s_median=med, control_steps_per_s=s["control_steps"] / med,
                 iteration_us=med * 1e6 / s["iterations"])
        modes[name] = s
    modes["first_come_leave"]["control_steps_per_s_ratio_to_park"] = (
        modes["first_come_leave"]["control_steps_per_s"] / modes["first_come_park"]["control_steps_per_s"])
    for k in ("scene_presence", "scene_enter"):
        kernels[k]["share_of_iteration"] = kernels[k]["us_per_launch_min"] / modes["first_come_leave_staggered"]["iteration_us"]
    out = dict(
        gpu=gpu,
        workload=f"{a.scenes} scenes x {K} vehicles (intersection approaches 1-4, recorded planner courses, 0-8 m along "
                 f"at 2-5 m/s), T = 13, outcomes only, max_steps = {a.steps}; first_come junction = (0, 0, {a.radius}); "
                 f"staggered: depart uniform in [0, {a.spread}) (seed 11); wall = construction + run(); kernels: "
                 f"B = {B}, {K - 1} mate slots, no skip mask, state after {a.mid} iterations of the staggered mode",
        rounds=a.rounds, modes=modes, kernel_state=state, kernels=kernels)
    print(json.dumps(out), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
