"""Cost of the per-episode outcome record (BatchedEpisodes(outcomes=True)).

Workload of tests/tools/bench_episodes.py: 65 536 episodes on the intersection course, T = 13, two constant-input
obstacles crossing the course, max_steps = 400.  Three modes, timed in one process, alternating (the order rotates every
round) after one warm-up round:
  history           today's run: History [max_steps, B, 8] and flags kept on the device and copied back
  history_outcomes  the same plus the outcome record
  outcomes          the outcome record without History
Per mode: wall time of construction + run() (host clock, run() ends in a device synchronise), its median over the
rounds, and torch.cuda.max_memory_allocated over construction + run (torch-owned buffers: the episode state, History,
outcome record; the engine's own cudaMalloc'd workspace is the same in all modes and not counted).  The card's name and
power limit are read in the same process.  The modes must agree: identical steps / done / state everywhere, identical
History and flags between the two History modes, identical outcome records between the two outcome modes.
Writes the JSON to --out (default profiles/r4_episode_outcomes.json).
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

MODES = {"history": dict(record_history=True, outcomes=False),
         "history_outcomes": dict(record_history=True, outcomes=True),
         "outcomes": dict(record_history=False, outcomes=True)}


def workload(course, B, seed=11):
    rng = np.random.default_rng(seed)
    state0 = np.repeat(np.array([[course[0, 0], course[0, 1], 0.0, course[0, 2]]]), B, axis=0)
    state0[:, 2] = rng.uniform(0, 3, B)
    obst = np.zeros((B, 2, 6))
    k = rng.integers(150, 400, (B, 2))
    ang = rng.uniform(-np.pi, np.pi, (B, 2))
    obst[:, :, 0] = course[k, 0] - 25 * np.cos(ang)
    obst[:, :, 1] = course[k, 1] - 25 * np.sin(ang)
    obst[:, :, 2] = rng.uniform(3, 8, (B, 2))
    obst[:, :, 3] = ang
    obst[:, :, 5] = rng.uniform(-.05, .05, (B, 2))
    return state0, obst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_episode_outcomes.json"))
    a = ap.parse_args()
    import torch
    from junction_mpc import synth
    from junction_mpc.batched import BatchedMPC
    from junction_mpc.episodes import BatchedEpisodes
    from oracle import collision_oracle as C
    if not torch.cuda.is_available():
        raise SystemExit("bench_episode_outcomes needs a CUDA device")
    gpu = dict(name=torch.cuda.get_device_name(0))
    try:
        gpu["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # noqa: BLE001
        gpu["power_limit"] = f"unavailable ({e})"
    course = synth.load_course("intersection")
    dl = float(np.linalg.norm(course[0, :2] - course[1, :2]))
    B, steps = a.B, a.steps
    engine = BatchedMPC([course], dl=dl, T=13, max_batch=B)
    state0, obst = workload(course, B)
    margin = C.cutoff_margin(C.CarGeometry(), dl)

    def one(mode):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        ep = BatchedEpisodes(engine, state0, obstacles=obst.copy(), frame_window=10, margin=margin, max_steps=steps,
                             **MODES[mode])
        res = ep.run(max_steps=steps)
        wall = time.perf_counter() - t0
        peak = torch.cuda.max_memory_allocated()
        del ep
        return wall, peak, res

    names = list(MODES)
    walls = {m: [] for m in names}
    peaks, last = {}, {}
    for r in range(a.rounds + 1):                # round 0 is the warm-up
        order = names[r % 3:] + names[:r % 3]
        for m in order:
            wall, peak, res = one(m)
            if r:
                walls[m].append(wall)
                peaks[m] = peak
                last[m] = res
            print(f"round {r} {m}: {wall * 1e3:.1f} ms, peak {peak / 2**20:.1f} MiB", flush=True)
    h, ho, o = last["history"], last["history_outcomes"], last["outcomes"]
    same = dict(
        steps_done_state=all(np.array_equal(h[k], x[k]) for x in (ho, o) for k in ("steps", "done", "state")),
        history_flags=bool(np.array_equal(h["history"], ho["history"], equal_nan=True)
                           and np.array_equal(h["flags"], ho["flags"])),
        outcomes=all(np.array_equal(ho["outcomes"][k], o["outcomes"][k]) for k in ho["outcomes"]))
    med = {m: statistics.median(walls[m]) for m in names}
    oc = o["outcomes"]
    out = dict(
        gpu=gpu,
        workload=f"{B} episodes, intersection course, T = 13, two constant-input obstacles, max_steps = {steps} "
                 "(tests/tools/bench_episodes.py); wall = construction + run(); memory = torch.cuda.max_memory_allocated",
        rounds=a.rounds, iterations=int(h["iterations"]), control_steps=int(h["steps"].sum()),
        modes={m: dict(wall_s=walls[m], wall_s_median=med[m], max_memory_allocated_bytes=int(peaks[m]))
               for m in names},
        history_outcomes_over_history=med["history_outcomes"] / med["history"] - 1.0,
        outcomes_over_history=med["outcomes"] / med["history"] - 1.0,
        memory_saved_bytes=int(peaks["history"] - peaks["outcomes"]),
        identical=same,
        batch=dict(contact=int((oc["first_contact_eval"] >= 0).sum()), cut=int((oc["cut_steps"] > 0).sum()),
                   failed_solves=int((oc["failed_solves"] > 0).sum()), limit=int((oc["limit_steps"] > 0).sum()),
                   done=int((o["done"] == 1).sum())))
    print(json.dumps({k: v for k, v in out.items() if k != "modes"}), flush=True)
    engine.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
