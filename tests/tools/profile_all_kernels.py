"""One launch (after warm-up) of every kernel in libjmpc.so at a representative size, for ncu:

    ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --csv \
        --log-file gpurun_out/r2_all_kernels.csv python tests/tools/profile_all_kernels.py

Sizes: config 2 (4096 x T=20, ordered queue -> schedule_kernel), config 3 (65 536 x T=13, 2 obstacles) for the step,
flag, plant, episode and obstacle kernels, 4096 planner searches, the table kernels of one course upload."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from junction_mpc import _cabi, synth  # noqa: E402
from junction_mpc.batched import BatchedMPC  # noqa: E402
from junction_mpc.episodes import BatchedEpisodes, scripted_obstacles  # noqa: E402
from junction_mpc import planner as P  # noqa: E402

dev = torch.device("cuda", 0)
t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)  # noqa: E731
reps = int(os.environ.get("REPS", "2"))

# config 2: step kernel T = 20 + schedule kernel
w = synth.make_workload(2)
mpc = BatchedMPC(w["courses"], dl=w["dl"], T=20, max_batch=4096, schedule="apriori")
args = [t(w["state"], torch.float64), t(w["target_ind"], torch.int32), t(w["oa"], torch.float64), t(w["od"], torch.float64)]
out = mpc.alloc_outputs(4096)
for _ in range(reps):
    mpc.step(args[0], args[1].clone(), args[2].clone(), args[3].clone(), out, course_len=t(w["course_len"], torch.int32))
torch.cuda.synchronize()

# config 3: flag kernel, step kernel T = 13, plant; closed loop kernels on the same batch
w = synth.make_workload(3)
B = w["B"]
mpc3 = BatchedMPC(w["courses"], dl=w["dl"], T=13, max_batch=B)          # arc_tables_kernel + circle_tables_kernel
state, tgt = t(w["state"], torch.float64), t(w["target_ind"], torch.int32)
oa, od = t(w["oa"], torch.float64), t(w["od"], torch.float64)
agent, v, obs = t(w["agent_idx"], torch.int32), t(w["state"][:, 2], torch.float64), t(w["obstacles"], torch.float64)
flag, clen = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
out3 = mpc3.alloc_outputs(B)
for _ in range(reps):
    mpc3.collision(agent, v, obs, 20, 72, flag, clen)
    tg = torch.minimum(tgt, clen - 1).contiguous()
    mpc3.step(state, tg, oa.clone(), od.clone(), out3, course_len=clen)
    mpc3.plant_step(state.clone(), out3.record[:, 1].contiguous(), out3.record[:, 0].contiguous())
torch.cuda.synchronize()
ep = BatchedEpisodes(mpc3, w["state"], obstacles=w["obstacles"], frame_window=20, margin=72, max_steps=4, record_history=True)
for _ in range(reps):
    ep.iterate()                     # episode_pre, collision, step, episode_post, obstacle_step, counter_add
torch.cuda.synchronize()
prog = scripted_obstacles([[dict(kind="roundabout", direction=1, offset=1., turning=True, speed=25 / 3.6, dt=0.2),
                            dict(kind="roundabout", direction=-1, offset=4., turning=True, speed=25 / 3.6, dt=0.2)]] * B)
ep2 = BatchedEpisodes(mpc3, w["state"], obstacle_program=prog, frame_window=20, margin=72, max_steps=4, record_history=False)
for _ in range(reps):
    ep2.iterate()                    # scripted_obstacle_kernel
torch.cuda.synchronize()

# planner: 4096 searches (the recorded variants, replicated)
z = np.load(os.path.join(ROOT, "tests", "golden", "planner.npz"))
names = [str(n) for n in z["variants"] if not np.isnan(z[f"{n}/cost"])]
g = lambda n, k: z[f"{n}/{k}"]             # noqa: E731
scenes = [[g(n, "hp")[k, :g(n, "hp_n")[k]] for k in range(len(g(n, "hp_n")))] for n in names]
idx = np.arange(4096) % len(names)
pl = P.BatchedPlanner(z["mp_points"], z["mp_total_length"], float(z["car_radius"]), z["car_circle_centers"])
for _ in range(reps):
    r = pl.plan(np.stack([g(names[i], "start") for i in idx]), np.stack([g(names[i], "goal_point") for i in idx]),
                np.stack([g(names[i], "goal_area") for i in idx]), [float(g(names[i], "allowed_dtheta")) for i in idx], scenes,
                scene_id=idx, weights=np.stack([g(names[i], "weights") for i in idx]), max_expansions=1024, max_path=32)
print("planner: %d searches, kernel %.3f ms, %.0f searches/s, found %d" % (4096, r.kernel_ms, 4096 / r.kernel_ms * 1e3,
                                                                             int((r.status == 0).sum())))
