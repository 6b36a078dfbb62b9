"""Wall time of one `step_host` call per host transfer mode (jmpc_set_host_transfer), the modes alternating in rounds
so that they share the same machine state.  Page-locked inputs and `host_outputs` by default, plain numpy arrays with
`--pageable`.  A -DJMPC_EXPERIMENT build (JMPC_LIB) with JMPC_TIMING=1 makes jmpc_step_host_io print its own
breakdown: one call per mode after the timed rounds does that.

    python tests/tools/e2e_breakdown.py --config 2
    python tests/tools/e2e_breakdown.py --config 2 --batch 1 --pageable
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "av-simulation-at-intersections_b200"))
import numpy as np  # noqa: E402
from junction_mpc import synth  # noqa: E402
from junction_mpc.batched import BatchedMPC  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4])
ap.add_argument("--batch", type=int, default=0, help="instances (default: the config's own size)")
ap.add_argument("--pageable", action="store_true", help="plain numpy inputs and results instead of page-locked ones")
ap.add_argument("--modes", nargs="+", default=list(BatchedMPC.HOST_TRANSFER), choices=list(BatchedMPC.HOST_TRANSFER))
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--calls", type=int, default=0, help="timed calls per mode and round (default: 200 for B <= 64, else 20)")
args = ap.parse_args()

w = synth.make_workload(args.config, B=args.batch or None)
B, T = w["B"], w["T"]
calls = args.calls or (200 if B <= 64 else 20)
mpc = BatchedMPC(w["courses"], dl=w["dl"], T=T, max_batch=B)
keys = ("state", "target_ind", "oa", "od", "course_len")
if args.pageable:
    hin, hout = {k: w[k] for k in keys}, None
else:
    hin = {}
    for key in keys:
        hin[key] = mpc.pinned_empty(w[key].shape, w[key].dtype)
        hin[key][...] = w[key]
    hout = mpc.host_outputs(B)


def call():
    return mpc.step_host(hin["state"], hin["target_ind"], hin["oa"], hin["od"], course_len=hin["course_len"], out=hout)


print(f"config {args.config}, B = {B}, T = {T}, {'pageable' if args.pageable else 'page-locked'} inputs and results, "
      f"{args.rounds} rounds x {calls} calls per mode", flush=True)
ms = {m: [] for m in args.modes}
ref = None
for r in range(args.rounds):
    for mode in args.modes:
        mpc.set_host_transfer(mode)
        for _ in range(3):
            out = call()
        if ref is None:
            ref = {k: getattr(out, k).copy() for k in ("oa", "od", "cost", "status", "iters", "target_ind")}
        for k, v in ref.items():            # the transfer mode must not change a result
            assert np.array_equal(getattr(out, k), v, equal_nan=True), (mode, k)
        t0 = time.perf_counter()
        for _ in range(calls):
            call()
        ms[mode].append((time.perf_counter() - t0) / calls * 1e3)
for mode, v in ms.items():
    print(f"mode {mode:18s} ms per call: median {np.median(v):.4f}  min {min(v):.4f}  max {max(v):.4f}  "
          f"rounds {' '.join(f'{x:.4f}' for x in v)}", flush=True)
os.environ["JMPC_TIMING"] = "1"
for mode in args.modes:
    mpc.set_host_transfer(mode)
    call()
    sys.stderr.flush()
mpc.close()
