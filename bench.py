#!/usr/bin/env python
"""bench.py -- batched MPC step solves/s on B200 (BASELINE.json metric) and the CPU reference arm.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (nearest index -> reference sampling -> rollout -> linearise/condense ->
QP solve -> outputs) over one batch of synthetic instances (SURVEY.md section 8d):

  config 2 (default, the configuration the metric is quoted on): 4096 ego instances x T=20 per GPU, weak scaling;
  config 3 / 4: 65 536 / 262 144 instances x T=13 per GPU with 2 / 4 obstacles each: the flag kernel runs first and
           its truncated course lengths feed the step, as the scenario loop orders them; solves/s (the step) and
           flags/s (the flag kernel) are timed and reported separately;
  config 5: the 1 048 576-instance parameter grid (T in {8, 13, 20, 25} x dt x six weight axes x 32 states), sorted
           by T (one launch per horizon), the GLOBAL batch sharded over the ranks (strong scaling).

Multi-GPU: no communication on the solve path; the packed per-instance result records are all-gathered by the
step kernel's own epilogue (NVLink peer stores into every rank's table) and made visible by a cross-GPU barrier.

Timed region: CUDA events on the launching stream around each step, L2 flushed (256 MiB write) and the in-place
warm-start buffers restored before every step outside the events; sum over K steps, max over ranks.

--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned (last_step_outputs) as
DIR/<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "av-simulation-at-intersections_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "batched MPC step solves/sec"
UNIT = "solves/s"


def flops_per_solve(T: int, iters: float) -> float:
    """Algorithmic flop count of the implemented algorithm (DESIGN.md section 5)."""
    n = 2 * T
    f_prep = 64.0 * T
    f_cond = 45.0 * n * (n + 1) / 2.0 + 70.0 * (T + 1) + 12.0 * T * (T + 1)   # O(1) entries from 23 suffix moments
    f_iter = n ** 3 / 3.0 + 7.0 * n * n + 240.0 * T
    return f_prep + f_cond + iters * f_iter


def bytes_per_solve(T: int) -> float:
    return 8.0 * (15 * T + 23)          # SURVEY.md section 8(d)


WORKLOADS = {
    2: ("intersection_T20: 4096 synthetic ego instances x T=20 per GPU (BASELINE.json configs[1])", "weak"),
    3: ("roundabout_T13: 65536 instances x T=13 per GPU, 2 randomised obstacles each, flag kernel -> truncated "
        "course -> step (BASELINE.json configs[2])", "weak"),
    4: ("multilane_T13: 262144 instances x T=13 per GPU, 4 obstacles each, flag kernel -> truncated course -> step "
        "(BASELINE.json configs[3])", "weak"),
    5: ("sensitivity grid: 1048576 instances = T in {8,13,20,25} x dt x w_perp x w_para x R x Rd (8192 points per "
        "horizon) x 32 states, sorted by T, the global batch sharded over the GPUs (BASELINE.json configs[4])",
        "strong"),
}
DEFAULT_B = {2: 4096, 3: 65536, 4: 262144}


def config_block(args):
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm of one configuration."""
    text, scaling = WORKLOADS[args.config]
    c = {"workload": f"config {args.config}: {text}", "config_id": args.config,
         "T": [8, 13, 20, 25] if args.config == 5 else [20 if args.config == 2 else 13],
         "l2": "GPU arm: L2 flushed with a 256 MiB write before every timed step; CPU arm: not applicable"}
    if args.config == 5:
        c["instances_total"] = 4 * 8192 * args.states_per_point
    else:
        c["instances_per_gpu"] = args.batch or DEFAULT_B[args.config]
    return c, scaling


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self._armed = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        self._armed.wait()                  # started early, records only inside the timed region
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def arm(self):
        self._armed.set()

    def finish(self):
        self._halt.set()
        self._armed.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- workloads --------------------------------------------------------------------------------------------------
def host_slices(args, rank, world):
    """The horizon-homogeneous slices this rank solves per step: a list of workload dicts (junction_mpc.synth).
    Configs 2-4: one slice, every rank its own seeded batch (weak scaling).  Config 5: one slice per horizon, this
    rank's contiguous shard of the global slice (strong scaling), `row0` = its first row in the gathered table."""
    from junction_mpc import synth
    from junction_mpc.distributed import shard_bounds
    if args.config != 5:
        w = synth.make_workload(args.config, B=args.batch or None, seed_offset=rank)
        w["row0"], w["rows_global"] = rank * w["B"], world * w["B"]
        return [w]
    out = []
    per_T = 8192 * args.states_per_point
    for k, T in enumerate(synth.SWEEP_HORIZONS):
        lo, hi = shard_bounds(per_T, world, rank)
        w = synth.make_sweep_shard(T, lo, hi, states_per_point=args.states_per_point)
        w["row0"], w["rows_global"] = k * per_T + lo, 4 * per_T
        out.append(w)
    return out


DUMP_BYTES = 60 << 20          # array data of --dump-outputs; the .npy headers fit in the rest of 64 MB


def last_step_outputs(devs, has_obs):
    """name -> float64 host array: what the timed step hands its caller (controls and target index updated in place,
    predicted states, reference, cost, status, solver iterations, result records; with obstacles the flags and the
    cut course lengths), instance-major.  Several horizon slices (config 5) are prefixed `T<T>_`.  When the whole
    batch would exceed DUMP_BYTES, every array of a slice holds the same seeded sample of instances, sorted, whose
    indices are `rows`."""
    import torch
    slices = []
    for d in devs:
        a = {"oa": d.oa, "od": d.od, "target_ind": d.tgt, "ox": d.out.ox, "oy": d.out.oy, "ov": d.out.ov,
             "oyaw": d.out.oyaw, "xref": d.out.xref, "cost": d.out.cost, "status": d.out.status, "iters": d.out.iters,
             "record": d.out.record}
        if has_obs:
            a["flag"], a["course_len"] = d.flag, d.clen
        slices.append(a)
    total = sum(8 * (sum(t.numel() for t in a.values()) + d.B) for d, a in zip(devs, slices))   # + d.B: `rows`
    frac = min(1.0, DUMP_BYTES / total)
    out = {}
    for d, a in zip(devs, slices):
        prefix = f"T{d.T}_" if len(devs) > 1 else ""
        rows = None
        if frac < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(d.B, int(d.B * frac), replace=False))
            out[prefix + "rows"] = rows.astype(np.float64)
            rows = torch.as_tensor(rows, device=d.oa.device)
        for name, t in a.items():
            out[prefix + name] = (t if rows is None else t.index_select(0, rows)).to(torch.float64).cpu().numpy()
    return out


def cpu_solver():
    """Which CPU implementation the CPU legs time: the reference's own solver stack when it imports here
    (cvxpy + ECOS through the reference's formulation, oracle/reference_solver.py), else the oracle port."""
    from oracle import reference_solver as RS
    pr = RS.probe()
    return ("reference" if pr["available"] else "port"), pr


def _cpu_one(job):
    from helpers import params_from_vector
    from oracle import mpc_oracle as O
    from oracle import reference_solver as RS
    kind, pv, T, state, oa, od, course, n, target = job
    p = params_from_vector(pv, T)
    fn = RS.mpc_step_reference_solver if kind == "reference" else O.mpc_step
    r = fn(p, state, oa, od, course[:n, 0], course[:n, 1], course[:n, 2], int(target))
    return r.status


def cpu_jobs(kind, slices, per_slice):
    from helpers import default_vector
    jobs = []
    for w in slices:
        base = default_vector(w)
        for k in range(min(per_slice, w["B"])):
            pv = base if w.get("params") is None else w["params"][k]
            jobs.append((kind, pv, w["T"], w["state"][k], w["oa"][k], w["od"][k], w["courses"][0],
                         int(w["course_len"][k]), int(w["target_ind"][k])))
    return jobs


def cpu_run(pool, jobs):
    """One instance per call, as the scenarios call the controller, spread over the pool's processes."""
    t0 = time.perf_counter()
    st = pool.map(_cpu_one, jobs, chunksize=max(1, len(jobs) // (4 * pool._processes)))
    dt = time.perf_counter() - t0
    assert all(s == 0 for s in st), "CPU arm: unsolved instances"
    return len(jobs) / dt, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, same
    configuration.  cvxpy + ECOS are probed at run time; when they do not import (they are not in this image and
    cannot be installed offline; the reference is pure Python, so there is no oracle/_ref to compile either) the
    oracle port runs instead and the line says so (`kind: "port"`, the probe's reason included)."""
    if rank != 0:
        return
    from helpers import make_pool
    cfg, scaling = config_block(args)
    kind, pr = cpu_solver()
    # the step of the reference arm: the whole batch for config 2 (same batch as the GPU arm), a bounded sample of
    # the batch otherwise (the full batches would take minutes per step on the CPU)
    slices = host_slices(args, 0, 1) if args.config != 5 else None
    if args.config == 5:
        from junction_mpc import synth
        per = max(1, args.ref_sample // 4)
        slices = [synth.make_sweep_sample(T, per, states_per_point=args.states_per_point) for T in synth.SWEEP_HORIZONS]
        per_slice = per
        sample = (f"{per} instances of each horizon slice per step (the first states of the slice's generator on {per} "
                  f"parameter points strided over the 8192-point grid)")
    elif args.config == 2:
        per_slice = slices[0]["B"]
        sample = f"the whole {per_slice}-instance batch per step (the GPU arm's batch, rank 0 seed)"
    else:
        per_slice = min(args.ref_sample, slices[0]["B"])
        sample = (f"first {per_slice} instances of the batch per step, full course length (the flag kernel's cut "
                  f"lengths come from the GPU arm)")
    cores = os.cpu_count() or 1
    jobs = cpu_jobs(kind, slices, per_slice)
    times = []
    with make_pool(cores) as pool:
        for k in range(args.warmup + args.steps):
            _, dt = cpu_run(pool, jobs)
            if k >= args.warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = len(jobs) / (ms * 1e-3)
    label = "reference CPU (cvxpy+ECOS)" if kind == "reference" else "CPU restatement (numpy fp64 oracle port)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "label": f"{label}, {cores} cores",
                         "sample": f"{sample}; one solve per call, multiprocessing over {cores} processes",
                         "solves_per_step": len(jobs), "reference_solver_probe": pr},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (configs 2-4; default: the config's own size)")
    ap.add_argument("--states-per-point", type=int, default=32, help="config 5: states per parameter point (32 = 1M instances)")
    ap.add_argument("--ref-sample", type=int, default=1024, help="reference arm: instances per step for configs 3-5")
    ap.add_argument("--cpu-sample", type=int, default=2048)
    ap.add_argument("--gather", default="barrier", choices=["barrier", "flags", "deferred", "nccl"],
                    help="N > 1: fused gather (record stores over NVLink in the step kernel's epilogue) completed by a "
                         "cross-GPU signal-pad barrier after every step (default: measured fastest and with the "
                         "tightest p99 at 4 and 8 GPUs); completed by flags the step kernel publishes, every step "
                         "waiting for its own table (flags) or for the previous step's (deferred: ranks run uncoupled, "
                         "the last step pays the skew); or one NCCL all-gather per step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs as DIR/<name>.npy (float64, at most 64 MB: a seeded "
                         "sample of instances when the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    if rank == 0 or not os.path.exists(os.path.join(g.PKG, "junction_mpc", "libjmpc.so")):
        g.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    if world > 1 and os.environ.get("BENCH_PIN") and hasattr(os, "sched_setaffinity"):
        # one disjoint set of host cores per rank (experiment: launch jitter of eight processes on one host)
        n = os.cpu_count() or world
        per = max(1, n // world)
        os.sched_setaffinity(0, set(range(local * per, min(n, (local + 1) * per))))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()

    from junction_mpc.batched import BatchedMPC
    from junction_mpc import _cabi
    from junction_mpc.distributed import allgather_records
    from oracle import collision_oracle as CO            # cutoff_margin only (a constant of the scenario scripts)

    cfg_block, scaling = config_block(args)
    slices = host_slices(args, rank, world)
    B_local = sum(w["B"] for w in slices)
    B_global = slices[0]["rows_global"]
    max_B = max(w["B"] for w in slices)
    mpc = BatchedMPC(slices[0]["courses"], dl=slices[0]["dl"], T=slices[0]["T"], max_batch=max_B, device=local,
                     max_T=max(w["T"] for w in slices))
    f64, i32 = torch.float64, torch.int32
    t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)  # noqa: E731
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    has_obs = slices[0].get("obstacles") is not None
    margin = CO.cutoff_margin(CO.CarGeometry(), slices[0]["dl"])

    class Dev:
        pass
    devs = []
    for w in slices:
        d = Dev()
        d.w, d.B, d.T = w, w["B"], w["T"]
        d.state, d.clen = t(w["state"], f64), t(w["course_len"], i32)
        d.tgt0, d.oa0, d.od0 = t(w["target_ind"], i32), t(w["oa"], f64), t(w["od"], f64)
        d.tgt, d.oa, d.od = d.tgt0.clone(), d.oa0.clone(), d.od0.clone()
        d.params = t(w.get("params"), f64)
        d.out = mpc.alloc_outputs(d.B, d.T)
        if has_obs:
            d.agent, d.v, d.obs = t(w["agent_idx"], i32), t(w["state"][:, 2], f64), t(w["obstacles"], f64)
            d.flag = torch.zeros(d.B, dtype=i32, device=dev)
            # the flag kernel's course lengths feed the step; the search start is clamped to the truncated course
            # once, outside the timed region (the inputs, hence the cut lengths, are the same every step)
            mpc.collision(d.agent, d.v, d.obs, w["frame_window"], margin, d.flag, d.clen)
            d.tgt0 = torch.minimum(d.tgt0, d.clen - 1).contiguous()
            d.tgt = d.tgt0.clone()
        devs.append(d)
    torch.cuda.synchronize()

    # multi-GPU gather of the result records: fused into the kernel epilogue over NVLink peer memory when symmetric
    # memory is available, otherwise one NCCL all-gather straight from the kernel's record buffer
    fused, gather_kind = None, "none (single GPU)"
    if world > 1:
        gather_kind = "nccl all_gather_into_tensor of the record buffer, every step"
        if args.gather != "nccl":
            try:
                from junction_mpc.distributed import FusedRecordGather
                fused = FusedRecordGather(mpc, B_global, slices[0]["row0"], sync="barrier" if args.gather == "barrier" else "flags")
                gather_kind = ("fused: the step kernel's epilogue stores every record into every rank's table (NVLink "
                               "symmetric memory, ring of %d tables); " % fused.buffers +
                               ("completion by flags: the kernel's last block publishes the step number to every rank, and "
                                "every step ends with the wait for all ranks' records of THIS step (a complete table "
                                "inside every timed step, no barrier kernel)" if args.gather == "flags" else
                                "completion by flags: the kernel's last block publishes the step number to every rank, and "
                                "every step ends with the wait for all ranks' records of the PREVIOUS step (the last timed "
                                "step also waits for its own and so pays the skew the ranks have built up), so the gather "
                                "runs one step behind the solves" if args.gather == "deferred" else
                                "cross-GPU signal-pad barrier after every step"))
            except Exception as exc:            # noqa: BLE001
                if rank == 0:
                    print(f"[bench] fused gather unavailable ({type(exc).__name__}: {exc}); using NCCL", file=sys.stderr)
                fused = None
    step_no = [0]

    def one_step(e0=None, e1=None, ec=None, cold=True, marks=None, final=False):
        flush.zero_()
        for d in devs:
            d.tgt.copy_(d.tgt0); d.oa.copy_(d.oa0); d.od.copy_(d.od0)
        if cold:
            # The bench re-solves the same batch every step.  The engine's default schedule orders the work queue
            # by the iteration counts of the previous step (meant for closed loops); on a repeated batch those
            # would be exact foreknowledge, so the headline forgets them before every step: the queue is ordered by
            # the a-priori key computed from this step's inputs only.
            mpc.reset_schedule_hints()
        if e0 is not None:
            e0.record()
        if has_obs:
            for d in devs:
                mpc.collision(d.agent, d.v, d.obs, d.w["frame_window"], margin, d.flag, d.clen)
            if ec is not None:
                ec.record()
        for k, d in enumerate(devs):
            if fused is not None:
                fused.begin_step(d.w["row0"], publish=(k == len(devs) - 1))
            mpc.step(d.state, d.tgt, d.oa, d.od, d.out, course_len=d.clen, params=d.params, T=d.T)
            if marks is not None:
                marks[k].record()
        step_no[0] += 1
        if fused is not None:
            fused.finish()                     # the records are already on their way into every peer's table
            if args.gather == "flags":
                fused.wait(fused.step_no)
            elif args.gather == "deferred":
                fused.wait(fused.step_no if final else fused.step_no - 1)
        elif world > 1:
            for d in devs:
                allgather_records(d.out.record)   # [world * B, 8] on every rank, straight from the kernel's buffer
        if e1 is not None:
            e1.record()

    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    if fused is not None and len(devs) == 1:   # the fused table must equal what the NCCL all-gather delivers
        one_step(final=True)
        torch.cuda.synchronize()
        got = fused.table_of(fused.step_no)
        ref = allgather_records(devs[0].out.record)
        torch.cuda.synchronize()
        same = torch.equal(torch.nan_to_num(got, nan=-1.0), torch.nan_to_num(ref, nan=-1.0))
        assert same, "fused record gather differs from the NCCL all-gather"
        assert not mpc.gather_timed_out(), "gather wait timed out"
    sampler = ClockSampler(local, period=float(os.environ.get("BENCH_SAMPLER_PERIOD", "0.005")))     # NVML init: milliseconds
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    evs = [(ev(), ev(), ev(), [ev() for _ in devs]) for _ in range(args.steps)]
    step_no[0] = 0
    # Align the ranks on the DEVICE right before the timed loop: the NCCL barrier is a kernel on each rank's stream, so
    # all streams leave it within microseconds.  (Anything host-side between the barrier and the loop -- NVML start-up,
    # event creation -- skews the ranks by milliseconds, and with a cross-rank gather inside the step the early ranks
    # then time their waiting for the late ones.)
    import gc
    sampler.start()                          # the thread idles until arm(): its start-up stays outside the timed region
    gc.collect()
    gc.disable()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    sampler.arm()
    launches0 = mpc.launch_count
    for k, (e0, e1, ec, marks) in enumerate(evs):
        one_step(e0, e1, ec, marks=marks, final=(k == len(evs) - 1))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.finish()
    gc.enable()
    launches = mpc.launch_count - launches0
    # taken now: the passes below overwrite the output buffers
    dump = last_step_outputs(devs, has_obs) if args.dump_outputs and rank == 0 else None
    # per step: [flag kernel] + step launches + gather.  The metric counts MPC step solves: flag production is timed
    # separately (SURVEY.md 8d: "solves/s must not be diluted or inflated by it").
    coll_ms = np.array([e0.elapsed_time(ec) for e0, e1, ec, _ in evs]) if has_obs else np.zeros(args.steps)
    total_step_ms = np.array([e0.elapsed_time(e1) for e0, e1, ec, _ in evs])
    per_step = total_step_ms - coll_ms                                        # ms: the solve (+ gather) part
    slice_ms = []
    for k in range(len(devs)):
        start = [(ec if has_obs else e0) if k == 0 else marks[k - 1] for e0, e1, ec, marks in evs]
        slice_ms.append(float(np.mean([s.elapsed_time(marks[k]) for s, (_, _, _, marks) in zip(start, evs)])))
    tot = torch.tensor([per_step.sum(), coll_ms.sum(), total_step_ms.sum()], dtype=f64, device=dev)
    per_rank_ms = [float(per_step.mean())]
    if world > 1:
        allr = [torch.zeros(1, dtype=f64, device=dev) for _ in range(world)]
        dist.all_gather(allr, torch.tensor([per_step.mean()], dtype=f64, device=dev))
        per_rank_ms = [float(x.item()) for x in allr]
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    ms_per_step = float(tot[0].item()) / args.steps
    coll_ms_per_step = float(tot[1].item()) / args.steps
    pipeline_ms = float(tot[2].item()) / args.steps
    solves_per_step = B_global if scaling == "strong" else world * B_local
    value = solves_per_step / (ms_per_step * 1e-3)
    status = np.concatenate([d.out.status.cpu().numpy() for d in devs])
    iters = [d.out.iters.cpu().numpy() for d in devs]
    not_solved = int((status != 0).sum())
    if has_obs:            # a cut right behind the search start can leave the index rule undefined (status 3)
        assert not_solved <= 1e-3 * len(status), f"{not_solved} instances not solved"
    else:
        assert not_solved == 0, f"{not_solved} instances not solved"

    # secondary figure (config 2): the same steps with the previous step's iteration counts as scheduling keys (what
    # a closed loop that re-solves slowly changing instances sees; on this repeated batch the keys are exact)
    hint = None
    if args.config == 2:
        hint_steps = max(3, min(args.steps, 20))
        one_step(cold=False)
        evs2 = [(ev(), ev()) for _ in range(hint_steps)]
        for e0, e1 in evs2:
            one_step(e0, e1, cold=False)
        torch.cuda.synchronize()
        hint_ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in evs2) / hint_steps], dtype=f64, device=dev)
        if world > 1:
            dist.all_reduce(hint_ms, op=dist.ReduceOp.MAX)
        hint = (float(hint_ms.item()), hint_steps)
    if fused is not None:
        torch.cuda.synchronize()
        assert not mpc.gather_timed_out(), "gather wait timed out"
        dist.barrier()
        fused.close()

    # end to end through the host API: inputs in page-locked host memory, H2D of the step's inputs and the results
    # back on the host inside the timed region (wall clock around the calls)
    e2e_steps = max(3, min(args.steps, 20 if B_local <= 65536 else 5))
    h2d = d2h = 0
    hio = []
    for d in devs:
        w, T1 = d.w, d.T + 1
        keys = ["state", "target_ind", "oa", "od", "course_len"] + (["params"] if w.get("params") is not None else []) \
            + (["agent_idx", "obstacles"] if has_obs else [])
        hin = {}
        for key in keys:
            hin[key] = mpc.pinned_empty(w[key].shape, w[key].dtype)
            hin[key][...] = w[key]
            h2d += hin[key].nbytes
        if has_obs:
            hin["v"] = mpc.pinned_empty((d.B,), np.float64)
            hin["v"][...] = w["state"][:, 2]
            hin["flag"], hin["clen"] = mpc.pinned_empty((d.B,), np.int32), mpc.pinned_empty((d.B,), np.int32)
            hin["tgt"] = mpc.pinned_empty((d.B,), np.int32)
            h2d += hin["v"].nbytes
            d2h += 8 * d.B
        hio.append((hin, mpc.host_outputs(d.B, d.T)))
        d2h += 8 * d.B * (2 * d.T + 4 * T1 + 4 * T1 + 1 + _cabi.RECORD_LEN) + 4 * d.B * 3

    def e2e_step():
        mpc.reset_schedule_hints()              # cold schedule, as in the device-timed region
        res = []
        for d, (hin, hout) in zip(devs, hio):
            clen, tgt = hin["course_len"], hin["target_ind"]
            if has_obs:
                mpc.collision_host(hin["agent_idx"], hin["v"], hin["obstacles"], d.w["frame_window"], margin,
                                   out=(hin["flag"], hin["clen"]))
                clen = hin["clen"]
                np.minimum(hin["target_ind"], clen - 1, out=hin["tgt"])
                tgt = hin["tgt"]
            res.append(mpc.step_host(hin["state"], tgt, hin["oa"], hin["od"], course_len=clen, params=hin.get("params"),
                                     T=d.T, out=hout))
        return res
    for _ in range(2):
        e2e_step()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ho = e2e_step()
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=f64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = solves_per_step / (float(e2e_ms.item()) * 1e-3)
    assert sum(int((h.status != 0).sum()) for h in ho) == not_solved

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # latency of one controller call for a single ego (what a scenario runner sees per timestep)
    w0 = slices[0]
    one = BatchedMPC(w0["courses"], dl=w0["dl"], T=w0["T"], max_batch=1, device=local)
    lat = []
    prm1 = None if w0.get("params") is None else w0["params"][:1]
    for k in range(60):
        t0 = time.perf_counter()
        one.step_host(w0["state"][:1], w0["target_ind"][:1], w0["oa"][:1], w0["od"][:1], course_len=w0["course_len"][:1],
                      params=prm1)
        if k >= 10:
            lat.append((time.perf_counter() - t0) * 1e3)
    one.close()

    # roofline of the dominant kernel (the step kernel of the slowest slice): CUDA-core FP64 FMA bound (DESIGN.md 5)
    fp64_peak, fp32_peak = mpc.measure_fma_peak()
    kdom = int(np.argmax(slice_ms))
    Td, Bd = devs[kdom].T, devs[kdom].B
    kernel_ms = slice_ms[kdom]
    mean_iters = float(iters[kdom].mean())
    fl = flops_per_solve(Td, mean_iters) * Bd
    achieved = fl / (kernel_ms * 1e-3) / 1e12
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tr = json.load(f)
        key = f"B{Bd}_T{Td}"
        if key in tr:
            traffic, traffic_src = tr[key]["dram_bytes_per_launch"], f"profiles/r2_traffic.json[{key}]"
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_ach = bytes_per_solve(Td) * Bd / (kernel_ms * 1e-3) / 1e9
    all_iters = np.concatenate(iters)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg_block,
        "run": {"instances_this_rank": B_local, "solves_per_step_all_ranks": solves_per_step,
                "solver": "condensed QP, Mehrotra predictor-corrector interior point, fp64 (DESIGN.md: an interior-point "
                          "method instead of the north star's ADMM sketch, for parity)",
                "instances_per_warp": {str(d.T): 2 if d.T <= 15 else 1 for d in devs},
                "mean_solver_iters": float(all_iters.mean()), "max_solver_iters": int(all_iters.max()),
                "not_solved": not_solved,
                "schedule": "longest-first work queue by an a-priori key from the step's inputs (speed-cap proximity); "
                            "previous-step iteration counts deliberately forgotten before every step",
                "gather": gather_kind, "ms_per_step_by_rank": per_rank_ms,
                "ms_by_step_rank0": [round(float(x), 3) for x in per_step[:64]],
                "slices": [{"T": d.T, "instances": d.B, "kernel_ms": ms, "mean_solver_iters": float(it.mean()),
                            "fp64_frac": flops_per_solve(d.T, float(it.mean())) * d.B / (ms * 1e-3) / 1e12 / fp64_peak}
                           for d, ms, it in zip(devs, slice_ms, iters)]},
        "p50_ms": float(np.percentile(per_step, 50)), "p99_ms": float(np.percentile(per_step, 99)),
        "single_instance_step_ms": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                    "api": f"step_host, B=1, T={w0['T']}, host in / host out"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": float(e2e_ms.item()), "steps": e2e_steps,
                "api": ("BatchedMPC.collision_host -> jmpc_collision_host, then " if has_obs else "") +
                       "BatchedMPC.step_host(out=host_outputs) -> jmpc_step_host_io: numpy inputs and results in "
                       "page-locked host memory; inputs copied host->device with cudaMemcpyAsync, results stored by the "
                       "kernels straight into the host arrays over PCIe (device mapping of the page-locked memory, no "
                       "device->host copy pass); wall clock around the calls, results readable on the host when they return"
                       + (" (the flag kernel's time is inside this figure)" if has_obs else "")},
        "gpu_launches": int(launches),
        "roofline": {"bound": "fp64_fma", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": achieved / fp64_peak if fp64_peak else None, "traffic": traffic,
                     "traffic_unit": f"bytes/launch (dram__bytes_read.sum + dram__bytes_write.sum, {traffic_src})",
                     "peak_source": "jmpc_measure_fma_peak: register-resident FP64 FMA loop on all SMs, measured in this run "
                                    "(MEASURED_PEAKS.json holds no FP64 figure)",
                     "flops_per_solve": flops_per_solve(Td, mean_iters), "kernel": f"jmpc::mpc_step_kernel<{Td}>",
                     "kernel_ms": kernel_ms, "kernel_instances": Bd, "fp32_peak_tflops": fp32_peak,
                     "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                             "bytes_per_solve": bytes_per_solve(Td),
                             "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback of B200_PROFILING.md"}},
    }
    if has_obs:
        flags_per_step = world * B_local
        line["flag_kernel"] = {"value": flags_per_step / (coll_ms_per_step * 1e-3), "unit": "flags/s",
                               "ms_per_step": coll_ms_per_step, "n_obs": int(slices[0]["obstacles"].shape[1]),
                               "frame_window": int(slices[0]["frame_window"]),
                               "flag_rate": float(devs[0].flag.float().mean().item()),
                               "pipeline_ms_per_step": pipeline_ms,
                               "note": "jmpc::collision_kernel, timed by its own events; not part of `value`"}
    if hint is not None:
        line["with_history_hints"] = {"value": solves_per_step / (hint[0] * 1e-3), "unit": UNIT, "ms_per_step": hint[0],
                                      "steps": hint[1],
                                      "note": "same steps with the work queue ordered by the previous step's iteration counts "
                                              "(the engine's closed-loop default); exact foreknowledge on this repeated batch, "
                                              "so it is reported beside the headline, not as it"}
    if world == 1 and not args.no_cpu:
        from helpers import make_pool
        kind, pr = cpu_solver()
        cores = os.cpu_count() or 1
        per_slice = max(1, min(args.cpu_sample, B_local) // len(slices))
        # the CPU leg sees the step's inputs as the GPU saw them (course lengths from the flag kernel)
        cw = [dict(d.w, course_len=d.clen.cpu().numpy(), target_ind=d.tgt0.cpu().numpy()) for d in devs]
        ok = []
        for d in devs:              # solved instances, strided over the slice (config 5: over its parameter points)
            good = np.nonzero(d.out.status.cpu().numpy() == 0)[0]
            ok.append(good[::max(1, len(good) // per_slice)][:per_slice])
        for w, sel in zip(cw, ok):
            for key in ("state", "oa", "od", "course_len", "target_ind") + (("params",) if w.get("params") is not None else ()):
                w[key] = w[key][sel]
            w["B"] = len(sel)
        jobs = cpu_jobs(kind, cw, per_slice)
        with make_pool(cores) as pool:
            cpu_run(pool, jobs[:64])                                  # warm the workers (imports, BLAS)
            rate, dt = cpu_run(pool, jobs)
        label = "reference CPU (cvxpy+ECOS)" if kind == "reference" else "CPU restatement (numpy fp64 oracle port)"
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "label": f"{label}, {cores} cores",
                                "sample": f"{per_slice} solved instances strided over each slice of the same batch "
                                          f"({len(jobs)} solves), one solve per call, {cores} processes, {dt:.1f} s wall",
                                "reference_solver_probe": pr}
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
