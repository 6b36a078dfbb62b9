"""BatchedMPC: thousands of independent MPC steps per call, on one GPU, through the C ABI.

Two entry styles:
  * host arrays (numpy, float64/int32, instance-major) -> `step_host`, `collision_host`: the library stages
    through pinned memory and returns numpy results;
  * device tensors (torch, same layout) -> `step`, `collision`, `plant_step`: pointers are handed to the
    library, work is enqueued on torch's current stream, nothing synchronises.
torch is used for device memory and streams only; all arithmetic is in libjmpc.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _cabi
from .config import MPCConfig, NPARAM


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def _i32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.int32)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


@dataclass
class StepOutput:
    """Results of one batched step (numpy on the host path, torch tensors on the device path)."""
    oa: object          # [B, T]
    od: object          # [B, T]
    ox: object          # [B, T+1]
    oy: object
    ov: object
    oyaw: object
    xref: object        # [B, 4, T+1]
    cost: object        # [B]
    status: object      # [B] int32 (jmpc_status)
    iters: object       # [B] int32
    target_ind: object  # [B] int32
    record: object = None  # [B, 8] packed {di, ai, cost, status, target_ind, iters, v_1, yaw_1}


class BatchedMPC:
    def __init__(self, courses: Sequence[np.ndarray], dl: float, T: Optional[int] = None,
                 config: Optional[MPCConfig] = None, dt: float = 0.2, L: float = 2.86, speed: float = 30.0 / 3.6,
                 max_batch: int = 1 << 20, device: int = 0, max_solver_iters: int = 40,
                 linearisation_iters: Optional[int] = None, mu_tol: float = 1e-13, warps_per_sm: int = 0,
                 max_T: Optional[int] = None, schedule: str = "history", du_th: float = 0.0):
        """courses: list of (N_c, >=3) arrays [x, y, yaw(smoothed)].  `du_th` > 0 switches on the early exit of the
        linearisation loop the reference left commented out (mpc.py:236-240)."""
        self._open(max(len(c) for c in courses), len(courses), dl, T, config, dt, L, speed, max_batch, device,
                   max_solver_iters, linearisation_iters, mu_tol, warps_per_sm, max_T, du_th)
        self.set_courses(courses)
        self.set_schedule(schedule)

    def _open(self, max_N, max_courses, dl, T, config, dt, L, speed, max_batch, device, max_solver_iters,
              linearisation_iters, mu_tol, warps_per_sm, max_T, du_th):
        self._lib = _cabi.load()
        cfg = config or MPCConfig.default()
        self.T = int(T if T is not None else cfg.T)
        self.config = cfg.with_T(self.T)
        self.dl, self.dt, self.L, self.speed = float(dl), float(dt), float(L), float(speed)
        self.default_params = self.config.param_vector(dl=self.dl, dt=self.dt, L=self.L, speed=self.speed)
        self.max_batch = int(max_batch)
        self.device = int(device)
        self.max_N = int(max_N)
        self.car_radius = 2.0 / 2 ** 0.5                 # jmpc_set_car_geometry's default (car_dimensions.py:82-90)
        self.course_ok = self.course_dl = None            # set by set_courses_from_plans
        opt = _cabi.Options(int(max_solver_iters), int(linearisation_iters or cfg.max_iter), float(mu_tol),
                            int(warps_per_sm), float(du_th))
        h = C.c_void_p()
        _cabi.check(self._lib.jmpc_create(self.device, self.max_batch, int(max_T or max(self.T, 25)), self.max_N,
                                          int(max_courses), _ptr(self.default_params), C.byref(opt), C.byref(h)),
                    "jmpc_create")
        self._h = h
        self._pinned = []
        self._host_out = {}

    @classmethod
    def from_plans(cls, plans, T: Optional[int] = None, config: Optional[MPCConfig] = None, dt: float = 0.2,
                   L: float = 2.86, speed: float = 30.0 / 3.6, max_N: Optional[int] = None, max_batch: int = 1 << 20,
                   device: int = 0, max_solver_iters: int = 40, linearisation_iters: Optional[int] = None,
                   mu_tol: float = 1e-13, warps_per_sm: int = 0, max_T: Optional[int] = None, schedule: str = "history",
                   du_th: float = 0.0) -> "BatchedMPC":
        """An engine whose courses are the planned ones of a `planner.DevicePlanBatch`, ingested on the device
        (`set_courses_from_plans`): course c = plan c.  `max_N` (default: the longest trajectory the plans can hold)
        bounds the course length; a longer plan is reported unusable.  The engine's default dl is that of the first
        usable course; `BatchedEpisodes.from_plans` gives every episode its own course's dl."""
        obj = cls.__new__(cls)
        obj._open(int(max_N or plans.traj.shape[1]), len(plans), float("nan"), T, config, dt, L, speed, max_batch, device,
                  max_solver_iters, linearisation_iters, mu_tol, warps_per_sm, max_T, du_th)
        obj.set_courses_from_plans(plans)
        obj.set_schedule(schedule)
        return obj

    def set_courses_from_plans(self, plans):
        """Replace the courses by the planned trajectories of `plans` (a `planner.DevicePlanBatch`) without a host round
        trip (jmpc_set_courses_device): yaw unwrapped as MPC.__init__ does it (mpc.py:260), dl of the first segment
        (mpc_intersection.py:73), collision tables built, on torch's current stream.  Sets `course_ok` (int32, 1 =
        usable) and `course_dl` (float64, NaN when unusable) as CUDA tensors [n_plans], and `course_len`."""
        import torch
        n = len(plans)
        dev = torch.device("cuda", self.device)
        ok = torch.empty(n, dtype=torch.int32, device=dev)
        dl = torch.empty(n, dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _cabi.check(self._lib.jmpc_set_courses_device(
            self._h, n, int(plans.traj.shape[1]), self._dp(plans.n_traj, torch.int32), self._dp(plans.traj, torch.float64),
            self._dp(plans.status, torch.int32), self._dp(dl, torch.float64), self._dp(ok, torch.int32),
            C.c_void_p(stream)), "jmpc_set_courses_device")
        self.course_len = self.get_courses(0, n, lengths_only=True)
        self.course_ok, self.course_dl = ok, dl
        self._ok_host, self._dl_host = ok.cpu().numpy(), dl.cpu().numpy()
        if self._ok_host.any():
            self.dl = float(self._dl_host[np.argmax(self._ok_host)])
            self.default_params = self.config.param_vector(dl=self.dl, dt=self.dt, L=self.L, speed=self.speed)
            _cabi.check(self._lib.jmpc_set_default_params(self._h, _ptr(self.default_params)), "jmpc_set_default_params")

    def get_courses(self, first: int = 0, n: Optional[int] = None, lengths_only: bool = False):
        """The uploaded courses first .. first + n - 1 as (N_c, 3) arrays [x, y, smoothed yaw] (jmpc_get_courses);
        with `lengths_only` just their lengths."""
        n = len(self.course_len) - first if n is None else int(n)
        lens = np.zeros(n, np.int32)
        if lengths_only:
            _cabi.check(self._lib.jmpc_get_courses(self._h, int(first), n, 0, _ptr(lens), None, None, None), "jmpc_get_courses")
            return lens
        stride = self.max_N
        tab = np.zeros((3, n, stride))
        _cabi.check(self._lib.jmpc_get_courses(self._h, int(first), n, stride, _ptr(lens), _ptr(tab[0]), _ptr(tab[1]),
                                               _ptr(tab[2])), "jmpc_get_courses")
        return [np.ascontiguousarray(tab[:, k, :lens[k]].T) for k in range(n)]

    def arc_table_flags(self, first: int = 0, n: Optional[int] = None) -> np.ndarray:
        """bool [n]: which of the uploaded courses first .. first + n - 1 got an arc-length table (jmpc_get_arc_tables);
        the collision kernel sums the arc lengths of the others on the fly."""
        n = len(self.course_len) - first if n is None else int(n)
        has = np.zeros(n, np.int32)
        _cabi.check(self._lib.jmpc_get_arc_tables(self._h, int(first), n, _ptr(has)), "jmpc_get_arc_tables")
        return has != 0

    # ---- configuration ----------------------------------------------------------------------------------
    def set_courses(self, courses: Sequence[np.ndarray]):
        lens = _i32([len(c) for c in courses])
        stride = int(lens.max())
        tab = np.zeros((3, len(courses), stride))
        for k, c in enumerate(courses):
            c = np.asarray(c, dtype=np.float64)
            tab[0, k, :len(c)] = c[:, 0]
            tab[1, k, :len(c)] = c[:, 1]
            tab[2, k, :len(c)] = c[:, 2]
        _cabi.check(self._lib.jmpc_set_courses(self._h, len(courses), stride, _ptr(lens), _ptr(tab[0]), _ptr(tab[1]),
                                               _ptr(tab[2])), "jmpc_set_courses")
        self.course_len = lens.copy()
        self.course_ok = self.course_dl = None

    def set_course_speed(self, speeds: Optional[Sequence[np.ndarray]]):
        """Reference speed profile per course point (`cv` of main/lib/mpc_with_speed.py:104): one array per uploaded
        course, or None to go back to the two-level v_ref / v_ref_cut parameters."""
        if speeds is None:
            _cabi.check(self._lib.jmpc_set_course_speed(self._h, 0, 0, None), "jmpc_set_course_speed")
            return
        if len(speeds) != len(self.course_len):
            raise ValueError("one speed profile per uploaded course")
        stride = int(self.course_len.max())
        tab = np.zeros((len(speeds), stride))
        for k, v in enumerate(speeds):
            v = np.asarray(v, dtype=np.float64)
            if len(v) < self.course_len[k]:
                raise ValueError("speed profile shorter than its course")
            tab[k, :self.course_len[k]] = v[:self.course_len[k]]
        _cabi.check(self._lib.jmpc_set_course_speed(self._h, len(speeds), stride, _ptr(tab)), "jmpc_set_course_speed")

    HOST_TRANSFER = {"staged": 0, "zero_copy_results": 1, "zero_copy": 2}

    def set_host_transfer(self, mode: str):
        """How `step_host` / `collision_host` move data: "zero_copy_results" (default: inputs by DMA, results stored by
        the kernel straight into page-locked host memory), "staged" (DMA both ways) or "zero_copy" (inputs read
        through the mapping as well) -- jmpc_set_host_transfer in include/jmpc.h."""
        _cabi.check(self._lib.jmpc_set_host_transfer(self._h, self.HOST_TRANSFER[mode]), "jmpc_set_host_transfer")

    def set_default_params(self, params: np.ndarray):
        self.default_params = _f64(params, (NPARAM,))
        _cabi.check(self._lib.jmpc_set_default_params(self._h, _ptr(self.default_params)), "jmpc_set_default_params")

    def set_car_geometry(self, front_offset: float, rear_offset: float, radius: float):
        _cabi.check(self._lib.jmpc_set_car_geometry(self._h, float(front_offset), float(rear_offset), float(radius)),
                    "jmpc_set_car_geometry")
        self.car_radius = float(radius)

    SCHEDULES = {"index": 0, "apriori": 1, "history": 2}

    def set_schedule(self, mode: str):
        """Order of the solver's work queue: "index", "apriori" (longest first by a key computed from the inputs) or
        "history" (by the iteration count of the same instance index in the previous step, a-priori key when there
        is none) -- see jmpc_set_schedule in include/jmpc.h."""
        _cabi.check(self._lib.jmpc_set_schedule(self._h, self.SCHEDULES[mode]), "jmpc_set_schedule")
        self.schedule = mode

    def reset_schedule_hints(self):
        _cabi.check(self._lib.jmpc_reset_schedule_hints(self._h), "jmpc_reset_schedule_hints")

    def set_skip_mask(self, mask):
        """`mask`: CUDA int32 tensor [B] (kept alive by the caller) or None.  Instances with mask != 0 are skipped by
        the step and collision kernels."""
        _cabi.check(self._lib.jmpc_set_skip_mask(self._h, None if mask is None else C.c_void_p(mask.data_ptr())),
                    "jmpc_set_skip_mask")

    def set_record_peers(self, peer_table_ptrs, rank_offset: int):
        """Fused all-gather: from now on the step kernel's epilogue also stores every instance's result record into
        row `rank_offset + b` of each peer GPU's gathered table.  `peer_table_ptrs`: device pointers (ints) of the
        [world * B, RECORD_LEN] tables of all ranks as seen from this GPU (symmetric memory `buffer_ptrs`); an empty
        list switches it off."""
        ptrs = (C.c_uint64 * max(len(peer_table_ptrs), 1))(*[int(p) for p in peer_table_ptrs])
        _cabi.check(self._lib.jmpc_set_record_peers(self._h, len(peer_table_ptrs), ptrs, int(rank_offset)),
                    "jmpc_set_record_peers")

    def set_record_flags(self, peer_flag_ptrs, step: int):
        """Completion flags of the fused all-gather (jmpc_set_record_flags): from now on the last retiring block of
        every step launch stores `step` into the given addresses (this rank's slot in every rank's flag array)."""
        ptrs = (C.c_uint64 * max(len(peer_flag_ptrs), 1))(*[int(p) for p in peer_flag_ptrs])
        _cabi.check(self._lib.jmpc_set_record_flags(self._h, len(peer_flag_ptrs), ptrs, int(step)), "jmpc_set_record_flags")

    def gather_wait(self, flags, world: int, step: int, stream: Optional[int] = None):
        """Enqueue the wait for all `world` ranks to have published `step` in the local flag array `flags` (CUDA int64)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        _cabi.check(self._lib.jmpc_gather_wait(self._h, C.c_void_p(flags.data_ptr()), int(world), int(step),
                                               C.c_void_p(stream)), "jmpc_gather_wait")

    def gather_timed_out(self) -> bool:
        v = C.c_int32(0)
        _cabi.check(self._lib.jmpc_gather_timed_out(self._h, C.byref(v)), "jmpc_gather_timed_out")
        return bool(v.value)

    def close(self):
        if getattr(self, "_h", None):
            self._host_out = {}
            for p in getattr(self, "_pinned", []):
                self._lib.jmpc_host_free(self._h, p)
            self._pinned = []
            self._lib.jmpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._lib.jmpc_launch_count(self._h))

    def measure_fma_peak(self):
        a, b = C.c_double(), C.c_double()
        _cabi.check(self._lib.jmpc_measure_fma_peak(self._h, C.byref(a), C.byref(b)), "jmpc_measure_fma_peak")
        return a.value, b.value

    def debug_linalg(self, A, b, x, full: bool = False, group_lanes: int = 32, which: int = 0):
        """Building-block self-test: returns (A^{-1} b, A x, ok) computed by the tiled routines on one lane group
        (`group_lanes` = 32: a warp; 16: half `which` of a warp whose two halves both run the problem)."""
        A = _f64(A)
        n = A.shape[0]
        b, x = _f64(b, (n,)), _f64(x, (n,))
        sol, prod = np.zeros(2 * n), np.zeros(2 * n)
        rc = self._lib.jmpc_debug_linalg_g(self._h, n, int(group_lanes), int(which), _ptr(A), _ptr(b), _ptr(x), _ptr(sol),
                                           _ptr(prod))
        if rc < 0:
            _cabi.check(rc, "jmpc_debug_linalg")
        if group_lanes != 32:               # only the solver-layout matvec exists for a half warp
            return (sol, prod, rc == 0) if full else (sol[:n], prod[n:], rc == 0)
        if n % 2 == 0 and not full:         # the matvec in the solver's row layout must agree with the tiled one
            np.testing.assert_allclose(prod[n:], prod[:n], rtol=1e-13, atol=1e-13 * np.abs(A).max())
        return (sol, prod, rc == 0) if full else (sol[:n], prod[:n], rc == 0)

    # ---- page-locked host arrays --------------------------------------------------------------------------
    def pinned_empty(self, shape, dtype=np.float64) -> np.ndarray:
        """numpy array in page-locked memory owned by this engine (freed by close())."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _cabi.check(self._lib.jmpc_host_alloc(self._h, n, C.byref(p)), "jmpc_host_alloc")
        self._pinned.append(p)
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def host_outputs(self, B: int, T: Optional[int] = None) -> StepOutput:
        """Reusable page-locked result arrays for `step_host(..., out=...)`: no allocation, page faults or staging
        copy per step.  Contents are overwritten by the next call that is given the same object."""
        T = int(T or self.T)
        key = (B, T)
        if key not in self._host_out:
            f, i = self.pinned_empty, lambda s: self.pinned_empty(s, np.int32)
            self._host_out[key] = StepOutput(oa=f((B, T)), od=f((B, T)), ox=f((B, T + 1)), oy=f((B, T + 1)),
                                             ov=f((B, T + 1)), oyaw=f((B, T + 1)), xref=f((B, 4, T + 1)), cost=f((B,)),
                                             status=i((B,)), iters=i((B,)), target_ind=i((B,)),
                                             record=f((B, _cabi.RECORD_LEN)))
        return self._host_out[key]

    # ---- host path --------------------------------------------------------------------------------------
    def step_host(self, state, target_ind, oa=None, od=None, course_id=None, course_len=None, warm=None,
                  params=None, T: Optional[int] = None, out: Optional[StepOutput] = None) -> StepOutput:
        T = int(T or self.T)
        if out is not None:
            return self._step_host_into(out, T, state, target_ind, oa, od, course_id, course_len, warm, params)
        state = _f64(state)
        B = state.shape[0]
        if state.shape != (B, 4):
            raise ValueError("state must be [B, 4] (x, y, v, yaw)")
        T1 = T + 1
        if oa is None or od is None:
            oa_b, od_b = np.zeros((B, T)), np.zeros((B, T))
            warm = np.zeros(B, np.int32)
        else:
            oa_b, od_b = _f64(oa, (B, T)).copy(), _f64(od, (B, T)).copy()
        tgt = _i32(target_ind, (B,)).copy()
        cid = None if course_id is None else _i32(course_id, (B,))
        clen = None if course_len is None else _i32(course_len, (B,))
        wrm = None if warm is None else _i32(warm, (B,))
        prm = None if params is None else _f64(params, (B, NPARAM))
        ox, oy, ov, oyaw = (np.zeros((B, T1)) for _ in range(4))
        xref = np.zeros((B, 4, T1))
        cost = np.full(B, np.nan)
        status = np.zeros(B, np.int32)
        iters = np.zeros(B, np.int32)
        record = np.zeros((B, _cabi.RECORD_LEN))
        _cabi.check(self._lib.jmpc_step_host(self._h, B, T, _ptr(state), _ptr(cid), _ptr(clen), _ptr(tgt), _ptr(wrm),
                                             _ptr(oa_b), _ptr(od_b), _ptr(prm), _ptr(ox), _ptr(oy), _ptr(ov),
                                             _ptr(oyaw), _ptr(xref), _ptr(cost), _ptr(status), _ptr(iters),
                                             _ptr(record)), "jmpc_step_host")
        return StepOutput(oa_b, od_b, ox, oy, ov, oyaw, xref, cost, status, iters, tgt, record)

    def _step_host_into(self, out, T, state, target_ind, oa, od, course_id, course_len, warm, params) -> StepOutput:
        """Results into the caller's (page-locked) `out`; the inputs are only read.  `oa` / `od` / `target_ind` may be
        `out`'s own arrays (a closed loop feeding its previous solution back), in which case nothing is copied."""
        state = _f64(state)
        B = state.shape[0]
        if out.oa.shape != (B, T):
            raise ValueError("`out` was made for another batch size / horizon")
        if oa is None or od is None:
            out.oa[...] = 0.0
            out.od[...] = 0.0
            oa_in, od_in = out.oa, out.od
            warm = np.zeros(B, np.int32)
        else:
            oa_in = oa if oa is out.oa else _f64(oa, (B, T))
            od_in = od if od is out.od else _f64(od, (B, T))
        tgt_in = target_ind if target_ind is out.target_ind else _i32(target_ind, (B,))
        cid = None if course_id is None else _i32(course_id, (B,))
        clen = None if course_len is None else _i32(course_len, (B,))
        wrm = None if warm is None else _i32(warm, (B,))
        prm = None if params is None else _f64(params, (B, NPARAM))
        _cabi.check(self._lib.jmpc_step_host_io(
            self._h, B, T, _ptr(state), _ptr(cid), _ptr(clen), _ptr(tgt_in), _ptr(wrm), _ptr(oa_in), _ptr(od_in),
            _ptr(prm), _ptr(out.target_ind), _ptr(out.oa), _ptr(out.od), _ptr(out.ox), _ptr(out.oy), _ptr(out.ov),
            _ptr(out.oyaw), _ptr(out.xref), _ptr(out.cost), _ptr(out.status), _ptr(out.iters), _ptr(out.record)),
            "jmpc_step_host_io")
        return out

    def collision_host(self, agent_idx, v, obstacles, frame_window: int, margin: int, course_id=None,
                       params=None, horizon_s: float = 7.0, out=None):
        """obstacles: [B, n_obs, 6].  Returns (flag[B] int32, course_len[B] int32); `out` = (flag, course_len) arrays
        to fill instead (page-locked ones from `pinned_empty` are written by the kernel directly)."""
        agent_idx = _i32(agent_idx)
        B = agent_idx.shape[0]
        obstacles = _f64(obstacles)
        n_obs = obstacles.shape[1] if obstacles.ndim == 3 else 0
        if out is not None:
            flag, clen = out
            if flag.dtype != np.int32 or clen.dtype != np.int32 or flag.shape != (B,) or clen.shape != (B,):
                raise ValueError("`out` must be two int32 arrays of shape [B]")
        else:
            flag = np.zeros(B, np.int32)
            clen = np.zeros(B, np.int32)
        _cabi.check(self._lib.jmpc_collision_host(
            self._h, B, _ptr(None if course_id is None else _i32(course_id, (B,))), _ptr(agent_idx), _ptr(_f64(v, (B,))),
            _ptr(obstacles) if n_obs else None, n_obs, int(frame_window), int(margin), float(horizon_s),
            _ptr(None if params is None else _f64(params, (B, NPARAM))), _ptr(flag), _ptr(clen)), "jmpc_collision_host")
        return flag, clen

    # ---- device path (torch tensors) -----------------------------------------------------------------------
    @staticmethod
    def _dp(t, dtype=None):
        if t is None:
            return None
        if not t.is_cuda or not t.is_contiguous():
            raise ValueError("device path needs contiguous CUDA tensors")
        if dtype is not None and t.dtype != dtype:
            raise ValueError(f"expected {dtype}, got {t.dtype}")
        return C.c_void_p(t.data_ptr())

    def alloc_outputs(self, B: int, T: Optional[int] = None):
        import torch
        T = int(T or self.T)
        dev = torch.device("cuda", self.device)
        f = lambda *s: torch.empty(*s, dtype=torch.float64, device=dev)  # noqa: E731
        i = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)    # noqa: E731
        return StepOutput(oa=None, od=None, ox=f(B, T + 1), oy=f(B, T + 1), ov=f(B, T + 1), oyaw=f(B, T + 1),
                          xref=f(B, 4, T + 1), cost=f(B), status=i(B), iters=i(B), target_ind=None,
                          record=f(B, _cabi.RECORD_LEN))

    def step(self, state, target_ind, oa, od, out: StepOutput, course_id=None, course_len=None, warm=None,
             params=None, T: Optional[int] = None, stream: Optional[int] = None) -> StepOutput:
        """All arguments are CUDA tensors; `target_ind`, `oa`, `od` are updated in place; `out` from alloc_outputs."""
        import torch
        T = int(T or self.T)
        B = state.shape[0]
        f64, i32 = torch.float64, torch.int32
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        _cabi.check(self._lib.jmpc_step(
            self._h, B, T, self._dp(state, f64), self._dp(course_id, i32), self._dp(course_len, i32),
            self._dp(target_ind, i32), self._dp(warm, i32), self._dp(oa, f64), self._dp(od, f64), self._dp(params, f64),
            self._dp(out.ox, f64), self._dp(out.oy, f64), self._dp(out.ov, f64), self._dp(out.oyaw, f64),
            self._dp(out.xref, f64), self._dp(out.cost, f64), self._dp(out.status, i32), self._dp(out.iters, i32),
            self._dp(out.record, f64), C.c_void_p(stream)), "jmpc_step")
        out.oa, out.od, out.target_ind = oa, od, target_ind
        return out

    def collision(self, agent_idx, v, obstacles, frame_window: int, margin: int, flag, course_len_out,
                  course_id=None, params=None, horizon_s: float = 7.0, stream: Optional[int] = None, plans=None,
                  n_planned: int = 0, consider=None):
        """Collision flags and cut lengths on the device.  plans [B, n_planned, plan_len, 2] float64 (optional): per-step
        (a, steer) inputs that predict obstacle slots 0 .. n_planned - 1 instead of their rows' constant inputs
        (jmpc_collision_planned in include/jmpc.h).  consider [B] int32 (optional): bit s set = obstacle slot s takes
        part in the cut; the others are ignored (jmpc_collision_masked)."""
        import torch
        B = agent_idx.shape[0]
        n_obs = int(obstacles.shape[1]) if obstacles is not None else 0
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        if plans is not None:
            n_planned = int(n_planned)
            if plans.dim() != 4 or plans.shape[0] != B or plans.shape[1] != n_planned or plans.shape[3] != 2:
                raise ValueError(f"plans must be [{B}, {n_planned}, plan_len, 2]")
        if consider is not None:
            if tuple(consider.shape) != (B,):
                raise ValueError(f"consider must be [{B}]")
            planned = plans is not None and n_planned > 0
            _cabi.check(self._lib.jmpc_collision_masked(
                self._h, B, self._dp(course_id, torch.int32), self._dp(agent_idx, torch.int32),
                self._dp(v, torch.float64), self._dp(obstacles, torch.float64), n_obs,
                self._dp(plans, torch.float64) if planned else None, n_planned if planned else 0,
                int(plans.shape[2]) if planned else 1, self._dp(consider, torch.int32), int(frame_window), int(margin),
                float(horizon_s), self._dp(params, torch.float64), self._dp(flag, torch.int32),
                self._dp(course_len_out, torch.int32), C.c_void_p(stream)), "jmpc_collision_masked")
            return flag, course_len_out
        if plans is not None:
            _cabi.check(self._lib.jmpc_collision_planned(
                self._h, B, self._dp(course_id, torch.int32), self._dp(agent_idx, torch.int32),
                self._dp(v, torch.float64), self._dp(obstacles, torch.float64), n_obs, self._dp(plans, torch.float64),
                n_planned, int(plans.shape[2]), int(frame_window), int(margin), float(horizon_s),
                self._dp(params, torch.float64), self._dp(flag, torch.int32), self._dp(course_len_out, torch.int32),
                C.c_void_p(stream)), "jmpc_collision_planned")
            return flag, course_len_out
        _cabi.check(self._lib.jmpc_collision(
            self._h, B, self._dp(course_id, torch.int32), self._dp(agent_idx, torch.int32), self._dp(v, torch.float64),
            self._dp(obstacles, torch.float64), n_obs, int(frame_window), int(margin), float(horizon_s),
            self._dp(params, torch.float64), self._dp(flag, torch.int32), self._dp(course_len_out, torch.int32),
            C.c_void_p(stream)), "jmpc_collision")
        return flag, course_len_out

    def plant_step(self, state, a, delta, params=None, stream: Optional[int] = None):
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        _cabi.check(self._lib.jmpc_plant_step(self._h, state.shape[0], self._dp(state, torch.float64),
                                              self._dp(a, torch.float64), self._dp(delta, torch.float64),
                                              self._dp(params, torch.float64), C.c_void_p(stream)), "jmpc_plant_step")
        return state
