/*
 * jmpc.h -- C ABI of libjmpc.so: the batched JunctionSim MPC step on B200 (sm_100a).
 *
 * This is the drop-in boundary for the per-timestep controller hot path of
 * SaeedRahmani/AV-Simulation-at-Intersections (paths below are relative to that repository).  The reference
 * has no FFI of its own (it is pure Python); the entry points here are what a ctypes binding placed behind
 * `lib.mpc.MPC` binds (INTEGRATION.md shows that stub).  Plain pointers and sizes only; no C++ or torch
 * types cross this boundary; no C++ exception escapes it.
 *
 * Memory convention
 *   - `jmpc_step` / `jmpc_collision` take DEVICE pointers (e.g. torch tensors' data_ptr()) and only enqueue
 *     work on `stream`; they never synchronise.
 *   - `jmpc_step_host[_io]` / `jmpc_collision_host` take HOST pointers, run the same kernels and return after the
 *     results are on the host (step: the kernel accesses page-locked host memory directly; collision: staged
 *     through pinned buffers owned by the handle).
 *   - Arrays are instance-major ("batch first"), float64 / int32, densely packed:
 *       state      [B][4]         x, y, v, yaw            (main/lib/mpc.py:291)
 *       oa, od     [B][T]         accelerations / steering angles; in: previous solution (the linearisation
 *                                 point, mpc.py:225-227,293-296; zeros when there is none), out: new solution
 *       ox,oy,ov,oyaw [B][T+1]    predicted states          (mpc.py:199-205)
 *       xref       [B][4][T+1]    sampled reference         (mpc.py:89-112)
 *       params     [B][JMPC_NPARAM]  optional per-instance parameters (NULL -> handle defaults)
 *       obstacles  [B][n_obs][6]  x, y, v, yaw, a, steer    (main/lib/moving_obstacles.py:229-232 `get()`)
 *   - A lane group (a warp, or half a warp for horizons T <= 15) owns an instance, so instance-major rows are
 *     what it reads coalesced.
 *
 * Threading: one handle per (host thread, device); calls on one handle must be serialised by the caller.
 */
#ifndef JMPC_H_
#define JMPC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JMPC_ABI_VERSION 2
#define JMPC_RECORD_LEN 8         /* doubles per instance in the packed result record, see jmpc_step */
#define JMPC_MAX_PEERS 8          /* GPUs of one NVSwitch box */
#define JMPC_MAX_T 31           /* horizon limit of the lane-per-stage kernels (reference GUI range 5..25) */

/* Row order of a parameter vector.  Derivations as in main/lib/mpc.py:14-39 and main/lib/simulation.py:23-25:
 * Qf_* already multiplied by T (mpc.py:28), max_dsteer in rad/s (mpc.py:37). */
enum jmpc_param {
  JMPC_P_DT = 0,        /* sample time [s]                          MPC(..., dt)            mpc.py:247 */
  JMPC_P_DL,            /* course tick [m]                          MPC(..., dl)                       */
  JMPC_P_L,             /* wheelbase                                car_dimensions.py:84               */
  JMPC_P_SPEED,         /* speed cap of the QP                      MPC(..., speed)         mpc.py:190 */
  JMPC_P_W_PERP, JMPC_P_W_PARA,                     /* mpc.py:23-24                                    */
  JMPC_P_R_A, JMPC_P_R_D,                           /* R  = diag(.,.)                        mpc.py:25 */
  JMPC_P_RD_A, JMPC_P_RD_D,                         /* Rd = diag(.,.)                        mpc.py:26 */
  JMPC_P_Q_V, JMPC_P_Q_YAW,                         /* Q_v_yaw                               mpc.py:27 */
  JMPC_P_QF_X, JMPC_P_QF_Y, JMPC_P_QF_V, JMPC_P_QF_YAW,  /* Qf * T                           mpc.py:28 */
  JMPC_P_REND_A, JMPC_P_REND_D,                     /* input weight once the course end is reached, mpc.py:181 */
  JMPC_P_MAX_DSTEER,    /* rad/s                                                             mpc.py:37 */
  JMPC_P_MAX_ACCEL, JMPC_P_MAX_DECEL,               /*                                       mpc.py:38-39 */
  JMPC_P_MAX_STEER,     /* Simulation.MAX_STEER                                        simulation.py:23 */
  JMPC_P_SIM_MAX_SPEED, /* Simulation.MAX_SPEED (rollout clamp, not the QP cap)        simulation.py:24 */
  JMPC_P_MIN_SPEED,     /* Simulation.MIN_SPEED                                        simulation.py:25 */
  JMPC_P_V_REF_MIN,     /* 10/3.6: floor of the reference-sampling speed                     mpc.py:99 */
  JMPC_P_V_REF,         /* reference speed profile, main/lib/mpc_with_speed.py:104,280-282: xref[2, t] = V_REF     */
  JMPC_P_V_REF_CUT,     /*   while the sampled course index is < V_REF_CUT, 0 beyond it (cv[cutoff_idx:] = 0);      */
                        /*   defaults 0 and 1e9 reproduce lib.mpc, whose xref speed row is always 0 (mpc.py:107)    */
  JMPC_NPARAM
};

/* Per-instance status word. */
enum jmpc_status {
  JMPC_OPTIMAL = 0,      /* cvxpy OPTIMAL / OPTIMAL_INACCURATE branch                     mpc.py:199-205 */
  JMPC_MAX_ITER = 1,     /* iteration cap hit without meeting even the reduced tolerances: a failed solve, handled
                            like any solver status other than OPTIMAL / OPTIMAL_INACCURATE (mpc.py:199-209):
                            control outputs are left untouched, xref/target_ind are valid, record.ai = MAX_DECEL */
  JMPC_INFEASIBLE = 2,   /* v0 outside [MIN_SPEED, speed]: reference prints "Cannot solve mpc", mpc.py:207-209;
                            control outputs are left untouched, xref/target_ind are valid                */
  JMPC_INDEX_RULE = 3    /* nearest-index rule failed: reference raises at trajectories.py:120;
                            nothing is written for the instance                                          */
};

typedef struct jmpc_handle_s* jmpc_handle;

/* Solver options (all have defaults; pass NULL to jmpc_create). */
typedef struct {
  int32_t max_solver_iters;   /* interior-point iteration cap (default 40)                                 */
  int32_t linearisation_iters;/* MAX_ITER of mpc_config.json (default 1)                     mpc.py:231   */
  double  mu_tol;             /* complementarity target (default 1e-13)                                    */
  int32_t warps_per_sm;       /* resident solver warps per SM, 0 = auto (auto also picks the low-latency
                                 kernels for launches of at most eight warps per SM; same results)          */
  double  du_th;              /* > 0: leave the linearisation loop once sum|oa - poa| + sum|od - pod| <= du_th;
                                 the exit the reference left commented out at mpc.py:236-240 (DU_TH of
                                 mpc_config.json).  Default 0 = off, as in the reference.                  */
} jmpc_options;

/* Library / ABI introspection. */
int32_t     jmpc_abi_version(void);
int32_t     jmpc_nparam(void);
const char* jmpc_last_error(void);          /* thread-local message of the last failing call */

/* Create a handle on CUDA device `device` able to run batches of up to `max_B` instances with horizon up to
 * `max_T` (<= JMPC_MAX_T) over courses of up to `max_N` points.  `default_params` is a JMPC_NPARAM vector used
 * when a call passes params == NULL.  Replaces the module-level configuration of mpc.py:14-39 and the
 * constructor state of `class MPC` (mpc.py:245-277).  Returns 0 on success, <0 on error. */
int32_t jmpc_create(int32_t device, int32_t max_B, int32_t max_T, int32_t max_N, int32_t max_courses,
                    const double* default_params, const jmpc_options* options, jmpc_handle* out);
int32_t jmpc_destroy(jmpc_handle h);

/* Replace the default parameter vector. */
int32_t jmpc_set_default_params(jmpc_handle h, const double* default_params);

/* Upload course tables (HOST pointers): course c has len[c] points, stored at cx + c*stride etc.  Yaw must
 * already be smoothed (mpc.py:46-58 is a once-per-course scan the Python wrapper does in place, as
 * MPC.__init__ does at mpc.py:260).  Replaces MPC.__init__/set_trajectory_fromarray (mpc.py:279-282): a
 * truncated course `trajectory_full[:k]` is expressed per instance by `course_len` in jmpc_step. */
int32_t jmpc_set_courses(jmpc_handle h, int32_t n_courses, int32_t stride, const int32_t* len,
                         const double* cx, const double* cy, const double* cyaw);

/* Reference speed profile per course point (HOST pointer, same layout as cx; NULL clears it): xref[2, t] = cv[idx_t]
 * as main/lib/mpc_with_speed.py:104 samples it.  Without a table the speed row of xref is the two-level profile of
 * JMPC_P_V_REF / JMPC_P_V_REF_CUT (0 for lib.mpc); a finite JMPC_P_V_REF_CUT still zeroes the profile from that
 * index on (mpc_with_speed.py:280-282).  Call after jmpc_set_courses. */
int32_t jmpc_set_course_speed(jmpc_handle h, int32_t n_courses, int32_t stride, const double* cv);

/* Collision-circle geometry of the car (main/lib/car_dimensions.py:62-79): x offsets of the front and rear
 * circle centres from the rear axle and the circle radius.  Defaults are BicycleModelDimensions
 * (car_dimensions.py:82-90): 2.18, 0.68, 2/sqrt(2). */
int32_t jmpc_set_car_geometry(jmpc_handle h, double front_offset, double rear_offset, double radius);

/* One MPC step (mpc.py:284-303 -> _iterative_linear_mpc_control :214-242) for B instances with horizon T.
 * DEVICE pointers; enqueues on `stream` (a cudaStream_t passed as void*).
 *   course_id  [B] or NULL (all course 0);  course_len [B] or NULL (full length)
 *   target_ind [B] in: search start, out: new nearest index            (mpc.py:94, :298)
 *   warm       [B] or NULL: 0 -> treat oa/od as zeros (mpc.py:225-227), 1 -> use them
 *   cost       [B]: objective value at the optimum, constants included (what `prob.value` would be)
 *   iters      [B] or NULL: solver iterations used
 *   record     [B][JMPC_RECORD_LEN] or NULL: packed per-instance result written by the kernel's epilogue --
 *              {di = od[0], ai = oa[0] (MAX_DECEL when not solved, mpc.py:298-301), cost, status, target_ind,
 *              iters, v_1, yaw_1} -- one contiguous buffer, the send buffer of the multi-GPU all-gather */
int32_t jmpc_step(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                  const int32_t* course_len, int32_t* target_ind, const int32_t* warm, double* oa, double* od,
                  const double* params, double* ox, double* oy, double* ov, double* oyaw, double* xref,
                  double* cost, int32_t* status, int32_t* iters, double* record, void* stream);

/* Skip mask (DEVICE pointer, [B] int32, or NULL to clear): instances with skip[b] != 0 are left untouched by
 * subsequent jmpc_step / jmpc_collision calls on the handle -- finished episodes of a closed-loop batch cost nothing.
 * The mask belongs to the device entry points: the *_host entry points refuse to run while one is set. */
int32_t jmpc_set_skip_mask(jmpc_handle h, const int32_t* skip);

/* Order in which the work queue hands instances to the solver warps.  A batch of one to a few waves of the resident
 * warps finishes when its slowest late-started instance does, so longest-first matters (config 2: 1.27 -> 0.90 ms
 * with exact knowledge).  mode 0: index order.  mode 1: by an a-priori key computed from the inputs (how many
 * horizon stages the speed cap can bind on).  mode 2: by the solver iteration count the same instance index needed
 * in the previous jmpc_step call on this handle with the same (B, T) -- the closed-loop case, where instance b is the
 * same ego one time step later and its active set changes slowly -- falling back to mode 1 when there is no such
 * previous call.  jmpc_reset_schedule_hints forgets the recorded counts (the next call is "cold").  Results do not
 * depend on the order. */
int32_t jmpc_set_schedule(jmpc_handle h, int32_t mode);
int32_t jmpc_reset_schedule_hints(jmpc_handle h);

/* Debug builds only (-DJMPC_CYCLES): per-region clock64() totals accumulated by the step kernel (32 slots), optionally
 * cleared.  Fails in a regular build. */
int32_t jmpc_debug_cycles(jmpc_handle h, uint64_t* out32, int32_t reset);

/* Fused all-gather of the result records (multi-GPU): after this call every jmpc_step on the handle also stores each
 * instance's record into row `rank_offset + b` of every table in `peer_tables` (DEVICE pointers valid on this GPU
 * for all `n_peers` ranks including this one -- NVLink peer / symmetric memory, e.g. the `buffer_ptrs` of a
 * torch.distributed._symmetric_memory rendezvous).  Each table is [world * B][JMPC_RECORD_LEN].  The stores are
 * issued by the step kernel's epilogue; the caller only has to run a cross-GPU barrier before reading the
 * tables.  n_peers = 0 switches it off. */
int32_t jmpc_set_record_peers(jmpc_handle h, int32_t n_peers, const uint64_t* peer_tables, int64_t rank_offset);

/* Completion flags of the fused all-gather.  After jmpc_set_record_flags every jmpc_step on the handle ends with the
 * last retiring block storing `step` (release, system scope, after all record stores of the launch) into
 * `peer_flags[p]` for every peer p: the address of THIS rank's slot in rank p's flag array (DEVICE pointers valid on
 * this GPU, uint64 slots, monotonically increasing step numbers).  n_peers = 0 switches it off.
 * jmpc_gather_wait enqueues a one-warp kernel on `stream` that returns once all `world` slots of the LOCAL flag array
 * hold a value >= step, i.e. once every rank's records of that step are in this GPU's table: the only synchronisation
 * of the gather, placed where (and as late as) the reader wants it.  It gives up after ~2 s instead of hanging the GPU;
 * jmpc_gather_timed_out reports (and synchronises the device for) that. */
int32_t jmpc_set_record_flags(jmpc_handle h, int32_t n_peers, const uint64_t* peer_flags, uint64_t step);
int32_t jmpc_gather_wait(jmpc_handle h, const uint64_t* flags, int32_t world, uint64_t step, void* stream);
int32_t jmpc_gather_timed_out(jmpc_handle h, int32_t* out);

/* Same with HOST pointers: runs the step and returns when the results are in the host arrays.  The inputs are
 * copied to the device with cudaMemcpyAsync; the results take no copy pass: the kernel's epilogue stores them into
 * page-locked host memory through its device mapping -- the caller's arrays where they are page-locked
 * (jmpc_host_alloc), the handle's staging block otherwise (one host memcpy per such array).  jmpc_set_host_transfer
 * selects the other two modes: 0 stages both directions through device memory, 2 also reads the inputs through the
 * mapping (measured slower: every warp waits a PCIe round trip when it picks an instance up). */
int32_t jmpc_step_host(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                       const int32_t* course_len, int32_t* target_ind, const int32_t* warm, double* oa,
                       double* od, const double* params, double* ox, double* oy, double* ov, double* oyaw,
                       double* xref, double* cost, int32_t* status, int32_t* iters, double* record);

int32_t jmpc_set_host_transfer(jmpc_handle h, int32_t mode);     /* 0, 1 (default) or 2, see above */

/* jmpc_step_host with separate read and write arrays for the in-out quantities: the previous solution and search
 * start are read from target_in / oa_in / od_in (never written), the new ones go to target_out / oa_out / od_out
 * (which receive the input values for instances that are not solved).  *_out may alias *_in, which is exactly
 * jmpc_step_host.  A controller that keeps its warm start (mpc.py:293-296) in one place and its outputs in another
 * (fresh arrays each step, mpc.py:199-205) saves a copy per step this way. */
int32_t jmpc_step_host_io(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                          const int32_t* course_len, const int32_t* target_in, const int32_t* warm,
                          const double* oa_in, const double* od_in, const double* params, int32_t* target_out,
                          double* oa_out, double* od_out, double* ox, double* oy, double* ov, double* oyaw,
                          double* xref, double* cost, int32_t* status, int32_t* iters, double* record);

/* Page-locked host memory for the *_host entry points: arrays placed in it are transferred without the staging
 * memcpy (any page-locked memory is recognised, e.g. cudaHostAlloc or torch pin_memory). */
int32_t jmpc_host_alloc(jmpc_handle h, size_t bytes, void** out);
int32_t jmpc_host_free(jmpc_handle h, void* p);

/* Collision flag + cut index for B instances (mpc_intersection.py:111-140, collision_avoidance.py:85-124,
 * 168-180, moving_obstacles_prediction.py:21-47, trajectories.py:58-86).  DEVICE pointers.
 *   agent_idx [B]: ego index on the full course (traj_agent_idx);  v [B]: ego speed
 *   obstacles [B][n_obs][6];  frame_window: FRAME_WINDOW;  margin: EXTRA_CUTOFF_MARGIN (in course points)
 *   flag [B]: 1 when a collision is predicted;  course_len_out [B]: effective course length to feed
 *   jmpc_step (full length when flag == 0).  flag = -1 (full length) reports an instance outside the kernel's table
 *   sizes: more than 160 kept ego points or more than 71 obstacle prediction steps (the reference's scenes: 49 / 35).
 * params [B][JMPC_NPARAM] or NULL: dt, L, max_accel and sim_max_speed are read per instance.
 * Arc lengths: a course with an arc-length table (jmpc_get_arc_tables) reads them from it; the others are summed on the
 * fly in shared memory, max_N doubles per warp.  Then the kernel runs 4, 2 or 1 warps per block, the most whose
 * (max_N + 288 n_obs + 32) * 8 + 320 bytes each fit in 200 KB, and the call fails when one warp does not fit:
 * max_N <= 25528 - 288 n_obs (23224 at 8 obstacles) whenever some uploaded course lacks a table. */
int32_t jmpc_collision(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                       const double* v, const double* obstacles, int32_t n_obs, int32_t frame_window,
                       int32_t margin, double horizon_s, const double* params, int32_t* flag,
                       int32_t* course_len_out, void* stream);
int32_t jmpc_collision_host(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                            const double* v, const double* obstacles, int32_t n_obs, int32_t frame_window,
                            int32_t margin, double horizon_s, const double* params, int32_t* flag,
                            int32_t* course_len_out);

/* jmpc_collision with per-step inputs for the first n_planned obstacle slots (DEVICE pointers; every other argument,
 * check, limit, the skip mask and the launch sizing as jmpc_collision; no extra shared memory).
 *   plans [B][n_planned][plan_len][2]: (a, steer) per predictor step; 0 <= n_planned <= n_obs, plan_len >= 1, plans
 *   may be NULL only when n_planned = 0.  A planned slot is predicted with the reference's constant-input recurrence
 *   (moving_obstacles_prediction.py:21-47) fed a sequence: predictor step t uses input min(t, plan_len - 1), so past
 *   the plan the last input is held (speed unclamped, as for a constant input).  Per step the position advances with
 *   the old v and yaw, then v += a_t dt, then yaw += (v / L) tan(steer_t) dt.  The rows' columns 4 and 5 are not read
 *   for planned slots; slots n_planned .. n_obs - 1 use them as jmpc_collision does.  A plan whose entries all equal
 *   the row's (a, steer) gives jmpc_collision's flags and cut lengths bit for bit. */
int32_t jmpc_collision_planned(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                               const double* v, const double* obstacles, int32_t n_obs, const double* plans,
                               int32_t n_planned, int32_t plan_len, int32_t frame_window, int32_t margin,
                               double horizon_s, const double* params, int32_t* flag, int32_t* course_len_out,
                               void* stream);

/* Plant step for B instances (Simulation.step, simulation.py:35-47 -> Bicycle.step, bicycle/main.py:28-41).
 * DEVICE pointers; state [B][4] is advanced in place with (a, delta). */
int32_t jmpc_plant_step(jmpc_handle h, int32_t B, double* state, const double* a, const double* delta,
                        const double* params, void* stream);

/* Closed-loop episodes on the device (the scenario loop around the step, main/scenarios/mpc_intersection.py:99-163).
 * DEVICE pointers; all arrays [B] unless noted; episodes with done != 0 are left untouched by all three.  done codes
 * (enum jmpc_done): 1 goal reached, 2 the index rule raised, 3 no planned course (jmpc_episode_init_from_courses: the
 * plan failed), 4 a scene mate has no planned course (jmpc_scene_init).
 *   jmpc_episode_pre : done |= is_goal(state) (mpc.py:314-330; done = 2 when the index rule raises), then
 *                      agent_idx = nearest forward index on the full course unless the truncated course has
 *                      collapsed onto the ego's point (mpc_intersection.py:107-109).  course_len = length of the
 *                      course the MPC was last given, steps = iterations executed so far.
 *   jmpc_episode_post: takes the step's record [B][JMPC_RECORD_LEN], applies (a, delta) to the plant
 *                      (simulation.py:35-47; a = MAX_DECEL and the previous delta when the solve failed,
 *                      mpc.py:298-301), stores target_ind, sets warm (0 after a failed solve: the next step starts
 *                      from zeros, mpc.py:225-227), increments steps and, if history != NULL, writes one
 *                      History row [B][8] = x, y, yaw, v, t, delta, a, xref_deviation (simulation.py:76-84).
 *   jmpc_episode_post_dev: the same with the loop iteration i read from device memory (iter_dev): the History row goes
 *                      to history_base[i] ([rows][B][8], skipped once i >= rows), the collision flags are copied to
 *                      flags_base[i] ([rows][B]), t = (i + 1) * dt_loop.  With jmpc_counter_add (*counter += delta,
 *                      one thread) closing the iteration, the whole loop body has no per-iteration host argument and
 *                      can be captured once as a CUDA graph and replayed.
 *   jmpc_obstacle_step: constant-input motion of obstacles [B][n_obs][6] (moving_obstacles_prediction.py:21-29), with
 *                      one `dt` for the whole batch: a params row's dt reaches the collision prediction and the plant,
 *                      not this step. */
enum jmpc_done {
  JMPC_DONE_RUNNING = 0,         /* still driving                                                                  */
  JMPC_DONE_GOAL = 1,            /* is_goal fired                                                    mpc.py:314-330 */
  JMPC_DONE_INDEX_RULE = 2,      /* the nearest-index rule raised                             trajectories.py:120 */
  JMPC_DONE_NO_COURSE = 3,       /* no usable planned course: never stepped      jmpc_episode_init_from_courses */
  JMPC_DONE_MATE_NO_COURSE = 4   /* a scene mate has no usable planned course: never stepped    jmpc_scene_init */
};
int32_t jmpc_episode_pre(jmpc_handle h, int32_t B, const double* state, const int32_t* course_id,
                         const int32_t* course_len, const int32_t* target_ind, const int32_t* steps,
                         int32_t* agent_idx, int32_t* done, double goal_dis, double stop_speed, void* stream);
int32_t jmpc_episode_post(jmpc_handle h, int32_t B, double* state, const int32_t* course_id, const double* record,
                          const double* params, int32_t* target_ind, int32_t* steps, int32_t* done, double* di,
                          int32_t* warm, double* history, double t_now, void* stream);
int32_t jmpc_episode_post_dev(jmpc_handle h, int32_t B, double* state, const int32_t* course_id, const double* record,
                              const double* params, int32_t* target_ind, int32_t* steps, int32_t* done, double* di,
                              int32_t* warm, double* history_base, int32_t history_rows, int32_t* flags_base,
                              const int32_t* flag, const int32_t* iter_dev, double dt_loop, void* stream);
int32_t jmpc_counter_add(jmpc_handle h, int32_t* counter, int32_t delta, void* stream);

/* Per-episode outcome record (DEVICE pointers): contact, clearance and comfort of each closed-loop episode, accumulated
 * on the device while it runs, so that a study needs neither the History nor the obstacle poses on the host.
 * outcomes [B][JMPC_OUTCOME_LEN]: the public columns of enum jmpc_outcome, then private running state (previous pose,
 * speed, applied a and clamped steer, executed steps).  One thread per episode; episodes with done != 0 are left
 * untouched (also a done = 2 that jmpc_episode_post set in the same iteration).
 *   Evaluation e pairs an ego pose with obstacle poses of the same instant.  e = 0: the start state with the obstacles'
 *   initial poses (initial = 1: writes the empty record for every episode, then evaluates; reads no step data, record /
 *   di / flag / iter_dev may be NULL).  e = i + 1 (initial = 0, i read from iter_dev): the state after loop iteration i
 *   (History row i) with the poses iteration i + 1's collision check reads -- so enqueue it after the obstacles have
 *   advanced (jmpc_scripted_obstacle_step(advance = 1) / jmpc_obstacle_step; a recording's frame min(i + 1, S - 1))
 *   and before jmpc_counter_add.  With no step data besides the record the call also works in a captured graph.
 *   Geometry is the collision kernel's (jmpc_set_car_geometry): two circles of radius r per car, for the ego at
 *   state (x, y, yaw) and for obstacle k at obstacles[b][k] (x, y, yaw = columns 0, 1, 3).  Clearance of (ego,
 *   obstacle) = min over the 4 circle pairs of dist - 2r; contact <=> dist <= 2r for some pair (the test jmpc_collision
 *   applies to predictions).  The record only observes:
 *   nothing here changes an episode.
 *   The step columns count executed steps: flag [B] is the iteration's jmpc_collision flag (NULL: no obstacles,
 *   counts 0), the applied controls and the xref deviation are recomputed from record, di, params and the previous
 *   pose exactly as jmpc_episode_post computes them; course_id [B] or NULL (course 0) locates the target point.
 *   obstacle_history [rows + 1][B][n_obs][6] or NULL: the poses of evaluation e go to row e (skipped once e > rows),
 *   so row i + 1 is simultaneous with History row i.  Episodes that are done get no row. */
#define JMPC_OUTCOME_LEN 22       /* doubles per episode in the outcome record (JMPC_NOUTCOME public, then private) */
enum jmpc_outcome {
  JMPC_O_MIN_CLEARANCE = 0,  /* min over evaluations and obstacles of the clearance [m]            empty: +inf */
  JMPC_O_MIN_CLEARANCE_EVAL, /* evaluation where that minimum was first reached (strict <)         empty: -1   */
  JMPC_O_MIN_CLEARANCE_OBS,  /*   and its obstacle (the lowest index within the evaluation)        empty: -1   */
  JMPC_O_FIRST_CONTACT_EVAL, /* first evaluation with contact                                      empty: -1   */
  JMPC_O_FIRST_CONTACT_OBS,  /*   and the lowest obstacle index in contact then                    empty: -1   */
  JMPC_O_CONTACT_EVALS,      /* evaluations with contact                                           empty: 0    */
  JMPC_O_CUT_STEPS,          /* executed steps whose collision flag was 1 (course cut)             empty: 0    */
  JMPC_O_LIMIT_STEPS,        /* executed steps whose flag was -1 (no valid collision check)        empty: 0    */
  JMPC_O_FAILED_SOLVES,      /* executed steps whose status was not JMPC_OPTIMAL (braked, MAX_DECEL) empty: 0  */
  JMPC_O_MAX_ABS_ACCEL,      /* max |a| applied                                                    empty: 0    */
  JMPC_O_MAX_ABS_JERK,       /* max |a_i - a_{i-1}| / dt over consecutive executed steps           empty: 0    */
  JMPC_O_MAX_ABS_STEER_RATE, /* the same for the applied steer clamp(delta, +-MAX_STEER)           empty: 0    */
  JMPC_O_MAX_ABS_LAT_ACCEL,  /* max |v * (v / L) * tan(steer)|, v the speed before the step        empty: 0    */
  JMPC_O_MAX_XREF_DEV,       /* max of the xref deviation over optimal solves (History column 7)   empty: 0    */
  JMPC_O_SUM_XREF_DEV,       /*   and its sum                                                      empty: 0    */
  JMPC_O_DISTANCE,           /* path length driven: sum of hypot(dx, dy) over executed steps [m]   empty: 0    */
  JMPC_NOUTCOME
};
int32_t jmpc_episode_outcomes(jmpc_handle h, int32_t B, const double* state, const int32_t* course_id,
                              const double* obstacles, int32_t n_obs, const double* record, const double* di,
                              const int32_t* flag, const double* params, const int32_t* done, const int32_t* iter_dev,
                              int32_t initial, double* outcomes, double* obstacle_history, int32_t history_rows,
                              void* stream);

/* Scenes of several MPC-driven vehicles that see each other as moving obstacles (DEVICE pointers).  k consecutive
 * episodes form a scene: episode b = s * k + j is vehicle j of scene s (B % k == 0, k >= 1).  Every vehicle runs the
 * single-vehicle loop above unchanged; only its obstacle rows come from its scene mates.
 *   jmpc_scene_exchange writes obstacles_out [B][n_obs][6], n_obs = (k - 1) + n_extra <= 8 (the collision and outcome
 *   kernels' limit), the obstacle rows of every episode:
 *     slots 0 .. k - 2: the scene mates in episode order, skipping the episode itself (the outcome record's *_obs
 *       columns index these slots).  A mate's row is (x, y, v, yaw, a, steer): its state at that instant, the
 *       acceleration it applied in its last executed step (MAX_DECEL after a failed solve, mpc.py:298-301) and the
 *       steer it applied, clamped to +-MAX_STEER as the plant clamps it (simulation.py:38-43) -- both from the step's
 *       record, di and params as jmpc_episode_post applies them; a = steer = 0 before the mate's first step (steps = 0).
 *       Parked rule: a mate with done != 0 no longer moves and stays in the scene at its last pose with
 *       v = a = steer = 0.
 *     slots k - 1 .. n_obs - 1: the episode's own extras [B][n_extra][6] (constant-input or scripted obstacles,
 *       advanced by jmpc_obstacle_step / jmpc_scripted_obstacle_step as for a single vehicle), copied.
 *   Timing: all vehicles move simultaneously.  Enqueue one exchange before evaluation 0 / loop iteration 0 (on the start
 *   states) and one per loop iteration after jmpc_episode_post_dev and the extras' advance, before jmpc_episode_outcomes:
 *   the rows written in iteration i are the poses of evaluation i + 1 and what iteration i + 1's jmpc_collision reads,
 *   the contract of a recording's frame.  No per-iteration host argument: the call can be captured in a CUDA graph.
 *   record [B][JMPC_RECORD_LEN], di, params ([B][JMPC_NPARAM] or NULL: handle defaults), done, steps: as
 *   jmpc_episode_post leaves them; extras NULL when n_extra = 0.  Rows of every episode are written, done or not.
 *   jmpc_scene_init: the scene pass after jmpc_episode_init_from_courses.  A scene in which some episode has done = 3 is
 *   not driven: its episodes with done = 0 get done = 4 (JMPC_DONE_MATE_NO_COURSE), so no mate row is ever absent. */
int32_t jmpc_scene_exchange(jmpc_handle h, int32_t B, int32_t k, int32_t n_extra, const double* state,
                            const double* record, const double* di, const double* params, const int32_t* done,
                            const int32_t* steps, const double* extras, double* obstacles_out, void* stream);
int32_t jmpc_scene_init(jmpc_handle h, int32_t B, int32_t k, int32_t* done, void* stream);

/* Shared plans (opt-in): scene mates predicted along their own MPC plans instead of their last applied controls.
 *   jmpc_scene_plans writes plans_out [B][k - 1][T - 1][2], the inputs jmpc_collision_planned reads for the mate slots
 *   0 .. k - 2 (n_planned = k - 1, plan_len = T - 1).  The mate rows of jmpc_scene_exchange are unchanged; only their
 *   prediction changes.  For mate m of a slot and predictor step t = 0 .. T - 2 the input is
 *   (oa[m][t + 1], clamp(od[m][t + 1], +-MAX_STEER of m)): the rest of the plan of m's last solve, whose step 0 m has
 *   just applied.  A mate without a valid plan -- done[m] != 0 (parked), or warm[m] = 0 (before its first step, after a
 *   failed solve) -- gets its row's (a, steer) repeated, so that its slot predicts exactly as the constant-input row.
 *   oa, od [B][T] and warm, done [B] as jmpc_step / jmpc_episode_post_dev leave them; params [B][JMPC_NPARAM] or NULL;
 *   obstacles [B][n_obs][6] the rows jmpc_scene_exchange wrote, n_obs in [k - 1, 8].  T >= 2.  k = 1 writes nothing.
 *   Timing: enqueue it after every jmpc_scene_exchange (before iteration 0 and once per iteration); no per-iteration
 *   host argument.  The predictor runs at the evaluating vehicle's dt, so the vehicles of a scene must share dt. */
int32_t jmpc_scene_plans(jmpc_handle h, int32_t B, int32_t k, int32_t T, const double* oa, const double* od,
                         const int32_t* warm, const int32_t* done, const double* params, const double* obstacles,
                         int32_t n_obs, double* plans_out, void* stream);

/* Right-of-way rules (opt-in): which scene mates a vehicle yields to.  Without a rule every vehicle cuts its course in
 * front of every mate whose prediction crosses it, so two vehicles that cross both stop and wait for each other.
 * A rule sets a per-episode consider mask, consider [B] int32: bit s set = obstacle slot s takes part in the episode's
 * collision cut (jmpc_collision_masked).  It changes nothing else: the mate rows, the outcome record (contacts with
 * ignored mates are still measured) and obstacle_history stay as they are.
 *   Always considered: the extras (slots k - 1 ..; they do not react) and parked mates (done != 0 at the collision
 *   instant).  A moving mate m is considered by b only if m comes before b in the scene's total order of keys
 *   (cls, key, episode index), compared lexicographically; so the first vehicle of a scene yields only to parked cars
 *   and extras, and no cycle of waiting forms between moving vehicles.  The mask has every bit set except the mate
 *   slots b ignores; a finished episode (done != 0) gets -1.  Mate slot s is mate s of jmpc_scene_exchange.
 *   JMPC_ROW_FIXED: cls 0, key = priority[b] (finite).
 *   JMPC_ROW_FIRST_COME: zone [B][2] = (entry, exit) from jmpc_right_of_way_init, a = agent_idx[b], dl = params
 *     JMPC_P_DL of b: committed (a >= entry; inside the zone or past it) cls 0, key (exit - a) * dl, so the vehicle
 *     closest to leaving or furthest past the zone goes first; approaching (a < entry) cls 1, key (entry - a) * dl;
 *     a course that never enters the zone (entry = -1) cls 2: it yields to every moving mate.  Distances are course
 *     indices x dl, the arc length on the uniformly resampled courses.
 * jmpc_right_of_way_init writes zone_out [B][2]: the first and last index i of episode b's course (course_id [B] or
 *   NULL = course 0) with dx * dx + dy * dy <= r * r, dx = cx[i] - x, dy = cy[i] - y, evaluated without fused
 *   multiply-add; -1 / -1 when no point is inside.  junction [n_junction][3] = (x, y, r): n_junction = 1 (one zone for
 *   every scene) or B / k (scene b / k).  Enqueue it once the course ids are final.
 * jmpc_right_of_way writes consider_out [B] from agent_idx, done (as jmpc_episode_pre leaves them), params
 *   ([B][JMPC_NPARAM] or NULL: handle defaults; first_come reads JMPC_P_DL), zone (first_come) and priority [B]
 *   (fixed).  k in [2, 9].  Timing: every iteration after jmpc_episode_pre and before jmpc_collision_masked; no
 *   per-iteration host argument, so the call can be captured in a CUDA graph.
 * jmpc_collision_masked: jmpc_collision (plans = NULL, n_planned = 0) or jmpc_collision_planned with every check, the
 *   skip mask and the launch sizing of those, where only the slots whose bit is set in consider [B] (DEVICE, not NULL)
 *   take part in the cut.  The result equals the same call on the considered rows (and plans) alone, in slot order; a
 *   mask with no bit set among the n_obs slots gives flag = 0 and the full course length, as n_obs = 0 does. */
enum jmpc_right_of_way_rule {
  JMPC_ROW_FIXED = 1,            /* key = priority[b]                                                              */
  JMPC_ROW_FIRST_COME = 2        /* committed before approaching, then by distance to the zone's exit / entry     */
};
int32_t jmpc_right_of_way_init(jmpc_handle h, int32_t B, int32_t k, const int32_t* course_id, const double* junction,
                               int32_t n_junction, int32_t* zone_out, void* stream);
int32_t jmpc_right_of_way(jmpc_handle h, int32_t B, int32_t k, int32_t rule, const int32_t* agent_idx,
                          const int32_t* done, const double* params, const int32_t* zone, const double* priority,
                          int32_t* consider_out, void* stream);
int32_t jmpc_collision_masked(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                              const double* v, const double* obstacles, int32_t n_obs, const double* plans,
                              int32_t n_planned, int32_t plan_len, const int32_t* consider, int32_t frame_window,
                              int32_t margin, double horizon_s, const double* params, int32_t* flag,
                              int32_t* course_len_out, void* stream);

/* The reference's scripted obstacles on the device (main/lib/moving_obstacles.py: MovingObstacleTIntersection :166-232,
 * MovingObstacleRoundabout :28-123 including its dt = 0.2 quirk at :45 and the theta overwrite inside its steering
 * property, MovingObstacleArterial :125-164).  DEVICE pointers.
 *   script [B][n_obs][JMPC_OBS_SCRIPT_LEN]  constant description of each obstacle (enum jmpc_obs_script)
 *   model  [B][n_obs][4]   in-out: Bicycle xc, yc, theta, step counter
 *   obstacles [B][n_obs][6] out: what `get()` returns (x, y, forward_velocity, theta, 0, steering_angle), the tuple
 *             jmpc_collision consumes
 *   advance: 0 = only evaluate get() (before the first loop iteration), 1 = step() first (moving_obstacles.py:113-116)
 * Episodes with done != 0 are left untouched. */
enum jmpc_obs_kind { JMPC_OBS_CONSTANT = 0, JMPC_OBS_TINTERSECTION = 1, JMPC_OBS_ROUNDABOUT = 2, JMPC_OBS_ARTERIAL = 3 };
enum jmpc_obs_script {
  JMPC_OBS_KIND = 0,     /* jmpc_obs_kind                                                                     */
  JMPC_OBS_DIRECTION,    /* +1 left to right, -1 right to left                        moving_obstacles.py:41 */
  JMPC_OBS_TURNING,      /* 0 / 1                                                                             */
  JMPC_OBS_SPEED,        /* forward speed once moving                                                         */
  JMPC_OBS_OFFSET,       /* seconds before it starts moving; <= 0: moves at once           :44, :107-111      */
  JMPC_OBS_DT_MODEL,     /* Bicycle.sample_time (the constructor's dt)                                        */
  JMPC_OBS_DT_OFFSET,    /* dt of the offset test: the constructor's dt, 0.2 for the roundabout class (:45)   */
  JMPC_OBS_AUX,          /* roundabout: arctan(L / 5), the turning steer angle (:15-25); arterial: initial speed */
  JMPC_OBS_SCRIPT_LEN
};
int32_t jmpc_scripted_obstacle_step(jmpc_handle h, int32_t B, int32_t n_obs, const double* script, double* model,
                                    double* obstacles, const int32_t* done, int32_t advance, void* stream);
int32_t jmpc_obstacle_step(jmpc_handle h, int32_t B, int32_t n_obs, double* obstacles, const int32_t* done,
                           double dt, void* stream);

/* Batched motion-primitive A* planner (SURVEY.md 8f row f4): B independent searches, one warp each.  Replaces
 * MotionPrimitiveSearch.run (main/lib/mp_search_ww_generic.py:136-140 -> AStar.run, main/lib/a_star.py:31-78,
 * neighbour / cost / heuristic / goal functions :147-243, path_to_full_trajectory :245-256, collision test
 * main/lib/obstacles.py:157-176).  HOST pointers; no handle: the call allocates its workspace on `device`, runs, copies
 * the results back and frees it.
 *   primitives  mp_pts [n_mp][n_pts][3] points relative to the start pose, mp_len [n_mp] total_length,
 *               mp_cc [n_mp][n_cc][2] collision-check points (resampled at the car radius, one per collision circle,
 *               mp_search_ww_generic.py:121-138 -- derived on the host, once per primitive set)
 *   scenes      hp [n_scenes][max_obs][JMPC_PLAN_MAX_HP][3] half-plane rows a, b, c of every obstacle
 *               (Obstacle.to_convex(margin), obstacles.py:83-95,135-150), hp_n [n_scenes][max_obs] rows used,
 *               n_obs [n_scenes]; scene_id [B] or NULL (all scene 0)
 *   searches    start, goal_point [B][3]; goal_area [B][4] = x1, y1, x2, y2 of the goal box; allowed [B]
 *               allowed_goal_theta_difference; weights [B][9] = wh_dist, wh_theta, wh_steering, wh_obstacle,
 *               wh_center, wc_dist, wc_steering, wc_obstacle, wc_center (mp_search_ww_generic.py:27-31)
 *   limits      max_expansions nodes expanded per search, max_path nodes per path
 *   results     cost [B] (NaN unless found), status [B] (jmpc_plan_status), n_path [B], path [B][max_path][3],
 *               path_mp [B][max_path] primitive index of every edge, n_traj [B],
 *               traj [B][(max_path-1)*(n_pts-1)][3] = trajectory_full, expansions [B];
 *               log [B][max_log][5] or NULL: g, h, x, y, theta of every expanded node in order (AStar debug data);
 *               kernel_ms or NULL: duration of the search kernel by CUDA events */
#define JMPC_PLAN_MAX_HP 8
enum jmpc_plan_status {
  JMPC_PLAN_FOUND = 0,
  JMPC_PLAN_NO_SOLUTION = 1,  /* the open list ran empty: the reference raises "No solution found." (a_star.py:78) */
  JMPC_PLAN_LIMIT = 2         /* max_expansions / max_path reached (the reference has no limit)                  */
};
int32_t jmpc_plan_host(int32_t device, int32_t B, int32_t n_mp, int32_t n_pts, int32_t n_cc, const double* mp_pts,
                       const double* mp_len, const double* mp_cc, int32_t n_scenes, int32_t max_obs, const double* hp,
                       const int32_t* hp_n, const int32_t* n_obs, const int32_t* scene_id, const double* start,
                       const double* goal_point, const double* goal_area, const double* allowed, const double* weights,
                       int32_t max_expansions, int32_t max_path, int32_t max_log, double* cost, int32_t* status,
                       int32_t* n_path, double* path, int32_t* path_mp, int32_t* n_traj, double* traj,
                       int32_t* expansions, double* log, double* kernel_ms);

/* Persistent planner: the same plan_kernel as jmpc_plan_host with the primitives, scenes and per-search workspace
 * allocated once, so that planned courses can stay on the device (jmpc_set_courses_device) instead of taking the
 * allocate / upload / run / download / free round trip of jmpc_plan_host on every call.  Replaces the per-scenario
 * MotionPrimitiveSearch(...).run() of main/scenarios/mpc_intersection.py:63-66 for a batch of scenarios.
 * One handle per (host thread, device); calls on one handle must be serialised by the caller (one stream).
 *
 * jmpc_planner_create: uploads the primitive set (layouts as jmpc_plan_host) and allocates, for max_B searches, the
 *   workspace of each search -- node pool (pool_cap = max_expansions * n_mp + 1 entries of 48 bytes), heap
 *   (pool_cap int32) and closed-set hash table (table_size = smallest power of two >= 2 * max_expansions + 2, at
 *   least 64, int32 slots) -- i.e. pool_cap * 52 + table_size * 4 bytes per search (about 2 MB at max_expansions =
 *   4096 with the reference's nine primitives).  max_log = 0 disables the expansion log. */
typedef struct jmpc_planner_s* jmpc_planner;
int32_t jmpc_planner_create(int32_t device, int32_t max_B, int32_t n_mp, int32_t n_pts, int32_t n_cc, const double* mp_pts,
                            const double* mp_len, const double* mp_cc, int32_t max_expansions, int32_t max_path,
                            int32_t max_log, jmpc_planner* out);
int32_t jmpc_planner_destroy(jmpc_planner p);
/* Scenes (HOST pointers, layouts as jmpc_plan_host), uploaded once and kept until the next call.  Waits for the
 * device to finish earlier work of the handle before replacing them. */
int32_t jmpc_planner_set_scenes(jmpc_planner p, int32_t n_scenes, int32_t max_obs, const double* hp, const int32_t* hp_n,
                                const int32_t* n_obs);
/* B <= max_B searches with DEVICE pointers; only enqueues on `stream` (no allocation, no synchronisation).  Inputs
 * and results have the layouts of jmpc_plan_host with the handle's max_path and max_log (log may be NULL; a handle
 * created with max_log = 0 writes none).  scene_id [B] or NULL (all scene 0); values outside [0, n_scenes) are
 * clamped, as device entry points cannot validate.  The results are bit-identical to jmpc_plan_host's for the same
 * inputs and limits, and do not depend on what an earlier call left in the workspace: the outputs are cleared first
 * and every search resets its own hash table. */
int32_t jmpc_plan(jmpc_planner p, int32_t B, const int32_t* scene_id, const double* start, const double* goal_point,
                  const double* goal_area, const double* allowed, const double* weights, double* cost, int32_t* status,
                  int32_t* n_path, double* path, int32_t* path_mp, int32_t* n_traj, double* traj, int32_t* expansions,
                  double* log, void* stream);

/* Course tables straight from the planner's output (DEVICE pointers): course c is traj[c][0 : n_traj[c]] of a
 * [n_courses][traj_stride][3] array (jmpc_plan's traj, x, y, raw yaw).  Replaces, for a batch, what the scenario
 * script does between planning and driving (mpc_intersection.py:63-79): MPC(trajectory_full) smoothing the yaw in
 * place (mpc.py:260 -> the sequential unwrap of mpc.py:46-58, one thread per course, the same compares with pi/2 and
 * the same adds of 2 pi, so bit-identical to it) and dl = norm(trajectory_full[0, :2] - trajectory_full[1, :2])
 * (mpc_intersection.py:73, as sqrt(dx*dx + dy*dy) without fused multiply-adds).  Then the circle and arc-length
 * tables of jmpc_set_courses are built, in O(1) launches for all courses.  No trajectory byte leaves the device; the
 * call reads the n_courses lengths back (one synchronisation of `stream`) so that the handle's course lengths and the
 * arc-table budget behave as after jmpc_set_courses.
 *   plan_status [n_courses] jmpc_plan_status or NULL (all found)
 *   dl_out [n_courses]: dl of the course, NaN when unusable;  course_ok [n_courses]: 1 usable, 0 unusable
 * A course whose plan failed (status != JMPC_PLAN_FOUND), with fewer than 2 or more than max_N points, or with a
 * non-finite value is unusable: it gets a one-point placeholder -- its first trajectory point (the start pose) when
 * the plan produced one, the origin otherwise -- and never fails the call.  The tables are built on `stream`; the
 * handle's own stream (the *_host entry points) is ordered after them, other streams must be ordered by the caller. */
int32_t jmpc_set_courses_device(jmpc_handle h, int32_t n_courses, int32_t traj_stride, const int32_t* n_traj,
                                const double* traj, const int32_t* plan_status, double* dl_out, int32_t* course_ok,
                                void* stream);

/* Read courses first .. first + n - 1 back (HOST pointers): len [n], and cx / cy / cyaw [n][stride] with the points
 * beyond a course's length zeroed (all three NULL: lengths only).  Waits for the device.  For tests and for callers
 * that want to keep what was planned and smoothed. */
int32_t jmpc_get_courses(jmpc_handle h, int32_t first, int32_t n, int32_t stride, int32_t* len, double* cx, double* cy,
                         double* cyaw);

/* Which courses first .. first + n - 1 got an arc-length table (HOST pointer): has_table [n], 1 = table, 0 = the
 * collision kernel sums the arc lengths on the fly.  A course of N points needs N (N + 1) / 2 doubles; the uploads
 * (jmpc_set_courses, jmpc_set_courses_device) place them in course order while they fit in 256 MB, skipping a course
 * that does not fit.  Both paths give bit-identical results; the table saves the collision kernel a sequential sum. */
int32_t jmpc_get_arc_tables(jmpc_handle h, int32_t first, int32_t n, int32_t* has_table);

/* Episode start on the ingested courses (DEVICE pointers), the reference's State(x=trajectory_full[0, 0],
 * y=trajectory_full[0, 1], yaw=trajectory_full[0, 2], v=0) of mpc_intersection.py:76-79 after the smoothing:
 *   state [B][4] = (cx[0], cy[0], 0, cyaw[0]) of course course_id[b] (NULL: course 0; clamped to the courses)
 *   params [B][JMPC_NPARAM] or NULL: row JMPC_P_DL = dl[course] (dl NULL: untouched); other rows are left as they are
 *   done [B] = 3 ("no planned course") where course_ok[course] == 0 (course_ok NULL: all usable); untouched otherwise */
int32_t jmpc_episode_init_from_courses(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* course_ok,
                                       const double* dl, double* state, double* params, int32_t* done, void* stream);

/* Number of kernel launches issued through this handle since creation (for bench.py's gpu_launches). */
int64_t jmpc_launch_count(jmpc_handle h);

/* Measured FP64 / FP32 FMA throughput of the device in TFLOP/s (a register-resident FMA loop on every SM);
 * the denominator of the solver kernel's roofline, which is CUDA-core bound (DESIGN.md). */
int32_t jmpc_measure_fma_peak(jmpc_handle h, double* fp64_tflops, double* fp32_tflops);

/* Self-test of the solver's building blocks (4x4-tiled symmetric matvec, Cholesky, triangular solves) on one
 * warp: A is a dense symmetric positive definite n x n matrix (row major, n <= 2*JMPC_MAX_T), HOST pointers.
 * prod = A x, sol = A^{-1} b, each with 2n entries: [0, n) the results; prod[n, 2n) holds A x once more, computed
 * by the matvec in the solver's own row layout (even n only, NaN otherwise); sol[n, 2n) is unused (NaN).  Returns 0 on success, 1 when the
 * factorisation met a non-positive pivot. */
int32_t jmpc_debug_linalg(jmpc_handle h, int32_t n, const double* A, const double* b, const double* x, double* sol,
                          double* prod);
/* The same on a lane group of `group_lanes` (16 or 32) lanes: with 16, both halves of the warp work on their own copy
 * and half `which` reports; prod[0, n) is only filled for group_lanes == 32. */
int32_t jmpc_debug_linalg_g(jmpc_handle h, int32_t n, int32_t group_lanes, int32_t which, const double* A,
                            const double* b, const double* x, double* sol, double* prod);

#ifdef __cplusplus
}
#endif
#endif /* JMPC_H_ */
