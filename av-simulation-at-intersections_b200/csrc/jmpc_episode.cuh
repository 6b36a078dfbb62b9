// jmpc_episode.cuh -- the pieces of the scenario loop around the MPC step, for B closed-loop episodes on the device.
//
// Reference loop: main/scenarios/mpc_intersection.py:99-163 (identical in mpc_roundabout.py / _multi_lane.py):
//   is_goal(state) -> break                                  mpc.py:314-330            [episode_pre_kernel]
//   traj_agent_idx = nearest forward index on the full course, unless the truncated course has collapsed onto
//                    the ego's point                         mpc_intersection.py:107-109 [episode_pre_kernel]
//   collision check -> truncated course length               :111-143                  [collision_kernel]
//   delta, a = mpc.step(state)                               :146                      [mpc_step_kernel]
//   xref deviation; plant step; history                      :163, mpc.py:305-312, simulation.py:35-61 [episode_post_kernel]
// Obstacles either move with constant inputs (obstacle_step_kernel: the update of their predictor,
// moving_obstacles_prediction.py:21-29) or follow the reference's scripted steering rules
// (scripted_obstacle_kernel: MovingObstacleTIntersection / Roundabout / Arterial, moving_obstacles.py:28-232).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/jmpc.h"
#include "jmpc_collision.cuh"
#include "jmpc_step.cuh"              // nearest_index

namespace jmpc {

struct EpisodeArgs {
  int B, T;
  const double* cx; const double* cy; const double* cyaw; const int* course_n; int course_stride;
  const int* course_id;
  const double* params; ParamBlock defaults;
  double goal_dis, stop_speed;
  double* state;            // [B][4] x, y, v, yaw   (in-out)
  int* agent_idx;           // [B]   traj_agent_idx  (in-out)
  int* course_len;          // [B]   length of the course the MPC was last given (len(mpc.cx))
  int* target_ind;          // [B]   mpc.target_ind
  int* done;                // [B]   1 once is_goal fired (or the index rule failed: done = 2)
  int* steps;               // [B]   loop iterations executed
  double* di;               // [B]   last commanded steer (kept when a solve fails, mpc.py:298-301)
  int* warm;                // [B]   1 when the next step may use oa/od as its linearisation point (mpc.py:225-227)
  const double* record;     // [B][JMPC_RECORD_LEN] from the step kernel
  double* history;          // [B][8] slice for this step: x, y, yaw, v, t, delta, a, xref_deviation; or nullptr
  double t_now;
  // device-indexed variant (jmpc_episode_post_dev): the loop iteration is read from device memory, so that a
  // captured CUDA graph of the loop body can be replayed without per-iteration host arguments
  const int* iter_dev;      // nullptr -> use history / t_now above
  double* history_base;     // [rows][B][8] or nullptr
  int* flags_base;          // [rows][B] or nullptr: per-iteration copy of the collision flags
  const int* flag;          // [B]
  int history_rows;
  double dt_loop;
};

// One warp per episode: goal test, then the ego's index on the full course.
__global__ void __launch_bounds__(128) episode_pre_kernel(const EpisodeArgs A) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= A.B) return;
  if (A.done[b]) return;
  const int cid = A.course_id ? A.course_id[b] : 0;
  const double* cx = A.cx + (size_t)cid * A.course_stride;
  const double* cy = A.cy + (size_t)cid * A.course_stride;
  const double* cyaw = A.cyaw + (size_t)cid * A.course_stride;
  const int N = A.course_n[cid];
  const double x = A.state[4 * b], y = A.state[4 * b + 1], v = A.state[4 * b + 2];
  // is_goal: distance to the end of the FULL course, target index against the CURRENT course length (mpc.py:322)
  const int len = A.course_len[b];
  const double d = hypot(x - cx[N - 1], y - cy[N - 1]);
  bool goal = d <= A.goal_dis;
  if (abs(A.target_ind[b] - len) >= 5) goal = false;
  if (goal && fabs(v) <= A.stop_speed) {
    if (lane == 0) A.done[b] = 1;
    return;
  }
  // mpc_intersection.py:107: skip the update when the truncated course ends exactly at the ego's course point
  int a0 = A.agent_idx[b];
  bool update = true;
  if (A.steps[b] > 0) {
    const int last = min(len, N) - 1;
    const int at = min(a0, last);                 // tmp_trajectory[traj_agent_idx] (a0 < len always holds: cut >= a0 + 1)
    update = (cx[at] != cx[last]) || (cy[at] != cy[last]) || (cyaw[at] != cyaw[last]);
  }
  if (update) {
    const int near = nearest_index<32>(cx, cy, N, a0, x, y, lane, 0xffffffffu);
    if (near < 0) { if (lane == 0) A.done[b] = 2; return; }     // reference raises (trajectories.py:120)
    a0 = near;
  }
  if (lane == 0) A.agent_idx[b] = a0;
}

// ---- per-step arithmetic shared by episode_post_kernel and episode_outcome_kernel ---------------------------------
// Applied controls of a step: any status but OPTIMAL is a failed solve, the previous steer `di` is kept and the ego
// brakes with MAX_DECEL (mpc.py:298-301); that includes JMPC_MAX_ITER, whose record carries no controls.
__device__ __forceinline__ bool applied_controls(const double* rec, const double* prm, double di, double& delta,
                                                 double& acc) {
  const bool ok = (int)rec[3] == JMPC_OPTIMAL;
  delta = ok ? rec[0] : di;
  acc = ok ? rec[1] : prm[JMPC_P_MAX_DECEL];
  return ok;
}
// get_current_xref_deviation (mpc.py:305-312) at the course point `at`; (x, y) = ox[0], oy[0], the current position
__device__ __forceinline__ double xref_deviation(const double* cx, const double* cy, const double* cyaw, size_t at,
                                                 double x, double y) {
  const double ang = cyaw[at] + M_PI / 2;
  const double ex = cx[at] - x, ey = cy[at] - y;
  const double px = cos(ang) * ex, py = sin(ang) * ey;
  return sqrt(__dadd_rn(__dmul_rn(px, px), __dmul_rn(py, py)));
}
// the steer the plant applies and its yaw rate (simulation.py:38-43)
__device__ __forceinline__ double clamped_steer(double delta, double max_steer) {
  return fmax(fmin(delta, max_steer), -max_steer);
}
__device__ __forceinline__ double yaw_rate(double v, double L, double steer) { return __dmul_rn(v / L, tan(steer)); }

// One thread per episode: controls from the step's record, xref deviation, plant step, history, counters.
__global__ void episode_post_kernel(const EpisodeArgs A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  double* history = A.history;
  double t_now = A.t_now;
  if (A.iter_dev) {
    const int it = *A.iter_dev;
    const bool in_rows = it < A.history_rows;
    history = (A.history_base && in_rows) ? A.history_base + (size_t)it * A.B * 8 : nullptr;
    t_now = (double)(it + 1) * A.dt_loop;
    if (A.flags_base && A.flag && in_rows) A.flags_base[(size_t)it * A.B + b] = A.flag[b];     // all episodes, as the host copy did
  }
  if (A.done[b]) return;
  const double* prm = A.params ? A.params + (size_t)b * JMPC_NPARAM : A.defaults.v;
  const double* rec = A.record + (size_t)b * JMPC_RECORD_LEN;
  const int status = (int)rec[3];
  if (status == JMPC_INDEX_RULE) { A.done[b] = 2; return; }
  const int cid = A.course_id ? A.course_id[b] : 0;
  const size_t coff = (size_t)cid * A.course_stride;
  double x = A.state[4 * b], y = A.state[4 * b + 1], v = A.state[4 * b + 2], yaw = A.state[4 * b + 3];
  const int target = (int)rec[4];
  A.target_ind[b] = target;
  double delta, acc;
  const bool ok = applied_controls(rec, prm, A.di[b], delta, acc);
  const double dev = ok ? xref_deviation(A.cx, A.cy, A.cyaw, coff + target, x, y) : nan("");
  A.di[b] = delta;
  if (A.warm) A.warm[b] = ok ? 1 : 0;
  // Simulation.step (simulation.py:35-47)
  const double dt = prm[JMPC_P_DT], L = prm[JMPC_P_L];
  const double dcl = clamped_steer(delta, prm[JMPC_P_MAX_STEER]);
  const double xd = __dmul_rn(v, cos(yaw)), yd = __dmul_rn(v, sin(yaw)), td = yaw_rate(v, L, dcl);
  x = __dadd_rn(x, __dmul_rn(xd, dt));
  y = __dadd_rn(y, __dmul_rn(yd, dt));
  yaw = __dadd_rn(yaw, __dmul_rn(td, dt));
  v = __dadd_rn(v, __dmul_rn(acc, dt));
  v = fmax(fmin(v, prm[JMPC_P_SIM_MAX_SPEED]), prm[JMPC_P_MIN_SPEED]);
  A.state[4 * b] = x; A.state[4 * b + 1] = y; A.state[4 * b + 2] = v; A.state[4 * b + 3] = yaw;
  A.steps[b] += 1;
  if (history) {
    double* hrow = history + (size_t)b * 8;          // History.store (simulation.py:76-84), raw delta as stored there
    hrow[0] = x; hrow[1] = y; hrow[2] = yaw; hrow[3] = v; hrow[4] = t_now + dt; hrow[5] = delta; hrow[6] = acc;
    hrow[7] = dev;
  }
}

__global__ void counter_add_kernel(int* counter, int delta) { *counter += delta; }

// ---- per-episode outcome record (enum jmpc_outcome) ----------------------------------------------------------------
// private running state after the public columns
enum { kOutPrevX = JMPC_NOUTCOME, kOutPrevY, kOutPrevV, kOutPrevA, kOutPrevSteer, kOutSteps, kOutEnd };
static_assert(kOutEnd == JMPC_OUTCOME_LEN, "JMPC_OUTCOME_LEN must cover the private columns");

struct OutcomeArgs {
  int B, n_obs, initial, history_rows;
  const double* cx; const double* cy; const double* cyaw; int course_stride;
  const int* course_id;
  const double* params; ParamBlock defaults;
  double off_front, off_rear, radius;       // jmpc_set_car_geometry, as the collision kernel uses it
  const double* state;                      // [B][4] after this iteration's plant step
  const double* obstacles;                  // [B][n_obs][6] poses of the same instant
  const double* record; const double* di; const int* flag; const int* done; const int* iter_dev;
  double* outcomes;                         // [B][JMPC_OUTCOME_LEN]
  double* obstacle_history;                 // [history_rows + 1][B][n_obs][6] or nullptr
  // scene_outcome_kernel only (jmpc_episode_outcomes_scene)
  const int* present;                       // [B] bit s = obstacle slot s is present, or nullptr: every slot
  const int* depart;                        // [B] entry iteration: evaluation depart[b] > 0 starts b's record
};

// One thread per episode, once before the first loop iteration (initial: evaluation 0) and once per iteration after
// the obstacles have advanced (evaluation i + 1).  At most kMaxObstacles x 4 circle pairs per evaluation.
// Scene: absent slots (bit clear in present[b]) are skipped and get a NaN track row, and evaluation depart[b] takes
// the path of evaluation 0 for b.
template <bool Scene>
__device__ __forceinline__ void episode_outcome_body(const OutcomeArgs& A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  double* out = A.outcomes + (size_t)b * JMPC_OUTCOME_LEN;
  const double x = A.state[4 * b], y = A.state[4 * b + 1], v = A.state[4 * b + 2], yaw = A.state[4 * b + 3];
  int e = 0;
  bool first = A.initial != 0;
  if (Scene && !first && !A.done[b]) {      // b entered after iteration e - 1 and has taken no step yet
    e = *A.iter_dev + 1;
    first = e == A.depart[b];
  }
  if (first) {
    out[JMPC_O_MIN_CLEARANCE] = INFINITY;
    for (int c = JMPC_O_MIN_CLEARANCE_EVAL; c <= JMPC_O_FIRST_CONTACT_OBS; ++c) out[c] = -1.0;
    for (int c = JMPC_O_CONTACT_EVALS; c < JMPC_NOUTCOME; ++c) out[c] = 0.0;
    out[kOutPrevA] = 0.0; out[kOutPrevSteer] = 0.0; out[kOutSteps] = 0.0;
    if (A.done[b]) return;
  } else {
    if (A.done[b]) return;                  // no step executed in this iteration (goal, index rule) or earlier
    e = *A.iter_dev + 1;
    // the step just executed, recomputed as episode_post_kernel computed it
    const double* prm = A.params ? A.params + (size_t)b * JMPC_NPARAM : A.defaults.v;
    const double* rec = A.record + (size_t)b * JMPC_RECORD_LEN;
    const double px = out[kOutPrevX], py = out[kOutPrevY], pv = out[kOutPrevV];
    double delta, acc;
    const bool ok = applied_controls(rec, prm, A.di[b], delta, acc);
    const double dt = prm[JMPC_P_DT];
    const double steer = clamped_steer(delta, prm[JMPC_P_MAX_STEER]);
    const double lat = __dmul_rn(pv, yaw_rate(pv, prm[JMPC_P_L], steer));
    const int f = A.flag ? A.flag[b] : 0;
    if (f == 1) out[JMPC_O_CUT_STEPS] += 1.0;
    if (f == -1) out[JMPC_O_LIMIT_STEPS] += 1.0;
    if (!ok) out[JMPC_O_FAILED_SOLVES] += 1.0;
    if (ok) {
      const int cid = A.course_id ? A.course_id[b] : 0;
      const double dev = xref_deviation(A.cx, A.cy, A.cyaw, (size_t)cid * A.course_stride + (int)rec[4], px, py);
      if (isfinite(dev)) {
        out[JMPC_O_MAX_XREF_DEV] = fmax(out[JMPC_O_MAX_XREF_DEV], dev);
        out[JMPC_O_SUM_XREF_DEV] = __dadd_rn(out[JMPC_O_SUM_XREF_DEV], dev);
      }
    }
    out[JMPC_O_MAX_ABS_ACCEL] = fmax(out[JMPC_O_MAX_ABS_ACCEL], fabs(acc));
    out[JMPC_O_MAX_ABS_LAT_ACCEL] = fmax(out[JMPC_O_MAX_ABS_LAT_ACCEL], fabs(lat));
    if (out[kOutSteps] > 0.0) {
      out[JMPC_O_MAX_ABS_JERK] = fmax(out[JMPC_O_MAX_ABS_JERK], fabs((acc - out[kOutPrevA]) / dt));
      out[JMPC_O_MAX_ABS_STEER_RATE] = fmax(out[JMPC_O_MAX_ABS_STEER_RATE], fabs((steer - out[kOutPrevSteer]) / dt));
    }
    out[JMPC_O_DISTANCE] = __dadd_rn(out[JMPC_O_DISTANCE], hypot(x - px, y - py));
    out[kOutPrevA] = acc; out[kOutPrevSteer] = steer; out[kOutSteps] += 1.0;
  }
  out[kOutPrevX] = x; out[kOutPrevY] = y; out[kOutPrevV] = v;

  // evaluation e: the ego's circles against every obstacle's, same centres as the collision kernel
  double s, c;
  sincos(yaw, &s, &c);
  double ex[2], ey[2];
  circle_centre(x, y, c, s, A.off_front, ex[0], ey[0]);
  circle_centre(x, y, c, s, A.off_rear, ex[1], ey[1]);
  const double reach = 2.0 * A.radius;
  double best = out[JMPC_O_MIN_CLEARANCE];
  int best_obs = -1, contact_obs = -1;
  double* track = (A.obstacle_history && e <= A.history_rows)
                      ? A.obstacle_history + ((size_t)e * A.B + b) * A.n_obs * 6 : nullptr;
  const unsigned present = (Scene && A.present) ? (unsigned)A.present[b] : 0xffffffffu;
  for (int k = 0; k < A.n_obs; ++k) {
    const double* o = A.obstacles + ((size_t)b * A.n_obs + k) * 6;
    if (Scene && !((present >> k) & 1u)) {
      if (track)
        for (int j = 0; j < 6; ++j) track[6 * k + j] = nan("");
      continue;
    }
    if (track)
      for (int j = 0; j < 6; ++j) track[6 * k + j] = o[j];
    sincos(o[3], &s, &c);
    double ox[2], oy[2];
    circle_centre(o[0], o[1], c, s, A.off_front, ox[0], oy[0]);
    circle_centre(o[0], o[1], c, s, A.off_rear, ox[1], oy[1]);
    double clear = INFINITY;
    bool touch = false;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const double dx = ex[p >> 1] - ox[p & 1], dy = ey[p >> 1] - oy[p & 1];
      const double d = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
      clear = fmin(clear, d - reach);
      touch |= d <= reach;
    }
    if (clear < best) { best = clear; best_obs = k; }
    if (touch && contact_obs < 0) contact_obs = k;
  }
  if (best_obs >= 0) {
    out[JMPC_O_MIN_CLEARANCE] = best;
    out[JMPC_O_MIN_CLEARANCE_EVAL] = (double)e;
    out[JMPC_O_MIN_CLEARANCE_OBS] = (double)best_obs;
  }
  if (contact_obs >= 0) {
    out[JMPC_O_CONTACT_EVALS] += 1.0;
    if (out[JMPC_O_FIRST_CONTACT_EVAL] < 0.0) {
      out[JMPC_O_FIRST_CONTACT_EVAL] = (double)e;
      out[JMPC_O_FIRST_CONTACT_OBS] = (double)contact_obs;
    }
  }
}
__global__ void episode_outcome_kernel(const OutcomeArgs A) { episode_outcome_body<false>(A); }
__global__ void scene_outcome_kernel(const OutcomeArgs A) { episode_outcome_body<true>(A); }

// ---- scenes of k vehicles that see each other as obstacles (jmpc_scene_exchange, jmpc_scene_init) -----------------
// One thread per (episode, slot) of obstacles_out [B][n_obs][6], n_obs = (k - 1) + n_extra.  Slots 0 .. k - 2 are the
// scene mates of episode b = s * k + j in episode order without b itself, slots k - 1 .. are b's own extras.  A mate's
// row is the tuple the flag kernel consumes: its pose and speed, and the (a, clamped steer) it applied in its last
// step; (0, 0) before its first step; a finished mate (done != 0) is parked: v = a = steer = 0.  Copies, a select and
// the shared clamp only, so the rows are bit-exact with the state and the applied controls.
// Mate slot `slot` (0 .. k - 2) of episode b = s * k + j: the scene's episodes in order, b itself skipped.
__device__ __forceinline__ int scene_mate(int b, int k, int slot) {
  const int j = b % k;
  return b - j + (slot < j ? slot : slot + 1);
}
__global__ void scene_exchange_kernel(int count, int k, int n_obs, const double* __restrict__ state,
                                      const double* __restrict__ record, const double* __restrict__ di,
                                      const double* __restrict__ params, const ParamBlock defaults,
                                      const int* __restrict__ done, const int* __restrict__ steps,
                                      const double* __restrict__ extras, double* __restrict__ obstacles_out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int b = t / n_obs, slot = t - b * n_obs;
  double* o = obstacles_out + (size_t)t * 6;
  if (slot >= k - 1) {
    const double* e = extras + ((size_t)b * (n_obs - (k - 1)) + (slot - (k - 1))) * 6;
    for (int c = 0; c < 6; ++c) o[c] = e[c];
    return;
  }
  const int m = scene_mate(b, k, slot);
  const double* s = state + 4 * (size_t)m;
  double v = s[2], acc = 0.0, steer = 0.0;
  if (done[m]) {
    v = 0.0;
  } else if (steps[m] > 0) {
    const double* prm = params ? params + (size_t)m * JMPC_NPARAM : defaults.v;
    double delta;
    applied_controls(record + (size_t)m * JMPC_RECORD_LEN, prm, di[m], delta, acc);
    steer = clamped_steer(delta, prm[JMPC_P_MAX_STEER]);
  }
  o[0] = s[0]; o[1] = s[1]; o[2] = v; o[3] = s[3]; o[4] = acc; o[5] = steer;
}

// One thread per (episode, mate slot, plan step) of plans_out [B][k - 1][T - 1][2] (jmpc_scene_plans): the input of
// predictor step t for mate m is what m's last solve planned for its step t + 1, (oa[m][t + 1], clamp(od[m][t + 1])).
// A mate without a valid plan -- finished (done != 0) or without a usable warm start (warm = 0: before its first step,
// after a failed solve) -- repeats its row's (a, steer), so that its slot predicts exactly as the constant-input row.
__global__ void scene_plans_kernel(int count, int k, int T, int n_obs, const double* __restrict__ oa,
                                   const double* __restrict__ od, const int* __restrict__ warm,
                                   const int* __restrict__ done, const double* __restrict__ params,
                                   const ParamBlock defaults, const double* __restrict__ obstacles,
                                   double* __restrict__ plans_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int row = i / (T - 1), t = i - row * (T - 1);       // row = b * (k - 1) + slot
  const int b = row / (k - 1), slot = row - b * (k - 1);
  const int m = scene_mate(b, k, slot);
  double acc, steer;
  if (done[m] == 0 && warm[m] != 0) {
    const double* prm = params ? params + (size_t)m * JMPC_NPARAM : defaults.v;
    acc = oa[(size_t)m * T + t + 1];
    steer = clamped_steer(od[(size_t)m * T + t + 1], prm[JMPC_P_MAX_STEER]);
  } else {
    const double* o = obstacles + ((size_t)b * n_obs + slot) * 6;
    acc = o[4];
    steer = o[5];
  }
  plans_out[2 * (size_t)i] = acc;
  plans_out[2 * (size_t)i + 1] = steer;
}

// ---- right-of-way rules (jmpc_right_of_way_init, jmpc_right_of_way) ----------------------------------------------
// One warp per episode: the first and last point of its course inside the junction zone of its scene b / k,
// dx * dx + dy * dy <= r * r without fused multiply-add; -1 / -1 when the course never enters it.  zone_out [B][2].
__global__ void __launch_bounds__(128) right_of_way_init_kernel(int B, int k, const double* __restrict__ cx,
                                                                const double* __restrict__ cy,
                                                                const int* __restrict__ course_n, int course_stride,
                                                                int n_courses, const int* __restrict__ course_id,
                                                                const double* __restrict__ junction, int per_scene,
                                                                int* __restrict__ zone_out) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int cid = course_id ? min(max(course_id[b], 0), n_courses - 1) : 0;
  const double* px = cx + (size_t)cid * course_stride;
  const double* py = cy + (size_t)cid * course_stride;
  const int N = course_n[cid];
  const double* J = junction + (per_scene ? 3 * (size_t)(b / k) : 0);
  const double jx = J[0], jy = J[1], r2 = __dmul_rn(J[2], J[2]);
  int entry = 0x7fffffff, exit = -1;
  for (int i = lane; i < N; i += 32) {
    const double dx = px[i] - jx, dy = py[i] - jy;
    if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= r2) { entry = min(entry, i); exit = max(exit, i); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    entry = min(entry, __shfl_xor_sync(0xffffffffu, entry, o));
    exit = max(exit, __shfl_xor_sync(0xffffffffu, exit, o));
  }
  if (lane == 0) {
    zone_out[2 * (size_t)b] = exit < 0 ? -1 : entry;
    zone_out[2 * (size_t)b + 1] = exit;
  }
}

// The right-of-way key (cls, key) of episode m, compared lexicographically and then by episode index.
//   JMPC_ROW_FIXED: (0, priority[m]).
//   JMPC_ROW_FIRST_COME, a = agent_idx[m], zone [entry, exit]: committed (a >= entry) (0, (exit - a) dl), approaching
//   (1, (entry - a) dl), a course that never enters the zone (2, 0).
struct RowKey { int cls; double key; int idx; };
__device__ __forceinline__ bool row_before(const RowKey& p, const RowKey& q) {
  if (p.cls != q.cls) return p.cls < q.cls;
  if (p.key != q.key) return p.key < q.key;
  return p.idx < q.idx;
}
__device__ __forceinline__ RowKey row_key(int m, int rule, const int* __restrict__ agent_idx,
                                          const double* __restrict__ params, const ParamBlock& defaults,
                                          const int* __restrict__ zone, const double* __restrict__ priority) {
  if (rule == JMPC_ROW_FIXED) return RowKey{0, priority[m], m};
  const int entry = zone[2 * (size_t)m], exit = zone[2 * (size_t)m + 1], a = agent_idx[m];
  if (entry < 0) return RowKey{2, 0.0, m};
  const double dl = (params ? params + (size_t)m * JMPC_NPARAM : defaults.v)[JMPC_P_DL];
  if (a >= entry) return RowKey{0, __dmul_rn((double)(exit - a), dl), m};
  return RowKey{1, __dmul_rn((double)(entry - a), dl), m};
}
// One thread per episode b: consider[b] has every bit set except the mate slots s (0 .. k - 2) whose mate is moving
// (done = 0) and does not come before b.  Parked mates and the extras are always considered; a finished b gets -1.
__global__ void right_of_way_kernel(int B, int k, int rule, const int* __restrict__ agent_idx,
                                    const int* __restrict__ done, const double* __restrict__ params,
                                    const ParamBlock defaults, const int* __restrict__ zone,
                                    const double* __restrict__ priority, int* __restrict__ consider) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  unsigned mask = 0xffffffffu;
  if (done[b] == 0) {
    const RowKey own = row_key(b, rule, agent_idx, params, defaults, zone, priority);
    for (int slot = 0; slot < k - 1; ++slot) {
      const int m = scene_mate(b, k, slot);
      if (done[m] == 0 && !row_before(row_key(m, rule, agent_idx, params, defaults, zone, priority), own))
        mask &= ~(1u << slot);
    }
  }
  consider[b] = (int)mask;
}

// One thread per scene: a scene with an episode that has no course (done = 3) is not driven; its other episodes get
// done = 4.
__global__ void scene_init_kernel(int n_scenes, int k, int* __restrict__ done) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_scenes) return;
  int* d = done + (size_t)s * k;
  bool unplannable = false;
  for (int j = 0; j < k; ++j) unplannable |= d[j] == JMPC_DONE_NO_COURSE;
  if (!unplannable) return;
  for (int j = 0; j < k; ++j)
    if (d[j] == JMPC_DONE_RUNNING) d[j] = JMPC_DONE_MATE_NO_COURSE;
}

// ---- lifetimes of scene vehicles (jmpc_scene_depart_init, jmpc_scene_enter, jmpc_scene_presence) ---------------
// One thread per episode: a vehicle that enters later waits (done 0 -> JMPC_WAITING where depart > 0).
__global__ void scene_depart_init_kernel(int B, const int* __restrict__ depart, int* __restrict__ done) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (done[b] == JMPC_DONE_RUNNING && depart[b] > 0) done[b] = JMPC_WAITING;
}
// One thread per episode, at the end of loop iteration i: the vehicles that take their first step in iteration i + 1
// enter (JMPC_WAITING -> 0), so that evaluation i + 1 sees them.
__global__ void scene_enter_kernel(int B, const int* __restrict__ depart, const int* __restrict__ iter_dev,
                                   int* __restrict__ done) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (done[b] == JMPC_WAITING && depart[b] <= *iter_dev + 1) done[b] = JMPC_DONE_RUNNING;
}
// One thread per episode b: clears bit s of mask[b] for every absent mate in slot s (waiting, or gone after its goal
// with leave != 0).  combine = 0 starts from -1, combine = 1 from mask[b] (a right-of-way rule's consider mask).
__global__ void scene_presence_kernel(int B, int k, int leave, const int* __restrict__ done, int* __restrict__ mask,
                                      int combine) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  unsigned m = combine ? (unsigned)mask[b] : 0xffffffffu;
  for (int slot = 0; slot < k - 1; ++slot) {
    const int d = done[scene_mate(b, k, slot)];
    if (d == JMPC_WAITING || (leave && d == JMPC_DONE_GOAL)) m &= ~(1u << slot);
  }
  mask[b] = (int)m;
}
// ---- trips through scene slots (jmpc_scene_trips, jmpc_scene_trips_finish) -----------------------------------------
enum { kTripPending = 0, kTripInSlot = 1, kTripClosed = 2 };

// The outcome record's clearance between two poses (x, y, ., yaw) >= gap.  far2: squared distance of the reference
// points beyond which no circle pair can come within gap (a shortcut that skips the exact test, never a decision).
__device__ __forceinline__ bool start_clear(const double* p, const double* q, double off_front, double off_rear,
                                            double reach, double gap, double far2) {
  const double rx = p[0] - q[0], ry = p[1] - q[1];
  if (rx * rx + ry * ry > far2) return true;
  double s, c, px[2], py[2], qx[2], qy[2];
  sincos(p[3], &s, &c);
  circle_centre(p[0], p[1], c, s, off_front, px[0], py[0]);
  circle_centre(p[0], p[1], c, s, off_rear, px[1], py[1]);
  sincos(q[3], &s, &c);
  circle_centre(q[0], q[1], c, s, off_front, qx[0], qy[0]);
  circle_centre(q[0], q[1], c, s, off_rear, qx[1], qy[1]);
  double clear = INFINITY;
#pragma unroll
  for (int n = 0; n < 4; ++n) {
    const double dx = px[n >> 1] - qx[n & 1], dy = py[n >> 1] - qy[n & 1];
    clear = fmin(clear, sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))) - reach);
  }
  return clear >= gap;
}

// Writes trip t's row from slot b: exit, steps, done and the public outcome columns.
__device__ __forceinline__ void close_trip(const jmpc_trips& P, int t, int b, int exit, int done) {
  P.exit[t] = exit;
  P.steps[t] = P.ep_steps[b];
  P.done[t] = done;
  if (P.outcomes && P.ep_outcomes)
    for (int c = 0; c < JMPC_NOUTCOME; ++c)
      P.outcomes[(size_t)t * JMPC_NOUTCOME + c] = P.ep_outcomes[(size_t)b * JMPC_OUTCOME_LEN + c];
}

// Slot b becomes a fresh vehicle on trip t, entering at evaluation `entry`.
__device__ __forceinline__ void load_trip(const jmpc_trips& P, int t, int b, int entry) {
  for (int c = 0; c < 4; ++c) P.state[4 * (size_t)b + c] = P.start[4 * (size_t)t + c];
  for (int c = 0; c < JMPC_NPARAM; ++c)
    P.ep_params[(size_t)b * JMPC_NPARAM + c] = P.params[(size_t)t * JMPC_NPARAM + c];
  for (int c = 0; c < P.T; ++c) { P.oa[(size_t)b * P.T + c] = 0.0; P.od[(size_t)b * P.T + c] = 0.0; }
  P.ep_course_id[b] = P.course_id[t];
  P.ep_course_len[b] = P.course_len[t];
  P.target_ind[b] = 0; P.agent_idx[b] = 0; P.ep_steps[b] = 0; P.warm[b] = 0; P.flag[b] = 0;
  P.di[b] = 0.0;
  if (P.ep_zone) { P.ep_zone[2 * (size_t)b] = P.zone[2 * (size_t)t]; P.ep_zone[2 * (size_t)b + 1] = P.zone[2 * (size_t)t + 1]; }
  if (P.ep_priority) P.ep_priority[b] = P.priority[t];
  P.depart[b] = entry;
  P.ep_done[b] = JMPC_DONE_RUNNING;
  P.slot_trip[b] = t;
  P.phase[t] = kTripInSlot;
  P.slot[t] = b;
  P.entry[t] = entry;
}

// One thread per scene: close, admit, load (jmpc_scene_trips in include/jmpc.h).  A thread per scene suffices: at
// most 9 slots; the walk starts at the scene's first pending trip, stops at the first trip not yet due, and once no
// slot is empty jumps from one unusable trip to the next (the waits for a slot are not written: every due pass of a
// trip either admits it, counts a blocked wait or is a slot wait, so the slot waits follow from entry and arrival).
__global__ void scene_trips_kernel(const jmpc_trips P, const int* __restrict__ iter_dev, int initial, double off_front,
                                   double off_rear, double radius) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= P.n_scenes) return;
  const int k = P.k, b0 = s * k;
  const int i = initial ? -1 : *iter_dev;
  const int entry = i + 1;
  unsigned empty = 0;
  for (int j = 0; j < k; ++j) {
    const int b = b0 + j;
    if (P.ep_done[b] == JMPC_DONE_GOAL) {
      const int t = P.slot_trip[b];
      close_trip(P, t, b, i, JMPC_DONE_GOAL);
      P.phase[t] = kTripClosed;
      P.slot_trip[b] = -1;
      P.ep_done[b] = JMPC_WAITING;
    }
    if (P.ep_done[b] == JMPC_WAITING) empty |= 1u << j;
  }
  const int last = P.scene_start[s + 1];
  int first = P.cursor[s];
  while (first < last && P.phase[first] != kTripPending) ++first;
  P.cursor[s] = first;
  const double reach = 2.0 * radius;
  const double far = P.entry_gap + reach + 2.0 * (fabs(off_front) + fabs(off_rear)) + 1.0;
  const double far2 = far * far;
  int admitted = 0;
  for (int t = first; t < last && P.arrival[t] <= entry; ++t) {
    if (!empty) {                           // the rest wait for a slot (counted by the caller): close unusable ones
      t = P.next_unusable[t];
      if (t >= last || P.arrival[t] > entry) break;
    }
    if (P.phase[t] != kTripPending) continue;
    if (!P.usable[t]) {
      P.done[t] = JMPC_DONE_NO_COURSE;
      P.phase[t] = kTripClosed;
      ++admitted;
      continue;
    }
    const double* st = P.start + 4 * (size_t)t;
    bool clear = true;
    for (int j = 0; j < k && clear; ++j)
      if (!((empty >> j) & 1u))
        clear = start_clear(st, P.state + 4 * (size_t)(b0 + j), off_front, off_rear, reach, P.entry_gap, far2);
    for (int u = first; u < t && clear; ++u)
      if (P.phase[u] == kTripPending)
        clear = start_clear(st, P.start + 4 * (size_t)u, off_front, off_rear, reach, P.entry_gap, far2);
    if (!clear) { P.blocked_waits[t] += 1; continue; }
    const int j = __ffs(empty) - 1;
    empty &= empty - 1;
    load_trip(P, t, b0 + j, entry);
    ++admitted;
  }
  if (admitted) P.pending[s] -= admitted;
}

// One thread per slot: the rows of the trips still in a slot when the run ends.
__global__ void scene_trips_finish_kernel(const jmpc_trips P, int n_iterations) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.n_scenes * P.k) return;
  const int t = P.slot_trip[b];
  if (t >= 0) close_trip(P, t, b, n_iterations, P.ep_done[b]);
}

// ---- fixed-time traffic signals (jmpc_signals) ----------------------------------------------------------------------
struct SignalArgs {
  jmpc_signal_plan plan;
  int B, k, n_courses;
  const int* offset;        // [B / k] or nullptr
  const int* owner;         // [B] or nullptr: owner = b
  const int* group;         // [n_owner]
  const int* zone;          // [n_owner][2]
  const int* course_id;     // [B] or nullptr
  const int* course_n;      // the handle's course lengths
  const int* agent_idx; const double* state; const double* params; double default_dl;
  const int* done;
  int checked;
  int* course_len;          // [B] in-out
  int* latch;               // [B][2] (owner, 1 HOLD / 0 GO)
  int* hold_steps; int* go;                 // [n_owner]
  int* slot_hold_steps; int* slot_go;       // [B] or nullptr
  const int* iter_dev;
};

// One thread per episode: the red-light cut at L = e - margin, decided once per red phase and owner.
__global__ void signal_kernel(const SignalArgs A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B || A.done[b] != JMPC_DONE_RUNNING) return;
  int len;
  if (A.checked) {
    len = A.course_len[b];
  } else {                                  // what a flag-0 collision check writes
    len = A.course_n[A.course_id ? min(max(A.course_id[b], 0), A.n_courses - 1) : 0];
    A.course_len[b] = len;
  }
  const int o = A.owner ? A.owner[b] : b;
  const int g = A.group[o], e = A.zone[2 * (size_t)o];
  bool red = false;
  if (g >= 0 && g < A.plan.n_groups && e >= 0) {
    const long long d = (long long)*A.iter_dev + (A.offset ? A.offset[b / A.k] : 0) - A.plan.green_start[g];
    long long m = d % A.plan.cycle;
    if (m < 0) m += A.plan.cycle;
    red = m >= A.plan.green_len[g];
  }
  int* latch = A.latch + 2 * (size_t)b;
  if (!red) {
    if (latch[0] != -1) {                   // most latches are already empty: store only to clear one
      latch[0] = -1;
      latch[1] = 0;
    }
    return;
  }
  const int a = A.agent_idx[b], L = e - A.plan.margin;
  int hold;
  if (latch[0] == o) {
    hold = latch[1];
  } else {
    const double v = A.state[4 * (size_t)b + 2];
    const double dl = A.params ? A.params[(size_t)b * JMPC_NPARAM + JMPC_P_DL] : A.default_dl;
    const double reach = __dmul_rn(__dmul_rn(__dmul_rn(2.0, A.plan.stop_decel), (double)(L - 1 - a)), dl);
    hold = (a < L && __dmul_rn(v, v) <= reach) ? 1 : 0;
    latch[0] = o;
    latch[1] = hold;
    if (!hold && a < L) {                   // could not stop before the line: a dilemma-zone pass
      A.go[o] += 1;
      if (A.slot_go) A.slot_go[b] += 1;
    }
  }
  if (hold) {
    A.course_len[b] = min(len, max(a + 1, L));
    A.hold_steps[o] += 1;
    if (A.slot_hold_steps) A.slot_hold_steps[b] += 1;
  }
}

// The extras of a waiting vehicle keep to the loop's clock: they advance as those of a running one.
__device__ __forceinline__ bool extras_advance(int done) { return done == JMPC_DONE_RUNNING || done == JMPC_WAITING; }

// Constant-input obstacle motion, one thread per obstacle: obstacles [B][n_obs][6] = x, y, v, yaw, a, steer.
__global__ void obstacle_step_kernel(int count, double* __restrict__ obs, const int* __restrict__ done, int n_obs,
                                     double dt, double L) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  if (done && !extras_advance(done[k / n_obs])) return;
  double* o = obs + (size_t)k * 6;
  double x = o[0], y = o[1], v = o[2], yaw = o[3];
  double s, c;
  sincos(yaw, &s, &c);
  x = __dadd_rn(x, __dmul_rn(__dmul_rn(v, c), dt));
  y = __dadd_rn(y, __dmul_rn(__dmul_rn(v, s), dt));
  v = __dadd_rn(v, __dmul_rn(o[4], dt));
  yaw = __dadd_rn(yaw, __dmul_rn(__dmul_rn(v / L, tan(o[5])), dt));
  o[0] = x; o[1] = y; o[2] = v; o[3] = yaw;
}

// ---- the reference's scripted obstacles (main/lib/moving_obstacles.py) -------------------------------------------
// One thread per obstacle.  `script` [count][JMPC_OBS_SCRIPT_LEN] is constant: kind, direction (+1 / -1), turning,
// speed, offset (<= 0: none), the Bicycle's sample time, the dt of the offset test (the roundabout class overwrites
// its own with 0.2, moving_obstacles.py:45, while its Bicycle keeps the constructor's), and one auxiliary value (the
// turning steer angle arctan(L / 5) of the roundabout rules, computed on the host; the arterial's initial speed).
// `model` [count][4] = Bicycle xc, yc, theta and the step counter.  `obs` [count][6] receives what `get()` returns:
// x, y, forward_velocity, theta, 0, steering_angle -- the tuple the flag kernel consumes.
//
// The scenario loop calls get() (prediction), then step() (mpc_intersection.py:123-125, 157-160).  get() evaluates
// its tuple left to right, so theta is read BEFORE the steering property runs, and the roundabout's steering property
// overwrites model.theta as a side effect (moving_obstacles.py:82-84, 98-100) -- both reproduced.
__device__ __forceinline__ double scripted_speed(const double* sc, double counter) {
  const int kind = (int)sc[JMPC_OBS_KIND];
  const double offset = sc[JMPC_OBS_OFFSET];
  const bool moving = !(offset > 0.0) || counter > __ddiv_rn(offset, sc[JMPC_OBS_DT_OFFSET]);
  if (moving) return sc[JMPC_OBS_SPEED];
  return kind == JMPC_OBS_ARTERIAL ? sc[JMPC_OBS_AUX] : 0.0;
}
__device__ __forceinline__ double scripted_steer(const double* sc, double xc, double yc, double& theta) {
  const int kind = (int)sc[JMPC_OBS_KIND];
  const bool right = sc[JMPC_OBS_DIRECTION] >= 0.0, turning = sc[JMPC_OBS_TURNING] != 0.0;
  double steer = 0.0;
  if (!turning) return steer;
  if (kind == JMPC_OBS_TINTERSECTION) {                 // moving_obstacles.py:197-213
    if (right) { if (xc >= -10.0 && theta > -M_PI / 2) steer = -0.38; }
    else if (xc <= 12.0 && theta < 3 * M_PI / 2) steer = 0.19;
  } else if (kind == JMPC_OBS_ROUNDABOUT) {             // moving_obstacles.py:66-103, the ifs in sequence
    const double ang = sc[JMPC_OBS_AUX];
    if (right) {
      if (-7.0 <= xc && xc <= -4.0 && yc < 0.0) steer = -ang;
      if (-3.0 < xc) steer = ang;
      if (yc > 0.0 && -5.0 <= xc && xc <= -3.0) steer = -ang;
      if (xc <= -3.0 && yc > 0.0) { theta = -M_PI; steer = 0.0; }
    } else {
      if (4.0 <= xc && xc <= 7.0 && yc > 0.0) steer = -ang;
      if (xc < 3.0) steer = ang;
      if (yc < 0.0 && 3.0 <= xc && xc <= 5.0) steer = -ang;
      if (3.0 <= xc && yc < 0.0) { theta = 0.0; steer = 0.0; }
    }
  }
  return steer;
}
__global__ void scripted_obstacle_kernel(int count, const double* __restrict__ script, double* __restrict__ model,
                                         double* __restrict__ obs, const int* __restrict__ done, int n_obs, int advance,
                                         double L) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  if (done && !extras_advance(done[k / n_obs])) return;
  const double* sc = script + (size_t)k * JMPC_OBS_SCRIPT_LEN;
  double* m = model + (size_t)k * 4;
  double xc = m[0], yc = m[1], theta = m[2], counter = m[3];
  if (advance) {                                        // step(): moving_obstacles.py:113-116, bicycle/main.py:28-41
    const double steer = scripted_steer(sc, xc, yc, theta);
    const double v = scripted_speed(sc, counter), dt = sc[JMPC_OBS_DT_MODEL];
    const double xd = __dmul_rn(v, cos(theta)), yd = __dmul_rn(v, sin(theta)), td = __dmul_rn(v / L, tan(steer));
    xc = __dadd_rn(xc, __dmul_rn(xd, dt));
    yc = __dadd_rn(yc, __dmul_rn(yd, dt));
    theta = __dadd_rn(theta, __dmul_rn(td, dt));
    counter += 1.0;
  }
  double* o = obs + (size_t)k * 6;                      // get(): moving_obstacles.py:118-120
  o[0] = xc; o[1] = yc; o[2] = scripted_speed(sc, counter); o[3] = theta; o[4] = 0.0;
  o[5] = scripted_steer(sc, xc, yc, theta);             // may overwrite theta (after it has been reported)
  m[0] = xc; m[1] = yc; m[2] = theta; m[3] = counter;
}

}  // namespace jmpc
