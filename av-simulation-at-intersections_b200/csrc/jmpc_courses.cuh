// jmpc_courses.cuh -- planned courses into the controller's course tables on the device (jmpc_set_courses_device), and
// the episode start on them (jmpc_episode_init_from_courses).
//
// Reference (relative to SaeedRahmani/AV-Simulation-at-Intersections):
//   main/scenarios/mpc_intersection.py:63-79   plan, dl of the first segment, MPC(trajectory_full), State at its start
//   main/lib/mpc.py:46-58, :260                the yaw unwrap MPC.__init__ applies to the course in place
//
// What the host pipeline did per course (slice the planner's output, unwrap the yaw in a Python loop, upload through a
// pinned row, one table kernel per course) is three launches for all courses here: course_ingest_kernel (one warp per
// course: AoS -> SoA copy by the lanes, the sequential unwrap by lane 0), then circle_tables_kernel and
// arc_tables_kernel with the course index in the grid's y dimension.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/jmpc.h"
#include "jmpc_collision.cuh"

namespace jmpc {

struct IngestArgs {
  int n_courses, traj_stride, max_N, course_stride;
  const int* n_traj; const double* traj; const int* plan_status;
  double* cx; double* cy; double* cyaw; int* course_n;
  double* dl; int* ok;
};

// One warp per course.
__global__ void __launch_bounds__(128) course_ingest_kernel(const IngestArgs A) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= A.n_courses) return;
  const unsigned full = 0xffffffffu;
  const double* src = A.traj + (size_t)c * A.traj_stride * 3;
  double* cx = A.cx + (size_t)c * A.course_stride;
  double* cy = A.cy + (size_t)c * A.course_stride;
  double* cyaw = A.cyaw + (size_t)c * A.course_stride;
  const int n = A.n_traj[c];
  const bool found = !A.plan_status || A.plan_status[c] == JMPC_PLAN_FOUND;
  bool ok = found && n >= 2 && n <= A.max_N && n <= A.traj_stride;
  if (ok) {                                   // a non-finite value would also make the unwrap below loop forever
    bool bad = false;
    for (int i = lane; i < n; i += 32)
      bad = bad || !isfinite(src[3 * i]) || !isfinite(src[3 * i + 1]) || !isfinite(src[3 * i + 2]);
    ok = !__any_sync(full, bad);
  }
  if (!ok) {                                  // one-point placeholder: the start pose when there is one
    if (lane == 0) {
      const bool have = n >= 1 && n <= A.traj_stride && isfinite(src[0]) && isfinite(src[1]) && isfinite(src[2]);
      cx[0] = have ? src[0] : 0.0; cy[0] = have ? src[1] : 0.0; cyaw[0] = have ? src[2] : 0.0;
      A.course_n[c] = 1; A.dl[c] = nan(""); A.ok[c] = 0;
    }
    return;
  }
  for (int i = lane; i < n; i += 32) { cx[i] = src[3 * i]; cy[i] = src[3 * i + 1]; }
  if (lane == 0) {
    // mpc.py:46-58 (synth.smooth_yaw_inplace): compares against the already-unwrapped predecessor
    const double half_pi = M_PI / 2.0, two_pi = 2.0 * M_PI;
    double prev = src[2];
    cyaw[0] = prev;
    for (int k = 1; k < n; ++k) {
      double y = src[3 * k + 2];
      while (y - prev >= half_pi) y -= two_pi;
      while (y - prev <= -half_pi) y += two_pi;
      cyaw[k] = y;
      prev = y;
    }
    const double dx = src[0] - src[3], dy = src[1] - src[4];
    A.dl[c] = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    A.course_n[c] = n; A.ok[c] = 1;
  }
}

// Circle-centre tables of every course: x = point, y = course.
__global__ void circle_tables_kernel(int n_courses, int stride, const int* __restrict__ course_n,
                                     const double* __restrict__ cx, const double* __restrict__ cy,
                                     const double* __restrict__ cyaw, double off_front, double off_rear,
                                     double* __restrict__ fx, double* __restrict__ fy, double* __restrict__ rx,
                                     double* __restrict__ ry) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (int c = blockIdx.y; c < n_courses; c += gridDim.y) {
    if (i >= course_n[c]) continue;
    const size_t o = (size_t)c * stride;
    circle_table_point(i, cx + o, cy + o, cyaw + o, off_front, off_rear, fx + o, fy + o, rx + o, ry + o);
  }
}

// Arc-length tables of every course that has a slot (arc_off[c] >= 0): x = start index, y = course.
__global__ void arc_tables_kernel(int n_courses, int stride, const int* __restrict__ course_n,
                                  const long long* __restrict__ arc_off, const double* __restrict__ cx,
                                  const double* __restrict__ cy, double* __restrict__ tab) {
  const int a0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int c = blockIdx.y; c < n_courses; c += gridDim.y) {
    const int N = course_n[c];
    if (a0 >= N || arc_off[c] < 0) continue;
    const size_t o = (size_t)c * stride;
    arc_table_row(a0, N, cx + o, cy + o, tab + arc_off[c]);
  }
}

// One thread per episode: start state on its course, its dl, done = 3 when the course is unusable.
__global__ void episode_init_kernel(int B, int n_courses, int stride, const int* __restrict__ course_id,
                                    const int* __restrict__ course_ok, const double* __restrict__ dl,
                                    const double* __restrict__ cx, const double* __restrict__ cy,
                                    const double* __restrict__ cyaw, double* __restrict__ state,
                                    double* __restrict__ params, int* __restrict__ done) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int c = course_id ? min(max(course_id[b], 0), n_courses - 1) : 0;
  const size_t o = (size_t)c * stride;
  state[4 * b] = cx[o]; state[4 * b + 1] = cy[o]; state[4 * b + 2] = 0.0; state[4 * b + 3] = cyaw[o];
  if (params && dl) params[(size_t)b * JMPC_NPARAM + JMPC_P_DL] = dl[c];
  if (course_ok && !course_ok[c]) done[b] = 3;
}

}  // namespace jmpc
