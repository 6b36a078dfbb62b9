// jmpc_collision.cuh -- collision flag + cut index, one warp per instance.
//
// Reference (relative to SaeedRahmani/AV-Simulation-at-Intersections):
//   main/scenarios/mpc_intersection.py:111-140   ego max-acceleration prediction, cut index
//   main/lib/trajectories.py:58-86               resample_curve
//   main/lib/moving_obstacles_prediction.py:21-47  constant-input obstacle prediction
//   main/lib/collision_avoidance.py:68-124,168-180 frame-shifted circle test, first-hit lookup
//
// The reference materialises a (frames * 4 * copies) x 2 table and takes the first row within 2 * radius.
// The row order -- frame, ego circle, obstacle copy (obstacle major, frame offset -fw..+fw minor), obstacle
// circle -- decides WHICH obstacle circle is reported, hence the cut index; the kernel walks the same order
// (frames in sequence, the 4 * copies pairs of one frame across the lanes, lowest pair index wins).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/jmpc.h"

namespace jmpc {

constexpr int kMaxObstacles = 8;
constexpr int kMaxFrameWindow = 32;
constexpr int kMaxObsFrames = 72;      // len(arange(0, horizon, dt)); 35 in the reference
constexpr int kMaxEgoFrames = 160;     // points kept by resample_curve (<= 49 in the reference's scenes)

struct ParamBlock { double v[JMPC_NPARAM]; };

struct CollisionArgs {
  int B, n_courses;
  const double* cx; const double* cy; const double* cyaw;
  const double* ccfx; const double* ccfy; const double* ccrx; const double* ccry;   // circle-centre tables
  const int* course_n; int course_stride;
  const int* course_id; const int* agent_idx; const double* v; const double* obstacles;
  int n_obs, frame_window, margin;
  double horizon_s;
  double off_front, off_rear, radius;
  const double* params; ParamBlock defaults;
  int* flag; int* course_len_out;
  int arc_cap;                                       // longest course (handle max_N)
  int arc_smem;                                      // doubles of shared memory per warp for the on-the-fly arc scan: arc_cap,
                                                     // or 0 when every course has a table (twice the resident warps then)
  // Optional per-course table of the running arc lengths from every start index (arc_tables_kernel): row a0 of course c
  // starts at arc_tab + arc_off[c] + a0 * N - a0 (a0 - 1) / 2 and has N - a0 entries; arc_off[c] < 0 = no table
  const double* arc_tab; const long long* arc_off;
  const int* skip;                                   // [B] or nullptr: skip[b] != 0 -> instance left untouched
  // collision_kernel<true> only: per-step inputs [B][n_planned][plan_len][2] (a, steer) of obstacle slots 0 ..
  // n_planned - 1; predictor step t uses input min(t, plan_len - 1)
  const double* plans; int n_planned, plan_len;
};

// dynamic shared memory of one warp: arc[arc_cap] | ocx[n_obs][kMaxObsFrames][2] | ocy[...] | bbox[kMaxObstacles][4] |
// ego_idx[kMaxEgoFrames]
__host__ __device__ inline size_t collision_warp_smem_bytes(int arc_cap, int n_obs) {
  return ((size_t)arc_cap + (size_t)4 * n_obs * kMaxObsFrames + 4 * kMaxObstacles) * sizeof(double) +
         (size_t)kMaxEgoFrames * sizeof(short);
}

// circle centres of a pose: same operation order as trajectories.py:27-34 with a zero lateral offset
// ((cos * off - sin * 0) + x): no fused multiply-add.
__device__ __forceinline__ void circle_centre(double x, double y, double c, double s, double off, double& ox, double& oy) {
  ox = __dadd_rn(__dmul_rn(c, off), x);
  oy = __dadd_rn(__dmul_rn(s, off), y);
}

// Start of row a0 in the arc-length table of a course of N points (rows of N, N - 1, ..., 1 entries).
__host__ __device__ inline long long arc_row_offset(int a0, int N) { return (long long)a0 * N - ((long long)a0 * (a0 - 1)) / 2; }

// dist(a, b) <= reach with numpy's sqrt(dx*dx + dy*dy); the square root is only evaluated when the squared
// comparison is within rounding distance of the threshold.
__device__ __forceinline__ bool within(double ax, double ay, double bx, double by, double reach, double reach2_lo,
                                       double reach2_hi) {
  const double dx = ax - bx, dy = ay - by;
  const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  if (d2 < reach2_lo) return true;
  if (d2 > reach2_hi) return false;
  return sqrt(d2) <= reach;
}

// consider[b] of the masked kernel, loaded where it is used (volatile: not merged with an earlier load of the same word
// and kept in a register across sections A and B).  The generic pointer is converted to the global window explicitly.
__device__ __forceinline__ unsigned ld_mask(const int* p) {
  unsigned m;
  asm volatile("{\n\t.reg .u64 g;\n\tcvta.to.global.u64 g, %1;\n\tld.global.nc.u32 %0, [g];\n\t}" : "=r"(m) : "l"(p));
  return m;
}

struct CollisionSmem {
  double* arc;          // segment lengths, then running arc length
  double* ocx;          // obstacle circle centres [obstacle][frame][circle]
  double* ocy;
  double* bbox;         // per obstacle: min x, max x, min y, max y of its predicted circle centres
  short* ego_idx;       // kept path points (relative to agent_idx)
  __device__ CollisionSmem(unsigned char* base, int arc_cap, int n_obs) {
    arc = reinterpret_cast<double*>(base);
    ocx = arc + arc_cap;
    ocy = ocx + (size_t)2 * n_obs * kMaxObsFrames;
    bbox = ocy + (size_t)2 * n_obs * kMaxObsFrames;
    ego_idx = reinterpret_cast<short*>(bbox + 4 * kMaxObstacles);
  }
  __device__ __forceinline__ int oi(int ob, int frame, int circle) const { return (ob * kMaxObsFrames + frame) * 2 + circle; }
};

// The body of collision_kernel and masked_collision_kernel, one warp per instance.
// Planned = false: every obstacle is predicted with the constant input (a, steer) of its row (columns 4, 5).
// Planned = true: slots < A.n_planned are predicted with their per-step inputs from A.plans instead; only section B
// differs, and a plan whose entries all equal the row's (a, steer) gives the constant-input prediction bit for bit.
// Masked = true: only the slots whose bit is set in consider[b] take part in section C.  Dropping slots keeps the
// reference's row order of the others (obstacle major within an ego circle), so the result is that of the same call on
// the considered rows alone; a mask without a bit among the n_obs slots is the n_obs = 0 case (flag 0, the full length:
// section C finds no pair, and the table-limit exit reports 0 instead of -1).  An ignored slot gets an empty bounding
// box (+inf .. -inf), which section C's box test skips like any box out of reach; the mask is read where it is used,
// so that no register holds it across sections A and B.
template <bool Planned, bool Masked>
__device__ __forceinline__ void collision_body(const CollisionArgs& A, const int* __restrict__ consider) {
  extern __shared__ unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int b = blockIdx.x * (blockDim.x >> 5) + wib;
  if (b >= A.B) return;
  if (A.skip && A.skip[b] != 0) return;
  CollisionSmem S(smem_raw + (size_t)wib * collision_warp_smem_bytes(A.arc_smem, A.n_obs), A.arc_smem, A.n_obs);
  const unsigned full = 0xffffffffu;

  const double* prm = A.params ? A.params + (size_t)b * JMPC_NPARAM : A.defaults.v;
  const double dt = prm[JMPC_P_DT], L = prm[JMPC_P_L];
  const double max_accel = prm[JMPC_P_MAX_ACCEL], max_speed = prm[JMPC_P_SIM_MAX_SPEED];
  const int cid = A.course_id ? min(max(A.course_id[b], 0), A.n_courses - 1) : 0;
  const size_t coff = (size_t)cid * A.course_stride;
  const double* cx = A.cx + coff; const double* cy = A.cy + coff;
  const double* fx = A.ccfx + coff; const double* fy = A.ccfy + coff;
  const double* rx = A.ccrx + coff; const double* ry = A.ccry + coff;
  const int N = A.course_n[cid];
  const int a0 = min(max(A.agent_idx[b], 0), N - 1);
  const int M = min(N - a0, A.arc_cap);               // points of trajectory_full[agent_idx:]
  const double v = A.v[b];

  if (A.n_obs == 0) {                                // check_collision_moving_cars returns None
    if (lane == 0) { A.flag[b] = 0; A.course_len_out[b] = N; }
    return;
  }

  // ---- A. ego prediction: resample_curve(path, dl_i) ------------------------------------------------
  const bool have_tab = A.arc_tab && A.arc_off[cid] >= 0 && M == N - a0;
  const double* arc = have_tab ? A.arc_tab + A.arc_off[cid] + arc_row_offset(a0, N) : S.arc;
  if (!have_tab) {
  for (int i = lane; i < M; i += 32) {
    double seg = 0.0;
    if (i > 0) {
      const double dx = cx[a0 + i] - cx[a0 + i - 1], dy = cy[a0 + i] - cy[a0 + i - 1];
      seg = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    }
    S.arc[i] = seg;
  }
  __syncwarp();
  if (lane == 0) {                                   // np.cumsum: strictly sequential float64 adds
    double acc = 0.0;
    for (int i = 0; i < M; ++i) { acc = __dadd_rn(acc, S.arc[i]); S.arc[i] = acc; }
  }
  __syncwarp();
  }
  int n_ego = 0;
  {
    const bool ramp = v < max_speed;                 // mpc_intersection.py:114
    const double dl_flat = __dmul_rn(dt, max_speed);
    for (int base = 0; base < M; base += 32) {
      const int i = base + lane;
      bool keep = false;
      if (i < M) {
        // bucket_i = floor(arc_i / dl_i), dl_i = dt * min(cumsum(max_accel)_i + v, max_speed)
        auto bucket = [&](int k) -> double {
          double dl = dl_flat;
          if (ramp) {
            // cumsum of a constant: k+1 sequential adds; every partial sum is exact for a small integer
            // constant (2.0 in every reference config), otherwise the additions are repeated literally
            double cs = 0.0;
            if (max_accel == rint(max_accel) && fabs(max_accel) < 1048576.0) cs = (double)(k + 1) * max_accel;
            else for (int q = 0; q <= k; ++q) cs = __dadd_rn(cs, max_accel);
            dl = __dmul_rn(dt, fmin(__dadd_rn(cs, v), max_speed));
          }
          return floor(arc[k] / dl);
        };
        keep = (i == 0) || (i == M - 1) || (bucket(i) - bucket(i - 1) >= 1.0);
      }
      const unsigned m = __ballot_sync(full, keep);
      if (keep) {
        const int pos = n_ego + __popc(m & ((1u << lane) - 1u));
        if (pos < kMaxEgoFrames) S.ego_idx[pos] = (short)i;
      }
      n_ego += __popc(m);
    }
  }
  // Limits of the per-warp shared-memory tables: an instance whose ego prediction keeps more than kMaxEgoFrames points
  // or whose obstacle prediction needs more than kMaxObsFrames - 1 steps cannot be decided here; it is reported
  // (flag = -1, full course length) instead of being silently truncated.  The reference's scenes need 49 / 35.
  if (n_ego > kMaxEgoFrames || (int)ceil(A.horizon_s / dt) > kMaxObsFrames - 1) {
    // a mask without a considered slot is the n_obs = 0 case: flag 0 (tested here, on this rare path, and not before
    // section A: a test up there costs the masked kernels spills of the loop state)
    if (lane == 0) {
      A.flag[b] = (Masked && (ld_mask(consider + b) & ((1u << A.n_obs) - 1u)) == 0u) ? 0 : -1;
      A.course_len_out[b] = N;
    }
    return;
  }

  // ---- B. obstacle predictions (moving_obstacles_prediction.py:21-47) ------------------------------
  // The yaw / speed recurrences need no trigonometry, so they are walked first (one lane per obstacle); then all lanes
  // evaluate sin / cos of the n_of + 1 distinct headings in parallel; then the positions are accumulated in sequence.
  // Each value is produced by the same operations in the same order as in the reference's loop, which evaluates
  // sin / cos of every heading twice (2 x 35 sequential sincos per obstacle on 2-4 active lanes before).
  const int n_of = min((int)ceil(A.horizon_s / dt), kMaxObsFrames - 1);
  // Planned slots: the recurrence is the same, with input min(k, plan_len - 1) at step k.  tan(steer_k) of every
  // (slot, step) is evaluated across the lanes first, into ocy[ob][k][1] (free until the centres are written); the
  // yaw / speed walk then replaces it with the speed before step k, which the position pass reads back.
  const double* plan = nullptr;
  if constexpr (Planned) {
    const double* pb = A.plans + (size_t)b * A.n_planned * A.plan_len * 2;
    for (int j = lane; j < A.n_planned * n_of; j += 32) {
      const int ob = j / n_of, k = j - ob * n_of;
      S.ocy[S.oi(ob, k, 1)] = tan(pb[((size_t)ob * A.plan_len + min(k, A.plan_len - 1)) * 2 + 1]);
    }
    if (lane < A.n_planned) plan = pb + (size_t)lane * A.plan_len * 2;
    __syncwarp();
  }
  if (lane < A.n_obs) {
    const double* o = A.obstacles + ((size_t)b * A.n_obs + lane) * 6;
    double vo = o[2], yaw = o[3];
    if (Planned && plan) {
      S.ocy[S.oi(lane, 0, 0)] = yaw;                 // scratch: heading k in ocy[ob][k][0]
      for (int k = 0; k < n_of; ++k) {
        const double tn = S.ocy[S.oi(lane, k, 1)];
        S.ocy[S.oi(lane, k, 1)] = vo;
        vo = __dadd_rn(vo, __dmul_rn(plan[2 * min(k, A.plan_len - 1)], dt));
        yaw = __dadd_rn(yaw, __dmul_rn(__dmul_rn(vo / L, tn), dt));
        S.ocy[S.oi(lane, k + 1, 0)] = yaw;
      }
    } else {
      const double acc = o[4], tn = tan(o[5]);
      S.ocy[S.oi(lane, 0, 0)] = yaw;
      for (int k = 0; k < n_of; ++k) {
        vo = __dadd_rn(vo, __dmul_rn(acc, dt));
        yaw = __dadd_rn(yaw, __dmul_rn(__dmul_rn(vo / L, tn), dt));
        S.ocy[S.oi(lane, k + 1, 0)] = yaw;
      }
    }
  }
  __syncwarp();
  for (int j = lane; j < A.n_obs * (n_of + 1); j += 32) {
    const int ob = j / (n_of + 1), k = j - ob * (n_of + 1);
    double s, c;
    sincos(S.ocy[S.oi(ob, k, 0)], &s, &c);
    S.ocx[S.oi(ob, k, 0)] = c; S.ocx[S.oi(ob, k, 1)] = s;      // scratch: cos / sin of heading k in ocx[ob][k][0 / 1]
  }
  __syncwarp();
  if (lane < A.n_obs) {
    const double* o = A.obstacles + ((size_t)b * A.n_obs + lane) * 6;
    double x = o[0], y = o[1], vo = o[2];
    const double acc = o[4];
    double c = S.ocx[S.oi(lane, 0, 0)], s = S.ocx[S.oi(lane, 0, 1)];
    for (int k = 0; k < n_of; ++k) {
      if (Planned && plan) vo = S.ocy[S.oi(lane, k, 1)];
      x = __dadd_rn(x, __dmul_rn(__dmul_rn(vo, c), dt));
      y = __dadd_rn(y, __dmul_rn(__dmul_rn(vo, s), dt));
      if (!(Planned && plan)) vo = __dadd_rn(vo, __dmul_rn(acc, dt));
      c = S.ocx[S.oi(lane, k + 1, 0)]; s = S.ocx[S.oi(lane, k + 1, 1)];       // heading after the step
      // slot k is overwritten with the circle centres only now that its cos / sin have been consumed
      circle_centre(x, y, c, s, A.off_front, S.ocx[S.oi(lane, k, 0)], S.ocy[S.oi(lane, k, 0)]);
      circle_centre(x, y, c, s, A.off_rear, S.ocx[S.oi(lane, k, 1)], S.ocy[S.oi(lane, k, 1)]);
    }
  }
  __syncwarp();

  // Bounding box of every obstacle's predicted circle centres.  An ego circle further than the reach outside the box
  // cannot touch any frame-shifted copy of that obstacle (the copies are clamped to the predicted frames), so the
  // whole group of 2 * span pair tests is skipped -- a conservative test, the decisions stay bit-exact.
  for (int ob = 0; ob < A.n_obs; ++ob) {
    double x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
    for (int j = lane; j < 2 * n_of; j += 32) {
      const double ox = S.ocx[S.oi(ob, j >> 1, j & 1)], oy = S.ocy[S.oi(ob, j >> 1, j & 1)];
      x0 = fmin(x0, ox); x1 = fmax(x1, ox); y0 = fmin(y0, oy); y1 = fmax(y1, oy);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      x0 = fmin(x0, __shfl_xor_sync(full, x0, o)); x1 = fmax(x1, __shfl_xor_sync(full, x1, o));
      y0 = fmin(y0, __shfl_xor_sync(full, y0, o)); y1 = fmax(y1, __shfl_xor_sync(full, y1, o));
    }
    if (Masked && !((ld_mask(consider + b) >> ob) & 1u)) { x0 = y0 = INFINITY; x1 = y1 = -INFINITY; }
    if (lane == 0) { S.bbox[4 * ob] = x0; S.bbox[4 * ob + 1] = x1; S.bbox[4 * ob + 2] = y0; S.bbox[4 * ob + 3] = y1; }
  }
  __syncwarp();

  // ---- C. first touching pair in the reference's row order ------------------------------------------
  const double reach = 2.0 * A.radius;
  const double pad = reach * (1.0 + 1e-9);
  const double reach2 = reach * reach, reach2_lo = reach2 * (1.0 - 1e-12), reach2_hi = reach2 * (1.0 + 1e-12);
  const int span = 2 * A.frame_window + 1;
  const int copies = A.n_obs * span;
  // per frame: 4 * copies pairs, ordered [ego circle][copy][obstacle circle]
  const int frames = max(n_ego, n_of);
  int hit_f = -1, hit_pair = 0;
  for (int f = 0; f < frames && hit_f < 0; ++f) {
    const int ei = a0 + S.ego_idx[min(f, n_ego - 1)];
    const int fc = min(f, n_of - 1);
    int best = 0x7fffffff;
    // pair index p = ac * 2 * copies + (ob * span + k) * 2 + oc, walked in increasing order by every lane without
    // integer divisions (the first version decoded p with / and %: a third of the kernel's instructions)
    for (int ac = 0; ac < 2 && best == 0x7fffffff; ++ac) {
      const double ax = ac ? rx[ei] : fx[ei], ay = ac ? ry[ei] : fy[ei];
      for (int ob = 0; ob < A.n_obs && best == 0x7fffffff; ++ob) {
        if (ax < S.bbox[4 * ob] - pad || ax > S.bbox[4 * ob + 1] + pad || ay < S.bbox[4 * ob + 2] - pad ||
            ay > S.bbox[4 * ob + 3] + pad)
          continue;
        const int pbase = ac * 2 * copies + ob * span * 2;
        for (int q = lane; q < 2 * span; q += 32) {
          const int oc = q & 1, off = (q >> 1) - A.frame_window;
          const int fi = min(max(fc - off, 0), n_of - 1);
          if (within(ax, ay, S.ocx[S.oi(ob, fi, oc)], S.ocy[S.oi(ob, fi, oc)], reach, reach2_lo, reach2_hi)) {
            best = pbase + q;
            break;
          }
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(full, best, o));
    if (best != 0x7fffffff) { hit_f = f; hit_pair = best; }
  }
  if (hit_f < 0) {
    if (lane == 0) { A.flag[b] = 0; A.course_len_out[b] = N; }
    return;
  }
  double wx, wy;
  {
    const int ac = hit_pair / (2 * copies), rem = hit_pair - ac * 2 * copies;
    const int j = rem >> 1, oc = rem & 1;
    const int ob = j / span, off = (j - ob * span) - A.frame_window;
    const int fi = min(max(min(hit_f, n_of - 1) - off, 0), n_of - 1);
    wx = S.ocx[S.oi(ob, fi, oc)]; wy = S.ocy[S.oi(ob, fi, oc)];
  }

  // ---- D. first point of the detailed path whose circle touches that obstacle circle -----------------
  // (front-circle rows come first in the reference's concatenation, then the rear-circle rows)
  int k_first = 0x7fffffff;
  for (int base = 0; base < M && k_first == 0x7fffffff; base += 32) {
    const int i = base + lane;
    const bool t = (i < M) && within(fx[a0 + i], fy[a0 + i], wx, wy, reach, reach2_lo, reach2_hi);
    const unsigned m = __ballot_sync(full, t);
    if (m) k_first = base + __ffs(m) - 1;
  }
  if (k_first == 0x7fffffff) {
    for (int base = 0; base < M && k_first == 0x7fffffff; base += 32) {
      const int i = base + lane;
      const bool t = (i < M) && within(rx[a0 + i], ry[a0 + i], wx, wy, reach, reach2_lo, reach2_hi);
      const unsigned m = __ballot_sync(full, t);
      if (m) k_first = base + __ffs(m) - 1;
    }
  }
  if (k_first == 0x7fffffff) k_first = 0;             // np.argmax of an all-False mask

  // ---- E. cut index: first course point within 1 mm of that path point, minus the margin ------------
  const double px = cx[a0 + k_first], py = cy[a0 + k_first];
  const double r1 = 0.001, r1_2 = r1 * r1;
  int first = 0x7fffffff;
  for (int base = 0; base < N && first == 0x7fffffff; base += 32) {
    const int i = base + lane;
    const bool t = (i < N) && within(cx[i], cy[i], px, py, r1, r1_2 * (1.0 - 1e-12), r1_2 * (1.0 + 1e-12));
    const unsigned m = __ballot_sync(full, t);
    if (m) first = base + __ffs(m) - 1;
  }
  if (lane == 0) {
    A.flag[b] = 1;
    A.course_len_out[b] = max(a0 + 1, first - A.margin);
  }
}

// jmpc_collision / jmpc_collision_planned
template <bool Planned>
__global__ void __launch_bounds__(128) collision_kernel(const CollisionArgs A) {
  collision_body<Planned, false>(A, nullptr);
}

// jmpc_collision_masked: consider [B] int32, bit s set = obstacle slot s takes part in the cut
template <bool Planned>
__global__ void __launch_bounds__(128) masked_collision_kernel(const CollisionArgs A, const int32_t* consider) {
  collision_body<Planned, true>(A, consider);
}

}  // namespace jmpc
