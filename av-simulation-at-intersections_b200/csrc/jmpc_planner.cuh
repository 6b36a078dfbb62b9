// jmpc_planner.cuh -- batched motion-primitive A* (SURVEY.md section 8f row f4): one warp runs one search.
//
// Reference (paths relative to SaeedRahmani/AV-Simulation-at-Intersections):
//   main/lib/a_star.py:31-78                   the search: heap of (g + h, g, node, predecessor) tuples, dict of expanded
//                                              nodes keyed by the exact (x, y, theta) floats
//   main/lib/mp_search_ww_generic.py:136-256   neighbours (one per collision-free primitive), edge cost, heuristic,
//                                              goal test, path -> full trajectory
//   main/lib/obstacles.py:157-176              collision: some check point inside ALL half-planes of some obstacle
//   main/lib/linalg.py, main/lib/maths.py      2-D transform of a primitive by a node, angle normalisation
//
// Many (start, goal, weights, scene) searches run at once, one per warp.  Inside a warp the lanes split the
// collision test of the popped node (primitive x check point pairs against every half-plane set) and the evaluation
// of its neighbours (lane m = primitive m: end pose, edge cost, heuristic, closed-set lookup); lane 0 owns the open
// list (binary heap in global memory, keys compared exactly as Python compares the reference's tuples: g + h, then g,
// then the node's floats, then the predecessor's) and the closed set (open-addressing hash on the node's floats, the
// reference's dict).  Everything is float64 and every decision (collision, closed-set membership, heap order, goal
// test) is taken on the same quantities as in the reference; sin / cos come from CUDA's libm, so node coordinates can
// differ from numpy's in the last bits (never observed to change a decision on the recorded searches).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/jmpc.h"

namespace jmpc {

struct PlanNode {           // one pushed tuple of the reference's heap
  double x, y, th, g, gh;
  int parent;               // pool index of the entry that was being expanded when this one was generated
  int mp;                   // primitive that leads from the parent's node to this node
};

struct PlanArgs {
  int B, n_mp, n_pts, n_cc, max_obs, n_scenes;
  // primitives (shared by all searches)
  const double* mp_pts;     // [n_mp][n_pts][3] points of each primitive, relative to its start pose
  const double* mp_len;     // [n_mp] total_length
  const double* mp_cc;      // [n_mp][n_cc][2] collision-check points (mp_search_ww_generic.py:121-138)
  // scenes: half-plane sets of the obstacles
  const double* hp;         // [n_scenes][max_obs][JMPC_PLAN_MAX_HP][3]
  const int* hp_n;          // [n_scenes][max_obs]
  const int* n_obs;         // [n_scenes]
  // searches
  const int* scene_id;      // [B]
  const double* start;      // [B][3]
  const double* goal_point; // [B][3]
  const double* goal_area;  // [B][4] x1, y1, x2, y2 of the goal box
  const double* allowed;    // [B] allowed_goal_theta_difference
  const double* weights;    // [B][9] wh_dist, wh_theta, wh_steering, wh_obstacle, wh_center, wc_dist, wc_steering, wc_obstacle, wc_center
  int max_expansions, max_path, max_traj, max_log;
  // workspace, per search
  PlanNode* pool; int pool_cap;
  int* heap;
  int* table; int table_size;     // power of two
  // results
  double* cost; int* status; int* n_path; double* path; int* path_mp; int* n_traj; double* traj; int* expansions;
  double* log;                     // [B][max_log][5] g, h, x, y, theta in expansion order, or nullptr
};

// Python's float %: the result takes the sign of the divisor
__device__ __forceinline__ double py_mod(double a, double b) {
  double r = fmod(a, b);
  if (r != 0.0) { if ((b < 0.0) != (r < 0.0)) r += b; }
  else r = copysign(0.0, b);
  return r;
}
__device__ __forceinline__ double plan_normalize_angle(double th) {       // maths.py
  th = py_mod(th, 2.0 * M_PI);
  if (th >= M_PI) th -= 2.0 * M_PI;
  return th;
}
__device__ __forceinline__ double plan_steer_cost(double a_th, double b_th) {      // mp_search_ww_generic.py:59-79
  double d = b_th - a_th;
  d = py_mod(d + M_PI, 2.0 * M_PI) - M_PI;
  return fabs(d);
}
// tuple comparison of two heap entries: (g + h, g, node, predecessor)
__device__ __forceinline__ bool plan_less(const PlanNode* pool, int a, int b) {
  const PlanNode& A = pool[a]; const PlanNode& Bn = pool[b];
  if (A.gh != Bn.gh) return A.gh < Bn.gh;
  if (A.g != Bn.g) return A.g < Bn.g;
  if (A.x != Bn.x) return A.x < Bn.x;
  if (A.y != Bn.y) return A.y < Bn.y;
  if (A.th != Bn.th) return A.th < Bn.th;
  const PlanNode& PA = pool[A.parent]; const PlanNode& PB = pool[Bn.parent];
  if (PA.x != PB.x) return PA.x < PB.x;
  if (PA.y != PB.y) return PA.y < PB.y;
  return PA.th < PB.th;
}
__device__ inline void plan_heap_push(const PlanNode* pool, int* heap, int& n, int e) {
  int i = n++;
  while (i > 0) {
    const int p = (i - 1) >> 1;
    if (!plan_less(pool, e, heap[p])) break;
    heap[i] = heap[p];
    i = p;
  }
  heap[i] = e;
}
__device__ inline int plan_heap_pop(const PlanNode* pool, int* heap, int& n) {
  const int top = heap[0];
  const int last = heap[--n];
  int i = 0;
  for (;;) {
    int c = 2 * i + 1;
    if (c >= n) break;
    if (c + 1 < n && plan_less(pool, heap[c + 1], heap[c])) ++c;
    if (!plan_less(pool, heap[c], last)) break;
    heap[i] = heap[c];
    i = c;
  }
  if (n > 0) heap[i] = last;
  return top;
}
// closed set = the reference's pred_dict: node floats -> pool entry that was expanded for it
__device__ __forceinline__ unsigned plan_hash(double x, double y, double th) {
  unsigned long long h = (unsigned long long)__double_as_longlong(x + 0.0) * 0x9E3779B97F4A7C15ull;
  h ^= (unsigned long long)__double_as_longlong(y + 0.0) * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2);
  h ^= (unsigned long long)__double_as_longlong(th + 0.0) * 0x165667B19E3779F9ull + (h << 6) + (h >> 2);
  return (unsigned)(h ^ (h >> 32));
}
__device__ inline int plan_find(const PlanNode* pool, const int* table, int mask, double x, double y, double th, int* slot_out) {
  unsigned s = plan_hash(x, y, th) & (unsigned)mask;
  for (;;) {
    const int e = table[s];
    if (e < 0) { if (slot_out) *slot_out = (int)s; return -1; }
    if (pool[e].x == x && pool[e].y == y && pool[e].th == th) { if (slot_out) *slot_out = (int)s; return e; }
    s = (s + 1) & (unsigned)mask;
  }
}

__global__ void __launch_bounds__(128) plan_kernel(const PlanArgs A) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= A.B) return;
  const unsigned full = 0xffffffffu;
  PlanNode* pool = A.pool + (size_t)b * A.pool_cap;
  int* heap = A.heap + (size_t)b * A.pool_cap;
  int* table = A.table + (size_t)b * A.table_size;
  const int mask = A.table_size - 1;
  for (int i = lane; i < A.table_size; i += 32) table[i] = -1;
  // jmpc_plan_host rejects an out-of-range scene id on the host; jmpc_plan's ids live on the device and are clamped here
  const int scene = A.scene_id ? min(max(A.scene_id[b], 0), A.n_scenes - 1) : 0;
  const double* hp = A.hp + (size_t)scene * A.max_obs * JMPC_PLAN_MAX_HP * 3;
  const int* hp_n = A.hp_n + (size_t)scene * A.max_obs;
  const int n_obs = A.n_obs[scene];
  const double* W = A.weights + (size_t)b * 9;
  const double wh_dist = W[0], wh_theta = W[1], wh_steering = W[2], wh_obstacle = W[3], wh_center = W[4];
  const double wc_dist = W[5], wc_steering = W[6], wc_obstacle = W[7], wc_center = W[8];
  const double sx = A.start[3 * b], sy = A.start[3 * b + 1], sth = A.start[3 * b + 2];
  const double gx = A.goal_point[3 * b], gy = A.goal_point[3 * b + 1], gth = A.goal_point[3 * b + 2];
  const double ax1 = A.goal_area[4 * b], ay1 = A.goal_area[4 * b + 1], ax2 = A.goal_area[4 * b + 2], ay2 = A.goal_area[4 * b + 3];
  const double allowed = A.allowed[b];
  __syncwarp();

  // distance_to_nearest_obstacle (mp_search_ww_generic.py:81-119): distance to the half-plane LINES, as written there
  auto nearest_obstacle = [&](double x, double y) -> double {
    double best = INFINITY;
    for (int o = 0; o < n_obs; ++o) {
      double dmin = INFINITY;
      for (int k = 0; k < hp_n[o]; ++k) {
        const double* h = hp + ((size_t)o * JMPC_PLAN_MAX_HP + k) * 3;
        const double num = fabs(__dadd_rn(__dadd_rn(__dmul_rn(h[0], x), __dmul_rn(h[1], y)), h[2]));
        const double d = num / sqrt(__dadd_rn(__dmul_rn(h[0], h[0]), __dmul_rn(h[1], h[1])));
        dmin = fmin(dmin, d);
      }
      if (dmin < best) best = dmin;
    }
    return best;
  };
  auto heuristic = [&](double x, double y, double th) -> double {          // distance_to_goal, :170-197
    const double ex = x - gx, ey = y - gy;
    const double dxy = sqrt(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)));
    const double dth = fmin(fabs(th - gth), fabs(th - gth) - allowed / 2);
    const double sc = plan_steer_cost(th, gth);
    double oc = 0.0, dc = 0.0;
    if (wh_obstacle != 0.0) { const double d = nearest_obstacle(x, y); oc = (d != 0.0) ? 1.0 / d : INFINITY; }
    if (wh_center != 0.0) dc = sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
    double h = __dmul_rn(wh_dist, dxy);
    h = __dadd_rn(h, __dmul_rn(wh_theta, dth));
    h = __dadd_rn(h, __dmul_rn(wh_steering, sc));
    h = __dadd_rn(h, __dmul_rn(wh_obstacle, oc));
    h = __dadd_rn(h, __dmul_rn(wh_center, dc));
    return h;
  };

  int pool_n = 0, heap_n = 0, expansions = 0;
  int status = JMPC_PLAN_NO_SOLUTION, goal_entry = -1;
  if (lane == 0) {
    pool[0] = PlanNode{sx, sy, sth, 0.0, 0.0, 0, -1};          // (0, 0, start, start)
    heap[0] = 0;
  }
  pool_n = 1; heap_n = 1;
  __syncwarp();

  for (;;) {
    // ---- pop until an entry that is not superseded (a_star.py:46-53)
    int e = -1;
    if (lane == 0) {
      while (heap_n > 0) {
        const int c = plan_heap_pop(pool, heap, heap_n);
        const int seen = plan_find(pool, table, mask, pool[c].x, pool[c].y, pool[c].th, nullptr);
        if (seen >= 0 && pool[c].g >= pool[seen].g) continue;
        e = c;
        break;
      }
    }
    e = __shfl_sync(full, e, 0);
    heap_n = __shfl_sync(full, heap_n, 0);
    if (e < 0) break;                                           // open list empty: "No solution found."
    if (expansions >= A.max_expansions) { status = JMPC_PLAN_LIMIT; break; }
    const double nx = pool[e].x, ny = pool[e].y, nth = pool[e].th, ng = pool[e].g;
    if (lane == 0) {
      if (A.log && expansions < A.max_log) {
        double* L = A.log + ((size_t)b * A.max_log + expansions) * 5;
        L[0] = ng; L[1] = pool[e].gh - ng; L[2] = nx; L[3] = ny; L[4] = nth;
      }
      int slot;
      plan_find(pool, table, mask, nx, ny, nth, &slot);
      table[slot] = e;                                          // pred_dict[node] = g, predecessor
    }
    ++expansions;
    __syncwarp();
    // ---- goal test (mp_search_ww_generic.py:147-152; BoxObstacle.distance_to_point, obstacles.py:93-101)
    {
      const double dx = fmax(fmax(ax1 - nx, 0.0), nx - ax2), dy = fmax(fmax(ay1 - ny, 0.0), ny - ay2);
      if (sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))) <= 1e-5 && fabs(nth - gth) <= allowed) {
        status = JMPC_PLAN_FOUND; goal_entry = e;
        break;
      }
    }
    if (pool_n + A.n_mp > A.pool_cap) { status = JMPC_PLAN_LIMIT; break; }
    // ---- neighbours (mp_search_ww_generic.py:210-243)
    double sn, cs;
    sincos(nth, &sn, &cs);
    // collision: check point (m, j) in world space against every obstacle's half-plane set
    unsigned collide = 0u;                                       // bit m: primitive m collides
    const int pairs = A.n_mp * A.n_cc;
    for (int base = 0; base < pairs; base += 32) {
      const int idx = base + lane;
      bool hit = false;
      int m = 0;
      if (idx < pairs) {
        m = idx / A.n_cc;
        const double px = A.mp_cc[2 * idx], py = A.mp_cc[2 * idx + 1];
        const double wx = fma(-sn, py, cs * px) + nx, wy = fma(cs, py, sn * px) + ny;
        for (int o = 0; o < n_obs && !hit; ++o) {
          bool inside = true;
          for (int k = 0; k < hp_n[o] && inside; ++k) {
            const double* h = hp + ((size_t)o * JMPC_PLAN_MAX_HP + k) * 3;
            inside = (fma(h[1], wy, h[0] * wx) + h[2]) <= 0.0;
          }
          hit = inside;
        }
      }
      // fold the lanes' verdicts into the per-primitive mask
      for (int src = 0; src < 32; ++src) {
        const int hm = __shfl_sync(full, hit ? m : -1, src);
        if (hm >= 0) collide |= 1u << hm;
      }
    }
    // lane m evaluates primitive m
    bool push = false;
    PlanNode cand;
    if (lane < A.n_mp && !((collide >> lane) & 1u)) {
      const double* endp = A.mp_pts + ((size_t)lane * A.n_pts + (A.n_pts - 1)) * 3;
      const double x = fma(-sn, endp[1], cs * endp[0]) + nx, y = fma(cs, endp[1], sn * endp[0]) + ny;
      const double th = plan_normalize_angle(endp[2] + nth);
      const double sc = plan_steer_cost(nth, th);
      double oc = 0.0, dc = 0.0;
      if (wh_obstacle != 0.0) { const double d = nearest_obstacle(x, y); oc = (d != 0.0) ? 1.0 / d : INFINITY; }   // (sic) wh, :234
      if (wc_center != 0.0) dc = sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
      double edge = __dmul_rn(wc_dist, A.mp_len[lane]);
      edge = __dadd_rn(edge, __dmul_rn(wc_steering, sc));
      edge = __dadd_rn(edge, __dmul_rn(wc_obstacle, oc));
      edge = __dadd_rn(edge, __dmul_rn(wc_center, dc));
      const double g2 = __dadd_rn(ng, edge);
      const int seen = plan_find(pool, table, mask, x, y, th, nullptr);
      if (seen < 0 || g2 < pool[seen].g) {                      // a_star.py:71
        push = true;
        cand = PlanNode{x, y, th, g2, __dadd_rn(g2, heuristic(x, y, th)), e, lane};
      }
    }
    const unsigned pm = __ballot_sync(full, push);
    if (push) pool[pool_n + __popc(pm & ((1u << lane) - 1u))] = cand;
    __syncwarp();
    if (lane == 0) {
      const int cnt = __popc(pm);
      for (int k = 0; k < cnt; ++k) plan_heap_push(pool, heap, heap_n, pool_n + k);
    }
    pool_n += __popc(pm);
    heap_n = __shfl_sync(full, heap_n, 0);
    __syncwarp();
  }

  // ---- path reconstruction through the closed set (a_star.py:58-67) and the full trajectory (:245-256)
  int n_path = 0, n_traj = 0;
  if (status == JMPC_PLAN_FOUND) {
    if (lane == 0) {
      // walk back: node <- predecessor, predecessor <- pred_dict[predecessor]
      int cur = goal_entry, len = 1;
      while (!(pool[cur].x == sx && pool[cur].y == sy && pool[cur].th == sth) && len <= A.pool_cap) {
        const PlanNode& P = pool[pool[cur].parent];
        cur = plan_find(pool, table, mask, P.x, P.y, P.th, nullptr);
        ++len;
      }
      n_path = len;
      if (len <= A.max_path) {
        cur = goal_entry;
        for (int i = len - 1; i >= 0; --i) {
          double* q = A.path + ((size_t)b * A.max_path + i) * 3;
          q[0] = pool[cur].x; q[1] = pool[cur].y; q[2] = pool[cur].th;
          if (i > 0) {
            A.path_mp[(size_t)b * A.max_path + i - 1] = pool[cur].mp;
            const PlanNode& P = pool[pool[cur].parent];
            cur = plan_find(pool, table, mask, P.x, P.y, P.th, nullptr);
          }
        }
      }
    }
    n_path = __shfl_sync(full, n_path, 0);
    __syncwarp();
    if (n_path > A.max_path) status = JMPC_PLAN_LIMIT;
    else {
      const int per = A.n_pts - 1;                              // motion_primitive_at(...)[:-1]
      n_traj = (n_path - 1) * per;
      if (n_traj > A.max_traj) status = JMPC_PLAN_LIMIT;
      else
        for (int edge = 0; edge < n_path - 1; ++edge) {
          const double* q = A.path + ((size_t)b * A.max_path + edge) * 3;
          const int m = A.path_mp[(size_t)b * A.max_path + edge];
          double sn, cs;
          sincos(q[2], &sn, &cs);
          for (int j = lane; j < per; j += 32) {
            const double* p = A.mp_pts + ((size_t)m * A.n_pts + j) * 3;
            double* out = A.traj + ((size_t)b * A.max_traj + (size_t)edge * per + j) * 3;
            out[0] = fma(-sn, p[1], cs * p[0]) + q[0];
            out[1] = fma(cs, p[1], sn * p[0]) + q[1];
            out[2] = p[2] + q[2];
          }
        }
    }
  }
  if (lane == 0) {
    A.status[b] = status;
    A.cost[b] = (status == JMPC_PLAN_FOUND) ? pool[goal_entry].g : nan("");
    A.n_path[b] = (status == JMPC_PLAN_FOUND) ? n_path : 0;
    A.n_traj[b] = (status == JMPC_PLAN_FOUND) ? n_traj : 0;
    A.expansions[b] = expansions;
  }
}

}  // namespace jmpc
