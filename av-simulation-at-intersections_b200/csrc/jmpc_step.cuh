// jmpc_step.cuh -- the fused MPC-step kernel: one lane group (a whole warp, or half a warp for horizons T <= 15)
// owns one instance.
//
// Pipeline per instance (reference lines relative to SaeedRahmani/AV-Simulation-at-Intersections):
//   1. nearest forward index on the course        main/lib/trajectories.py:100-126
//   2. reference sampling xref / reaches_end      main/lib/mpc.py:89-112
//   3. operating-point rollout xbar               main/lib/mpc.py:115-129, main/lib/simulation.py:35-47,
//                                                 main/bicycle/main.py:28-41
//   4. linearisation + exact condensing           main/lib/mpc.py:61-82,132-138,151-194  (states eliminated; the
//      unknowns are the cumulative accelerations s_k = a_0 + .. + a_k and the steering angles: see step_prep)
//   5. QP solve: Mehrotra predictor-corrector interior point on the n = 2T condensed problem; the normal
//      matrix K = P + A' diag(w) A lives in shared memory, its Cholesky factor overwrites it in place
//      (replaces cvxpy + ECOS, mpc.py:196-197)
//   6. outputs: controls, predicted states, cost, status             main/lib/mpc.py:199-209
//
// All arithmetic is float64: the index decisions (rint, 3-nearest rule) must match numpy bit for bit, and
// the condensed Hessians have cond ~1e6..1e7 (SURVEY.md section 6), far outside what fp32 factors resolve
// at the 1e-4 control tolerance.
//
// Lane groups.  Lane k of a group owns horizon stage k, so an instance needs T + 1 lanes: with the reference's
// default horizon (T = 13) a warp-per-instance mapping leaves 18 of 32 lanes idle in all the row work and pays every
// synchronisation, every redundant diagonal-block factorisation and every shuffle reduction for one instance only.
// The kernel is therefore a template on G, the lanes per instance: G = 16 packs two independent instances into a
// warp (one per half), G = 32 is the whole warp (T >= 16).  The groups of a warp run in lock step: every phase is
// uniform control flow (a group that is finished, failed or has no instance left keeps executing on its own
// shared-memory region with its commits switched off).  Phases A and C have group-uniform early exits, so their
// shuffles and synchronisations are group-scoped and never depend on the halves being converged; the solve phase has
// none and names the whole warp (step_solve).
//
// Two instantiations per horizon: the throughput kernel (four warps per block, 128 registers, sweeps through shared
// memory) and the low-latency kernel for launches of at most eight warps per SM (one warp per block, ~190 registers,
// sweeps with the vector in registers).  Same results bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/jmpc.h"
#include "jmpc_linalg.cuh"

namespace jmpc {

constexpr int kMaxT = JMPC_MAX_T;
constexpr unsigned kFull = 0xffffffffu;

struct ParamVec { double v[JMPC_NPARAM]; };

struct StepArgs {
  int B, T;
  int lin_iters;            // MAX_ITER of the reference config
  int max_iters;            // interior-point iteration cap
  double mu_tol;
  double tol_res;           // primal / (scaled) dual residual tolerance of the strict exit
  double init_mu;           // > 0: centred start lambda = init_mu / s ; 0: lambda = 1
  double du_th;             // > 0: leave the linearisation loop once sum|du| <= du_th (mpc.py:236-240, commented out there)
  // course tables
  const double* cx; const double* cy; const double* cyaw;
  const double* cv;         // reference speed profile per course point (mpc_with_speed.py:104) or nullptr
  const int* course_n; int course_stride; int n_courses;
  // inputs
  const double* state; const int* course_id; const int* course_len; const int* warm;
  const double* params;     // [B][NPARAM] or nullptr
  double defaults[JMPC_NPARAM];
  // in-out: read from target_ind / oa / od, written to the *_out twins (the same arrays for jmpc_step; the host
  // entry point reads device copies and writes page-locked host memory directly)
  const int* target_ind; const double* oa; const double* od;
  int* target_out; double* oa_out; double* od_out;
  double* ox; double* oy; double* ov; double* oyaw; double* xref; double* cost; int* status; int* iters;
  double* record;           // [B][JMPC_RECORD_LEN] or nullptr
  // fused all-gather: the epilogue also stores the record into every peer GPU's gathered table (NVLink peer
  // memory, jmpc_set_record_peers); peer p's table is [world * B][JMPC_RECORD_LEN], this rank owns rows
  // rank_offset .. rank_offset + B - 1
  const int* skip;          // [B] or nullptr: instances with skip[b] != 0 are left untouched (finished episodes)
  const int* order;         // [B] or nullptr: the work queue hands out order[ticket] instead of ticket (longest first)
  int* work_hint;           // [B] or nullptr: solver iterations this step, the next step's scheduling key
  double* peer_rec[JMPC_MAX_PEERS];
  int n_peers;
  long long rank_offset;
  // completion flags of the fused all-gather (jmpc_set_record_flags): when the last block of the launch retires it
  // stores gather_step into this rank's slot of every peer's flag array (release, system scope), after every record
  unsigned long long* peer_flag[JMPC_MAX_PEERS];
  int n_flag_peers;
  unsigned long long gather_step;
  unsigned int* blocks_done;       // retired-block counter of the launch (reset by the last block)
  // scratch
  double* pscratch;         // [resident groups][tiles_doubles(n)] condensed Hessian on tiles, L2 resident
  unsigned int* counter;    // dynamic work queue
};

constexpr int kSlotHi3 = JMPC_NPARAM, kSlotLo3 = JMPC_NPARAM + 1, kSlotLim = JMPC_NPARAM + 2;   // derived bounds
constexpr int kSlotGscale = JMPC_NPARAM + 3;     // the solver's dual-residual scale
constexpr int kParamSlots = 32;
static_assert(JMPC_NPARAM + 4 <= kParamSlots, "parameter block too small");

// suffix-moment slots of the Hessian assembly (step_prep): weight x centred prefix products
enum MomentSlot {
  MOM_11, MOM_11_B, MOM_11_BB,
  MOM_12, MOM_12_B, MOM_12_K, MOM_12_BK,
  MOM_22, MOM_22_K, MOM_22_KK,
  MOM_QPSI, MOM_WX, MOM_WY, MOM_COUNT
};

// shared-memory doubles one instance needs for horizon T (every sub-array starts 16-byte aligned)
__host__ __device__ inline int even_up(int x) { return (x + 1) & ~1; }
// the K region also hosts the suffix moments during the condensing (short horizons need more room for those)
__host__ __device__ inline int k_region_doubles(int T) {
  const int a = tiles_doubles(2 * T), b = MOM_COUNT * even_up(T + 1);
  return a > b ? a : b;
}
#ifndef JMPC_PAD_T1E
#define JMPC_PAD_T1E 0          // layout experiments: unused (T + 1)-arrays between epsi and vb
#endif
__host__ __device__ inline int inst_smem_doubles(int T) {
  const int n = 2 * T, n4 = nblk(n) << 2, T1e = even_up(T + 1), Te = even_up(T);
  return k_region_doubles(T)    // K / L on 4x4 tiles (and the condensing's moment tables)
         + 4 * n4               // u, q, rhs, grad
         + (9 + JMPC_PAD_T1E) * T1e   // alp, cb, wvs, ck (condensing); WeX, WeY, epsi; vb, th
         + 4 * Te               // per-iteration barrier terms wA, wD, wR, wS
         + kParamSlots          // the instance's parameter vector + derived row bounds
         + 2;                   // mbarrier of the TMA Hessian copy (8 bytes, padded to 16)
}

// lanes per instance for horizon T: lane k owns stage k and horizon point k (T + 1 points)
__host__ __device__ inline int group_lanes_for(int T) { return (T + 1 <= 16) ? 16 : 32; }

// dynamic shared memory of a block of `wpb` warps with `groups` instances each: the instances' regions plus the
// block-shared Cholesky task table
__host__ __device__ inline size_t step_block_smem_bytes(int T, int wpb, int groups) {
  return (size_t)wpb * groups * inst_smem_doubles(T) * sizeof(double) + chol_lut_bytes(nblk(2 * T));
}

__device__ __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }

// ---- group-scoped collectives: G lanes, `gm` = the group's lane mask, `gl` = lane index inside the group ----------
template <int G>
__device__ __forceinline__ unsigned group_mask(int lane) {
  if constexpr (G == 32) return kFull;
  else return ((1u << G) - 1u) << (lane & ~(G - 1));
}
// a > b ? a : b -- two selects; fmax() costs a NaN fix-up and three more moves per call, and nothing here is NaN unless
// the solve has already failed
__device__ __forceinline__ double dmax(double a, double b) { return a > b ? a : b; }
template <int G>
__device__ __forceinline__ double grp_sum(double v, unsigned gm) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gm, v, o);
  return v;
}
template <int G>
__device__ __forceinline__ double grp_max(double v, unsigned gm) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = dmax(v, __shfl_xor_sync(gm, v, o));
  return v;
}
// true when `p` holds on every lane of the group.  The half-warp kernels vote with the whole warp (their groups run
// in lock step through every place this is used) and look at their own half of the ballot.
template <int G>
__device__ __forceinline__ bool grp_all(bool p) {
  if constexpr (G == 32) return __all_sync(kFull, p);
  else {
    const unsigned sh = (threadIdx.x & 31u) & ~(unsigned)(G - 1), ones = (1u << G) - 1u;
    return ((__ballot_sync(kFull, p) >> sh) & ones) == ones;
  }
}
// One step of a scan inside a lane group: v += the value held `o` lanes below (above), when that lane belongs to
// the group.  shfl.sync reports that in a predicate, which saves the lane-index compares of `if (gl >= o) v += t`
// (ptxas still turns the predicated add into an add and a select): 4 % fewer instructions in the solver loop.
template <int G>
__device__ __forceinline__ void scan_step_up(double& v, unsigned o, unsigned gm) {
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 lo, hi, tlo, thi;\n\t.reg .f64 t;\n\t"
               "mov.b64 {lo, hi}, %0;\n\t"
               "shfl.sync.up.b32 tlo|p, lo, %1, %2, %3;\n\t"
               "shfl.sync.up.b32 thi, hi, %1, %2, %3;\n\t"
               "mov.b64 t, {tlo, thi};\n\t"
               "@p add.rn.f64 %0, %0, t;\n\t}"
               : "+d"(v) : "r"(o), "n"((32 - G) << 8), "r"(gm));
}
template <int G>
__device__ __forceinline__ void scan_step_down(double& v, unsigned o, unsigned gm) {
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 lo, hi, tlo, thi;\n\t.reg .f64 t;\n\t"
               "mov.b64 {lo, hi}, %0;\n\t"
               "shfl.sync.down.b32 tlo|p, lo, %1, %2, %3;\n\t"
               "shfl.sync.down.b32 thi, hi, %1, %2, %3;\n\t"
               "mov.b64 t, {tlo, thi};\n\t"
               "@p add.rn.f64 %0, %0, t;\n\t}"
               : "+d"(v) : "r"(o), "n"(((32 - G) << 8) | 0x1f), "r"(gm));
}
// inclusive prefix sum over the group's lanes
template <int G>
__device__ __forceinline__ double grp_scan(double v, int gl, unsigned gm) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) scan_step_up<G>(v, (unsigned)o, gm);
  (void)gl;
  return v;
}
// inclusive suffix sum: out[gl] = sum_{l >= gl} v[l]
template <int G>
__device__ __forceinline__ double grp_rscan(double v, int gl, unsigned gm) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) scan_step_down<G>(v, (unsigned)o, gm);
  (void)gl;
  return v;
}

// One lane writes the instance's result record locally and, when peers are set, into every peer's gathered table
// (one 64-byte store each; with NVSwitch every peer is one hop away, and the stores are the only communication of
// the whole step -- the all-gather is fused into the solve kernel's epilogue).
__device__ __forceinline__ void write_record(const StepArgs& A, int b, double r0, double r1, double r2, double r3,
                                             double r4, double r5, double r6, double r7) {
  if (A.record) {
    double2* rec = reinterpret_cast<double2*>(A.record + (size_t)b * JMPC_RECORD_LEN);
    rec[0] = make_double2(r0, r1); rec[1] = make_double2(r2, r3); rec[2] = make_double2(r4, r5); rec[3] = make_double2(r6, r7);
  }
  for (int p = 0; p < A.n_peers; ++p) {
    double2* rec = reinterpret_cast<double2*>(A.peer_rec[p] + ((size_t)A.rank_offset + b) * JMPC_RECORD_LEN);
    rec[0] = make_double2(r0, r1); rec[1] = make_double2(r2, r3); rec[2] = make_double2(r4, r5); rec[3] = make_double2(r6, r7);
  }
}

// An instance that is not solved keeps its in-out values: when the write side is a different array (host entry
// points) they are carried over here.
__device__ __forceinline__ void carry_inout(const StepArgs& A, int b, int T, int gl) {
  if (A.oa_out != A.oa && gl < T) A.oa_out[(size_t)b * T + gl] = A.oa[(size_t)b * T + gl];
  if (A.od_out != A.od && gl < T) A.od_out[(size_t)b * T + gl] = A.od[(size_t)b * T + gl];
  if (A.target_out != A.target_ind && gl == 0) A.target_out[b] = A.target_ind[b];
}

// ---- candidate list for the 3-nearest rule: ascending by (d2, index) --------------------------------
struct Near3 {
  double d0, d1, d2; int i0, i1, i2;
};
__device__ __forceinline__ bool closer(double da, int ia, double db, int ib) {
  return (da < db) || (da == db && ia < ib);
}
__device__ __forceinline__ void near3_insert(Near3& s, double d, int i) {
  if (closer(d, i, s.d2, s.i2)) {
    if (closer(d, i, s.d1, s.i1)) {
      s.d2 = s.d1; s.i2 = s.i1;
      if (closer(d, i, s.d0, s.i0)) { s.d1 = s.d0; s.i1 = s.i0; s.d0 = d; s.i0 = i; }
      else { s.d1 = d; s.i1 = i; }
    } else { s.d2 = d; s.i2 = i; }
  }
}

// Nearest forward index (trajectories.py:100-126).  Returns -1 when the rule raises.
// Distances are compared squared (monotone in the reference's sqrt); products are kept unfused so the
// ordering matches numpy's dx*dx + dy*dy.  Ties break towards the lower index.
template <int G>
__device__ inline int nearest_index(const double* __restrict__ cx, const double* __restrict__ cy, int n_course,
                                    int start, double x, double y, int gl, unsigned gm) {
  const int m = n_course - start;
  if (m <= 1) return start;
  if (m == 2) return start + 1;
  Near3 s;
  s.d0 = s.d1 = s.d2 = INFINITY;
  s.i0 = s.i1 = s.i2 = 0x7fffffff;
  for (int j = start + gl; j < n_course; j += G) {
    const double ex = cx[j] - x, ey = cy[j] - y;
    const double d = __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey));
    near3_insert(s, d, j - start);
  }
  int res[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    // global best among the lanes' heads
    double bd = s.d0; int bi = s.i0;
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(gm, bd, o);
      const int oi = __shfl_xor_sync(gm, bi, o);
      if (closer(od, oi, bd, bi)) { bd = od; bi = oi; }
    }
    res[r] = bi;
    if (s.i0 == bi) {   // the owner pops its head
      s.d0 = s.d1; s.i0 = s.i1; s.d1 = s.d2; s.i1 = s.i2; s.d2 = INFINITY; s.i2 = 0x7fffffff;
    }
  }
  if (abs(res[1] - res[2]) == 2) return res[0] + start;
  if (abs(res[0] - res[1]) == 1) return max(res[0], res[1]) + start;
  return -1;
}

// ---- per-instance shared-memory views ------------------------------------------------------------------
struct WarpMem {
  double *K, *u, *q, *rhs, *grad;
  double *alp, *cb, *wvs, *ck;          // condensing: alpha_{k+1}, centred prefix sums B, speed weight per stage, K
  double *WeX, *WeY, *epsi, *vb, *th;
  double *wA, *wD, *wR, *wS;            // solver: barrier terms of K (wA / wD diagonal, wS / wR sub-diagonal, s / steering block)
  double *prm;
  unsigned long long* mbar;
  __device__ WarpMem(double* base, int T) {
    const int n = 2 * T, n4 = nblk(n) << 2, T1e = even_up(T + 1), Te = even_up(T);
    double* p = base;
    K = p; p += k_region_doubles(T);
    u = p; p += n4; q = p; p += n4; rhs = p; p += n4; grad = p; p += n4;
    // grad .. epsi are dead while the solver runs: 4 (2T) + 7 (T + 1) >= 8T doubles, the solver's row stash
    alp = p; p += T1e; cb = p; p += T1e; wvs = p; p += T1e; ck = p; p += T1e;
    WeX = p; p += T1e; WeY = p; p += T1e; epsi = p; p += T1e;
    p += JMPC_PAD_T1E * T1e;
    vb = p; p += T1e; th = p; p += T1e;
    wA = p; p += Te; wD = p; p += Te; wR = p; p += Te; wS = p; p += Te;
    prm = p; p += kParamSlots;
    mbar = reinterpret_cast<unsigned long long*>(p);
  }
};

// ---- TMA 1-D bulk copy global -> shared (cp.async.bulk, SASS UBLKCP) completing on an mbarrier --------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
// one lane: order the warp's earlier generic-proxy accesses before the async proxy, arm the barrier with the byte
// count and issue the copy (bytes: multiple of 16; both addresses 16-byte aligned)
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
  asm volatile("fence.proxy.async;\n" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}

// z = A u for the stage rows (u = [s; delta] in shared memory): acceleration s_k - s_{k-1}, steering angle, steering
// rate delta_{k+1} - delta_k, cumulative acceleration s_k (the speed row).  Rows beyond the horizon are garbage here
// and switched off by the caller.
template <int G>
__device__ __forceinline__ void rows_apply(const double* u, int T, int gl, unsigned gm, double z[4]) {
  const double sk = (gl < T) ? u[gl] : 0.0, sm = (gl >= 1 && gl <= T) ? u[gl - 1] : 0.0;
  const double d = (gl < T) ? u[T + gl] : 0.0;
  const double dn = __shfl_down_sync(gm, d, 1, G);
  z[0] = sk - sm; z[1] = d; z[2] = dn - d; z[3] = sk;
}
// the same for a vector held in registers (a = entry gl, d = entry T + gl; 0 beyond the horizon), with exact zeros
// on the dead rows (z[1], z[3] are zero there by construction)
template <int G>
__device__ __forceinline__ void rows_apply_reg(double a, double d, int gl, unsigned gm, bool live013, bool live2,
                                               double z[4]) {
  const double dn = __shfl_down_sync(gm, d, 1, G);
  double am = __shfl_up_sync(gm, a, 1, G);
  if (gl == 0) am = 0.0;
  z[0] = live013 ? a - am : 0.0; z[1] = d; z[2] = live2 ? dn - d : 0.0; z[3] = a;
}
// (A' t): this lane's entries for s_k (ra) and delta_k (rd); dead rows must carry t = 0
template <int G>
__device__ __forceinline__ void rows_apply_T(const double t[4], int gl, unsigned gm, double& ra, double& rd) {
  const double t0n = __shfl_down_sync(gm, t[0], 1, G);     // the acceleration row of stage k + 1 (0 behind the horizon;
  ra = t[0] - t0n + t[3];                                  //  the group's last lane is never a live stage)
  double up = __shfl_up_sync(gm, t[2], 1, G);
  if (gl == 0) up = 0.0;
  rd = t[1] - t[2] + up;
}

// reference speed of horizon point `idx` (xref[2]): 0 for lib.mpc (mpc.py:107); the speed profile of
// mpc_with_speed.py:104 is either a per-course table or the two-level profile its set_trajectory_fromarray builds
// (V_REF before the cut index, 0 from there on); a cut index also applies on top of a table
__device__ __forceinline__ double ref_speed(const StepArgs& A, const double* prm, int cid, int idx) {
  if (!((double)idx < prm[JMPC_P_V_REF_CUT])) return 0.0;
  return A.cv ? A.cv[(size_t)cid * A.course_stride + idx] : prm[JMPC_P_V_REF];
}

// ---- phase A: index, reference sampling, rollout, linearisation, condensing --------------------------------
// Leaves everything the later phases need in shared memory / the L2 scratch; returns a jmpc_status
// (JMPC_OPTIMAL = go on and solve).  `active` = this group holds a real instance (its failures are reported).
template <int TT, int G>
__device__ __noinline__ int step_prep(const StepArgs& A, int b, bool active, double* smem_base, double* pscr, int gl,
                                      unsigned gm, int lin, int total_iters, double oa_k, double od_k, double ov_k,
                                      int& target, int& idx_out, unsigned& end_mask_out) {
  const int T = (TT > 0) ? TT : A.T;
  const int n = 2 * T, T1 = T + 1, nb = nblk(n), n4 = nb << 2;
  WarpMem M(smem_base, T);
  auto P = [&](int k) -> double { return M.prm[k]; };
  const int cid = A.course_id ? min(max(A.course_id[b], 0), A.n_courses - 1) : 0;     // device arrays are clamped, host arrays validated
  const double* cx = A.cx + (size_t)cid * A.course_stride;
  const double* cy = A.cy + (size_t)cid * A.course_stride;
  const double* cyaw = A.cyaw + (size_t)cid * A.course_stride;
  int n_course = A.course_n[cid];
  if (A.course_len) n_course = min(n_course, max(A.course_len[b], 1));
  const double x0 = A.state[(size_t)b * 4 + 0], y0 = A.state[(size_t)b * 4 + 1];
  const double v0 = A.state[(size_t)b * 4 + 2], yaw0 = A.state[(size_t)b * 4 + 3];
  const double dt = P(JMPC_P_DT), dl = P(JMPC_P_DL), Lw = P(JMPC_P_L), speed = P(JMPC_P_SPEED);
  const double min_speed = P(JMPC_P_MIN_SPEED);
  if (lin == 0) target = min(max(target, 0), n_course);      // numpy slicing clamps an out-of-range start
  // ---------------- 1. nearest index --------------------------------------------------------------
  const int near = nearest_index<G>(cx, cy, n_course, target, x0, y0, gl, gm);
  if (near < 0) {                        // group-uniform; the rest of the phase only touches this group's memory
    if (active) {
      carry_inout(A, b, T, gl);
      if (gl == 0) {
        A.status[b] = JMPC_INDEX_RULE; if (A.iters) A.iters[b] = total_iters;
        write_record(A, b, nan(""), nan(""), nan(""), JMPC_INDEX_RULE, A.target_ind[b], total_iters, nan(""), nan(""));
      }
    }
    return JMPC_INDEX_RULE;
  }
  target = near;

  // ---------------- 2. reference sampling ---------------------------------------------------------
  // travel = cumsum(|ov| dt): sequential float64 adds, reproduced literally (lane k owns point k)
  double sp_k;
  if (lin == 0) sp_k = fabs(fmax(v0, P(JMPC_P_V_REF_MIN))) * dt; else sp_k = fabs(ov_k) * dt;
  double travel = 0.0;
  {
    double acc = 0.0;
    for (int j = 0; j <= T; ++j) {          // uniform trip count: every lane takes part in the shuffle
      const double sj = __shfl_sync(gm, sp_k, j, G);
      if (j <= gl) acc = (j == 0) ? sj : __dadd_rn(acc, sj);
    }
    travel = acc;
  }
  int idx = 0;
  bool at_end = false;
  double xr = 0.0, yr = 0.0, psir = 0.0, vr = 0.0;
  if (gl <= T) {
    const long long hop = (long long)rint(travel / dl);
    long long id = hop + (long long)target;
    if (id > (long long)(n_course - 1)) id = n_course - 1;
    if (id < 0) id = 0;
    idx = (int)id;
    at_end = (idx == n_course - 1);
    xr = cx[idx]; yr = cy[idx]; psir = cyaw[idx];
    vr = ref_speed(A, M.prm, cid, idx);     // mpc_with_speed.py:104; 0 for lib.mpc
  }
  // bit t = reaches_end[t]
  const unsigned end_mask = (__ballot_sync(gm, at_end) >> ((threadIdx.x & 31) & ~(G - 1))) & (unsigned)((1ull << G) - 1ull);

  // ---------------- 3. operating-point rollout ----------------------------------------------------
  // The speed recurrence (with the plant's clamp) is walked by every lane redundantly, one shuffle per stage; lane t
  // keeps vbar_t.  The heading is a running sum of per-stage terms that only need the lane's own vbar_t, so it is one
  // group scan instead of a second shuffle, an fp64 division (v / L: ~50 instructions) and the adds on every stage of
  // the walk.  The scan adds in a different order than the reference's loop, and v * (1 / L) differs from v / L in
  // the last bit: the operating point moves by ~1e-16 relative, like the libm differences in tan / sincos (DESIGN.md
  // section 3); no integer decision depends on it.
  const double max_steer = P(JMPC_P_MAX_STEER), vmax_sim = P(JMPC_P_SIM_MAX_SPEED);
  const double tan_k = tan(fmax(fmin(od_k, max_steer), -max_steer));
  double vb = v0;                     // lane t ends up holding vbar_t
  {
    double v = v0;
    const double adt_k = __dmul_rn(oa_k, dt);
    for (int t = 0; t < T; ++t) {
      v = __dadd_rn(v, __shfl_sync(gm, adt_k, t, G));
      v = v > vmax_sim ? vmax_sim : v;
      v = v < min_speed ? min_speed : v;
      if (gl == t + 1) vb = v;
    }
  }
  const double inv_L = 1.0 / Lw;
  const double dth = (gl < T) ? __dmul_rn(__dmul_rn(__dmul_rn(vb, inv_L), tan_k), dt) : 0.0;   // heading gained on stage t
  const double th = yaw0 + (grp_scan<G>(dth, gl, gm) - dth);                                     // phibar_t
  double sn, cs;
  sincos(th, &sn, &cs);
  // (x, y) are only reported (xbar rows 0,1 do not enter the QP); the QP needs vbar, phibar.
  // ---------------- 4. linearisation + condensing -------------------------------------------------
  // per-stage coefficients (stage t = lane, t < T)
  double al = 0.0, be = 0.0, ga = 0.0, ka = 0.0, gk = 0.0;
  if (gl < T) {
    al = dt * cs; be = dt * vb * sn; ga = dt * sn; ka = dt * vb * cs; gk = dt * vb / Lw;
  }
  // The unknowns of the condensed problem are the CUMULATIVE accelerations s_k = a_0 + ... + a_k and the steering
  // angles delta_k: v_t = v0 + dt s_{t-1}, so a speed row is a box on s_k and an acceleration row the difference
  // s_k - s_{k-1} -- no running sums in A or A' (seven group scans per interior-point iteration in the a_k form), and
  // the barrier term A' W A is tridiagonal in both blocks.  A position depends on s_k through v_{k+1} only:
  //   dX_t / ds_k = dt alpha_{k+1},  dY_t / ds_k = dt gamma_{k+1}   for t >= k + 2,
  // constant in t, so the s-block of the Hessian needs plain suffix sums of the stage weights.  The steering
  // sensitivities are  dX_t / ddelta_i = -g_i (B_t - B_{i+1}),  dY_t / ddelta_i = g_i (K_t - K_{i+1})  with the
  // exclusive prefix sums B, K of beta, kappa (lane t: t = 0..T).  Only differences of B, K are ever used, so both
  // are centred on their mid-horizon value: that halves the magnitudes entering the moment expansion below.
  double cb_t = grp_scan<G>(be, gl, gm) - be, ck_t = grp_scan<G>(ka, gl, gm) - ka;
  cb_t -= __shfl_sync(gm, cb_t, T >> 1, G); ck_t -= __shfl_sync(gm, ck_t, T >> 1, G);
  // alpha_{k+1}, gamma_{k+1} for stage k (0 for k = T - 1: s_{T-1} moves no position inside the horizon)
  const double al_next = __shfl_down_sync(gm, al, 1, G), ga_next = __shfl_down_sync(gm, ga, 1, G);
  // free response (u = 0): v = v0, psi = yaw0
  const double fx_term = (gl < T) ? (al * v0 - be * (yaw0 - th)) : 0.0;
  const double fy_term = (gl < T) ? (ga * v0 + ka * (yaw0 - th)) : 0.0;
  const double xf_t = x0 + (grp_scan<G>(fx_term, gl, gm) - fx_term);
  const double yf_t = y0 + (grp_scan<G>(fy_term, gl, gm) - fy_term);
  // stage weights (t = lane, meaningful for 1 <= t <= T)
  double w11 = 0.0, w12 = 0.0, w22 = 0.0, wv = 0.0, wpsi = 0.0;
  if (gl >= 1 && gl <= T) {
    if (at_end) {
      w11 = P(JMPC_P_QF_X); w22 = P(JMPC_P_QF_Y); wv = P(JMPC_P_QF_V); wpsi = P(JMPC_P_QF_YAW);
    } else {
      double s1, c1, s2, c2;
      sincos(psir + 0.5 * M_PI, &s1, &c1);
      sincos(psir, &s2, &c2);
      const double wp = P(JMPC_P_W_PERP), wl = P(JMPC_P_W_PARA);
      w11 = (c1 * c1) * wp + (c2 * c2) * wl;
      w12 = (c1 * s1) * wp + (c2 * s2) * wl;
      w22 = (s1 * s1) * wp + (s2 * s2) * wl;
      wv = P(JMPC_P_Q_V); wpsi = P(JMPC_P_Q_YAW);
    }
  }
  // Suffix moments  mom[m][t0] = sum_{t >= t0} W_t * (product of centred prefix values at t),  13 sequences, kept
  // in the K region (free until the solver starts).  With them every Hessian entry is O(1):
  //   sum_{t>=t0} W (F_t - F0)(G_t - G0) = M_WFG - G0 M_WF - F0 M_WG + F0 G0 M_W.
  const double ex = xf_t - xr, ey = yf_t - yr, ev = v0 - vr, eps = yaw0 - psir;
  const double wex = w11 * ex + w12 * ey, wey = w12 * ex + w22 * ey;
  {
    const bool vt = (gl >= 1 && gl <= T);
    const double B_ = vt ? cb_t : 0.0, K_ = vt ? ck_t : 0.0;
    double* mom = M.K;
    const int ms = even_up(T + 1);
    // every lane (stage) stores its terms; the suffix sums are then taken along the stages by one lane per sequence
    // (a serial add chain of T + 1 terms in shared memory instead of a group scan of 4-5 shuffle steps per sequence)
    auto put = [&](int m, double v) { if (gl <= T) mom[m * ms + gl] = v; };
    put(MOM_11, w11); put(MOM_11_B, w11 * B_); put(MOM_11_BB, w11 * B_ * B_);
    put(MOM_12, w12); put(MOM_12_B, w12 * B_); put(MOM_12_K, w12 * K_); put(MOM_12_BK, w12 * B_ * K_);
    put(MOM_22, w22); put(MOM_22_K, w22 * K_); put(MOM_22_KK, w22 * K_ * K_);
    put(MOM_QPSI, wpsi); put(MOM_WX, vt ? wex : 0.0); put(MOM_WY, vt ? wey : 0.0);
    __syncwarp(gm);
    for (int m = gl; m < MOM_COUNT; m += G) {
      double* seq = mom + m * ms;
      double acc = 0.0;
      for (int t = T; t >= 0; --t) { acc += seq[t]; seq[t] = acc; }
    }
  }
  if (gl <= T) {
    M.cb[gl] = cb_t; M.ck[gl] = ck_t;
    M.WeX[gl] = wex; M.WeY[gl] = wey;
    M.epsi[gl] = wpsi * eps;          // weighted yaw error per stage
    M.grad[gl] = wv * ev;             // weighted speed error per stage (grad is free until the solver starts)
    M.wvs[gl] = wv;                   // speed weight of stage t (the s-block's diagonal)
  }
  if (gl < T) { M.alp[gl] = al_next; M.wD[gl] = ga_next; }    // alpha_{k+1}, gamma_{k+1} (gamma borrows wD, free until the solver starts)
  if (gl < T) M.wA[gl] = gk;          // g_k borrows wA during condensing
  if (gl <= T) { M.vb[gl] = vb; M.th[gl] = th; }       // operating point, reused by the epilogue
  if (gl == 0) {                      // derived row bounds, read back by the solver
    M.prm[kSlotHi3] = (speed - v0) / dt; M.prm[kSlotLo3] = (min_speed - v0) / dt;
    M.prm[kSlotLim] = P(JMPC_P_MAX_DSTEER) * dt;
  }
  __syncwarp(gm);

  const double Ra = P(JMPC_P_R_A), Rd_ = P(JMPC_P_R_D), Rda = P(JMPC_P_RD_A), Rdd = P(JMPC_P_RD_D);
  const double Rea = P(JMPC_P_REND_A), Red = P(JMPC_P_REND_D);
  const double dt2 = dt * dt;
  // Hessian on 4x4 tiles (jmpc_linalg.cuh), variable order [s_0..s_{T-1}, delta_0..delta_{T-1}]; the last
  // block row is cleared first so that the identity padding (n -> multiple of 4) is in place
  {
    const int last0 = tile_off(nb - 1, 0), last1 = tiles_doubles(n);
    for (int e = last0 + gl; e < last1; e += G) pscr[e] = 0.0;
    __syncwarp(gm);
    if (gl < n4 - n) pscr[elem_off(n + gl, n + gl)] = 1.0;
  }
  {
    // Three passes, one per block type (s x s, steer x s, steer x steer): a single pass over the packed
    // triangle mixed steer x s and steer x steer entries in every group of lanes, so the warp executed both paths.
    const int ms = even_up(T + 1);
    // S(W; F, G)(F0, G0) = sum_{t >= t0} W_t (F_t - F0)(G_t - G0) from the suffix moments
    auto S = [&](const double* mom, int mW, int mWF, int mWG, int mWFG, double F0, double G0) -> double {
      return mom[mWFG * ms] - G0 * mom[mWF * ms] - F0 * mom[mWG * ms] + F0 * G0 * mom[mW * ms];
    };
    auto store = [&](int i, int j, double acc) {
      pscr[elem_off(i, j)] = acc;
      if (i != j && (i >> 2) == (j >> 2)) pscr[elem_off(j, i)] = acc;      // diagonal tiles are stored full
    };
    // input and input-rate weights on the (block-)diagonal and first sub-diagonal (mpc.py:180-187)
    auto input_weights = [&](int ki, int kj, double r_run, double r_end, double rd_w) -> double {
      if (ki == kj) {
        const bool e_t = (end_mask >> ki) & 1u;
        const int nbr = (T >= 2) ? ((ki == 0 || ki == T - 1) ? 1 : 2) : 0;
        return 2.0 * (e_t ? r_end : r_run) + 2.0 * rd_w * nbr;
      }
      return (ki == kj + 1) ? -2.0 * rd_w : 0.0;
    };
    // the tridiagonal input-weight matrix of the a_k formulation, any index order, zero outside the horizon
    auto Mw = [&](int i, int j, double r_run, double r_end, double rd_w) -> double {
      if (i >= T || j >= T) return 0.0;
      return input_weights(max(i, j), min(i, j), r_run, r_end, rd_w);
    };
    {                                  // s x s: sX_{t,k} = dt alpha_{k+1}, sY_{t,k} = dt gamma_{k+1} for t >= k + 2; sV_{k+1,k} = dt
      int ki = 0, kj = gl;
      while (kj > ki) { kj -= ki + 1; ++ki; }
      for (int e = gl; e < tri(T); e += G) {
        const double* mom = M.K + min(ki + 2, T);              // t0 = max(ki, kj) + 2 (the factor in front is 0 beyond T)
        const double ai = M.alp[ki], gi = M.wD[ki], aj = M.alp[kj], gj = M.wD[kj];
        double acc = ai * aj * mom[MOM_11 * ms] + (ai * gj + gi * aj) * mom[MOM_12 * ms] + gi * gj * mom[MOM_22 * ms];
        if (ki == kj) acc += M.wvs[ki + 1];
        acc *= 2.0 * dt2;
        // input weights: a = D s (a_k = s_k - s_{k-1}), so the band is D' M D, pentadiagonal
        if (ki - kj <= 2)
          acc += Mw(ki, kj, Ra, Rea, Rda) - Mw(ki + 1, kj, Ra, Rea, Rda) - Mw(ki, kj + 1, Ra, Rea, Rda) +
                 Mw(ki + 1, kj + 1, Ra, Rea, Rda);
        store(ki, kj, acc);
        kj += G;
        while (kj > ki) { kj -= ki + 1; ++ki; }
      }
    }
    for (int e = gl; e < T * T; e += G) {                      // steer (row) x s (col): sX_i = -g (B - B0), sY_i = g (K - K0)
      const int ki = e / T, kj = e - ki * T;
      const double* mom = M.K + min(max(ki + 1, kj + 2), T);
      const double bi = M.cb[ki + 1], kki = M.ck[ki + 1], aj = M.alp[kj], gj = M.wD[kj];
      const double s11 = mom[MOM_11 * ms], s12 = mom[MOM_12 * ms], s22 = mom[MOM_22 * ms];
      double acc = -aj * (mom[MOM_11_B * ms] - bi * s11) - gj * (mom[MOM_12_B * ms] - bi * s12)
                 + aj * (mom[MOM_12_K * ms] - kki * s12) + gj * (mom[MOM_22_K * ms] - kki * s22);
      acc *= 2.0 * M.wA[ki] * dt;
      store(T + ki, kj, acc);
    }
    {                                  // steer x steer, plus the yaw weight
      int ki = 0, kj = gl;
      while (kj > ki) { kj -= ki + 1; ++ki; }
      for (int e = gl; e < tri(T); e += G) {
        const double* mom = M.K + ki + 1;
        const double bi = M.cb[ki + 1], kki = M.ck[ki + 1], bj = M.cb[kj + 1], kkj = M.ck[kj + 1];
        double acc = S(mom, MOM_11, MOM_11_B, MOM_11_B, MOM_11_BB, bi, bj) - S(mom, MOM_12, MOM_12_B, MOM_12_K, MOM_12_BK, bi, kkj)
                   - S(mom, MOM_12, MOM_12_K, MOM_12_B, MOM_12_BK, kki, bj) + S(mom, MOM_22, MOM_22_K, MOM_22_K, MOM_22_KK, kki, kkj)
                   + mom[MOM_QPSI * ms];
        acc = 2.0 * M.wA[ki] * M.wA[kj] * acc + input_weights(ki, kj, Rd_, Red, Rdd);
        store(T + ki, T + kj, acc);
        kj += G;
        while (kj > ki) { kj -= ki + 1; ++ki; }
      }
    }
  }
  // linear term
  if (gl < T) {
    const int k = gl;
    const double bi = M.cb[k + 1], kki = M.ck[k + 1];
    const int ms = even_up(T + 1);
    const double* mom = M.K + min(k + 2, T);
    const double qs = dt * (M.alp[k] * mom[MOM_WX * ms] + M.wD[k] * mom[MOM_WY * ms]) + dt * M.grad[k + 1];
    double qd = 0.0;
    for (int t = k + 1; t <= T; ++t)
      qd += gk * (-(M.cb[t] - bi) * M.WeX[t] + (M.ck[t] - kki) * M.WeY[t]) + gk * M.epsi[t];
    M.q[k] = 2.0 * qs; M.q[T + k] = 2.0 * qd;
    M.u[k] = 0.0; M.u[T + k] = 0.0;
  }
  if (gl < n4 - n) { M.q[n + gl] = 0.0; M.u[n + gl] = 0.0; M.rhs[n + gl] = 0.0; M.grad[n + gl] = 0.0; }
  __threadfence();                     // the Hessian scratch is read back by TMA (async proxy) in the solver
  __syncwarp(gm);

  // feasibility predicate (SURVEY.md 8a row 8): the t = 0 speed rows act on the fixed v0
  if (!(min_speed <= v0 && v0 <= speed)) {
    if (active) {
      carry_inout(A, b, T, gl);
      // xref / target are still reported, as the reference assigns them before the solve result
      if (gl <= T) {
        double* xo = A.xref + (size_t)b * 4 * T1;
        xo[gl] = xr; xo[T1 + gl] = yr; xo[2 * T1 + gl] = vr; xo[3 * T1 + gl] = psir;
      }
      if (gl == 0) {
        A.status[b] = JMPC_INFEASIBLE; A.target_out[b] = target; if (A.iters) A.iters[b] = total_iters;
        A.cost[b] = nan("");
        write_record(A, b, nan(""), P(JMPC_P_MAX_DECEL), nan(""), JMPC_INFEASIBLE, target, total_iters, nan(""), nan(""));
      }
    }
    return JMPC_INFEASIBLE;
  }
  idx_out = idx; end_mask_out = end_mask;
  return JMPC_OPTIMAL;
}

// 1 / s of a lane's slacks, recomputed after the factorisation and after the triangular solves instead of being held
// across them: 16 registers fewer live through the solver loop's register peaks.  rcp_pos with a volatile seed, so that
// the recomputations are not merged back into one value; the same instructions on the same slacks, the same bits.
__device__ __forceinline__ double rcp_pos_again(double a) {
  double y;
  asm volatile("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  double e = fma(-a, y, 1.0);
  y = fma(y, e, y);
  e = fma(-a, y, 1.0);
  return fma(y, e, y);
}
__device__ __forceinline__ void slack_rcp(const double sh[4], const double sl[4], double ish[4], double isl[4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r) { ish[r] = rcp_pos_again(sh[r]); isl[r] = rcp_pos_again(sl[r]); }
}

// ---- phase B: Mehrotra predictor-corrector on the condensed QP -----------------------------------------------
// Returns the group's iteration count; `converged_out` says whether its KKT tolerances were met.  The groups of a
// warp iterate in lock step until all of them are done; a group that is done (or never active) keeps executing on
// its own data with its commits switched off, so the iterate it reports is the one it was done with.
template <int TT, int G, bool LAT>
__device__ __noinline__ int step_solve(const StepArgs& A, bool active, double* smem_base, const double* pscr, int gl,
                                       bool& converged_out, unsigned& tma_parity, const chol_task* lut) {
  // The groups of a warp go through this whole phase in lock step (uniform control flow, see above), so its
  // shuffles and synchronisations name the whole warp: a mask held in a register costs a MATCH / REDUX / VOTE
  // sequence in front of every group of shuffles (3.5 % of the half-warp kernel's instructions); the shuffles' width
  // (G) keeps the groups' data apart.  Phases A and C have group-uniform early exits and keep the group masks.
  constexpr unsigned gm = kFull;
  const int T = (TT > 0) ? TT : A.T;
  const int n = 2 * T, nb = nblk(n);
  WarpMem M(smem_base, T);
  auto P = [&](int k) -> double { return M.prm[k]; };
  // ---------------- 5. interior-point solve -------------------------------------------------------
  // Stage k = lane owns four two-sided rows: r = 0 acceleration box (on s_k - s_{k-1}), 1 steer box, 2 steer rate
  // k -> k+1, 3 speed (a box on s_k, the running sum of a up to k).  Only slacks and multipliers stay in registers across the factorisation;
  // bounds are rebuilt from the parameter block when needed.
  // Dead rows (lanes beyond the horizon; the rate row of the last stage) keep lambda = 0 and ds = dl = 0 exactly for
  // the whole solve, so every product with their multipliers vanishes by itself: only the quantities that would
  // otherwise be non-zero on them (row residuals, the rate / running-sum rows of A du, the centring term) are
  // switched off explicitly.
  double sh[4], sl[4], lh[4], ll[4];
  const bool live013 = gl < T, live2 = gl < T - 1;
  auto is_live = [&](int r) -> bool { return r == 2 ? live2 : live013; };
  auto bound_hi = [&](int r) -> double {
    return r == 0 ? P(JMPC_P_MAX_ACCEL) : r == 1 ? P(JMPC_P_MAX_STEER) : r == 2 ? P(kSlotLim) : P(kSlotHi3);
  };
  auto bound_lo = [&](int r) -> double {
    return r == 0 ? P(JMPC_P_MAX_DECEL) : r == 1 ? -P(JMPC_P_MAX_STEER) : r == 2 ? -P(kSlotLim) : P(kSlotLo3);
  };
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    sh[r] = fmax(bound_hi(r), 1e-2); sl[r] = fmax(-bound_lo(r), 1e-2);      // u = 0 -> A u = 0
    if (A.init_mu > 0.0) { lh[r] = is_live(r) ? A.init_mu / sh[r] : 0.0; ll[r] = is_live(r) ? A.init_mu / sl[r] : 0.0; }
    else { lh[r] = is_live(r) ? 1.0 : 0.0; ll[r] = lh[r]; }
  }
  const double inv_rows = 1.0 / (double)(2 * (4 * T - 1));
  {
    double gscale = 0.0;
    if (gl < T) gscale = fmax(fabs(M.q[gl]), fabs(M.q[T + gl]));
    gscale = 1.0 + grp_max<G>(gscale, gm);
    if (gl == 0) M.prm[kSlotGscale] = gscale;    // read back by the exit tests (not held in a register across the loop)
  }
  const int ntd = tiles_doubles(n);
  bool converged = false;
  bool acceptable = false;          // last evaluated iterate meets the reduced tolerances (see below)
  // kLock: several groups share the warp and iterate in lock step.  A whole-warp instance (G = 32) leaves the loop the
  // moment it is done, so `done` never guards anything there and the compiler sees the single-instance loop.
  constexpr bool kLock = (G != 32);
  bool done = kLock ? !active : false;      // this group's solve is over (its state is frozen from then on)
  int my_iters = 0;
#ifdef JMPC_DEBUG_RESID
  double dbg_mu = 0, dbg_rp = 0, dbg_rd = 0;
#endif
  int it = 0;
  // P -> shared with one TMA bulk copy per iteration (the scratch copy is L2 resident).  The copy for iteration
  // it + 1 is issued as soon as the corrector's triangular solves have read the factor for the last time, so it
  // runs under the direction recovery, the step and the next iteration's row work.  Every exit of the loop lies
  // behind the wait for the copy in flight (and none is issued for an iteration that will not run), so the
  // barrier's phase stays in step and nothing lands in K after the solver has left.  The last reads of K are
  // behind a group __syncwarp; the fence inside tma_load_1d orders them (generic proxy) before the copy (async proxy).
  if (gl == 0 && A.max_iters > 0) tma_load_1d(M.K, pscr, (unsigned)(ntd * sizeof(double)), M.mbar);
  for (it = 0; it < A.max_iters; ++it) {
    JMPC_TICK(ts_);
    // The primal row residuals rph / rpl are needed again in both direction phases.  They are parked in shared memory
    // (the rhs / grad / prefix-sum arrays are dead during the solve) instead of being held across the factorisation
    // and the triangular solves: with them in registers the compiler spilled 0.5 KB per thread to local memory,
    // which misses the small L1 left beside 222 KB of shared memory and waits on L2.
    double* stash = M.grad;                         // [8][T]: rph[0..3], rpl[0..3] of stage = lane
    double z[4], t4[4];
    rows_apply<G>(M.u, T, gl, gm, z);
    double mu = 0.0, rpmax = 0.0;                   // rpmax: this lane's largest primal row residual
    double w2, w3;
    {
      double w[4], ish[4], isl[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const bool lv = is_live(r);
        ish[r] = rcp_pos(sh[r]); isl[r] = rcp_pos(sl[r]);
        const double rph_r = lv ? (z[r] + sh[r] - bound_hi(r)) : 0.0;
        const double rpl_r = lv ? (-z[r] + sl[r] + bound_lo(r)) : 0.0;
        if (gl < T) { stash[r * T + gl] = rph_r; stash[(4 + r) * T + gl] = rpl_r; }
        // predictor (affine) complementarity target rc = lambda s:  (lambda rp - rc) / s = lambda (rp - s) / s
        t4[r] = fma(lh[r], rph_r, -lh[r] * sh[r]) * ish[r] - fma(ll[r], rpl_r, -ll[r] * sl[r]) * isl[r];
        w[r] = fma(lh[r], ish[r], ll[r] * isl[r]);
        mu += lh[r] * sh[r] + ll[r] * sl[r];
        rpmax = dmax(rpmax, dmax(fabs(rph_r), fabs(rpl_r)));
      }
      w2 = w[2]; w3 = w[3];
      double wup = __shfl_up_sync(gm, w2, 1, G);
      if (gl == 0) wup = 0.0;
      const double w0n = __shfl_down_sync(gm, w[0], 1, G);          // acceleration row of the next stage (0 behind the horizon)
      // A' W A is tridiagonal in both blocks: the diagonal terms (wA: s block, wD: steering block) and the
      // sub-diagonal ones (wS: -w0_k at (k, k-1); wR: -w2_{k-1} at (T+k, T+k-1))
      if (gl < T) { M.wA[gl] = w[0] + w0n + w3; M.wS[gl] = w[0]; M.wD[gl] = w[1] + w2 + wup; M.wR[gl] = w2; }
    }
    mu = grp_sum<G>(mu, gm) * inv_rows;
    double ra_p, rd_p;                              // A' (predictor row terms)
    rows_apply_T<G>(t4, gl, gm, ra_p, rd_p);
    // P u is formed from the clean Hessian: folding the barrier weights in first and subtracting them again
    // would cancel catastrophically once w ~ 1e12
    JMPC_TOCK(ts_, 0);
    mbar_wait(M.mbar, tma_parity);
    tma_parity ^= 1u;
    __syncwarp(gm);
    JMPC_TOCK(ts_, 1);
    double pu0, pu1;                              // rows gl and T + gl of P u
    symv_rows<(TT > 0) ? ((2 * TT + 3) >> 2) : 0>(M.K, M.u, T, nb, gl, pu0, pu1);
#pragma unroll
    for (int r = 0; r < 4; ++r) t4[r] = lh[r] - ll[r];
    double ra, rd;
    rows_apply_T<G>(t4, gl, gm, ra, rd);
    // gradient of the Lagrangian (dual residual), kept in registers: g0 for s_gl, g1 for delta_gl
    const double g0 = (gl < T) ? pu0 + M.q[gl] + ra : 0.0, g1 = (gl < T) ? pu1 + M.q[T + gl] + rd : 0.0;
    __syncwarp(gm);                               // every lane is done reading P before K is assembled in place
    JMPC_TOCK(ts_, 2);
    // K = P + A' diag(w) A: a tridiagonal in each block (only the lower triangle is read by the factorisation)
    if (gl < T) {
      const int i = T + gl;
      M.K[elem_off(gl, gl)] += M.wA[gl];
      M.K[elem_off(i, i)] += M.wD[gl];
      if (gl >= 1) { M.K[elem_off(gl, gl - 1)] -= M.wS[gl]; M.K[elem_off(i, i - 1)] -= M.wR[gl - 1]; }
    }
    // The exit tests only compare the largest primal / dual residual of the group with three thresholds each, so the
    // lanes compare their own maxima and vote (six votes) instead of reducing two maxima over the group (ten
    // 64-bit shuffle steps with their compares and selects).
    const double rdmax_l = dmax(fabs(g0), fabs(g1));
    const bool rp_strict = grp_all<G>(rpmax <= A.tol_res), rp_red = grp_all<G>(rpmax <= 1e-7), rp_brk = grp_all<G>(rpmax <= 1e-9);
    const double gscale = M.prm[kSlotGscale];
    const bool rd_strict = grp_all<G>(rdmax_l <= A.tol_res * gscale), rd_red = grp_all<G>(rdmax_l <= 1e-7 * gscale);
    const bool rd_brk = grp_all<G>(rdmax_l <= 1e-9 * gscale);
#ifdef JMPC_DEBUG_RESID
    const double rpmax_g = grp_max<G>(rpmax, gm), rdmax = grp_max<G>(rdmax_l, gm);
#endif
    __syncwarp(gm);
    if (!kLock || !done) {
      if (mu <= A.mu_tol && rp_strict && rd_strict) { converged = true; done = true; }
      // Complementarity three orders below its target with the primal rows satisfied: the iterate has converged;
      // what is left in the dual residual is multiplier noise on the active rows (w ~ 1e16 by now, their slacks are
      // at roundoff), which lies in the span of the active normals and does not move u.  Iterating further only
      // amplifies it.  Measured on 200k instances: controls at such exits are within 1e-8 of the oracle.
      else if (mu <= 1e-3 * A.mu_tol && rp_strict) { converged = true; done = true; }
      // Reduced tolerances, the analogue of the OPTIMAL_INACCURATE status the reference accepts (mpc.py:199): used
      // when the factorisation breaks down numerically a step or two before the strict target (w ~ 1e13 by then),
      // or the iteration cap is hit.  Measured: such iterates are still 5-6x inside the control tolerance.
      else acceptable = (mu <= 1e-9 && rp_red && rd_red);
      if (kLock && done) my_iters = it;
#ifdef JMPC_DEBUG_RESID
      dbg_mu = mu; dbg_rp = rpmax_g; dbg_rd = rdmax / gscale;
#endif
    }
    if (kLock ? __all_sync(kFull, done) : done) break;

    JMPC_TOCK(ts_, 3);
    // The predictor's right-hand side needs nothing from the factor, so its forward substitution rides along with
    // the factorisation (one triangular sweep out of four per iteration saved).
    if (gl < T) { M.rhs[gl] = -g0 - ra_p; M.rhs[T + gl] = -g1 - rd_p; }
    __syncwarp(gm);
    const bool clean = chol_tiles<G>(M.K, nb, gl, gm, lut, M.rhs);     // non-positive pivots are replaced, never fatal
    JMPC_TOCK(ts_, 4);
    // Numerical breakdown of the factorisation (a pivot lost to roundoff, w ~ 1e13 by then) on an iterate that is
    // already two orders inside the reduced tolerances: stop here.  The step computed from the patched factor is
    // usually harmless, but on a few instances in 10^5 (weakly active speed rows, T = 25) it threw the iterate far
    // enough out that the iteration cap was reached; which instances depended on the build.
    if ((!kLock || !done) && !clean && mu <= 1e-11 && rp_brk && rd_brk) {
      acceptable = true; done = true;
      if (kLock) my_iters = it;
    }
    if (!kLock && done) break;

    // dlh / dll enter each phase's direction recovery holding the complementarity targets rc: l s for the predictor, l s
    // + ds_aff dl_aff - sigma mu for the corrector (formed at the end of the predictor, so that only rc and not the four
    // affine directions live into the corrector)
    double dsh[4], dsl[4], dlh[4], dll[4];
    double aff_step = 0.0;
#pragma unroll 1
    for (int phase = 0; phase < 2; ++phase) {
      double sw_lo = 0.0, sw_hi = 0.0;
      (void)sw_lo; (void)sw_hi;
      // the primal row residual k (rph[0..3], rpl[0..3]), read from the stash where it is used
      auto rp = [&](int k) -> double { return (gl < T) ? stash[k * T + gl] : 0.0; };
      if (phase == 1) {
        double th[4], ish[4], isl[4];
        slack_rcp(sh, sl, ish, isl);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          // th = a_h - a_l with a_l rounded and a_h's product fused into the difference, written out: left to the
          // compiler, which of the two products it fuses changes with the surrounding code, and so would the iterates
          const double a_l = __dmul_rn(fma(ll[r], rp(4 + r), -dll[r]), isl[r]);
          th[r] = fma(fma(lh[r], rp(r), -dlh[r]), ish[r], -a_l);
        }
        rows_apply_T<G>(th, gl, gm, ra, rd);
        if (gl < T) { M.rhs[gl] = -g0 - ra; M.rhs[T + gl] = -g1 - rd; }
        __syncwarp(gm);
        JMPC_TOCK(ts_, 5);
        if constexpr (LAT) {
          sweep_load<G>(M.rhs, nb << 2, gl, sw_lo, sw_hi);
          solve_forward_regs<G>(M.K, nb, gl, gm, sw_lo, sw_hi);
        } else {
          solve_forward_tiles<G>(M.K, M.rhs, nb, gl, gm);
        }
      } else {
        if constexpr (LAT) sweep_load<G>(M.rhs, nb << 2, gl, sw_lo, sw_hi);   // the forward substitution rode along with the factorisation
#pragma unroll
        for (int r = 0; r < 4; ++r) { dlh[r] = lh[r] * sh[r]; dll[r] = ll[r] * sl[r]; }
        JMPC_TOCK(ts_, 5);
      }
      if constexpr (LAT) {
        // low-latency kernels: the sweeps keep the vector in registers in a cyclic layout (lane -> entries gl, gl + G);
        // the stage rows want entries gl and T + gl, so it takes one trip through shared memory
        solve_backward_regs<G>(M.K, nb, gl, gm, sw_lo, sw_hi);
        __syncwarp(gm);
        sweep_store<G>(M.rhs, nb << 2, gl, sw_lo, sw_hi);
      } else {
        solve_backward_tiles<G>(M.K, M.rhs, nb, gl, gm);
      }
      __syncwarp(gm);
      if (phase == 1 && gl == 0 && it + 1 < A.max_iters) tma_load_1d(M.K, pscr, (unsigned)(ntd * sizeof(double)), M.mbar);
      const double du0 = (gl < T) ? M.rhs[gl] : 0.0, du1 = (gl < T) ? M.rhs[T + gl] : 0.0;
      JMPC_TOCK(ts_, 6);
      double dz[4];
      rows_apply_reg<G>(du0, du1, gl, gm, live013, live2, dz);
      // largest step keeping s, lambda > 0: alpha_max = 1 / max(-ds/s, -dl/l).  The slacks' reciprocals are at hand
      // (ish, isl), so their ratios are one multiplication each; the multipliers' ratios are tracked as a
      // (numerator, denominator) pair compared by cross-multiplication and turned into a ratio once per lane (no
      // fp64 division anywhere: ~20 instructions each).  Dead rows carry zero directions and never bind.
      double rho = 0.0, wn = 0.0, wd = 1.0, ish[4], isl[4];
      slack_rcp(sh, sl, ish, isl);
      auto cand = [&](double num, double den) { if (num * wd > wn * den) { wn = num; wd = den; } };
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const double rch = dlh[r], rcl = dll[r];
        dsh[r] = -rp(r) - dz[r];
        dsl[r] = -rp(4 + r) + dz[r];
        dlh[r] = -(fma(lh[r], dsh[r], rch)) * ish[r];
        dll[r] = -(fma(ll[r], dsl[r], rcl)) * isl[r];
        rho = dmax(rho, dmax(-dsh[r] * ish[r], -dsl[r] * isl[r]));
        cand(-dlh[r], lh[r]); cand(-dll[r], ll[r]);
      }
      rho = dmax(rho, wn * rcp_pos(wd));
      rho = grp_max<G>(rho, gm);
      // only amax < 1 / 0.99 matters below (the step is capped at 1)
      const double amax = (rho > 0.5) ? rcp_pos(rho) : 2.0;
      if (phase == 0) {
        const double aa = fmin(1.0, amax);
        aff_step = aa;
        double mu_aff = 0.0;
#pragma unroll
        for (int r = 0; r < 4; ++r)
          mu_aff += fma(aa, dlh[r], lh[r]) * fma(aa, dsh[r], sh[r]) + fma(aa, dll[r], ll[r]) * fma(aa, dsl[r], sl[r]);
        mu_aff = grp_sum<G>(mu_aff, gm) * inv_rows;
        const double ratio = mu_aff * rcp_pos(mu);
        const double sigma_mu = ratio * ratio * ratio * mu;
        const double sm013 = live013 ? sigma_mu : 0.0, sm2 = live2 ? sigma_mu : 0.0;
#pragma unroll
        for (int r = 0; r < 4; ++r) {                // the corrector's rc
          const double sm = (r == 2) ? sm2 : sm013;
          dlh[r] = fma(lh[r], sh[r], dsh[r] * dlh[r] - sm); dll[r] = fma(ll[r], sl[r], dsl[r] * dll[r] - sm);
        }
      } else if (!kLock || !done) {
        // Fraction to the boundary tied to the length aa of the affine (predictor) step: a long predictor step
        // means the iterate is well centred and the corrector may go almost to the boundary (0.9999); a short
        // one keeps the classical 0.99.  Saves ~13 % of the iterations; a rule driven by mu alone (1 - mu) made
        // a few instances in 10^4 oscillate between a tiny predictor step and a pure centring step.
        const double alpha = fmin(1.0, fmin(0.9999, fmax(0.99, 1.0 - 0.1 * (1.0 - aff_step) * (1.0 - aff_step))) * amax);
        if (gl < T) { M.u[gl] = fma(alpha, du0, M.u[gl]); M.u[T + gl] = fma(alpha, du1, M.u[T + gl]); }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          sh[r] = fma(alpha, dsh[r], sh[r]); sl[r] = fma(alpha, dsl[r], sl[r]);
          lh[r] = fma(alpha, dlh[r], lh[r]); ll[r] = fma(alpha, dll[r], ll[r]);
        }
      }
      __syncwarp(gm);
      JMPC_TOCK(ts_, 7);
    }
  }
  if (!kLock || !done) my_iters = it;
#ifdef JMPC_DEBUG_RESID
  if (gl == 0) { M.prm[29] = dbg_mu; M.prm[30] = dbg_rp; M.prm[31] = dbg_rd; }
  __syncwarp(gm);
#endif
  converged_out = converged || acceptable;
  return my_iters;
}

// ---- phase C: states of the linearised model for the solution, objective, outputs ---------------------------
// Returns true when the group's results have been written (last linearisation pass, DU_TH exit, or failed solve).
template <int TT, int G>
__device__ __noinline__ bool step_output(const StepArgs& A, int b, bool active, double* smem_base, int gl, unsigned gm,
                                         bool last, bool solved, int target, int idx, unsigned end_mask,
                                         int total_iters, double& oa_k, double& od_k, double& ov_k) {
  const int T = (TT > 0) ? TT : A.T;
  const int T1 = T + 1;
  WarpMem M(smem_base, T);
  auto P = [&](int k) -> double { return M.prm[k]; };
  const double x0 = A.state[(size_t)b * 4 + 0], y0 = A.state[(size_t)b * 4 + 1];
  const double v0 = A.state[(size_t)b * 4 + 2], yaw0 = A.state[(size_t)b * 4 + 3];
  const double dt = P(JMPC_P_DT), Lw = P(JMPC_P_L);
  // per-lane data of phase A, re-read or recomputed instead of being held in registers across the solve
  const int cid = A.course_id ? min(max(A.course_id[b], 0), A.n_courses - 1) : 0;
  double xr = 0.0, yr = 0.0, psir = 0.0, vr = 0.0, vb = 0.0, th = 0.0;
  if (gl <= T) {
    const size_t off = (size_t)cid * A.course_stride + idx;
    xr = A.cx[off]; yr = A.cy[off]; psir = A.cyaw[off];
    vr = ref_speed(A, M.prm, cid, idx);
    vb = M.vb[gl]; th = M.th[gl];
  }
  if (!solved) {
    // The solver hit its iteration cap without meeting even the reduced tolerances: a failed solve, as when the
    // reference's solver status is neither OPTIMAL nor OPTIMAL_INACCURATE (mpc.py:199-209): no controls are
    // reported (the in-out arrays keep their values), xref / target are, and the record brakes with MAX_DECEL.
    if (active) {
      carry_inout(A, b, T, gl);
      if (gl <= T) {
        double* xo = A.xref + (size_t)b * 4 * T1;
        xo[gl] = xr; xo[T1 + gl] = yr; xo[2 * T1 + gl] = vr; xo[3 * T1 + gl] = psir;
      }
      if (gl == 0) {
        A.status[b] = JMPC_MAX_ITER; A.target_out[b] = target; if (A.iters) A.iters[b] = total_iters;
        if (A.work_hint) A.work_hint[b] = total_iters;
        A.cost[b] = nan("");
        write_record(A, b, nan(""), P(JMPC_P_MAX_DECEL), nan(""), JMPC_MAX_ITER, target, total_iters, nan(""), nan(""));
      }
    }
    return true;
  }
  double sn, cs;
  sincos(th, &sn, &cs);
  double al = 0.0, be = 0.0, ga = 0.0, ka = 0.0, gk = 0.0;
  if (gl < T) { al = dt * cs; be = dt * vb * sn; ga = dt * sn; ka = dt * vb * cs; gk = dt * vb / Lw; }
  // ---------------- 6. states of the linearised model for the solution ---------------------------
  // the solver's unknowns are the cumulative accelerations s_k: a_k = s_k - s_{k-1}, v_t = v0 + dt s_{t-1}
  const double s_sol = (gl < T) ? M.u[gl] : 0.0, d_sol = (gl < T) ? M.u[T + gl] : 0.0;
  double s_prev = __shfl_up_sync(gm, s_sol, 1, G);
  if (gl == 0) s_prev = 0.0;
  const double a_sol = (gl < T) ? s_sol - s_prev : 0.0;
  const double v_t = v0 + dt * s_prev;                                                // lane t: v_t
  const double gd = gk * d_sol;
  const double psi_t = yaw0 + (grp_scan<G>(gd, gl, gm) - gd);
  const double tx = (gl < T) ? (al * v_t - be * (psi_t - th)) : 0.0;
  const double ty = (gl < T) ? (ga * v_t + ka * (psi_t - th)) : 0.0;
  const double X_t = x0 + (grp_scan<G>(tx, gl, gm) - tx);
  const double Y_t = y0 + (grp_scan<G>(ty, gl, gm) - ty);

  if (!last && A.du_th > 0.0) {
    // the exit the reference left commented out (mpc.py:236-240): du = sum|oa - poa| + sum|od - pod| <= DU_TH
    const double du = grp_sum<G>((gl < T) ? fabs(a_sol - oa_k) + fabs(d_sol - od_k) : 0.0, gm);
    last = du <= A.du_th;
  }
  if (!last) {
    // feed the solution back as the next linearisation point (mpc.py:231-236)
    oa_k = a_sol; od_k = d_sol; ov_k = v_t;
    return false;
  }
  // objective value, evaluated term by term as mpc.py:159-187 writes it
  const double Ra = P(JMPC_P_R_A), Rd_ = P(JMPC_P_R_D), Rda = P(JMPC_P_RD_A), Rdd = P(JMPC_P_RD_D);
  const double Rea = P(JMPC_P_REND_A), Red = P(JMPC_P_REND_D);
  double cterm = 0.0;
  if (gl >= 1 && gl <= T) {
    double w11, w12 = 0.0, w22, wv, wpsi;             // stage weights, recomputed as in step_prep
    if ((end_mask >> gl) & 1u) {
      w11 = P(JMPC_P_QF_X); w22 = P(JMPC_P_QF_Y); wv = P(JMPC_P_QF_V); wpsi = P(JMPC_P_QF_YAW);
    } else {
      double s1, c1, s2, c2;
      sincos(psir + 0.5 * M_PI, &s1, &c1);
      sincos(psir, &s2, &c2);
      const double wp = P(JMPC_P_W_PERP), wl = P(JMPC_P_W_PARA);
      w11 = (c1 * c1) * wp + (c2 * c2) * wl;
      w12 = (c1 * s1) * wp + (c2 * s2) * wl;
      w22 = (s1 * s1) * wp + (s2 * s2) * wl;
      wv = P(JMPC_P_Q_V); wpsi = P(JMPC_P_Q_YAW);
    }
    const double dx = xr - X_t, dy = yr - Y_t, dv = vr - v_t, dp = psir - psi_t;
    cterm = dx * (w11 * dx + w12 * dy) + dy * (w12 * dx + w22 * dy) + wv * dv * dv + wpsi * dp * dp;
  }
  if (gl < T) {
    const bool e_t = (end_mask >> gl) & 1u;
    cterm += (e_t ? Rea : Ra) * a_sol * a_sol + (e_t ? Red : Rd_) * d_sol * d_sol;
  }
  const double a_next = __shfl_down_sync(gm, a_sol, 1, G), d_next = __shfl_down_sync(gm, d_sol, 1, G);
  if (gl < T - 1) cterm += Rda * (a_next - a_sol) * (a_next - a_sol) + Rdd * (d_next - d_sol) * (d_next - d_sol);
  const double cost = grp_sum<G>(cterm, gm);
  const double v1 = __shfl_sync(gm, v_t, 1, G), yaw1 = __shfl_sync(gm, psi_t, 1, G);
  if (active) {
    if (gl < T) { A.oa_out[(size_t)b * T + gl] = a_sol; A.od_out[(size_t)b * T + gl] = d_sol; }
    if (gl <= T) {
      A.ox[(size_t)b * T1 + gl] = X_t; A.oy[(size_t)b * T1 + gl] = Y_t;
      A.ov[(size_t)b * T1 + gl] = v_t; A.oyaw[(size_t)b * T1 + gl] = psi_t;
      double* xo = A.xref + (size_t)b * 4 * T1;
      xo[gl] = xr; xo[T1 + gl] = yr; xo[2 * T1 + gl] = vr; xo[3 * T1 + gl] = psir;
    }
    if (gl == 0) {
      A.cost[b] = cost; A.status[b] = JMPC_OPTIMAL; A.target_out[b] = target;
      if (A.iters) A.iters[b] = total_iters;
      if (A.work_hint) A.work_hint[b] = total_iters;
#ifdef JMPC_DEBUG_RESID
      write_record(A, b, M.prm[29], a_sol, cost, JMPC_OPTIMAL, target, total_iters, M.prm[30], M.prm[31]);
#else
      write_record(A, b, d_sol, a_sol, cost, JMPC_OPTIMAL, target, total_iters, v1, yaw1);
#endif
    }
  }
  return true;
}

// The fused step for the instances of one warp (one per lane group).  TT > 0 fixes the horizon at compile time
// (every shared-memory offset and tile count becomes an immediate); TT == 0 is the generic runtime-T version.  The
// three phases are separate functions so that the solver's register allocation is not burdened by the values the
// preparation and the epilogue need; they communicate through the group's shared memory.
template <int TT, int G, bool LAT>
__device__ __forceinline__ void mpc_step_instance(const StepArgs& A, int b, bool active, double* smem_base, double* pscr,
                                                  int gl, unsigned gm, unsigned& tma_parity, const chol_task* lut) {
  const int T = (TT > 0) ? TT : A.T;
  WarpMem M(smem_base, T);
  // the instance's parameter vector lives in shared memory (uniform reads, no registers held across phases)
  for (int k = gl; k < JMPC_NPARAM; k += G) M.prm[k] = A.params ? A.params[(size_t)b * JMPC_NPARAM + k] : A.defaults[k];
  __syncwarp(gm);
  // warm start = linearisation point (mpc.py:225-227: None -> zeros)
  const bool use_warm = A.warm ? (A.warm[b] != 0) : true;
  double oa_k = 0.0, od_k = 0.0, ov_k = 0.0;       // ov: |ov| feedback for lin_iters > 1 (lane k <-> horizon point k)
  if (use_warm && gl < T) { oa_k = A.oa[(size_t)b * T + gl]; od_k = A.od[(size_t)b * T + gl]; }
  int target = A.target_ind[b];
  int total_iters = 0;
  for (int lin = 0; lin < A.lin_iters; ++lin) {
    int idx = 0; unsigned end_mask = 0;
    JMPC_TICK(ti_);
    const int st = step_prep<TT, G>(A, b, active, smem_base, pscr, gl, gm, lin, total_iters, oa_k, od_k, ov_k, target,
                                    idx, end_mask);
    if (st != JMPC_OPTIMAL) active = false;        // reported by step_prep; the group idles through the rest
    if (G == 32 ? !active : !__any_sync(kFull, active)) return;
    JMPC_TOCK(ti_, 10);
    bool converged = false;
    total_iters += step_solve<TT, G, LAT>(A, active, smem_base, pscr, gl, converged, tma_parity, lut);
    JMPC_TOCK(ti_, 11);
    const bool finished = step_output<TT, G>(A, b, active, smem_base, gl, gm, lin == A.lin_iters - 1, converged, target,
                                             idx, end_mask, total_iters, oa_k, od_k, ov_k);
    if (finished) active = false;
    JMPC_TOCK(ti_, 12);
    __syncwarp(gm);
    if (G == 32 ? !active : !__any_sync(kFull, active)) return;
  }
}

// ---- scheduling: longest instances first ------------------------------------------------------------------------
// A batch of one to a few waves of instances (4096 instances on 2368 resident warps) finishes when its slowest
// late-started instance does: interior-point iteration counts spread from 6 to 23 around a mean of 10, and an
// instance that needs 23 iterations and is only picked up when the first wave retires decides the kernel time
// (measured on config 2: 1.27 ms in index order, 0.90 ms longest-first).  The queue therefore hands instances out
// by descending key: the iteration count of the same instance in the previous step when the caller runs a closed
// loop (work_hint; the active set, and with it the iteration count, changes slowly from step to step), otherwise
// an a-priori key: the number of horizon stages on which the speed cap can bind at full throttle (v0 close to the
// cap => many active, nearly degenerate speed rows) plus the stages on which the acceleration box binds while a slow
// ego catches up with the reference points (correlation 0.56 with the iteration count on config 2).
constexpr int kSchedKeys = 64;
constexpr int kSchedThreads = 1024;
__device__ __forceinline__ int schedule_key(int b, int T, const int* __restrict__ hint, const double* __restrict__ state,
                                            const double* __restrict__ params, const ParamVec& defaults, double acc_weight) {
  int key;
  if (hint) {
    key = hint[b];
  } else {
    const double* pv = params ? params + (size_t)b * JMPC_NPARAM : defaults.v;
    const double v0 = state[(size_t)b * 4 + 2];
    const double dv_stage = fmax(pv[JMPC_P_MAX_ACCEL] * pv[JMPC_P_DT], 1e-9);        // speed gained per stage at full throttle
    // stages on which the speed cap can bind
    const double cap_stages = fmin(fmax((double)T - (pv[JMPC_P_SPEED] - v0) / dv_stage, 0.0), (double)T);
    // stages at full throttle to reach the speed the reference points advance with (mpc.py:98: max(v, 10/3.6)); the
    // acceleration box binds on those and, to close the gap opened meanwhile, on about as many again
    const double acc_stages = fmin(fmax((pv[JMPC_P_V_REF_MIN] - v0) / dv_stage, 0.0), (double)T);
    key = (int)(2.0 * (cap_stages + acc_weight * acc_stages));
  }
  return min(max(key, 0), kSchedKeys - 1);
}
// Counting sort on 64 key values in two launches over any number of blocks (a block owns a contiguous chunk of the
// batch): (1) keys and the global histogram, (2) every block reserves, per key, a range of the output for its chunk
// with one global atomic and scatters into it.  The order inside a key class is not deterministic (it only affects
// timing, never results).  work: [0, 64) histogram, [64, 128) per-key cursors, both zeroed before the first launch.
__global__ void __launch_bounds__(kSchedThreads) schedule_count_kernel(int B, int T, const int* __restrict__ hint,
                                                                       const double* __restrict__ state,
                                                                       const double* __restrict__ params, ParamVec defaults,
                                                                       double acc_weight, unsigned char* __restrict__ keys,
                                                                       int* __restrict__ work) {
  __shared__ int count[kSchedKeys];
  for (int k = threadIdx.x; k < kSchedKeys; k += blockDim.x) count[k] = 0;
  __syncthreads();
  const int chunk = (B + gridDim.x - 1) / gridDim.x, lo = blockIdx.x * chunk, hi = min(B, lo + chunk);
  for (int b = lo + threadIdx.x; b < hi; b += blockDim.x) {
    const int key = schedule_key(b, T, hint, state, params, defaults, acc_weight);
    keys[b] = (unsigned char)key;
    atomicAdd(&count[key], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < kSchedKeys; k += blockDim.x) if (count[k]) atomicAdd(&work[k], count[k]);
}
__global__ void __launch_bounds__(kSchedThreads) schedule_place_kernel(int B, const unsigned char* __restrict__ keys,
                                                                       int* __restrict__ work, int* __restrict__ order) {
  __shared__ int count[kSchedKeys];
  __shared__ int base[kSchedKeys];
  for (int k = threadIdx.x; k < kSchedKeys; k += blockDim.x) count[k] = 0;
  __syncthreads();
  const int chunk = (B + gridDim.x - 1) / gridDim.x, lo = blockIdx.x * chunk, hi = min(B, lo + chunk);
  for (int b = lo + threadIdx.x; b < hi; b += blockDim.x) atomicAdd(&count[keys[b]], 1);
  __syncthreads();
  if (threadIdx.x < kSchedKeys) {
    const int k = threadIdx.x;
    int start = 0;                                     // descending keys: everything with a larger key comes first
    for (int q = k + 1; q < kSchedKeys; ++q) start += work[q];
    base[k] = start + (count[k] ? atomicAdd(&work[kSchedKeys + k], count[k]) : 0);
  }
  __syncthreads();
  for (int b = lo + threadIdx.x; b < hi; b += blockDim.x) order[atomicAdd(&base[keys[b]], 1)] = b;
}

// Persistent kernel: every resident warp pulls instances (one per lane group) from a global counter.
#ifndef JMPC_MINBLOCKS
#define JMPC_MINBLOCKS 4
#endif
#ifndef JMPC_WPB
#define JMPC_WPB 4                 // warps per block; JMPC_WPB x JMPC_MINBLOCKS resident warps per SM set the register budget
#endif
// resident blocks per SM the register budget is set for: short horizons leave shared memory for more warps, and at
// T = 8 the extra warps pay for the tighter register budget (80 registers, 24 warps: +5 %; at T = 13 / 20 they do
// not).  At T = 25 shared memory (18.4 KB per instance) admits only three blocks of four warps anyway, so the kernel
// is compiled for three: 168 registers instead of 128 (measured: 16.8 -> 15.5 ms on 65 536 instances).
#ifndef JMPC_T8_BLOCKS
#define JMPC_T8_BLOCKS ((JMPC_MINBLOCKS * 3) / 2)
#endif
// At T = 13 three blocks (168 registers, no spills, 24 resident instances) have overtaken four (128 registers, 32
// instances) since the solver loop lost a third of its instructions: +2 % (profiles/r2_ab_variants.txt, session mb3);
// at T = 20 the two are equal and four stay.
constexpr int step_min_blocks(int TT) {
  return TT == 8 ? JMPC_T8_BLOCKS : ((TT == 25 || TT == 13) && JMPC_MINBLOCKS > 3) ? 3 : JMPC_MINBLOCKS;
}
// LAT selects the low-latency solve phase (triangular sweeps with the vector in registers, jmpc_linalg.cuh): for
// launches that leave the SMs nearly empty -- a single ego's step -- where one warp's dependency chains are the whole
// kernel time.  Same results bit for bit.
// The low-latency kernels are launched with one warp per block and no occupancy target, so they get the full 255
// registers (no spills: the 128-register budget of the throughput kernels costs a warp that runs alone ~20 %).
template <int TT, int G, bool LAT = false>
__global__ void __launch_bounds__(LAT ? 32 : 32 * JMPC_WPB, LAT ? 1 : step_min_blocks(TT)) mpc_step_kernel(
    const __grid_constant__ StepArgs A) {
  extern __shared__ __align__(16) double smem[];
  constexpr int NG = 32 / G;                       // instances per warp
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int gl = lane & (G - 1), sub = lane / G;
  const unsigned gm = group_mask<G>(lane);
  const int warps_per_block = blockDim.x >> 5;
  const int T = (TT > 0) ? TT : A.T;
  double* base = smem + (size_t)(wib * NG + sub) * inst_smem_doubles(T);
  const int gg = (blockIdx.x * warps_per_block + wib) * NG + sub;      // resident-group index
  const int n = 2 * T;
  double* pscr = A.pscratch + (size_t)gg * tiles_doubles(n);
  unsigned tma_parity = 0;
  {
    WarpMem M0(base, T);
    if (gl == 0) mbar_init(M0.mbar, 1);
    __syncwarp();
  }
  // block-shared task table of the Cholesky trailing update, behind the instances' regions
  chol_task* lut = reinterpret_cast<chol_task*>(smem + (size_t)warps_per_block * NG * inst_smem_doubles(T));
  chol_lut_build(lut, nblk(n), threadIdx.x, blockDim.x);
  __syncthreads();
  for (;;) {
    // the warp takes NG consecutive tickets: with the longest-first order neighbours in the queue have similar
    // keys, so the instances that share a warp tend to need a similar number of iterations
    unsigned t0 = 0;
    if (lane == 0) t0 = atomicAdd(A.counter, (unsigned)NG);
    t0 = __shfl_sync(kFull, t0, 0);
    if (t0 >= (unsigned)A.B) break;
    const unsigned ticket = t0 + (unsigned)sub;
    bool active = ticket < (unsigned)A.B;
    unsigned b = active ? ticket : t0;             // a group without a ticket idles on the warp's first instance (reads only)
    if (A.order) b = (unsigned)A.order[b];
    if (A.skip && A.skip[b] != 0) active = false;
    if (!__any_sync(kFull, active)) continue;
    mpc_step_instance<TT, G, LAT>(A, (int)b, active, base, pscr, gl, gm, tma_parity, lut);
    __syncwarp();
  }
  // Fused all-gather, completion signal: the block that retires last has (through the fences and the counter) every
  // record store of this launch before it; it publishes the step number to every peer.  A reader waits for all ranks'
  // flags (gather_wait_kernel) and then owns a complete table -- no barrier kernel, no collective call.
  if (A.n_flag_peers > 0) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      const unsigned prev = atomicAdd(A.blocks_done, 1u);
      if (prev == gridDim.x - 1) {
        *A.blocks_done = 0u;
        __threadfence_system();
        for (int p = 0; p < A.n_flag_peers; ++p)
          asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(A.peer_flag[p]), "l"(A.gather_step) : "memory");
      }
    }
  }
}

// Wait until every rank of the fused all-gather has published `step` (or a later one): lane p watches rank p's slot
// of the local flag array.  Gives up after ~2 s of spinning and reports it in *timed_out instead of hanging the GPU.
__global__ void gather_wait_kernel(const unsigned long long* flags, int world, unsigned long long step, int* timed_out) {
  const int p = threadIdx.x;
  if (p >= world) return;
  unsigned long long v = 0;
  for (long long spin = 0; spin < (1ll << 24); ++spin) {
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(flags + p) : "memory");
    if (v >= step) return;
    __nanosleep(100);
  }
  atomicExch(timed_out, 1);
}

}  // namespace jmpc
