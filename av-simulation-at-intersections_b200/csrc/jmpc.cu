// jmpc.cu -- C ABI of libjmpc.so (see include/jmpc.h): handle management, launches, host staging.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <chrono>
#include <vector>

#include "../../include/jmpc.h"
#include "jmpc_collision.cuh"
#include "jmpc_step.cuh"
#include "jmpc_episode.cuh"
#include "jmpc_planner.cuh"
#include "jmpc_courses.cuh"

namespace {

thread_local std::string g_err;

int fail(const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
  else snprintf(buf, sizeof buf, "%s", what);
  g_err = buf;
  return -1;
}

#define CK(call)                                          \
  do {                                                    \
    cudaError_t e_ = (call);                              \
    if (e_ != cudaSuccess) return fail(#call, e_);        \
  } while (0)

}  // namespace

struct jmpc_handle_s {
  int device = 0;
  int max_B = 0, max_T = 0, max_N = 0, max_courses = 0;
  int sm_count = 0;
  jmpc_options opt{};
  double defaults[JMPC_NPARAM];
  // courses
  double *d_cx = nullptr, *d_cy = nullptr, *d_cyaw = nullptr;
  double* d_cv = nullptr; bool have_cv = false;                                          // reference speed profile (jmpc_set_course_speed)
  double *d_ccfx = nullptr, *d_ccfy = nullptr, *d_ccrx = nullptr, *d_ccry = nullptr;   // collision-circle tables
  double* d_arc = nullptr; long long* d_arc_off = nullptr;                                // arc-length tables (collision kernel)
  bool arc_all = false;                                                                   // every uploaded course has a table
  std::vector<int> arc_has;                                                               // per course: 1 = has a table (jmpc_get_arc_tables)
  double off_front = 2.86 / 2 + (3.5 / 2 - 1.0), off_rear = 2.86 / 2 - (3.5 / 2 - 1.0), radius = 2.0 / 1.4142135623730951;
  int* d_course_n = nullptr;
  int n_courses = 0, course_stride = 0;
  std::vector<int> course_n;
  // solver scratch
  double* d_pscratch = nullptr;
  size_t pscratch_doubles = 0;
  unsigned int* d_counter = nullptr;
  // staging for the *_host entry points
  char* d_stage = nullptr; size_t d_stage_bytes = 0;
  char* h_stage = nullptr; size_t h_stage_bytes = 0;
  cudaStream_t own_stream = nullptr;
  long long launches = 0;
  // fused all-gather targets (jmpc_set_record_peers)
  double* peer_rec[JMPC_MAX_PEERS] = {};
  int n_peers = 0;
  long long rank_offset = 0;
  unsigned long long* peer_flag[JMPC_MAX_PEERS] = {};      // jmpc_set_record_flags
  int n_flag_peers = 0;
  unsigned long long gather_step = 0;
  int* d_gather_timeout = nullptr;
  bool collision_attr_set = false, collision_planned_attr_set = false;
  bool collision_masked_attr_set[2] = {false, false};   // masked_collision_kernel<false / true>
  const int* skip = nullptr;           // jmpc_set_skip_mask
  // longest-first scheduling (jmpc_set_schedule)
  int host_transfer = 1;               // jmpc_set_host_transfer
  int schedule = 0;                     // 0 index order, 1 a-priori key, 2 previous step's iteration counts (+ 1 as fallback)
  int* d_order = nullptr; int* d_hint = nullptr; unsigned char* d_keys = nullptr; int* d_sched_work = nullptr;
  int hint_B = 0, hint_T = 0;           // batch the hints were recorded for (0 = none)
  struct HostBlock { char* base; size_t bytes; char* dev; };
  std::vector<HostBlock> host_blocks;   // page-locked blocks from jmpc_host_alloc (+ h_stage) with their device mapping
  // launch geometry of the step kernel per horizon, resolved once (function attributes, occupancy)
  struct Geom {
    bool ready = false;
    void (*kernel)(const jmpc::StepArgs) = nullptr;
    void (*kernel_lat)(const jmpc::StepArgs) = nullptr;      // low-latency variant, one warp per block
    int groups = 1, wpb = 0, per_sm = 0;
    size_t smem = 0, smem_lat = 0;
  };
  Geom geom[JMPC_MAX_T + 1];
};

namespace {

// launch geometry of the step kernel for horizon T
struct StepGeom { int blocks, threads; size_t smem; int groups_total; };

using StepKernel = void (*)(const jmpc::StepArgs);

// Horizons with a compile-time specialisation; anything else runs a generic kernel.  Horizons up to 15 (T + 1 <= 16
// horizon points) run two instances per warp, one per half (jmpc_step.cuh).
// `lat`: the low-latency variant (jmpc_step.cuh), for launches of a handful of instances.
template <bool LAT>
StepKernel step_kernel_variant(int T, int groups) {
#ifdef JMPC_EXPERIMENT
  if (getenv("JMPC_GENERIC")) return groups == 2 ? jmpc::mpc_step_kernel<0, 16, LAT> : jmpc::mpc_step_kernel<0, 32, LAT>;
#endif
  switch (T) {
    case 8: return jmpc::mpc_step_kernel<8, 16, LAT>;
    case 13: return jmpc::mpc_step_kernel<13, 16, LAT>;
    case 20: return jmpc::mpc_step_kernel<20, 32, LAT>;
    case 25: return jmpc::mpc_step_kernel<25, 32, LAT>;
    default: return groups == 2 ? jmpc::mpc_step_kernel<0, 16, LAT> : jmpc::mpc_step_kernel<0, 32, LAT>;
  }
}
StepKernel step_kernel_for(int T, int* groups, bool lat = false) {
  *groups = 32 / jmpc::group_lanes_for(T);
  return lat ? step_kernel_variant<true>(T, *groups) : step_kernel_variant<false>(T, *groups);
}

// Function attributes and occupancy are resolved once per (handle, T): the single-ego call runs this path every
// time step.  (Experiment builds, -DJMPC_EXPERIMENT, re-read their environment knobs on every call instead.)
int step_geometry(jmpc_handle h, int B, int T, StepGeom* g, StepKernel* kernel) {
  jmpc_handle_s::Geom& c = h->geom[T];
#ifdef JMPC_EXPERIMENT
  c.ready = false;
#endif
  if (!c.ready) {
    int wpb = JMPC_WPB;
    int carve = cudaSharedmemCarveoutMaxShared;
    int cap = h->opt.warps_per_sm;
#ifdef JMPC_EXPERIMENT
    if (const char* e = getenv("JMPC_WPB")) wpb = std::max(1, std::min(JMPC_WPB, atoi(e)));
    if (const char* e = getenv("JMPC_CARVEOUT")) carve = atoi(e);          // percent of the unified L1 / shared memory given to shared
    if (const char* e = getenv("JMPC_WARPS_PER_SM")) cap = atoi(e);
#endif
    int groups = 1;
    StepKernel k = step_kernel_for(T, &groups);
    const size_t smem = jmpc::step_block_smem_bytes(T, wpb, groups);
    CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, wpb * 32, smem));
    if (per_sm < 1) return fail("step kernel does not fit on an SM for this horizon");
    if (cap > 0) per_sm = std::max(1, std::min(per_sm, cap / wpb));
    // Shared memory and L1 share 256 KB per SM.  Ask for no more shared memory than the resident blocks use: T = 20 /
    // T = 8 fit into the 196 KB configuration, which leaves 60 KB of L1 instead of 28 KB for the course tables and
    // the T = 8 kernel's spilled registers (measured when the T = 20 solver loop still spilled: 0.833 -> 0.808 ms on
    // config 2, T = 8 +1.5 %; with that loop spill-free the two configurations time the same on config 2,
    // profiles/r5_ab.txt); T = 13 / T = 25 need the full 228 KB either way.
    if (carve == cudaSharedmemCarveoutMaxShared) {
      int smem_sm = 0;
      CK(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, h->device));
      const size_t need = (size_t)per_sm * (smem + 1024);       // 1 KB per block is reserved by the system
      if (smem_sm > 0) {
        const int pct = (int)std::min<size_t>(100, (need * 100 + (size_t)smem_sm - 1) / (size_t)smem_sm);
        CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
        int check = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&check, k, wpb * 32, smem));
        if (check < per_sm) CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
        else carve = pct;
      }
    }
    // the low-latency variant runs one warp per block, so that a handful of instances spread over as many SMs
    StepKernel kl = step_kernel_for(T, &groups, true);
    const size_t smem_lat = jmpc::step_block_smem_bytes(T, 1, groups);
    CK(cudaFuncSetAttribute(kl, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CK(cudaFuncSetAttribute(kl, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    c.kernel = k; c.kernel_lat = kl; c.groups = groups; c.wpb = wpb; c.per_sm = per_sm; c.smem = smem; c.smem_lat = smem_lat;
    c.ready = true;
    if (getenv("JMPC_DEBUG"))
      fprintf(stderr, "[jmpc] step geometry: T=%d %d instance(s) per warp, %d blocks per SM x %d warps, smem/block=%zu, carve-out %d\n",
              T, groups, per_sm, wpb, smem, carve);
  }
  // A launch of at most eight warps per SM is latency-bound on single warps: it gets the low-latency kernel, one warp
  // per block (a single ego's step at T = 20: 0.27 -> 0.24 ms; 2368 instances at T = 13: 0.43 -> 0.33 ms; from twelve
  // warps per SM on its ~190 registers cost a second wave and the throughput kernel wins:
  // profiles/r2_lat_threshold.txt).
  long long lat_warps_per_sm = 8;
#ifdef JMPC_EXPERIMENT
  if (const char* e = getenv("JMPC_LAT_WARPS_PER_SM")) lat_warps_per_sm = atoll(e);
#endif
  if ((long long)B <= lat_warps_per_sm * h->sm_count * c.groups && h->opt.warps_per_sm <= 0) {
    const int blocks = (B + c.groups - 1) / c.groups;
    g->blocks = blocks; g->threads = 32; g->smem = c.smem_lat; g->groups_total = blocks * c.groups;
    *kernel = c.kernel_lat;
    return 0;
  }
  int blocks = h->sm_count * c.per_sm;
  const int per_block = c.wpb * c.groups;
  const int need = (B + per_block - 1) / per_block;
  if (blocks > need) blocks = need;
  g->blocks = blocks; g->threads = c.wpb * 32; g->smem = c.smem; g->groups_total = blocks * per_block;
  *kernel = c.kernel;
  return 0;
}

int ensure_scratch(jmpc_handle h, size_t doubles) {
  if (doubles <= h->pscratch_doubles) return 0;
  if (h->d_pscratch) cudaFree(h->d_pscratch);
  h->d_pscratch = nullptr; h->pscratch_doubles = 0;
  CK(cudaMalloc(&h->d_pscratch, doubles * sizeof(double)));
  h->pscratch_doubles = doubles;
  return 0;
}

int ensure_stage(jmpc_handle h, size_t bytes) {
  if (bytes > h->d_stage_bytes) {
    if (h->d_stage) cudaFree(h->d_stage);
    h->d_stage = nullptr; h->d_stage_bytes = 0;
    CK(cudaMalloc(&h->d_stage, bytes));
    h->d_stage_bytes = bytes;
  }
  if (bytes > h->h_stage_bytes) {
    if (h->h_stage) cudaFreeHost(h->h_stage);
    h->h_stage = nullptr; h->h_stage_bytes = 0;
    CK(cudaMallocHost(&h->h_stage, bytes));
    h->h_stage_bytes = bytes;
  }
  return 0;
}

// ---- small kernels that live here -----------------------------------------------------------------------

// Simulation.step (simulation.py:35-47) + Bicycle.step (bicycle/main.py:28-41), one thread per instance.
__global__ void plant_step_kernel(int B, double* __restrict__ state, const double* __restrict__ a,
                                  const double* __restrict__ delta, const double* __restrict__ params,
                                  jmpc::ParamBlock defaults) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double* prm = params ? params + (size_t)b * JMPC_NPARAM : defaults.v;
  const double dt = prm[JMPC_P_DT], L = prm[JMPC_P_L], ms = prm[JMPC_P_MAX_STEER];
  double x = state[4 * b], y = state[4 * b + 1], v = state[4 * b + 2], yaw = state[4 * b + 3];
  const double d = fmax(fmin(delta[b], ms), -ms);
  const double xd = __dmul_rn(v, cos(yaw)), yd = __dmul_rn(v, sin(yaw)), td = __dmul_rn(v / L, tan(d));
  x = __dadd_rn(x, __dmul_rn(xd, dt));
  y = __dadd_rn(y, __dmul_rn(yd, dt));
  yaw = __dadd_rn(yaw, __dmul_rn(td, dt));
  v = __dadd_rn(v, __dmul_rn(a[b], dt));
  v = fmax(fmin(v, prm[JMPC_P_SIM_MAX_SPEED]), prm[JMPC_P_MIN_SPEED]);
  state[4 * b] = x; state[4 * b + 1] = y; state[4 * b + 2] = v; state[4 * b + 3] = yaw;
}

int refresh_circle_tables(jmpc_handle h) {
  CK(cudaSetDevice(h->device));
  for (int c = 0; c < h->n_courses; ++c) {
    const size_t off = (size_t)c * h->course_stride;
    const int n = h->course_n[c];
    jmpc::circle_table_kernel<<<(n + 127) / 128, 128, 0, h->own_stream>>>(
        n, h->d_cx + off, h->d_cy + off, h->d_cyaw + off, h->off_front, h->off_rear, h->d_ccfx + off,
        h->d_ccfy + off, h->d_ccrx + off, h->d_ccry + off);
    CK(cudaGetLastError());
    h->launches++;
  }
  CK(cudaStreamSynchronize(h->own_stream));
  return 0;
}

// Arc-length tables of the uploaded courses (jmpc_collision.cuh: arc_table_kernel), N (N + 1) / 2 doubles per course;
// courses are left without a table (the kernel then sums on the fly) once 256 MB are used.  Frees the old tables,
// places the courses of h->course_n and allocates the new block; off[c] = -1 for a course without a table.
int place_arc_tables(jmpc_handle h, std::vector<long long>& off) {
  if (h->d_arc) { cudaFree(h->d_arc); h->d_arc = nullptr; }
  if (!h->d_arc_off) CK(cudaMalloc(&h->d_arc_off, (size_t)h->max_courses * sizeof(long long)));
  off.assign(h->n_courses, -1);
  h->arc_has.assign(h->n_courses, 0);
  long long total = 0;
  h->arc_all = true;
  const long long cap = (256ll << 20) / (long long)sizeof(double);
  for (int c = 0; c < h->n_courses; ++c) {
    const long long n = h->course_n[c], need = n * (n + 1) / 2;
    if (total + need > cap) { h->arc_all = false; continue; }
    off[c] = total; total += need; h->arc_has[c] = 1;
  }
  if (total > 0) CK(cudaMalloc(&h->d_arc, (size_t)total * sizeof(double)));
  return 0;
}

int refresh_arc_tables(jmpc_handle h) {
  CK(cudaSetDevice(h->device));
  std::vector<long long> off;
  if (place_arc_tables(h, off)) return -1;
  for (int c = 0; c < h->n_courses; ++c) {
    if (off[c] < 0) continue;
    const size_t coff = (size_t)c * h->course_stride;
    const int n = h->course_n[c];
    jmpc::arc_table_kernel<<<(n + 63) / 64, 64, 0, h->own_stream>>>(n, h->d_cx + coff, h->d_cy + coff, h->d_arc + off[c]);
    CK(cudaGetLastError());
    h->launches++;
  }
  CK(cudaMemcpyAsync(h->d_arc_off, off.data(), (size_t)h->n_courses * sizeof(long long), cudaMemcpyHostToDevice, h->own_stream));
  CK(cudaStreamSynchronize(h->own_stream));
  return 0;
}

template <typename F>
__global__ void fma_peak_kernel(F* out, int iters) {
  F a0 = (F)threadIdx.x * (F)1e-3, a1 = a0 + (F)1, a2 = a0 + (F)2, a3 = a0 + (F)3;
  F a4 = a0 + (F)4, a5 = a0 + (F)5, a6 = a0 + (F)6, a7 = a0 + (F)7;
  const F m = (F)0.999, c = (F)1e-3;
  for (int i = 0; i < iters; ++i) {
    a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
    a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

template <typename F>
int measure_fma(jmpc_handle h, double* tflops) {
  const int blocks = h->sm_count * 8, threads = 256, iters = 1 << 14;
  F* d = nullptr;
  CK(cudaMalloc(&d, (size_t)blocks * threads * sizeof(F)));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0, h->own_stream));
    fma_peak_kernel<F><<<blocks, threads, 0, h->own_stream>>>(d, iters);
    CK(cudaEventRecord(e1, h->own_stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    h->launches++;
    const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return 0;
}

}  // namespace

extern "C" {

int32_t jmpc_abi_version(void) { return JMPC_ABI_VERSION; }
int32_t jmpc_nparam(void) { return JMPC_NPARAM; }
const char* jmpc_last_error(void) { return g_err.c_str(); }

int32_t jmpc_create(int32_t device, int32_t max_B, int32_t max_T, int32_t max_N, int32_t max_courses,
                    const double* default_params, const jmpc_options* options, jmpc_handle* out) {
  if (!out) return fail("jmpc_create: out is NULL");
  *out = nullptr;
  if (max_T < 2 || max_T > JMPC_MAX_T) return fail("jmpc_create: max_T must be in [2, JMPC_MAX_T]");
  if (max_B < 1 || max_N < 1 || max_courses < 1) return fail("jmpc_create: sizes must be positive");
  if (max_N > 32767) return fail("jmpc_create: max_N must be <= 32767 (16-bit path indices in the collision kernel)");
  if (!default_params) return fail("jmpc_create: default_params is NULL");
  int count = 0;
  CK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail("jmpc_create: no such CUDA device");
  CK(cudaSetDevice(device));
  jmpc_handle h = new (std::nothrow) jmpc_handle_s();
  if (!h) return fail("jmpc_create: out of host memory");
  h->device = device; h->max_B = max_B; h->max_T = max_T; h->max_N = max_N; h->max_courses = max_courses;
  h->opt.max_solver_iters = 40; h->opt.linearisation_iters = 1; h->opt.mu_tol = 1e-13; h->opt.warps_per_sm = 0;
  h->opt.du_th = 0.0;
  if (options) {
    if (options->du_th > 0) h->opt.du_th = options->du_th;
    if (options->max_solver_iters > 0) h->opt.max_solver_iters = options->max_solver_iters;
    if (options->linearisation_iters > 0) h->opt.linearisation_iters = options->linearisation_iters;
    if (options->mu_tol > 0) h->opt.mu_tol = options->mu_tol;
    if (options->warps_per_sm > 0) h->opt.warps_per_sm = options->warps_per_sm;
  }
  memcpy(h->defaults, default_params, sizeof h->defaults);
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { delete h; return fail("cudaGetDeviceProperties", e); }
  h->sm_count = prop.multiProcessorCount;
  h->course_stride = max_N;
  const size_t cbytes = (size_t)max_courses * max_N * sizeof(double);
  if ((e = cudaMalloc(&h->d_cx, cbytes)) != cudaSuccess || (e = cudaMalloc(&h->d_cy, cbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_cyaw, cbytes)) != cudaSuccess || (e = cudaMalloc(&h->d_cv, cbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_ccfx, cbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_ccfy, cbytes)) != cudaSuccess || (e = cudaMalloc(&h->d_ccrx, cbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_ccry, cbytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_course_n, max_courses * sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_counter, 64)) != cudaSuccess || (e = cudaMemset(h->d_counter, 0, 64)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_gather_timeout, sizeof(int))) != cudaSuccess ||
      (e = cudaMemset(h->d_gather_timeout, 0, sizeof(int))) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    jmpc_destroy(h);
    return fail("jmpc_create: device allocation failed", e);
  }
  *out = h;
  return 0;
}

int32_t jmpc_destroy(jmpc_handle h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaFree(h->d_cx); cudaFree(h->d_cy); cudaFree(h->d_cyaw); cudaFree(h->d_cv); cudaFree(h->d_course_n);
  cudaFree(h->d_ccfx); cudaFree(h->d_ccfy); cudaFree(h->d_ccrx); cudaFree(h->d_ccry); cudaFree(h->d_arc); cudaFree(h->d_arc_off);
  cudaFree(h->d_pscratch); cudaFree(h->d_counter); cudaFree(h->d_stage); cudaFree(h->d_order); cudaFree(h->d_hint);
  cudaFree(h->d_keys); cudaFree(h->d_sched_work); cudaFree(h->d_gather_timeout);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return 0;
}

int32_t jmpc_set_default_params(jmpc_handle h, const double* p) {
  if (!h || !p) return fail("jmpc_set_default_params: NULL argument");
  memcpy(h->defaults, p, sizeof h->defaults);
  return 0;
}

int32_t jmpc_set_courses(jmpc_handle h, int32_t n_courses, int32_t stride, const int32_t* len, const double* cx,
                         const double* cy, const double* cyaw) {
  if (!h || !len || !cx || !cy || !cyaw) return fail("jmpc_set_courses: NULL argument");
  if (n_courses < 1 || n_courses > h->max_courses) return fail("jmpc_set_courses: n_courses out of range");
  for (int c = 0; c < n_courses; ++c)             // validate everything before the handle's state is touched
    if (len[c] < 1 || len[c] > h->max_N || len[c] > stride) return fail("jmpc_set_courses: course length out of range");
  CK(cudaSetDevice(h->device));
  // Uploads go through the handle's pinned block on its own stream, the stream the table kernels below run on: a
  // pageable cudaMemcpy on the legacy stream has no ordering against a non-blocking stream.
  const size_t row = (size_t)h->max_N * sizeof(double);
  if (ensure_stage(h, 3 * row + (size_t)n_courses * sizeof(int))) return -1;
  cudaStream_t st = h->own_stream;
  for (int c = 0; c < n_courses; ++c) {
    const size_t off = (size_t)c * h->course_stride, src = (size_t)c * stride, nb = (size_t)len[c] * sizeof(double);
    memcpy(h->h_stage, cx + src, nb); memcpy(h->h_stage + row, cy + src, nb); memcpy(h->h_stage + 2 * row, cyaw + src, nb);
    CK(cudaMemcpyAsync(h->d_cx + off, h->h_stage, nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_cy + off, h->h_stage + row, nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_cyaw + off, h->h_stage + 2 * row, nb, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));                  // the staging rows are reused by the next course
  }
  memcpy(h->h_stage, len, (size_t)n_courses * sizeof(int));
  CK(cudaMemcpyAsync(h->d_course_n, h->h_stage, (size_t)n_courses * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  h->course_n.assign(len, len + n_courses);
  h->n_courses = n_courses;
  h->have_cv = false;                               // a speed profile belongs to the courses it was uploaded for
  if (refresh_arc_tables(h)) return -1;
  return refresh_circle_tables(h);
}

int32_t jmpc_set_course_speed(jmpc_handle h, int32_t n_courses, int32_t stride, const double* cv) {
  if (!h) return fail("jmpc_set_course_speed: NULL handle");
  if (!cv) { h->have_cv = false; return 0; }
  if (n_courses != h->n_courses) return fail("jmpc_set_course_speed: n_courses differs from the uploaded courses");
  for (int c = 0; c < n_courses; ++c)
    if (h->course_n[c] > stride) return fail("jmpc_set_course_speed: stride shorter than a course");
  CK(cudaSetDevice(h->device));
  if (ensure_stage(h, (size_t)h->max_N * sizeof(double))) return -1;
  cudaStream_t st = h->own_stream;
  for (int c = 0; c < n_courses; ++c) {
    const size_t nb = (size_t)h->course_n[c] * sizeof(double);
    memcpy(h->h_stage, cv + (size_t)c * stride, nb);
    CK(cudaMemcpyAsync(h->d_cv + (size_t)c * h->course_stride, h->h_stage, nb, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
  }
  h->have_cv = true;
  return 0;
}

int32_t jmpc_set_car_geometry(jmpc_handle h, double front_offset, double rear_offset, double radius) {
  if (!h) return fail("jmpc_set_car_geometry: NULL handle");
  if (!(radius > 0)) return fail("jmpc_set_car_geometry: radius must be positive");
  h->off_front = front_offset; h->off_rear = rear_offset; h->radius = radius;
  return h->n_courses ? refresh_circle_tables(h) : 0;
}

namespace {
// Launch of the step kernel.  The in-out arrays have separate read and write pointers: jmpc_step passes the same
// array twice, jmpc_step_host reads device copies and writes page-locked host memory.
int launch_step(jmpc_handle h, int B, int T, const double* state, const int* course_id, const int* course_len,
                const int* target_in, int* target_out, const int* warm, const double* oa_in, const double* od_in,
                double* oa_out, double* od_out, const double* params, double* ox, double* oy, double* ov,
                double* oyaw, double* xref, double* cost, int* status, int* iters, double* record, cudaStream_t s) {
  StepGeom g;
  StepKernel kernel = nullptr;
  if (step_geometry(h, B, T, &g, &kernel)) return -1;
  const int n = 2 * T;
  if (ensure_scratch(h, (size_t)g.groups_total * jmpc::tiles_doubles(n))) return -1;
  jmpc::StepArgs a;
  a.B = B; a.T = T; a.lin_iters = h->opt.linearisation_iters; a.max_iters = h->opt.max_solver_iters;
  a.mu_tol = h->opt.mu_tol; a.du_th = h->opt.du_th;
  a.tol_res = 1e-9; a.init_mu = 0.0;
#ifdef JMPC_EXPERIMENT
  if (const char* e = getenv("JMPC_TOL_RES")) a.tol_res = atof(e);          // solver experiments (tests/tools/tune_solver.py)
  if (const char* e = getenv("JMPC_INIT_MU")) a.init_mu = atof(e);
#endif
  a.cx = h->d_cx; a.cy = h->d_cy; a.cyaw = h->d_cyaw; a.cv = h->have_cv ? h->d_cv : nullptr; a.course_n = h->d_course_n;
  a.course_stride = h->course_stride; a.n_courses = h->n_courses;
  a.state = state; a.course_id = course_id; a.course_len = course_len; a.warm = warm; a.params = params;
  memcpy(a.defaults, h->defaults, sizeof a.defaults);
  a.target_ind = target_in; a.oa = oa_in; a.od = od_in;
  a.target_out = target_out; a.oa_out = oa_out; a.od_out = od_out;
  a.ox = ox; a.oy = oy; a.ov = ov; a.oyaw = oyaw; a.xref = xref;
  a.cost = cost; a.status = status; a.iters = iters; a.record = record;
  a.n_peers = h->n_peers; a.rank_offset = h->rank_offset; a.skip = h->skip;
  for (int p = 0; p < JMPC_MAX_PEERS; ++p) { a.peer_rec[p] = h->peer_rec[p]; a.peer_flag[p] = h->peer_flag[p]; }
  a.n_flag_peers = h->n_flag_peers; a.gather_step = h->gather_step; a.blocks_done = h->d_counter + 1;
  a.pscratch = h->d_pscratch; a.counter = h->d_counter;
  a.order = nullptr; a.work_hint = nullptr;
  if (h->schedule > 0) {
    if (!h->d_order) {
      CK(cudaMalloc(&h->d_order, (size_t)h->max_B * sizeof(int)));
      CK(cudaMalloc(&h->d_hint, (size_t)h->max_B * sizeof(int)));
      CK(cudaMalloc(&h->d_keys, (size_t)h->max_B));
      CK(cudaMalloc(&h->d_sched_work, 2 * jmpc::kSchedKeys * sizeof(int)));
      CK(cudaMemsetAsync(h->d_hint, 0, (size_t)h->max_B * sizeof(int), s));
    }
    // Ordering pays in two ways: a batch of a few waves of the resident instance slots finishes when its slowest
    // late-started instance does (longest first), and on the half-warp kernels neighbours in the queue share a warp
    // and iterate in lock step (similar keys = less idling).  With the previous step's iteration counts as keys it
    // pays at any size (measured on 65 536 / 262 144 instances, T = 13: +8 % / +6 %); the a-priori key is a weaker
    // predictor and is only used while the batch is a few waves deep.
    long long sched_max_waves = 16;
    double acc_weight = 2.0;                         // weight of the acceleration-saturation stages in the a-priori key
#ifdef JMPC_EXPERIMENT
    if (const char* e = getenv("JMPC_SCHED_MAX_WAVES")) sched_max_waves = atoll(e);
    if (const char* e = getenv("JMPC_KEY_ACC_WEIGHT")) acc_weight = atof(e);
#endif
    const bool have_hint = h->schedule >= 2 && h->hint_B == B && h->hint_T == T;
    // (two instances per warp: with the previous step's counts the pairing alone pays, even when the whole batch is resident)
    const bool pairing = have_hint && h->geom[T].groups > 1 && B >= 1024;
    if (pairing || (B > g.groups_total && (have_hint || (long long)B <= sched_max_waves * (long long)g.groups_total))) {
      jmpc::ParamVec dv;
      memcpy(dv.v, h->defaults, sizeof dv.v);
      const int sblocks = std::max(1, std::min((B + jmpc::kSchedThreads - 1) / jmpc::kSchedThreads, 2 * h->sm_count));
      CK(cudaMemsetAsync(h->d_sched_work, 0, 2 * jmpc::kSchedKeys * sizeof(int), s));
      jmpc::schedule_count_kernel<<<sblocks, jmpc::kSchedThreads, 0, s>>>(B, T, have_hint ? h->d_hint : nullptr, state, params, dv,
                                                                         acc_weight, h->d_keys, h->d_sched_work);
      jmpc::schedule_place_kernel<<<sblocks, jmpc::kSchedThreads, 0, s>>>(B, h->d_keys, h->d_sched_work, h->d_order);
      CK(cudaGetLastError());
      h->launches += 2;
      a.order = h->d_order;
    }
    if (h->schedule >= 2) { a.work_hint = h->d_hint; h->hint_B = B; h->hint_T = T; }
  }
  CK(cudaMemsetAsync(h->d_counter, 0, sizeof(unsigned int), s));
  kernel<<<g.blocks, g.threads, g.smem, s>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}
}  // namespace

int32_t jmpc_step(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                  const int32_t* course_len, int32_t* target_ind, const int32_t* warm, double* oa, double* od,
                  const double* params, double* ox, double* oy, double* ov, double* oyaw, double* xref,
                  double* cost, int32_t* status, int32_t* iters, double* record, void* stream) {
  if (!h) return fail("jmpc_step: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_step: B out of range");
  if (T < 2 || T > h->max_T) return fail("jmpc_step: T out of range");
  if (!state || !target_ind || !oa || !od || !ox || !oy || !ov || !oyaw || !xref || !cost || !status)
    return fail("jmpc_step: NULL array");
  if (h->n_courses < 1) return fail("jmpc_step: no courses uploaded (jmpc_set_courses)");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  return launch_step(h, B, T, state, course_id, course_len, target_ind, target_ind, warm, oa, od, oa, od, params, ox, oy,
                     ov, oyaw, xref, cost, status, iters, record, (cudaStream_t)stream);
}

int32_t jmpc_host_alloc(jmpc_handle h, size_t bytes, void** out) {
  if (!h || !out) return fail("jmpc_host_alloc: NULL argument");
  CK(cudaSetDevice(h->device));
  CK(cudaMallocHost(out, bytes ? bytes : 1));
  void* dev = nullptr;
  if (cudaHostGetDevicePointer(&dev, *out, 0) != cudaSuccess) { cudaGetLastError(); dev = nullptr; }
  if (dev) h->host_blocks.push_back({(char*)*out, bytes ? bytes : 1, (char*)dev});
  return 0;
}

int32_t jmpc_host_free(jmpc_handle h, void* p) {
  if (!h) return fail("jmpc_host_free: NULL handle");
  if (p) {
    for (size_t k = 0; k < h->host_blocks.size(); ++k)
      if (h->host_blocks[k].base == (char*)p) { h->host_blocks.erase(h->host_blocks.begin() + k); break; }
    CK(cudaFreeHost(p));
  }
  return 0;
}

namespace {
// Page-locked?  If so `mapped` receives the device-side address.  Blocks handed out by jmpc_host_alloc are recognised
// from the handle's own list (no driver call: cudaPointerGetAttributes costs ~1.5 us, twenty of them per step add up).
bool is_pinned(jmpc_handle h, const void* p, void** mapped) {
  const char* c = (const char*)p;
  for (const auto& r : h->host_blocks)
    if (c >= r.base && c < r.base + r.bytes) { *mapped = r.dev + (c - r.base); return true; }
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  if (at.type != cudaMemoryTypeHost) return false;
  *mapped = at.devicePointer;
  return true;
}
}  // namespace

int32_t jmpc_debug_cycles(jmpc_handle h, uint64_t* out32, int32_t reset) {
  if (!h || !out32) return fail("jmpc_debug_cycles: NULL argument");
#ifdef JMPC_CYCLES
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpyFromSymbol(out32, jmpc::g_cycles, 32 * sizeof(uint64_t)));
  if (reset) { uint64_t z[32] = {}; CK(cudaMemcpyToSymbol(jmpc::g_cycles, z, sizeof z)); }
  return 0;
#else
  (void)reset;
  return fail("jmpc_debug_cycles: library built without -DJMPC_CYCLES");
#endif
}

int32_t jmpc_set_schedule(jmpc_handle h, int32_t mode) {
  if (!h) return fail("jmpc_set_schedule: NULL handle");
  if (mode < 0 || mode > 2) return fail("jmpc_set_schedule: mode must be 0, 1 or 2");
  h->schedule = mode; h->hint_B = 0; h->hint_T = 0;
  return 0;
}

int32_t jmpc_reset_schedule_hints(jmpc_handle h) {
  if (!h) return fail("jmpc_reset_schedule_hints: NULL handle");
  h->hint_B = 0; h->hint_T = 0;
  return 0;
}

int32_t jmpc_set_host_transfer(jmpc_handle h, int32_t mode) {
  if (!h) return fail("jmpc_set_host_transfer: NULL handle");
  if (mode < 0 || mode > 2) return fail("jmpc_set_host_transfer: mode must be 0, 1 or 2");
  h->host_transfer = mode;
  return 0;
}

int32_t jmpc_set_skip_mask(jmpc_handle h, const int32_t* skip) {
  if (!h) return fail("jmpc_set_skip_mask: NULL handle");
  h->skip = skip;
  return 0;
}

int32_t jmpc_set_record_peers(jmpc_handle h, int32_t n_peers, const uint64_t* peer_tables, int64_t rank_offset) {
  if (!h) return fail("jmpc_set_record_peers: NULL handle");
  if (n_peers < 0 || n_peers > JMPC_MAX_PEERS) return fail("jmpc_set_record_peers: n_peers out of range");
  if (n_peers > 0 && !peer_tables) return fail("jmpc_set_record_peers: NULL table list");
  if (rank_offset < 0) return fail("jmpc_set_record_peers: negative rank_offset");
  for (int p = 0; p < JMPC_MAX_PEERS; ++p) h->peer_rec[p] = (p < n_peers) ? reinterpret_cast<double*>(peer_tables[p]) : nullptr;
  h->n_peers = n_peers; h->rank_offset = rank_offset;
  return 0;
}

int32_t jmpc_set_record_flags(jmpc_handle h, int32_t n_peers, const uint64_t* peer_flags, uint64_t step) {
  if (!h) return fail("jmpc_set_record_flags: NULL handle");
  if (n_peers < 0 || n_peers > JMPC_MAX_PEERS) return fail("jmpc_set_record_flags: n_peers out of range");
  if (n_peers > 0 && !peer_flags) return fail("jmpc_set_record_flags: NULL flag list");
  for (int p = 0; p < JMPC_MAX_PEERS; ++p)
    h->peer_flag[p] = (p < n_peers) ? reinterpret_cast<unsigned long long*>(peer_flags[p]) : nullptr;
  h->n_flag_peers = n_peers; h->gather_step = step;
  return 0;
}

int32_t jmpc_gather_wait(jmpc_handle h, const uint64_t* flags, int32_t world, uint64_t step, void* stream) {
  if (!h || !flags) return fail("jmpc_gather_wait: NULL argument");
  if (world < 1 || world > JMPC_MAX_PEERS) return fail("jmpc_gather_wait: world out of range");
  CK(cudaSetDevice(h->device));
  jmpc::gather_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long*>(flags), world, step,
                                                              h->d_gather_timeout);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_gather_timed_out(jmpc_handle h, int32_t* out) {
  if (!h || !out) return fail("jmpc_gather_timed_out: NULL argument");
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpy(out, h->d_gather_timeout, sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int32_t jmpc_step_host(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                       const int32_t* course_len, int32_t* target_ind, const int32_t* warm, double* oa,
                       double* od, const double* params, double* ox, double* oy, double* ov, double* oyaw,
                       double* xref, double* cost, int32_t* status, int32_t* iters, double* record) {
  return jmpc_step_host_io(h, B, T, state, course_id, course_len, target_ind, warm, oa, od, params, target_ind, oa, od,
                           ox, oy, ov, oyaw, xref, cost, status, iters, record);
}

int32_t jmpc_step_host_io(jmpc_handle h, int32_t B, int32_t T, const double* state, const int32_t* course_id,
                          const int32_t* course_len, const int32_t* target_in, const int32_t* warm,
                          const double* oa_in, const double* od_in, const double* params, int32_t* target_out,
                          double* oa_out, double* od_out, double* ox, double* oy, double* ov, double* oyaw,
                          double* xref, double* cost, int32_t* status, int32_t* iters, double* record) {
  if (!h) return fail("jmpc_step_host: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_step_host: B out of range");
  if (T < 2 || T > h->max_T) return fail("jmpc_step_host: T out of range");
  if (!state || !target_in || !oa_in || !od_in || !target_out || !oa_out || !od_out || !ox || !oy || !ov || !oyaw ||
      !xref || !cost || !status)
    return fail("jmpc_step_host: NULL array");
  if (h->n_courses < 1) return fail("jmpc_step_host: no courses uploaded (jmpc_set_courses)");
  if (h->skip) return fail("jmpc_step_host: a skip mask is set (jmpc_set_skip_mask is for the device entry points)");
  if (course_id)             // host arrays can be validated (the device entry points clamp instead, jmpc_step.cuh)
    for (int k = 0; k < B; ++k)
      if (course_id[k] < 0 || course_id[k] >= h->n_courses) return fail("jmpc_step_host: course_id out of range");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  const size_t T1 = T + 1, b = (size_t)B;
  // Staging block layout [inputs | outputs], the same offsets on the device (d_stage) and in the handle's
  // page-locked host block (h_stage).  Transfer modes (jmpc_set_host_transfer):
  //   1  (default) inputs by cudaMemcpyAsync into d_stage; the kernel stores its results directly into page-locked
  //      host memory through the device mapping (unified addressing): the caller's own array where that is
  //      page-locked (jmpc_host_alloc, cudaHostAlloc, torch pin_memory), the h_stage slot otherwise (one host
  //      memcpy).  A warp writes ~1.7 KB when it is done with an instance; the stores ride under the other warps'
  //      solves, and at ~6 GB/s of results the PCIe link is far from saturated, so the device -> host transfer
  //      leaves the critical path (measured: 1.61 -> 1.43 ms per 4096-instance step).
  //   2  the kernel also reads its inputs from page-locked host memory (no copy engine at all).  Measured slower
  //      than 1: every warp waits a PCIe round trip when it picks an instance up (kernel 1.24 -> 1.30 ms).
  //   0  staged DMA both ways (results to d_stage, cudaMemcpyAsync back).
  // Instances that fail the index rule or are infeasible get their input values in oa_out / od_out / target_out
  // (the kernel carries them over), so "in-out arrays keep their values" holds whether or not the arrays alias.
  struct Seg { size_t off, bytes; void* host; bool pinned; void* mapped; };
  size_t off = 0;
  Seg segs[20];
  int ns = 0;
#ifdef JMPC_EXPERIMENT
  const bool timing = getenv("JMPC_TIMING") != nullptr;                 // host-side breakdown on stderr
#else
  const bool timing = false;
#endif
  auto now = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_begin = timing ? now() : 0.0;
  const int mode = h->host_transfer;
  auto seg = [&](size_t bytes, const void* host) -> Seg& {
    Seg& s = segs[ns++];
    s.off = off; s.bytes = host ? bytes : 0; s.host = const_cast<void*>(host);
    s.mapped = nullptr;
    s.pinned = host ? is_pinned(h, host, &s.mapped) : false;
    off += (s.bytes + 15) & ~size_t(15);
    return s;
  };
  const Seg& s_state = seg(b * 4 * 8, state);
  const Seg& s_params = seg(b * JMPC_NPARAM * 8, params);
  const Seg& s_cid = seg(b * 4, course_id);
  const Seg& s_clen = seg(b * 4, course_len);
  const Seg& s_warm = seg(b * 4, warm);
  const Seg& s_oa_in = seg(b * T * 8, oa_in);
  const Seg& s_od_in = seg(b * T * 8, od_in);
  const Seg& s_tgt_in = seg(b * 4, target_in);
  const int first_out = ns;
  const size_t in_end = off;
  const Seg& s_oa = seg(b * T * 8, oa_out);
  const Seg& s_od = seg(b * T * 8, od_out);
  const Seg& s_tgt = seg(b * 4, target_out);
  const Seg& s_ox = seg(b * T1 * 8, ox);
  const Seg& s_oy = seg(b * T1 * 8, oy);
  const Seg& s_ov = seg(b * T1 * 8, ov);
  const Seg& s_oyaw = seg(b * T1 * 8, oyaw);
  const Seg& s_xref = seg(b * 4 * T1 * 8, xref);
  const Seg& s_cost = seg(b * 8, cost);
  const Seg& s_status = seg(b * 4, status);
  const Seg& s_iters = seg(b * 4, iters);
  const Seg& s_rec = seg(b * JMPC_RECORD_LEN * 8, record);
  const size_t total = off;
  if (ensure_stage(h, total)) return -1;
  char* hs = h->h_stage; char* ds = h->d_stage;
  cudaStream_t st = h->own_stream;
  // device mappings of the page-locked arrays
  char* hs_dev = nullptr;
  bool map_ok = mode >= 1;
  if (map_ok && cudaHostGetDevicePointer((void**)&hs_dev, hs, 0) != cudaSuccess) { cudaGetLastError(); map_ok = false; }
  for (int k = 0; k < ns && map_ok; ++k) {
    Seg& s = segs[k];
    if (!s.bytes) continue;
    if (s.pinned) { if (!s.mapped) map_ok = false; }
    else s.mapped = hs_dev + s.off;
  }
  const bool zc_out = map_ok, zc_in = map_ok && mode >= 2;
  // ---- inputs
  if (zc_in) {
    for (int k = 0; k < first_out; ++k)
      if (segs[k].bytes && !segs[k].pinned) memcpy(hs + segs[k].off, segs[k].host, segs[k].bytes);
  } else {
    bool any_pinned_in = false;
    for (int k = 0; k < first_out; ++k) any_pinned_in = any_pinned_in || (segs[k].bytes && segs[k].pinned);
    if (!any_pinned_in) {
      for (int k = 0; k < first_out; ++k)
        if (segs[k].bytes) memcpy(hs + segs[k].off, segs[k].host, segs[k].bytes);
      CK(cudaMemcpyAsync(ds, hs, in_end, cudaMemcpyHostToDevice, st));
    } else {
      for (int k = 0; k < first_out; ++k) {
        const Seg& s = segs[k];
        if (!s.bytes) continue;
        const void* src = s.host;
        if (!s.pinned) { memcpy(hs + s.off, s.host, s.bytes); src = hs + s.off; }
        CK(cudaMemcpyAsync(ds + s.off, src, s.bytes, cudaMemcpyHostToDevice, st));
      }
    }
  }
  auto rp = [&](const Seg& s) -> char* { return s.bytes ? (zc_in ? (char*)s.mapped : ds + s.off) : nullptr; };    // read side
  auto wp = [&](const Seg& s) -> char* { return s.bytes ? (zc_out ? (char*)s.mapped : ds + s.off) : nullptr; };   // write side
  const double t_prep = timing ? now() : 0.0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (timing) { cudaEventCreate(&ev0); cudaEventCreate(&ev1); cudaEventRecord(ev0, st); }
  int rc = launch_step(h, B, T, (const double*)rp(s_state), (const int*)rp(s_cid), (const int*)rp(s_clen),
                       (const int*)rp(s_tgt_in), (int*)wp(s_tgt), (const int*)rp(s_warm), (const double*)rp(s_oa_in),
                       (const double*)rp(s_od_in), (double*)wp(s_oa), (double*)wp(s_od), (const double*)rp(s_params),
                       (double*)wp(s_ox), (double*)wp(s_oy), (double*)wp(s_ov), (double*)wp(s_oyaw), (double*)wp(s_xref),
                       (double*)wp(s_cost), (int*)wp(s_status), (int*)wp(s_iters), (double*)wp(s_rec), st);
  if (rc) return rc;
  if (timing) cudaEventRecord(ev1, st);
  const double t_launch = timing ? now() : 0.0;
  // ---- results
  if (!zc_out) {
    for (int k = first_out; k < ns; ++k) {
      const Seg& s = segs[k];
      if (!s.bytes) continue;
      CK(cudaMemcpyAsync(s.pinned ? s.host : (void*)(hs + s.off), ds + s.off, s.bytes, cudaMemcpyDeviceToHost, st));
    }
  }
  CK(cudaStreamSynchronize(st));
  const double t_sync = timing ? now() : 0.0;
  for (int k = first_out; k < ns; ++k) {
    const Seg& s = segs[k];
    if (s.bytes && !s.pinned) memcpy(s.host, hs + s.off, s.bytes);
  }
  if (timing) {
    float kms = 0.f;
    cudaEventElapsedTime(&kms, ev0, ev1);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    fprintf(stderr, "[jmpc] step_host B=%d mode=%d: prep %.1f us, launch %.1f us, wait %.1f us (kernel %.1f us by events), post %.1f us\n",
            B, mode, t_prep - t_begin, t_launch - t_prep, t_sync - t_launch, kms * 1e3, now() - t_sync);
  }
  return 0;
}

// jmpc_collision, jmpc_collision_planned and jmpc_collision_masked: the same checks and launch sizing for every
// instantiation of the kernel (section B of the planned one and the mask use no extra shared memory).
extern "C++" {
template <bool Planned, bool Masked = false>
static int32_t launch_collision(const char* name, jmpc_handle h, int32_t B, const int32_t* course_id,
                                const int32_t* agent_idx, const double* v, const double* obstacles, int32_t n_obs,
                                const double* plans, int32_t n_planned, int32_t plan_len, int32_t frame_window,
                                int32_t margin, double horizon_s, const double* params, int32_t* flag,
                                int32_t* course_len_out, void* stream, const int32_t* consider = nullptr) {
  char msg[160];
  auto err = [&](const char* what) { snprintf(msg, sizeof msg, "%s: %s", name, what); return fail(msg); };
  if (!h) return err("NULL handle");
  if (B < 0 || B > h->max_B) return err("B out of range");
  if (!agent_idx || !v || !flag || !course_len_out) return err("NULL array");
  if (n_obs < 0 || n_obs > jmpc::kMaxObstacles) return err("n_obs out of range");
  if (n_obs > 0 && !obstacles) return err("obstacles is NULL");
  if (frame_window < 0 || frame_window > jmpc::kMaxFrameWindow) return err("frame_window out of range");
  if (h->n_courses < 1) return err("no courses uploaded (jmpc_set_courses)");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::CollisionArgs a;
  a.B = B; a.n_courses = h->n_courses; a.cx = h->d_cx; a.cy = h->d_cy; a.cyaw = h->d_cyaw; a.course_n = h->d_course_n;
  a.ccfx = h->d_ccfx; a.ccfy = h->d_ccfy; a.ccrx = h->d_ccrx; a.ccry = h->d_ccry;
  a.arc_tab = h->d_arc; a.arc_off = h->d_arc_off;
#ifdef JMPC_EXPERIMENT
  if (getenv("JMPC_NO_ARC_TABLE")) a.arc_tab = nullptr;
#endif
  a.off_front = h->off_front; a.off_rear = h->off_rear; a.radius = h->radius; a.arc_cap = h->max_N;
  a.course_stride = h->course_stride; a.course_id = course_id; a.agent_idx = agent_idx; a.v = v;
  a.obstacles = obstacles; a.n_obs = n_obs; a.frame_window = frame_window; a.margin = margin;
  a.horizon_s = horizon_s; a.params = params;
  memcpy(a.defaults.v, h->defaults, sizeof h->defaults);
  a.flag = flag; a.course_len_out = course_len_out; a.skip = h->skip;
  a.plans = plans; a.n_planned = n_planned; a.plan_len = plan_len;
  // with a table for every course the kernel needs no shared memory for the arc scan: 5 KB per warp instead of 12.6 KB
  // at max_N = 960 and two obstacles, i.e. more than twice the resident warps of this latency-bound kernel
  a.arc_smem = (a.arc_tab && h->arc_all) ? 0 : h->max_N;
  // 4 warps per block unless a long course's arc scan does not leave room for them: then 2, or 1 (jmpc.h states the
  // resulting max_N limit).  The warps of a block share nothing, so the results do not depend on the count.
  const size_t smem_cap = 200 * 1024, warp_smem = jmpc::collision_warp_smem_bytes(a.arc_smem, n_obs);
  if (warp_smem > smem_cap) return err("course too long for the shared-memory arc scan");
  int wpb = 4;
  while (wpb > 1 && wpb * warp_smem > smem_cap) wpb >>= 1;
  const int blocks = (B + wpb - 1) / wpb;
  const size_t smem = wpb * warp_smem;
  bool& attr_set = Masked ? h->collision_masked_attr_set[Planned]
                          : (Planned ? h->collision_planned_attr_set : h->collision_attr_set);
  if constexpr (Masked) {
    if (!attr_set) {                        // per handle: function attributes are per device
      CK(cudaFuncSetAttribute(jmpc::masked_collision_kernel<Planned>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)smem_cap));
      attr_set = true;
    }
    jmpc::masked_collision_kernel<Planned><<<blocks, wpb * 32, smem, (cudaStream_t)stream>>>(a, consider);
  } else {
    if (!attr_set) {
      CK(cudaFuncSetAttribute(jmpc::collision_kernel<Planned>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)smem_cap));
      attr_set = true;
    }
    jmpc::collision_kernel<Planned><<<blocks, wpb * 32, smem, (cudaStream_t)stream>>>(a);
  }
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}
}  // extern "C++"

int32_t jmpc_collision(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                       const double* v, const double* obstacles, int32_t n_obs, int32_t frame_window,
                       int32_t margin, double horizon_s, const double* params, int32_t* flag,
                       int32_t* course_len_out, void* stream) {
  return launch_collision<false>("jmpc_collision", h, B, course_id, agent_idx, v, obstacles, n_obs, nullptr, 0, 1,
                                 frame_window, margin, horizon_s, params, flag, course_len_out, stream);
}

int32_t jmpc_collision_planned(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                               const double* v, const double* obstacles, int32_t n_obs, const double* plans,
                               int32_t n_planned, int32_t plan_len, int32_t frame_window, int32_t margin,
                               double horizon_s, const double* params, int32_t* flag, int32_t* course_len_out,
                               void* stream) {
  if (n_planned < 0 || n_planned > n_obs) return fail("jmpc_collision_planned: n_planned must be in [0, n_obs]");
  if (plan_len < 1) return fail("jmpc_collision_planned: plan_len must be >= 1");
  if (n_planned > 0 && !plans) return fail("jmpc_collision_planned: plans is NULL");
  return launch_collision<true>("jmpc_collision_planned", h, B, course_id, agent_idx, v, obstacles, n_obs, plans,
                                n_planned, plan_len, frame_window, margin, horizon_s, params, flag, course_len_out,
                                stream);
}

int32_t jmpc_collision_masked(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                              const double* v, const double* obstacles, int32_t n_obs, const double* plans,
                              int32_t n_planned, int32_t plan_len, const int32_t* consider, int32_t frame_window,
                              int32_t margin, double horizon_s, const double* params, int32_t* flag,
                              int32_t* course_len_out, void* stream) {
  if (n_planned < 0 || n_planned > n_obs) return fail("jmpc_collision_masked: n_planned must be in [0, n_obs]");
  if (plan_len < 1) return fail("jmpc_collision_masked: plan_len must be >= 1");
  if (n_planned > 0 && !plans) return fail("jmpc_collision_masked: plans is NULL");
  if (!consider) return fail("jmpc_collision_masked: consider is NULL");
  if (n_planned > 0)
    return launch_collision<true, true>("jmpc_collision_masked", h, B, course_id, agent_idx, v, obstacles, n_obs, plans,
                                        n_planned, plan_len, frame_window, margin, horizon_s, params, flag,
                                        course_len_out, stream, consider);
  return launch_collision<false, true>("jmpc_collision_masked", h, B, course_id, agent_idx, v, obstacles, n_obs,
                                       nullptr, 0, 1, frame_window, margin, horizon_s, params, flag, course_len_out,
                                       stream, consider);
}

int32_t jmpc_collision_host(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* agent_idx,
                            const double* v, const double* obstacles, int32_t n_obs, int32_t frame_window,
                            int32_t margin, double horizon_s, const double* params, int32_t* flag,
                            int32_t* course_len_out) {
  if (!h) return fail("jmpc_collision_host: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_collision_host: B out of range");
  if (!agent_idx || !v || !flag || !course_len_out) return fail("jmpc_collision_host: NULL array");
  if (n_obs < 0 || n_obs > jmpc::kMaxObstacles) return fail("jmpc_collision_host: n_obs out of range");
  if (n_obs > 0 && !obstacles) return fail("jmpc_collision_host: obstacles is NULL");
  if (h->skip) return fail("jmpc_collision_host: a skip mask is set (jmpc_set_skip_mask is for the device entry points)");
  if (course_id)
    for (int k = 0; k < B; ++k)
      if (course_id[k] < 0 || course_id[k] >= h->n_courses) return fail("jmpc_collision_host: course_id out of range");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  const size_t b = (size_t)B;
  // Inputs: page-locked caller arrays (jmpc_host_alloc) are copied to the device straight from where they are, others
  // through the handle's pinned block.  Results: the kernel stores flag / course_len_out into page-locked host memory
  // through its device mapping (the caller's arrays when they are page-locked, the pinned block + one memcpy otherwise),
  // as the step's host entry point does: no device->host copy pass.
  struct Seg { size_t off, bytes; const void* host; bool pinned; void* mapped; };
  Seg segs[7];
  int ns = 0;
  size_t off = 0;
  auto seg = [&](size_t bytes, const void* host) -> Seg& {
    Seg& s = segs[ns++];
    s.off = off; s.bytes = host ? bytes : 0; s.host = host; s.mapped = nullptr;
    s.pinned = (host && s.bytes) ? is_pinned(h, host, &s.mapped) : false;
    off += (s.bytes + 15) & ~size_t(15);
    return s;
  };
  const Seg& s_v = seg(b * 8, v);
  const Seg& s_obs = seg(b * n_obs * 6 * 8, n_obs ? obstacles : nullptr);
  const Seg& s_prm = seg(b * JMPC_NPARAM * 8, params);
  const Seg& s_cid = seg(b * 4, course_id);
  const Seg& s_idx = seg(b * 4, agent_idx);
  const int first_out = ns;
  Seg& s_flag = seg(b * 4, flag);
  Seg& s_len = seg(b * 4, course_len_out);
  if (ensure_stage(h, off)) return -1;
  char* hs = h->h_stage; char* ds = h->d_stage;
  cudaStream_t st = h->own_stream;
  for (int k = 0; k < first_out; ++k) {
    const Seg& s = segs[k];
    if (!s.bytes) continue;
    const void* src = s.host;
    if (!s.pinned) { memcpy(hs + s.off, s.host, s.bytes); src = hs + s.off; }
    CK(cudaMemcpyAsync(ds + s.off, src, s.bytes, cudaMemcpyHostToDevice, st));
  }
  char* hs_dev = nullptr;
  bool zc_out = h->host_transfer >= 1;
  if (zc_out && cudaHostGetDevicePointer((void**)&hs_dev, hs, 0) != cudaSuccess) { cudaGetLastError(); zc_out = false; }
  for (int k = first_out; k < ns && zc_out; ++k) {
    Seg& s = segs[k];
    if (s.pinned) { if (!s.mapped) zc_out = false; }
    else s.mapped = hs_dev + s.off;
  }
  auto rp = [&](const Seg& s) -> const char* { return s.bytes ? ds + s.off : nullptr; };
  auto wp = [&](const Seg& s) -> char* { return zc_out ? (char*)s.mapped : ds + s.off; };
  int rc = jmpc_collision(h, B, (const int*)rp(s_cid), (const int*)rp(s_idx), (const double*)rp(s_v),
                          (const double*)rp(s_obs), n_obs, frame_window, margin, horizon_s, (const double*)rp(s_prm),
                          (int*)wp(s_flag), (int*)wp(s_len), (void*)st);
  if (rc) return rc;
  if (!zc_out)
    for (int k = first_out; k < ns; ++k)
      CK(cudaMemcpyAsync(segs[k].pinned ? const_cast<void*>(segs[k].host) : (void*)(hs + segs[k].off), ds + segs[k].off,
                         segs[k].bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int k = first_out; k < ns; ++k)
    if (!segs[k].pinned) memcpy(const_cast<void*>(segs[k].host), hs + segs[k].off, segs[k].bytes);
  return 0;
}

int32_t jmpc_plant_step(jmpc_handle h, int32_t B, double* state, const double* a, const double* delta,
                        const double* params, void* stream) {
  if (!h) return fail("jmpc_plant_step: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_plant_step: B out of range");
  if (!state || !a || !delta) return fail("jmpc_plant_step: NULL array");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::ParamBlock d;
  memcpy(d.v, h->defaults, sizeof h->defaults);
  plant_step_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, state, a, delta, params, d);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

namespace {
void fill_episode_args(jmpc_handle h, jmpc::EpisodeArgs& a, int B, const int* course_id, const double* params) {
  memset(&a, 0, sizeof a);
  a.B = B; a.cx = h->d_cx; a.cy = h->d_cy; a.cyaw = h->d_cyaw; a.course_n = h->d_course_n;
  a.course_stride = h->course_stride; a.course_id = course_id; a.params = params;
  memcpy(a.defaults.v, h->defaults, sizeof h->defaults);
}
}  // namespace

int32_t jmpc_episode_pre(jmpc_handle h, int32_t B, const double* state, const int32_t* course_id,
                         const int32_t* course_len, const int32_t* target_ind, const int32_t* steps,
                         int32_t* agent_idx, int32_t* done, double goal_dis, double stop_speed, void* stream) {
  if (!h) return fail("jmpc_episode_pre: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_episode_pre: B out of range");
  if (!state || !course_len || !target_ind || !steps || !agent_idx || !done) return fail("jmpc_episode_pre: NULL array");
  if (h->n_courses < 1) return fail("jmpc_episode_pre: no courses uploaded (jmpc_set_courses)");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::EpisodeArgs a;
  fill_episode_args(h, a, B, course_id, nullptr);
  a.state = const_cast<double*>(state); a.course_len = const_cast<int*>(course_len);
  a.target_ind = const_cast<int*>(target_ind); a.steps = const_cast<int*>(steps);
  a.agent_idx = agent_idx; a.done = done; a.goal_dis = goal_dis; a.stop_speed = stop_speed;
  jmpc::episode_pre_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_episode_post(jmpc_handle h, int32_t B, double* state, const int32_t* course_id, const double* record,
                          const double* params, int32_t* target_ind, int32_t* steps, int32_t* done, double* di,
                          int32_t* warm, double* history, double t_now, void* stream) {
  if (!h) return fail("jmpc_episode_post: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_episode_post: B out of range");
  if (!state || !record || !target_ind || !steps || !done || !di) return fail("jmpc_episode_post: NULL array");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::EpisodeArgs a;
  fill_episode_args(h, a, B, course_id, params);
  a.state = state; a.record = record; a.target_ind = target_ind; a.steps = steps; a.done = done; a.di = di;
  a.warm = warm; a.history = history; a.t_now = t_now;
  jmpc::episode_post_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_episode_post_dev(jmpc_handle h, int32_t B, double* state, const int32_t* course_id, const double* record,
                              const double* params, int32_t* target_ind, int32_t* steps, int32_t* done, double* di,
                              int32_t* warm, double* history_base, int32_t history_rows, int32_t* flags_base,
                              const int32_t* flag, const int32_t* iter_dev, double dt_loop, void* stream) {
  if (!h) return fail("jmpc_episode_post_dev: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_episode_post_dev: B out of range");
  if (!state || !record || !target_ind || !steps || !done || !di || !iter_dev) return fail("jmpc_episode_post_dev: NULL array");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::EpisodeArgs a;
  fill_episode_args(h, a, B, course_id, params);
  a.state = state; a.record = record; a.target_ind = target_ind; a.steps = steps; a.done = done; a.di = di;
  a.warm = warm; a.history = nullptr; a.t_now = 0.0;
  a.iter_dev = iter_dev; a.history_base = history_base; a.history_rows = history_rows; a.flags_base = flags_base;
  a.flag = flag; a.dt_loop = dt_loop;
  jmpc::episode_post_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_counter_add(jmpc_handle h, int32_t* counter, int32_t delta, void* stream) {
  if (!h || !counter) return fail("jmpc_counter_add: NULL argument");
  CK(cudaSetDevice(h->device));
  jmpc::counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter, delta);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_episode_outcomes(jmpc_handle h, int32_t B, const double* state, const int32_t* course_id,
                              const double* obstacles, int32_t n_obs, const double* record, const double* di,
                              const int32_t* flag, const double* params, const int32_t* done, const int32_t* iter_dev,
                              int32_t initial, double* outcomes, double* obstacle_history, int32_t history_rows,
                              void* stream) {
  if (!h) return fail("jmpc_episode_outcomes: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_episode_outcomes: B out of range");
  if (n_obs < 0 || n_obs > jmpc::kMaxObstacles) return fail("jmpc_episode_outcomes: n_obs out of range");
  if (history_rows < 0) return fail("jmpc_episode_outcomes: negative history_rows");
  if (!state || !done || !outcomes) return fail("jmpc_episode_outcomes: NULL array");
  if (n_obs > 0 && !obstacles) return fail("jmpc_episode_outcomes: obstacles is NULL");
  if (!initial) {
    if (!record || !di || !iter_dev) return fail("jmpc_episode_outcomes: NULL step array");
    if (h->n_courses < 1) return fail("jmpc_episode_outcomes: no courses uploaded (jmpc_set_courses)");
  }
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::OutcomeArgs a;
  memset(&a, 0, sizeof a);
  a.B = B; a.n_obs = n_obs; a.initial = initial ? 1 : 0; a.history_rows = history_rows;
  a.cx = h->d_cx; a.cy = h->d_cy; a.cyaw = h->d_cyaw; a.course_stride = h->course_stride; a.course_id = course_id;
  a.params = params;
  memcpy(a.defaults.v, h->defaults, sizeof h->defaults);
  a.off_front = h->off_front; a.off_rear = h->off_rear; a.radius = h->radius;
  a.state = state; a.obstacles = obstacles; a.record = record; a.di = di; a.flag = flag; a.done = done;
  a.iter_dev = iter_dev; a.outcomes = outcomes; a.obstacle_history = obstacle_history;
  jmpc::episode_outcome_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_scene_exchange(jmpc_handle h, int32_t B, int32_t k, int32_t n_extra, const double* state,
                            const double* record, const double* di, const double* params, const int32_t* done,
                            const int32_t* steps, const double* extras, double* obstacles_out, void* stream) {
  if (!h) return fail("jmpc_scene_exchange: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_scene_exchange: B out of range");
  if (k < 1 || B % k != 0) return fail("jmpc_scene_exchange: B must be a multiple of k >= 1");
  if (n_extra < 0 || (k - 1) + n_extra > jmpc::kMaxObstacles)
    return fail("jmpc_scene_exchange: (k - 1) + n_extra must be in [0, 8]");
  if (!state || !record || !di || !done || !steps || !obstacles_out) return fail("jmpc_scene_exchange: NULL array");
  if (n_extra > 0 && !extras) return fail("jmpc_scene_exchange: extras is NULL");
  const int n_obs = (k - 1) + n_extra;
  if (B == 0 || n_obs == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::ParamBlock defaults;
  memcpy(defaults.v, h->defaults, sizeof h->defaults);
  const int count = B * n_obs;
  jmpc::scene_exchange_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      count, k, n_obs, state, record, di, params, defaults, done, steps, extras, obstacles_out);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_scene_plans(jmpc_handle h, int32_t B, int32_t k, int32_t T, const double* oa, const double* od,
                         const int32_t* warm, const int32_t* done, const double* params, const double* obstacles,
                         int32_t n_obs, double* plans_out, void* stream) {
  if (!h) return fail("jmpc_scene_plans: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_scene_plans: B out of range");
  if (k < 1 || B % k != 0) return fail("jmpc_scene_plans: B must be a multiple of k >= 1");
  if (T < 2) return fail("jmpc_scene_plans: T must be >= 2");
  if (n_obs < k - 1 || n_obs > jmpc::kMaxObstacles) return fail("jmpc_scene_plans: n_obs must be in [k - 1, 8]");
  if (B == 0 || k == 1) return 0;
  if (!oa || !od || !warm || !done || !obstacles || !plans_out) return fail("jmpc_scene_plans: NULL array");
  CK(cudaSetDevice(h->device));
  jmpc::ParamBlock defaults;
  memcpy(defaults.v, h->defaults, sizeof h->defaults);
  const long long count = (long long)B * (k - 1) * (T - 1);
  if (count > INT32_MAX) return fail("jmpc_scene_plans: B * (k - 1) * (T - 1) too large");
  jmpc::scene_plans_kernel<<<(unsigned)((count + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      (int)count, k, T, n_obs, oa, od, warm, done, params, defaults, obstacles, plans_out);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_right_of_way_init(jmpc_handle h, int32_t B, int32_t k, const int32_t* course_id, const double* junction,
                               int32_t n_junction, int32_t* zone_out, void* stream) {
  if (!h) return fail("jmpc_right_of_way_init: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_right_of_way_init: B out of range");
  if (k < 1 || B % k != 0) return fail("jmpc_right_of_way_init: B must be a multiple of k >= 1");
  if (n_junction != 1 && n_junction != B / k) return fail("jmpc_right_of_way_init: n_junction must be 1 or B / k");
  if (!junction || !zone_out) return fail("jmpc_right_of_way_init: NULL array");
  if (h->n_courses < 1) return fail("jmpc_right_of_way_init: no courses uploaded (jmpc_set_courses)");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::right_of_way_init_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(
      B, k, h->d_cx, h->d_cy, h->d_course_n, h->course_stride, h->n_courses, course_id, junction,
      n_junction > 1 ? 1 : 0, zone_out);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_right_of_way(jmpc_handle h, int32_t B, int32_t k, int32_t rule, const int32_t* agent_idx,
                          const int32_t* done, const double* params, const int32_t* zone, const double* priority,
                          int32_t* consider_out, void* stream) {
  if (!h) return fail("jmpc_right_of_way: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_right_of_way: B out of range");
  if (k < 2 || k > jmpc::kMaxObstacles + 1 || B % k != 0)
    return fail("jmpc_right_of_way: B must be a multiple of k in [2, 9]");
  if (rule != JMPC_ROW_FIXED && rule != JMPC_ROW_FIRST_COME) return fail("jmpc_right_of_way: unknown rule");
  if (!agent_idx || !done || !consider_out) return fail("jmpc_right_of_way: NULL array");
  if (rule == JMPC_ROW_FIXED && !priority) return fail("jmpc_right_of_way: the fixed rule needs priority");
  if (rule == JMPC_ROW_FIRST_COME && !zone) return fail("jmpc_right_of_way: the first-come rule needs zone");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::ParamBlock defaults;
  memcpy(defaults.v, h->defaults, sizeof h->defaults);
  jmpc::right_of_way_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, k, rule, agent_idx, done, params,
                                                                               defaults, zone, priority, consider_out);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_scene_init(jmpc_handle h, int32_t B, int32_t k, int32_t* done, void* stream) {
  if (!h) return fail("jmpc_scene_init: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_scene_init: B out of range");
  if (k < 1 || B % k != 0) return fail("jmpc_scene_init: B must be a multiple of k >= 1");
  if (!done) return fail("jmpc_scene_init: NULL array");
  if (B == 0 || k == 1) return 0;
  CK(cudaSetDevice(h->device));
  const int n_scenes = B / k;
  jmpc::scene_init_kernel<<<(n_scenes + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_scenes, k, done);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_obstacle_step(jmpc_handle h, int32_t B, int32_t n_obs, double* obstacles, const int32_t* done,
                           double dt, void* stream) {
  if (!h) return fail("jmpc_obstacle_step: NULL handle");
  if (B < 0 || B > h->max_B || n_obs < 0) return fail("jmpc_obstacle_step: size out of range");
  if (B == 0 || n_obs == 0) return 0;
  if (!obstacles) return fail("jmpc_obstacle_step: NULL array");
  CK(cudaSetDevice(h->device));
  const int count = B * n_obs;
  jmpc::obstacle_step_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(count, obstacles, done, n_obs, dt,
                                                                                   h->defaults[JMPC_P_L]);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_scripted_obstacle_step(jmpc_handle h, int32_t B, int32_t n_obs, const double* script, double* model,
                                    double* obstacles, const int32_t* done, int32_t advance, void* stream) {
  if (!h) return fail("jmpc_scripted_obstacle_step: NULL handle");
  if (B < 0 || B > h->max_B || n_obs < 0) return fail("jmpc_scripted_obstacle_step: size out of range");
  if (B == 0 || n_obs == 0) return 0;
  if (!script || !model || !obstacles) return fail("jmpc_scripted_obstacle_step: NULL array");
  CK(cudaSetDevice(h->device));
  const int count = B * n_obs;
  jmpc::scripted_obstacle_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      count, script, model, obstacles, done, n_obs, advance, h->defaults[JMPC_P_L]);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int32_t jmpc_plan_host(int32_t device, int32_t B, int32_t n_mp, int32_t n_pts, int32_t n_cc, const double* mp_pts,
                       const double* mp_len, const double* mp_cc, int32_t n_scenes, int32_t max_obs, const double* hp,
                       const int32_t* hp_n, const int32_t* n_obs, const int32_t* scene_id, const double* start,
                       const double* goal_point, const double* goal_area, const double* allowed, const double* weights,
                       int32_t max_expansions, int32_t max_path, int32_t max_log, double* cost, int32_t* status,
                       int32_t* n_path, double* path, int32_t* path_mp, int32_t* n_traj, double* traj,
                       int32_t* expansions, double* log, double* kernel_ms) {
  if (!mp_pts || !mp_len || !mp_cc || !hp || !hp_n || !n_obs || !start || !goal_point || !goal_area || !allowed || !weights ||
      !cost || !status || !n_path || !path || !path_mp || !n_traj || !traj || !expansions)
    return fail("jmpc_plan_host: NULL argument");
  if (B < 0 || n_mp < 1 || n_mp > 32 || n_pts < 2 || n_cc < 1 || n_scenes < 1 || max_obs < 0)
    return fail("jmpc_plan_host: size out of range (1 <= n_mp <= 32)");
  if (max_expansions < 1 || max_path < 2 || max_log < 0) return fail("jmpc_plan_host: limits out of range");
  for (int s = 0; s < n_scenes; ++s) {
    if (n_obs[s] < 0 || n_obs[s] > max_obs) return fail("jmpc_plan_host: n_obs out of range");
    for (int o = 0; o < n_obs[s]; ++o)
      if (hp_n[(size_t)s * max_obs + o] < 1 || hp_n[(size_t)s * max_obs + o] > JMPC_PLAN_MAX_HP)
        return fail("jmpc_plan_host: hp_n out of range");
  }
  if (scene_id)
    for (int b = 0; b < B; ++b)
      if (scene_id[b] < 0 || scene_id[b] >= n_scenes) return fail("jmpc_plan_host: scene_id out of range");
  if (B == 0) return 0;
  int count = 0;
  CK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail("jmpc_plan_host: no such CUDA device");
  CK(cudaSetDevice(device));
  jmpc::PlanArgs a;
  memset(&a, 0, sizeof a);
  a.B = B; a.n_mp = n_mp; a.n_pts = n_pts; a.n_cc = n_cc; a.max_obs = max_obs; a.n_scenes = n_scenes;
  a.max_expansions = max_expansions; a.max_path = max_path; a.max_traj = (max_path - 1) * (n_pts - 1); a.max_log = max_log;
  a.pool_cap = max_expansions * n_mp + 1;
  int ts = 64;
  while (ts < 2 * max_expansions + 2) ts <<= 1;
  a.table_size = ts;
  const size_t b = (size_t)B;
  // one device block [inputs | workspace | results]
  size_t off = 0;
  auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
  const size_t hp_doubles = (size_t)n_scenes * max_obs * JMPC_PLAN_MAX_HP * 3;
  const size_t o_pts = seg((size_t)n_mp * n_pts * 3 * 8), o_len = seg((size_t)n_mp * 8), o_cc = seg((size_t)n_mp * n_cc * 2 * 8);
  const size_t o_hp = seg(hp_doubles * 8), o_hpn = seg((size_t)n_scenes * max_obs * 4 + 4), o_nobs = seg((size_t)n_scenes * 4);
  const size_t o_sid = seg(b * 4), o_start = seg(b * 24), o_goal = seg(b * 24), o_area = seg(b * 32), o_allow = seg(b * 8);
  const size_t o_w = seg(b * 72);
  const size_t o_pool = seg(b * a.pool_cap * sizeof(jmpc::PlanNode)), o_heap = seg(b * a.pool_cap * 4), o_tab = seg(b * ts * 4);
  const size_t o_res = off;
  const size_t o_cost = seg(b * 8), o_status = seg(b * 4), o_npath = seg(b * 4), o_path = seg(b * max_path * 24);
  const size_t o_pmp = seg(b * max_path * 4), o_ntraj = seg(b * 4), o_traj = seg(b * a.max_traj * 24), o_exp = seg(b * 4);
  const size_t o_log = seg(log ? b * max_log * 40 : 0);
  char* d = nullptr;
  cudaError_t err = cudaMalloc(&d, off);
  if (err != cudaSuccess) return fail("jmpc_plan_host: workspace allocation failed (lower max_expansions or B)", err);
  cudaStream_t st = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  int rc = 0;
  auto up = [&](size_t o, const void* src, size_t bytes) {
    if (!rc && bytes && cudaMemcpyAsync(d + o, src, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = fail("jmpc_plan_host: upload failed");
  };
  auto down = [&](void* dst, size_t o, size_t bytes) {
    if (!rc && bytes && cudaMemcpyAsync(dst, d + o, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = fail("jmpc_plan_host: download failed");
  };
  if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&e0) != cudaSuccess ||
      cudaEventCreate(&e1) != cudaSuccess)
    rc = fail("jmpc_plan_host: stream / event creation failed");
  up(o_pts, mp_pts, (size_t)n_mp * n_pts * 24); up(o_len, mp_len, (size_t)n_mp * 8); up(o_cc, mp_cc, (size_t)n_mp * n_cc * 16);
  up(o_hp, hp, hp_doubles * 8); up(o_hpn, hp_n, (size_t)n_scenes * max_obs * 4); up(o_nobs, n_obs, (size_t)n_scenes * 4);
  if (scene_id) up(o_sid, scene_id, b * 4);
  up(o_start, start, b * 24); up(o_goal, goal_point, b * 24); up(o_area, goal_area, b * 32); up(o_allow, allowed, b * 8);
  up(o_w, weights, b * 72);
  if (!rc) {
    a.mp_pts = (const double*)(d + o_pts); a.mp_len = (const double*)(d + o_len); a.mp_cc = (const double*)(d + o_cc);
    a.hp = (const double*)(d + o_hp); a.hp_n = (const int*)(d + o_hpn); a.n_obs = (const int*)(d + o_nobs);
    a.scene_id = scene_id ? (const int*)(d + o_sid) : nullptr;
    a.start = (const double*)(d + o_start); a.goal_point = (const double*)(d + o_goal); a.goal_area = (const double*)(d + o_area);
    a.allowed = (const double*)(d + o_allow); a.weights = (const double*)(d + o_w);
    a.pool = (jmpc::PlanNode*)(d + o_pool); a.heap = (int*)(d + o_heap); a.table = (int*)(d + o_tab);
    a.cost = (double*)(d + o_cost); a.status = (int*)(d + o_status); a.n_path = (int*)(d + o_npath); a.path = (double*)(d + o_path);
    a.path_mp = (int*)(d + o_pmp); a.n_traj = (int*)(d + o_ntraj); a.traj = (double*)(d + o_traj); a.expansions = (int*)(d + o_exp);
    a.log = log ? (double*)(d + o_log) : nullptr;
    if (cudaMemsetAsync(d + o_res, 0, off - o_res, st) != cudaSuccess) rc = fail("jmpc_plan_host: memset failed");
  }
  if (!rc) {
    cudaEventRecord(e0, st);
    jmpc::plan_kernel<<<(B + 3) / 4, 128, 0, st>>>(a);
    cudaEventRecord(e1, st);
    if ((err = cudaGetLastError()) != cudaSuccess) rc = fail("jmpc_plan_host: launch failed", err);
  }
  down(cost, o_cost, b * 8); down(status, o_status, b * 4); down(n_path, o_npath, b * 4); down(path, o_path, b * max_path * 24);
  down(path_mp, o_pmp, b * max_path * 4); down(n_traj, o_ntraj, b * 4); down(traj, o_traj, b * a.max_traj * 24);
  down(expansions, o_exp, b * 4);
  if (log) down(log, o_log, b * max_log * 40);
  if (!rc && (err = cudaStreamSynchronize(st)) != cudaSuccess) rc = fail("jmpc_plan_host: kernel failed", err);
  if (!rc && kernel_ms) { float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1); *kernel_ms = ms; }
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (st) cudaStreamDestroy(st);
  cudaFree(d);
  return rc;
}

}  // extern "C"

struct jmpc_planner_s {
  int device = 0, max_B = 0, n_mp = 0, n_pts = 0, n_cc = 0;
  int max_expansions = 0, max_path = 0, max_log = 0, pool_cap = 0, table_size = 0;
  double *d_pts = nullptr, *d_len = nullptr, *d_cc = nullptr;                    // primitives
  double* d_hp = nullptr; int* d_hp_n = nullptr; int* d_n_obs = nullptr;           // scenes
  size_t hp_bytes = 0, hpn_bytes = 0, nobs_bytes = 0;
  int n_scenes = 0, max_obs = 0;
  jmpc::PlanNode* d_pool = nullptr; int* d_heap = nullptr; int* d_table = nullptr; // per-search workspace
};

namespace {
// (re)allocate *p to hold `bytes` when it is smaller
template <typename T>
int grow(T** p, size_t* have, size_t bytes) {
  if (bytes <= *have) return 0;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  CK(cudaMalloc(p, bytes));
  *have = bytes;
  return 0;
}
}  // namespace

extern "C" {

int32_t jmpc_planner_create(int32_t device, int32_t max_B, int32_t n_mp, int32_t n_pts, int32_t n_cc, const double* mp_pts,
                            const double* mp_len, const double* mp_cc, int32_t max_expansions, int32_t max_path,
                            int32_t max_log, jmpc_planner* out) {
  if (!out) return fail("jmpc_planner_create: out is NULL");
  *out = nullptr;
  if (!mp_pts || !mp_len || !mp_cc) return fail("jmpc_planner_create: NULL argument");
  if (max_B < 1 || n_mp < 1 || n_mp > 32 || n_pts < 2 || n_cc < 1)
    return fail("jmpc_planner_create: size out of range (max_B >= 1, 1 <= n_mp <= 32)");
  if (max_expansions < 1 || max_path < 2 || max_log < 0) return fail("jmpc_planner_create: limits out of range");
  int count = 0;
  CK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail("jmpc_planner_create: no such CUDA device");
  CK(cudaSetDevice(device));
  jmpc_planner p = new (std::nothrow) jmpc_planner_s();
  if (!p) return fail("jmpc_planner_create: out of host memory");
  p->device = device; p->max_B = max_B; p->n_mp = n_mp; p->n_pts = n_pts; p->n_cc = n_cc;
  p->max_expansions = max_expansions; p->max_path = max_path; p->max_log = max_log;
  p->pool_cap = max_expansions * n_mp + 1;                  // as jmpc_plan_host sizes them
  int ts = 64;
  while (ts < 2 * max_expansions + 2) ts <<= 1;
  p->table_size = ts;
  const size_t b = (size_t)max_B, pts = (size_t)n_mp * n_pts * 3, cc = (size_t)n_mp * n_cc * 2;
  cudaError_t e;
  if ((e = cudaMalloc(&p->d_pts, pts * 8)) != cudaSuccess || (e = cudaMalloc(&p->d_len, (size_t)n_mp * 8)) != cudaSuccess ||
      (e = cudaMalloc(&p->d_cc, cc * 8)) != cudaSuccess ||
      (e = cudaMalloc(&p->d_pool, b * p->pool_cap * sizeof(jmpc::PlanNode))) != cudaSuccess ||
      (e = cudaMalloc(&p->d_heap, b * p->pool_cap * sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&p->d_table, b * ts * sizeof(int))) != cudaSuccess ||
      (e = cudaMemcpy(p->d_pts, mp_pts, pts * 8, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(p->d_len, mp_len, (size_t)n_mp * 8, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(p->d_cc, mp_cc, cc * 8, cudaMemcpyHostToDevice)) != cudaSuccess) {
    jmpc_planner_destroy(p);
    return fail("jmpc_planner_create: workspace allocation failed (lower max_B or max_expansions)", e);
  }
  *out = p;
  return 0;
}

int32_t jmpc_planner_destroy(jmpc_planner p) {
  if (!p) return 0;
  cudaSetDevice(p->device);
  cudaFree(p->d_pts); cudaFree(p->d_len); cudaFree(p->d_cc); cudaFree(p->d_hp); cudaFree(p->d_hp_n); cudaFree(p->d_n_obs);
  cudaFree(p->d_pool); cudaFree(p->d_heap); cudaFree(p->d_table);
  delete p;
  return 0;
}

int32_t jmpc_planner_set_scenes(jmpc_planner p, int32_t n_scenes, int32_t max_obs, const double* hp, const int32_t* hp_n,
                                const int32_t* n_obs) {
  if (!p || !hp || !hp_n || !n_obs) return fail("jmpc_planner_set_scenes: NULL argument");
  if (n_scenes < 1 || max_obs < 0) return fail("jmpc_planner_set_scenes: size out of range");
  for (int s = 0; s < n_scenes; ++s) {
    if (n_obs[s] < 0 || n_obs[s] > max_obs) return fail("jmpc_planner_set_scenes: n_obs out of range");
    for (int o = 0; o < n_obs[s]; ++o)
      if (hp_n[(size_t)s * max_obs + o] < 1 || hp_n[(size_t)s * max_obs + o] > JMPC_PLAN_MAX_HP)
        return fail("jmpc_planner_set_scenes: hp_n out of range");
  }
  CK(cudaSetDevice(p->device));
  CK(cudaDeviceSynchronize());                             // searches in flight may still read the old scenes
  const size_t hpd = (size_t)n_scenes * max_obs * JMPC_PLAN_MAX_HP * 3, hpn = (size_t)n_scenes * max_obs;
  if (grow(&p->d_hp, &p->hp_bytes, std::max<size_t>(hpd, 1) * 8) || grow(&p->d_hp_n, &p->hpn_bytes, std::max<size_t>(hpn, 1) * 4) ||
      grow(&p->d_n_obs, &p->nobs_bytes, (size_t)n_scenes * 4))
    return -1;
  if (hpd) CK(cudaMemcpy(p->d_hp, hp, hpd * 8, cudaMemcpyHostToDevice));
  if (hpn) CK(cudaMemcpy(p->d_hp_n, hp_n, hpn * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(p->d_n_obs, n_obs, (size_t)n_scenes * 4, cudaMemcpyHostToDevice));
  p->n_scenes = n_scenes; p->max_obs = max_obs;
  return 0;
}

int32_t jmpc_plan(jmpc_planner p, int32_t B, const int32_t* scene_id, const double* start, const double* goal_point,
                  const double* goal_area, const double* allowed, const double* weights, double* cost, int32_t* status,
                  int32_t* n_path, double* path, int32_t* path_mp, int32_t* n_traj, double* traj, int32_t* expansions,
                  double* log, void* stream) {
  if (!p) return fail("jmpc_plan: NULL handle");
  if (B < 0 || B > p->max_B) return fail("jmpc_plan: B out of range (B <= max_B of jmpc_planner_create)");
  if (!start || !goal_point || !goal_area || !allowed || !weights || !cost || !status || !n_path || !path || !path_mp ||
      !n_traj || !traj || !expansions)
    return fail("jmpc_plan: NULL argument");
  if (p->n_scenes < 1) return fail("jmpc_plan: no scenes (jmpc_planner_set_scenes)");
  if (B == 0) return 0;
  CK(cudaSetDevice(p->device));
  cudaStream_t st = (cudaStream_t)stream;
  jmpc::PlanArgs a;
  memset(&a, 0, sizeof a);
  a.B = B; a.n_mp = p->n_mp; a.n_pts = p->n_pts; a.n_cc = p->n_cc; a.max_obs = p->max_obs; a.n_scenes = p->n_scenes;
  a.max_expansions = p->max_expansions; a.max_path = p->max_path; a.max_traj = (p->max_path - 1) * (p->n_pts - 1);
  a.max_log = log ? p->max_log : 0;
  a.pool_cap = p->pool_cap; a.table_size = p->table_size;
  a.mp_pts = p->d_pts; a.mp_len = p->d_len; a.mp_cc = p->d_cc;
  a.hp = p->d_hp; a.hp_n = p->d_hp_n; a.n_obs = p->d_n_obs;
  a.scene_id = scene_id; a.start = start; a.goal_point = goal_point; a.goal_area = goal_area; a.allowed = allowed;
  a.weights = weights;
  a.pool = p->d_pool; a.heap = p->d_heap; a.table = p->d_table;
  a.cost = cost; a.status = status; a.n_path = n_path; a.path = path; a.path_mp = path_mp; a.n_traj = n_traj;
  a.traj = traj; a.expansions = expansions; a.log = a.max_log ? log : nullptr;
  // the kernel writes path / trajectory / log rows only as far as a search got: clear them, as jmpc_plan_host does
  const size_t b = (size_t)B;
  CK(cudaMemsetAsync(cost, 0, b * 8, st)); CK(cudaMemsetAsync(status, 0, b * 4, st)); CK(cudaMemsetAsync(n_path, 0, b * 4, st));
  CK(cudaMemsetAsync(path, 0, b * p->max_path * 24, st)); CK(cudaMemsetAsync(path_mp, 0, b * p->max_path * 4, st));
  CK(cudaMemsetAsync(n_traj, 0, b * 4, st)); CK(cudaMemsetAsync(traj, 0, b * a.max_traj * 24, st));
  CK(cudaMemsetAsync(expansions, 0, b * 4, st));
  if (a.log) CK(cudaMemsetAsync(log, 0, b * a.max_log * 40, st));
  jmpc::plan_kernel<<<(B + 3) / 4, 128, 0, st>>>(a);
  CK(cudaGetLastError());
  return 0;
}

int32_t jmpc_set_courses_device(jmpc_handle h, int32_t n_courses, int32_t traj_stride, const int32_t* n_traj,
                                const double* traj, const int32_t* plan_status, double* dl_out, int32_t* course_ok,
                                void* stream) {
  if (!h || !n_traj || !traj || !dl_out || !course_ok) return fail("jmpc_set_courses_device: NULL argument");
  if (n_courses < 1 || n_courses > h->max_courses) return fail("jmpc_set_courses_device: n_courses out of range");
  if (traj_stride < 1) return fail("jmpc_set_courses_device: traj_stride must be positive");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  jmpc::IngestArgs a;
  a.n_courses = n_courses; a.traj_stride = traj_stride; a.max_N = h->max_N; a.course_stride = h->course_stride;
  a.n_traj = n_traj; a.traj = traj; a.plan_status = plan_status;
  a.cx = h->d_cx; a.cy = h->d_cy; a.cyaw = h->d_cyaw; a.course_n = h->d_course_n; a.dl = dl_out; a.ok = course_ok;
  jmpc::course_ingest_kernel<<<(n_courses + 3) / 4, 128, 0, st>>>(a);
  CK(cudaGetLastError());
  h->launches++;
  // the lengths decide the arc-table budget (and are what course_len reports): the call's one readback
  if (ensure_stage(h, (size_t)n_courses * sizeof(int))) return -1;
  CK(cudaMemcpyAsync(h->h_stage, h->d_course_n, (size_t)n_courses * sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const int* lens = (const int*)h->h_stage;
  h->course_n.assign(lens, lens + n_courses);
  h->n_courses = n_courses;
  h->have_cv = false;
  int max_n = 1;
  for (int c = 0; c < n_courses; ++c) max_n = std::max(max_n, h->course_n[c]);
  std::vector<long long> off;
  if (place_arc_tables(h, off)) return -1;
  CK(cudaMemcpyAsync(h->d_arc_off, off.data(), (size_t)n_courses * sizeof(long long), cudaMemcpyHostToDevice, st));
  const unsigned gy = (unsigned)std::min(n_courses, 65535);
  if (h->d_arc) {
    jmpc::arc_tables_kernel<<<dim3((max_n + 63) / 64, gy), 64, 0, st>>>(n_courses, h->course_stride, h->d_course_n,
                                                                      h->d_arc_off, h->d_cx, h->d_cy, h->d_arc);
    CK(cudaGetLastError());
    h->launches++;
  }
  jmpc::circle_tables_kernel<<<dim3((max_n + 127) / 128, gy), 128, 0, st>>>(
      n_courses, h->course_stride, h->d_course_n, h->d_cx, h->d_cy, h->d_cyaw, h->off_front, h->off_rear, h->d_ccfx,
      h->d_ccfy, h->d_ccrx, h->d_ccry);
  CK(cudaGetLastError());
  h->launches++;
  // the *_host entry points run on the handle's own stream: order it after the tables without a host wait
  cudaEvent_t ev;
  CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  cudaError_t e = cudaEventRecord(ev, st);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(h->own_stream, ev, 0);
  cudaEventDestroy(ev);
  if (e != cudaSuccess) return fail("jmpc_set_courses_device: stream ordering failed", e);
  return 0;
}

int32_t jmpc_get_courses(jmpc_handle h, int32_t first, int32_t n, int32_t stride, int32_t* len, double* cx, double* cy,
                         double* cyaw) {
  if (!h || !len) return fail("jmpc_get_courses: NULL argument");
  const bool pts = cx || cy || cyaw;
  if (pts && !(cx && cy && cyaw)) return fail("jmpc_get_courses: give all of cx, cy, cyaw or none");
  if (first < 0 || n < 0 || first + n > h->n_courses) return fail("jmpc_get_courses: course range out of range");
  int width = 0;
  for (int k = 0; k < n; ++k) { len[k] = h->course_n[first + k]; width = std::max(width, len[k]); }
  if (!pts || n == 0) return 0;
  if (stride < width) return fail("jmpc_get_courses: stride shorter than a course");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  const size_t spitch = (size_t)h->course_stride * 8, dpitch = (size_t)stride * 8, off = (size_t)first * h->course_stride;
  CK(cudaMemcpy2D(cx, dpitch, h->d_cx + off, spitch, (size_t)width * 8, n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(cy, dpitch, h->d_cy + off, spitch, (size_t)width * 8, n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(cyaw, dpitch, h->d_cyaw + off, spitch, (size_t)width * 8, n, cudaMemcpyDeviceToHost));
  for (int k = 0; k < n; ++k) {
    const size_t o = (size_t)k * stride + len[k], cnt = (size_t)stride - len[k];
    memset(cx + o, 0, cnt * 8); memset(cy + o, 0, cnt * 8); memset(cyaw + o, 0, cnt * 8);
  }
  return 0;
}

int32_t jmpc_get_arc_tables(jmpc_handle h, int32_t first, int32_t n, int32_t* has_table) {
  if (!h || !has_table) return fail("jmpc_get_arc_tables: NULL argument");
  if (first < 0 || n < 0 || first + n > h->n_courses) return fail("jmpc_get_arc_tables: course range out of range");
  for (int k = 0; k < n; ++k) has_table[k] = h->arc_has[first + k];
  return 0;
}

int32_t jmpc_episode_init_from_courses(jmpc_handle h, int32_t B, const int32_t* course_id, const int32_t* course_ok,
                                       const double* dl, double* state, double* params, int32_t* done, void* stream) {
  if (!h) return fail("jmpc_episode_init_from_courses: NULL handle");
  if (B < 0 || B > h->max_B) return fail("jmpc_episode_init_from_courses: B out of range");
  if (!state || !done) return fail("jmpc_episode_init_from_courses: NULL array");
  if (h->n_courses < 1) return fail("jmpc_episode_init_from_courses: no courses uploaded");
  if (B == 0) return 0;
  CK(cudaSetDevice(h->device));
  jmpc::episode_init_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      B, h->n_courses, h->course_stride, course_id, course_ok, dl, h->d_cx, h->d_cy, h->d_cyaw, state, params, done);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int64_t jmpc_launch_count(jmpc_handle h) { return h ? h->launches : 0; }

int32_t jmpc_debug_linalg(jmpc_handle h, int32_t n, const double* A, const double* b, const double* x, double* sol,
                          double* prod) {
  return jmpc_debug_linalg_g(h, n, 32, 0, A, b, x, sol, prod);
}

int32_t jmpc_debug_linalg_g(jmpc_handle h, int32_t n, int32_t group_lanes, int32_t which, const double* A,
                            const double* b, const double* x, double* sol, double* prod) {
  if (!h || !A || !b || !x || !sol || !prod) return fail("jmpc_debug_linalg: NULL argument");
  if (n < 1 || n > 2 * JMPC_MAX_T) return fail("jmpc_debug_linalg: n out of range");
  if (group_lanes != 16 && group_lanes != 32) return fail("jmpc_debug_linalg: group_lanes must be 16 or 32");
  const int groups = 32 / group_lanes;
  if (which < 0 || which >= groups) return fail("jmpc_debug_linalg: no such lane group");
  CK(cudaSetDevice(h->device));
  const size_t nn = (size_t)n * n;
  const size_t in_doubles = nn + 2 * (size_t)n, out_doubles = 4 * (size_t)n + 2;
  if (ensure_stage(h, (in_doubles + out_doubles) * sizeof(double))) return -1;
  // everything on the handle's own stream, through its pinned block
  double* hs = (double*)h->h_stage;
  double* d = (double*)h->d_stage;
  memcpy(hs, A, nn * sizeof(double)); memcpy(hs + nn, b, n * sizeof(double)); memcpy(hs + nn + n, x, n * sizeof(double));
  double *dA = d, *db = dA + nn, *dx = db + n, *dsol = dx + n, *dprod = dsol + 2 * n;
  int* dok = (int*)(dprod + 2 * n);
  cudaStream_t st = h->own_stream;
  CK(cudaMemcpyAsync(d, hs, in_doubles * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(dsol, 0xff, out_doubles * sizeof(double), st));          // NaN where the kernel writes nothing
  const int nb = jmpc::nblk(n);
  const size_t smem = (size_t)groups * (jmpc::tiles_doubles(n) + 8 * nb) * sizeof(double) +
                      jmpc::chol_lut_bytes(nb) + 16;
  if (group_lanes == 32) jmpc::linalg_selftest_kernel<32><<<1, 32, smem, st>>>(n, which, dA, db, dx, dsol, dprod, dok);
  else jmpc::linalg_selftest_kernel<16><<<1, 32, smem, st>>>(n, which, dA, db, dx, dsol, dprod, dok);
  CK(cudaGetLastError());
  h->launches++;
  CK(cudaMemcpyAsync(hs + in_doubles, dsol, out_doubles * sizeof(double), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memcpy(sol, hs + in_doubles, 2 * (size_t)n * sizeof(double));
  memcpy(prod, hs + in_doubles + 2 * n, 2 * (size_t)n * sizeof(double));
  int ok = 0;
  memcpy(&ok, hs + in_doubles + 4 * n, sizeof(int));
  return ok == 1 ? 0 : 1;
}

int32_t jmpc_measure_fma_peak(jmpc_handle h, double* fp64_tflops, double* fp32_tflops) {
  if (!h || !fp64_tflops || !fp32_tflops) return fail("jmpc_measure_fma_peak: NULL argument");
  CK(cudaSetDevice(h->device));
  if (measure_fma<double>(h, fp64_tflops)) return -1;
  if (measure_fma<float>(h, fp32_tflops)) return -1;
  return 0;
}

}  // extern "C"
