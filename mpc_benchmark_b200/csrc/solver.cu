// libmpcb200.so — CUDA kernels (sm_100a) + the C-ABI of include/mpcb200.h.
//
// One solver handle = one batch of independent MPC instances on one GPU.  Kernels:
//   k_init         CTA / instance   run() prologue (warm start copy, x0 forcing, BCL reset)
//   k_eval<D>      CTA / (instance, knot)   per-knot evaluation (+ derivatives, LQ assembly when D)
//   k_decide_eval  CTA / instance   reductions + BCL outer-loop logic
//   k_riccati      CTA / instance   proximal Riccati backward + forward, directional derivative
//   k_apply_step   CTA / instance   trial point x (+) alpha dx
//   k_decide_ls    CTA / instance   Armijo test / next alpha / accept
// There is deliberately NO CPU fallback: every entry point fails if CUDA is unavailable.
#include "driver.hpp"
#include "ws_alloc.hpp"
#include "rbd_terms.cuh"
#include "gait_host.hpp"
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

using namespace mpcdev;

static thread_local std::string g_err;
static int fail(const std::string &m) { g_err = m; return 1; }
#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_));          \
  } while (0)

// ------------------------------------------------------------------ kernels
__global__ void k_init(Ws w, const double *xs_in, const double *us_in, int max_iters, int first) { init_instance(w, first + blockIdx.x, xs_in, us_in, max_iters); }

// Evaluation kernel launch shape: G knots per CTA (one group of TH threads each, own shared-memory slice and named barrier).
// The groups of a CTA start together and run the same instruction stream, which is what keeps the (large, mostly
// straight-line) evaluation code from being fetched G times per SM: ncu showed 59 % instruction-cache hits and
// "no instruction" as the second stall reason with one knot per CTA.
template <int KIND, bool DERIV> struct EvalShape {
  // full-dynamics derivative pass: FOUR knots of 96 threads per SM (same 384 threads / register budget as three of 128; the tangent
  // matrices live in the L2-resident global scratch, which brings a knot's shared memory under 56 KB).  Values-only passes (full /
  // kinodynamic): five knots of 96 threads in one CTA measured 16 % faster than 2 CTAs of 2 x 128.
  static constexpr int TH = (KIND == MPC_KIND_CENT) ? 32 : (KIND == MPC_KIND_KINO && DERIV) ? 128 : 96;
  static constexpr int G = (KIND == MPC_KIND_CENT) ? 4 : DERIV ? ((KIND == MPC_KIND_FULL) ? 4 : 3) : 5; // knots per CTA
  static constexpr size_t raw = sizeof(typename KindTraits<KIND>::template EvalWs<DERIV>);
  static constexpr size_t slice = (raw + 15) / 16 * 16;
  static_assert(G * slice <= 232448, "evaluation groups exceed the 227 KB opt-in shared memory");
};
template <int KIND, bool DERIV> __global__ void __launch_bounds__(EvalShape<KIND, DERIV>::TH * EvalShape<KIND, DERIV>::G, 1)
k_eval(Ws w, const int32_t *list, int nitems) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T1 = w.T + 1;
  const int item = blockIdx.x * EvalShape<KIND, DERIV>::G + threadIdx.y;
  if (item >= nitems) return;
  const int b = list[item / T1], k = item % T1;
  eval_dispatch<KIND, DERIV>(w, b, k, smem_raw + threadIdx.y * EvalShape<KIND, DERIV>::slice);
}
template <int KIND, bool DERIV> static void launch_eval(const Ws &w, const int32_t *list, int nitems, cudaStream_t s) {
  using Sh = EvalShape<KIND, DERIV>;
  k_eval<KIND, DERIV><<<(nitems + Sh::G - 1) / Sh::G, dim3(Sh::TH, Sh::G), Sh::G * Sh::slice, s>>>(w, list, nitems);
}

__global__ void k_decide_eval(Ws w, const int32_t *list, int32_t *next_eval) {
  __shared__ double red[8];
  decide_eval(w, list[blockIdx.x], red, next_eval);
}

// ROLLOUT_NONLINEAR: nonlinear forward rollout and the complete Armijo linesearch of one instance per CTA (one evaluation group:
// the knots are visited in sequence, each trial state is produced by the previous knot's dynamics)
template <int KIND> struct RolloutShape {
  static constexpr int TH = EvalShape<KIND, false>::TH;
  static constexpr size_t smem = EvalShape<KIND, false>::slice + 256 * sizeof(double);
};
template <int KIND> __global__ void __launch_bounds__(RolloutShape<KIND>::TH) k_rollout_ls(Ws w, const int32_t *list, int32_t *next_eval) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red[8];
  rollout_linesearch<KIND>(w, list[blockIdx.x], smem_raw, reinterpret_cast<double *>(smem_raw + EvalShape<KIND, false>::slice), red, next_eval);
}

template <int KIND> __global__ void __launch_bounds__(256) k_riccati(Ws w, const int32_t *list) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  riccati_dispatch<KIND>(w, list[blockIdx.x], reinterpret_cast<double *>(smem_raw));
}

__global__ void k_apply_step(Ws w, const int32_t *list) {
  if (blockIdx.x == 0 && threadIdx.x == 0) w.counters[0] = 0; // next linesearch list starts empty
  apply_step(w, list[blockIdx.x]);
}

__global__ void k_decide_ls(Ws w, const int32_t *list, int32_t *ls_out, int32_t *next_eval) {
  __shared__ double red[8];
  decide_ls(w, list[blockIdx.x], red, ls_out, next_eval);
}

// shift the horizon by one knot (replaceStageCircular / cycleAppend, fulldynamic_talos.py:496-497)
__global__ void k_cycle(Ws w, const mpc_knot_t *last) {
  const int b = blockIdx.x, nd = sizeof(mpc_knot_t) / 8;
  double *kn = reinterpret_cast<double *>(w.knots + (size_t)b * w.T);
  // serial over knots, parallel over the doubles of one knot: knot k <- knot k+1
  for (int k = 0; k + 1 < w.T; k++) {
    for (int i = threadIdx.x; i < nd; i += blockDim.x) kn[k * nd + i] = kn[(k + 1) * nd + i];
    __syncthreads();
  }
  for (int i = threadIdx.x; i < nd; i += blockDim.x) kn[(w.T - 1) * nd + i] = reinterpret_cast<const double *>(last + b)[i];
}

// rigid-body terms of the whole-body QPs for `count` states (rbd_terms.cuh): one 128-thread CTA per state
__global__ void __launch_bounds__(128) k_rbd_terms(const DevModel *model, const double *x, int count, double *M, double *nle, double *Jc, double *dJv, double *vf) {
  extern __shared__ double rbd_smem[];
  const int i = blockIdx.x;
  if (i >= count) return;
  FullWsT<false> &w = *reinterpret_cast<FullWsT<false> *>(rbd_smem);
  rbd_terms_group(*model, x + (size_t)i * (NQ + NV), w, M + (size_t)i * NV * NV, nle + (size_t)i * NV, Jc + (size_t)i * 12 * NV, dJv + (size_t)i * 12, vf + (size_t)i * 12);
}

// the same terms plus the IKID QP's task terms (ikid_terms_group) of two frames for `count` states, one 128-thread CTA per state
struct IkidFrames {
  int32_t body[2];
  double place[24];
};
__global__ void __launch_bounds__(128) k_ikid_terms(const DevModel *model, const double *x, int count, const IkidFrames fr, double *M, double *nle, double *Jc,
                                                    double *dJv, double *Ag, double *dAgv, double *Jang, double *dJang) {
  extern __shared__ double rbd_smem[];
  const int i = blockIdx.x;
  if (i >= count) return;
  FullWsT<false> &w = *reinterpret_cast<FullWsT<false> *>(rbd_smem);
  ikid_terms_group(*model, x + (size_t)i * (NQ + NV), fr.body, fr.place, w, M + (size_t)i * NV * NV, nle + (size_t)i * NV, Jc + (size_t)i * 12 * NV,
                   dJv + (size_t)i * 12, Ag + (size_t)i * 6 * NV, dAgv + (size_t)i * 6, Jang + (size_t)i * 6 * NV, dJang + (size_t)i * 6);
}

// device-side gait bookkeeping (gait.cuh): one 128-thread CTA per robot rewrites its T knots and terminal block
__global__ void __launch_bounds__(128) k_gait_tick(Ws w, const GaitCfg *g, GaitRobot *robots, int t, const double *lf, const double *rf) {
  __shared__ double sm[16];
  const size_t b = blockIdx.x;
  gait_tick_group(*g, robots[b], t, lf ? lf + b * 12 : nullptr, rf ? rf + b * 12 : nullptr, w.knots + b * w.T, w.terms + b, sm);
}
// sole placements at the state the next tick starts from (the model prediction xs[1]): forward kinematics of the evaluation kernel
__global__ void __launch_bounds__(128) k_feet_of_prediction(Ws w, const DevModel *model, double *lf, double *rf) {
  extern __shared__ double rbd_smem[];
  const size_t b = blockIdx.x;
  FullWsT<false> &ws = *reinterpret_cast<FullWsT<false> *>(rbd_smem);
  const double *x = w.xs + b * ((size_t)w.T + 1) * w.nx + w.nx;
  PAR_FOR(i, NQ + NV) ws.x[i] = x[i];
  SYNC();
  mb_kinematics(*model, ws);
  PAR_FOR(i, 12) { lf[b * 12 + i] = ws.ofoot[i]; rf[b * 12 + i] = ws.ofoot[12 + i]; }
}

// fp64 peak micro-benchmark: 8 independent DFMA chains per thread
__global__ void k_dfma_peak(double *out, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// fp64 tensor-pipe peak: 8 independent DMMA.8x8x4 accumulator chains per warp (512 FLOP per warp instruction)
__global__ void k_dmma_peak(double *out, int iters) {
  double c[8][2];
#pragma unroll
  for (int j = 0; j < 8; j++) { c[j][0] = 0.0; c[j][1] = 0.0; }
  const double a = 1.0 + threadIdx.x * 1e-9, b = 1e-9 * (threadIdx.x & 7);
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int j = 0; j < 8; j++) dmma_8x8x4(c[j][0], c[j][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) s += c[j][0] + c[j][1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ------------------------------------------------------------------ host side
struct mpc_solver {
  int device = 0;
  Ws w{};
  DevModel *d_model = nullptr;
  DevModel h_model;
  std::vector<void *> allocs;
  double *d_xs_in = nullptr, *d_us_in = nullptr, *d_meas = nullptr;
  mpc_knot_t *d_last = nullptr;
  int32_t *h_counters = nullptr; // pinned
  cudaStream_t stream = nullptr, stream_copy = nullptr; // stream_copy: uploads / downloads of mpc_run_pipelined
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_part[2 * 8] = {};
  double *d_k0 = nullptr; // first feedback gains, packed (mpc_run_pipelined)
  InstState *h_st = nullptr; // pinned copy of the per-instance summaries (mpc_run_pipelined)
  int num_sms = 148;
  int last_launches = 0;
  float last_ms = 0;
  size_t bytes = 0;
  bool setup_done = false;
  // per-kernel-category device timing of the last run: 0 eval+derivatives, 1 riccati, 2 trial evaluation, 3 bookkeeping
  std::vector<cudaEvent_t> evpool;
  std::vector<int> evcat;
  double cat_ms[4] = {0, 0, 0, 0};
  int cat_launches[4] = {0, 0, 0, 0};
  bool profile = true;
  // device-side gait generator (mpc_gait_setup / mpc_gait_tick)
  GaitCfg *d_gait = nullptr;
  GaitRobot *d_gait_robots = nullptr;
  int8_t *d_gait_phases = nullptr;
  double *d_gait_urefs = nullptr, *d_feet = nullptr; // d_feet: [2][B][12]
  int gait_t = 0;
  bool gait_ready = false;
  int tail_mode = 0; // warm start of the knot appended by mpc_tick (mpc_set_tail_warmstart)
};

struct CudaBackend {
  mpc_solver *h;
  cudaStream_t s;
  cudaError_t err = cudaSuccess;
  void mark(int cat) { // event before a launch of category `cat`; the matching end event is the next mark (or run end)
    if (!h->profile) return;
    size_t i = h->evcat.size();
    if (i >= h->evpool.size()) { cudaEvent_t e; cudaEventCreate(&e); h->evpool.push_back(e); }
    cudaEventRecord(h->evpool[i], s);
    h->evcat.push_back(cat);
  }
  void reset_counters() { mark(3); cudaMemsetAsync(h->w.counters, 0, 4 * sizeof(int32_t), s); }
  void eval(bool d, const int32_t *list, int n) {
    const int nitems = n * (h->w.T + 1);
    mark(d ? 0 : 2);
    dispatch_kind(h->w.kind, [&](auto kind) {
      if (d) launch_eval<decltype(kind)::value, true>(h->w, list, nitems, s);
      else launch_eval<decltype(kind)::value, false>(h->w, list, nitems, s);
    });
  }
  void decide_eval(const int32_t *list, int n, int32_t *next_eval) { mark(3); k_decide_eval<<<n, 128, 0, s>>>(h->w, list, next_eval); }
  void riccati(const int32_t *list, int n) {
    mark(1);
    dispatch_kind(h->w.kind, [&](auto kind) {
      using K = KindTraits<decltype(kind)::value>;
      k_riccati<decltype(kind)::value><<<n, K::ric_threads(n, h->num_sms), K::ric_smem, s>>>(h->w, list);
    });
  }
  void rollout_ls(const int32_t *list, int n, int32_t *next_eval) {
    mark(2);
    dispatch_kind(h->w.kind, [&](auto kind) {
      using Sh = RolloutShape<decltype(kind)::value>;
      k_rollout_ls<decltype(kind)::value><<<n, Sh::TH, Sh::smem, s>>>(h->w, list, next_eval);
    });
    mark(-1);
  }
  void apply_step(const int32_t *list, int n) { mark(3); k_apply_step<<<n, 128, 0, s>>>(h->w, list); }
  void decide_ls(const int32_t *list, int n, int32_t *ls_out, int32_t *next_eval) { mark(3); k_decide_ls<<<n, 128, 0, s>>>(h->w, list, ls_out, next_eval); mark(-1); }
  void read_counters(int *c) {
    cudaError_t e = cudaMemcpyAsync(h->h_counters, h->w.counters, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { err = e; for (int i = 0; i < 4; i++) c[i] = 0; return; }
    for (int i = 0; i < 4; i++) c[i] = h->h_counters[i];
  }
};

// the SM count (Riccati launch shape) and the dynamic shared memory of the handle's kernels
static int set_kernel_attrs(mpc_solver *h) {
  { int dev = 0, sms = 0; if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) h->num_sms = sms; }
  return dispatch_kind(h->w.kind, [&](auto kind) {
    constexpr int KIND = decltype(kind)::value;
    CK(cudaFuncSetAttribute(k_eval<KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EvalShape<KIND, true>::G * EvalShape<KIND, true>::slice)));
    CK(cudaFuncSetAttribute(k_eval<KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EvalShape<KIND, false>::G * EvalShape<KIND, false>::slice)));
    CK(cudaFuncSetAttribute(k_rollout_ls<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RolloutShape<KIND>::smem));
    CK(cudaFuncSetAttribute(k_riccati<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, KindTraits<KIND>::ric_smem));
    return 0;
  });
}

// multipliers of every instance back to zero (a fresh solver.setup())
static int zero_multipliers(mpc_solver *h, cudaStream_t s) {
  const Ws &w = h->w;
  const size_t T1 = w.T + 1;
  CK(cudaMemsetAsync(w.vs, 0, w.B * T1 * w.nc * 8, s));
  CK(cudaMemsetAsync(w.lams, 0, w.B * T1 * w.n * 8, s));
  return 0;
}

// upload `last` (host, [batch]) and append it to the horizon (k_cycle), on the handle's stream
static int cycle_knots(mpc_solver *h, const mpc_knot_t *last) {
  if (!h->d_last) CK(cudaMalloc(&h->d_last, sizeof(mpc_knot_t) * h->w.B)); // owned by the handle, released in mpc_destroy
  CK(cudaMemcpyAsync(h->d_last, last, sizeof(mpc_knot_t) * h->w.B, cudaMemcpyHostToDevice, h->stream));
  k_cycle<<<h->w.B, 96, 0, h->stream>>>(h->w, h->d_last);
  return 0;
}

// device time of the last run (ev0 -> ev1, ev1 complete) and its per-category split from the marks of CudaBackend
static int read_run_times(mpc_solver *h) {
  CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  for (int c = 0; c < 4; c++) { h->cat_ms[c] = 0; h->cat_launches[c] = 0; }
  for (size_t i = 0; i + 1 < h->evcat.size(); i++) {
    int c = h->evcat[i];
    if (c < 0) continue;
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, h->evpool[i], h->evpool[i + 1]));
    h->cat_ms[c] += ms; h->cat_launches[c]++;
  }
  return 0;
}

extern "C" {

const char *mpc_last_error(void) { return g_err.c_str(); }

mpc_solver_t *mpc_create(const mpc_robot_t *robot, const mpc_config_t *cfg, int32_t batch, int32_t device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_err = "no CUDA device: libmpcb200 has no CPU fallback"; return nullptr; }
  if (!robot || !cfg) { g_err = "mpc_create: null robot / config"; return nullptr; }
  if (cfg->kind != MPC_KIND_FULL && cfg->kind != MPC_KIND_CENT && cfg->kind != MPC_KIND_KINO) { g_err = "unknown model kind"; return nullptr; }
  if (batch <= 0 || cfg->T <= 0) { g_err = "mpc_create: batch and horizon must be positive"; return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { g_err = "cudaSetDevice failed"; return nullptr; }
  mpc_solver *h = new mpc_solver;
  h->device = device;
  const char *err = nullptr;
  if (build_dev_model(robot, cfg, &h->h_model, &err)) { g_err = err; delete h; return nullptr; }
  // every failure below releases what was created so far through mpc_destroy (all members start null)
  auto bail = [&](const char *what, cudaError_t e) -> mpc_solver_t * { g_err = std::string(what) + ": " + cudaGetErrorString(e); mpc_destroy(h); return nullptr; };
  cudaError_t e;
  if ((e = cudaMalloc(&h->d_model, sizeof(DevModel))) != cudaSuccess) return bail("cudaMalloc(model)", e);
  if ((e = cudaMemcpy(h->d_model, &h->h_model, sizeof(DevModel), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy(model)", e);
  init_ws(h->w, *cfg, batch, h->d_model);
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaEventCreate(&h->ev0)) != cudaSuccess || (e = cudaEventCreate(&h->ev1)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaMallocHost(&h->h_counters, 4 * sizeof(int32_t))) != cudaSuccess) return bail("cudaMallocHost", e);
  if (set_kernel_attrs(h)) { std::string keep = g_err; mpc_destroy(h); g_err = keep; return nullptr; }
  return h;
}

void mpc_destroy(mpc_solver_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (void *p : h->allocs) cudaFree(p);
  for (cudaEvent_t e : h->evpool) cudaEventDestroy(e);
  if (h->d_xs_in) cudaFree(h->d_xs_in);
  if (h->d_us_in) cudaFree(h->d_us_in);
  if (h->d_meas) cudaFree(h->d_meas);
  if (h->d_last) cudaFree(h->d_last);
  if (h->d_model) cudaFree(h->d_model);
  if (h->h_counters) cudaFreeHost(h->h_counters);
  if (h->h_st) cudaFreeHost(h->h_st);
  if (h->d_k0) cudaFree(h->d_k0);
  cudaFree(h->d_gait); cudaFree(h->d_gait_robots); cudaFree(h->d_gait_phases); cudaFree(h->d_gait_urefs); cudaFree(h->d_feet);
  for (cudaEvent_t e : h->ev_part) if (e) cudaEventDestroy(e);
  if (h->stream_copy) cudaStreamDestroy(h->stream_copy);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int32_t mpc_setup(mpc_solver_t *h, const mpc_knot_t *knots, const mpc_term_t *terms, const double *x0) {
  CK(cudaSetDevice(h->device));
  Ws &w = h->w;
  const size_t T1 = w.T + 1;
  if (!h->setup_done) {
    bool ok = true;
    h->bytes = alloc_ws(w, [&](size_t bytes) -> void * {
      void *p = nullptr;
      if (!ok) return nullptr;
      if (cudaMalloc(&p, bytes ? bytes : 8) != cudaSuccess) { ok = false; return nullptr; }
      cudaMemsetAsync(p, 0, bytes ? bytes : 8, h->stream);
      h->allocs.push_back(p);
      return p;
    });
    if (!ok) return fail("cudaMalloc(workspace) failed: batch too large for this GPU");
    CK(cudaMalloc(&h->d_xs_in, w.B * T1 * w.nx * 8));
    CK(cudaMalloc(&h->d_us_in, (size_t)w.B * w.T * w.m * 8));
    h->setup_done = true;
  } else {
    // solver.setup() re-creates the workspace: multipliers restart from zero (fulldynamic_talos.py:539)
    if (zero_multipliers(h, h->stream)) return 1;
  }
  CK(cudaMemcpyAsync(w.knots, knots, sizeof(mpc_knot_t) * w.B * w.T, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(w.terms, terms, sizeof(mpc_term_t) * w.B, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(w.x0, x0, 8 * (size_t)w.B * w.nx, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_update_knots(mpc_solver_t *h, const mpc_knot_t *knots, int32_t first, int32_t count) {
  CK(cudaSetDevice(h->device));
  Ws &w = h->w;
  if (!h->setup_done) return fail("mpc_update_knots before mpc_setup");
  if (first < 0 || count < 0 || first + count > w.T) return fail("knot range out of bounds");
  // host layout [batch][count]
  CK(cudaMemcpy2DAsync(w.knots + first, sizeof(mpc_knot_t) * w.T, knots, sizeof(mpc_knot_t) * count, sizeof(mpc_knot_t) * count, w.B,
                       cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_update_terms(mpc_solver_t *h, const mpc_term_t *terms) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_update_terms before mpc_setup");
  CK(cudaMemcpyAsync(h->w.terms, terms, sizeof(mpc_term_t) * h->w.B, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_cycle(mpc_solver_t *h, const mpc_knot_t *last) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_cycle before mpc_setup");
  if (cycle_knots(h, last)) return 1;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// Warm-start shift of the multipliers by n knots (solver.cycleProblem without setup, kinodynamic_talos.py:488).  The constraint
// multipliers of the RUNNING knots and the co-states of x_1 .. x_T move n knots to the left, the vacated slots repeat the last
// running knot / the last co-state (as the trajectory warm start repeats its last knot); the terminal constraint's multiplier
// vs[T] and the initial-condition co-state lams[0] belong to constraints that do not move and stay where they are.  (Round 1
// shifted all T + 1 slots and zero-filled: that puts the terminal multiplier on a running knot and zeroes the last co-state —
// the kept-multiplier closed loop diverged within 40 ticks with it and is healthy with this, profiles/r2_closed_loop_kino_keep.txt.)
__global__ void k_shift_multipliers(Ws w, int n) {
  const size_t b = blockIdx.x, T1 = (size_t)w.T + 1;
  double *V = w.vs + b * T1 * w.nc, *L = w.lams + b * T1 * w.n;
  for (int k = 0; k < w.T; k++) {
    const int sv = (k + n < w.T) ? k + n : w.T - 1, sl = (k + 1 + n <= w.T) ? k + 1 + n : w.T;
    for (int i = threadIdx.x; i < w.nc; i += blockDim.x) V[(size_t)k * w.nc + i] = V[(size_t)sv * w.nc + i];
    for (int i = threadIdx.x; i < w.n; i += blockDim.x) L[(size_t)(k + 1) * w.n + i] = L[(size_t)sl * w.n + i];
    __syncthreads();
  }
}

int32_t mpc_shift_multipliers(mpc_solver_t *h, int32_t n) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_shift_multipliers before mpc_setup");
  if (n <= 0) return 0;
  k_shift_multipliers<<<h->w.B, 128, 0, h->stream>>>(h->w, n);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// swap in new model / weight constants without touching the workspace (same kind, horizon and batch)
int32_t mpc_reconfigure(mpc_solver_t *h, const mpc_robot_t *robot, const mpc_config_t *cfg) {
  CK(cudaSetDevice(h->device));
  if (cfg->kind != h->w.kind || cfg->T != h->w.T) return fail("mpc_reconfigure: kind / horizon must not change");
  const char *err = nullptr;
  if (build_dev_model(robot, cfg, &h->h_model, &err)) return fail(err);
  h->w.sc = default_consts(cfg->tol, cfg->mu_init, cfg->rollout);
  CK(cudaMemcpyAsync(h->d_model, &h->h_model, sizeof(DevModel), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_set_x0(mpc_solver_t *h, const double *x0) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_set_x0 before mpc_setup");
  CK(cudaMemcpyAsync(h->w.x0, x0, 8 * (size_t)h->w.B * h->w.nx, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

static int run_impl(mpc_solver *h, const double *d_xs, const double *d_us, int max_iters, cudaStream_t s, bool sync_events) {
  if (!h->setup_done) return fail("mpc_run before mpc_setup");
  CK(cudaEventRecord(h->ev0, s));
  h->evcat.clear();
  CudaBackend be{h, s};
  be.mark(3);
  k_init<<<h->w.B, 128, 0, s>>>(h->w, d_xs, d_us, max_iters, 0);
  h->last_launches = 1 + run_loop(be, h->w, max_iters, h->w.sc);
  be.mark(-1);
  CK(cudaEventRecord(h->ev1, s));
  if (be.err != cudaSuccess) return fail(std::string("kernel failure: ") + cudaGetErrorString(be.err));
  CK(cudaGetLastError());
  if (sync_events) {
    CK(cudaEventSynchronize(h->ev1));
    return read_run_times(h);
  }
  return 0;
}

// closed-loop warm start (fulldynamic_talos.py:532-536): xs <- xs[1:] + [xs[-1]], us <- us[1:] + [us[-1]], x0 <- measured state
// (x_meas, or the model prediction xs[1] when x_meas == nullptr: ideal plant)
// tail_mode 0: the reference scripts' warm start, us = us[1:] + [us[-1]] (fulldynamic_talos.py:534): the appended knot starts from the previous knot's control.
// tail_mode 1: it starts from the control of the NEAREST KNOT OF THE HORIZON WITH THE SAME CONTACT PHASE.  With mode 0 the first double-support knot after a
// swing phase inherits single-support torques (and the first swing knot double-support ones): under the rigid-contact full dynamics that is 36 N of cone
// violation at the end of the horizon, from which the one-iteration loop does not recover (DESIGN section 7); with mode 1 the same loop walks.
__global__ void k_shift_warmstart(Ws w, double *xs_in, double *us_in, const double *x_meas, int tail_mode) {
  const size_t b = blockIdx.x, T1 = (size_t)w.T + 1, T = w.T;
  const double *X = w.xs + b * T1 * w.nx, *U = w.us + b * T * w.m;
  double *Xo = xs_in + b * T1 * w.nx, *Uo = us_in + b * T * w.m;
  __shared__ int tail_src;
  if (threadIdx.x == 0) {
    int src = (int)T - 1; // index into the OLD trajectory: old knot T - 1 = new knot T - 2 (the copy of the reference)
    if (tail_mode == 1 && T >= 2) {
      const mpc_knot_t *kn = w.knots + b * T; // already rotated: slot j of the new horizon
      const double c0 = kn[T - 1].cs[0], c1 = kn[T - 1].cs[1];
      for (int j = (int)T - 2; j >= 0; j--)
        if (kn[j].cs[0] == c0 && kn[j].cs[1] == c1) { src = j + 1; break; } // new slot j = old knot j + 1
    }
    tail_src = src;
  }
  __syncthreads();
  for (size_t i = threadIdx.x; i < T1 * w.nx; i += blockDim.x) { size_t k = i / w.nx, c = i % w.nx; Xo[i] = X[(k < T ? k + 1 : T) * w.nx + c]; }
  for (size_t i = threadIdx.x; i < T * w.m; i += blockDim.x) { size_t k = i / w.m, c = i % w.m; Uo[i] = U[(k + 1 < T ? k + 1 : (size_t)tail_src) * w.m + c]; }
  for (int i = threadIdx.x; i < w.nx; i += blockDim.x) w.x0[b * w.nx + i] = x_meas ? x_meas[b * w.nx + i] : X[w.nx + i];
}

// One closed-loop MPC tick entirely on the device (SURVEY 8f row f-2; fulldynamic_talos.py:496-497,532-540):
// rotate the horizon (append `last`), shift the warm start, take x0 from x_meas (host [batch][nx]) or from the model
// prediction, reset (setup-per-tick, full/cent) or shift (cycleProblem, kino) the multipliers, run max_iters iterations.
int32_t mpc_tick(mpc_solver_t *h, const mpc_knot_t *last, const double *x_meas, int32_t keep_multipliers, int32_t max_iters) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_tick before mpc_setup");
  Ws &w = h->w;
  if (last && cycle_knots(h, last)) return 1;
  double *d_meas = nullptr;
  if (x_meas) {
    if (!h->d_meas) CK(cudaMalloc(&h->d_meas, (size_t)w.B * w.nx * 8));
    CK(cudaMemcpyAsync(h->d_meas, x_meas, (size_t)w.B * w.nx * 8, cudaMemcpyHostToDevice, h->stream));
    d_meas = h->d_meas;
  }
  k_shift_warmstart<<<w.B, 128, 0, h->stream>>>(w, h->d_xs_in, h->d_us_in, d_meas, h->tail_mode);
  if (keep_multipliers) k_shift_multipliers<<<w.B, 128, 0, h->stream>>>(w, 1);
  else if (zero_multipliers(h, h->stream)) return 1;
  CK(cudaGetLastError());
  return run_impl(h, h->d_xs_in, h->d_us_in, max_iters, h->stream, true);
}

int32_t mpc_set_tail_warmstart(mpc_solver_t *h, int32_t mode) {
  if (!h) return fail("null handle");
  if (mode != 0 && mode != 1) return fail("mpc_set_tail_warmstart: mode must be 0 (previous knot) or 1 (nearest knot of the same contact phase)");
  h->tail_mode = mode;
  return 0;
}

int32_t mpc_reset_multipliers(mpc_solver_t *h, uint64_t stream) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_reset_multipliers before mpc_setup");
  return zero_multipliers(h, stream ? reinterpret_cast<cudaStream_t>(stream) : h->stream);
}

int32_t mpc_run(mpc_solver_t *h, const double *xs_init, const double *us_init, int32_t max_iters) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_run before mpc_setup");
  Ws &w = h->w;
  const size_t T1 = w.T + 1;
  CK(cudaMemcpyAsync(h->d_xs_in, xs_init, w.B * T1 * w.nx * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_us_in, us_init, (size_t)w.B * w.T * w.m * 8, cudaMemcpyHostToDevice, h->stream));
  return run_impl(h, h->d_xs_in, h->d_us_in, max_iters, h->stream, true);
}

// pack what the MPC loop consumes (fulldynamic_talos.py:548-550) of the instances [first, first + gridDim.x): the first feedback
// gain into K0 [instance][m][n] and the summary into info [instance][8] (either may be null)
__global__ void k_pack_k0_info(Ws w, double *K0, double *info, int first) {
  const size_t b = first + blockIdx.x, sz = (size_t)w.m * w.n;
  if (K0) for (size_t i = threadIdx.x; i < sz; i += blockDim.x) K0[b * sz + i] = w.Kfb[b * (size_t)w.T * sz + i];
  if (info && threadIdx.x == 0) {
    const InstState &t = w.st[b];
    double *o = info + b * 8;
    o[0] = t.prim_infeas; o[1] = t.dual_infeas; o[2] = t.traj_cost; o[3] = t.merit; o[4] = (double)t.num_iters; o[5] = (double)t.conv; o[6] = (double)t.status; o[7] = t.alpha;
  }
}

int32_t mpc_run_pipelined(mpc_solver_t *h, const double *xs_init, const double *us_init, int32_t max_iters, int32_t parts, double *xs_out,
                          double *us_out, double *K0_out, mpc_info_t *info_out) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_run_pipelined before mpc_setup");
  Ws &w = h->w;
  const size_t T1 = w.T + 1, sx = T1 * w.nx, su = (size_t)w.T * w.m, sk = (size_t)w.m * w.n;
  if (parts < 1) parts = 1;
  if (parts > 8) parts = 8;
  if (parts > w.B) parts = w.B;
  if (!h->stream_copy) CK(cudaStreamCreateWithFlags(&h->stream_copy, cudaStreamNonBlocking));
  for (int i = 0; i < 2 * parts; i++) if (!h->ev_part[i]) CK(cudaEventCreateWithFlags(&h->ev_part[i], cudaEventDisableTiming));
  if (K0_out && !h->d_k0) CK(cudaMalloc(&h->d_k0, (size_t)w.B * sk * 8));
  if (info_out && !h->h_st) CK(cudaMallocHost(&h->h_st, sizeof(InstState) * w.B));
  cudaStream_t s = h->stream, sc = h->stream_copy;
  auto lo = [&](int p) { return (int)((long long)w.B * p / parts); };
  // every upload is queued at once on the copy stream; the solve of part p waits for its own
  for (int p = 0; p < parts; p++) {
    const size_t o = lo(p), n = lo(p + 1) - lo(p);
    CK(cudaMemcpyAsync(h->d_xs_in + o * sx, xs_init + o * sx, n * sx * 8, cudaMemcpyHostToDevice, sc));
    CK(cudaMemcpyAsync(h->d_us_in + o * su, us_init + o * su, n * su * 8, cudaMemcpyHostToDevice, sc));
    CK(cudaEventRecord(h->ev_part[p], sc));
  }
  CK(cudaEventRecord(h->ev0, s));
  h->evcat.clear();
  CudaBackend be{h, s};
  int launches = 0;
  for (int p = 0; p < parts; p++) {
    const int o = lo(p), n = lo(p + 1) - o;
    CK(cudaStreamWaitEvent(s, h->ev_part[p], 0));
    be.mark(3);
    k_init<<<n, 128, 0, s>>>(w, h->d_xs_in, h->d_us_in, max_iters, o);
    launches += 1 + run_loop(be, w, max_iters, w.sc, o, n); // returns with the part finished (its last counter read synchronises)
    be.mark(-1);
    if (be.err != cudaSuccess) return fail(std::string("kernel failure: ") + cudaGetErrorString(be.err));
    // the download of this part overlaps the solve of the next one
    CK(cudaEventRecord(h->ev_part[parts + p], s));
    CK(cudaStreamWaitEvent(sc, h->ev_part[parts + p], 0));
    if (xs_out) CK(cudaMemcpyAsync(xs_out + (size_t)o * sx, w.xs + (size_t)o * sx, (size_t)n * sx * 8, cudaMemcpyDeviceToHost, sc));
    if (us_out) CK(cudaMemcpyAsync(us_out + (size_t)o * su, w.us + (size_t)o * su, (size_t)n * su * 8, cudaMemcpyDeviceToHost, sc));
    if (K0_out) {
      k_pack_k0_info<<<n, 128, 0, sc>>>(w, h->d_k0, nullptr, o);
      CK(cudaMemcpyAsync(K0_out + (size_t)o * sk, h->d_k0 + (size_t)o * sk, (size_t)n * sk * 8, cudaMemcpyDeviceToHost, sc));
    }
    if (info_out) CK(cudaMemcpyAsync(h->h_st + o, w.st + o, sizeof(InstState) * n, cudaMemcpyDeviceToHost, sc));
  }
  CK(cudaEventRecord(h->ev1, s));
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(sc));
  CK(cudaEventSynchronize(h->ev1));
  h->last_launches = launches;
  if (read_run_times(h)) return 1;
  if (info_out)
    for (int b = 0; b < w.B; b++) info_out[b] = info_of(h->h_st[b]);
  return 0;
}

int32_t mpc_run_device(mpc_solver_t *h, uint64_t xs_dev, uint64_t us_dev, int32_t max_iters, uint64_t stream) {
  CK(cudaSetDevice(h->device));
  cudaStream_t s = stream ? reinterpret_cast<cudaStream_t>(stream) : h->stream;
  return run_impl(h, reinterpret_cast<const double *>(xs_dev), reinterpret_cast<const double *>(us_dev), max_iters, s, true);
}

int32_t mpc_get_results(mpc_solver_t *h, double *xs, double *us, double *K, double *vs, double *lams, mpc_info_t *info) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_get_results before mpc_setup");
  Ws &w = h->w;
  const size_t T1 = w.T + 1;
  cudaStream_t s = h->stream;
  if (xs) CK(cudaMemcpyAsync(xs, w.xs, w.B * T1 * w.nx * 8, cudaMemcpyDeviceToHost, s));
  if (us) CK(cudaMemcpyAsync(us, w.us, (size_t)w.B * w.T * w.m * 8, cudaMemcpyDeviceToHost, s));
  if (K) CK(cudaMemcpyAsync(K, w.Kfb, (size_t)w.B * w.T * w.m * w.n * 8, cudaMemcpyDeviceToHost, s));
  if (vs) CK(cudaMemcpyAsync(vs, w.vs, w.B * T1 * w.nc * 8, cudaMemcpyDeviceToHost, s));
  if (lams) CK(cudaMemcpyAsync(lams, w.lams, w.B * T1 * w.n * 8, cudaMemcpyDeviceToHost, s));
  std::vector<InstState> st;
  if (info) { st.resize(w.B); CK(cudaMemcpyAsync(st.data(), w.st, sizeof(InstState) * w.B, cudaMemcpyDeviceToHost, s)); }
  CK(cudaStreamSynchronize(s));
  if (info)
    for (int b = 0; b < w.B; b++) info[b] = info_of(st[b]);
  return 0;
}

int32_t mpc_result_ptrs(mpc_solver_t *h, uint64_t *xs, uint64_t *us, uint64_t *K, uint64_t *info) {
  if (!h->setup_done) return fail("mpc_result_ptrs before mpc_setup");
  if (xs) *xs = (uint64_t)h->w.xs;
  if (us) *us = (uint64_t)h->w.us;
  if (K) *K = (uint64_t)h->w.Kfb;
  if (info) *info = (uint64_t)h->w.st;
  return 0;
}

// xs, us, K0 and the per-instance summary into device buffers, e.g. for a gather over NVLink
int32_t mpc_export_results_device(mpc_solver_t *h, uint64_t xs_dev, uint64_t us_dev, uint64_t K0_dev, uint64_t info_dev, uint64_t stream) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_export_results_device before mpc_setup");
  Ws &w = h->w;
  cudaStream_t s = stream ? reinterpret_cast<cudaStream_t>(stream) : h->stream;
  if (xs_dev) CK(cudaMemcpyAsync(reinterpret_cast<void *>(xs_dev), w.xs, (size_t)w.B * (w.T + 1) * w.nx * 8, cudaMemcpyDeviceToDevice, s));
  if (us_dev) CK(cudaMemcpyAsync(reinterpret_cast<void *>(us_dev), w.us, (size_t)w.B * w.T * w.m * 8, cudaMemcpyDeviceToDevice, s));
  if (K0_dev || info_dev) {
    k_pack_k0_info<<<w.B, 128, 0, s>>>(w, reinterpret_cast<double *>(K0_dev), reinterpret_cast<double *>(info_dev), 0);
    CK(cudaGetLastError());
  }
  return 0;
}

int32_t mpc_get_stage_data(mpc_solver_t *h, int32_t k, double *xdot, double *contact_force) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_get_stage_data before mpc_setup");
  Ws &w = h->w;
  if (k < 0 || k >= w.T) return fail("stage index out of range");
  const size_t T1 = w.T + 1;
  if (xdot) CK(cudaMemcpy2D(xdot, w.n * 8, w.xdot + (size_t)k * 56, T1 * 56 * 8, w.n * 8, w.B, cudaMemcpyDeviceToHost));
  if (contact_force) CK(cudaMemcpy2D(contact_force, 12 * 8, w.lamc + (size_t)k * 12, T1 * 12 * 8, 12 * 8, w.B, cudaMemcpyDeviceToHost));
  return 0;
}

int32_t mpc_last_launches(mpc_solver_t *h) { return h->last_launches; }
double mpc_last_kernel_ms(mpc_solver_t *h, int32_t category) { return (category >= 0 && category < 4) ? h->cat_ms[category] : -1.0; }
int32_t mpc_last_kernel_launches(mpc_solver_t *h, int32_t category) { return (category >= 0 && category < 4) ? h->cat_launches[category] : -1; }
void mpc_set_profiling(mpc_solver_t *h, int32_t on) { h->profile = on != 0; }

int32_t mpc_get_feedback(mpc_solver_t *h, int32_t k, double *K) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_get_feedback before mpc_setup");
  Ws &w = h->w;
  if (k < 0 || k >= w.T) return fail("stage index out of range");
  const size_t sz = (size_t)w.m * w.n * 8;
  CK(cudaMemcpy2DAsync(K, sz, w.Kfb + (size_t)k * w.m * w.n, (size_t)w.T * sz, sz, w.B, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}
double mpc_last_device_ms(mpc_solver_t *h) { return h->last_ms; }
uint64_t mpc_workspace_bytes(mpc_solver_t *h) { return h->bytes; }
// per-phase cycle counters of the Riccati kernel for instance 0 (all zero unless built with -DMPC_PHASE_TIMING)
int32_t mpc_debug_phases(mpc_solver_t *h, double *out64) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_debug_phases before mpc_setup");
  CK(cudaMemcpy(out64, h->w.phase, 64 * 8, cudaMemcpyDeviceToHost)); // [0:16)+[48:64) Riccati, [16:32) derivative eval, [32:48) values eval
  return 0;
}

int32_t mpc_debug_lq(mpc_solver_t *h, const double *xs, const double *us, int32_t inst, double *AB, double *H, double *g, double *gap,
                     double *hval, double *scal) {
  CK(cudaSetDevice(h->device));
  if (!h->setup_done) return fail("mpc_debug_lq before mpc_setup");
  Ws &w = h->w;
  const size_t T1 = w.T + 1, T = w.T;
  if (inst < 0 || inst >= w.B) return fail("instance out of range");
  CK(cudaMemcpyAsync(h->d_xs_in, xs, w.B * T1 * w.nx * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_us_in, us, (size_t)w.B * w.T * w.m * 8, cudaMemcpyHostToDevice, h->stream));
  k_init<<<w.B, 128, 0, h->stream>>>(w, h->d_xs_in, h->d_us_in, 1, 0);
  CudaBackend be{h, h->stream};
  be.reset_counters();
  be.eval(true, eval_list(w, 0), w.B); be.decide_eval(eval_list(w, 0), w.B, eval_list(w, 1));
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  const size_t b = inst;
  if (AB) CK(cudaMemcpy(AB, w.AB + b * T * w.n * w.nz, T * w.n * w.nz * 8, cudaMemcpyDeviceToHost));
  if (H) CK(cudaMemcpy(H, w.H + b * T1 * w.nz * w.nz, T1 * w.nz * w.nz * 8, cudaMemcpyDeviceToHost));
  if (g) CK(cudaMemcpy(g, w.g + b * T1 * w.nz, T1 * w.nz * 8, cudaMemcpyDeviceToHost));
  if (gap) CK(cudaMemcpy(gap, w.gap + b * T * w.n, T * w.n * 8, cudaMemcpyDeviceToHost));
  if (hval) CK(cudaMemcpy(hval, w.h + b * T1 * w.nc, T1 * w.nc * 8, cudaMemcpyDeviceToHost));
  if (scal) CK(cudaMemcpy(scal, w.scal + b * T1 * SC_COUNT, T1 * SC_COUNT * 8, cudaMemcpyDeviceToHost));
  return 0;
}

__global__ void k_gemm_tn_test(int mt, int nt, int K, const double *A, int lda, const double *B, int ldb, double *C, int ldc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *sA = reinterpret_cast<double *>(smem_raw), *sB = sA + K * lda, *sC = sB + K * ldb;
  for (int i = threadIdx.x; i < K * lda; i += blockDim.x) sA[i] = A[i];
  for (int i = threadIdx.x; i < K * ldb; i += blockDim.x) sB[i] = B[i];
  __syncthreads();
  mma_tn(mt, nt, K, sA, lda, sB, ldb, sC, ldc, nullptr, 0, 0, 0, false);
  for (int i = threadIdx.x; i < 8 * mt * ldc; i += blockDim.x) C[i] = sC[i];
}

// unit-test hook for the DMMA tile GEMM: C (8mt x 8nt) = A^T B, A [K][lda], B [K][ldb], host pointers
int32_t mpc_debug_gemm_tn(int32_t mt, int32_t nt, int32_t K, const double *A, int32_t lda, const double *B, int32_t ldb, double *C, int32_t ldc) {
  double *dA, *dB, *dC;
  size_t sa = (size_t)K * lda * 8, sb = (size_t)K * ldb * 8, sc = (size_t)8 * mt * ldc * 8;
  CK(cudaMalloc(&dA, sa)); CK(cudaMalloc(&dB, sb)); CK(cudaMalloc(&dC, sc));
  CK(cudaMemcpy(dA, A, sa, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dB, B, sb, cudaMemcpyHostToDevice));
  CK(cudaFuncSetAttribute(k_gemm_tn_test, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sa + sb + sc)));
  k_gemm_tn_test<<<1, 256, sa + sb + sc>>>(mt, nt, K, dA, lda, dB, ldb, dC, ldc);
  CK(cudaGetLastError());
  CK(cudaMemcpy(C, dC, sc, cudaMemcpyDeviceToHost));
  cudaFree(dA); cudaFree(dB); cudaFree(dC);
  return 0;
}

// TFLOP/s of a peak kernel: 8 CTAs of 256 threads per SM, one warm-up launch of warm_iters, best of five timed launches of iters
// (flop_per_thread: FLOP per thread and iteration)
static double time_peak(int device, void (*kernel)(double *, int), int warm_iters, int iters, double flop_per_thread) {
  if (cudaSetDevice(device) != cudaSuccess) { g_err = "no CUDA device"; return -1.0; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  double *out = nullptr;
  if (cudaMalloc(&out, (size_t)blocks * threads * 8) != cudaSuccess) return -1.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  kernel<<<blocks, threads>>>(out, warm_iters);
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0);
    kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  cudaFree(out); cudaEventDestroy(e0); cudaEventDestroy(e1);
  double flops = flop_per_thread * (double)iters * blocks * threads;
  return flops / (best * 1e-3) / 1e12;
}

double mpc_measure_fp64_peak(int32_t device) { return time_peak(device, k_dfma_peak, 1024, 1 << 16, 2.0 * 8); }
double mpc_measure_fp64_peak_dmma(int32_t device) { return time_peak(device, k_dmma_peak, 256, 1 << 14, 512.0 * 8 / 32); }

// ---- rigid-body terms in front of the whole-body QPs (include/mpcb200.h)
int32_t mpc_rbd_terms_device(mpc_solver_t *h, int32_t count, uint64_t x_dev, uint64_t M_dev, uint64_t nle_dev, uint64_t Jc_dev, uint64_t dJv_dev, uint64_t vf_dev,
                             uint64_t stream) {
  if (!h) return fail("null handle");
  if (h->w.kind == MPC_KIND_CENT) return fail("mpc_rbd_terms: the centroidal model has no rigid-body tree");
  if (count <= 0) return fail("mpc_rbd_terms: count out of range");
  CK(cudaSetDevice(h->device));
  const size_t smem = sizeof(FullWsT<false>);
  CK(cudaFuncSetAttribute(k_rbd_terms, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); // per device: set on every call (microseconds)
  k_rbd_terms<<<count, 128, smem, stream ? (cudaStream_t)stream : h->stream>>>(h->d_model, (const double *)x_dev, count, (double *)M_dev, (double *)nle_dev,
                                                                                  (double *)Jc_dev, (double *)dJv_dev, (double *)vf_dev);
  CK(cudaGetLastError());
  return 0;
}
int32_t mpc_rbd_terms(mpc_solver_t *h, int32_t count, const double *x, double *M, double *nle, double *Jc, double *dJv, double *vf) {
  if (!h) return fail("null handle");
  if (count <= 0) return fail("mpc_rbd_terms: count out of range");
  CK(cudaSetDevice(h->device));
  const size_t B = count, per = (NQ + NV) + NV * NV + NV + 12 * NV + 12 + 12;
  double *d = nullptr;
  CK(cudaMalloc(&d, 8 * B * per));
  double *dx = d, *dM = dx + B * (NQ + NV), *dn = dM + B * NV * NV, *dJ = dn + B * NV, *dd = dJ + B * 12 * NV, *dv = dd + B * 12;
  int rc = 0;
  if (cudaMemcpyAsync(dx, x, 8 * B * (NQ + NV), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) rc = fail("H2D of the states failed");
  if (!rc) rc = mpc_rbd_terms_device(h, count, (uint64_t)dx, (uint64_t)dM, (uint64_t)dn, (uint64_t)dJ, (uint64_t)dd, (uint64_t)dv, 0);
  auto back = [&](double *dst, const double *src, size_t n) { if (!rc && dst && cudaMemcpyAsync(dst, src, 8 * B * n, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) rc = fail("D2H failed"); };
  back(M, dM, NV * NV); back(nle, dn, NV); back(Jc, dJ, 12 * NV); back(dJv, dd, 12); back(vf, dv, 12);
  if (cudaStreamSynchronize(h->stream) != cudaSuccess && !rc) rc = fail("mpc_rbd_terms: kernel failed");
  cudaFree(d);
  return rc;
}

int32_t mpc_ikid_terms_device(mpc_solver_t *h, int32_t count, uint64_t x_dev, const int32_t frame_body[2], const double frame_place[2][12], uint64_t M_dev,
                              uint64_t nle_dev, uint64_t Jc_dev, uint64_t dJv_dev, uint64_t Ag_dev, uint64_t dAgv_dev, uint64_t Jang_dev, uint64_t dJang_dev,
                              uint64_t stream) {
  if (!h || !frame_body || !frame_place) return fail("null handle / frames");
  if (h->w.kind == MPC_KIND_CENT) return fail("mpc_ikid_terms: the centroidal model has no rigid-body tree");
  if (count <= 0) return fail("mpc_ikid_terms: count out of range");
  if (frame_body[0] < 0 || frame_body[0] >= NB || frame_body[1] < 0 || frame_body[1] >= NB) return fail("mpc_ikid_terms: frame body out of range [0, nb)");
  CK(cudaSetDevice(h->device));
  IkidFrames fr;
  for (int f = 0; f < 2; f++) {
    fr.body[f] = frame_body[f];
    for (int i = 0; i < 12; i++) fr.place[12 * f + i] = frame_place[f][i];
  }
  const size_t smem = sizeof(FullWsT<false>);
  CK(cudaFuncSetAttribute(k_ikid_terms, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_ikid_terms<<<count, 128, smem, stream ? (cudaStream_t)stream : h->stream>>>(h->d_model, (const double *)x_dev, count, fr, (double *)M_dev, (double *)nle_dev,
                                                                                   (double *)Jc_dev, (double *)dJv_dev, (double *)Ag_dev, (double *)dAgv_dev,
                                                                                   (double *)Jang_dev, (double *)dJang_dev);
  CK(cudaGetLastError());
  return 0;
}
int32_t mpc_ikid_terms(mpc_solver_t *h, int32_t count, const double *x, const int32_t frame_body[2], const double frame_place[2][12], double *M, double *nle,
                       double *Jc, double *dJv, double *Ag, double *dAgv, double *Jang, double *dJang) {
  if (!h) return fail("null handle");
  if (count <= 0) return fail("mpc_ikid_terms: count out of range");
  CK(cudaSetDevice(h->device));
  const size_t B = count, per = (NQ + NV) + NV * NV + NV + 12 * NV + 12 + 6 * NV + 6 + 6 * NV + 6;
  double *d = nullptr;
  CK(cudaMalloc(&d, 8 * B * per));
  double *dx = d, *dM = dx + B * (NQ + NV), *dn = dM + B * NV * NV, *dJ = dn + B * NV, *dd = dJ + B * 12 * NV, *dA = dd + B * 12, *dAv = dA + B * 6 * NV,
         *dJa = dAv + B * 6, *dJav = dJa + B * 6 * NV;
  int rc = 0;
  if (cudaMemcpyAsync(dx, x, 8 * B * (NQ + NV), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) rc = fail("H2D of the states failed");
  if (!rc) rc = mpc_ikid_terms_device(h, count, (uint64_t)dx, frame_body, frame_place, (uint64_t)dM, (uint64_t)dn, (uint64_t)dJ, (uint64_t)dd, (uint64_t)dA,
                                      (uint64_t)dAv, (uint64_t)dJa, (uint64_t)dJav, 0);
  auto back = [&](double *dst, const double *src, size_t n) { if (!rc && dst && cudaMemcpyAsync(dst, src, 8 * B * n, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) rc = fail("D2H failed"); };
  back(M, dM, NV * NV); back(nle, dn, NV); back(Jc, dJ, 12 * NV); back(dJv, dd, 12);
  back(Ag, dA, 6 * NV); back(dAgv, dAv, 6); back(Jang, dJa, 6 * NV); back(dJang, dJav, 6);
  if (cudaStreamSynchronize(h->stream) != cudaSuccess && !rc) rc = fail("mpc_ikid_terms: kernel failed");
  cudaFree(d);
  return rc;
}

// ---- device-side gait / swing-foot references (include/mpcb200.h, SURVEY 8f row f-4)
int32_t mpc_gait_setup(mpc_solver_t *h, const mpc_gait_t *gait, const int32_t *mirror, const double *urefs) {
  if (!h || !gait) return fail("null handle / gait");
  if (!h->setup_done) return fail("mpc_gait_setup before mpc_setup");
  if (gait->T_ds <= 0 || gait->T_ss <= 0 || gait->cycles < 0 || gait->cycles > 3) return fail("mpc_gait_setup: schedule out of range (T_ds, T_ss > 0, cycles <= 3)");
  if (h->w.kind != MPC_KIND_FULL && (gait->n_uref <= 0 || !urefs)) return fail("mpc_gait_setup: the kinodynamic / centroidal gaits need the control-reference table");
  CK(cudaSetDevice(h->device));
  Ws &w = h->w;
  GaitCfg g;
  std::memset(&g, 0, sizeof g);
  gait_fill_cfg(*gait, w.kind, w.T, g);
  std::vector<int8_t> phases;
  gait_build_schedule(*gait, w.T, phases, g);
  cudaFree(h->d_gait); cudaFree(h->d_gait_robots); cudaFree(h->d_gait_phases); cudaFree(h->d_gait_urefs); cudaFree(h->d_feet);
  h->d_gait = nullptr; h->d_gait_robots = nullptr; h->d_gait_phases = nullptr; h->d_gait_urefs = nullptr; h->d_feet = nullptr;
  CK(cudaMalloc(&h->d_gait, sizeof(GaitCfg)));
  CK(cudaMalloc(&h->d_gait_robots, sizeof(GaitRobot) * w.B));
  CK(cudaMalloc(&h->d_gait_phases, phases.size()));
  CK(cudaMalloc(&h->d_feet, 8 * (size_t)w.B * 24));
  CK(cudaMemcpy(h->d_gait_phases, phases.data(), phases.size(), cudaMemcpyHostToDevice));
  g.phases = h->d_gait_phases;
  if (gait->n_uref > 0 && urefs) {
    CK(cudaMalloc(&h->d_gait_urefs, 8 * (size_t)gait->n_uref * MPC_MAXU));
    CK(cudaMemcpy(h->d_gait_urefs, urefs, 8 * (size_t)gait->n_uref * MPC_MAXU, cudaMemcpyHostToDevice));
    g.urefs = h->d_gait_urefs;
  }
  CK(cudaMemcpy(h->d_gait, &g, sizeof g, cudaMemcpyHostToDevice));
  const std::vector<GaitRobot> rs = gait_init_robots(*gait, w.B, mirror);
  CK(cudaMemcpy(h->d_gait_robots, rs.data(), sizeof(GaitRobot) * w.B, cudaMemcpyHostToDevice));
  h->gait_t = 0;
  h->gait_ready = true;
  return 0;
}

int32_t mpc_gait_tick(mpc_solver_t *h, const double *lf, const double *rf) {
  if (!h) return fail("null handle");
  if (!h->gait_ready) return fail("mpc_gait_tick before mpc_gait_setup");
  if ((lf == nullptr) != (rf == nullptr)) return fail("mpc_gait_tick: pass both measured placements or neither");
  CK(cudaSetDevice(h->device));
  Ws &w = h->w;
  double *dl = h->d_feet, *dr = h->d_feet + (size_t)w.B * 12;
  if (lf) {
    CK(cudaMemcpyAsync(dl, lf, 8 * (size_t)w.B * 12, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dr, rf, 8 * (size_t)w.B * 12, cudaMemcpyHostToDevice, h->stream));
  } else if (w.kind == MPC_KIND_CENT) {
    dl = dr = nullptr; // the centroidal state carries no feet: the soles are taken where last tick's plan wanted them (exact tracking)
  } else {
    const size_t smem = sizeof(FullWsT<false>);
    CK(cudaFuncSetAttribute(k_feet_of_prediction, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); // per device: set on every call
    k_feet_of_prediction<<<w.B, 128, smem, h->stream>>>(w, h->d_model, dl, dr);
  }
  k_gait_tick<<<w.B, 128, 0, h->stream>>>(w, h->d_gait, h->d_gait_robots, h->gait_t, dl, dr);
  CK(cudaGetLastError());
  h->gait_t++;
  return 0;
}

int32_t mpc_get_knots(mpc_solver_t *h, mpc_knot_t *knots, mpc_term_t *terms) {
  if (!h) return fail("null handle");
  if (!h->setup_done) return fail("mpc_get_knots before mpc_setup");
  CK(cudaSetDevice(h->device));
  Ws &w = h->w;
  if (knots) CK(cudaMemcpyAsync(knots, w.knots, sizeof(mpc_knot_t) * (size_t)w.B * w.T, cudaMemcpyDeviceToHost, h->stream));
  if (terms) CK(cudaMemcpyAsync(terms, w.terms, sizeof(mpc_term_t) * (size_t)w.B, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_abi_sizeof(int32_t which) {
  switch (which) {
  case 0: return sizeof(mpc_robot_t);
  case 1: return sizeof(mpc_config_t);
  case 2: return sizeof(mpc_knot_t);
  case 3: return sizeof(mpc_term_t);
  case 4: return sizeof(mpc_info_t);
  case 5: return sizeof(mpc_gait_t);
  }
  return -1;
}

} // extern "C"
