// libmpcb200.so — batched dense QP (SURVEY 8f row f-3): kernels + the C-ABI of include/mpcqp_b200.h.
// One CTA (128 threads) per QP, everything in shared memory (qp.cuh).  No CPU fallback: creation fails without a CUDA device.
#include "qp.cuh"
#include "cuda_owned.hpp"
#include "../../include/mpcb200.h"
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <string>

using namespace mpcdev;

namespace {

constexpr int QP_THREADS = 128;

__global__ void __launch_bounds__(QP_THREADS) k_qp_solve(const QPArgs P) {
  extern __shared__ __align__(16) double qp_smem[];
  for (int inst = blockIdx.x; inst < P.batch; inst += gridDim.x) {
    qp_solve_group(P, inst, qp_smem);
    SYNC();
  }
}

struct AsmArgs {
  const double *M, *nle, *Jc, *gamma, *a, *forces;
  const int32_t *cs;
  double mu, L, W;
  double *A, *b, *C, *l;
  int batch;
};
__global__ void __launch_bounds__(QP_THREADS) k_qp_assemble_id(const AsmArgs P) {
  const int i = blockIdx.x;
  if (i >= P.batch) return;
  qp_assemble_id_group(P.M + i * 784, P.nle + i * 28, P.Jc + i * 336, P.gamma + i * 12, P.a + i * 28, P.forces + i * 12, P.cs + i * 2, P.mu, P.L, P.W,
                       P.A + (size_t)i * 2480, P.b + i * 40, P.C + (size_t)i * 1116, P.l + i * 18);
}

struct IkidAsmArgs {
  const double *M, *nle, *Jc, *dJv, *Ag, *dAgv, *Jang, *dJang, *task, *forces, *gains;
  const int32_t *cs;
  double wt[5], mu, L, W;
  double *H, *g, *A, *b, *C, *l;
  int batch;
};
__global__ void __launch_bounds__(QP_THREADS) k_qp_assemble_ikid(const IkidAsmArgs P) {
  __shared__ double sm[24 * 28 + 24 + 12 + 28];
  const int i = blockIdx.x;
  if (i >= P.batch) return;
  qp_assemble_ikid_group(P.M + i * 784, P.nle + i * 28, P.Jc + i * 336, P.dJv + i * 12, P.Ag + i * 168, P.dAgv + i * 6, P.Jang + i * 168, P.dJang + i * 6,
                         P.task + i * 98, P.forces + i * 12, P.cs + i * 2, P.wt, P.gains, P.mu, P.L, P.W, sm, P.H + (size_t)i * 3844, P.g + i * 62,
                         P.A + (size_t)i * 2480, P.b + i * 40, P.C + (size_t)i * 1116, P.l + i * 18);
}

// gamma = (dJ v + kd (v_lin + v_ang) on the linear rows) of the active contacts (QP_utils.py:524-528), in place over dJv
__global__ void k_qp_gamma(double *dJv, const double *vf, const int32_t *cs, double kd, int batch) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= batch * 12) return;
  const int i = e / 12, r = e % 12, c = r / 6, rr = r % 6;
  double g = dJv[e];
  if (rr < 3) g += kd * (vf[i * 12 + c * 6 + rr] + vf[i * 12 + c * 6 + 3 + rr]);
  dJv[e] = cs[i * 2 + c] ? g : 0.0;
}

thread_local std::string g_err;
int fail(const std::string &m) { g_err = m; return 1; }
#define CUQ(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

struct Slot { // one data array of the handle: device buffer sized for the full batch, current batch stride
  CudaArray<double> d;
  size_t per = 0;
  long long stride = 0;
  bool set = false;
};

} // namespace

struct mpc_qp {
  int n, ne, ni, box, nz, max_batch, device, batch = 0;
  CudaStream stream;
  CudaEvent ev0, ev1;
  Slot H, g, A, b, C, l, u, lb, ub;
  CudaArray<double> dx, dy, dz, dscratch, dstate; // dstate: [B][57] states + [B][12] frame velocities
  CudaArray<double> dikid; // IKID assembly only, allocated by its first call: gains [1658] + [B][98] task errors + [B] task terms (IkidScratch)
  CudaArray<mpc_qp_info_t> dinfo;
  CudaArray<long long> dphase; // instrumented builds only
  size_t smem_bytes = 0;
  int sms = 0, ctas_per_sm = 1;
};

namespace {

// the preamble of every entry point that takes a handle: a null handle fails before any CUDA call, then the device becomes current
int enter(const mpc_qp *h, const char *fn) {
  if (!h) return fail(std::string(fn) + ": null handle");
  CUQ(cudaSetDevice(h->device));
  return 0;
}

// checks, launch shape, buffers, stream and events of a new handle (mpc_qp_create)
int init_qp(mpc_qp *h, int n, int n_eq, int n_in, int box, int max_batch, int device) {
  if (n <= 0 || n > MPC_QP_MAXN || n_eq < 0 || n_eq > MPC_QP_MAXEQ || n_in < 0 || n_in > MPC_QP_MAXIN || max_batch <= 0)
    return fail("mpc_qp_create: dimensions out of range (n <= 64, n_eq <= 64, n_in <= 32, max_batch > 0)");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= device || device < 0) return fail("mpc_qp_create: no CUDA device (this library has no CPU fallback)");
  h->n = n; h->ne = n_eq; h->ni = n_in; h->box = box ? 1 : 0; h->nz = n_in + (box ? n : 0); h->max_batch = max_batch; h->device = device;
  if (cudaSetDevice(device) != cudaSuccess) return fail("cudaSetDevice failed");
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  h->sms = prop.multiProcessorCount;
  h->smem_bytes = 8 * (size_t)qp_smem_doubles(n, n_eq, n_in, h->box);
  if (h->smem_bytes > (size_t)prop.sharedMemPerBlockOptin) return fail("QP does not fit the shared memory of one SM");
  if (cudaFuncSetAttribute(k_qp_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes) != cudaSuccess)
    return fail("cudaFuncSetAttribute(k_qp_solve) failed");
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->ctas_per_sm, k_qp_solve, QP_THREADS, h->smem_bytes);
  const size_t B = max_batch;
  struct { Slot *s; size_t per; } slots[] = {{&h->H, (size_t)n * n}, {&h->g, (size_t)n}, {&h->A, (size_t)n_eq * n}, {&h->b, (size_t)n_eq}, {&h->C, (size_t)n_in * n},
                                             {&h->l, (size_t)n_in},  {&h->u, (size_t)n_in}, {&h->lb, (size_t)n},       {&h->ub, (size_t)n}};
  for (auto &sl : slots) {
    sl.s->per = sl.per;
    if (sl.s->d.ensure((sl.per ? sl.per : 1) * B) != cudaSuccess) return fail("cudaMalloc of the QP data failed");
    cudaMemset(sl.s->d, 0, 8 * (sl.per ? sl.per : 1) * B);
  }
  if (h->dx.ensure(B * n) != cudaSuccess || h->dy.ensure(B * (n_eq ? n_eq : 1)) != cudaSuccess || h->dz.ensure(B * (h->nz ? h->nz : 1)) != cudaSuccess ||
      h->dinfo.ensure(B) != cudaSuccess || h->dscratch.ensure(B * (784 + 28 + 336 + 12 + 28 + 12 + 1)) != cudaSuccess || h->dstate.ensure(B * (57 + 12)) != cudaSuccess)
    return fail("cudaMalloc of the QP results failed");
#ifdef MPC_QP_PHASE_TIMING
  if (h->dphase.ensure(8) != cudaSuccess) return fail("cudaMalloc failed");
  cudaMemset(h->dphase, 0, 64);
#endif
  if (h->stream.ensure(cudaStreamDefault) != cudaSuccess || h->ev0.ensure(cudaEventDefault) != cudaSuccess || h->ev1.ensure(cudaEventDefault) != cudaSuccess)
    return fail("stream / event creation failed");
  return 0;
}

int upload(mpc_qp *h, Slot &s, const double *src, long long stride, int batch, const char *name) {
  if (!src) return 0;
  if (stride != 0 && stride < (long long)s.per) return fail(std::string("stride of ") + name + " smaller than one QP's array");
  if (stride == 0) CUQ(cudaMemcpyAsync(s.d, src, 8 * s.per, cudaMemcpyHostToDevice, h->stream));
  else if (stride == (long long)s.per) CUQ(cudaMemcpyAsync(s.d, src, 8 * s.per * batch, cudaMemcpyHostToDevice, h->stream));
  else CUQ(cudaMemcpy2DAsync(s.d, 8 * s.per, src, 8 * stride, 8 * s.per, batch, cudaMemcpyHostToDevice, h->stream));
  s.stride = stride == 0 ? 0 : (long long)s.per;
  s.set = true;
  return 0;
}

// inputs of k_qp_assemble_id for B QPs, carved out of the handle's scratch: M, nle, Jc, gamma, a, forces, cs
struct AsmScratch {
  double *M, *nle, *Jc, *gamma, *a, *forces;
  int32_t *cs;
  AsmScratch(double *s, size_t B)
      : M(s), nle(M + B * 784), Jc(nle + B * 28), gamma(Jc + B * 336), a(gamma + B * 12), forces(a + B * 28), cs((int32_t *)(forces + B * 12)) {}
};

// the slots a device assembly filled hold one array per QP of the batch
void set_assembled(mpc_qp *h, std::initializer_list<Slot *> slots, int batch) { for (Slot *s : slots) { s->stride = s->per; s->set = true; } h->batch = batch; }

// assemble the whole-body ID QPs from the scratch into the handle's A, b, C, l, which then hold one array per QP
int assemble_id(mpc_qp *h, const AsmScratch &s, int batch, double mu, double L, double W) {
  AsmArgs P;
  P.M = s.M; P.nle = s.nle; P.Jc = s.Jc; P.gamma = s.gamma; P.a = s.a; P.forces = s.forces; P.cs = s.cs; P.mu = mu; P.L = L; P.W = W;
  P.A = h->A.d; P.b = h->b.d; P.C = h->C.d; P.l = h->l.d; P.batch = batch;
  k_qp_assemble_id<<<batch, QP_THREADS, 0, h->stream>>>(P);
  CUQ(cudaGetLastError());
  set_assembled(h, {&h->A, &h->b, &h->C, &h->l}, batch);
  return 0;
}

// start of both assemblies from measured states: checks, then states x [B][57] into dstate, forces and contact flags into the scratch
int begin_from_state(mpc_qp *h, const char *fn, bool ikid, const mpc_solver *solver, int batch, const double *x, const double *forces, const int32_t *cs) {
  if (enter(h, fn)) return 1;
  if (!solver || !x || !forces || !cs) return fail(std::string(fn) + ": null solver handle / argument");
  if (h->n != 62 || h->ne != 40 || h->ni != 18 || (ikid && !h->box))
    return fail(std::string(fn) + (ikid ? ": handle is not the IKID shape (n 62, n_eq 40, n_in 18, box constraints)" : ": handle is not the whole-body ID shape (n 62, n_eq 40, n_in 18)"));
  if (batch <= 0 || batch > h->max_batch) return fail(std::string(fn) + ": batch out of range");
  const size_t B = batch;
  const AsmScratch s(h->dscratch, B);
  CUQ(cudaMemcpyAsync(h->dstate, x, 8 * B * 57, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.forces, forces, 8 * B * 12, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.cs, cs, 4 * B * 2, cudaMemcpyHostToDevice, h->stream));
  return 0;
}

// the IKID assembly's inputs beyond AsmScratch, for B QPs: the shared gains, then per QP the task errors and the task terms
constexpr size_t IKID_GAINS = 2 * 784 + 2 * 36 + 2 * 9, IKID_PER = 98 + 168 + 6 + 168 + 6;
struct IkidScratch {
  double *gains, *task, *Ag, *dAgv, *Jang, *dJang;
  IkidScratch(double *s, size_t B) : gains(s), task(gains + IKID_GAINS), Ag(task + B * 98), dAgv(Ag + B * 168), Jang(dAgv + B * 6), dJang(Jang + B * 168) {}
};

int launch(mpc_qp *h, const QPArgs &P, cudaStream_t stream) {
  if (P.batch <= 0) return 0;
  const int grid = P.batch; // one CTA per QP: QPs take different numbers of Newton steps, the hardware scheduler balances them
  CUQ(cudaEventRecord(h->ev0, stream));
  k_qp_solve<<<grid, QP_THREADS, h->smem_bytes, stream>>>(P);
  CUQ(cudaGetLastError());
  CUQ(cudaEventRecord(h->ev1, stream));
  return 0;
}

} // namespace

extern "C" {

const char *mpc_qp_last_error(void) { return g_err.c_str(); }

void mpc_qp_default_settings(mpc_qp_settings_t *s) {
  s->eps_abs = 1e-5; s->eps_rel = 0.0; s->rho = 1e-6; s->mu_eq = 1e-3; s->mu_in = 1e-1; s->alpha_bcl = 0.1; s->beta_bcl = 0.9;
  s->mu_update_factor = 0.1; s->mu_min_eq = 1e-4; s->mu_min_in = 1e-4; s->max_iter = 10000; s->max_iter_in = 1500;
  s->check_duality_gap = 0; s->warm_start = 0;
}

int32_t mpc_qp_abi_sizeof(int32_t which) { return which == 0 ? (int32_t)sizeof(mpc_qp_settings_t) : which == 1 ? (int32_t)sizeof(mpc_qp_info_t) : -1; }

void mpc_qp_destroy(mpc_qp_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  delete h;
}

mpc_qp_t *mpc_qp_create(int32_t n, int32_t n_eq, int32_t n_in, int32_t box, int32_t max_batch, int32_t device) {
  std::unique_ptr<mpc_qp> h(new mpc_qp); // a failure releases what was created so far
  return init_qp(h.get(), n, n_eq, n_in, box, max_batch, device) ? nullptr : h.release();
}

int32_t mpc_qp_update(mpc_qp_t *h, int32_t batch, const double *H, int64_t sH, const double *g, int64_t sg, const double *A, int64_t sA, const double *b,
                      int64_t sb, const double *C, int64_t sC, const double *l, int64_t sl, const double *u, int64_t su, const double *l_box, int64_t slb,
                      const double *u_box, int64_t sub) {
  if (enter(h, "mpc_qp_update")) return 1;
  if (batch <= 0 || batch > h->max_batch) return fail("mpc_qp_update: batch out of range");
  h->batch = batch;
  if (upload(h, h->H, H, sH, batch, "H") || upload(h, h->g, g, sg, batch, "g") || upload(h, h->A, A, sA, batch, "A") || upload(h, h->b, b, sb, batch, "b") ||
      upload(h, h->C, C, sC, batch, "C") || upload(h, h->l, l, sl, batch, "l") || upload(h, h->u, u, su, batch, "u"))
    return 1;
  if (h->box && (upload(h, h->lb, l_box, slb, batch, "l_box") || upload(h, h->ub, u_box, sub, batch, "u_box"))) return 1;
  return 0;
}

static int fill_args(mpc_qp *h, QPArgs &P, const mpc_qp_settings_t *settings) {
  if (!settings) return fail("null settings");
  P.phase = h->dphase;
  P.n = h->n; P.ne = h->ne; P.ni = h->ni; P.box = h->box; P.batch = h->batch;
  P.st = *settings;
  return 0;
}

int32_t mpc_qp_solve(mpc_qp_t *h, const mpc_qp_settings_t *settings, double *x, double *y, double *z, mpc_qp_info_t *info) {
  if (enter(h, "mpc_qp_solve")) return 1;
  if (h->batch <= 0) return fail("mpc_qp_solve: no data (call mpc_qp_update first)");
  if (!h->H.set || !h->g.set || (h->ne && (!h->A.set || !h->b.set)) || (h->ni && (!h->C.set || !h->l.set || !h->u.set)) || (h->box && (!h->lb.set || !h->ub.set)))
    return fail("mpc_qp_solve: QP data incomplete (init must pass every array of the declared shape)");
  QPArgs P;
  if (fill_args(h, P, settings)) return 1;
  const size_t B = h->batch;
  if (settings->warm_start) {
    if (!x || !y || !z) return fail("warm start needs x, y, z");
    CUQ(cudaMemcpyAsync(h->dx, x, 8 * B * h->n, cudaMemcpyHostToDevice, h->stream));
    if (h->ne) CUQ(cudaMemcpyAsync(h->dy, y, 8 * B * h->ne, cudaMemcpyHostToDevice, h->stream));
    if (h->nz) CUQ(cudaMemcpyAsync(h->dz, z, 8 * B * h->nz, cudaMemcpyHostToDevice, h->stream));
  }
  P.H = h->H.d; P.sH = h->H.stride; P.g = h->g.d; P.sg = h->g.stride; P.A = h->A.d; P.sA = h->A.stride; P.b = h->b.d; P.sb = h->b.stride;
  P.C = h->C.d; P.sC = h->C.stride; P.l = h->l.d; P.sl = h->l.stride; P.u = h->u.d; P.su = h->u.stride;
  P.lb = h->lb.d; P.slb = h->lb.stride; P.ub = h->ub.d; P.sub = h->ub.stride;
  P.x = h->dx; P.y = h->dy; P.z = h->dz; P.info = h->dinfo;
  if (launch(h, P, h->stream)) return 1;
  if (x) CUQ(cudaMemcpyAsync(x, h->dx, 8 * B * h->n, cudaMemcpyDeviceToHost, h->stream));
  if (y && h->ne) CUQ(cudaMemcpyAsync(y, h->dy, 8 * B * h->ne, cudaMemcpyDeviceToHost, h->stream));
  if (z && h->nz) CUQ(cudaMemcpyAsync(z, h->dz, 8 * B * h->nz, cudaMemcpyDeviceToHost, h->stream));
  if (info) CUQ(cudaMemcpyAsync(info, h->dinfo, sizeof(mpc_qp_info_t) * B, cudaMemcpyDeviceToHost, h->stream));
  CUQ(cudaStreamSynchronize(h->stream));
  return 0;
}

int32_t mpc_qp_solve_device(mpc_qp_t *h, int32_t batch, const mpc_qp_settings_t *settings, uint64_t H, int64_t sH, uint64_t g, int64_t sg, uint64_t A, int64_t sA,
                            uint64_t b, int64_t sb, uint64_t C, int64_t sC, uint64_t l, int64_t sl, uint64_t u, int64_t su, uint64_t l_box, int64_t slb,
                            uint64_t u_box, int64_t sub, uint64_t x, uint64_t y, uint64_t z, uint64_t info, uint64_t stream) {
  if (enter(h, "mpc_qp_solve_device")) return 1;
  if (batch <= 0) return fail("mpc_qp_solve_device: batch out of range");
  QPArgs P;
  const bool all_caller_owned = H && g && (A || !h->ne) && (b || !h->ne) && (C || !h->ni) && (l || !h->ni) && (u || !h->ni) && (!h->box || (l_box && u_box)) && x && y && z && info;
  if (batch > h->max_batch && !all_caller_owned) return fail("mpc_qp_solve_device: batch above the handle's capacity needs caller-owned buffers for every array");
  h->batch = batch;
  if (fill_args(h, P, settings)) return 1;
  auto pick = [](uint64_t p, int64_t s, const Slot &sl, const double *&out, long long &so) { if (p) { out = (const double *)p; so = s; } else { out = sl.d; so = sl.stride; } };
  pick(H, sH, h->H, P.H, P.sH); pick(g, sg, h->g, P.g, P.sg); pick(A, sA, h->A, P.A, P.sA); pick(b, sb, h->b, P.b, P.sb); pick(C, sC, h->C, P.C, P.sC);
  pick(l, sl, h->l, P.l, P.sl); pick(u, su, h->u, P.u, P.su); pick(l_box, slb, h->lb, P.lb, P.slb); pick(u_box, sub, h->ub, P.ub, P.sub);
  P.x = x ? (double *)x : h->dx; P.y = y ? (double *)y : h->dy; P.z = z ? (double *)z : h->dz;
  P.info = info ? (mpc_qp_info_t *)info : h->dinfo;
  return launch(h, P, stream ? (cudaStream_t)stream : h->stream);
}

/* instrumented builds (-DMPC_QP_PHASE_TIMING, never the product library): cycles per phase summed over the QPs since the last call */
int32_t mpc_qp_debug_phases(mpc_qp_t *h, double *out8) {
  if (enter(h, "mpc_qp_debug_phases")) return 1;
  long long c[8] = {0};
  if (h->dphase) { CUQ(cudaMemcpyAsync(c, h->dphase, 64, cudaMemcpyDeviceToHost, h->stream)); CUQ(cudaMemsetAsync(h->dphase, 0, 64, h->stream)); }
  CUQ(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < 8; i++) out8[i] = (double)c[i];
  return 0;
}

double mpc_qp_last_device_ms(mpc_qp_t *h) {
  if (enter(h, "mpc_qp_last_device_ms")) return -1.0;
  float ms = 0;
  if (cudaEventSynchronize(h->ev1) != cudaSuccess || cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.0;
  return ms;
}

int32_t mpc_qp_assemble_id(mpc_qp_t *h, int32_t batch, const double *M, const double *nle, const double *Jc, const double *gamma, const double *a,
                           const double *forces, const int32_t *cs, double mu, double L, double W) {
  if (enter(h, "mpc_qp_assemble_id")) return 1;
  if (h->n != 62 || h->ne != 40 || h->ni != 18) return fail("mpc_qp_assemble_id: handle is not the whole-body ID shape (n 62, n_eq 40, n_in 18)");
  if (batch <= 0 || batch > h->max_batch) return fail("mpc_qp_assemble_id: batch out of range");
  const size_t B = batch;
  const AsmScratch s(h->dscratch, B);
  CUQ(cudaMemcpyAsync(s.M, M, 8 * B * 784, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.nle, nle, 8 * B * 28, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.Jc, Jc, 8 * B * 336, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.gamma, gamma, 8 * B * 12, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.a, a, 8 * B * 28, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.forces, forces, 8 * B * 12, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(s.cs, cs, 4 * B * 2, cudaMemcpyHostToDevice, h->stream));
  return assemble_id(h, s, batch, mu, L, W);
}

int32_t mpc_qp_assemble_id_from_state(mpc_qp_t *h, struct mpc_solver *solver, int32_t batch, const double *x, const double *a, const double *forces,
                                      const int32_t *cs, double mu, double L, double W, double kd) {
  if (begin_from_state(h, "mpc_qp_assemble_id_from_state", false, solver, batch, x, forces, cs)) return 1;
  const size_t B = batch;
  // M, nle, Jc and gamma come from the rigid-body terms of the states (held in dstate with the frame velocities behind them)
  const AsmScratch s(h->dscratch, B);
  CUQ(cudaMemcpyAsync(s.a, a, 8 * B * 28, cudaMemcpyHostToDevice, h->stream));
  if (mpc_rbd_terms_device(solver, batch, (uint64_t)h->dstate.get(), (uint64_t)s.M, (uint64_t)s.nle, (uint64_t)s.Jc, (uint64_t)s.gamma, (uint64_t)(h->dstate + B * 57), (uint64_t)h->stream.get()) != 0)
    return fail(mpc_last_error());
  k_qp_gamma<<<(batch * 12 + 127) / 128, 128, 0, h->stream>>>(s.gamma, h->dstate + B * 57, s.cs, kd, batch);
  return assemble_id(h, s, batch, mu, L, W);
}

int32_t mpc_qp_assemble_ikid_from_state(mpc_qp_t *h, struct mpc_solver *solver, int32_t batch, const double *x, const double *task, const double *forces,
                                        const int32_t *cs, const double weights[5], const double *gains, const int32_t frame_body[2],
                                        const double frame_place[2][12], double mu, double L, double W) {
  if (begin_from_state(h, "mpc_qp_assemble_ikid_from_state", true, solver, batch, x, forces, cs)) return 1;
  if (!task || !weights || !gains || !frame_body || !frame_place) return fail("mpc_qp_assemble_ikid_from_state: null argument");
  if (h->dikid.ensure(IKID_GAINS + (size_t)h->max_batch * IKID_PER) != cudaSuccess)
    return fail("mpc_qp_assemble_ikid_from_state: cudaMalloc of the IKID scratch failed");
  const size_t B = batch;
  // M, nle, Jc and dJv (in the gamma slot) come from the rigid-body terms of the states, the task terms go to the IKID scratch
  const AsmScratch s(h->dscratch, B);
  const IkidScratch k(h->dikid, B);
  CUQ(cudaMemcpyAsync(k.task, task, 8 * B * 98, cudaMemcpyHostToDevice, h->stream));
  CUQ(cudaMemcpyAsync(k.gains, gains, 8 * IKID_GAINS, cudaMemcpyHostToDevice, h->stream));
  if (mpc_ikid_terms_device(solver, batch, (uint64_t)h->dstate.get(), frame_body, frame_place, (uint64_t)s.M, (uint64_t)s.nle, (uint64_t)s.Jc, (uint64_t)s.gamma,
                            (uint64_t)k.Ag, (uint64_t)k.dAgv, (uint64_t)k.Jang, (uint64_t)k.dJang, (uint64_t)h->stream.get()) != 0)
    return fail(mpc_last_error());
  IkidAsmArgs P;
  P.M = s.M; P.nle = s.nle; P.Jc = s.Jc; P.dJv = s.gamma; P.Ag = k.Ag; P.dAgv = k.dAgv; P.Jang = k.Jang; P.dJang = k.dJang; P.task = k.task;
  P.forces = s.forces; P.gains = k.gains; P.cs = s.cs;
  for (int i = 0; i < 5; i++) P.wt[i] = weights[i];
  P.mu = mu; P.L = L; P.W = W;
  P.H = h->H.d; P.g = h->g.d; P.A = h->A.d; P.b = h->b.d; P.C = h->C.d; P.l = h->l.d; P.batch = batch;
  k_qp_assemble_ikid<<<batch, QP_THREADS, 0, h->stream>>>(P);
  CUQ(cudaGetLastError());
  set_assembled(h, {&h->H, &h->g, &h->A, &h->b, &h->C, &h->l}, batch);
  return 0;
}

} // extern "C"
