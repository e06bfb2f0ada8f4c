// TEST-ONLY host emulation of the CUDA kernel sources (mpc_benchmark_b200/csrc/*.cuh compiled with
// -DMPC_HOST_EMU: PAR_FOR = serial loop, SYNC = no-op).  Lets the CPU test-suite check kernel LOGIC against the
// oracle without a GPU.  It is never loaded by the product package and is not a fallback.
#define MPC_HOST_EMU 1
#include "../../mpc_benchmark_b200/csrc/driver.hpp"
#include "../../mpc_benchmark_b200/csrc/ws_alloc.hpp"
#include "../../mpc_benchmark_b200/csrc/qp.cuh"
#include "../../mpc_benchmark_b200/csrc/rbd_terms.cuh"
#include "../../mpc_benchmark_b200/csrc/gait_host.hpp"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace mpcdev;

struct EmuBackend {
  Ws w;
  LegWs lw{}; // allocated for cfg.lq_legs >= 2: the time-parallel LQ solve (riccati_par.cuh)
  std::vector<double> smem;
  EmuBackend() : smem(40000, 0.0) {}
  void reset_counters() { for (int i = 0; i < 4; i++) w.counters[i] = 0; }
  void eval(bool d, const int32_t *list, int n) {
    dispatch_kind(w.kind, [&](auto kind) {
      for (int i = 0; i < n; i++)
        for (int k = 0; k <= w.T; k++) {
          if (d) eval_dispatch<decltype(kind)::value, true>(w, list[i], k, smem.data());
          else eval_dispatch<decltype(kind)::value, false>(w, list[i], k, smem.data());
        }
    });
  }
  void decide_eval(const int32_t *list, int n, int32_t *next_eval) { double red[8]; for (int i = 0; i < n; i++) mpcdev::decide_eval(w, list[i], red, next_eval); }
  void riccati(const int32_t *list, int n) {
    dispatch_kind(w.kind, [&](auto kind) {
      constexpr int KIND = decltype(kind)::value;
      if (lw.L < 2) { for (int i = 0; i < n; i++) riccati_dispatch<KIND>(w, list[i], smem.data()); return; }
      // the four phases as the CUDA backend launches them: A and C over every (instance, leg), B and D over every instance
      double sh[64];
      for (int e = 0; e < n * lw.L; e++) ric_par_legs<KIND>(w, lw, list[e / lw.L], e % lw.L);
      for (int i = 0; i < n; i++) ric_par_consensus<KIND>(w, lw, list[i], sh);
      for (int e = 0; e < n * lw.L; e++) ric_par_resolve<KIND>(w, lw, list[e / lw.L], e % lw.L, smem.data());
      for (int i = 0; i < n; i++) ric_par_finish<KIND>(w, lw, list[i]);
    });
  }
  void apply_step(const int32_t *list, int n) { w.counters[0] = 0; for (int i = 0; i < n; i++) mpcdev::apply_step(w, list[i]); }
  void decide_ls(const int32_t *list, int n, int32_t *ls_out, int32_t *next_eval) {
    double red[8];
    for (int i = 0; i < n; i++) mpcdev::decide_ls(w, list[i], red, ls_out, next_eval);
  }
  void rollout_ls(const int32_t *list, int n, int32_t *next_eval) {
    double red[8], xv[256];
    dispatch_kind(w.kind, [&](auto kind) { for (int i = 0; i < n; i++) rollout_linesearch<decltype(kind)::value>(w, list[i], smem.data(), xv, red, next_eval); });
  }
  void read_counters(int *c) { for (int i = 0; i < 4; i++) c[i] = w.counters[i]; }
};

static std::string g_err;
extern "C" const char *emu_last_error() { return g_err.c_str(); }

// robots / cfgs [batch] are nullable, as in mpc_set_instance_models.  If either is given, every instance gets its own DevModel
// (Ws::model_stride 1), built and checked by build_instance_models like the C-ABI's, a null array standing for rb / cfg.  With both null
// the batch shares one DevModel (model_stride 0).  A rejected model returns 1 with the message in emu_last_error().
extern "C" int emu_solve(const mpc_robot_t *rb, const mpc_config_t *cfg, const mpc_robot_t *robots, const mpc_config_t *cfgs, int batch,
                         const mpc_knot_t *knots, const mpc_term_t *terms, const double *x0, double *xs, double *us, double *K, double *vs,
                         double *lams, mpc_info_t *info, double *stage0, int max_iters,
                         double *lq_dump /* optional: AB,H,g of instance 0 after the first derivative pass */) {
  static_assert(sizeof(FullWsT<true>) <= 40000 * 8 && sizeof(KinoWsT<true>) <= 40000 * 8, "smem");
  std::vector<DevModel> shared(1), models;
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, shared.data(), &err)) { g_err = err; return 1; }
  if (robots || cfgs) {
    models.resize(batch);
    g_err = build_instance_models(shared[0], robots, cfgs, batch, models.data());
    if (!g_err.empty()) return 1;
  }
  EmuBackend be;
  Ws &w = be.w;
  init_ws(w, *cfg, batch, models.empty() ? shared.data() : models.data());
  w.model_stride = models.empty() ? 0 : 1;
  std::vector<void *> allocs;
  auto calloc_ = [&](size_t bytes) { void *p = calloc(bytes ? bytes : 8, 1); allocs.push_back(p); return p; };
  alloc_ws(w, calloc_);
  if (cfg->lq_legs >= 2) alloc_leg_ws(w, be.lw, cfg->lq_legs, calloc_);
  const size_t T1 = w.T + 1;
  std::memcpy(w.knots, knots, sizeof(mpc_knot_t) * batch * w.T);
  std::memcpy(w.terms, terms, sizeof(mpc_term_t) * batch);
  std::memcpy(w.x0, x0, 8 * batch * w.nx);
  if (vs) std::memcpy(w.vs, vs, 8 * batch * T1 * w.nc);
  if (lams) std::memcpy(w.lams, lams, 8 * batch * T1 * w.n);
  for (int b = 0; b < batch; b++) init_instance(w, b, xs, us, max_iters);
  if (lq_dump) { // single derivative pass, dump instance 0
    be.reset_counters(); be.eval(true, eval_list(w, 0), w.B); be.decide_eval(eval_list(w, 0), w.B, eval_list(w, 1));
    size_t o = 0;
    auto put = [&](const double *p, size_t n) { std::memcpy(lq_dump + o, p, 8 * n); o += n; };
    put(w.AB, (size_t)w.T * w.n * w.nz); put(w.H, T1 * w.nz * w.nz); put(w.g, T1 * w.nz); put(w.gap, (size_t)w.T * w.n); put(w.h, T1 * w.nc);
    put(w.scal, T1 * SC_COUNT);
  } else run_loop(be, w, max_iters, w.sc);
  if (getenv("EMU_NCA_HIST")) { // test tooling: active-row counts per knot of the last pass (sizes the kernel's shared-memory fast path)
    for (int b = 0; b < batch; b++) { fprintf(stderr, "nca[%d]:", b); for (size_t k = 0; k < T1; k++) fprintf(stderr, " %d", w.nca[b * T1 + k]); fprintf(stderr, "\n"); }
  }
  std::memcpy(xs, w.xs, 8 * batch * T1 * w.nx);
  std::memcpy(us, w.us, 8 * batch * w.T * w.m);
  if (K) std::memcpy(K, w.Kfb, 8 * (size_t)batch * w.T * w.m * w.n);
  if (vs) std::memcpy(vs, w.vs, 8 * batch * T1 * w.nc);
  if (lams) std::memcpy(lams, w.lams, 8 * batch * T1 * w.n);
  for (int b = 0; b < batch; b++) {
    if (info) info[b] = info_of(w.st[b]);
    if (stage0) { std::memcpy(stage0 + b * 68, w.xdot + b * T1 * 56, 8 * 56); std::memcpy(stage0 + b * 68 + 56, w.lamc + b * T1 * 12, 8 * 12); }
  }
  for (void *p : allocs) free(p);
  return 0;
}

// ---- batched dense QP (qp.cuh) run serially: same source as k_qp_solve / k_qp_assemble_id
extern "C" int emu_qp_solve(int n, int ne, int ni, int box, int batch, const mpc_qp_settings_t *st, const double *H, long sH, const double *g, long sg,
                            const double *A, long sA, const double *b, long sb, const double *C, long sC, const double *l, long sl, const double *u, long su,
                            const double *lb, long slb, const double *ub, long sub, double *x, double *y, double *z, mpc_qp_info_t *info) {
  QPArgs P;
  P.n = n; P.ne = ne; P.ni = ni; P.box = box; P.batch = batch; P.st = *st;
  P.H = H; P.sH = sH; P.g = g; P.sg = sg; P.A = A; P.sA = sA; P.b = b; P.sb = sb; P.C = C; P.sC = sC; P.l = l; P.sl = sl; P.u = u; P.su = su;
  P.lb = lb; P.slb = slb; P.ub = ub; P.sub = sub; P.x = x; P.y = y; P.z = z; P.info = info;
  std::vector<double> smem(qp_smem_doubles(n, ne, ni, box), 0.0);
  for (int i = 0; i < batch; i++) qp_solve_group(P, i, smem.data());
  return 0;
}
extern "C" void emu_qp_assemble_id(int batch, const double *M, const double *nle, const double *Jc, const double *gamma, const double *a, const double *forces,
                                   const int32_t *cs, double mu, double L, double W, double *A, double *b, double *C, double *l) {
  for (int i = 0; i < batch; i++)
    qp_assemble_id_group(M + i * 784, nle + i * 28, Jc + i * 336, gamma + i * 12, a + i * 28, forces + i * 12, cs + i * 2, mu, L, W, A + i * 2480, b + i * 40,
                         C + i * 1116, l + i * 18);
}

// ---- rigid-body terms in front of the whole-body QPs (rbd_terms.cuh), serial
extern "C" int emu_rbd_terms(const mpc_robot_t *rb, const mpc_config_t *cfg, int count, const double *x, double *M, double *nle, double *Jc, double *dJv, double *vf) {
  DevModel *model = new DevModel;
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, model, &err)) { delete model; return 1; }
  std::vector<double> smem(sizeof(FullWsT<false>) / 8 + 8, 0.0);
  FullWsT<false> &w = *reinterpret_cast<FullWsT<false> *>(smem.data());
  for (int i = 0; i < count; i++)
    rbd_terms_group(*model, x + (size_t)i * 57, w, M + (size_t)i * 784, nle + (size_t)i * 28, Jc + (size_t)i * 336, dJv + (size_t)i * 12, vf + (size_t)i * 12);
  delete model;
  return 0;
}

// ---- IKID task terms (k_ikid_terms) of `count` states, serial
extern "C" int emu_ikid_terms(const mpc_robot_t *rb, const mpc_config_t *cfg, int count, const double *x, const int32_t *frame_body, const double *frame_place,
                              double *M, double *nle, double *Jc, double *dJv, double *Ag, double *dAgv, double *Jang, double *dJang) {
  DevModel *model = new DevModel;
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, model, &err)) { delete model; return 1; }
  std::vector<double> smem(sizeof(FullWsT<false>) / 8 + 8, 0.0);
  FullWsT<false> &w = *reinterpret_cast<FullWsT<false> *>(smem.data());
  for (int i = 0; i < count; i++)
    ikid_terms_group(*model, x + (size_t)i * 57, frame_body, frame_place, w, M + (size_t)i * 784, nle + (size_t)i * 28, Jc + (size_t)i * 336, dJv + (size_t)i * 12,
                     Ag + (size_t)i * 168, dAgv + (size_t)i * 6, Jang + (size_t)i * 168, dJang + (size_t)i * 6);
  delete model;
  return 0;
}
// k_qp_assemble_ikid, serial
extern "C" void emu_qp_assemble_ikid(int batch, const double *M, const double *nle, const double *Jc, const double *dJv, const double *Ag, const double *dAgv,
                                     const double *Jang, const double *dJang, const double *task, const double *forces, const int32_t *cs, const double *weights,
                                     const double *gains, double mu, double L, double W, double *H, double *g, double *A, double *b, double *C, double *l) {
  double sm[24 * 28 + 24 + 12 + 28];
  for (int i = 0; i < batch; i++)
    qp_assemble_ikid_group(M + i * 784, nle + i * 28, Jc + i * 336, dJv + i * 12, Ag + i * 168, dAgv + i * 6, Jang + i * 168, dJang + i * 6, task + i * 98,
                           forces + i * 12, cs + i * 2, weights, gains, mu, L, W, sm, H + (size_t)i * 3844, g + i * 62, A + (size_t)i * 2480, b + i * 40,
                           C + (size_t)i * 1116, l + i * 18);
}

// ---- device gait generator (gait.cuh) run serially: `ticks` ticks of `batch` robots; lf / rf [ticks][batch][12] measured sole placements;
// knots_out [ticks][batch][T], terms_out [ticks][batch]
extern "C" int emu_gait(int kind, int T, const mpc_gait_t *gait, int batch, const int32_t *mirror, const double *urefs, int ticks, const double *lf,
                        const double *rf, mpc_knot_t *knots_out, mpc_term_t *terms_out) {
  GaitCfg g;
  std::memset(&g, 0, sizeof g);
  gait_fill_cfg(*gait, kind, T, g);
  std::vector<int8_t> phases;
  gait_build_schedule(*gait, T, phases, g);
  g.phases = phases.data();
  g.urefs = urefs;
  std::vector<GaitRobot> rs = gait_init_robots(*gait, batch, mirror);
  double sm[16];
  for (int t = 0; t < ticks; t++)
    for (int b = 0; b < batch; b++)
      gait_tick_group(g, rs[b], t, lf + ((size_t)t * batch + b) * 12, rf + ((size_t)t * batch + b) * 12, knots_out + ((size_t)t * batch + b) * T,
                      terms_out + (size_t)t * batch + b, sm);
  return 0;
}
