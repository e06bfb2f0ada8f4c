// TEST-ONLY host emulation of the solver with the time-parallel LQ solve (cfg.lq_legs >= 2): the kernel sources of
// mpc_benchmark_b200/csrc compiled with -DMPC_HOST_EMU (PAR_FOR = serial loop, SYNC = no-op), the phases of riccati_par.cuh run
// as the CUDA backend launches them (A and C over every (instance, leg), then B and D over every instance).  Never loaded by the
// product package and not a fallback.
#define MPC_HOST_EMU 1
#include "../../mpc_benchmark_b200/csrc/driver.hpp"
#include "../../mpc_benchmark_b200/csrc/ws_alloc.hpp"
#include <cstdlib>
#include <cstring>
#include <vector>

using namespace mpcdev;

struct LegEmuBackend {
  Ws w;
  LegWs lw{};
  int legs = 0;
  std::vector<double> smem;
  LegEmuBackend() : smem(40000, 0.0) {}
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
      if (legs < 2) { for (int i = 0; i < n; i++) riccati_dispatch<KIND>(w, list[i], smem.data()); return; }
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

// emu_solve of tests/emu/emu.cpp with cfg->lq_legs honoured; multipliers vs / lams are the warm start (in) and the result (out)
extern "C" int emu_solve_legs(const mpc_robot_t *rb, const mpc_config_t *cfg, int batch, const mpc_knot_t *knots, const mpc_term_t *terms,
                              const double *x0, double *xs, double *us, double *K, double *vs, double *lams, mpc_info_t *info, int max_iters) {
  DevModel *model = new DevModel;
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, model, &err)) { delete model; return 1; }
  LegEmuBackend be;
  Ws &w = be.w;
  init_ws(w, *cfg, batch, model);
  std::vector<void *> allocs;
  auto calloc_ = [&](size_t bytes) { void *p = calloc(bytes ? bytes : 8, 1); allocs.push_back(p); return p; };
  alloc_ws(w, calloc_);
  be.legs = cfg->lq_legs;
  if (be.legs >= 2) alloc_leg_ws(w, be.lw, be.legs, calloc_);
  const size_t T1 = w.T + 1;
  std::memcpy(w.knots, knots, sizeof(mpc_knot_t) * batch * w.T);
  std::memcpy(w.terms, terms, sizeof(mpc_term_t) * batch);
  std::memcpy(w.x0, x0, 8 * batch * w.nx);
  std::memcpy(w.vs, vs, 8 * batch * T1 * w.nc);
  std::memcpy(w.lams, lams, 8 * batch * T1 * w.n);
  for (int b = 0; b < batch; b++) init_instance(w, b, xs, us, max_iters);
  run_loop(be, w, max_iters, w.sc);
  std::memcpy(xs, w.xs, 8 * batch * T1 * w.nx);
  std::memcpy(us, w.us, 8 * batch * w.T * w.m);
  std::memcpy(K, w.Kfb, 8 * (size_t)batch * w.T * w.m * w.n);
  std::memcpy(vs, w.vs, 8 * batch * T1 * w.nc);
  std::memcpy(lams, w.lams, 8 * batch * T1 * w.n);
  for (int b = 0; b < batch; b++) info[b] = info_of(w.st[b]);
  for (void *p : allocs) free(p);
  delete model;
  return 0;
}
