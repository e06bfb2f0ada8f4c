// TEST-ONLY host emulation of a batch with per-instance models (mpc_set_instance_models): the kernel sources of emu.cpp (included
// here, so this library carries every emu_* entry point too) run with Ws::model = one DevModel per instance and model_stride 1, the
// models built and checked by build_instance_models (csrc/model.cuh), the same code as the C-ABI.  Built by tests/emu_models_lib.py.
#include "emu.cpp"
#include <string>

static std::string g_models_err;
extern "C" const char *emu_models_last_error() { return g_models_err.c_str(); }

// emu_solve with robots / cfgs [batch] (null: the shared rb / cfg for every instance); a rejected model returns 1 with the message in
// emu_models_last_error()
extern "C" int emu_solve_models(const mpc_robot_t *rb, const mpc_config_t *cfg, const mpc_robot_t *robots, const mpc_config_t *cfgs, int batch,
                                const mpc_knot_t *knots, const mpc_term_t *terms, const double *x0, double *xs, double *us, double *K, double *vs,
                                double *lams, mpc_info_t *info, int max_iters) {
  std::vector<DevModel> shared(1), models(batch);
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, shared.data(), &err)) { g_models_err = err; return 1; }
  g_models_err = build_instance_models(shared[0], robots, cfgs, batch, models.data());
  if (!g_models_err.empty()) return 1;
  EmuBackend be;
  Ws &w = be.w;
  init_ws(w, *cfg, batch, models.data());
  w.model_stride = 1;
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
  run_loop(be, w, max_iters, w.sc);
  std::memcpy(xs, w.xs, 8 * batch * T1 * w.nx);
  std::memcpy(us, w.us, 8 * batch * w.T * w.m);
  if (K) std::memcpy(K, w.Kfb, 8 * (size_t)batch * w.T * w.m * w.n);
  if (vs) std::memcpy(vs, w.vs, 8 * batch * T1 * w.nc);
  if (lams) std::memcpy(lams, w.lams, 8 * batch * T1 * w.n);
  if (info) for (int b = 0; b < batch; b++) info[b] = info_of(w.st[b]);
  for (void *p : allocs) free(p);
  return 0;
}
