// Device-side ProxDDP state machine shared by the CUDA kernels (solver.cu).
//
// Replaces the control flow of aligator::SolverProxDDPTpl::run / innerLoop (reached from
// fulldynamic_talos.py:393-397,540) with a per-instance state machine so that thousands of independent MPC
// instances advance in lock-step kernel launches:
//   MODE_EVAL --(eval<deriv> + decide_eval)--> MODE_STEP --(riccati)--> MODE_LS --(apply_step, eval<values>,
//   decide_ls)*--> MODE_EVAL ... --> MODE_DONE
// Constants of the BCL outer loop / Armijo linesearch: DESIGN.md "solver constants" (SURVEY App. A6).
#pragma once
#include "eval_cent.cuh"
#include "eval_full.cuh"
#include "eval_kino.cuh"
#include "riccati.cuh"
#include "riccati_fast.cuh"
#include "riccati_par.cuh"

namespace mpcdev {

enum { MODE_EVAL = 0, MODE_STEP = 1, MODE_LS = 2, MODE_DONE = 3 };

struct SolverConst {
  double tol, mu_init;
  int max_al_iters;
  double prim_alpha, prim_beta, dual_alpha, dual_beta, mu_update_factor, mu_lower_bound;
  double reg_init, reg_min, reg_max, reg_inc, reg_dec;
  double ls_c1, ls_alpha_min, ls_contr_min, ls_contr_max, ls_dphi_rel;
  int ls_max_steps;
  int rollout; // 0 ROLLOUT_LINEAR (every reference script), 1 ROLLOUT_NONLINEAR (fused rollout + linesearch kernel)
};
inline SolverConst default_consts(double tol, double mu_init, int rollout = 0) {
  SolverConst c;
  c.tol = tol; c.mu_init = mu_init; c.max_al_iters = 100;
  c.prim_alpha = 0.1; c.prim_beta = 0.9; c.dual_alpha = 1.0; c.dual_beta = 1.0; c.mu_update_factor = 0.01; c.mu_lower_bound = 1e-8;
  c.reg_init = 1e-9; c.reg_min = 1e-10; c.reg_max = 1e9; c.reg_inc = 10.0; c.reg_dec = 1.0 / 3.0;
  c.ls_c1 = 1e-4; c.ls_alpha_min = 1e-7; c.ls_contr_min = 0.5; c.ls_contr_max = 0.8; c.ls_max_steps = 20; c.ls_dphi_rel = 1e-11;
  c.rollout = rollout;
  return c;
}

struct InstState {
  double mu, inner_tol, prim_tol, preg;
  double prim_infeas, dual_infeas, inner_crit, traj_cost, merit;
  double dphi0, alpha, a_prev, phi_prev;
  int32_t num_iters, al_iters, conv, status, mode, ls_it, max_iters, ls_evals;
};

struct Ws {
  int B, T, kind, nx, n, m, nc, nz;
  const DevModel *model;
  int model_stride; // DevModels between consecutive instances: 0 = one model shared by the batch, 1 = one per instance
  SolverConst sc;
  mpc_knot_t *knots; mpc_term_t *terms; double *x0;
  double *xs, *us, *vs, *lams, *vs_prev, *lams_prev;
  double *txs, *tus, *tvs, *tlams;
  double *dxs, *dus, *dvs, *dlams;
  double *AB, *H, *lxu, *g, *T6, *E6, *gE, *fbar, *dbar, *vplus, *lplus, *CDact;
  int32_t *nca, *act_idx;
  double *gap, *h, *scal, *tscal, *xdot, *lamc;
  double *W, *pt, *K, *Kfb, *dphi;
  double *ric_scratch; size_t ric_scratch_stride; // per-instance scratch of the Riccati kernel (doubles per instance)
  InstState *st;
  int32_t *counters; // [0] instances still in MODE_LS (next ls list), [2] instances to evaluate in the next pass
  double *phase;     // 16 doubles: per-phase cycle counters of instance 0 (MPC_PHASE_TIMING builds)
  int32_t *lists;    // [4][B] compacted instance lists: 0,1 = evaluation lists (double-buffered), 2,3 = linesearch lists
};
// the robot / problem constants of instance b
HDH const DevModel &model_of(const Ws &w, int b) { return w.model[(size_t)b * w.model_stride]; }
HDH int32_t *eval_list(const Ws &w, int which) { return w.lists + (size_t)(which & 1) * w.B; }
HDH int32_t *ls_list(const Ws &w, int which) { return w.lists + (size_t)(2 + (which & 1)) * w.B; }

HD KnotIO make_io(const Ws &w, int b, int k, bool trial) {
  KnotIO io;
  const size_t T1 = (size_t)w.T + 1, kb = (size_t)b * T1 + k, kT = (size_t)b * w.T + k;
  const double *X = trial ? w.txs : w.xs, *U = trial ? w.tus : w.us, *V = trial ? w.tvs : w.vs, *L = trial ? w.tlams : w.lams;
  io.x = X + kb * w.nx;
  io.u = (k < w.T) ? U + kT * w.m : nullptr;
  io.xn = (k < w.T) ? X + (kb + 1) * w.nx : nullptr;
  io.kn = (k < w.T) ? w.knots + kT : nullptr;
  io.tm = w.terms + b;
  io.v = V + kb * w.nc; io.v_prev = w.vs_prev + kb * w.nc;
  io.lam_k = L + kb * w.n;
  io.lam_n = (k < w.T) ? L + (kb + 1) * w.n : nullptr;
  io.lam_n_prev = (k < w.T) ? w.lams_prev + (kb + 1) * w.n : nullptr;
  io.mu = w.st[b].mu; io.preg = w.st[b].preg; io.k = k; io.T = w.T;
  io.AB = w.AB + kT * w.n * w.nz; io.H = w.H + kb * w.nz * w.nz; io.lxu = w.lxu + kb * w.nz; io.g = w.g + kb * w.nz;
  io.T6 = w.T6 + kT * 36; io.E6 = w.E6 + kT * 36; io.gE_next = w.gE + (kb + 1) * 6;
  io.fbar = w.fbar + kT * w.n; io.dbar = w.dbar + kb * w.nc; io.vplus = w.vplus + kb * w.nc; io.lplus = w.lplus + (kb + 1) * w.n;
  io.CDact = w.CDact + kb * w.nc * w.nz; io.nca = w.nca + kb; io.act_idx = w.act_idx + kb * w.nc;
  io.gap = w.gap + kT * w.n; io.h = w.h + kb * w.nc; io.scal = (trial ? w.tscal : w.scal) + kb * SC_COUNT;
  io.xdot = w.xdot + kb * 56; io.lamc = w.lamc + kb * 12;
  io.scratch = (k < w.T) ? w.W + kT * w.n * w.nz : nullptr;
  io.slack = nullptr; io.xn_out = nullptr;
  io.phase_out = (b == 0 && k == 1) ? w.phase + (trial ? 32 : 16) : nullptr;
  return io;
}

// ---- run() prologue for one instance (one CTA): copy the warm start, force x0, reset BCL state
HD void init_instance(const Ws &w, int b, const double *xs_in, const double *us_in, int max_iters) {
  const size_t T1 = (size_t)w.T + 1;
  PAR_FOR(i, (int)(T1 * w.nx)) w.xs[b * T1 * w.nx + i] = xs_in[b * T1 * w.nx + i];
  PAR_FOR(i, w.T * w.m) w.us[(size_t)b * w.T * w.m + i] = us_in[(size_t)b * w.T * w.m + i];
  SYNC();
  // force_initial_condition is uniform over the batch (build_instance_models): instance 0's model answers for every instance
  if (w.model->cfg.force_initial_condition) PAR_FOR(i, w.nx) w.xs[b * T1 * w.nx + i] = w.x0[(size_t)b * w.nx + i];
  PAR_FOR(i, (int)(T1 * w.nc)) w.vs_prev[b * T1 * w.nc + i] = w.vs[b * T1 * w.nc + i];
  PAR_FOR(i, (int)(T1 * w.n)) w.lams_prev[b * T1 * w.n + i] = w.lams[b * T1 * w.n + i];
  PAR_FOR(i, 6) w.gE[b * T1 * 6 + i] = 0.0;
  ONE_THREAD {
    eval_list(w, 0)[b] = b;
    InstState &s = w.st[b];
    const SolverConst &c = w.sc;
    s.mu = c.mu_init; s.preg = c.reg_init;
    s.prim_tol = fmax(pow(s.mu, c.prim_alpha), c.tol);
    s.inner_tol = fmax(pow(s.mu, c.dual_alpha), c.tol);
    s.num_iters = 0; s.al_iters = 0; s.conv = 0; s.status = 1; s.ls_it = 0; s.max_iters = max_iters; s.ls_evals = 0;
    s.mode = (max_iters > 0) ? MODE_EVAL : MODE_DONE;
    s.prim_infeas = s.dual_infeas = s.inner_crit = s.traj_cost = s.merit = 0;
    s.dphi0 = s.alpha = s.a_prev = s.phi_prev = 0;
  }
}

// ---- after eval<deriv>: reduce the per-knot partials, finish the dual residual (base block of E^T lam), BCL logic
HD void decide_eval(const Ws &w, int b, double *red /* shared, >= 8 doubles */, int32_t *next_eval) {
  const size_t T1 = (size_t)w.T + 1;
  InstState &s = w.st[b];
  // the mode is snapshotted once: thread 0 rewrites s.mode below, and a warp scheduled late must not see the new value,
  // skip the group barrier and its share of the copies
  ONE_THREAD red[1] = (double)s.mode;
  SYNC();
  if (red[1] != (double)MODE_EVAL) return;
  // add E_{k-1}^T lam_k (base block) to g_k[0:6] and fold it into the dual residual
  const bool has_base = (w.kind != MPC_KIND_CENT);
  if (has_base) {
    PAR_FOR(e, w.T * 6) {
      int k = 1 + e / 6, j = e % 6;
      w.g[(b * T1 + k) * w.nz + j] += w.gE[(b * T1 + k) * 6 + j];
    }
    SYNC();
  }
  ONE_THREAD {
    double cost = 0, pen = 0, prim = 0, dual = 0, inner = 0;
    for (int k = 0; k <= w.T; k++) {
      const double *sc = w.scal + (b * T1 + k) * SC_COUNT;
      cost += sc[SC_COST]; pen += sc[SC_PEN];
      prim = fmax(prim, sc[SC_PRIM]); dual = fmax(dual, sc[SC_DUAL]); inner = fmax(inner, sc[SC_INNER]);
      if (has_base && k >= 1) for (int j = 0; j < 6; j++) dual = fmax(dual, fabs(w.g[(b * T1 + k) * w.nz + j]));
    }
    inner = fmax(inner, dual);
    s.traj_cost = cost; s.merit = cost + pen; s.prim_infeas = prim; s.dual_infeas = dual; s.inner_crit = inner;
    red[0] = 0; // accept multipliers flag
    const SolverConst &c = w.sc;
    if (!isfinite(s.merit)) { s.status = 2; s.mode = MODE_DONE; }
    else if (inner <= s.inner_tol) {
      if (prim <= s.prim_tol) {
        s.prim_tol *= pow(s.mu, c.prim_beta); s.inner_tol *= pow(s.mu, c.dual_beta);
        red[0] = 1;
        if (fmax(prim, dual) <= c.tol) { s.conv = 1; s.status = 0; s.mode = MODE_DONE; }
      } else {
        s.mu = fmax(s.mu * c.mu_update_factor, c.mu_lower_bound);
        s.prim_tol = pow(s.mu, c.prim_alpha); s.inner_tol = pow(s.mu, c.dual_alpha);
      }
      if (s.mode != MODE_DONE) {
        s.inner_tol = fmax(s.inner_tol, 0.01 * c.tol); s.prim_tol = fmax(s.prim_tol, c.tol);
        s.al_iters++;
        if (s.al_iters >= c.max_al_iters) s.mode = MODE_DONE; // else stays MODE_EVAL: re-evaluate with the new estimates
        else next_eval[ATOMIC_INC(&w.counters[2])] = b;
      }
    } else s.mode = MODE_STEP;
  }
  SYNC();
  if (red[0] != 0.0) {
    PAR_FOR(i, (int)(T1 * w.nc)) w.vs_prev[b * T1 * w.nc + i] = w.vs[b * T1 * w.nc + i];
    PAR_FOR(i, (int)(T1 * w.n)) w.lams_prev[b * T1 * w.n + i] = w.lams[b * T1 * w.n + i];
  }
}

// ---- trial point for the current alpha
HD void apply_step(const Ws &w, int b) {
  const InstState &s = w.st[b];
  if (s.mode != MODE_LS) return;
  const size_t T1 = (size_t)w.T + 1;
  const double al = s.alpha;
  if (w.kind == MPC_KIND_CENT) {
    PAR_FOR(i, (int)(T1 * w.nx)) w.txs[b * T1 * w.nx + i] = w.xs[b * T1 * w.nx + i] + al * w.dxs[b * T1 * w.n + i];
  } else {
    PAR_FOR(k, (int)T1) {
      const double *x = w.xs + (b * T1 + k) * w.nx, *d = w.dxs + (b * T1 + k) * w.n;
      double *o = w.txs + (b * T1 + k) * w.nx;
      double xi[6], e[12], R[9], pn[3];
      for (int i = 0; i < 6; i++) xi[i] = al * d[i];
      exp6(xi, e); quat_to_R(x + 3, R); mat3_vec(R, e + 9, pn);
      for (int i = 0; i < 3; i++) o[i] = x[i] + pn[i];
      quat_integrate(x + 3, xi + 3, o + 3);
    }
    PAR_FOR(e, (int)(T1 * (NJ + NV))) {
      int k = e / (NJ + NV), i = e % (NJ + NV);
      w.txs[(b * T1 + k) * w.nx + 7 + i] = w.xs[(b * T1 + k) * w.nx + 7 + i] + al * w.dxs[(b * T1 + k) * w.n + 6 + i];
    }
  }
  PAR_FOR(i, w.T * w.m) w.tus[(size_t)b * w.T * w.m + i] = w.us[(size_t)b * w.T * w.m + i] + al * w.dus[(size_t)b * w.T * w.m + i];
  PAR_FOR(i, (int)(T1 * w.nc)) w.tvs[b * T1 * w.nc + i] = w.vs[b * T1 * w.nc + i] + al * w.dvs[b * T1 * w.nc + i];
  PAR_FOR(i, (int)(T1 * w.n)) w.tlams[b * T1 * w.n + i] = w.lams[b * T1 * w.n + i] + al * w.dlams[b * T1 * w.n + i];
}

// ---- after riccati: start the linesearch
HD void start_linesearch(const Ws &w, int b) {
  ONE_THREAD {
    InstState &s = w.st[b];
    if (s.mode == MODE_STEP) { s.dphi0 = w.dphi[b]; s.alpha = 1.0; s.ls_it = 0; s.a_prev = 0; s.phi_prev = 0; s.mode = MODE_LS; }
  }
}

// ---- after eval<values> at the trial point: Armijo test, next alpha or accept (proxsuite-nlp style backtracking)
HD void decide_ls(const Ws &w, int b, double *red, int32_t *ls_out, int32_t *next_eval) {
  const size_t T1 = (size_t)w.T + 1;
  InstState &s = w.st[b];
  ONE_THREAD red[1] = (double)s.mode; // snapshot (see decide_eval)
  SYNC();
  if (red[1] != (double)MODE_LS) return;
  ONE_THREAD {
    const SolverConst &c = w.sc;
    double cost = 0, pen = 0;
    for (int k = 0; k <= w.T; k++) { const double *sc = w.tscal + (b * T1 + k) * SC_COUNT; cost += sc[SC_COST]; pen += sc[SC_PEN]; }
    const double phi = cost + pen, phi0 = s.merit, dphi0 = s.dphi0, alpha = s.alpha;
    s.ls_evals++;
    bool accept = (phi <= phi0 + c.ls_c1 * alpha * dphi0) || alpha <= c.ls_alpha_min || s.ls_it + 1 >= c.ls_max_steps ||
                  (fabs(dphi0) <= c.ls_dphi_rel * fmax(1.0, fabs(phi0)) && isfinite(phi)); // decrease below merit resolution
    red[0] = accept ? 1.0 : 0.0;
    if (accept) {
      if (!isfinite(phi)) { s.status = 2; s.mode = MODE_DONE; red[0] = 0.0; }
      else {
        s.merit = phi; s.traj_cost = cost;
        if (alpha <= c.ls_alpha_min) {
          if (s.preg >= c.reg_max) { s.status = 3; s.mode = MODE_DONE; }
          else s.preg = fmin(s.preg * c.reg_inc, c.reg_max);
        } else s.preg = fmax(s.preg * c.reg_dec, c.reg_min);
        s.num_iters++;
        if (s.mode != MODE_DONE) s.mode = (s.num_iters < s.max_iters) ? MODE_EVAL : MODE_DONE;
      }
    } else {
      double a_new;
      if (s.ls_it == 0) a_new = -dphi0 * alpha * alpha / (2.0 * (phi - phi0 - dphi0 * alpha));
      else {
        double r1 = phi - phi0 - dphi0 * alpha, r2 = s.phi_prev - phi0 - dphi0 * s.a_prev;
        double den = alpha * alpha * s.a_prev * s.a_prev * (alpha - s.a_prev);
        double a = (s.a_prev * s.a_prev * r1 - alpha * alpha * r2) / den;
        double bq = (-s.a_prev * s.a_prev * s.a_prev * r1 + alpha * alpha * alpha * r2) / den;
        if (fabs(a) < 1e-300) a_new = -dphi0 / (2.0 * bq);
        else { double disc = bq * bq - 3.0 * a * dphi0; a_new = (-bq + sqrt(disc)) / (3.0 * a); }
      }
      if (!(a_new >= c.ls_contr_min * alpha)) a_new = c.ls_contr_min * alpha;
      if (a_new > c.ls_contr_max * alpha) a_new = c.ls_contr_max * alpha;
      s.a_prev = alpha; s.phi_prev = phi;
      s.alpha = fmax(a_new, c.ls_alpha_min);
      s.ls_it++;
    }
    if (s.mode == MODE_LS) { if (ls_out) ls_out[ATOMIC_INC(&w.counters[0])] = b; } // (null: the fused rollout kernel loops by itself)
    else if (s.mode == MODE_EVAL) next_eval[ATOMIC_INC(&w.counters[2])] = b;
  }
  SYNC();
  if (red[0] != 0.0) { // accept: trial -> current
    PAR_FOR(i, (int)(T1 * w.nx)) w.xs[b * T1 * w.nx + i] = w.txs[b * T1 * w.nx + i];
    PAR_FOR(i, w.T * w.m) w.us[(size_t)b * w.T * w.m + i] = w.tus[(size_t)b * w.T * w.m + i];
    PAR_FOR(i, (int)(T1 * w.nc)) w.vs[b * T1 * w.nc + i] = w.tvs[b * T1 * w.nc + i];
    PAR_FOR(i, (int)(T1 * w.n)) w.lams[b * T1 * w.n + i] = w.tlams[b * T1 * w.n + i];
  }
}

// ---- what differs between the model kinds: dimensions, the evaluation workspace and stage functions, the Riccati solver and
// its launch shape.  KIND is a compile-time parameter so every model gets its own kernels (registers, shared memory and spills
// of one stage type do not tax the others); the host turns the runtime kind into KIND with dispatch_kind (driver.hpp).
template <int KIND> struct KindTraits;
template <> struct KindTraits<MPC_KIND_FULL> {
  static constexpr int nx = 57, n = 56, m = 22, nc = 78;
  static constexpr int ncap = 23; // active rows of the Riccati's shared-memory carving: what fits over the dead P | G buffers (two instances per SM)
  template <bool D> using EvalWs = FullWsT<D>;
  template <bool D, bool ROLL = false> static HD void knot(const DevModel &md, const KnotIO &io, EvalWs<D> &f) { eval_full_knot<D, ROLL>(md, io, f); }
  template <bool D> static HD void term(const DevModel &md, const KnotIO &io, EvalWs<D> &f) { eval_mb_term<D, true, FNZ, FNC>(md, io, f); }
  static HD void riccati(const RiccatiIO &r, double *smem) { riccati_instance_fast<n, m, nc, ncap>(r, smem); }
  static HD void riccati_seeded(const RiccatiIO &r, double *smem) { riccati_instance_fast<n, m, nc, ncap, true>(r, smem); }
  static constexpr bool lie6 = true;
  static constexpr int ric_smem = RicFastLayout<n, m, nc, ncap>::total * 8, ric_scratch = RicFastLayout<n, m, nc, ncap>::scratch;
  // two 128-thread instances per SM when the launch fills the GPU; 256 threads per instance when SMs would idle (latency)
  static constexpr int ric_threads(int count, int num_sms) { return count <= num_sms ? 256 : 128; }
};
template <> struct KindTraits<MPC_KIND_KINO> {
  static constexpr int nx = 57, n = 56, m = 34, nc = 68;
  static constexpr int ncap = 54; // knots with more active rows (up to all 68) solve their KKT out of global scratch
  template <bool D> using EvalWs = KinoWsT<D>;
  template <bool D, bool ROLL = false> static HD void knot(const DevModel &md, const KnotIO &io, EvalWs<D> &f) { eval_kino_knot<D, ROLL>(md, io, f); }
  template <bool D> static HD void term(const DevModel &md, const KnotIO &io, EvalWs<D> &f) { eval_mb_term<D, false, KNZ, KNC>(md, io, f); }
  static HD void riccati(const RiccatiIO &r, double *smem) { riccati_instance_fast<n, m, nc, ncap>(r, smem); }
  static HD void riccati_seeded(const RiccatiIO &r, double *smem) { riccati_instance_fast<n, m, nc, ncap, true>(r, smem); }
  static constexpr bool lie6 = true;
  static constexpr int ric_smem = RicFastLayout<n, m, nc, ncap>::total * 8, ric_scratch = RicFastLayout<n, m, nc, ncap>::scratch;
  static constexpr int ric_threads(int, int) { return 256; }
};
template <> struct KindTraits<MPC_KIND_CENT> {
  static constexpr int nx = 9, n = 9, m = 12, nc = 34;
  static constexpr int ncap = nc; // the generic Riccati kernel holds every row in shared memory
  template <bool D> using EvalWs = CentWs;
  template <bool D, bool ROLL = false> static HD void knot(const DevModel &md, const KnotIO &io, CentWs &f) { eval_cent_knot<D, ROLL>(md, io, f); }
  template <bool D> static HD void term(const DevModel &md, const KnotIO &io, CentWs &f) { eval_cent_term<D>(md, io, f); }
  static HD void riccati(const RiccatiIO &r, double *smem) { riccati_instance<n, m, nc>(r, smem); }
  static HD void riccati_seeded(const RiccatiIO &r, double *smem) { riccati_instance<n, m, nc, true>(r, smem); }
  static constexpr bool lie6 = false;
  static constexpr int ric_smem = riccati_smem_doubles<n, m, nc>() * 8, ric_scratch = 2; // no global scratch: a token block
  static constexpr int ric_threads(int, int) { return 128; }
};
static_assert(KindTraits<MPC_KIND_FULL>::ric_smem <= 232448 && KindTraits<MPC_KIND_KINO>::ric_smem <= 232448 && KindTraits<MPC_KIND_CENT>::ric_smem <= 232448,
              "Riccati shared memory exceeds the 227 KB opt-in limit");

// ---- one (instance, knot) evaluation.  smem: KindTraits<KIND>::EvalWs<DERIV> storage.
template <int KIND, bool DERIV> HD void eval_dispatch(const Ws &w, int b, int k, void *smem) {
  using K = KindTraits<KIND>;
  const int mode = w.st[b].mode;
  if (mode != (DERIV ? MODE_EVAL : MODE_LS)) return;
  KnotIO io = make_io(w, b, k, !DERIV);
  auto &f = *reinterpret_cast<typename K::template EvalWs<DERIV> *>(smem);
  const DevModel &md = model_of(w, b);
  if (k < w.T) K::template knot<DERIV>(md, io, f); else K::template term<DERIV>(md, io, f);
}

// ---- ROLLOUT_NONLINEAR: one trial point of the fused rollout + linesearch kernel (one CTA = one evaluation group per instance).
// The affine policy of the LQ solve is rolled out through the NONLINEAR dynamics, knot after knot (oracle: Solver::try_step_nonlinear):
//   dx_k = x+_k (-) x_k,  du = alpha ku + Ku dx_k,  dv = alpha kv + Kv dx_k (active rows; alpha dbar/mu otherwise),
//   dlam' = alpha pt + W [dx_k; du],  x+_{k+1} = f(x+_k, u+_k) (+) mu_d (lam_e - lam'+)   (set inside the knot evaluation),
// and every knot's merit terms land in tscal exactly as in a linear-rollout trial, so decide_ls applies unchanged.
// xv: >= 64 + 96 + 64 doubles of shared memory next to the evaluation workspace.
template <int KIND> HD void rollout_trial(const Ws &w, int b, double alpha, void *smem, double *xv) {
  using K = KindTraits<KIND>;
  auto &f = *reinterpret_cast<typename K::template EvalWs<false> *>(smem);
  const size_t T1 = (size_t)w.T + 1;
  const int n = w.n, m = w.m, nc = w.nc, nz = w.nz, nx = w.nx, NRk = 1 + n, S = m + nc, T = w.T;
  const int ldw = (KIND == MPC_KIND_CENT) ? nz : ((nz + 7) & ~7);
  double *dx = xv, *z = xv + 64, *slack = xv + 160;
  const double mu = w.st[b].mu, mu_d = mu;
  const DevModel &md = model_of(w, b);
  const double *xs = w.xs + b * T1 * nx, *us = w.us + (size_t)b * T * m, *vs = w.vs + b * T1 * nc, *lams = w.lams + b * T1 * n;
  double *txs = w.txs + b * T1 * nx, *tus = w.tus + (size_t)b * T * m, *tvs = w.tvs + b * T1 * nc, *tlams = w.tlams + b * T1 * n;
  const double *lams_prev = w.lams_prev + b * T1 * n, *dbar = w.dbar + b * T1 * nc;
  auto state_diff = [&](const double *x0, const double *x1) { // dx = x1 (-) x0
    if (KIND == MPC_KIND_CENT) { PAR_FOR(i, n) dx[i] = x1[i] - x0[i]; }
    else {
      ONE_THREAD {
        double M0[12], M1[12], D[12];
        quat_to_R(x0 + 3, M0); M0[9] = x0[0]; M0[10] = x0[1]; M0[11] = x0[2];
        quat_to_R(x1 + 3, M1); M1[9] = x1[0]; M1[10] = x1[1]; M1[11] = x1[2];
        se3_inv_mul(M0, M1, D);
        log6(D, dx);
      }
      PAR_FOR(i, NJ + NV) dx[6 + i] = x1[7 + i] - x0[7 + i];
    }
  };
  PAR_FOR(i, nx) txs[i] = xs[i];
  PAR_FOR(i, n) tlams[i] = lams[i] + alpha * w.dlams[b * T1 * n + i];
  SYNC();
  for (int k = 0; k <= T; k++) {
    const size_t kb = b * T1 + k;
    const int nca = w.nca[kb];
    const int32_t *ai = w.act_idx + kb * nc;
    state_diff(xs + (size_t)k * nx, txs + (size_t)k * nx);
    PAR_FOR(r, nc) tvs[(size_t)k * nc + r] = vs[(size_t)k * nc + r] + alpha * dbar[(size_t)k * nc + r] / mu; // rows outside the active set
    SYNC();
    if (k == T) { // terminal rows: dv = (alpha dbar + C dx) / mu
      const double *CT = w.CDact + kb * nc * nz;
      PAR_FOR(a, nca) {
        const int row = ai[a];
        double t = alpha * dbar[(size_t)k * nc + row];
        for (int j = 0; j < n; j++) t += CT[a * nz + j] * dx[j];
        tvs[(size_t)k * nc + row] = vs[(size_t)k * nc + row] + t / mu;
      }
      SYNC();
      KnotIO io = make_io(w, b, k, true);
      K::template term<false>(md, io, f);
      SYNC();
      break;
    }
    const double *Kk = w.K + ((size_t)b * T + k) * S * NRk;
    PAR_FOR(i, m + nca) {
      double t = alpha * Kk[i * NRk];
      for (int j = 0; j < n; j++) t += Kk[i * NRk + 1 + j] * dx[j];
      if (i < m) { z[n + i] = t; tus[(size_t)k * m + i] = us[(size_t)k * m + i] + t; }
      else { const int row = ai[i - m]; tvs[(size_t)k * nc + row] = vs[(size_t)k * nc + row] + t; }
    }
    PAR_FOR(j, n) z[j] = dx[j];
    SYNC();
    const double *Wk = w.W + (size_t)b * T * n * ((nz + 7) & ~7) + (size_t)k * n * ldw, // (instance stride as in make_riccati_io)
                  *ptk = w.pt + ((size_t)b * T + k) * n;
    PAR_FOR(i, n) {
      double t = alpha * ptk[i];
      for (int j = 0; j < nz; j++) t += Wk[i * ldw + j] * z[j];
      const size_t id = (size_t)(k + 1) * n + i;
      const double tl = lams[id] + t;
      tlams[id] = tl;
      slack[i] = mu_d * (lams_prev[id] - tl);
    }
    SYNC();
    KnotIO io = make_io(w, b, k, true);
    io.xn = io.x; io.slack = slack; io.xn_out = txs + (size_t)(k + 1) * nx;
    K::template knot<false, true>(md, io, f);
    SYNC();
  }
}
// the whole linesearch of one instance: trial rollouts until decide_ls accepts (or gives up)
template <int KIND> HD void rollout_linesearch(const Ws &w, int b, void *smem, double *xv, double *red /* shared, >= 8 */, int32_t *next_eval) {
  for (int it = 0; it <= w.sc.ls_max_steps; it++) {
    ONE_THREAD { red[2] = (double)w.st[b].mode; red[3] = w.st[b].alpha; }
    SYNC();
    const double mode = red[2], alpha = red[3];
    SYNC();
    if (mode != (double)MODE_LS) break;
    rollout_trial<KIND>(w, b, alpha, smem, xv);
    decide_ls(w, b, red, nullptr, next_eval);
    SYNC();
  }
}

HD RiccatiIO make_riccati_io(const Ws &w, int b) {
  const size_t T1 = (size_t)w.T + 1, T = w.T;
  RiccatiIO r;
  r.T = w.T; r.mu = w.st[b].mu; r.mu_d = w.st[b].mu;
  r.AB = w.AB + b * T * w.n * w.nz; r.H = w.H + b * T1 * w.nz * w.nz; r.g = w.g + b * T1 * w.nz; r.fbar = w.fbar + b * T * w.n;
  r.T6 = w.T6 + b * T * 36; r.CDact = w.CDact + b * T1 * w.nc * w.nz; r.dbar = w.dbar + b * T1 * w.nc; r.nca = w.nca + b * T1;
  r.act_idx = w.act_idx + b * T1 * w.nc; r.lxu = w.lxu + b * T1 * w.nz; r.vplus = w.vplus + b * T1 * w.nc; r.v = w.vs + b * T1 * w.nc;
  r.lplus = w.lplus + b * T1 * w.n; r.lam = w.lams + b * T1 * w.n;
  r.W = w.W + b * T * w.n * ((w.nz + 7) & ~7); r.scratch = w.ric_scratch + b * w.ric_scratch_stride; r.pt = w.pt + b * T * w.n; r.K = w.K + b * T * (w.m + w.nc) * (1 + w.n); r.Kfb = w.Kfb + b * T * w.m * w.n;
  r.dxs = w.dxs + b * T1 * w.n; r.dus = w.dus + b * T * w.m; r.dvs = w.dvs + b * T1 * w.nc; r.dlams = w.dlams + b * T1 * w.n;
  r.dphi = w.dphi + b;
  r.phase_out = (b == 0) ? w.phase : nullptr;
  return r;
}

template <int KIND> HD void riccati_dispatch(const Ws &w, int b, double *smem) {
  if (w.st[b].mode != MODE_STEP) return;
  KindTraits<KIND>::riccati(make_riccati_io(w, b), smem);
  start_linesearch(w, b);
}

// ---- time-parallel LQ solve (riccati_par.cuh), lq_legs = L >= 2: per-(instance, leg) blocks, indexed b * L + j
struct LegWs {
  int L;
  double *sum, *ws, *buf, *scratch; // LegLayout::sum / ::ws / ::buf and KindTraits::ric_scratch doubles per (instance, leg)
};
template <int KIND> struct LegDims {
  using K = KindTraits<KIND>;
  using Lay = LegLayout<K::n, K::m, K::nc>;
};
// phase A: leg j of instance b
template <int KIND> HD void ric_par_legs(const Ws &w, const LegWs &lw, int b, int j) {
  using K = KindTraits<KIND>;
  using Lay = typename LegDims<KIND>::Lay;
  if (w.st[b].mode != MODE_STEP) return;
  const size_t i = (size_t)b * lw.L + j;
  ric_leg_param<K::n, K::m, K::nc, K::lie6>(make_riccati_io(w, b), leg_start(w.T, lw.L, j), leg_start(w.T, lw.L, j + 1), j + 1 == lw.L, lw.ws + i * Lay::ws,
                                             lw.sum + i * Lay::sum);
}
// phase B: the boundaries of instance b.  sh: >= n doubles of shared memory
template <int KIND> HD void ric_par_consensus(const Ws &w, const LegWs &lw, int b, double *sh) {
  using K = KindTraits<KIND>;
  using Lay = typename LegDims<KIND>::Lay;
  if (w.st[b].mode != MODE_STEP) return;
  const size_t i = (size_t)b * lw.L;
  ric_consensus<K::n, K::m, K::nc>(lw.L, lw.sum + i * Lay::sum, Lay::sum, lw.buf + i * Lay::buf, Lay::buf, sh);
}
// phase C: exact re-solve of leg j of instance b with the model's Riccati kernel.  smem: KindTraits::ric_smem bytes
template <int KIND> HD void ric_par_resolve(const Ws &w, const LegWs &lw, int b, int j, double *smem) {
  using K = KindTraits<KIND>;
  using Lay = typename LegDims<KIND>::Lay;
  if (w.st[b].mode != MODE_STEP) return;
  const size_t i = (size_t)b * lw.L + j;
  double *bf = lw.buf + i * Lay::buf;
  RiccatiIO r = make_riccati_io(w, b);
  r.k0 = leg_start(w.T, lw.L, j); r.k1 = leg_start(w.T, lw.L, j + 1);
  r.seedP = (j + 1 < lw.L) ? bf : nullptr; r.seedp = bf + Lay::off_seedp; r.dx0 = bf + Lay::off_x;
  r.dphi = bf + Lay::off_dphi;
  r.scratch = lw.scratch + i * K::ric_scratch;
  r.phase_out = (b == 0 && j == 0) ? w.phase : nullptr;
  K::riccati_seeded(r, smem);
}
// phase D: the legs' merit derivative partials in leg order, then what riccati_dispatch does after the serial kernel
template <int KIND> HD void ric_par_finish(const Ws &w, const LegWs &lw, int b) {
  using Lay = typename LegDims<KIND>::Lay;
  if (w.st[b].mode != MODE_STEP) return;
  ONE_THREAD {
    double s = 0;
    for (int j = 0; j < lw.L; j++) s += lw.buf[((size_t)b * lw.L + j) * Lay::buf + Lay::off_dphi];
    w.dphi[b] = s;
  }
  SYNC();
  start_linesearch(w, b);
}

} // namespace mpcdev
