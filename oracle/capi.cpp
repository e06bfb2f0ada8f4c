// ORACLE (test infrastructure, not product code) — C entry points used by tests/, smoke() and
// bench.py's cpu_baseline leg ONLY.  The product path (mpc_benchmark_b200 + libmpcb200.so) never loads this.
// PARITY UNPINNED against upstream Aligator/Pinocchio (absent from /root/reference, README.md:10-18).
#include "proxddp.hpp"
#include "qp.hpp"
#include "riccati_par.hpp"
#include <cstdio>
#include <omp.h>

using namespace orc;

extern "C" {

int orc_sizeof(int which) {
  switch (which) {
  case 0: return sizeof(mpc_robot_t);
  case 1: return sizeof(mpc_config_t);
  case 2: return sizeof(mpc_knot_t);
  case 3: return sizeof(mpc_term_t);
  case 4: return sizeof(mpc_info_t);
  case 5: return sizeof(mpc_qp_settings_t);
  case 6: return sizeof(mpc_qp_info_t);
  }
  return -1;
}

// ---- Lie group checks: max |analytic - AD| of Jlog6 at M and Jexp6 at xi
double orc_check_jlog6(const double *M12) {
  SE3<double> M = se3_from12<double>(M12);
  M6<double> J = Jlog6(M);
  double err = 0;
  for (int k = 0; k < 6; k++) {
    V6<Dual> d = zero6<Dual>(); d[k] = Dual(0, 1);
    SE3<Dual> Md = se3_cast<Dual>(M12);
    V6<Dual> l = log6(mul(Md, exp6(d)));
    for (int i = 0; i < 6; i++) err = std::max(err, std::fabs(l[i].d - J[6 * i + k]));
  }
  return err;
}
double orc_check_jexp6(const double *xi6) {
  V6<double> xi; for (int i = 0; i < 6; i++) xi[i] = xi6[i];
  M6<double> J = Jexp6(xi);
  SE3<double> M0 = exp6(xi);
  double err = 0;
  for (int k = 0; k < 6; k++) {
    // exp6(xi + e d) = exp6(xi) exp6(J e d)  =>  d/de log6(exp6(xi)^-1 exp6(xi + e d)) = J[:,k]
    V6<Dual> x; for (int i = 0; i < 6; i++) x[i] = Dual(xi[i], i == k ? 1.0 : 0.0);
    SE3<Dual> Mi; for (int i = 0; i < 9; i++) Mi.R[i] = M0.R[i]; for (int i = 0; i < 3; i++) Mi.p[i] = M0.p[i];
    SE3<Dual> D = mul(inverse(Mi), exp6(x));
    // log6 derivative at identity is the tangent itself
    V6<Dual> l = log6(D);
    for (int i = 0; i < 6; i++) err = std::max(err, std::fabs(l[i].d - J[6 * i + k]));
  }
  return err;
}
void orc_exp6(const double *xi, double *M12) {
  V6<double> x; for (int i = 0; i < 6; i++) x[i] = xi[i];
  SE3<double> M = exp6(x);
  for (int i = 0; i < 9; i++) M12[i] = M.R[i];
  for (int i = 0; i < 3; i++) M12[9 + i] = M.p[i];
}
void orc_log6(const double *M12, double *xi) { V6<double> l = log6(se3_from12<double>(M12)); for (int i = 0; i < 6; i++) xi[i] = l[i]; }
void orc_integrate(const double *x, const double *dx, double *out) { mb_integrate<double>(x, dx, out); }
void orc_difference(const double *x0, const double *x1, double *out) { mb_difference<double>(x0, x1, out); }
void orc_cone_matrix(double mu, double L, double W, double *A) { cone_matrix(mu, L, W, A); }

// ---- kinematics outputs for KATs
void orc_kinematics(const mpc_robot_t *rb, const double *x, double *com, double *mass, double *hg, double *lf12, double *rf12, double *M, double *b) {
  Tree tr(rb);
  static Kin<double> k;
  forward_kin<double>(tr, x, x + NQ, k);
  for (int i = 0; i < 3; i++) com[i] = k.com[i];
  *mass = k.mass;
  V6<double> h = centroidal_momentum(k);
  for (int i = 0; i < 6; i++) hg[i] = h[i];
  for (int f = 0; f < 2; f++) {
    SE3<double> Mf = mul(k.oM[rb->foot_body[f]], se3_cast<double>(rb->foot_place[f]));
    double *o = f == 0 ? lf12 : rf12;
    for (int i = 0; i < 9; i++) o[i] = Mf.R[i];
    for (int i = 0; i < 3; i++) o[9 + i] = Mf.p[i];
  }
  if (M) crba(tr, k, M);
  if (b) rnea<double>(tr, k, x + NQ, nullptr, nullptr, b);
}
// tau = RNEA(q,v,a)
void orc_rnea(const mpc_robot_t *rb, const double *x, const double *a, double *tau) {
  Tree tr(rb);
  static Kin<double> k;
  forward_kin<double>(tr, x, x + NQ, k);
  rnea<double>(tr, k, x + NQ, a, nullptr, tau);
}

// constrained dynamics values + analytic derivatives + AD check (errs[6]: da_dq, da_dv, da_dtau, dl_dq, dl_dv, dl_dtau)
void orc_cdyn(const mpc_robot_t *rb, const mpc_config_t *cfg, const double *x, const double *tau, const int *active_, double *a, double *lam,
              double *da_dq, double *da_dv, double *da_dtau, double *dl_dq, double *dl_dv, double *dl_dtau, double *errs) {
  Tree tr(rb);
  bool active[2] = {active_[0] != 0, active_[1] != 0};
  static CDyn<double> d;
  constrained_dynamics<double>(tr, *cfg, x, x + NQ, tau, active, d);
  for (int i = 0; i < NV; i++) a[i] = d.a[i];
  for (int i = 0; i < 12; i++) lam[i] = d.lam[i];
  static CDynDerivs dd;
  constrained_dynamics_derivatives(tr, *cfg, x + NQ, d, dd);
  auto cp = [](double *dst, const double *src, int n) { if (dst) for (int i = 0; i < n; i++) dst[i] = src[i]; };
  cp(da_dq, dd.da_dq, NV * NV); cp(da_dv, dd.da_dv, NV * NV); cp(da_dtau, dd.da_dtau, NV * NV);
  cp(dl_dq, dd.dl_dq, 12 * NV); cp(dl_dv, dd.dl_dv, 12 * NV); cp(dl_dtau, dd.dl_dtau, 12 * NV);
  if (!errs) return;
  for (int i = 0; i < 6; i++) errs[i] = 0;
  static CDyn<Dual> dz;
  for (int which = 0; which < 3; which++)
    for (int j = 0; j < NV; j++) {
      Dual xd[NQ + NV], taud[NV];
      for (int i = 0; i < NV; i++) taud[i] = Dual(tau[i], (which == 2 && i == j) ? 1.0 : 0.0);
      if (which == 0) {
        Dual x0[NQ + NV], dx[2 * NV];
        for (int i = 0; i < NQ + NV; i++) x0[i] = Dual(x[i]);
        for (int i = 0; i < 2 * NV; i++) dx[i] = Dual(0, i == j ? 1.0 : 0.0);
        mb_integrate<Dual>(x0, dx, xd);
      } else {
        for (int i = 0; i < NQ + NV; i++) xd[i] = Dual(x[i], (which == 1 && i == NQ + j) ? 1.0 : 0.0);
      }
      constrained_dynamics<Dual>(tr, *cfg, xd, xd + NQ, taud, active, dz);
      const double *A = which == 0 ? dd.da_dq : which == 1 ? dd.da_dv : dd.da_dtau;
      const double *Lm = which == 0 ? dd.dl_dq : which == 1 ? dd.dl_dv : dd.dl_dtau;
      for (int i = 0; i < NV; i++) errs[which] = std::max(errs[which], std::fabs(dz.a[i].d - A[i * NV + j]));
      for (int i = 0; i < 12; i++) errs[3 + which] = std::max(errs[3 + which], std::fabs(dz.lam[i].d - Lm[i * NV + j]));
    }
}

// centroidal momentum derivative check: returns max |analytic - AD| over dh/dq, dh/dv and Jcom
double orc_check_centroidal(const mpc_robot_t *rb, const double *x) {
  Tree tr(rb);
  static Kin<double> k;
  forward_kin<double>(tr, x, x + NQ, k);
  double dhq[6 * NV], Ag[6 * NV], Jc[3 * NV];
  centroidal_derivatives(tr, k, dhq, Ag);
  com_jacobian(k, Jc);
  double err = 0;
  static Kin<Dual> kd;
  for (int which = 0; which < 2; which++)
    for (int j = 0; j < NV; j++) {
      Dual xd[NQ + NV];
      if (which == 0) {
        Dual x0[NQ + NV], dx[2 * NV];
        for (int i = 0; i < NQ + NV; i++) x0[i] = Dual(x[i]);
        for (int i = 0; i < 2 * NV; i++) dx[i] = Dual(0, i == j ? 1.0 : 0.0);
        mb_integrate<Dual>(x0, dx, xd);
      } else for (int i = 0; i < NQ + NV; i++) xd[i] = Dual(x[i], i == NQ + j ? 1.0 : 0.0);
      forward_kin<Dual>(tr, xd, xd + NQ, kd);
      V6<Dual> h = centroidal_momentum(kd);
      for (int i = 0; i < 6; i++) err = std::max(err, std::fabs(h[i].d - (which == 0 ? dhq : Ag)[i * NV + j]));
      if (which == 0) for (int i = 0; i < 3; i++) err = std::max(err, std::fabs(kd.com[i].d - Jc[i * NV + j]));
    }
  return err;
}

// ---- knot evaluation (dense). Any output may be NULL. k == -1 evaluates the terminal knot.
void orc_eval_knot(const mpc_robot_t *rb, const mpc_config_t *cfg, const mpc_knot_t *kn, const mpc_term_t *tm, const double *x, const double *u,
                   const double *xn, int derivs, double *xnext, double *gap, double *A, double *B, double *E6, double *cost, double *lx,
                   double *lu, double *H, double *h, double *Cx, double *Cu, int *ctype, double *lo, double *hi, double *xdot, double *lam) {
  Problem P(rb, *cfg);
  KnotEval e; e.resize(P.d);
  if (kn) eval_knot(P, *kn, x, u, xn, derivs != 0, e); else eval_term(P, *tm, x, e);
  auto cp = [](double *dst, const std::vector<double> &src) { if (dst) std::copy(src.begin(), src.end(), dst); };
  cp(xnext, e.xnext); cp(gap, e.gap); cp(A, e.A); cp(B, e.B); cp(E6, e.E6); cp(lx, e.lx); cp(lu, e.lu); cp(H, e.H);
  cp(h, e.h); cp(Cx, e.Cx); cp(Cu, e.Cu); cp(lo, e.lo); cp(hi, e.hi);
  if (cost) *cost = e.cost;
  if (ctype) std::copy(e.ctype.begin(), e.ctype.end(), ctype);
  if (xdot) std::copy(e.xdot, e.xdot + 56, xdot);
  if (lam) std::copy(e.lam, e.lam + 12, lam);
}

// ---- proximal Riccati on dense caller data (all knots share sizes). Layouts as mpc_riccati_dense (mpcb200.h).
// H [T][nz][nz], g [T][nz], AB [T][n][nz], f [T][n], CD [T][nc][nz], d [T][nc], HT [n][n], gT [n]
// E6 [T][36] or NULL; CT [nct][n], dT [nct] or NULL.  legs >= 2: the leg-parallel solve (riccati_par.hpp), else the serial one
static void riccati_dense(int n, int m, int nc, int T, double mu_d, double mu, const double *H, const double *g, const double *AB, const double *f,
                          const double *CD, const double *dd, const double *E6, const double *HT, const double *gT, const double *CT, const double *dT,
                          int nct, int legs, double *dxs, double *dus, double *dvs, double *dlams, double *K) {
  int nz = n + m;
  std::vector<std::vector<double>> A(T), B(T), C(T), D(T);
  std::vector<LQKnot> kn(T);
  for (int k = 0; k < T; k++) {
    A[k].resize(n * n); B[k].resize(n * m); C[k].resize(nc * n); D[k].resize(nc * m);
    for (int i = 0; i < n; i++) { for (int j = 0; j < n; j++) A[k][i * n + j] = AB[((size_t)k * n + i) * nz + j]; for (int j = 0; j < m; j++) B[k][i * m + j] = AB[((size_t)k * n + i) * nz + n + j]; }
    for (int i = 0; i < nc; i++) { for (int j = 0; j < n; j++) C[k][i * n + j] = CD[((size_t)k * nc + i) * nz + j]; for (int j = 0; j < m; j++) D[k][i * m + j] = CD[((size_t)k * nc + i) * nz + n + j]; }
    kn[k] = {H + (size_t)k * nz * nz, g + (size_t)k * nz, A[k].data(), B[k].data(), E6 ? E6 + (size_t)k * 36 : nullptr, f + (size_t)k * n,
             C[k].data(), D[k].data(), dd + (size_t)k * nc};
  }
  LQSolution sol;
  if (legs >= 2) riccati_solve_par(n, m, nc, T, kn.data(), HT, n, gT, CT, dT, nct, mu_d, mu, legs, sol);
  else riccati_solve(n, m, nc, T, kn.data(), HT, n, gT, CT, dT, nct, mu_d, mu, sol);
  std::copy(sol.dxs.begin(), sol.dxs.end(), dxs); std::copy(sol.dus.begin(), sol.dus.end(), dus);
  if (dvs) std::copy(sol.dvs.begin(), sol.dvs.end(), dvs);
  if (dlams) std::copy(sol.dlams.begin(), sol.dlams.end(), dlams);
  if (K) std::copy(sol.K.begin(), sol.K.end(), K);
}
void orc_riccati(int n, int m, int nc, int T, double mu_d, double mu, const double *H, const double *g, const double *AB, const double *f,
                 const double *CD, const double *dd, const double *E6, const double *HT, const double *gT, const double *CT, const double *dT,
                 int nct, double *dxs, double *dus, double *dvs, double *dlams, double *K) {
  riccati_dense(n, m, nc, T, mu_d, mu, H, g, AB, f, CD, dd, E6, HT, gT, CT, dT, nct, 0, dxs, dus, dvs, dlams, K);
}
void orc_riccati_par(int n, int m, int nc, int T, double mu_d, double mu, const double *H, const double *g, const double *AB, const double *f,
                     const double *CD, const double *dd, const double *E6, const double *HT, const double *gT, const double *CT, const double *dT,
                     int nct, int legs, double *dxs, double *dus, double *dvs, double *dlams, double *K) {
  riccati_dense(n, m, nc, T, mu_d, mu, H, g, AB, f, CD, dd, E6, HT, gT, CT, dT, nct, legs, dxs, dus, dvs, dlams, K);
}

// ---- ProxDDP: batch of instances, OpenMP over instances (knot_threads > 1: over knots, batch serial)
// knots [batch][T], terms [batch], x0 [batch][nx], xs [batch][T+1][nx] in/out, us [batch][T][nu] in/out,
// K [batch][T][nu][ndx], vs [batch][T+1][nc] in/out, lams [batch][T+1][ndx] in/out (multipliers warm start; zero after setup)
// stage0 [batch][56+12]: xdot and contact forces of knot 0 at the last evaluated iterate (NULL = skip)
int orc_solve(const mpc_robot_t *rb, const mpc_config_t *cfg, int batch, const mpc_knot_t *knots, const mpc_term_t *terms, const double *x0,
              double *xs, double *us, double *K, double *vs, double *lams, mpc_info_t *info, double *stage0, int max_iters, int inst_threads,
              int knot_threads) {
  Problem P(rb, *cfg);
  Dims d = P.d;
  int T = cfg->T;
  SolverParams prm;
  prm.tol = cfg->tol; prm.mu_init = cfg->mu_init; prm.max_iters = max_iters;
  prm.par_knots = knot_threads > 1;
  prm.rollout = cfg->rollout;
  // ablation switches (see SolverParams); unset = the normative algorithm
  if (const char *e = getenv("ORC_MU_DYN_SCALE")) prm.mu_dyn_scale = atof(e);
  if (const char *e = getenv("ORC_LS_MODE")) prm.ls_mode = atoi(e);
  if (const char *e = getenv("ORC_LS_WINDOW")) prm.ls_window = atoi(e);
  if (const char *e = getenv("ORC_LS_ALPHA_MIN")) prm.ls_alpha_min = atof(e);
  if (const char *e = getenv("ORC_DUAL_WEIGHT")) prm.dual_weight = atof(e);
  if (const char *e = getenv("ORC_REG_INIT")) prm.reg_init = atof(e);
  if (knot_threads > 1) omp_set_num_threads(knot_threads);
  else omp_set_num_threads(inst_threads > 0 ? inst_threads : 1);
#pragma omp parallel if (knot_threads <= 1 && inst_threads > 1)
  {
    Solver S(P, prm);
    S.setup(T);
#pragma omp for schedule(dynamic)
    for (int b = 0; b < batch; b++) {
      Instance in;
      in.T = T; in.knots = knots + (size_t)b * T; in.term = terms[b];
      in.x0.assign(x0 + (size_t)b * d.nx, x0 + (size_t)(b + 1) * d.nx);
      size_t nxs = (size_t)(T + 1) * d.nx, nus = (size_t)T * d.m, nvs = (size_t)(T + 1) * d.nc, nls = (size_t)(T + 1) * d.n;
      if (vs) std::copy(vs + b * nvs, vs + (b + 1) * nvs, S.vs.begin()); else std::fill(S.vs.begin(), S.vs.end(), 0.0);
      if (lams) std::copy(lams + b * nls, lams + (b + 1) * nls, S.lams.begin()); else std::fill(S.lams.begin(), S.lams.end(), 0.0);
      S.run(in, xs + b * nxs, us + b * nus, max_iters);
      std::copy(S.xs.begin(), S.xs.end(), xs + b * nxs);
      std::copy(S.us.begin(), S.us.end(), us + b * nus);
      if (K) std::copy(S.Kfb.begin(), S.Kfb.end(), K + (size_t)b * T * d.m * d.n);
      if (vs) std::copy(S.vs.begin(), S.vs.end(), vs + b * nvs);
      if (lams) std::copy(S.lams.begin(), S.lams.end(), lams + b * nls);
      if (info) {
        mpc_info_t &o = info[b];
        o.prim_infeas = S.prim_infeas; o.dual_infeas = S.dual_infeas; o.traj_cost = S.traj_cost; o.merit = S.merit; o.mu = S.mu;
        o.num_iters = S.num_iters; o.al_iters = S.al_iters; o.conv = S.conv; o.status = S.status; o.alpha = S.alpha_last; o.ls_evals = S.ls_evals; o.pad_ = 0;
      }
      if (stage0) { std::copy(S.ev[0].xdot, S.ev[0].xdot + 56, stage0 + (size_t)b * 68); std::copy(S.ev[0].lam, S.ev[0].lam + 12, stage0 + (size_t)b * 68 + 56); }
    }
  }
  return 0;
}

// kinodynamic base acceleration: analytic Jacobians (from eval_knot_kino's xdot rows) vs forward-mode AD; returns max abs error
double orc_check_kino(const mpc_robot_t *rb, const mpc_config_t *cfg, const mpc_knot_t *kn, const double *x, const double *u) {
  Problem P(rb, *cfg);
  KnotEval e; e.resize(P.d);
  eval_knot(P, *kn, x, u, x, true, e);
  // A = d gap/dx includes the integrator; compare instead the acceleration map through AD of kino_dynamics + the integrator chain
  // by finite AD on xnext: d xnext / d(x,u) via Dual on (integrate(x, dx(x,u)))
  bool active[2] = {kn->cs[0] != 0.0, kn->cs[1] != 0.0};
  double err = 0;
  static Kin<Dual> kd;
  for (int j = 0; j < 56 + 34; j++) {
    Dual xd[NQ + NV], ud[34];
    for (int i = 0; i < 34; i++) ud[i] = Dual(u[i], (j >= 56 && j - 56 == i) ? 1.0 : 0.0);
    if (j < 56) {
      Dual x0[NQ + NV], dx[2 * NV];
      for (int i = 0; i < NQ + NV; i++) x0[i] = Dual(x[i]);
      for (int i = 0; i < 2 * NV; i++) dx[i] = Dual(0, i == j ? 1.0 : 0.0);
      mb_integrate<Dual>(x0, dx, xd);
    } else for (int i = 0; i < NQ + NV; i++) xd[i] = Dual(x[i]);
    forward_kin<Dual>(P.tree, xd, xd + NQ, kd);
    KinoVals<Dual> kv;
    kino_dynamics<Dual>(P.tree, *rb, active, kd, xd + NQ, ud, kv);
    // step and gap against xn = x (value point): gap = difference(x, integrate(xd, dxs))
    Dual dxs[2 * NV], xn2[NQ + NV], xref[NQ + NV], gap[2 * NV];
    for (int i = 0; i < NV; i++) { dxs[NV + i] = Dual(cfg->dt) * kv.a[i]; dxs[i] = Dual(cfg->dt) * (xd[NQ + i] + dxs[NV + i]); }
    mb_integrate<Dual>(xd, dxs, xn2);
    for (int i = 0; i < NQ + NV; i++) xref[i] = Dual(x[i]);
    mb_difference<Dual>(xref, xn2, gap);
    for (int i = 0; i < 56; i++) {
      double an = (j < 56) ? e.A[i * 56 + j] : e.B[i * 34 + (j - 56)];
      err = std::max(err, std::fabs(gap[i].d - an));
    }
  }
  return err;
}

int orc_num_procs() { return omp_get_num_procs(); }

// ---- dense QP (SURVEY 8f row f-3): batch of QPs, OpenMP over the batch; strides in doubles per QP (0 = shared)
void orc_qp_default_settings(mpc_qp_settings_t *s) { qp_default_settings(*s); }
int orc_qp_solve(int n, int ne, int ni, int box, int batch, const mpc_qp_settings_t *st, const double *H, long sH, const double *g, long sg,
                 const double *A, long sA, const double *b, long sb, const double *C, long sC, const double *l, long sl, const double *u, long su,
                 const double *lb, long slb, const double *ub, long sub, double *x, double *y, double *z, mpc_qp_info_t *info, int threads) {
  const int nz = ni + (box ? n : 0);
  int worst = 0;
#pragma omp parallel for schedule(dynamic) num_threads(threads > 0 ? threads : omp_get_max_threads()) reduction(max : worst)
  for (int i = 0; i < batch; i++) {
    QP q{n, ne, ni, box != 0, H + i * sH, g + i * sg, A + i * sA, b + i * sb, C + i * sC, l + i * sl, u + i * su,
         box ? lb + i * slb : nullptr, box ? ub + i * sub : nullptr};
    const int s = qp_solve(q, *st, x + (long)i * n, y + (long)i * ne, z + (long)i * nz, info ? info + i : nullptr);
    worst = std::max(worst, s);
  }
  return worst;
}
void orc_qp_assemble_id(int batch, const double *M, const double *nle, const double *Jc, const double *gamma, const double *a, const double *forces,
                        const int32_t *cs, double mu, double L, double W, double *A, double *b, double *C, double *l) {
  for (int i = 0; i < batch; i++)
    qp_assemble_id(M + i * 784, nle + i * 28, Jc + i * 336, gamma + i * 12, a + i * 28, forces + i * 12, cs + i * 2, mu, L, W, A + i * 2480, b + i * 40,
                   C + i * 1116, l + i * 18);
}

// ---- IKID task terms (IKIDSolver_f6) on the oracle's own rigid-body code (rbd.hpp), not on the kernels' composite formulation.
// Ag [6][NV] (centroidal_derivatives), dAgv [6] (centroidal_rate at qdd = 0, gravity excluded), the angular rows of the LOCAL Jacobians
// of two frames Jang [2][3][NV] and their dJ v [2][3] column by column from forward_kin, plus the frame placements oMf [2][12].
// Any output may be NULL.
void orc_ikid_terms(const mpc_robot_t *rb, const double *x, const int *frame_body, const double *frame_place, double *Ag, double *dAgv,
                    double *Jang, double *dJang, double *oMf) {
  Tree tr(rb);
  static Kin<double> k;
  forward_kin<double>(tr, x, x + NQ, k);
  double dhq[6 * NV], ag[6 * NV];
  centroidal_derivatives(tr, k, dhq, ag);
  if (Ag) for (int i = 0; i < 6 * NV; i++) Ag[i] = ag[i];
  // centroidal_rate folds gravity in as a_world = -g: remove its wrench at the CoM, [m (-g); 0]
  V6<double> F = centroidal_rate<double>(tr, k, x + NQ, nullptr);
  if (dAgv) for (int i = 0; i < 6; i++) dAgv[i] = F[i] + (i < 3 ? k.mass * rb->gravity[i] : 0.0);
  V6<double> a[NB];
  body_accels<double>(tr, k, x + NQ, nullptr, false, a);
  for (int f = 0; f < 2; f++) {
    const int b = frame_body[f];
    SE3<double> Mf = mul(k.oM[b], se3_cast<double>(frame_place + 12 * f));
    for (int j = 0; j < NV; j++) {
      V6<double> col = tr.anc[body_of_dof(j)][b] ? actinv_motion(Mf, k.S[j]) : zero6<double>();
      if (Jang) for (int r = 0; r < 3; r++) Jang[(3 * f + r) * NV + j] = col[3 + r];
    }
    V6<double> acc = actinv_motion(Mf, a[b]);
    if (dJang) for (int r = 0; r < 3; r++) dJang[3 * f + r] = acc[3 + r];
    if (oMf) {
      for (int i = 0; i < 9; i++) oMf[12 * f + i] = Mf.R[i];
      for (int i = 0; i < 3; i++) oMf[12 * f + 9 + i] = Mf.p[i];
    }
  }
}
}
