// What the full-dynamics and kinodynamic evaluations of a Talos knot share: the knot's I/O, the world-frame rigid-body phases
// (kinematics, subtree sums, body forces, bias pass, CRBA, sole motion, centroidal map, composite inertias and force-derivative
// columns; rbd_terms.cuh runs them too), the multibody cost stack (state, centroidal momentum, foot placements), the normal-cone
// projection, the back end of a running knot (constraint rows and shooting gap -> merit partials and LQ blocks) and the terminal knot.
// Each model file keeps its own dynamics solve, tangent assembly, constraint-row definitions and extra cost terms.
#pragma once
#include "model.cuh"

namespace mpcdev {

constexpr int FN = 56; // tangent dimension of the multibody state

// merit / infeasibility partials written per knot
enum { SC_COST = 0, SC_PEN, SC_PRIM, SC_DUAL, SC_INNER, SC_COUNT = 8 };

struct KnotIO {
  // inputs
  const double *x, *u, *xn;        // x_k, u_k, x_{k+1}
  const mpc_knot_t *kn;
  const mpc_term_t *tm;
  const double *v, *v_prev;        // constraint multipliers of this knot (current / BCL estimate)
  const double *lam_k;             // co-state of x_k (dynamics k-1, or initial condition for k = 0)
  const double *lam_n, *lam_n_prev;// co-state of x_{k+1}
  double mu, preg;
  int k, T;
  // outputs (derivative pass)
  double *AB, *H, *lxu, *g, *T6, *E6, *gE_next, *fbar, *dbar, *vplus, *lplus, *CDact;
  int32_t *nca, *act_idx;
  // outputs (both passes)
  double *gap, *h, *scal, *xdot, *lamc;
  // ROLLOUT_NONLINEAR (fused rollout kernel, values pass only): x_{k+1} is not an input but DEFINED here as f(x, u) (+) slack and written out
  const double *slack; double *xn_out;
  double *scratch;   // derivative pass: this knot's slot of the Riccati W buffer (n x nz doubles, dead until the Riccati kernel writes it):
                     // holds the tangent X = da/dz (NV x nz) and dlam/dz (12 x nz), which stay L2-resident between the phases
  double *phase_out; // profiling builds only
};

// ------------------------------------------------------------------ rigid-body phases
// One copy of each recursion of the evaluations and of rbd_terms.cuh, after the oracle's (oracle/rbd.hpp).  A helper is either one
// PAR_FOR phase or the body of one work item; none has a barrier inside, so every caller keeps its own SYNC() placement.

// subtree sums dst_b = sum_{d in sub(b)} src_d of a per-body quantity W doubles wide, one thread per element
template <int W> HD void mb_subtree_sum(const DevModel &m, const double *src, double *dst) {
  PAR_FOR(e, NB * W) {
    const int b = e / W, c = e % W;
    const uint32_t mask = m.sub_mask[b];
    double s = 0;
    for (int d = b; d < NB; d++) if (mask >> d & 1) s += src[W * d + c];
    dst[e] = s;
  }
}

// body force I_b a_b + v_b x* (I_b v_b) for the body acceleration ab (hb = I_b v_b from mb_kinematics)
template <class WS> HD void mb_body_force(const WS &w, int b, const double *ab, double *fb) {
  double t1[6], t2[6];
  inertia_mul(w.I + 10 * b, ab, t1);
  cross_mf(w.v + 6 * b, w.hb + 6 * b, t2);
  for (int i = 0; i < 6; i++) fb[i] = t1[i] + t2[i];
}

// ------------------------------------------------------------------ kinematics shared by running / terminal knots
// fills oM, S, I, v, hb, Ic, hsub, com, ofoot, Jf
template <class WS> HD void mb_kinematics(const DevModel &m, WS &w) {
  const mpc_robot_t &rb = m.rb;
  const double *q = w.x, *qd = w.x + NQ;
  // every body's placement relative to its parent (joint placement x joint rotation) is independent of the tree: all bodies
  // in parallel, off the level chain; the chain itself is then one SE(3) product per level
  PAR_FOR(b, NB) {
    double *o = w.oM + 12 * b;
    if (b == 0) { quat_to_R(q + 3, o); o[9] = q[0]; o[10] = q[1]; o[11] = q[2]; }
    else {
      // Rodrigues with the unit joint axis: R = I + sin(q) [a]x + (1 - cos q) [a]x^2
      double sn, cs, jr[12], K[9], K2[9];
      sincos(q[6 + b], &sn, &cs);
      skew3(rb.axis[b], K); mat3_mul(K, K, K2);
      for (int i = 0; i < 9; i++) jr[i] = ((i % 4 == 0) ? 1.0 : 0.0) + sn * K[i] + (1.0 - cs) * K2[i];
      jr[9] = jr[10] = jr[11] = 0;
      se3_mul(rb.jplace[b], jr, o);
    }
  }
  SYNC();
  for (int l = 1; l < m.nlevels; l++) {
    int n = m.level_start[l + 1] - m.level_start[l];
    PAR_FOR(t, n) {
      int b = m.level_body[m.level_start[l] + t];
      double loc[12];
      for (int i = 0; i < 12; i++) loc[i] = w.oM[12 * b + i];
      se3_mul(w.oM + 12 * rb.parent[b], loc, w.oM + 12 * b);
    }
    SYNC();
  }
  PAR_FOR(j, NV) {
    int b = body_of_dof(j);
    double e[6] = {0, 0, 0, 0, 0, 0};
    if (j < 6) e[j] = 1.0; else { e[3] = rb.axis[b][0]; e[4] = rb.axis[b][1]; e[5] = rb.axis[b][2]; }
    se3_act_motion(w.oM + 12 * b, e, w.S + 6 * j);
  }
  PAR_FOR(b, NB) {
    const double *o = w.oM + 12 * b;
    double cw[3], RI[9], Iw[9];
    mat3_vec(o, rb.com[b], cw);
    for (int i = 0; i < 3; i++) cw[i] += o[9 + i];
    mat3_mul(o, rb.inertia[b], RI);
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) Iw[3 * i + j] = RI[3 * i] * o[3 * j] + RI[3 * i + 1] * o[3 * j + 1] + RI[3 * i + 2] * o[3 * j + 2];
    double ms = rb.mass[b], c2 = dot3(cw, cw);
    double *I = w.I + 10 * b;
    I[0] = ms; I[1] = ms * cw[0]; I[2] = ms * cw[1]; I[3] = ms * cw[2];
    I[4] = Iw[0] + ms * (c2 - cw[0] * cw[0]); I[5] = Iw[1] - ms * cw[0] * cw[1]; I[6] = Iw[2] - ms * cw[0] * cw[2];
    I[7] = Iw[4] + ms * (c2 - cw[1] * cw[1]); I[8] = Iw[5] - ms * cw[1] * cw[2]; I[9] = Iw[8] + ms * (c2 - cw[2] * cw[2]);
  }
  PAR_FOR(f, 2) se3_mul(w.oM + 12 * rb.foot_body[f], rb.foot_place[f], w.ofoot + 12 * f);
  SYNC();
  PAR_FOR(e, NB * 6) {
    int b = e / 6, c = e % 6;
    uint32_t mask = m.ancdof_mask[b];
    double s = 0;
    for (int j = 0; j < NV; j++) if (mask >> j & 1) s += w.S[6 * j + c] * qd[j];
    w.v[e] = s;
  }
  PAR_FOR(e, 2 * NV) {
    int f = e / NV, j = e % NV;
    double col[6] = {0, 0, 0, 0, 0, 0};
    if (m.ancdof_mask[rb.foot_body[f]] >> j & 1) se3_actinv_motion(w.ofoot + 12 * f, w.S + 6 * j, col);
    for (int r = 0; r < 6; r++) w.Jf[(6 * f + r) * NV + j] = col[r];
  }
  mb_subtree_sum<10>(m, w.I, w.Ic);
  SYNC();
  PAR_FOR(b, NB) inertia_mul(w.I + 10 * b, w.v + 6 * b, w.hb + 6 * b);
  PAR_FOR(j, NV) inertia_mul(w.Ic + 10 * body_of_dof(j), w.S + 6 * j, w.U + 6 * j);
  SYNC();
  mb_subtree_sum<6>(m, w.hb, w.hsub);
  ONE_THREAD { for (int i = 0; i < 3; i++) w.com[i] = w.Ic[1 + i] / w.Ic[0]; }
  SYNC();
}

// Composite B of every subtree, Bc_b e_c = sum_{k in sub(b)} I_k (e_c x v_k) + e_c x* (I_k v_k) + v_k x* (I_k e_c):
// first each body's own 6 x 6 block (one column per work item, all bodies in parallel), then the subtree sums with one
// thread per matrix element walking the bodies leaves-to-root (bodies are ordered parents-first, so a child is complete
// before it is added to its parent): no barrier inside the accumulation and no O(subtree) work per item.
template <class WS> HD void mb_composite_B(const DevModel &m, WS &w) {
  PAR_FOR(e, NB * 6) {
    const int b = e / 6, c = e % 6;
    double ec[6] = {0, 0, 0, 0, 0, 0}, t0[6], t1[6], t2[6], t3[6], t4[6];
    ec[c] = 1.0;
    cross_mm(ec, w.v + 6 * b, t0);
    inertia_mul(w.I + 10 * b, t0, t1);
    cross_mf(ec, w.hb + 6 * b, t2);
    inertia_mul(w.I + 10 * b, ec, t3);
    cross_mf(w.v + 6 * b, t3, t4);
    for (int i = 0; i < 6; i++) w.Bc[36 * b + 6 * i + c] = t1[i] + t2[i] + t4[i];
  }
  SYNC();
  PAR_FOR(e, 36) {
    for (int b = NB - 1; b > 0; b--) w.Bc[36 * m.rb.parent[b] + e] += w.Bc[36 * b + e];
  }
  SYNC();
}

// bias pass: body accelerations with gravity folded in (a0 = [-g; 0] at the root) into w.a and body forces into w.f, for zero
// joint accelerations or, with JACC, for qdd = [0; qdd_j] (the kinodynamic joint accelerations; the base term comes later)
template <bool JACC = false, class WS> HD void mb_bias_forces(const DevModel &m, WS &w, const double *a0, const double *qdd_j = nullptr) {
  PAR_FOR(b, NB) {
    double acc[6] = {a0[0], a0[1], a0[2], 0, 0, 0};
    const uint32_t mask = m.anc_mask[b];
    for (int k = 1; k <= b; k++)
      if (mask >> k & 1) {
        double sj[6], c[6];
        for (int i = 0; i < 6; i++) sj[i] = w.S[6 * (5 + k) + i] * w.x[NQ + 5 + k];
        cross_mm(w.v + 6 * k, sj, c);
        if (JACC) for (int i = 0; i < 6; i++) acc[i] += c[i] + w.S[6 * (5 + k) + i] * qdd_j[k - 1];
        else for (int i = 0; i < 6; i++) acc[i] += c[i];
      }
    for (int i = 0; i < 6; i++) w.a[6 * b + i] = acc[i];
    mb_body_force(w, b, acc, w.f + 6 * b);
  }
}

// composite-rigid-body mass matrix M (NV x NV) from S and U = Ic S
template <class WS> HD void mb_crba(const DevModel &m, const WS &w, double *M) {
  PAR_FOR(e, NV * NV) {
    const int i = e / NV, j = e % NV, bi = body_of_dof(i), bj = body_of_dof(j);
    double v = 0;
    if (m.anc_mask[bj] >> bi & 1) v = dot6(w.S + 6 * i, w.U + 6 * j);
    else if (m.anc_mask[bi] >> bj & 1) v = dot6(w.S + 6 * j, w.U + 6 * i);
    M[e] = v;
  }
}

// LOCAL velocity of sole f and, with ACC, its acceleration at zero joint acceleration (dJ v: the bias acceleration w.a minus a0)
template <bool ACC = true, class WS> HD void mb_sole_motion(const DevModel &m, const WS &w, int f, const double *a0, double *vel, double *dJv = nullptr) {
  const int fb = m.rb.foot_body[f];
  se3_actinv_motion(w.ofoot + 12 * f, w.v + 6 * fb, vel);
  if (ACC) {
    double an[6];
    for (int i = 0; i < 6; i++) an[i] = w.a[6 * fb + i] - a0[i];
    se3_actinv_motion(w.ofoot + 12 * f, an, dJv);
  }
}

// centroidal momentum matrix A_g (6 x NV, linear rows first): column j = shift_to_com(U_j)
template <class WS> HD void mb_centroidal_map(const WS &w, double *Ag) {
  PAR_FOR(j, NV) {
    const double *Uj = w.U + 6 * j;
    double c[3];
    cross3(w.com, Uj, c);
    for (int r = 0; r < 3; r++) { Ag[r * NV + j] = Uj[r]; Ag[(3 + r) * NV + j] = Uj[3 + r] - c[r]; }
  }
}

// force-derivative column of dof j at body mb of subtree(J), J = body_of_dof(j): g = Ic_mb c_j + Bc_mb w_j (the oracle's
// total_force_derivatives), kind 0 (d/dq_j): w_j = s_j x v_pJ, c_j = s_j x a_pJ - w_j x v_pJ; kind 1 (d/dv_j): w_j = s_j,
// c_j = -s_j x (v_J + v_pJ); v_pJ, a_pJ of the parent of J, zero velocity and a0 at the root
template <class WS> HD void mb_force_column(const DevModel &m, const WS &w, int kind, int j, int mb, const double *a0, double *g) {
  const int J = body_of_dof(j), pJ = m.rb.parent[J];
  const double *s = w.S + 6 * j;
  double vp[6] = {0, 0, 0, 0, 0, 0}, ap[6] = {a0[0], a0[1], a0[2], 0, 0, 0};
  if (pJ >= 0) for (int i = 0; i < 6; i++) { vp[i] = w.v[6 * pJ + i]; ap[i] = w.a[6 * pJ + i]; }
  double cj[6], wj[6], t1[6], g2[6];
  if (kind == 0) {
    cross_mm(s, vp, wj);
    cross_mm(s, ap, cj);
    cross_mm(wj, vp, t1);
    for (int i = 0; i < 6; i++) cj[i] -= t1[i];
  } else {
    for (int i = 0; i < 6; i++) { wj[i] = s[i]; t1[i] = w.v[6 * J + i] + vp[i]; }
    cross_mm(s, t1, cj);
    for (int i = 0; i < 6; i++) cj[i] = -cj[i];
  }
  inertia_mul(w.Ic + 10 * mb, cj, g);
  mat6_vec(w.Bc + 36 * mb, wj, g2);
  for (int i = 0; i < 6; i++) g[i] += g2[i];
}

// centroidal momentum residual + Jacobian [dh/dq | A_g] (6 x 56), pose residuals + Jacobians, state error and — for running
// knots (gap_out != nullptr) — the base part of the semi-implicit Euler step, the shooting gap and the 6x6 Lie-group blocks
// P1 = Jlog6(D) Jexp6(dq), P2 = Jlog6(D) Ad(exp6(dq))^-1, E6 = -Jlog6(D) Ad(D^-1), T6 = -E6^-1 = Ad(D) Jexp6(log6 D).
// The single-thread Lie-group tasks are spread over the 4 warps in two dependent stages, the 6x6 products over all threads.
template <class WS, bool ROLL = false> HD void mb_cost_terms(const DevModel &m, WS &w, const double *lf_ref, const double *rf_ref, bool derivs, double *gap_out, const double *slack = nullptr) {
  const mpc_robot_t &rb = m.rb;
  // stage 1a: the relative placements whose logarithms are needed: both foot poses, the state error and the shooting gap
  PAR_FOR(task, 3 * 32) {
    if (task == 0) { // centroidal momentum value; integrator base block and gap placement
      const double *h = w.hsub;
      double c[3];
      cross3(w.com, h, c);
      for (int i = 0; i < 3; i++) { w.rcent[i] = h[i]; w.rcent[3 + i] = h[3 + i] - c[i]; }
      if (gap_out) {
        double pn[3], Mn[12], Mp[12];
        exp6(w.dx, w.eexp);
        mat3_vec(w.oM, w.eexp + 9, pn);
        for (int i = 0; i < 3; i++) w.xnext[i] = w.x[i] + pn[i];
        quat_integrate(w.x + 3, w.dx + 3, w.xnext + 3);
        if (ROLL) { // nonlinear rollout: x_{k+1} := f(x, u) (+) slack (base part; joints and velocities below)
          double es[12], Rn[9], ps[3];
          exp6(slack, es); quat_to_R(w.xnext + 3, Rn); mat3_vec(Rn, es + 9, ps);
          for (int i = 0; i < 3; i++) w.xn[i] = w.xnext[i] + ps[i];
          quat_integrate(w.xnext + 3, slack + 3, w.xn + 3);
        }
        quat_to_R(w.xn + 3, Mn); Mn[9] = w.xn[0]; Mn[10] = w.xn[1]; Mn[11] = w.xn[2];
        quat_to_R(w.xnext + 3, Mp); Mp[9] = w.xnext[0]; Mp[10] = w.xnext[1]; Mp[11] = w.xnext[2];
        se3_inv_mul(Mn, Mp, w.Dgap);
      }
    } else if (task == 32 || task == 64) { // foot pose placements
      int f = task == 32 ? 0 : 1;
      se3_inv_mul(f == 0 ? lf_ref : rf_ref, w.ofoot + 12 * f, w.Dl + 12 * f);
    } else if (task == 65) { // state error e = x (-) x_ref (second lane of the third warp: groups may have only three warps)
      double Mr[12], Mx[12];
      quat_to_R(m.cfg.x_ref + 3, Mr); Mr[9] = m.cfg.x_ref[0]; Mr[10] = m.cfg.x_ref[1]; Mr[11] = m.cfg.x_ref[2];
      for (int i = 0; i < 12; i++) Mx[i] = w.oM[i];
      se3_inv_mul(Mr, Mx, w.Dl + 24);
    }
  }
  SYNC();
  // stage 1b: ONE copy of log6 / Jlog6 run by up to four lanes of a warp side by side (the evaluation kernels are
  // instruction-fetch bound: every inlined copy of these long routines costs cold instruction-cache misses)
  PAR_FOR(item, gap_out ? 4 : 3) {
    const double *D = (item == 3) ? w.Dgap : w.Dl + 12 * item;
    double *out = (item < 2) ? w.rpose + 6 * item : (item == 2) ? w.estate : w.lgap;
    log6(D, out);
    if (derivs) Jlog6_from_log(out, (item < 2) ? w.Jlp + 36 * item : (item == 2) ? w.Jls : w.late.Jlg);
  }
  SYNC();
  if (gap_out) PAR_FOR(i, 6) gap_out[i] = w.fbr[i] = w.lgap[i]; // fbr temporarily holds the gap
  PAR_FOR(i, FN - 6) {
    int a = 6 + i;
    w.estate[a] = (a < NV) ? (w.x[7 + a - 6] - m.cfg.x_ref[7 + a - 6]) : (w.x[NQ + a - NV] - m.cfg.x_ref[NQ + a - NV]);
  }
  if (gap_out) {
    PAR_FOR(i, NJ) { w.xnext[7 + i] = w.x[7 + i] + w.dx[6 + i]; if (ROLL) w.xn[7 + i] = w.xnext[7 + i] + slack[6 + i]; gap_out[6 + i] = w.fbr[6 + i] = w.xnext[7 + i] - w.xn[7 + i]; }
    PAR_FOR(i, NV) { w.xnext[NQ + i] = w.x[NQ + i] + w.dx[NV + i]; if (ROLL) w.xn[NQ + i] = w.xnext[NQ + i] + slack[NV + i]; gap_out[NV + i] = w.fbr[NV + i] = w.xnext[NQ + i] - w.xn[NQ + i]; }
  }
  SYNC();
  if (!derivs) return;
  if (gap_out) {
    PAR_FOR(task, 3 * 32) {
      const double id[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
      if (task == 0) { double inv[12]; se3_inv_mul(w.Dgap, id, inv); se3_action_matrix(inv, w.late.AdDi); }
      else if (task == 32 || task == 33) Jexp6(task == 32 ? w.dx : w.lgap, task == 32 ? w.late.Jd : w.late.Jrg); // two lanes, one copy
      else if (task == 64) { double einv[12]; se3_inv_mul(w.eexp, id, einv); se3_action_matrix(einv, w.late.Ade); se3_action_matrix(w.Dgap, w.late.AdD); }
    }
  }
  PAR_FOR(e, 2 * 6 * NV) { // Jpose = Jlog6 * Jf
    int f = e / (6 * NV), r = (e / NV) % 6, j = e % NV;
    const double *Jl = w.Jlp + 36 * f;
    double s = 0;
    for (int k = 0; k < 6; k++) s += Jl[6 * r + k] * w.Jf[(6 * f + k) * NV + j];
    w.cj.Jpose[e] = s;
  }
  PAR_FOR(j, NV) { // centroidal derivative columns
    int J = body_of_dof(j), pJ = rb.parent[J];
    const double *s = w.S + 6 * j;
    double vp[6] = {0, 0, 0, 0, 0, 0};
    if (pJ >= 0) for (int i = 0; i < 6; i++) vp[i] = w.v[6 * pJ + i];
    double wj[6], t1[6], t2[6], dho[6], Is[6];
    cross_mm(s, vp, wj);
    cross_mf(s, w.hsub + 6 * J, t1);
    inertia_mul(w.Ic + 10 * J, wj, t2);
    for (int i = 0; i < 6; i++) dho[i] = t1[i] - t2[i];
    inertia_mul(w.Ic + 10 * J, s, Is);
    const double im_ = rcp_(w.Ic[0]);
    double dc[3] = {Is[0] * im_, Is[1] * im_, Is[2] * im_};
    double c1[3], c2[3], c3[3];
    cross3(dc, w.hsub, c1); cross3(w.com, dho, c2); cross3(w.com, Is, c3);
    for (int r = 0; r < 3; r++) {
      w.cj.Jcent[r * FN + j] = dho[r]; w.cj.Jcent[(3 + r) * FN + j] = dho[3 + r] - c1[r] - c2[r];
      w.cj.Jcent[r * FN + NV + j] = Is[r]; w.cj.Jcent[(3 + r) * FN + NV + j] = Is[3 + r] - c3[r];
    }
  }
  SYNC();
  if (gap_out) {
    PAR_FOR(e, 4 * 36) {
      int which = e / 36, i = (e % 36) / 6, j = e % 6;
      const double *A = (which == 3) ? w.late.AdD : w.late.Jlg;
      const double *B = (which == 0) ? w.late.AdDi : (which == 1) ? w.late.Jd : (which == 2) ? w.late.Ade : w.late.Jrg;
      double sacc = 0;
      for (int k = 0; k < 6; k++) sacc += A[6 * i + k] * B[6 * k + j];
      if (which == 0) w.late.E6[6 * i + j] = -sacc; else if (which == 1) w.late.P1[6 * i + j] = sacc; else if (which == 2) w.late.P2[6 * i + j] = sacc; else w.late.T6[6 * i + j] = sacc;
    }
    SYNC();
  }
}

// value + gradient + Gauss-Newton Hessian contributions of the multibody cost stack at (a, b) / z
template <class WS> HD double mb_cost_value(const WS &w, const double *wx, const double *wcent, const double *wlf, const double *wrf) {
  double c = 0;
  for (int i = 0; i < FN; i++) c += 0.5 * wx[i] * w.estate[i] * w.estate[i];
  for (int i = 0; i < 6; i++) c += 0.5 * (wcent[i] * w.rcent[i] * w.rcent[i] + wlf[i] * w.rpose[i] * w.rpose[i] + wrf[i] * w.rpose[6 + i] * w.rpose[6 + i]);
  return c;
}
template <class WS> HD double mb_cost_grad(const WS &w, const double *wx, const double *wcent, const double *wlf, const double *wrf, int z) {
  double g = 0;
  if (z < 6) { for (int r = 0; r < 6; r++) g += wx[r] * w.Jls[6 * r + z] * w.estate[r]; }
  else if (z < FN) g += wx[z] * w.estate[z];
  if (z < FN) for (int r = 0; r < 6; r++) g += wcent[r] * w.cj.Jcent[r * FN + z] * w.rcent[r];
  if (z < NV) for (int r = 0; r < 6; r++) g += wlf[r] * w.cj.Jpose[r * NV + z] * w.rpose[r] + wrf[r] * w.cj.Jpose[(6 + r) * NV + z] * w.rpose[6 + r];
  return g;
}
template <class WS> HD double mb_cost_hess(const WS &w, const double *wx, const double *wcent, const double *wlf, const double *wrf, int a, int b) {
  double h = 0; // a <= b
  if (b < 6) { for (int r = 0; r < 6; r++) h += wx[r] * w.Jls[6 * r + a] * w.Jls[6 * r + b]; }
  else if (a == b && a < FN) h += wx[a];
  if (b < FN) for (int r = 0; r < 6; r++) if (wcent[r] != 0.0) h += wcent[r] * w.cj.Jcent[r * FN + a] * w.cj.Jcent[r * FN + b];
  if (b < NV) for (int r = 0; r < 6; r++) h += wlf[r] * w.cj.Jpose[r * NV + a] * w.cj.Jpose[r * NV + b] + wrf[r] * w.cj.Jpose[(6 + r) * NV + a] * w.cj.Jpose[(6 + r) * NV + b];
  return h;
}

// normal-cone projection pieces (SURVEY App. A6, C14)
HD double vplus_row(int type, double h, double ve, double mu, double lo, double hi, int &act, double &prim) {
  double wv = h + mu * ve;
  if (type == 0) { act = 1; prim = h; return wv * rcp_(mu); }
  if (type == 1) { if (wv > 0) { act = 1; prim = h; return wv * rcp_(mu); } act = 0; prim = h - wv; return 0.0; }
  if (type == 2) {
    if (wv > hi) { act = 1; prim = h - hi; return (wv - hi) * rcp_(mu); }
    if (wv < lo) { act = 1; prim = h - lo; return (wv - lo) * rcp_(mu); }
    act = 0; prim = h - wv; return 0.0;
  }
  act = 0; prim = 0; return 0.0;
}

// ------------------------------------------------------------------ back end of a running knot
// The caller defines its rows and cost terms and keeps the phase order and the barriers between phases; the merit pieces are
// accumulated per thread (acc_*) and reduced once in mb_merit_finish.

// constraint row r once its (type, h, lo, hi) is known: projected multiplier, activity, dbar and the row's merit pieces;
// v / v_prev are this knot's multipliers (current / BCL estimate), wherever the caller reads them from
template <class WS> HD void mb_row_epilogue(WS &w, const KnotIO &io, int r, int type, double hv, double lo, double hi, const double *v,
                                            const double *v_prev, double &acc_pen, double &acc_prim, double &acc_inner) {
  int act = 0; double prim = 0;
  const double vp = vplus_row(type, hv, v_prev[r], io.mu, lo, hi, act, prim), dv = vp - v[r];
  w.ctype[r] = type; w.late.hval[r] = hv; w.late.vpl[r] = vp; w.isact[r] = act;
  w.late.dbr[r] = io.mu * dv;
  io.h[r] = hv;
  if (type >= 0) {
    acc_pen += 0.5 * io.mu * (vp * vp + dv * dv);
    acc_prim = fmax(acc_prim, fabs(prim));
    acc_inner = fmax(acc_inner, fabs(io.mu * dv));
  }
}

// dynamics rows (fbr holds the shooting gap on entry, mu (lplus - lam_{k+1}) on exit) and the state cost;
// lam_n / lam_n_prev: co-state of x_{k+1} and its estimate
template <class WS> HD void mb_dynamics_rows(const DevModel &m, WS &w, const KnotIO &io, const double *lam_n, const double *lam_n_prev,
                                             double &acc_cost, double &acc_pen, double &acc_prim, double &acc_inner) {
  PAR_FOR(i, FN) {
    const double gap = w.fbr[i], lp = lam_n_prev[i] + gap * rcp_(io.mu), dl = lp - lam_n[i]; // fbr = gap here
    w.lpl[i] = lp;
    w.fbr[i] = io.mu * dl;
    acc_pen += 0.5 * io.mu * (lp * lp + dl * dl);
    acc_prim = fmax(acc_prim, fabs(gap));
    acc_inner = fmax(acc_inner, fabs(io.mu * dl));
    acc_cost += 0.5 * m.cfg.wx[i] * w.estate[i] * w.estate[i];
  }
}

// group-wide reduction of the merit pieces into w.scal (dual residual 0 until mb_dual_scal), then the active rows compacted
template <int NC, class WS> HD void mb_merit_finish(WS &w, double acc_cost, double acc_pen, double acc_prim, double acc_inner) {
  reduce_sum2_max2(acc_cost, acc_pen, acc_prim, acc_inner, w.part, w.part + 16);
  ONE_THREAD { w.scal[SC_COST] = w.part[16]; w.scal[SC_PEN] = w.part[17]; w.scal[SC_PRIM] = w.part[18]; w.scal[SC_INNER] = w.part[19]; w.scal[SC_DUAL] = 0; }
  compact_flags(w.isact, NC, w.act_idx, &w.nca, reinterpret_cast<int32_t *>(w.part));
}

// per-row LQ vectors to HBM
template <int NC, class WS> HD void mb_store_rows(const WS &w, const KnotIO &io) {
  PAR_FOR(i, NC) { io.dbar[i] = w.late.dbr[i]; io.vplus[i] = w.late.vpl[i]; io.act_idx[i] = (i < w.nca) ? w.act_idx[i] : -1; }
  PAR_FOR(i, FN) { io.fbar[i] = w.fbr[i]; io.lplus[i] = w.lpl[i]; }
  PAR_FOR(i, 36) { io.T6[i] = w.late.T6[i]; io.E6[i] = w.late.E6[i]; }
  ONE_THREAD io.nca[0] = w.nca;
}

// column z of [A B] (NV rows of the semi-implicit Euler step of q, the base rows mapped by P1 / P2, then NV rows of v) from the
// tangent column da/dz = xc[i * stride]; returns lam_{k+1}' [A B] e_z
template <int NZ, class WS> HD double mb_ab_column(const WS &w, const KnotIO &io, int z, const double *xc, int stride, double dt, const double *lam_n) {
  const double dt2 = dt * dt;
  double d6[6], acc = 0;
  for (int k = 0; k < 6; k++) d6[k] = dt2 * xc[k * stride] + ((z == NV + k) ? dt : 0.0);
  for (int i = 0; i < 6; i++) {
    double s = (z < 6) ? w.late.P2[6 * i + z] : 0.0;
    for (int k = 0; k < 6; k++) s += w.late.P1[6 * i + k] * d6[k];
    io.AB[i * NZ + z] = s; acc += s * lam_n[i];
  }
  for (int i = 6; i < NV; i++) {
    double s = dt2 * xc[i * stride] + ((z == NV + i) ? dt : 0.0) + ((z == i) ? 1.0 : 0.0);
    io.AB[i * NZ + z] = s; acc += s * lam_n[i];
  }
  for (int i = 0; i < NV; i++) {
    double s = dt * xc[i * stride] + ((z == NV + i) ? 1.0 : 0.0);
    io.AB[(NV + i) * NZ + z] = s; acc += s * lam_n[NV + i];
  }
  return acc;
}

// E_k' lam_{k+1}, base block, for the next knot's gradient
template <class WS> HD void mb_gE_next(const WS &w, const KnotIO &io, const double *lam_n) {
  PAR_FOR(j, 6) {
    double s = 0;
    for (int i = 0; i < 6; i++) s += w.late.E6[6 * i + j] * lam_n[i];
    io.gE_next[j] = s;
  }
}

// Gauss-Newton Hessian H = sum_r w_r J_r' J_r (+ preg and the state / control diagonals) on 4 x 4 register tiles of the upper
// triangle.  model_rows(rank1) adds the weighted rows of the model's own cost terms, rank1(J_r, ncols, w_r); the multibody cost
// stack (centroidal momentum, foot poses, base block of the state error) follows.
template <int NZ, class WS, class Rows> HD void mb_gn_hessian(const WS &w, const KnotIO &io, const mpc_config_t &cfg, const mpc_knot_t &kn, Rows model_rows) {
  constexpr int HT = (NZ + 3) / 4;
  PAR_FOR(t, HT * HT) {
    const int ta = t / HT, tb = t % HT;
    if (tb < ta) continue;
    const int a0 = 4 * ta, b0 = 4 * tb;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) acc[i][j] = 0.0;
    auto rank1 = [&](const double *J, int ncols, double wgt) {
      double va[4], vb[4];
#pragma unroll
      for (int i = 0; i < 4; i++) { va[i] = (a0 + i < ncols) ? wgt * J[a0 + i] : 0.0; vb[i] = (b0 + i < ncols) ? J[b0 + i] : 0.0; }
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] += va[i] * vb[j];
    };
    model_rows(rank1);
    if (a0 < FN) {
      for (int r = 0; r < 6; r++) if (cfg.w_cent[r] != 0.0) rank1(w.cj.Jcent + r * FN, FN, cfg.w_cent[r]);
      if (a0 < NV && b0 < NV)
        for (int r = 0; r < 6; r++) {
          if (kn.w_lf[r] != 0.0) rank1(w.cj.Jpose + r * NV, NV, kn.w_lf[r]);
          if (kn.w_rf[r] != 0.0) rank1(w.cj.Jpose + (6 + r) * NV, NV, kn.w_rf[r]);
        }
      if (b0 < 8 && a0 < 8) for (int r = 0; r < 6; r++) rank1(w.Jls + 6 * r, 6, cfg.wx[r]);
    }
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int a = a0 + i, b = b0 + j;
        if (a >= NZ || b >= NZ || b < a) continue;
        double hv = acc[i][j];
        if (a == b) { hv += io.preg; if (a >= FN) hv += cfg.wu[a - FN]; else if (a >= 6) hv += cfg.wx[a]; }
        io.H[a * NZ + b] = hv; io.H[b * NZ + a] = hv;
      }
  }
}

// once g is complete: dual residual of this knot without the base block of the x-gradient (finalised in the reduction kernel),
// then every merit / infeasibility partial to HBM
template <int NZ, class WS> HD void mb_dual_scal(WS &w, const KnotIO &io) {
  SYNC();
  PAR_FOR(c, 8) {
    double dual = 0;
    for (int z = 6 + c; z < NZ; z += 8) {
      if (io.k == 0 && z < FN) continue;
      dual = fmax(dual, fabs(w.late.g[z]));
    }
    w.part[c] = dual;
  }
  SYNC();
  PAR_FOR(i, SC_COUNT) {
    double v = w.scal[i];
    if (i == SC_DUAL) for (int c = 0; c < 8; c++) v = fmax(v, w.part[c]);
    io.scal[i] = v;
  }
}

// ------------------------------------------------------------------ terminal knot
// optional CoM equality on rows 0-2 (fulldynamic_talos.py:499-507, kinodynamic_talos.py:176-180,276); COST adds the multibody cost
// stack with the *_term weights (fulldynamic_talos.py:234-245), the kinodynamic terminal cost is empty (kinodynamic_talos.py:175)
template <bool DERIV, bool COST, int NZ, int NC, class WS> HD void eval_mb_term(const DevModel &m, const KnotIO &io, WS &w) {
  const mpc_config_t &cfg = m.cfg;
  PAR_FOR(i, NQ + NV) w.x[i] = io.x[i];
  SYNC();
  mb_kinematics(m, w);
  if (COST) mb_cost_terms(m, w, io.tm->lf_ref, io.tm->rf_ref, DERIV, nullptr);
  const bool has_c = io.tm->has_com_cstr != 0.0;
  PAR_FOR(r, NC) {
    int type = -1; double hv = 0;
    if (r < 3 && has_c) { type = 0; hv = w.com[r] - io.tm->com_ref[r]; }
    int act = 0; double prim = 0;
    double vp = vplus_row(type, hv, io.v_prev[r], io.mu, 0, 0, act, prim);
    w.ctype[r] = type; w.late.hval[r] = hv; w.late.vpl[r] = vp; w.isact[r] = act; w.late.dbr[r] = io.mu * (vp - io.v[r]); w.late.rowtmp[r] = fabs(prim);
    io.h[r] = hv;
  }
  SYNC();
  ONE_THREAD {
    double cost = COST ? mb_cost_value(w, cfg.wx_term, cfg.w_cent_term, cfg.w_foot_term, cfg.w_foot_term) : 0.0, pen = 0, prim = 0, inner = 0;
    int nca = 0;
    for (int r = 0; r < 3; r++) {
      if (w.ctype[r] < 0) continue;
      double dv = w.late.vpl[r] - io.v[r];
      pen += 0.5 * io.mu * (w.late.vpl[r] * w.late.vpl[r] + dv * dv);
      prim = fmax(prim, w.late.rowtmp[r]); inner = fmax(inner, fabs(w.late.dbr[r]));
      if (w.isact[r]) w.act_idx[nca++] = r;
    }
    w.nca = nca;
    w.scal[SC_COST] = cost; w.scal[SC_PEN] = pen; w.scal[SC_PRIM] = prim; w.scal[SC_INNER] = inner; w.scal[SC_DUAL] = 0;
  }
  SYNC();
  if (!DERIV) { PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i]; return; }
  PAR_FOR(i, NC) { io.dbar[i] = w.late.dbr[i]; io.vplus[i] = w.late.vpl[i]; io.act_idx[i] = (i < w.nca) ? w.act_idx[i] : -1; }
  ONE_THREAD io.nca[0] = w.nca;
  PAR_FOR(z, NZ) {
    double lz = (COST && z < FN) ? mb_cost_grad(w, cfg.wx_term, cfg.w_cent_term, cfg.w_foot_term, cfg.w_foot_term, z) : 0.0;
    io.lxu[z] = lz;
    double gz = lz;
    if (z < NV && has_c) for (int r = 0; r < 3; r++) gz += io.v[r] * w.U[6 * z + r] * rcp_(w.Ic[0]);
    if (z >= 6 && z < FN) gz -= io.lam_k[z];
    w.late.g[z] = gz; io.g[z] = gz;
  }
  PAR_FOR(e, NZ * NZ) {
    int a = e / NZ, b = e % NZ;
    double hv = 0;
    if (!COST) hv = (a == b && a < FN) ? io.preg : 0.0;
    else if (a < FN && b < FN) { hv = (a <= b) ? mb_cost_hess(w, cfg.wx_term, cfg.w_cent_term, cfg.w_foot_term, cfg.w_foot_term, a, b)
                                               : mb_cost_hess(w, cfg.wx_term, cfg.w_cent_term, cfg.w_foot_term, cfg.w_foot_term, b, a);
      if (a == b) hv += io.preg; }
    io.H[e] = hv;
  }
  PAR_FOR(e, w.nca * NZ) {
    int ai = e / NZ, z = e % NZ, r = w.act_idx[ai];
    io.CDact[e] = (z < NV) ? w.U[6 * z + r] * rcp_(w.Ic[0]) : 0.0; // Jcom column = lin(Ic_J s_j) / mass
  }
  SYNC();
  ONE_THREAD {
    double dual = 0;
    for (int z = 6; z < FN; z++) dual = fmax(dual, fabs(w.late.g[z]));
    w.scal[SC_DUAL] = dual;
  }
  SYNC();
  PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i];
}

} // namespace mpcdev
