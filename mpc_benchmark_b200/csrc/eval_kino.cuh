// Per-knot evaluation of the KINODYNAMIC Talos stage: one CTA per (instance, knot).
//
// Replaces KinodynamicsFwdDynamics + IntegratorSemiImplEuler (kinodynamic_talos.py:107-112), the CostStack of
// kinodynamic_talos.py:137-157 (state, control, CentroidalMomentumResidual, CentroidalMomentumDerivativeResidual,
// FramePlacementResidual x2) and the constraints of :161-171 (joint box, CentroidalWrenchConeResidual + zero LOCAL
// FrameVelocityResidual per active contact).  u = [w_L(6), w_R(6), a_joint(22)]; the base acceleration solves
//   A_g[:, :6] a_b = hdot'(q, u) - F_g(q, v, [0; a_j])           (SURVEY App. A5; F_g with a_world = -g, see oracle/rbd.hpp)
// and its derivatives reuse the world-frame tangent machinery of eval_mb.cuh: d F_o / d q_j = s_j x* F_J - (Ic_J c_j + Bc_J w_j).
#pragma once
#include "eval_mb.cuh"

namespace mpcdev {

constexpr int KM = 34, KNZ = 90, KNC = 68;

template <bool WITH_DERIV> struct KinoWsT {
  static constexpr int XS = WITH_DERIV ? NV * KNZ : 8, TOPS = WITH_DERIV ? 2 * NV * 6 : 8, BCS = WITH_DERIV ? NB * 36 : 8;
  static constexpr int CJ1 = WITH_DERIV ? 6 * FN : 8, CJ2 = WITH_DERIV ? 2 * 6 * NV : 8, M6 = WITH_DERIV ? 36 : 1, ZS = WITH_DERIV ? KNZ : 8;
  static constexpr int CV = WITH_DERIV ? 12 * FN : 8, JCD = WITH_DERIV ? 6 * KNZ : 8, HQ = WITH_DERIV ? 6 * NV : 8;
  double x[NQ + NV], u[KM], xn[NQ + NV];
  double kn[sizeof(mpc_knot_t) / 8];
  double oM[NB * 12], S[NV * 6], v[NB * 6], a[NB * 6], I[NB * 10], Ic[NB * 10];
  double hb[NB * 6], hsub[NB * 6], f[NB * 6], Fsub[NB * 6];
  union {
    double Bc[BCS];
    struct { double Jcent[CJ1], Jpose[CJ2]; } cj;
  };
  double U[NV * 6];
  struct {
    double P1[M6], P2[M6], E6[M6], T6[M6], Jlg[M6], Jrg[M6], AdD[M6], AdDi[M6], Jd[M6], Ade[M6];
    double lxu[ZS], g[ZS], hval[KNC], vpl[KNC], dbr[KNC], rowtmp[KNC];
  } late;
  double acc[NV];
  double ofoot[24], Jf[2 * 6 * NV];
  double Ag[6 * NV], Abi[36], hd[6], Fg0[6], vl[12];
  double X[XS];       // [da/dx | da/du]  (NV x KNZ)
  double top[TOPS];   // dF_o/dq_j, dF_o/dv_j
  double hdq[HQ];     // d hdot'/dq (6 x NV)
  double Jcd[JCD];    // momentum-derivative residual Jacobian, dense rows over z
  double Cvel[CV];    // zero-frame-velocity constraint rows [dq | dv] for both feet (12 x 56)
  double rcent[6], rpose[12], Jlp[2 * M6];
  double estate[FN], Jls[M6];
  double dx[FN], xnext[NQ + NV], lgap[6], eexp[12], Dgap[12], Dl[36];
  double lpl[FN], fbr[FN];
  double com[3], scal[SC_COUNT], part[32];
  int32_t active[2], ctype[KNC], isact[KNC], act_idx[KNC], nca;
};

// constraint row layout: [0,22) joint box; contact f: base = 22 + 23 f: 17 cone rows then 6 velocity rows
HD double kino_c_entry(const DevModel &m, const double *Cvel, int r, int z) {
  if (r < 22) return (z == 6 + r) ? -1.0 : 0.0;
  int f = (r - 22) / 23, rr = (r - 22) % 23;
  if (rr < 17) { int k = z - FN - 6 * f; return (k >= 0 && k < 6) ? m.Acone[6 * rr + k] : 0.0; }
  return (z < FN) ? Cvel[(6 * f + rr - 17) * FN + z] : 0.0;
}

template <bool DERIV, bool ROLL = false> HD void eval_kino_knot(const DevModel &m, const KnotIO &io, KinoWsT<DERIV> &w) {
  const mpc_robot_t &rb = m.rb;
  const mpc_config_t &cfg = m.cfg;
  const double dt = cfg.dt;
  PAR_FOR(i, NQ + NV) { w.x[i] = io.x[i]; w.xn[i] = io.xn[i]; }
  PAR_FOR(i, KM) w.u[i] = io.u[i];
  PAR_FOR(i, (int)(sizeof(mpc_knot_t) / 8)) w.kn[i] = reinterpret_cast<const double *>(io.kn)[i];
  SYNC();
  const mpc_knot_t &kn = *reinterpret_cast<const mpc_knot_t *>(w.kn);
  ONE_THREAD { w.active[0] = kn.cs[0] != 0.0; w.active[1] = kn.cs[1] != 0.0; }
  mb_kinematics(m, w);
  const double a0[6] = {-rb.gravity[0], -rb.gravity[1], -rb.gravity[2], 0, 0, 0};
  mb_bias_forces<true>(m, w, a0, w.u + 12); // qdd = [0; a_j]
  mb_centroidal_map(w, w.Ag);
  SYNC();
  PAR_FOR(task, 64) {
    if (task == 0) { // total bias force at the CoM
      double F[6] = {0, 0, 0, 0, 0, 0}, c[3];
      for (int b = 0; b < NB; b++) for (int i = 0; i < 6; i++) F[i] += w.f[6 * b + i];
      cross3(w.com, F, c);
      for (int i = 0; i < 3; i++) { w.Fg0[i] = F[i]; w.Fg0[3 + i] = F[3 + i] - c[i]; }
    } else if (task == 32) { // contact wrench resultant hdot' and inverse of A_b
      double hl[3] = {0, 0, 0}, ha[3] = {0, 0, 0};
      for (int f = 0; f < 2; f++) {
        if (!w.active[f]) continue;
        const double *fo = w.u + 6 * f;
        double d[3] = {w.ofoot[12 * f + 9] - w.com[0], w.ofoot[12 * f + 10] - w.com[1], w.ofoot[12 * f + 11] - w.com[2]}, c[3];
        cross3(d, fo, c);
        for (int i = 0; i < 3; i++) { hl[i] += fo[i]; ha[i] += c[i] + fo[3 + i]; }
      }
      for (int i = 0; i < 3; i++) { w.hd[i] = hl[i]; w.hd[3 + i] = ha[i]; }
      double Ab[36];
      for (int i = 0; i < 6; i++) for (int j = 0; j < 6; j++) Ab[6 * i + j] = w.Ag[i * NV + j];
      inv6(Ab, w.Abi);
    }
  }
  SYNC();
  PAR_FOR(i, NV) {
    if (i < 6) { double s = 0; for (int k = 0; k < 6; k++) s += w.Abi[6 * i + k] * (w.hd[k] - w.Fg0[k]); w.acc[i] = s; }
    else w.acc[i] = w.u[12 + i - 6];
  }
  PAR_FOR(f, 2) { // LOCAL sole velocities (zero-velocity constraint values)
    double vl[6];
    mb_sole_motion<false>(m, w, f, a0, vl);
    for (int r = 0; r < 6; r++) w.vl[6 * f + r] = vl[r];
  }
  SYNC();
  PAR_FOR(i, NV) { io.xdot[i] = w.x[NQ + i]; io.xdot[NV + i] = w.acc[i]; }
  PAR_FOR(i, 12) io.lamc[i] = w.active[i / 6] ? w.u[i] : 0.0;

  if (DERIV) {
    // full accelerations: the base acceleration moves every body
    PAR_FOR(e, NB * 6) {
      int c = e % 6;
      double s = w.a[e];
      for (int j = 0; j < 6; j++) s += w.S[6 * j + c] * w.acc[j];
      w.a[e] = s;
    }
    PAR_FOR(e, NV * KNZ) w.X[e] = 0.0;
    SYNC();
    PAR_FOR(b, NB) mb_body_force(w, b, w.a + 6 * b, w.f + 6 * b);
    SYNC();
    mb_subtree_sum<6>(m, w.f, w.Fsub);
    mb_composite_B(m, w);
    PAR_FOR(e, 2 * NV) { // top vectors: d F_o/d q_j (kind 0), d F_o/d v_j (kind 1)
      const int kind = e / NV, j = e % NV, J = body_of_dof(j);
      double g[6], t1[6];
      mb_force_column(m, w, kind, j, J, a0, g);
      if (kind == 0) { cross_mf(w.S + 6 * j, w.Fsub + 6 * J, t1); for (int i = 0; i < 6; i++) w.top[6 * j + i] = t1[i] - g[i]; }
      else for (int i = 0; i < 6; i++) w.top[6 * (NV + j) + i] = g[i];
    }
    PAR_FOR(j, NV) { // d hdot'/dq_j (angular rows): sum_i (dp_i/dq_j - dc/dq_j) x f_i
      const double im_ = rcp_(w.Ic[0]);
      double dc[3] = {w.U[6 * j] * im_, w.U[6 * j + 1] * im_, w.U[6 * j + 2] * im_}, acc3[3] = {0, 0, 0};
      for (int f = 0; f < 2; f++) {
        if (!w.active[f]) continue;
        double dp[3] = {0, 0, 0};
        if (m.ancdof_mask[rb.foot_body[f]] >> j & 1) {
          cross3(w.S + 6 * j + 3, w.ofoot + 12 * f + 9, dp);
          for (int i = 0; i < 3; i++) dp[i] += w.S[6 * j + i];
        }
        double d[3] = {dp[0] - dc[0], dp[1] - dc[1], dp[2] - dc[2]}, c[3];
        cross3(d, w.u + 6 * f, c);
        for (int i = 0; i < 3; i++) acc3[i] += c[i];
      }
      for (int r = 0; r < 3; r++) { w.hdq[r * NV + j] = 0.0; w.hdq[(3 + r) * NV + j] = acc3[r]; }
    }
    PAR_FOR(e, 2 * NV) { // zero-velocity constraint rows for both feet
      int f = e / NV, j = e % NV, fb = rb.foot_body[f];
      double wl[6] = {0, 0, 0, 0, 0, 0};
      const bool on = (m.ancdof_mask[fb] >> j & 1) != 0;
      if (on) {
        int J = body_of_dof(j), pJ = rb.parent[J];
        double vp[6] = {0, 0, 0, 0, 0, 0}, wj[6];
        if (pJ >= 0) for (int i = 0; i < 6; i++) vp[i] = w.v[6 * pJ + i];
        cross_mm(w.S + 6 * j, vp, wj);
        se3_actinv_motion(w.ofoot + 12 * f, wj, wl);
      }
      for (int r = 0; r < 6; r++) { w.Cvel[(6 * f + r) * FN + j] = -wl[r]; w.Cvel[(6 * f + r) * FN + NV + j] = on ? w.Jf[(6 * f + r) * NV + j] : 0.0; }
    }
    SYNC();
    PAR_FOR(z, KNZ) { // base-acceleration Jacobian column z: A_b da_b = d hdot' - d F_g|_a - A_j da_j
      double rhs[6] = {0, 0, 0, 0, 0, 0};
      const double *Fo = w.Fsub; // total force about the origin
      if (z < NV) {
        const double *tq = w.top + 6 * z;
        const double im_ = rcp_(w.Ic[0]);
        double dc[3] = {w.U[6 * z] * im_, w.U[6 * z + 1] * im_, w.U[6 * z + 2] * im_}, c1[3], c2[3];
        cross3(dc, Fo, c1); cross3(w.com, tq, c2);
        for (int r = 0; r < 3; r++) { rhs[r] = w.hdq[r * NV + z] - tq[r]; rhs[3 + r] = w.hdq[(3 + r) * NV + z] - (tq[3 + r] - c1[r] - c2[r]); }
      } else if (z < FN) {
        const double *tv = w.top + 6 * (NV + z - NV);
        double c2[3];
        cross3(w.com, tv, c2);
        for (int r = 0; r < 3; r++) { rhs[r] = -tv[r]; rhs[3 + r] = -(tv[3 + r] - c2[r]); }
      } else {
        int jj = z - FN;
        if (jj < 12) {
          int f = jj / 6, k = jj % 6;
          if (w.active[f]) {
            if (k < 3) {
              double d[3] = {w.ofoot[12 * f + 9] - w.com[0], w.ofoot[12 * f + 10] - w.com[1], w.ofoot[12 * f + 11] - w.com[2]}, e3[3] = {0, 0, 0}, c[3];
              e3[k] = 1.0;
              cross3(d, e3, c);
              rhs[k] = 1.0;
              for (int r = 0; r < 3; r++) rhs[3 + r] = c[r];
            } else rhs[k] = 1.0;
          }
        } else for (int r = 0; r < 6; r++) rhs[r] = -w.Ag[r * NV + 6 + (jj - 12)];
      }
      for (int i = 0; i < 6; i++) { double s = 0; for (int k = 0; k < 6; k++) s += w.Abi[6 * i + k] * rhs[k]; w.X[i * KNZ + z] = s; }
      if (z >= FN + 12) w.X[(6 + z - FN - 12) * KNZ + z] = 1.0;
      // momentum-derivative residual Jacobian rows over z
      for (int r = 0; r < 6; r++) {
        double val = 0;
        if (z < NV) val = w.hdq[r * NV + z];
        else if (z >= FN && z < FN + 12) {
          int f = (z - FN) / 6, k = (z - FN) % 6;
          if (w.active[f]) {
            if (k < 3) {
              if (r == k) val = 1.0;
              else if (r >= 3) {
                double d[3] = {w.ofoot[12 * f + 9] - w.com[0], w.ofoot[12 * f + 10] - w.com[1], w.ofoot[12 * f + 11] - w.com[2]}, e3[3] = {0, 0, 0}, c[3];
                e3[k] = 1.0; cross3(d, e3, c); val = c[r - 3];
              }
            } else if (r == k) val = 1.0;
          }
        }
        w.Jcd[r * KNZ + z] = val;
      }
    }
    SYNC();
  }

  // ---- semi-implicit Euler + gap + cost terms
  PAR_FOR(i, NV) { double dv = dt * w.acc[i]; w.dx[NV + i] = dv; w.dx[i] = dt * (w.x[NQ + i] + dv); }
  SYNC();
  mb_cost_terms<KinoWsT<DERIV>, ROLL>(m, w, kn.lf_ref, kn.rf_ref, DERIV, io.gap, io.slack);
  if (ROLL) PAR_FOR(i, NQ + NV) io.xn_out[i] = w.xn[i];

  // ---- constraint values, multiplier estimates, activity
  // every thread accumulates the merit pieces of the rows / coordinates it owns; one group-wide reduction at the end
  double acc_cost = 0.0, acc_pen = 0.0, acc_prim = 0.0, acc_inner = 0.0;
  PAR_FOR(r, KNC) {
    int type = -1; double hv = 0, lo = 0, hi = 0;
    if (r < 22) { type = 2; hv = -w.x[7 + r]; lo = -rb.q_hi[r]; hi = -rb.q_lo[r]; }
    else {
      int f = (r - 22) / 23, rr = (r - 22) % 23;
      if (w.active[f]) {
        if (rr < 17) { type = 1; for (int k = 0; k < 6; k++) hv += m.Acone[6 * rr + k] * w.u[6 * f + k]; }
        else { type = 0; hv = w.vl[6 * f + rr - 17]; }
      }
    }
    mb_row_epilogue(w, io, r, type, hv, lo, hi, io.v, io.v_prev, acc_pen, acc_prim, acc_inner);
  }
  mb_dynamics_rows(m, w, io, io.lam_n, io.lam_n_prev, acc_cost, acc_pen, acc_prim, acc_inner);
  PAR_FOR(i, KM) { const double e = w.u[i] - kn.u_ref[i]; acc_cost += 0.5 * cfg.wu[i] * e * e; }
  PAR_FOR(i, 6) {
    const double rcd = w.hd[i] + (i < 3 ? m.total_mass * rb.gravity[i] : 0.0);
    acc_cost += 0.5 * (cfg.w_cent[i] * w.rcent[i] * w.rcent[i] + kn.w_lf[i] * w.rpose[i] * w.rpose[i] + kn.w_rf[i] * w.rpose[6 + i] * w.rpose[6 + i] +
                       cfg.w_centder[i] * rcd * rcd);
  }
  mb_merit_finish<KNC>(w, acc_cost, acc_pen, acc_prim, acc_inner);
  if (!DERIV) { PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i]; return; }

  // ---- LQ blocks to HBM
  mb_store_rows<KNC>(w, io);
  PAR_FOR(z, KNZ) {
    const double acc = mb_ab_column<KNZ>(w, io, z, w.X + z, KNZ, dt, io.lam_n);
    double lz = mb_cost_grad(w, cfg.wx, cfg.w_cent, kn.w_lf, kn.w_rf, z < FN ? z : FN);
    if (z >= FN) lz = cfg.wu[z - FN] * (w.u[z - FN] - kn.u_ref[z - FN]);
    for (int r = 0; r < 6; r++) {
      double rcd = w.hd[r] + (r < 3 ? m.total_mass * rb.gravity[r] : 0.0);
      lz += cfg.w_centder[r] * w.Jcd[r * KNZ + z] * rcd;
    }
    w.late.lxu[z] = lz; io.lxu[z] = lz;
    double gz = lz + acc;
    for (int r = 0; r < KNC; r++) {
      double vr = io.v[r];
      if (vr == 0.0 || w.ctype[r] < 0) continue;
      gz += kino_c_entry(m, w.Cvel, r, z) * vr;
    }
    if (z < FN) { if (io.k == 0) gz += io.lam_k[z]; else if (z >= 6) gz -= io.lam_k[z]; }
    w.late.g[z] = gz; io.g[z] = gz;
  }
  mb_gE_next(w, io, io.lam_n);
  mb_gn_hessian<KNZ>(w, io, cfg, kn, [&](auto &rank1) { // momentum-derivative cost rows
    for (int r = 0; r < 6; r++) if (cfg.w_centder[r] != 0.0) rank1(w.Jcd + r * KNZ, KNZ, cfg.w_centder[r]);
  });
  PAR_FOR(e, w.nca * KNZ) {
    int ai = e / KNZ, z = e % KNZ;
    io.CDact[e] = kino_c_entry(m, w.Cvel, w.act_idx[ai], z);
  }
  mb_dual_scal<KNZ>(w, io);
}

} // namespace mpcdev
