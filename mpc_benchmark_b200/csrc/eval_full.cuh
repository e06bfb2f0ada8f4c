// Per-knot evaluation of the FULL-DYNAMICS Talos stage: one CTA per (instance, knot).
//
// Replaces, for one knot, what the reference obtains from five independent Aligator objects that each re-run
// pinocchio::constraintDynamics + computeConstraintDynamicsDerivatives (SURVEY finding 7):
//   MultibodyConstraintFwdDynamics + IntegratorSemiImplEuler      fulldynamic_talos.py:100-111
//   ContactForceResidual x2, MultibodyWrenchConeResidual x2        fulldynamic_talos.py:188-201, 211-225
//   QuadraticState/Control cost, CentroidalMomentumResidual, FramePlacementResidual x2   :160-185
//   torque / joint-limit boxes                                     :206-209
// Here (a, lambda, da, dlambda) are computed ONCE in shared memory and every cost/constraint reads them.
//
// World-frame formulation (all spatial quantities at the world origin, world axes): subtree accumulations are
// plain sums.  Derivative columns use composite quantities (DESIGN.md "RBD derivatives"):
//   dtau_i/dq_j = -S_i.(Ic_m c_j + Bc_m w_j),  m = body(i) in subtree(body(j));  ancestors: S_i.(s_j x* F_J - g_J)
//   dtau_i/dv_j = +S_i.(Ic_m c'_j + Bc_m s_j)
#pragma once
#include <cstddef>
#include "dmma.cuh"
#include "eval_mb.cuh"

namespace mpcdev {

// optional per-phase cycle counters of the evaluation kernel (-DMPC_PHASE_TIMING builds; knot 1 of instance 0)
#if defined(MPC_PHASE_TIMING) && !defined(MPC_HOST_EMU)
#define EPH_DECL long long eph_last = clock64(); long long eph_acc[16] = {0}
#define EPH(i) do { SYNC(); if (threadIdx.x == 0) { long long t_ = clock64(); eph_acc[i] += t_ - eph_last; eph_last = t_; } } while (0)
#define EPH_DUMP(ptr) do { if (threadIdx.x == 0 && (ptr)) for (int i_ = 0; i_ < 16; i_++) (ptr)[i_] = (double)eph_acc[i_]; } while (0)
#else
#define EPH_DECL
#define EPH(i)
#define EPH_DUMP(ptr)
#endif


constexpr int FM = 22, FNZ = 78, FNC = 78;

template <bool WITH_DERIV> struct FullWsT {
  static constexpr int TOPS = WITH_DERIV ? 2 * NV * 6 : 8, BCS = WITH_DERIV ? NB * 36 : 8, HROWS = WITH_DERIV ? 40 : 1;
  static constexpr int CJ1 = WITH_DERIV ? 6 * FN : 8, CJ2 = WITH_DERIV ? 2 * 6 * NV : 8, M6 = WITH_DERIV ? 36 : 1, ZS = WITH_DERIV ? FNZ : 8;
  double x[NQ + NV], u[FM], xn[NQ + NV];
  double kn[sizeof(mpc_knot_t) / 8];
  double oM[NB * 12], S[NV * 6], v[NB * 6], a[NB * 6], I[NB * 10], Ic[NB * 10];
  double hb[NB * 6], hsub[NB * 6], f[NB * 6], Fsub[NB * 6];
  union { // Bc is dead once the derivative columns are built; the cost Jacobians are built afterwards
    double Bc[BCS];
    struct { double Jcent[CJ1], Jpose[CJ2]; } cj;
  };
  double top[TOPS]; // directly behind Bc: [Bc | top] doubles as the scratch of the explicit mass-matrix inverse (both are free until then)
  double U[NV * 6];
  union { // the mass-matrix factor is dead after X = M^-1 R1; the output-phase vectors live afterwards
    double M[NV * NV];
    struct {
      double P1[M6], P2[M6], E6[M6], T6[M6], Jlg[M6], Jrg[M6], AdD[M6], AdDi[M6], Jd[M6], Ade[M6];
      double lxu[ZS], g[ZS], hval[FNC], vpl[FNC], dbr[FNC], rowtmp[FNC];
    } late;
  };
  double acc[NV];
  double ofoot[24], Jf[2 * 6 * NV];
  double vc[12], gam[12], astar[12], c1Mc2[24], JlAd[2 * M6], lam[12], lgc[12];
  union { // the contact-solve scratch is dead once da/dlam are formed; the multipliers are staged into it afterwards
    struct { double Y[NV * 13], G[144], rhs[12], dinvM[4 * 64], dinvG[2 * 64]; };
    struct { double mv[FNC], mvp[FNC], mln[FN], mlnp[FN], mlk[FN]; }; // v, v_prev, lam_{k+1}, its estimate, lam_k
  };
  double rcent[6], rpose[12], Jlp[2 * M6];
  double estate[FN], Jls[M6];
  double dx[FN], xnext[NQ + NV], lgap[6], eexp[12], Dgap[12], Dl[36];
  double lpl[FN], fbr[FN];
  double com[3], scal[SC_COUNT], part[32];
  // Gauss-Newton Hessian as ONE tensor-core product H = sum_k w_k J_k' J_k: the weighted residual-Jacobian rows stay where they are
  // (dlam/dz rows in the global scratch, Jcent, Jpose, Jls in shared memory) and are addressed through this table
  double hrow_w[HROWS];
  int32_t hrow_len[HROWS];
  int32_t act[2], nact, sidx[2], ctype[FNC], isact[FNC], act_idx[FNC], nca;
};
using FullWs = FullWsT<true>;
static_assert(offsetof(FullWs, top) == offsetof(FullWs, Bc) + sizeof(double) * FullWs::BCS, "[Bc | top] must be contiguous");
static_assert(FullWs::BCS + FullWs::TOPS >= NV * NV + 3 * 64, "mass-matrix inverse scratch does not fit in [Bc | top]");

// constraint row layout: [0,22) torque box; [22,44) joint box; contact f: base = 44 + 17 f, wrench-cone rows over dlam/dz (DL,
// rows of the active contacts in sidx order)
HD double full_c_entry(const DevModel &m, const double *DL, const int32_t *sidx, int r, int z) {
  if (r < 22) return (z == FN + r) ? 1.0 : 0.0;
  if (r < 44) return (z == 6 + r - 22) ? -1.0 : 0.0;
  int f = (r - 44) / 17, rr = (r - 44) % 17; const double *Dl = DL + 6 * sidx[f] * FNZ; double c = 0; for (int k = 0; k < 6; k++) c += m.Acone[6 * rr + k] * Dl[k * FNZ + z];
  return c;
}

// ------------------------------------------------------------------ running knot
template <bool DERIV, bool ROLL = false> HD void eval_full_knot(const DevModel &m, const KnotIO &io, FullWsT<DERIV> &w) {
  EPH_DECL;
  const mpc_robot_t &rb = m.rb;
  const mpc_config_t &cfg = m.cfg;
  const double dt = cfg.dt;
  PAR_FOR(i, NQ + NV) { w.x[i] = io.x[i]; w.xn[i] = io.xn[i]; }
  PAR_FOR(i, FM) w.u[i] = io.u[i];
  PAR_FOR(i, (int)(sizeof(mpc_knot_t) / 8)) w.kn[i] = reinterpret_cast<const double *>(io.kn)[i];
  SYNC();
  const mpc_knot_t &kn = *reinterpret_cast<const mpc_knot_t *>(w.kn);
  ONE_THREAD {
    bool l = kn.cs[0] != 0.0, r = kn.cs[1] != 0.0;
    if (!l && !r) l = r = true; // fulldynamic_talos.py:108-110: no-contact falls through to both contacts
    w.nact = 0; w.sidx[0] = w.sidx[1] = -1;
    if (l) { w.sidx[0] = w.nact; w.act[w.nact++] = 0; }
    if (r) { w.sidx[1] = w.nact; w.act[w.nact++] = 1; }
  }
  EPH(0);
  mb_kinematics(m, w);
  EPH(1);
  const int nact = w.nact, nk = 6 * nact;
  // derivative kernel: explicit mass-matrix inverse, raw right-hand sides [tau - b | J'] (NV x 13) in Yr; values kernel: solve in place in Y
  // [L^-1 (NV x NV) | 64 doubles of scratch per warp] in the free [Bc | top] block; the raw right-hand sides go to the global scratch
  double *Ls = reinterpret_cast<double *>(&w) + offsetof(FullWsT<DERIV>, Bc) / sizeof(double); // spans [Bc | top]
  double *X = io.scratch, *DL = io.scratch + NV * FNZ; // derivative pass only (null otherwise)
  double *Yr = DERIV ? DL : w.Y;
  const double a0[6] = {-rb.gravity[0], -rb.gravity[1], -rb.gravity[2], 0, 0, 0};
  mb_bias_forces(m, w, a0); // qdd = 0
  SYNC();
  mb_subtree_sum<6>(m, w.f, w.Fsub);
  mb_crba(m, w, w.M);
  PAR_FOR(c, nact) { // contact kinematics + Baumgarte terms
    const int f = w.act[c];
    mb_sole_motion(m, w, f, a0, w.vc + 6 * c, w.gam + 6 * c);
    se3_inv_mul(w.ofoot + 12 * f, cfg.contact_place[f], w.c1Mc2 + 12 * c);
    double lg[6];
    log6(w.c1Mc2 + 12 * c, lg);
    for (int r = 0; r < 6; r++) w.astar[6 * c + r] = cfg.kp[r] * lg[r] - cfg.kd[r] * w.vc[6 * c + r];
    for (int r = 0; r < 6; r++) w.lgc[6 * c + r] = lg[r];
  }
  SYNC();
  PAR_FOR(j, NV) { // b = S^T Fsub ; rhs column 0 = tau - b ; columns 1.. = J^T
    double bj = dot6(w.S + 6 * j, w.Fsub + 6 * body_of_dof(j));
    Yr[j * 13] = (j >= 6 ? w.u[j - 6] : 0.0) - bj;
    for (int r = 0; r < nk; r++) Yr[j * 13 + 1 + r] = w.Jf[(6 * w.act[r / 6] + r % 6) * NV + j];
  }
  SYNC();
  EPH(2);
  if (DERIV) {
    // M <- M^-1 explicitly (one Cholesky + inverse factor + product): every solve with the mass matrix is then a plain matrix
    // product without barriers (Y here, the 78 right-hand sides of the tangent later).  The values-only kernel has just the
    // 13 columns of Y and keeps the factor + blocked triangular solves.
    spd_inverse_blocked(w.M, NV, NV, w.dinvM, Ls);
    EPH(3);
    PAR_FOR(e, NV * (1 + nk)) {
      const int i = e / (1 + nk), c = e % (1 + nk);
      double s = 0;
      for (int k = 0; k < NV; k++) s += w.M[i * NV + k] * Yr[k * 13 + c];
      w.Y[i * 13 + c] = s;
    }
    SYNC();
  } else {
    chol_blocked(w.M, NV, NV, w.dinvM);
    EPH(3);
    trsm_blocked(w.M, NV, NV, w.dinvM, w.Y, 1 + nk, 13);
  }
  PAR_FOR(e, nk * (nk + 1)) {
    int r = e / (nk + 1), c = e % (nk + 1);
    const double *Jr = w.Jf + (6 * w.act[r / 6] + r % 6) * NV;
    double s = 0;
    for (int i = 0; i < NV; i++) s += Jr[i] * w.Y[i * 13 + c];
    if (c == 0) w.rhs[r] = w.astar[r] - w.gam[r] - s;
    else w.G[r * 12 + c - 1] = s + ((r == c - 1) ? cfg.mu_contact : 0.0);
  }
  SYNC();
  if (DERIV) { // G <- G^-1 as well (6 x 6 or 12 x 12): lambda now, the 78 columns of dlambda later, all without triangular solves
    spd_inverse_blocked(w.G, nk, 12, w.dinvG, w.top); // `top` is free until the tangent columns are built
    PAR_FOR(r, nk) { double s = 0; for (int c = 0; c < nk; c++) s += w.G[r * 12 + c] * w.rhs[c]; w.astar[r] = s; }
    SYNC();
    PAR_FOR(r, nk) w.rhs[r] = w.astar[r];
    SYNC();
  } else {
    chol_blocked(w.G, nk, 12, w.dinvG);
    trsm_blocked(w.G, nk, 12, w.dinvG, w.rhs, 1, 1);
  }
  PAR_FOR(i, NV) {
    double s = w.Y[i * 13];
    for (int r = 0; r < nk; r++) s += w.Y[i * 13 + 1 + r] * w.rhs[r];
    w.acc[i] = s;
  }
  PAR_FOR(i, 12) { int f = i / 6; w.lam[i] = (w.sidx[f] >= 0) ? w.rhs[6 * w.sidx[f] + i % 6] : 0.0; }
  SYNC();
  PAR_FOR(i, NV) { io.xdot[i] = w.x[NQ + i]; io.xdot[NV + i] = w.acc[i]; }
  PAR_FOR(i, 12) io.lamc[i] = w.lam[i];

  EPH(4);
  if (DERIV) {
    // ---- inverse-dynamics tangent at (q, v, a) with the contact wrenches as external forces
    PAR_FOR(c, nact) { // JlAd = Jlog6(c1Mc2) * Ad(c2Mc1)
      double Jl[36], Ad[36], inv[12], id[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
      Jlog6_from_log(w.lgc + 6 * c, Jl);
      se3_inv_mul(w.c1Mc2 + 12 * c, id, inv);
      se3_action_matrix(inv, Ad);
      mat6_mul(Jl, Ad, w.JlAd + 36 * c);
    }
    PAR_FOR(e, NB * 6) { // full accelerations
      int b = e / 6, c = e % 6;
      uint32_t mask = m.ancdof_mask[b];
      double s = w.a[e];
      for (int j = 0; j < NV; j++) if (mask >> j & 1) s += w.S[6 * j + c] * w.acc[j];
      w.a[e] = s;
    }
    SYNC();
    PAR_FOR(b, NB) {
      double fb[6];
      mb_body_force(w, b, w.a + 6 * b, fb);
      for (int c = 0; c < nact; c++)
        if (rb.foot_body[w.act[c]] == b) {
          double fw[6];
          se3_act_force(w.ofoot + 12 * w.act[c], w.rhs + 6 * c, fw);
          for (int i = 0; i < 6; i++) fb[i] -= fw[i];
        }
      for (int i = 0; i < 6; i++) w.f[6 * b + i] = fb[i];
    }
    PAR_FOR(e, NV * FNZ) X[e] = 0.0;
    PAR_FOR(e, 12 * FNZ) DL[e] = 0.0;
    SYNC();
    mb_subtree_sum<6>(m, w.f, w.Fsub);
    EPH(5);
    mb_composite_B(m, w);
    EPH(6);
    PAR_FOR(e, 2 * m.npairs) {
      const int kind = e / m.npairs, p = e % m.npairs, j = m.pair_j[p], mb = m.pair_m[p], J = body_of_dof(j);
      double g[6], t1[6];
      mb_force_column(m, w, kind, j, mb, a0, g);
      int i0 = first_dof(mb), nd = ndof_of(mb);
      for (int d = 0; d < nd; d++) {
        double val = dot6(w.S + 6 * (i0 + d), g);
        X[(i0 + d) * FNZ + kind * NV + j] = kind == 0 ? -val : val;
      }
      if (mb == J) {
        if (kind == 0) { cross_mf(w.S + 6 * j, w.Fsub + 6 * J, t1); for (int i = 0; i < 6; i++) w.top[6 * j + i] = t1[i] - g[i]; }
        else for (int i = 0; i < 6; i++) w.top[6 * (NV + j) + i] = g[i];
      }
    }
    PAR_FOR(e, NJ) X[(6 + e) * FNZ + 2 * NV + e] = -1.0; // R1 for u: -B_act
    // R2 = d(alpha - astar)/d(q,v) for the active contacts
    PAR_FOR(e, nact * NV) {
      int c = e / NV, j = e % NV, f = w.act[c], fb = rb.foot_body[f];
      if (!(m.ancdof_mask[fb] >> j & 1)) continue;
      int J = body_of_dof(j), pJ = rb.parent[J];
      const double *s = w.S + 6 * j, *of = w.ofoot + 12 * f;
      double vp[6] = {0, 0, 0, 0, 0, 0}, ap[6] = {0, 0, 0, 0, 0, 0};
      if (pJ >= 0) for (int i = 0; i < 6; i++) { vp[i] = w.v[6 * pJ + i]; ap[i] = w.a[6 * pJ + i] - a0[i]; }
      double wj[6], cj[6], t1[6], t2[6], dq_[6], dv_[6], wl[6], Jc[6], dlog[6];
      cross_mm(s, vp, wj);
      cross_mm(s, ap, cj);
      cross_mm(wj, vp, t1);
      cross_mm(wj, w.v + 6 * fb, t2);
      for (int i = 0; i < 6; i++) t1[i] = cj[i] - t1[i] + t2[i];
      se3_actinv_motion(of, t1, dq_);
      for (int i = 0; i < 6; i++) t2[i] = w.v[6 * fb + i] - w.v[6 * J + i] - vp[i];
      cross_mm(s, t2, t1);
      se3_actinv_motion(of, t1, dv_);
      se3_actinv_motion(of, wj, wl);
      for (int r = 0; r < 6; r++) Jc[r] = w.Jf[(6 * f + r) * NV + j];
      mat6_vec(w.JlAd + 36 * c, Jc, dlog);
      for (int r = 0; r < 6; r++) {
        DL[(6 * c + r) * FNZ + j] = -dq_[r] - (-cfg.kp[r] * dlog[r] + cfg.kd[r] * wl[r]);
        DL[(6 * c + r) * FNZ + NV + j] = dv_[r] + cfg.kd[r] * Jc[r];
      }
    }
    SYNC();
    PAR_FOR(e, m.nanc) {
      int i = m.anc_i[e], j = m.anc_j[e];
      X[i * FNZ + j] = dot6(w.S + 6 * i, w.top + 6 * j);
      X[i * FNZ + NV + j] = dot6(w.S + 6 * i, w.top + 6 * (NV + j));
    }
    SYNC();
    EPH(7);
#ifdef MPC_HOST_EMU
    PAR_FOR(z, FNZ) { // X = M^-1 R1, one column per thread (column in registers, written back in place)
      double col[NV];
#pragma unroll
      for (int k = 0; k < NV; k++) col[k] = X[k * FNZ + z];
      for (int i = 0; i < NV; i++) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < NV; k++) s += w.M[i * NV + k] * col[k];
        X[i * FNZ + z] = s;
      }
    }
    SYNC();
    EPH(8);
    PAR_FOR(z, FNZ) { // per column of z: dlam = G^-1 (J X - DL), then da/dz = -X + Y dlam (X column and dlam in registers)
      double xc[NV], t[12], dl[12];
#pragma unroll
      for (int i = 0; i < NV; i++) xc[i] = X[i * FNZ + z];
#pragma unroll
      for (int r = 0; r < 12; r++) {
        t[r] = 0.0;
        if (r < nk) {
          const double *Jr = w.Jf + (6 * w.act[r / 6] + r % 6) * NV;
          double s = -DL[r * FNZ + z];
#pragma unroll
          for (int i = 0; i < NV; i++) s += Jr[i] * xc[i];
          t[r] = s;
        }
      }
#pragma unroll
      for (int r = 0; r < 12; r++) {
        dl[r] = 0.0;
        if (r < nk) {
          double s = 0;
#pragma unroll
          for (int c = 0; c < 12; c++) if (c < nk) s += w.G[r * 12 + c] * t[c];
          dl[r] = s;
          DL[r * FNZ + z] = s;
        }
      }
#pragma unroll
      for (int i = 0; i < NV; i++) {
        double s = -xc[i];
#pragma unroll
        for (int r = 0; r < 12; r++) if (r < nk) s += w.Y[i * 13 + 1 + r] * dl[r];
        X[i * FNZ + z] = s; // da/dz
      }
    }
    SYNC();
#else
    { // Tangent of the constrained dynamics on the FP64 tensor pipe, one 8-column tile of z per warp, no block barrier inside:
      //   X <- M^-1 R1;  T = J X - DL;  dlam = G^-1 T (-> DL);  da/dz = -X + Y dlam (-> X)
      // Accumulator tiles that feed the next product as its K operand are transposed through a per-warp slice of the dead
      // [Bc | top] block (32 x 8 for X, 16 x 8 for T / dlam); the right-hand sides of the next tile are fetched from the
      // L2-resident scratch while the current one is being processed.
      const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
      double *Xs = Ls + 384 * WARP_ID, *Ts = Xs + 256;
      static_assert(FullWsT<DERIV>::BCS + FullWsT<DERIV>::TOPS >= 3 * 384 || !DERIV, "per-warp transpose tiles do not fit in [Bc | top]");
      const double *Jb = w.Jf + 6 * w.act[0] * NV; // rows of the active contacts are contiguous in Jf
      const int ks2 = (nk + 3) / 4;
      constexpr int NCT = (FNZ + 7) / 8;
      double bx[7], bnext[7], xn[4][2];
      { const int cb = 8 * WARP_ID + g;
#pragma unroll
        for (int s_ = 0; s_ < 7; s_++) bnext[s_] = (WARP_ID < NCT && cb < FNZ) ? X[(4 * s_ + t) * FNZ + cb] : 0.0; }
      for (int ct = WARP_ID; ct < NCT; ct += NWARPS) {
        const int cc = 8 * ct + 2 * t;
        const bool okc = cc < FNZ;
#pragma unroll
        for (int s_ = 0; s_ < 7; s_++) bx[s_] = bnext[s_];
        { const int cbn = 8 * (ct + NWARPS) + g; // right-hand sides of this warp's next tile
#pragma unroll
          for (int s_ = 0; s_ < 7; s_++) bnext[s_] = (ct + NWARPS < NCT && cbn < FNZ) ? X[(4 * s_ + t) * FNZ + cbn] : 0.0; }
#pragma unroll
        for (int ti = 0; ti < 4; ti++) {
          const int row = 8 * ti + g;
          double c0 = 0.0, c1 = 0.0;
#pragma unroll
          for (int s_ = 0; s_ < 7; s_++) dmma_8x8x4(c0, c1, (row < NV) ? w.M[(4 * s_ + t) * NV + row] : 0.0, bx[s_]);
          xn[ti][0] = c0; xn[ti][1] = c1;
          *reinterpret_cast<double2 *>(Xs + row * 8 + 2 * t) = make_double2(c0, c1);
        }
        __syncwarp();
#pragma unroll
        for (int s_ = 0; s_ < 7; s_++) bx[s_] = Xs[(4 * s_ + t) * 8 + g];
#pragma unroll
        for (int ti = 0; ti < 2; ti++) {
          const int row = 8 * ti + g;
          double c0 = 0.0, c1 = 0.0;
          if (row < nk && okc) { const double2 d = *reinterpret_cast<const double2 *>(DL + row * FNZ + cc); c0 = -d.x; c1 = -d.y; }
#pragma unroll
          for (int s_ = 0; s_ < 7; s_++) dmma_8x8x4(c0, c1, (row < nk) ? Jb[row * NV + 4 * s_ + t] : 0.0, bx[s_]);
          *reinterpret_cast<double2 *>(Ts + row * 8 + 2 * t) = make_double2(c0, c1);
        }
        __syncwarp();
        double dl[2][2];
#pragma unroll
        for (int ti = 0; ti < 2; ti++) {
          const int row = 8 * ti + g;
          double c0 = 0.0, c1 = 0.0;
          for (int s_ = 0; s_ < ks2; s_++) {
            const int k = 4 * s_ + t;
            dmma_8x8x4(c0, c1, (row < nk && k < nk) ? w.G[row * 12 + k] : 0.0, (k < nk) ? Ts[k * 8 + g] : 0.0);
          }
          dl[ti][0] = c0; dl[ti][1] = c1;
        }
        __syncwarp();
#pragma unroll
        for (int ti = 0; ti < 2; ti++) {
          const int row = 8 * ti + g;
          *reinterpret_cast<double2 *>(Ts + row * 8 + 2 * t) = make_double2(dl[ti][0], dl[ti][1]);
          if (row < nk && okc) *reinterpret_cast<double2 *>(DL + row * FNZ + cc) = make_double2(dl[ti][0], dl[ti][1]);
        }
        __syncwarp();
#pragma unroll
        for (int ti = 0; ti < 4; ti++) {
          const int row = 8 * ti + g;
          double c0 = -xn[ti][0], c1 = -xn[ti][1];
          for (int s_ = 0; s_ < ks2; s_++) {
            const int k = 4 * s_ + t;
            dmma_8x8x4(c0, c1, (row < NV && k < nk) ? w.Y[row * 13 + 1 + k] : 0.0, (k < nk) ? Ts[k * 8 + g] : 0.0);
          }
          if (row < NV && okc) *reinterpret_cast<double2 *>(X + row * FNZ + cc) = make_double2(c0, c1);
        }
        __syncwarp();
      }
    }
    SYNC();
#endif
  }

  EPH(9);
  // ---- semi-implicit Euler + gap (App. A2)
  PAR_FOR(i, NV) { double dv = dt * w.acc[i]; w.dx[NV + i] = dv; w.dx[i] = dt * (w.x[NQ + i] + dv); }
  // stage the multipliers (their global-load latency hides behind the cost-term phase)
  PAR_FOR(i, FNC) { w.mv[i] = io.v[i]; w.mvp[i] = io.v_prev[i]; }
  PAR_FOR(i, FN) { w.mln[i] = io.lam_n[i]; w.mlnp[i] = io.lam_n_prev[i]; w.mlk[i] = io.lam_k[i]; }
  SYNC();
  mb_cost_terms<FullWsT<DERIV>, ROLL>(m, w, kn.lf_ref, kn.rf_ref, DERIV, io.gap, io.slack);
  if (ROLL) PAR_FOR(i, NQ + NV) io.xn_out[i] = w.xn[i];

  EPH(10);
  if (DERIV) {
    // the kinematics block [oM | S | v | a | I | Ic] is dead from here on: stage the dlam/dz rows of the active contacts into it, so the
    // gradient / Hessian / constraint-row phases below read them from shared memory instead of the L2-resident scratch
    static_assert(NB * 12 + NV * 6 + 2 * NB * 6 + 2 * NB * 10 >= 12 * FNZ, "dlam/dz does not fit in the dead kinematics block");
    double *DLs = reinterpret_cast<double *>(&w) + offsetof(FullWsT<DERIV>, oM) / sizeof(double); // the whole block, not just oM
    PAR_FOR(e, nk * FNZ) DLs[e] = DL[e];
    DL = DLs; // (the barrier before the first read is the one inside the merit reduction below)
  }
  // ---- constraint values, multiplier estimates, activity
  // every thread accumulates the merit pieces of the rows / coordinates it owns; one group-wide reduction at the end
  double acc_cost = 0.0, acc_pen = 0.0, acc_prim = 0.0, acc_inner = 0.0;
  PAR_FOR(r, FNC) {
    int type = -1; double hv = 0, lo = 0, hi = 0;
    if (r < 22) { type = 2; hv = w.u[r]; lo = -rb.tau_max[r]; hi = rb.tau_max[r]; }
    else if (r < 44) { int i = r - 22; type = 2; hv = -w.x[7 + i]; lo = -rb.q_hi[i]; hi = -rb.q_lo[i]; }
    else {
      int f = (r - 44) / 17, rr = (r - 44) % 17;
      if (w.sidx[f] >= 0) { type = 1; for (int k = 0; k < 6; k++) hv += m.Acone[6 * rr + k] * w.lam[6 * f + k]; }
    }
    mb_row_epilogue(w, io, r, type, hv, lo, hi, w.mv, w.mvp, acc_pen, acc_prim, acc_inner);
  }
  mb_dynamics_rows(m, w, io, w.mln, w.mlnp, acc_cost, acc_pen, acc_prim, acc_inner);
  PAR_FOR(i, FM) { const double e = w.u[i] - kn.u_ref[i]; acc_cost += 0.5 * cfg.wu[i] * e * e; }
  PAR_FOR(i, 6) acc_cost += 0.5 * (cfg.w_cent[i] * w.rcent[i] * w.rcent[i] + kn.w_lf[i] * w.rpose[i] * w.rpose[i] + kn.w_rf[i] * w.rpose[6 + i] * w.rpose[6 + i]);
  PAR_FOR(e, 12) {
    const int f = e / 6, i = e % 6;
    if (kn.fcost[f] != 0.0) { const double d = w.lam[e] - kn.f_ref[e]; acc_cost += 0.5 * cfg.w_force[i] * d * d; }
  }
  mb_merit_finish<FNC>(w, acc_cost, acc_pen, acc_prim, acc_inner);
  if (!DERIV) {
    PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i];
    EPH(11);
    EPH_DUMP(io.phase_out);
    return;
  }

  EPH(11);
  // ---- LQ blocks to HBM: AB (56 x 78), Lagrangian gradient, cost gradient / Hessian, active constraint rows
  mb_store_rows<FNC>(w, io);
  PAR_FOR(z, FNZ) {
    double xc[NV];
#pragma unroll
    for (int i = 0; i < NV; i++) xc[i] = X[i * FNZ + z]; // one pass over the column of the tangent (L2-resident scratch)
    const double acc = mb_ab_column<FNZ>(w, io, z, xc, 1, dt, w.mln);
    // cost gradient
    double lz = mb_cost_grad(w, cfg.wx, cfg.w_cent, kn.w_lf, kn.w_rf, z);
    if (z >= FN) lz += cfg.wu[z - FN] * (w.u[z - FN] - kn.u_ref[z - FN]);
    for (int f = 0; f < 2; f++)
      if (kn.fcost[f] != 0.0) {
        const double *Dl = DL + 6 * w.sidx[f] * FNZ;
        for (int r = 0; r < 6; r++) lz += cfg.w_force[r] * Dl[r * FNZ + z] * (w.lam[6 * f + r] - kn.f_ref[6 * f + r]);
      }
    w.late.lxu[z] = lz; io.lxu[z] = lz;
    // Lagrangian gradient: + C^T v  (+ E_{k-1}^T lam_k: vector part here, base block added by the reduction kernel)
    double gz = lz + acc;
    for (int r = 0; r < FNC; r++) {
      double vr = w.mv[r];
      if (vr == 0.0 || w.ctype[r] < 0) continue;
      gz += full_c_entry(m, DL, w.sidx, r, z) * vr;
    }
    if (z < FN) { if (io.k == 0) gz += w.mlk[z]; else if (z >= 6) gz -= w.mlk[z]; }
    w.late.g[z] = gz; io.g[z] = gz;
  }
  mb_gE_next(w, io, w.mln);
  EPH(12);
#ifdef MPC_HOST_EMU
  mb_gn_hessian<FNZ>(w, io, cfg, kn, [&](auto &rank1) { // contact-force cost rows dlam/dz
    for (int f = 0; f < 2; f++)
      if (kn.fcost[f] != 0.0) for (int r = 0; r < 6; r++) rank1(DL + (6 * w.sidx[f] + r) * FNZ, FNZ, cfg.w_force[r]);
  });
#else
  { // Gauss-Newton Hessian H = sum_k w_k J_k' J_k (+ state/control diagonals) as ONE tensor-core product over the 36 weighted
    // residual-Jacobian rows (12 contact-force rows dlam/dz, 6 centroidal momentum, 12 foot pose, 6 of the base block of the state
    // error; absent costs keep weight 0).  The rows stay where they are in shared memory and are addressed through a table of
    // offsets; every warp takes 2 x 2 blocks of 8 x 8 tiles of the FULL matrix, so the result leaves as row-major 16-byte stores.
    const double *base = reinterpret_cast<const double *>(&w);
    PAR_FOR(k, 36) {
      const double *p = w.Jls; int len = 0; double wgt = 0.0;
      if (k < 12) { const int f = k / 6, r = k % 6; if (kn.fcost[f] != 0.0 && w.sidx[f] >= 0) { p = DL + (6 * w.sidx[f] + r) * FNZ; len = FNZ; wgt = cfg.w_force[r]; } }
      else if (k < 18) { p = w.cj.Jcent + (k - 12) * FN; len = FN; wgt = cfg.w_cent[k - 12]; }
      else if (k < 30) { const int j = k - 18, r = j % 6; p = w.cj.Jpose + j * NV; len = NV; wgt = (j < 6) ? kn.w_lf[r] : kn.w_rf[r]; }
      else { p = w.Jls + 6 * (k - 30); len = 6; wgt = cfg.wx[k - 30]; }
      w.hrow_len[k] = (int32_t)(p - base) | (len << 20); // offset (doubles) and row length packed in one word
      w.hrow_w[k] = wgt;
    }
    SYNC();
    constexpr int NBK = ((FNZ + 7) / 8 + 1) / 2; // 5 blocks of 16 per side
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    for (int p = WARP_ID; p < NBK * NBK; p += NWARPS) {
      const int ti = 2 * (p / NBK), tj = 2 * (p % NBK);
      const int ia = ti * 8 + g, ib = tj * 8 + g;
      double c[2][2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
#pragma unroll 3
      for (int k0 = 0; k0 < 36; k0 += 4) {
        const int packed = w.hrow_len[k0 + t], off = packed & 0xFFFFF, len = packed >> 20;
        const double wk = w.hrow_w[k0 + t];
        const double *row = base + off;
        const double a0 = (ia < len) ? wk * row[ia] : 0.0, a1 = (ia + 8 < len) ? wk * row[ia + 8] : 0.0;
        const double b0 = (ib < len) ? row[ib] : 0.0, b1 = (ib + 8 < len) ? row[ib + 8] : 0.0;
        dmma_8x8x4(c[0][0][0], c[0][0][1], a0, b0);
        dmma_8x8x4(c[0][1][0], c[0][1][1], a0, b1);
        dmma_8x8x4(c[1][0][0], c[1][0][1], a1, b0);
        dmma_8x8x4(c[1][1][0], c[1][1][1], a1, b1);
      }
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const int r = (ti + a) * 8 + g, cc = (tj + b) * 8 + 2 * t;
          if (r >= FNZ || cc >= FNZ) continue;
          double h0 = c[a][b][0], h1 = c[a][b][1];
          const double dg = io.preg + ((r >= FN) ? cfg.wu[r - FN] : ((r >= 6) ? cfg.wx[r] : 0.0));
          if (r == cc) h0 += dg; else if (r == cc + 1) h1 += dg;
          *reinterpret_cast<double2 *>(io.H + r * FNZ + cc) = make_double2(h0, h1);
        }
    }
  }
#endif
  EPH(13);
  PAR_FOR(e, w.nca * FNZ) { // active constraint rows, compacted
    int ai = e / FNZ, z = e % FNZ;
    io.CDact[e] = full_c_entry(m, DL, w.sidx, w.act_idx[ai], z);
  }
  mb_dual_scal<FNZ>(w, io);
  EPH(14);
  EPH_DUMP(io.phase_out);
}

} // namespace mpcdev
