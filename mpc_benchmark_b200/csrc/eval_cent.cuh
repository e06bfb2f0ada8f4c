// Per-knot evaluation of the CENTROIDAL Talos stage (closed form): one CTA (one warp) per (instance, knot).
//
// Replaces CentroidalFwdDynamics + IntegratorEuler (centroidal_talos.py:202-205), the CostStack of
// centroidal_talos.py:212-240 (control, CoM, linear/angular momentum, angular/linear acceleration residuals)
// and the CentroidalWrenchConeResidual constraints (centroidal_talos.py:242-245).
//   x = [c, h_lin, h_ang], u = [f_L, tau_L, f_R, tau_R];  xdot = [h_lin/m; m g + sum f; sum (p_i - c) x f_i + tau_i]
#pragma once
#include "eval_mb.cuh"

namespace mpcdev {

constexpr int CN = 9, CM = 12, CNZ = 21, CNC = 34;

struct CentWs {
  double x[CN], u[CM], xn[CN];
  double kn[sizeof(mpc_knot_t) / 8];
  double xd[CN], Fx[CN * CN], Fu[CN * CM];
  double J[6 * CNZ], r[6], wgt[6]; // rows: angular-acc (3), linear-acc (3)
  double lxu[CNZ], g[CNZ], gap[CN];
  double hval[CNC], vpl[CNC], dbr[CNC], rowtmp[CNC], lpl[CN], fbr[CN];
  double scal[SC_COUNT];
  int32_t ctype[CNC], isact[CNC], act_idx[CNC], nca;
};

template <bool DERIV, bool ROLL = false> HD void eval_cent_knot(const DevModel &m, const KnotIO &io, CentWs &w) {
  const mpc_config_t &cfg = m.cfg;
  const double mass = cfg.mass, dt = cfg.dt;
  PAR_FOR(i, CN) { w.x[i] = io.x[i]; w.xn[i] = io.xn[i]; }
  PAR_FOR(i, CM) w.u[i] = io.u[i];
  PAR_FOR(i, (int)(sizeof(mpc_knot_t) / 8)) w.kn[i] = reinterpret_cast<const double *>(io.kn)[i];
  PAR_FOR(i, CN * CN) w.Fx[i] = 0.0;
  PAR_FOR(i, CN * CM) w.Fu[i] = 0.0;
  PAR_FOR(i, 6 * CNZ) w.J[i] = 0.0;
  SYNC();
  const mpc_knot_t &kn = *reinterpret_cast<const mpc_knot_t *>(w.kn);
  ONE_THREAD {
    double ft[3] = {0, 0, 0};
    for (int i = 0; i < 3; i++) { w.xd[i] = w.x[3 + i] / mass; w.xd[3 + i] = mass * m.rb.gravity[i]; w.xd[6 + i] = 0; w.Fx[i * CN + 3 + i] = 1.0 / mass; }
    for (int k = 0; k < 2; k++) {
      if (kn.cs[k] == 0.0) continue;
      const double *f = w.u + 6 * k, *t = f + 3;
      double d[3] = {kn.cpos[3 * k] - w.x[0], kn.cpos[3 * k + 1] - w.x[1], kn.cpos[3 * k + 2] - w.x[2]}, mo[3], px[9];
      cross3(d, f, mo);
      skew3(d, px);
      for (int i = 0; i < 3; i++) {
        w.xd[3 + i] += f[i]; w.xd[6 + i] += mo[i] + t[i]; ft[i] += f[i];
        w.Fu[(3 + i) * CM + 6 * k + i] = 1.0; w.Fu[(6 + i) * CM + 6 * k + 3 + i] = 1.0;
        for (int j = 0; j < 3; j++) w.Fu[(6 + i) * CM + 6 * k + j] = px[3 * i + j];
      }
    }
    double fx[9];
    skew3(ft, fx); // d/dc sum (p - c) x f = [f]x
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) w.Fx[(6 + i) * CN + j] = fx[3 * i + j];
    for (int i = 0; i < CN; i++) {
      double xn = w.x[i] + dt * w.xd[i];
      if (ROLL) { w.xn[i] = xn + io.slack[i]; io.xn_out[i] = w.xn[i]; } // nonlinear rollout: x_{k+1} := f(x, u) + slack
      w.gap[i] = xn - w.xn[i]; io.gap[i] = w.gap[i]; io.xdot[i] = w.xd[i];
    }
    // residual rows: angular acceleration = xdot[6:9] (cent:217-219), linear acceleration = g + sum f / m (cent:214-216)
    for (int i = 0; i < 3; i++) {
      w.r[i] = w.xd[6 + i]; w.wgt[i] = cfg.w_angacc[i];
      w.r[3 + i] = w.xd[3 + i] / mass; w.wgt[3 + i] = cfg.w_linacc[i];
      for (int j = 0; j < CN; j++) w.J[i * CNZ + j] = w.Fx[(6 + i) * CN + j];
      for (int j = 0; j < CM; j++) { w.J[i * CNZ + CN + j] = w.Fu[(6 + i) * CM + j]; w.J[(3 + i) * CNZ + CN + j] = w.Fu[(3 + i) * CM + j] / mass; }
    }
  }
  SYNC();
  PAR_FOR(r, CNC) {
    int k = r / 17, rr = r % 17, type = -1;
    double hv = 0;
    if (kn.cs[k] != 0.0) { type = 1; for (int j = 0; j < 6; j++) hv += m.Acone[6 * rr + j] * w.u[6 * k + j]; }
    int act = 0; double prim = 0;
    double vp = vplus_row(type, hv, io.v_prev[r], io.mu, 0, 0, act, prim);
    w.ctype[r] = type; w.hval[r] = hv; w.vpl[r] = vp; w.isact[r] = act; w.dbr[r] = io.mu * (vp - io.v[r]); w.rowtmp[r] = fabs(prim);
    io.h[r] = hv;
  }
  PAR_FOR(i, CN) { w.lpl[i] = io.lam_n_prev[i] + w.gap[i] / io.mu; w.fbr[i] = io.mu * (w.lpl[i] - io.lam_n[i]); }
  SYNC();
  ONE_THREAD {
    double cost = 0, pen = 0, prim = 0, inner = 0;
    for (int i = 0; i < CM; i++) { double e = w.u[i] - kn.u_ref[i]; cost += 0.5 * cfg.wu[i] * e * e; }
    for (int i = 0; i < 3; i++) {
      double ec = w.x[i] - cfg.com_ref[i];
      cost += 0.5 * (cfg.w_com[i] * ec * ec + cfg.w_linmom[i] * w.x[3 + i] * w.x[3 + i] + cfg.w_angmom[i] * w.x[6 + i] * w.x[6 + i]);
    }
    for (int i = 0; i < 6; i++) cost += 0.5 * w.wgt[i] * w.r[i] * w.r[i];
    int nca = 0;
    for (int r = 0; r < CNC; r++) {
      if (w.ctype[r] < 0) continue;
      double dv = w.vpl[r] - io.v[r];
      pen += 0.5 * io.mu * (w.vpl[r] * w.vpl[r] + dv * dv);
      prim = fmax(prim, w.rowtmp[r]); inner = fmax(inner, fabs(w.dbr[r]));
      if (w.isact[r]) w.act_idx[nca++] = r;
    }
    for (int i = 0; i < CN; i++) {
      double dl = w.lpl[i] - io.lam_n[i];
      pen += 0.5 * io.mu * (w.lpl[i] * w.lpl[i] + dl * dl);
      prim = fmax(prim, fabs(w.gap[i])); inner = fmax(inner, fabs(io.mu * dl));
    }
    w.nca = nca;
    w.scal[SC_COST] = cost; w.scal[SC_PEN] = pen; w.scal[SC_PRIM] = prim; w.scal[SC_INNER] = inner; w.scal[SC_DUAL] = 0;
  }
  SYNC();
  if (!DERIV) { PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i]; return; }
  PAR_FOR(i, CNC) { io.dbar[i] = w.dbr[i]; io.vplus[i] = w.vpl[i]; io.act_idx[i] = (i < w.nca) ? w.act_idx[i] : -1; }
  PAR_FOR(i, CN) { io.fbar[i] = w.fbr[i]; io.lplus[i] = w.lpl[i]; }
  PAR_FOR(i, 36) { double e = (i % 7 == 0) ? 1.0 : 0.0; io.T6[i] = e; io.E6[i] = -e; }
  ONE_THREAD io.nca[0] = w.nca;
  PAR_FOR(z, CNZ) {
    double acc = 0;
    for (int i = 0; i < CN; i++) {
      double s = (z < CN) ? ((i == z ? 1.0 : 0.0) + dt * w.Fx[i * CN + z]) : dt * w.Fu[i * CM + z - CN];
      io.AB[i * CNZ + z] = s; acc += s * io.lam_n[i];
    }
    double lz = 0;
    if (z >= CN) lz += cfg.wu[z - CN] * (w.u[z - CN] - kn.u_ref[z - CN]);
    else if (z < 3) lz += cfg.w_com[z] * (w.x[z] - cfg.com_ref[z]);
    else if (z < 6) lz += cfg.w_linmom[z - 3] * w.x[z];
    else lz += cfg.w_angmom[z - 6] * w.x[z];
    for (int r = 0; r < 6; r++) lz += w.wgt[r] * w.J[r * CNZ + z] * w.r[r];
    w.lxu[z] = lz; io.lxu[z] = lz;
    double gz = lz + acc;
    if (z >= CN) {
      int k = (z - CN) / 6, j = (z - CN) % 6;
      for (int rr = 0; rr < 17; rr++) { double vr = io.v[17 * k + rr]; if (vr != 0.0 && w.ctype[17 * k + rr] >= 0) gz += m.Acone[6 * rr + j] * vr; }
    } else gz += (io.k == 0) ? io.lam_k[z] : -io.lam_k[z];
    w.g[z] = gz; io.g[z] = gz;
  }
  PAR_FOR(j, 6) io.gE_next[j] = 0.0; // vector space: E = -I handled in-knot
  PAR_FOR(e, CNZ * CNZ) {
    int a = e / CNZ, b = e % CNZ;
    double hv = 0;
    if (a == b) {
      hv = io.preg;
      if (a >= CN) hv += cfg.wu[a - CN]; else if (a < 3) hv += cfg.w_com[a]; else if (a < 6) hv += cfg.w_linmom[a - 3]; else hv += cfg.w_angmom[a - 6];
    }
    for (int r = 0; r < 6; r++) hv += w.wgt[r] * w.J[r * CNZ + a] * w.J[r * CNZ + b];
    io.H[e] = hv;
  }
  PAR_FOR(e, w.nca * CNZ) {
    int ai = e / CNZ, z = e % CNZ, r = w.act_idx[ai], k = r / 17, rr = r % 17;
    io.CDact[e] = (z >= CN + 6 * k && z < CN + 6 * k + 6) ? m.Acone[6 * rr + z - CN - 6 * k] : 0.0;
  }
  SYNC();
  ONE_THREAD {
    double dual = 0;
    for (int z = (io.k == 0 ? CN : 0); z < CNZ; z++) dual = fmax(dual, fabs(w.g[z]));
    w.scal[SC_DUAL] = dual;
  }
  SYNC();
  PAR_FOR(i, SC_COUNT) io.scal[i] = w.scal[i];
}

// terminal knot: empty CostStack, no constraint (centroidal_talos.py:249,261)
template <bool DERIV> HD void eval_cent_term(const DevModel &m, const KnotIO &io, CentWs &w) {
  PAR_FOR(r, CNC) { io.h[r] = 0.0; if (DERIV) { io.dbar[r] = -io.mu * io.v[r]; io.vplus[r] = 0.0; io.act_idx[r] = -1; } }
  if (DERIV) {
    ONE_THREAD io.nca[0] = 0;
    PAR_FOR(z, CNZ) { io.lxu[z] = 0.0; io.g[z] = (z < CN) ? -io.lam_k[z] : 0.0; }
    PAR_FOR(e, CNZ * CNZ) io.H[e] = (e / CNZ == e % CNZ && e / CNZ < CN) ? io.preg : 0.0;
  }
  SYNC();
  ONE_THREAD {
    double dual = 0;
    if (DERIV) for (int z = 0; z < CN; z++) dual = fmax(dual, fabs(io.lam_k[z]));
    io.scal[SC_COST] = 0; io.scal[SC_PEN] = 0; io.scal[SC_PRIM] = 0; io.scal[SC_INNER] = 0; io.scal[SC_DUAL] = dual;
  }
}

} // namespace mpcdev
