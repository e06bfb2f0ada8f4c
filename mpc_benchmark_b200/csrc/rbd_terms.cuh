// Rigid-body terms of the whole-body QPs (SURVEY 8f row f-3, the step in front of the QP): for one measured state x = (q, v)
// what the reference computes with pinocchio before every ID_solver.solve (kinodynamic_talos.py:425-431, QP_utils.py:515-528):
//   M      = pin.crba(q)                                             [nv][nv]
//   nle    = pin.nonLinearEffects(q, v)                              [nv]
//   Jc     = pin.getFrameJacobian(..., LOCAL) of both sole frames    [12][nv]
//   dJv    = pin.getFrameJacobianTimeVariation(..., LOCAL) @ v       [12]   (spatial acceleration of the frame at zero joint acceleration)
//   vf     = pin.getFrameVelocity(...)  (LOCAL: linear, angular)     [2][6]
// One group of threads per state, on the kinematics / composite-inertia phases of the evaluation kernel
// (mb_kinematics and the bias-force phase of eval_full_knot), world-frame formulation, everything in the group's shared memory.
// ikid_terms_group adds the task terms of the IKID QP (centroidal momentum matrix, base / torso orientation Jacobians) on the same phases.
#pragma once
#include "eval_mb.cuh"

namespace mpcdev {

template <class WS> HD void rbd_terms_group(const DevModel &m, const double *x, WS &w, double *M_out, double *nle_out, double *Jc_out, double *dJv_out, double *vf_out) {
  const mpc_robot_t &rb = m.rb;
  PAR_FOR(i, NQ + NV) w.x[i] = x[i];
  SYNC();
  mb_kinematics(m, w);
  const double a0[6] = {-rb.gravity[0], -rb.gravity[1], -rb.gravity[2], 0, 0, 0};
  // bias accelerations (joint accelerations zero, gravity folded in) and bias forces per body
  PAR_FOR(b, NB) {
    double acc[6] = {a0[0], a0[1], a0[2], 0, 0, 0};
    const uint32_t mask = m.anc_mask[b];
    for (int k = 1; k <= b; k++)
      if (mask >> k & 1) {
        double sj[6], c[6];
        for (int i = 0; i < 6; i++) sj[i] = w.S[6 * (5 + k) + i] * w.x[NQ + 5 + k];
        cross_mm(w.v + 6 * k, sj, c);
        for (int i = 0; i < 6; i++) acc[i] += c[i];
      }
    for (int i = 0; i < 6; i++) w.a[6 * b + i] = acc[i];
    double t1[6], t2[6];
    inertia_mul(w.I + 10 * b, acc, t1);
    cross_mf(w.v + 6 * b, w.hb + 6 * b, t2);
    for (int i = 0; i < 6; i++) w.f[6 * b + i] = t1[i] + t2[i];
  }
  SYNC();
  PAR_FOR(e, NB * 6) { // subtree sums of the bias forces
    const int b = e / 6, c = e % 6;
    const uint32_t mask = m.sub_mask[b];
    double s = 0;
    for (int d = b; d < NB; d++) if (mask >> d & 1) s += w.f[6 * d + c];
    w.Fsub[e] = s;
  }
  PAR_FOR(e, NV * NV) { // composite-rigid-body mass matrix, straight to the output
    const int i = e / NV, j = e % NV, bi = body_of_dof(i), bj = body_of_dof(j);
    double v = 0;
    if (m.anc_mask[bj] >> bi & 1) v = dot6(w.S + 6 * i, w.U + 6 * j);
    else if (m.anc_mask[bi] >> bj & 1) v = dot6(w.S + 6 * j, w.U + 6 * i);
    M_out[e] = v;
  }
  PAR_FOR(f, 2) { // frame velocity and dJ v of both soles in their LOCAL frames
    const int fb = rb.foot_body[f];
    se3_actinv_motion(w.ofoot + 12 * f, w.v + 6 * fb, vf_out + 6 * f);
    double an[6];
    for (int i = 0; i < 6; i++) an[i] = w.a[6 * fb + i] - a0[i];
    se3_actinv_motion(w.ofoot + 12 * f, an, dJv_out + 6 * f);
  }
  PAR_FOR(e, 12 * NV) Jc_out[e] = w.Jf[e];
  SYNC();
  PAR_FOR(j, NV) nle_out[j] = dot6(w.S + 6 * j, w.Fsub + 6 * body_of_dof(j));
}

// Task terms of the IKID QP (IKIDSolver_f6, QP_utils.py:666-675,684,690) on top of rbd_terms_group, for the same state:
//   Ag    [6][nv]    data.Ag, centroidal momentum matrix about the CoM (linear rows, then angular), column j = shift_to_com(U_j)
//   dAgv  [6]        data.dAg @ v: rate of the centroidal momentum at zero joint acceleration, gravity excluded
//   Jang  [2][3][nv] angular rows of the LOCAL Jacobian of the frames (frame_body[f], frame_place[f]): R_frame' * ang(S_j)
//   dJang [2][3]     angular part of those frames' LOCAL acceleration at zero joint acceleration (dJ v)
// The frame velocities of rbd_terms_group go to w.vc, which nothing else here uses.
template <class WS>
HD void ikid_terms_group(const DevModel &m, const double *x, const int32_t *frame_body, const double *frame_place, WS &w, double *M_out, double *nle_out,
                         double *Jc_out, double *dJv_out, double *Ag_out, double *dAgv_out, double *Jang_out, double *dJang_out) {
  rbd_terms_group(m, x, w, M_out, nle_out, Jc_out, dJv_out, w.vc);
  // U, com, Ic, a and Fsub were complete before rbd_terms_group's last barrier, and its last phase writes none of them
  PAR_FOR(j, NV) {
    const double *Uj = w.U + 6 * j;
    double c[3];
    cross3(w.com, Uj, c);
    for (int r = 0; r < 3; r++) { Ag_out[r * NV + j] = Uj[r]; Ag_out[(3 + r) * NV + j] = Uj[3 + r] - c[r]; }
  }
  PAR_FOR(e, 2 * NV) {
    const int f = e / NV, j = e % NV, fb = frame_body[f];
    double col[6] = {0, 0, 0, 0, 0, 0};
    if (m.ancdof_mask[fb] >> j & 1) {
      double of[12];
      se3_mul(w.oM + 12 * fb, frame_place + 12 * f, of);
      se3_actinv_motion(of, w.S + 6 * j, col);
    }
    for (int r = 0; r < 3; r++) Jang_out[(3 * f + r) * NV + j] = col[3 + r];
  }
  PAR_FOR(f, 2) {
    const int fb = frame_body[f];
    const double a0[6] = {-m.rb.gravity[0], -m.rb.gravity[1], -m.rb.gravity[2], 0, 0, 0};
    double of[12], an[6], loc[6];
    se3_mul(w.oM + 12 * fb, frame_place + 12 * f, of);
    for (int i = 0; i < 6; i++) an[i] = w.a[6 * fb + i] - a0[i];
    se3_actinv_motion(of, an, loc);
    for (int r = 0; r < 3; r++) dJang_out[3 * f + r] = loc[3 + r];
  }
  ONE_THREAD { // total bias force (Fsub of the root) at the CoM, minus the gravity wrench [m a_world; 0] folded into it
    const double *F = w.Fsub;
    double c[3];
    cross3(w.com, F, c);
    for (int r = 0; r < 3; r++) { dAgv_out[r] = F[r] + w.Ic[0] * m.rb.gravity[r]; dAgv_out[3 + r] = F[3 + r] - c[r]; }
  }
}

} // namespace mpcdev
