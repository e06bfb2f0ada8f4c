// Rigid-body terms of the whole-body QPs (SURVEY 8f row f-3, the step in front of the QP): for one measured state x = (q, v)
// what the reference computes with pinocchio before every ID_solver.solve (kinodynamic_talos.py:425-431, QP_utils.py:515-528):
//   M      = pin.crba(q)                                             [nv][nv]
//   nle    = pin.nonLinearEffects(q, v)                              [nv]
//   Jc     = pin.getFrameJacobian(..., LOCAL) of both sole frames    [12][nv]
//   dJv    = pin.getFrameJacobianTimeVariation(..., LOCAL) @ v       [12]   (spatial acceleration of the frame at zero joint acceleration)
//   vf     = pin.getFrameVelocity(...)  (LOCAL: linear, angular)     [2][6]
// One group of threads per state, on the kinematics / composite-inertia phases of the evaluation kernel
// (mb_kinematics and the bias-force phase of eval_full_knot), world-frame formulation, everything in the group's shared memory.
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

} // namespace mpcdev
