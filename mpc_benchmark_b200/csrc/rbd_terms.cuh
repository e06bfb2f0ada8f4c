// Rigid-body terms of the whole-body QPs (SURVEY 8f row f-3, the step in front of the QP): for one measured state x = (q, v)
// what the reference computes with pinocchio before every ID_solver.solve (kinodynamic_talos.py:425-431, QP_utils.py:515-528):
//   M      = pin.crba(q)                                             [nv][nv]
//   nle    = pin.nonLinearEffects(q, v)                              [nv]
//   Jc     = pin.getFrameJacobian(..., LOCAL) of both sole frames    [12][nv]
//   dJv    = pin.getFrameJacobianTimeVariation(..., LOCAL) @ v       [12]   (spatial acceleration of the frame at zero joint acceleration)
//   vf     = pin.getFrameVelocity(...)  (LOCAL: linear, angular)     [2][6]
// One group of threads per state on the rigid-body phases of eval_mb.cuh that the full-dynamics knot also runs (kinematics, bias
// pass at zero joint acceleration, subtree sums, CRBA, sole motion), world-frame formulation, everything in the group's shared memory.
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
  mb_bias_forces(m, w, a0);
  SYNC();
  mb_subtree_sum<6>(m, w.f, w.Fsub);
  mb_crba(m, w, M_out);
  PAR_FOR(f, 2) mb_sole_motion(m, w, f, a0, vf_out + 6 * f, dJv_out + 6 * f);
  PAR_FOR(e, 12 * NV) Jc_out[e] = w.Jf[e];
  SYNC();
  PAR_FOR(j, NV) nle_out[j] = dot6(w.S + 6 * j, w.Fsub + 6 * body_of_dof(j));
}

// Task terms of the IKID QP (IKIDSolver_f6, QP_utils.py:666-675,684,690) on top of rbd_terms_group, for the same state:
//   Ag    [6][nv]    data.Ag, centroidal momentum matrix about the CoM (linear rows, then angular; mb_centroidal_map)
//   dAgv  [6]        data.dAg @ v: rate of the centroidal momentum at zero joint acceleration, gravity excluded
//   Jang  [2][3][nv] angular rows of the LOCAL Jacobian of the frames (frame_body[f], frame_place[f]): R_frame' * ang(S_j)
//   dJang [2][3]     angular part of those frames' LOCAL acceleration at zero joint acceleration (dJ v)
// The frame velocities of rbd_terms_group go to w.vc, which nothing else here uses.
template <class WS>
HD void ikid_terms_group(const DevModel &m, const double *x, const int32_t *frame_body, const double *frame_place, WS &w, double *M_out, double *nle_out,
                         double *Jc_out, double *dJv_out, double *Ag_out, double *dAgv_out, double *Jang_out, double *dJang_out) {
  rbd_terms_group(m, x, w, M_out, nle_out, Jc_out, dJv_out, w.vc);
  // U, com, Ic, a and Fsub were complete before rbd_terms_group's last barrier, and its last phase writes none of them
  mb_centroidal_map(w, Ag_out);
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
