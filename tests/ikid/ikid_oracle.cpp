// TEST-ONLY reference for the IKID task terms, written on the CPU oracle's own rigid-body code (oracle/rbd.hpp), not on the kernels'
// composite formulation.  Parity with pinocchio is unpinned, like the rest of the oracle.
#include "../../oracle/rbd.hpp"

using namespace orc;

// Ag [6][NV] (centroidal_derivatives), dAgv [6] (centroidal_rate at qdd = 0, gravity excluded), the angular rows of the LOCAL Jacobians
// of two frames Jang [2][3][NV] and their dJ v [2][3] column by column from forward_kin, plus the frame placements oMf [2][12].
// Any output may be NULL.
extern "C" void orc_ikid_terms(const mpc_robot_t *rb, const double *x, const int *frame_body, const double *frame_place, double *Ag, double *dAgv,
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
