// TEST-ONLY host emulation of the IKID kernel sources (ikid_terms_group in csrc/rbd_terms.cuh, qp_assemble_ikid_group in csrc/qp.cuh),
// compiled with -DMPC_HOST_EMU (PAR_FOR = serial loop, SYNC = no-op) like tests/emu/emu.cpp.  Lets the CPU test-suite check the
// kernel logic of the IKID path without a GPU.  Never loaded by the product package and not a fallback.
#define MPC_HOST_EMU 1
#include "../../mpc_benchmark_b200/csrc/eval_full.cuh"
#include "../../mpc_benchmark_b200/csrc/qp.cuh"
#include "../../mpc_benchmark_b200/csrc/rbd_terms.cuh"
#include <vector>

using namespace mpcdev;

// k_qp_assemble_ikid run serially
extern "C" void emu_qp_assemble_ikid(int batch, const double *M, const double *nle, const double *Jc, const double *dJv, const double *Ag, const double *dAgv,
                                     const double *Jang, const double *dJang, const double *task, const double *forces, const int32_t *cs, const double *weights,
                                     const double *gains, double mu, double L, double W, double *H, double *g, double *A, double *b, double *C, double *l) {
  double sm[24 * 28 + 24 + 12 + 28];
  for (int i = 0; i < batch; i++)
    qp_assemble_ikid_group(M + i * 784, nle + i * 28, Jc + i * 336, dJv + i * 12, Ag + i * 168, dAgv + i * 6, Jang + i * 168, dJang + i * 6, task + i * 98,
                           forces + i * 12, cs + i * 2, weights, gains, mu, L, W, sm, H + (size_t)i * 3844, g + i * 62, A + (size_t)i * 2480, b + i * 40,
                           C + (size_t)i * 1116, l + i * 18);
}

// k_ikid_terms run serially: rigid-body and IKID task terms of `count` states
extern "C" int emu_ikid_terms(const mpc_robot_t *rb, const mpc_config_t *cfg, int count, const double *x, const int32_t *frame_body, const double *frame_place,
                              double *M, double *nle, double *Jc, double *dJv, double *Ag, double *dAgv, double *Jang, double *dJang) {
  DevModel *model = new DevModel;
  const char *err = nullptr;
  if (build_dev_model(rb, cfg, model, &err)) { delete model; return 1; }
  std::vector<double> smem(sizeof(FullWsT<false>) / 8 + 8, 0.0);
  FullWsT<false> &w = *reinterpret_cast<FullWsT<false> *>(smem.data());
  for (int i = 0; i < count; i++)
    ikid_terms_group(*model, x + (size_t)i * 57, frame_body, frame_place, w, M + (size_t)i * 784, nle + (size_t)i * 28, Jc + (size_t)i * 336, dJv + (size_t)i * 12,
                     Ag + (size_t)i * 168, dAgv + (size_t)i * 6, Jang + (size_t)i * 168, dJang + (size_t)i * 6);
  delete model;
  return 0;
}
