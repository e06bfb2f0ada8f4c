// Device-side model block: robot tree + problem constants + tree index tables, built once on the host
// (mpc_create) and read by every kernel.  Replaces the per-object pinocchio::Model / aligator StageModel
// parameter storage of the reference (fulldynamic_talos.py:27-97,121-151).
#pragma once
#include "../../include/mpcb200.h"
#include "dev_common.cuh"
#include <string>

namespace mpcdev {

constexpr int NB = MPC_NB, NV = MPC_NV, NQ = MPC_NQ, NJ = MPC_NJ;
constexpr int MAX_PAIRS = NV * NB;

struct DevModel {
  mpc_robot_t rb;
  mpc_config_t cfg;
  double Acone[17 * 6];
  // tree tables
  int32_t nlevels, level_start[NB + 1], level_body[NB];
  uint32_t anc_mask[NB];   // bit a set: body a is ancestor-or-self of b
  uint32_t sub_mask[NB];   // bit d set: body d is in the subtree of b (incl. b)
  uint32_t ancdof_mask[NB];// bit j set: dof j belongs to an ancestor-or-self body of b
  int32_t npairs, pair_j[MAX_PAIRS], pair_m[MAX_PAIRS]; // (dof j, body m) with m in subtree(body(j))
  int32_t nanc, anc_i[NV * NV], anc_j[NV * NV];         // (dof i, dof j) with body(i) a STRICT ancestor of body(j)
  double total_mass;
};

#ifdef MPC_HOST_EMU
#define HDH inline
#else
#define HDH __host__ __device__ __forceinline__
#endif
HDH int body_of_dof(int j) { return j < 6 ? 0 : j - 5; }
HDH int first_dof(int b) { return b == 0 ? 0 : 5 + b; }
HDH int ndof_of(int b) { return b == 0 ? 6 : 1; }

#if 1
inline void cone_matrix_host(double mu, double L, double W, double *A) {
  for (int i = 0; i < 17 * 6; i++) A[i] = 0;
  auto row = [&](int r, double fx, double fy, double fz, double tx, double ty, double tz) {
    double *a = A + 6 * r; a[0] = fx; a[1] = fy; a[2] = fz; a[3] = tx; a[4] = ty; a[5] = tz;
  };
  row(0, 0, 0, -1, 0, 0, 0);
  row(1, 1, 0, -mu, 0, 0, 0); row(2, -1, 0, -mu, 0, 0, 0);
  row(3, 0, 1, -mu, 0, 0, 0); row(4, 0, -1, -mu, 0, 0, 0);
  row(5, 0, 0, -W, 1, 0, 0); row(6, 0, 0, -W, -1, 0, 0);
  row(7, 0, 0, -L, 0, 1, 0); row(8, 0, 0, -L, 0, -1, 0);
  int r = 9;
  for (int s1 = 1; s1 >= -1; s1 -= 2)
    for (int s2 = 1; s2 >= -1; s2 -= 2) row(r++, s1 * W, s2 * L, -mu * (L + W), -s1 * mu, -s2 * mu, -1);
  for (int s1 = 1; s1 >= -1; s1 -= 2)
    for (int s2 = 1; s2 >= -1; s2 -= 2) row(r++, s1 * W, s2 * L, -mu * (L + W), s1 * mu, s2 * mu, 1);
}

// returns 0 on success, fills err otherwise
inline int build_dev_model(const mpc_robot_t *rb, const mpc_config_t *cfg, DevModel *m, const char **err) {
  m->rb = *rb;
  m->cfg = *cfg;
  if (rb->nb != NB) { *err = "robot must have 23 bodies (free-flyer + 22 revolute)"; return 1; }
  if (rb->parent[0] != -1) { *err = "body 0 must be the root"; return 1; }
  for (int b = 1; b < NB; b++) if (rb->parent[b] < 0 || rb->parent[b] >= b) { *err = "bodies must be ordered parents-first"; return 1; }
  cone_matrix_host(cfg->mu_fric, cfg->foot_L, cfg->foot_W, m->Acone);
  int depth[NB];
  depth[0] = 0;
  int maxd = 0;
  for (int b = 1; b < NB; b++) { depth[b] = depth[rb->parent[b]] + 1; if (depth[b] > maxd) maxd = depth[b]; }
  m->nlevels = maxd + 1;
  int pos = 0;
  for (int l = 0; l <= maxd; l++) { m->level_start[l] = pos; for (int b = 0; b < NB; b++) if (depth[b] == l) m->level_body[pos++] = b; }
  m->level_start[maxd + 1] = pos;
  for (int b = 0; b < NB; b++) { m->anc_mask[b] = 0; m->sub_mask[b] = 0; m->ancdof_mask[b] = 0; }
  for (int b = 0; b < NB; b++)
    for (int k = b; k >= 0; k = rb->parent[k]) {
      m->anc_mask[b] |= 1u << k; m->sub_mask[k] |= 1u << b;
      for (int d = 0; d < ndof_of(k); d++) m->ancdof_mask[b] |= 1u << (first_dof(k) + d);
    }
  m->npairs = 0; m->nanc = 0;
  for (int j = 0; j < NV; j++) {
    int J = body_of_dof(j);
    for (int b = 0; b < NB; b++) if (m->sub_mask[J] >> b & 1) { m->pair_j[m->npairs] = j; m->pair_m[m->npairs] = b; m->npairs++; }
    for (int i = 0; i < NV; i++) { int bi = body_of_dof(i); if (bi != J && (m->anc_mask[J] >> bi & 1)) { m->anc_i[m->nanc] = i; m->anc_j[m->nanc] = j; m->nanc++; } }
  }
  m->total_mass = 0;
  for (int b = 0; b < NB; b++) m->total_mass += rb->mass[b];
  return 0;
}

// Per-instance models of a batch (mpc_set_instance_models): out[i] is built from robots[i] / cfgs[i], or from the shared robot / config
// of `shared` where the array is null.  What the kernels of one launch must agree on stays uniform and is checked here: the model kind,
// horizon and time step (workspace shape and Riccati dimensions), the solver constants (one BCL / linesearch schedule per handle, read from
// Ws::sc and instance 0's model) and the tree topology (parent array and sole bodies: the tree tables are built once per shape).  Returns
// an empty string, or an error naming the first offending instance and field.
inline std::string build_instance_models(const DevModel &shared, const mpc_robot_t *robots, const mpc_config_t *cfgs, int batch, DevModel *out) {
  const mpc_robot_t &r0 = shared.rb;
  const mpc_config_t &c0 = shared.cfg;
  for (int i = 0; i < batch; i++) {
    const mpc_robot_t &r = robots ? robots[i] : r0;
    const mpc_config_t &c = cfgs ? cfgs[i] : c0;
    auto bad = [&](const char *field) { return "mpc_set_instance_models: instance " + std::to_string(i) + ": " + field + " differs from the handle's"; };
    if (c.kind != c0.kind) return bad("cfg.kind");
    if (c.T != c0.T) return bad("cfg.T");
    if (c.dt != c0.dt) return bad("cfg.dt");
    if (c.tol != c0.tol) return bad("cfg.tol");
    if (c.mu_init != c0.mu_init) return bad("cfg.mu_init");
    if (c.max_iters != c0.max_iters) return bad("cfg.max_iters");
    if (c.force_initial_condition != c0.force_initial_condition) return bad("cfg.force_initial_condition");
    if (c.rollout != c0.rollout) return bad("cfg.rollout");
    if (c.lq_legs != c0.lq_legs) return bad("cfg.lq_legs");
    if (r.nb != r0.nb) return bad("robot.nb");
    for (int b = 0; b < NB; b++) if (r.parent[b] != r0.parent[b]) return bad("robot.parent");
    if (r.foot_body[0] != r0.foot_body[0] || r.foot_body[1] != r0.foot_body[1]) return bad("robot.foot_body");
    const char *err = nullptr;
    if (build_dev_model(&r, &c, out + i, &err)) return "mpc_set_instance_models: instance " + std::to_string(i) + ": " + err;
  }
  return std::string();
}
#endif

} // namespace mpcdev
