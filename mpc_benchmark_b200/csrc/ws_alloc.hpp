// Workspace layout of one solver handle: every array is [batch][knot][...] row-major fp64 in HBM
// (results layout of SURVEY 8b: xs [B,T+1,nx], us [B,T,nu], K [B,T,nu,ndx]).
#pragma once
#include "driver.hpp"
#include <cstddef>
#include <cstring>

namespace mpcdev {

// state, tangent, control and constraint dimensions of a model kind (KindTraits)
inline void dims_of_kind(int kind, int &nx, int &n, int &m, int &nc) {
  dispatch_kind(kind, [&](auto k) {
    using K = KindTraits<decltype(k)::value>;
    nx = K::nx; n = K::n; m = K::m; nc = K::nc;
  });
}

// shape and solver constants of a workspace for `batch` instances of cfg's model kind; every array pointer starts null (alloc_ws)
inline void init_ws(Ws &w, const mpc_config_t &cfg, int batch, const DevModel *model) {
  std::memset(&w, 0, sizeof w);
  w.B = batch; w.T = cfg.T; w.kind = cfg.kind;
  dims_of_kind(cfg.kind, w.nx, w.n, w.m, w.nc);
  w.nz = w.n + w.m;
  w.model = model;
  w.sc = default_consts(cfg.tol, cfg.mu_init, cfg.rollout);
}

// alloc(bytes) must return zero-initialised memory
template <class Alloc> size_t alloc_ws(Ws &w, Alloc &&alloc) {
  const size_t B = w.B, T = w.T, T1 = T + 1, nx = w.nx, n = w.n, m = w.m, nc = w.nc, nz = w.nz;
  size_t total = 0;
  auto D = [&](double *&p, size_t count) { p = (double *)alloc(count * 8); total += count * 8; };
  auto I = [&](int32_t *&p, size_t count) { p = (int32_t *)alloc(count * 4); total += count * 4; };
  w.knots = (mpc_knot_t *)alloc(B * T * sizeof(mpc_knot_t)); total += B * T * sizeof(mpc_knot_t);
  w.terms = (mpc_term_t *)alloc(B * sizeof(mpc_term_t)); total += B * sizeof(mpc_term_t);
  D(w.x0, B * nx);
  D(w.xs, B * T1 * nx); D(w.us, B * T * m); D(w.vs, B * T1 * nc); D(w.lams, B * T1 * n);
  D(w.vs_prev, B * T1 * nc); D(w.lams_prev, B * T1 * n);
  D(w.txs, B * T1 * nx); D(w.tus, B * T * m); D(w.tvs, B * T1 * nc); D(w.tlams, B * T1 * n);
  D(w.dxs, B * T1 * n); D(w.dus, B * T * m); D(w.dvs, B * T1 * nc); D(w.dlams, B * T1 * n);
  D(w.AB, B * T * n * nz); D(w.H, B * T1 * nz * nz); D(w.lxu, B * T1 * nz); D(w.g, B * T1 * nz);
  D(w.T6, B * T * 36); D(w.E6, B * T * 36); D(w.gE, B * T1 * 6 + 6);
  D(w.fbar, B * T * n); D(w.dbar, B * T1 * nc); D(w.vplus, B * T1 * nc); D(w.lplus, B * T1 * n + n);
  D(w.CDact, B * T1 * nc * nz);
  I(w.nca, B * T1); I(w.act_idx, B * T1 * nc);
  D(w.gap, B * T * n); D(w.h, B * T1 * nc); D(w.scal, B * T1 * SC_COUNT); D(w.tscal, B * T1 * SC_COUNT);
  D(w.xdot, B * T1 * 56); D(w.lamc, B * T1 * 12);
  D(w.W, B * T * n * ((nz + 7) & ~(size_t)7)); D(w.pt, B * T * n); D(w.K, B * T * (m + nc) * (1 + n)); D(w.Kfb, B * T * m * n); D(w.dphi, B); D(w.phase, 64);
  w.ric_scratch_stride = dispatch_kind(w.kind, [](auto kind) { return KindTraits<decltype(kind)::value>::ric_scratch; });
  D(w.ric_scratch, B * w.ric_scratch_stride);
  w.st = (InstState *)alloc(B * sizeof(InstState)); total += B * sizeof(InstState);
  I(w.counters, 4); I(w.lists, 4 * B);
  return total;
}

// doubles per instance of the trajectory arrays the C-ABI moves in and out: xs, us, vs, lams and the feedback gains Kfb
struct TrajSizes {
  size_t xs, us, vs, lams, K;
};
inline TrajSizes traj_sizes(const Ws &w) {
  const size_t T = w.T, T1 = T + 1;
  return {T1 * w.nx, T * w.m, T1 * w.nc, T1 * w.n, T * w.m * w.n};
}

// the time-parallel LQ solve's per-(instance, leg) blocks for `legs` legs (lq_legs >= 2), allocated on first need; returns bytes
template <class Alloc> size_t alloc_leg_ws(const Ws &w, LegWs &lw, int legs, Alloc &&alloc) {
  size_t sz[4];
  dispatch_kind(w.kind, [&](auto k) {
    using Lay = typename LegDims<decltype(k)::value>::Lay;
    sz[0] = Lay::sum; sz[1] = Lay::ws; sz[2] = Lay::buf; sz[3] = KindTraits<decltype(k)::value>::ric_scratch;
  });
  const size_t n = (size_t)w.B * legs;
  double **p[4] = {&lw.sum, &lw.ws, &lw.buf, &lw.scratch};
  size_t total = 0;
  for (int i = 0; i < 4; i++) { *p[i] = (double *)alloc(n * sz[i] * 8); total += n * sz[i] * 8; }
  lw.L = legs;
  return total;
}

} // namespace mpcdev
