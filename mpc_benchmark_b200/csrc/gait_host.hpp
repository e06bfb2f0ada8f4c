// Host side of the device gait generator (gait.cuh): builds the contact-phase schedule and the countdown seeds of one gait from
// the parameters of include/mpcb200.h `mpc_gait_t` (fulldynamic_talos.py:248-280, kinodynamic_talos.py:183-198, centroidal_talos.py:100-116).
#pragma once
#include "gait.cuh"
#include <vector>

namespace mpcdev {

// phases[mirror][i] = (left, right) in contact; mirror: the first swing is made with the other foot
inline void gait_build_schedule(const mpc_gait_t &p, int nsteps, std::vector<int8_t> &phases, GaitCfg &g) {
  std::vector<int8_t> one;
  auto push = [&](std::vector<int8_t> &v, int l, int r, int n) { for (int i = 0; i < n; i++) { v.push_back((int8_t)l); v.push_back((int8_t)r); } };
  phases.clear();
  for (int mir = 0; mir < 2; mir++) {
    std::vector<int8_t> v;
    const int al = mir ? 0 : 1, ar = mir ? 1 : 0; // first single support: left foot down (right swings) unless mirrored
    push(v, 1, 1, p.T_ds);
    for (int c = 0; c < p.cycles; c++) { push(v, al, ar, p.T_ss); push(v, 1, 1, p.T_ds); push(v, ar, al, p.T_ss); push(v, 1, 1, p.T_ds); }
    if (p.half_cycle) { push(v, al, ar, p.T_ss); push(v, 1, 1, p.T_ds); }
    push(v, 1, 1, 2 * nsteps);
    const int nph = (int)v.size() / 2;
    g.nph = nph;
    for (int e = 0; e < 4; e++) g.n_ev[mir][e] = 0;
    for (int i = 1; i < nph; i++) {
      const int pl = v[2 * i], pr = v[2 * i + 1], ql = v[2 * i - 2], qr = v[2 * i - 1];
      int e = -1;
      if (pl && !pr && ql && qr) e = 0;        // right foot takes off
      else if (!pl && pr && ql && qr) e = 1;   // left foot takes off
      else if (pl && pr && ql && !qr) e = 2;   // right foot lands
      else if (pl && pr && !ql && qr) e = 3;   // left foot lands
      if (e >= 0 && g.n_ev[mir][e] < 8) g.ev[mir][e][g.n_ev[mir][e]++] = i + nsteps;
    }
    phases.insert(phases.end(), v.begin(), v.end());
  }
}

inline void gait_fill_cfg(const mpc_gait_t &p, int kind, int nsteps, GaitCfg &g) {
  g.kind = kind; g.T = nsteps; g.T_ds = p.T_ds; g.T_ss = p.T_ss; g.keep_forward = p.keep_forward; g.n_uref = p.n_uref; g.pad_ = 0;
  g.x_forward = p.x_forward; g.y_forward = p.y_forward; g.foot_yaw = p.foot_yaw; g.y_gap = p.y_gap; g.z_height = p.z_height; g.apex = p.swing_apex;
  for (int i = 0; i < 12; i++) { g.lf0[i] = p.lf0[i]; g.rf0[i] = p.rf0[i]; }
  for (int i = 0; i < 3; i++) g.com0[i] = p.com0[i];
  g.f_half = p.f_half; g.w_lfrf = p.w_lfrf;
  g.phases = nullptr; g.urefs = nullptr;
}

// every robot starts with both soles at the gait's initial placements; mirror (optional, [batch]): robots whose first swing is made with the other foot
inline std::vector<GaitRobot> gait_init_robots(const mpc_gait_t &p, int batch, const int32_t *mirror) {
  std::vector<GaitRobot> rs(batch);
  for (int b = 0; b < batch; b++) {
    for (int i = 0; i < 12; i++) { rs[b].start_l[i] = rs[b].final_l[i] = rs[b].next_l[i] = p.lf0[i]; rs[b].start_r[i] = rs[b].final_r[i] = rs[b].next_r[i] = p.rf0[i]; }
    rs[b].mirror = mirror ? (mirror[b] != 0) : 0; rs[b].pad_ = 0;
  }
  return rs;
}

} // namespace mpcdev
