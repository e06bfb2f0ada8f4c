// ORACLE (test infrastructure, not product code): normative CPU restatement of the time-parallel LQ solve
// (csrc/riccati_par.cuh).  The horizon is cut into L legs, each leg is solved as a function of the co-state theta at its end, a small serial consensus over the L boundaries finds the
// exact boundary value functions and states, and every leg is then re-solved exactly.  Fills the same LQSolution as the serial
// orc::riccati_solve (oracle/riccati.hpp), up to rounding.
//
// Value function of a leg at its start, as a function of the start state x and the end co-state theta (end state x'):
//   V(x; theta) = 1/2 x'P x + x'(p + Pi theta) + 1/2 theta'Psi theta + psi'theta,    x' = dV/dtheta = Pi'x + Psi theta + psi.
// The recursion is the serial one with the affine column p widened to [p | Pi] (1 + n columns) from (P, [p | Pi]) = (0, [0 | I])
// at the leg's end, plus the theta-only terms, which the serial recursion has no need to carry:
//   proximal step (Moreau envelope of the next value):  Psi -= mu_d Pi'Lambda^-1 Pi,  psi += (Lambda^-1 Pi)'(f - mu_d p)
//   control / multiplier step (saddle value 1/2 r'z):   Psi += gh_u,theta' ku_theta,  psi += gh_u,theta' ku
// Consensus, backward over the boundaries: with the exact (P, p) at the leg's end, theta = P x' + p, i.e.
//   (I - P Psi) theta = P (Pi'x + psi) + p   =>   theta = G x + h,   P_start = P_leg + Pi G (symmetrised),  p_start = p_leg + Pi h;
// forward: dx_0 = 0, theta_j = G_j x_{t_j} + h_j, x_{t_{j+1}} = Pi_j'x_{t_j} + Psi_j theta_j + psi_j.  P is never inverted.
#pragma once
#include "riccati.hpp"
#include <algorithm>

namespace orc {

// first knot of leg j of L over a horizon of T knots (csrc/riccati_par.cuh: leg_start)
inline int leg_start(int T, int L, int j) { return (int)((long long)j * T / L); }

// Backward recursion over knots k1 - 1 down to k0 from the value function (P, pa) at k1; pa holds na affine columns.  With
// na = 1 + n the theta terms accumulate into Psi / psi; with sol the knots' gains go to sol (na = 1).
inline void ric_backward(int n, int m, int nc, const LQKnot *kn, int k0, int k1, double mu_d, double mu, std::vector<double> &P, std::vector<double> &pa,
                         int na, double *Psi, double *psi, LQSolution *sol) {
  const int nz = n + m, s = m + nc, nr = 1 + n, nt = na - 1, nk = na + n;
  std::vector<double> G(n * n), Pt(n * n), ptl(n * na), AB(n * nz), W(n * nz), Hh(nz * nz), gh(nz * na), KK(s * s), ra(s * nk), Pn(n * n);
  std::vector<int> arow(nc);
  for (int k = k1 - 1; k >= k0; k--) {
    const LQKnot &q = kn[k];
    double T6[36];
    if (q.E6) { double Ei[36]; inv6(q.E6, Ei); for (int i = 0; i < 36; i++) T6[i] = -Ei[i]; }
    else for (int i = 0; i < 36; i++) T6[i] = (i % 7 == 0) ? 1.0 : 0.0;
    if (sol) std::memcpy(&sol->T6[(size_t)k * 36], T6, sizeof T6);
    if (n >= 6 && q.E6) {
      for (int i = 0; i < n; i++) { double r6[6]; for (int j = 0; j < 6; j++) { double t = 0; for (int l = 0; l < 6; l++) t += P[i * n + l] * T6[6 * l + j]; r6[j] = t; } for (int j = 0; j < 6; j++) P[i * n + j] = r6[j]; }
      for (int j = 0; j < n; j++) { double c6[6]; for (int i = 0; i < 6; i++) { double t = 0; for (int l = 0; l < 6; l++) t += T6[6 * l + i] * P[l * n + j]; c6[i] = t; } for (int i = 0; i < 6; i++) P[i * n + j] = c6[i]; }
      for (int c = 0; c < na; c++) { double c6[6]; for (int i = 0; i < 6; i++) { double t = 0; for (int l = 0; l < 6; l++) t += T6[6 * l + i] * pa[l * na + c]; c6[i] = t; } for (int i = 0; i < 6; i++) pa[i * na + c] = c6[i]; }
    }
    // Lambda = I + mu_d P;  Pt = Lambda^-1 P;  ptl = Lambda^-1 ([p | Pi] + P f e_0')
    for (int i = 0; i < n * n; i++) G[i] = mu_d * P[i];
    for (int i = 0; i < n; i++) G[i * n + i] += 1.0;
    chol_d(G.data(), n);
    Pt = P; chol_solve_d(G.data(), n, Pt.data(), n);
    for (int i = 0; i < n; i++) {
      for (int c = 0; c < na; c++) ptl[i * na + c] = pa[i * na + c];
      double t = pa[i * na]; for (int j = 0; j < n; j++) t += P[i * n + j] * q.f[j]; ptl[i * na] = t;
    }
    chol_solve_d(G.data(), n, ptl.data(), na);
    for (int a = 0; a < nt; a++) {
      double t = 0;
      for (int i = 0; i < n; i++) t += ptl[i * na + 1 + a] * (q.f[i] - mu_d * pa[i * na]);
      psi[a] += t;
      for (int b = 0; b < nt; b++) { double u = 0; for (int i = 0; i < n; i++) u += pa[i * na + 1 + a] * ptl[i * na + 1 + b]; Psi[a * nt + b] -= mu_d * u; }
    }
    // W = Pt [A B];  Hh = H + [A B]'W;  gh = [g | 0] + [A B]'ptl
    for (int i = 0; i < n; i++) { std::memcpy(&AB[i * nz], &q.A[i * n], sizeof(double) * n); std::memcpy(&AB[i * nz + n], &q.B[i * m], sizeof(double) * m); }
    std::fill(W.begin(), W.end(), 0.0);
    gemm_nn(n, nz, n, Pt.data(), AB.data(), W.data());
    std::memcpy(Hh.data(), q.H, sizeof(double) * nz * nz);
    gemm_tn(nz, nz, n, AB.data(), W.data(), Hh.data());
    for (int i = 0; i < nz; i++)
      for (int c = 0; c < na; c++) { double t = (c == 0) ? q.g[i] : 0.0; for (int l = 0; l < n; l++) t += AB[l * nz + i] * ptl[l * na + c]; gh[i * na + c] = t; }
    if (sol) {
      std::memcpy(&sol->W[(size_t)k * n * nz], W.data(), sizeof(double) * n * nz);
      for (int i = 0; i < n; i++) sol->pt[(size_t)k * n + i] = ptl[i * na];
    }
    // KKT over the active rows, right-hand side columns [affine (na) | x (n)]
    int nact = 0;
    for (int r = 0; r < nc; r++) {
      bool nzr = false;
      for (int j = 0; j < n && !nzr; j++) nzr = q.C[r * n + j] != 0.0;
      for (int j = 0; j < m && !nzr; j++) nzr = q.D[r * m + j] != 0.0;
      if (nzr) arow[nact++] = r;
    }
    const int sa = m + nact;
    std::fill(KK.begin(), KK.begin() + sa * sa, 0.0);
    for (int i = 0; i < m; i++) for (int j = 0; j < m; j++) KK[i * sa + j] = 0.5 * (Hh[(n + i) * nz + n + j] + Hh[(n + j) * nz + n + i]);
    for (int a = 0; a < nact; a++) { int r = arow[a]; for (int j = 0; j < m; j++) { KK[(m + a) * sa + j] = q.D[r * m + j]; KK[j * sa + m + a] = q.D[r * m + j]; } KK[(m + a) * sa + m + a] = -mu; }
    std::fill(ra.begin(), ra.begin() + sa * nk, 0.0);
    for (int i = 0; i < m; i++) { for (int c = 0; c < na; c++) ra[i * nk + c] = -gh[(n + i) * na + c]; for (int j = 0; j < n; j++) ra[i * nk + na + j] = -Hh[j * nz + n + i]; }
    for (int a = 0; a < nact; a++) { int r = arow[a]; ra[(m + a) * nk] = -q.d[r]; for (int j = 0; j < n; j++) ra[(m + a) * nk + na + j] = -q.C[r * n + j]; }
    ldlt(KK.data(), sa);
    ldlt_solve(KK.data(), sa, ra.data(), nk);
    for (int a = 0; a < nt; a++) {
      double t = 0;
      for (int i = 0; i < m; i++) t += gh[(n + i) * na + 1 + a] * ra[i * nk];
      psi[a] += t;
      for (int b = 0; b < nt; b++) { double u = 0; for (int i = 0; i < m; i++) u += gh[(n + i) * na + 1 + a] * ra[i * nk + 1 + b]; Psi[a * nt + b] += u; }
    }
    if (sol) {
      double *Kk = &sol->K[(size_t)k * s * nr];
      for (int i = 0; i < s * nr; i++) Kk[i] = 0.0;
      for (int i = 0; i < m; i++) { Kk[i * nr] = ra[i * nk]; for (int j = 0; j < n; j++) Kk[i * nr + 1 + j] = ra[i * nk + na + j]; }
      for (int r = 0; r < nc; r++) Kk[(m + r) * nr] = q.d[r] / mu;
      for (int a = 0; a < nact; a++) { double *row = &Kk[(m + arow[a]) * nr]; row[0] = ra[(m + a) * nk]; for (int j = 0; j < n; j++) row[1 + j] = ra[(m + a) * nk + na + j]; }
    }
    // P = Qh + Sh Ku + C'Kv (symmetrised);  [p | Pi] = gh + Sh [ku | Ku_theta] + C'[kv | Kv_theta]
    for (int i = 0; i < n; i++) {
      for (int c = 0; c < na; c++) {
        double t = gh[i * na + c];
        for (int l = 0; l < m; l++) t += Hh[i * nz + n + l] * ra[l * nk + c];
        for (int a = 0; a < nact; a++) t += q.C[arow[a] * n + i] * ra[(m + a) * nk + c];
        pa[i * na + c] = t;
      }
      for (int j = 0; j < n; j++) {
        double t = Hh[i * nz + j];
        for (int l = 0; l < m; l++) t += Hh[i * nz + n + l] * ra[l * nk + na + j];
        for (int a = 0; a < nact; a++) t += q.C[arow[a] * n + i] * ra[(m + a) * nk + na + j];
        Pn[i * n + j] = t;
      }
    }
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) P[i * n + j] = 0.5 * (Pn[i * n + j] + Pn[j * n + i]);
  }
}

// Solve A X = B in place (A: n x n general, B: n x nrhs), Gaussian elimination with partial pivoting
inline void lu_solve(double *A, int n, double *B, int nrhs) {
  for (int c = 0; c < n; c++) {
    int piv = c;
    for (int r = c + 1; r < n; r++) if (std::fabs(A[r * n + c]) > std::fabs(A[piv * n + c])) piv = r;
    if (piv != c) { for (int j = 0; j < n; j++) std::swap(A[c * n + j], A[piv * n + j]); for (int j = 0; j < nrhs; j++) std::swap(B[c * nrhs + j], B[piv * nrhs + j]); }
    const double d = 1.0 / A[c * n + c];
    for (int r = c + 1; r < n; r++) {
      const double l = A[r * n + c] * d;
      if (l == 0.0) continue;
      for (int j = c + 1; j < n; j++) A[r * n + j] -= l * A[c * n + j];
      for (int j = 0; j < nrhs; j++) B[r * nrhs + j] -= l * B[c * nrhs + j];
    }
  }
  for (int c = n - 1; c >= 0; c--) {
    for (int j = 0; j < nrhs; j++) {
      double t = B[c * nrhs + j];
      for (int l = c + 1; l < n; l++) t -= A[c * n + l] * B[l * nrhs + j];
      B[c * nrhs + j] = t / A[c * n + c];
    }
  }
}

inline void riccati_solve_par(int n, int m, int nc, int T, const LQKnot *kn, const double *HT, int ldh, const double *gT, const double *CT,
                              const double *dT, int nct, double mu_d, double mu, int L, LQSolution &sol) {
  const int nz = n + m, s = m + nc, nr = 1 + n, na = 1 + n;
  sol.n = n; sol.m = m; sol.nc = nc; sol.T = T; sol.nct = nct;
  sol.K.assign((size_t)T * s * nr, 0.0); sol.W.assign((size_t)T * n * nz, 0.0); sol.pt.assign((size_t)T * n, 0.0); sol.T6.assign((size_t)T * 36, 0.0);
  sol.dxs.assign((size_t)(T + 1) * n, 0.0); sol.dus.assign((size_t)T * m, 0.0); sol.dvs.assign((size_t)(T + 1) * nc, 0.0); sol.dlams.assign((size_t)(T + 1) * n, 0.0);
  std::vector<double> PT(n * n), pT(n);
  for (int i = 0; i < n; i++) { pT[i] = gT[i]; for (int j = 0; j < n; j++) PT[i * n + j] = HT[i * ldh + j]; }
  for (int r = 0; r < nct; r++)
    for (int i = 0; i < n; i++) { double c = CT[r * n + i] / mu; if (c == 0.0) continue; pT[i] += c * dT[r]; for (int j = 0; j < n; j++) PT[i * n + j] += c * CT[r * n + j]; }
  sol.PT = PT; sol.pT = pT;
  // A. every leg but the last as a function of its end co-state; the last leg from the terminal value function
  std::vector<std::vector<double>> VP(L), Vp(L), Psi(L), psi(L);
  for (int j = 0; j < L; j++) {
    const int k0 = leg_start(T, L, j), k1 = leg_start(T, L, j + 1);
    if (j + 1 < L) {
      VP[j].assign(n * n, 0.0); Vp[j].assign(n * na, 0.0); Psi[j].assign(n * n, 0.0); psi[j].assign(n, 0.0);
      for (int i = 0; i < n; i++) Vp[j][i * na + 1 + i] = 1.0;
      ric_backward(n, m, nc, kn, k0, k1, mu_d, mu, VP[j], Vp[j], na, Psi[j].data(), psi[j].data(), nullptr);
    } else {
      VP[j] = PT; Vp[j] = pT;
      ric_backward(n, m, nc, kn, k0, k1, mu_d, mu, VP[j], Vp[j], 1, nullptr, nullptr, nullptr);
    }
  }
  // B. consensus: exact value functions at the boundaries (backward), boundary states (forward)
  std::vector<std::vector<double>> SP(L), Sp(L), Gh(L), xb(L);
  std::vector<double> Pc = VP[L - 1], pc = Vp[L - 1], Mm(n * n);
  for (int j = L - 2; j >= 0; j--) {
    SP[j] = Pc; Sp[j] = pc; // exact value function at t_{j+1}: the seed of leg j
    const std::vector<double> &Pi = Vp[j], &Ps = Psi[j], &ps = psi[j];
    Gh[j].assign(n * (n + 1), 0.0);
    for (int i = 0; i < n; i++) {
      for (int b = 0; b < n; b++) {
        double t = (i == b) ? 1.0 : 0.0, u = 0;
        for (int a = 0; a < n; a++) { t -= Pc[i * n + a] * Ps[a * n + b]; u += Pc[i * n + a] * Pi[b * na + 1 + a]; }
        Mm[i * n + b] = t; Gh[j][i * (n + 1) + b] = u;
      }
      double u = pc[i];
      for (int a = 0; a < n; a++) u += Pc[i * n + a] * ps[a];
      Gh[j][i * (n + 1) + n] = u;
    }
    lu_solve(Mm.data(), n, Gh[j].data(), n + 1);
    std::vector<double> Pq(n * n);
    for (int i = 0; i < n; i++) {
      for (int c = 0; c <= n; c++) {
        double t = (c < n) ? VP[j][i * n + c] : Vp[j][i * na];
        for (int a = 0; a < n; a++) t += Pi[i * na + 1 + a] * Gh[j][a * (n + 1) + c];
        if (c < n) Pq[i * n + c] = t; else pc[i] = t;
      }
    }
    for (int i = 0; i < n; i++) for (int c = 0; c < n; c++) Pc[i * n + c] = 0.5 * (Pq[i * n + c] + Pq[c * n + i]);
  }
  sol.P0 = Pc; sol.p0 = pc;
  xb[0].assign(n, 0.0);
  for (int j = 0; j + 1 < L; j++) {
    std::vector<double> th(n);
    xb[j + 1].assign(n, 0.0);
    for (int a = 0; a < n; a++) { double t = Gh[j][a * (n + 1) + n]; for (int b = 0; b < n; b++) t += Gh[j][a * (n + 1) + b] * xb[j][b]; th[a] = t; }
    for (int a = 0; a < n; a++) {
      double t = psi[j][a];
      for (int i = 0; i < n; i++) t += Vp[j][i * na + 1 + a] * xb[j][i];
      for (int b = 0; b < n; b++) t += Psi[j][a * n + b] * th[b];
      xb[j + 1][a] = t;
    }
  }
  // C. exact re-solve of every leg from its seed, forward from its boundary state
  std::vector<double> z(nz), tmp(n), dx(n);
  for (int j = 0; j < L; j++) {
    const int k0 = leg_start(T, L, j), k1 = leg_start(T, L, j + 1);
    std::vector<double> P = (j + 1 < L) ? SP[j] : PT, p = (j + 1 < L) ? Sp[j] : pT;
    ric_backward(n, m, nc, kn, k0, k1, mu_d, mu, P, p, 1, nullptr, nullptr, &sol);
    if (j == 0) for (int i = 0; i < n; i++) sol.dlams[i] = -p[i];
    dx = xb[j];
    for (int k = k0; k < k1; k++) {
      const double *Kk = &sol.K[(size_t)k * s * nr];
      for (int i = 0; i < s; i++) {
        double t = Kk[i * nr]; for (int c = 0; c < n; c++) t += Kk[i * nr + 1 + c] * dx[c];
        if (i < m) sol.dus[(size_t)k * m + i] = t; else sol.dvs[(size_t)k * nc + i - m] = t;
      }
      for (int c = 0; c < n; c++) z[c] = dx[c];
      for (int c = 0; c < m; c++) z[n + c] = sol.dus[(size_t)k * m + c];
      const double *Wk = &sol.W[(size_t)k * n * nz];
      double *dl = &sol.dlams[(size_t)(k + 1) * n], *dxn = &sol.dxs[(size_t)(k + 1) * n];
      for (int i = 0; i < n; i++) {
        double t = sol.pt[(size_t)k * n + i], a = kn[k].f[i];
        for (int c = 0; c < nz; c++) t += Wk[i * nz + c] * z[c];
        for (int c = 0; c < n; c++) a += kn[k].A[i * n + c] * z[c];
        for (int c = 0; c < m; c++) a += kn[k].B[i * m + c] * z[n + c];
        dl[i] = t; tmp[i] = a - mu_d * t;
      }
      const double *T6 = &sol.T6[(size_t)k * 36];
      for (int i = 0; i < n; i++) {
        if (i < 6 && n >= 6 && kn[k].E6) { double t = 0; for (int l = 0; l < 6; l++) t += T6[6 * i + l] * tmp[l]; dxn[i] = t; } else dxn[i] = tmp[i];
      }
      for (int c = 0; c < n; c++) dx[c] = dxn[c];
    }
  }
  for (int r = 0; r < nct; r++) { double t = dT[r]; for (int c = 0; c < n; c++) t += CT[r * n + c] * sol.dxs[(size_t)T * n + c]; sol.dvs[(size_t)T * nc + r] = t / mu; }
}

} // namespace orc
