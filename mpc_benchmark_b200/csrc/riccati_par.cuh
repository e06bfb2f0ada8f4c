// Time-parallel proximal Riccati (aligator's LQ_SOLVER_PARALLEL): the horizon is cut into L legs, knots t_j <= k < t_{j+1}
// with t_j = leg_start(T, L, j); the last leg also owns the terminal knot.  Four phases, each a launch of its own:
//   A  every leg at once: the leg's value function at its start as a function of the start state x and of the co-state theta
//      at its end (ric_leg_param; the last leg: the exact recursion from the terminal value function);
//   B  one group per instance, serial over the L boundaries: the exact value function and state at every boundary (ric_consensus);
//   C  every leg at once: the model's own Riccati kernel re-solves the leg exactly, seeded with the boundary value function and
//      started from the boundary state (riccati_instance / riccati_instance_fast with SEEDED = true);
//   D  one group per instance: the merit derivative partials of the legs, summed in leg order.
// The per-instance critical path is ~T/L knots of A, L small steps of B and ~T/L knots of C instead of T knots.
//
// Leg value function, theta = co-state at the leg's end in the coordinates of dx (x' = end state):
//   V(x; theta) = 1/2 x'P x + x'(p + Pi theta) + 1/2 theta'Psi theta + psi'theta,    x' = dV/dtheta = Pi'x + Psi theta + psi.
// It is the serial recursion (riccati.cuh) from (P, [p | Pi]) = (0, [0 | I]) with the affine column widened to 1 + n columns (the E
// normalisation T6 and the KKT right-hand side treat the theta columns like the affine one), plus the theta-only terms:
//   proximal step (the Moreau envelope of the next value):  Psi -= mu_d Pi'Lambda^-1 Pi,  psi += (Lambda^-1 Pi)'(fbar - mu_d p)
//   control / multiplier step (the KKT saddle value):       Psi += gh_u,theta' ku_theta,  psi += gh_u,theta' ku
// (an empty leg would be Psi = -mu_d I, x' = x - mu_d theta).  Consensus, backward: given the exact (P, p) at t_{j+1}, the leg's
// co-state is theta = P x' + p, i.e.
//   (I - P Psi) theta = P (Pi'x + psi) + p   =>   theta = G x + h,   P(t_j) = P_leg + Pi G (symmetrised),   p(t_j) = p_leg + Pi h,
// the generalisation of Lambda = I + mu_d P; the system is solved by LU with partial pivoting, P is never inverted.  Forward:
// dx_0 = 0, theta_j = G_j dx_{t_j} + h_j, dx_{t_{j+1}} = Pi_j'dx_{t_j} + Psi_j theta_j + psi_j.
#pragma once
#include "riccati.cuh"

namespace mpcdev {

// first knot of leg j of L over a horizon of T knots: near-equal legs, every leg non-empty for L <= T
HDH int leg_start(int T, int L, int j) { return (int)((long long)j * T / L); }

template <int N, int M, int NC> struct LegLayout {
  static constexpr int NZ = N + M, NA = 1 + N, NK = NA + N + NC;
  static constexpr int NB = ((N > M ? (N > NC ? N : NC) : (M > NC ? M : NC)) + 7) / 8;
  // phase A output per (instance, leg): P | [p | Pi] (N x NA) | Psi | psi
  static constexpr int sum = 2 * N * N + N * NA + N;
  // phase A work space per (instance, leg), global memory (L2-resident at the batch sizes a latency-bound user runs)
  static constexpr int ws = 3 * N * N + 2 * N * NA + 2 * N * NZ + NZ * NZ + NZ * NA + M * NK + M * M + NC * NZ + NC * NC + NC * (NA + N) + 64 * NB + 36 + N + NC;
  // phase B / C / D per (instance, leg): seed P | seed p (exact value function at the leg's end) | start state | [G | h] | LU work | dphi
  static constexpr int buf = 2 * N * N + 2 * N + N * (N + 1) + 2;
  static constexpr int off_seedp = N * N, off_x = N * N + N, off_gh = N * N + 2 * N, off_lu = N * N + 2 * N + N * (N + 1), off_dphi = buf - 2;
};

// A: value function at the leg's start as a function of (x, theta) for knots [k0, k1) (last: exact, from the terminal knot)
template <int N, int M, int NC, bool LIE6> HD void ric_leg_param(const RiccatiIO &io, int k0, int k1, bool last, double *ws, double *sum) {
  using Lay = LegLayout<N, M, NC>;
  constexpr int NZ = Lay::NZ, NA = Lay::NA, NK = Lay::NK;
  const double mu = io.mu, mu_d = io.mu_d;
  const int na = last ? 1 : NA, nt = na - 1, nk = na + N;
  double *VP = sum, *pa = VP + N * N, *Psi = pa + N * NA, *psi = Psi + N * N; // pa: stride NA
  double *G = ws, *Pt = G + N * N, *Pn = Pt + N * N, *ptl = Pn + N * N, *tpa = ptl + N * NA, *AB = tpa + N * NA, *W = AB + N * NZ, *Hh = W + N * NZ;
  double *gh = Hh + NZ * NZ, *Z = gh + NZ * NA, *Rh = Z + M * NK, *CD = Rh + M * M, *Sg = CD + NC * NZ, *Kv = Sg + NC * NC, *dinv = Kv + NC * (NA + N);
  double *T6 = dinv + 64 * Lay::NB, *fb = T6 + 36, *dbr = fb + N; // ptl, gh, Kv: stride na / na / nk
  if (last) {
    ric_terminal_value<N, M, NC>(io, VP, N, pa, NA);
  } else {
    PAR_FOR(e, N * N) { VP[e] = 0.0; Psi[e] = 0.0; }
    PAR_FOR(e, N * NA) pa[e] = ((e % NA) == 1 + e / NA) ? 1.0 : 0.0;
    PAR_FOR(i, N) psi[i] = 0.0;
  }
  SYNC();
  for (int k = k1 - 1; k >= k0; k--) {
    const int nca = io.nca[k];
    // 1. load; P <- T'P T, [p | Pi] <- T'[p | Pi]
    if (LIE6) PAR_FOR(e, 36) T6[e] = io.T6[(size_t)k * 36 + e];
    PAR_FOR(i, N) fb[i] = io.fbar[(size_t)k * N + i];
    PAR_FOR(e, N * NZ) AB[e] = io.AB[(size_t)k * N * NZ + e];
    SYNC();
    if (LIE6 && N >= 6) {
      PAR_FOR(e, N * 6) { const int i = e / 6, j = e % 6; double s = 0; for (int l = 0; l < 6; l++) s += VP[i * N + l] * T6[6 * l + j]; Pn[e] = s; }
      SYNC();
      PAR_FOR(e, N * 6) { const int i = e / 6, j = e % 6; VP[i * N + j] = Pn[e]; }
      SYNC();
      PAR_FOR(e, 6 * N) { const int i = e / N, j = e % N; double s = 0; for (int l = 0; l < 6; l++) s += T6[6 * l + i] * VP[l * N + j]; Pn[e] = s; }
      PAR_FOR(e, 6 * na) { const int i = e / na, c = e % na; double s = 0; for (int l = 0; l < 6; l++) s += T6[6 * l + i] * pa[l * NA + c]; tpa[e] = s; }
      SYNC();
      PAR_FOR(e, 6 * N) VP[e] = Pn[e];
      PAR_FOR(e, 6 * na) { const int i = e / na, c = e % na; pa[i * NA + c] = tpa[e]; }
      SYNC();
    }
    // 2. Lambda = I + mu_d P = G G';  Pt = Lambda^-1 P;  ptl = Lambda^-1 ([p | Pi] + P fbar e_0')
    PAR_FOR(e, N * N) { G[e] = mu_d * VP[e] + ((e / N == e % N) ? 1.0 : 0.0); Pt[e] = VP[e]; }
    PAR_FOR(e, N * na) {
      const int i = e / na, c = e % na;
      double s = pa[i * NA + c];
      if (c == 0) for (int j = 0; j < N; j++) s += VP[i * N + j] * fb[j];
      ptl[e] = s;
    }
    SYNC();
    chol_blocked(G, N, N, dinv);
    trsm_blocked(G, N, N, dinv, Pt, N, N);
    trsm_blocked(G, N, N, dinv, ptl, na, na);
    PAR_FOR(e, nt * nt) { const int a = e / nt, b = e % nt; double u = 0; for (int i = 0; i < N; i++) u += pa[i * NA + 1 + a] * ptl[i * na + 1 + b]; Psi[a * N + b] -= mu_d * u; }
    PAR_FOR(a, nt) { double t = 0; for (int i = 0; i < N; i++) t += ptl[i * na + 1 + a] * (fb[i] - mu_d * pa[i * NA]); psi[a] += t; }
    // 3. W = Pt [A B];  Hh = H_k + [A B]'W;  gh = [g | 0] + [A B]'ptl
    PAR_FOR(e, NZ * NZ) Hh[e] = io.H[(size_t)k * NZ * NZ + e];
    gemm_par<false>(N, NZ, N, Pt, N, AB, NZ, W, NZ, 0.0);
    gemm_par<true>(NZ, NZ, N, AB, NZ, W, NZ, Hh, NZ, 1.0);
    PAR_FOR(e, NZ * na) {
      const int i = e / na, c = e % na;
      double s = (c == 0) ? io.g[(size_t)k * NZ + i] : 0.0;
      for (int l = 0; l < N; l++) s += AB[l * NZ + i] * ptl[l * na + c];
      gh[e] = s;
    }
    // 4. KKT by block elimination, Z columns [gh_u (na) | Sh' (N) | D' (nca)]
    const int ncol = nk + nca;
    const int32_t *ai = io.act_idx + (size_t)k * NC;
    PAR_FOR(e, nca * NZ) CD[e] = io.CDact[(size_t)k * NC * NZ + e];
    PAR_FOR(r, nca) dbr[r] = io.dbar[(size_t)k * NC + ai[r]];
    PAR_FOR(e, M * M) { const int i = e / M, j = e % M; Rh[e] = 0.5 * (Hh[(N + i) * NZ + N + j] + Hh[(N + j) * NZ + N + i]); }
    SYNC();
    PAR_FOR(e, M * ncol) {
      const int i = e / ncol, c = e % ncol;
      Z[e] = (c < na) ? gh[(N + i) * na + c] : (c < nk ? Hh[(c - na) * NZ + N + i] : CD[(c - nk) * NZ + N + i]);
    }
    SYNC();
    chol_blocked(Rh, M, M, dinv);
    trsm_blocked(Rh, M, M, dinv, Z, ncol, ncol);
    ric_kkt_schur<N, M, true>(nca, na, nk, mu, CD, dbr, Z, ncol, Sg, Kv);
    if (nca > 0) { chol_blocked(Sg, nca, nca, dinv); trsm_blocked(Sg, nca, nca, dinv, Kv, nk, nk); }
    ric_kkt_ku<M>(nca, nk, Z, ncol, Kv); // [ku | Ku_theta | Ku]
    PAR_FOR(e, nt * nt) { const int a = e / nt, b = e % nt; double u = 0; for (int i = 0; i < M; i++) u += gh[(N + i) * na + 1 + a] * Z[i * ncol + 1 + b]; Psi[a * N + b] += u; }
    PAR_FOR(a, nt) { double t = 0; for (int i = 0; i < M; i++) t += gh[(N + i) * na + 1 + a] * Z[i * ncol]; psi[a] += t; }
    // 5. P = Qh + Sh Ku + C'Kv (symmetrised);  [p | Pi] = gh_x + Sh [ku | Ku_theta] + C'[kv | Kv_theta]
    PAR_FOR(e, N * nk) {
      const int i = e / nk, c = e % nk;
      double s = (c < na) ? gh[i * na + c] : Hh[i * NZ + c - na];
      for (int l = 0; l < M; l++) s += Hh[i * NZ + N + l] * Z[l * ncol + c];
      for (int r = 0; r < nca; r++) s += CD[r * NZ + i] * Kv[r * nk + c];
      if (c < na) pa[i * NA + c] = s; else Pn[i * N + c - na] = s;
    }
    SYNC();
    PAR_FOR(e, N * N) { const int i = e / N, j = e % N; VP[e] = 0.5 * (Pn[i * N + j] + Pn[j * N + i]); }
    SYNC();
  }
}

// A X = B in place (A: n x n general, B: n x nrhs), Gaussian elimination with partial pivoting; sh: 1 double of shared memory
HD void lu_solve_par(double *A, int n, double *B, int nrhs, double *sh) {
  for (int c = 0; c < n; c++) {
    ONE_THREAD {
      int piv = c;
      for (int r = c + 1; r < n; r++) if (fabs(A[r * n + c]) > fabs(A[piv * n + c])) piv = r;
      sh[0] = (double)piv;
    }
    SYNC();
    const int piv = (int)sh[0];
    if (piv != c) {
      PAR_FOR(j, n + nrhs) {
        double *x = (j < n) ? A + c * n + j : B + c * nrhs + j - n, *y = (j < n) ? A + piv * n + j : B + piv * nrhs + j - n;
        const double t = *x; *x = *y; *y = t;
      }
      SYNC();
    }
    const int rem = n - c - 1, wd = rem + nrhs;
    PAR_FOR(e, rem * wd) {
      const int r = c + 1 + e / wd, q = e % wd;
      const double l = A[r * n + c] / A[c * n + c];
      if (q < rem) A[r * n + c + 1 + q] -= l * A[c * n + c + 1 + q];
      else B[r * nrhs + q - rem] -= l * B[c * nrhs + q - rem];
    }
    SYNC();
  }
  PAR_FOR(j, nrhs) {
    for (int c = n - 1; c >= 0; c--) {
      double t = B[c * nrhs + j];
      for (int l = c + 1; l < n; l++) t -= A[c * n + l] * B[l * nrhs + j];
      B[c * nrhs + j] = t / A[c * n + c];
    }
  }
  SYNC();
}

// B: exact value functions at the boundaries (backward) and the boundary states (forward) of one instance.  sum / buf: leg 0's
// phase-A summary / leg buffer, legs at strides ss / bs.  sh: >= N doubles of shared memory.
template <int N, int M, int NC> HD void ric_consensus(int L, const double *sum, size_t ss, double *buf, size_t bs, double *sh) {
  using Lay = LegLayout<N, M, NC>;
  constexpr int NA = Lay::NA;
  { // the last leg's start value function is exact: the seed of leg L - 2
    const double *s = sum + (size_t)(L - 1) * ss;
    double *b = buf + (size_t)(L - 2) * bs;
    PAR_FOR(e, N * N) b[e] = s[e];
    PAR_FOR(i, N) b[Lay::off_seedp + i] = s[N * N + i * NA];
  }
  SYNC();
  for (int j = L - 2; j >= 0; j--) {
    const double *s = sum + (size_t)j * ss, *VP = s, *pa = VP + N * N, *Psi = pa + N * NA, *psi = Psi + N * N;
    double *b = buf + (size_t)j * bs, *Pc = b, *pc = b + Lay::off_seedp, *Gh = b + Lay::off_gh, *Mm = b + Lay::off_lu;
    PAR_FOR(e, N * N) {
      const int i = e / N, c = e % N;
      double t = (i == c) ? 1.0 : 0.0, u = 0.0;
      for (int a = 0; a < N; a++) { t -= Pc[i * N + a] * Psi[a * N + c]; u += Pc[i * N + a] * pa[c * NA + 1 + a]; }
      Mm[e] = t; Gh[i * (N + 1) + c] = u;
    }
    PAR_FOR(i, N) { double u = pc[i]; for (int a = 0; a < N; a++) u += Pc[i * N + a] * psi[a]; Gh[i * (N + 1) + N] = u; }
    SYNC();
    lu_solve_par(Mm, N, Gh, N + 1, sh);
    if (j == 0) break;
    double *bo = buf + (size_t)(j - 1) * bs; // P(t_j) = P_leg + Pi G, p(t_j) = p_leg + Pi h: the seed of leg j - 1
    PAR_FOR(e, N * (N + 1)) {
      const int i = e / (N + 1), c = e % (N + 1);
      double t = (c < N) ? VP[i * N + c] : pa[i * NA];
      for (int a = 0; a < N; a++) t += pa[i * NA + 1 + a] * Gh[a * (N + 1) + c];
      if (c < N) Mm[i * N + c] = t; else bo[Lay::off_seedp + i] = t;
    }
    SYNC();
    PAR_FOR(e, N * N) { const int i = e / N, c = e % N; bo[e] = 0.5 * (Mm[i * N + c] + Mm[c * N + i]); }
    SYNC();
  }
  PAR_FOR(i, N) buf[Lay::off_x + i] = 0.0;
  SYNC();
  for (int j = 0; j + 1 < L; j++) {
    const double *s = sum + (size_t)j * ss, *pa = s + N * N, *Psi = pa + N * NA, *psi = Psi + N * N;
    const double *b = buf + (size_t)j * bs, *x = b + Lay::off_x, *Gh = b + Lay::off_gh;
    double *xn = buf + (size_t)(j + 1) * bs + Lay::off_x;
    PAR_FOR(a, N) { double t = Gh[a * (N + 1) + N]; for (int c = 0; c < N; c++) t += Gh[a * (N + 1) + c] * x[c]; sh[a] = t; }
    SYNC();
    PAR_FOR(a, N) {
      double t = psi[a];
      for (int i = 0; i < N; i++) t += pa[i * NA + 1 + a] * x[i];
      for (int c = 0; c < N; c++) t += Psi[a * N + c] * sh[c];
      xn[a] = t;
    }
    SYNC();
  }
}

} // namespace mpcdev
