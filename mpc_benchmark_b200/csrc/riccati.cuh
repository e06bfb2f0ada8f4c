// Batched proximal Riccati (backward + forward) — one CTA per MPC instance, stage matrices in shared memory.
//
// Replaces aligator::gar::ProximalRiccatiSolver::backward/forward, reached from SolverProxDDP.run
// (selected at fulldynamic_talos.py:383; kinodynamic_talos.py:289; centroidal_talos.py:274).
// Recursion: SURVEY App. A6 (dual-regularised LQ, E normalised through T6 = -E6^-1).  Differences from the
// textbook dense form, all exact algebra:
//   * only ACTIVE constraint rows enter the KKT (the evaluation kernel compacts them); inactive rows decouple
//     to dv = dbar/mu;
//   * the quasi-definite KKT [R D'; D -mu I] is solved by block elimination: Cholesky(R), then Cholesky of the
//     Schur complement mu I + D R^-1 D' (both SPD) — no condensing into R + D'D/mu;
//   * the forward pass reuses W = Pt [A B] and pt stored by the backward pass: dlam' = W z + pt,
//     dx' = T6 (A dx + B du + fbar - mu_d dlam').
#pragma once
#include "dev_common.cuh"

namespace mpcdev {

// ------------------------------------------------------------------ block-cooperative dense helpers
// C (M x N, ldc) = beta*C + A^T B  with A (K x M, lda), B (K x N, ldb)        [TA = true]
// C (M x N, ldc) = beta*C + A   B  with A (M x K, lda), B (K x N, ldb)        [TA = false]
template <bool TA> HD void gemm_par(int M, int N, int K, const double *A, int lda, const double *B, int ldb, double *C, int ldc, double beta) {
  const int tm = (M + 3) / 4, tn = (N + 3) / 4;
  PAR_FOR(t, tm * tn) {
    int i0 = (t / tn) * 4, j0 = (t % tn) * 4;
    double acc[4][4];
    for (int a = 0; a < 4; a++) for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
    int mi = M - i0 < 4 ? M - i0 : 4, nj = N - j0 < 4 ? N - j0 : 4;
    if (mi == 4 && nj == 4) {
      for (int k = 0; k < K; k++) {
        double av[4], bv[4];
        for (int a = 0; a < 4; a++) av[a] = TA ? A[k * lda + i0 + a] : A[(i0 + a) * lda + k];
        for (int b = 0; b < 4; b++) bv[b] = B[k * ldb + j0 + b];
        for (int a = 0; a < 4; a++) for (int b = 0; b < 4; b++) acc[a][b] += av[a] * bv[b];
      }
    } else {
      for (int k = 0; k < K; k++)
        for (int a = 0; a < mi; a++) {
          double av = TA ? A[k * lda + i0 + a] : A[(i0 + a) * lda + k];
          for (int b = 0; b < nj; b++) acc[a][b] += av * B[k * ldb + j0 + b];
        }
    }
    for (int a = 0; a < mi; a++)
      for (int b = 0; b < nj; b++) { double *c = &C[(i0 + a) * ldc + j0 + b]; *c = (beta == 0.0 ? 0.0 : beta * *c) + acc[a][b]; }
  }
  SYNC();
}

// per-instance pointers (all device/global unless noted)
struct RiccatiIO {
  int T;
  double mu_d, mu;
  // LQ data written by the evaluation kernel, per knot k (k = T: terminal)
  const double *AB;      // [T][N][NZ]
  const double *H;       // [T+1][NZ][NZ]
  const double *g;       // [T+1][NZ]   Lagrangian gradient (q, r)
  const double *fbar;    // [T][N]
  const double *T6;      // [T][36]
  const double *CDact;   // [T+1][NC][NZ]  compacted active rows
  const double *dbar;    // [T+1][NC]      all rows
  const int32_t *nca;    // [T+1]
  const int32_t *act_idx;// [T+1][NC]
  // for the directional derivative of the merit function
  const double *lxu;     // [T+1][NZ] cost gradient
  const double *vplus, *v;   // [T+1][NC]
  const double *lplus, *lam; // [T+1][N]  (index k+1 belongs to dynamics k)
  // outputs
  double *W, *pt;        // [T][N][NZ] (fast kernels: [T][N][round8(NZ)], column NZ = pt), [T][N]
  double *K;             // [T][M+NC][1+N]   rows 0..M-1: [ku|Ku]; then compact active [kv|Kv]
  double *Kfb;           // [T][M][N]        controlFeedbacks()
  double *dxs, *dus, *dvs, *dlams; // [T+1][N], [T][M], [T+1][NC], [T+1][N]
  double *dphi;          // scalar
  double *scratch;       // per-instance global block for the KKT buffers of knots whose active rows exceed the shared-memory carving
  double *phase_out;     // optional 16 per-phase cycle counters (MPC_PHASE_TIMING builds), else nullptr
  // SEEDED solves (one leg of the time-parallel solve, riccati_par.cuh): knots [k0, k1) only, backward from the value function
  // (seedP, seedp) at k1 (nullptr: the terminal knot, k1 = T), forward from dx0 at k0
  int k0, k1;
  const double *seedP, *seedp, *dx0;
};

// ------------------------------------------------------------------ steps shared by the Riccati kernels (riccati_instance,
// riccati_instance_fast, ric_leg_param); they differ only in leading dimensions and buffer placement
// terminal value function: P = H_T[xx] + C'C/mu (leading dimension ldp), p = g_T[x] + C'd/mu (stride ps)
template <int N, int M, int NC> HD void ric_terminal_value(const RiccatiIO &io, double *P, int ldp, double *p, int ps) {
  constexpr int NZ = N + M;
  const int T = io.T;
  const double mu = io.mu;
  const double *HT = io.H + (size_t)T * NZ * NZ, *gT = io.g + (size_t)T * NZ;
  const int nca = io.nca[T];
  const double *CT = io.CDact + (size_t)T * NC * NZ, *dT = io.dbar + (size_t)T * NC;
  const int32_t *ai = io.act_idx + (size_t)T * NC;
  PAR_FOR(e, N * N) {
    int i = e / N, j = e % N;
    double s = HT[i * NZ + j];
    for (int r = 0; r < nca; r++) s += CT[r * NZ + i] * CT[r * NZ + j] / mu;
    P[i * ldp + j] = s;
  }
  PAR_FOR(i, N) {
    double s = gT[i];
    for (int r = 0; r < nca; r++) s += CT[r * NZ + i] * dT[ai[r]] / mu;
    p[i * ps] = s;
  }
}

// value function the backward sweep starts from: the seed (RiccatiIO::seedP) of a seeded leg, else the terminal value function
template <int N, int M, int NC> HD void ric_start_value(const RiccatiIO &io, bool seeded, double *P, int ldp, double *p) {
  if (seeded) {
    PAR_FOR(e, N * N) P[(e / N) * ldp + e % N] = io.seedP[e];
    PAR_FOR(i, N) p[i] = io.seedp[i];
    SYNC();
  } else {
    ric_terminal_value<N, M, NC>(io, P, ldp, p, 1);
    SYNC();
  }
}

// KKT by block elimination, after Z (M rows, leading dimension ldz) <- R^-1 [gh_u (na columns) | Sh' (N) | D' (nca)], nk = na + N:
// Schur complement Sg = mu I + D Z_D;  right-hand side Kv = [dbar | 0 | C] - D Z[:, 0:nk] (nca x nk).  CD: the active rows (NZ wide).
// THETA: na may exceed 1 (the co-state columns of ric_leg_param); the serial kernels pass na = 1
template <int N, int M, bool THETA = false>
HD void ric_kkt_schur(int nca, int na, int nk, double mu, const double *CD, const double *dbr, const double *Z, int ldz, double *Sg, double *Kv) {
  constexpr int NZ = N + M;
  PAR_FOR(e, nca * nca) {
    int r = e / nca, c = e % nca;
    double s = (r == c) ? mu : 0.0;
    for (int l = 0; l < M; l++) s += CD[r * NZ + N + l] * Z[l * ldz + nk + c];
    Sg[e] = s;
  }
  PAR_FOR(e, nca * nk) {
    int r = e / nk, c = e % nk;
    double s = (c == 0) ? dbr[r] : ((THETA && c < na) ? 0.0 : CD[r * NZ + c - na]);
    for (int l = 0; l < M; l++) s -= CD[r * NZ + N + l] * Z[l * ldz + c];
    Kv[e] = s;
  }
  SYNC();
}
// ... then, once Kv <- Sg^-1 Kv:  [ku | Ku] = -Z0 - Z_D Kv  (into Z0's place)
template <int M> HD void ric_kkt_ku(int nca, int nk, double *Z, int ldz, const double *Kv) {
  PAR_FOR(e, M * nk) {
    int i = e / nk, c = e % nk;
    double s = -Z[i * ldz + c];
    for (int r = 0; r < nca; r++) s -= Z[i * ldz + nk + r] * Kv[r * nk + c];
    Z[i * ldz + c] = s;
  }
  SYNC();
}

// store the gains of knot k: rows 0..M-1 = [ku | Ku] (and Ku into Kfb), rows M.. = [kv | Kv] (active rows, compact)
template <int N, int M, int NC> HD void ric_store_gains(const RiccatiIO &io, int k, const double *Z, int ldz, const double *Kv, int nca) {
  constexpr int NR = 1 + N, S = M + NC;
  double *gK = io.K + (size_t)k * S * NR;
  PAR_FOR(e, M * NR) { int i = e / NR, c = e % NR; double v = Z[i * ldz + c]; gK[e] = v; if (c > 0) io.Kfb[((size_t)k * M + i) * N + c - 1] = v; }
  PAR_FOR(e, nca * NR) gK[M * NR + e] = Kv[e];
}

// forward sweep start: dx = dx0 of a SEEDED leg, else 0 (force_initial_condition, fulldynamic_talos.py:384); knot k0 = 0 also writes
// dxs_0 and dlams_0 = -p
template <int N, bool SEEDED> HD void ric_forward_start(const RiccatiIO &io, int K0, const double *p, double *dx) {
  if (SEEDED) {
    PAR_FOR(i, N) { dx[i] = io.dx0[i]; if (K0 == 0) { io.dxs[i] = io.dx0[i]; io.dlams[i] = -p[i]; } }
  } else PAR_FOR(i, N) { dx[i] = 0.0; io.dxs[i] = 0.0; io.dlams[i] = -p[i]; }
}

template <int N, int M, int NC> constexpr int riccati_smem_doubles() {
  constexpr int NZ = N + M, NR = 1 + N;
  constexpr int phase1 = 2 * N * N + 2 * N * NZ;
  constexpr int phase2 = NC * NZ + NC * NC + M * (NR + NC) + NC * NR + M * M;
  return NZ * NZ + (phase1 > phase2 ? phase1 : phase2) + 8 * NZ + 36 + 2 * NC + 512 + 64 * ((NC + 7) / 8 + (N + 7) / 8) + 16;
}

// Backward + forward sweep for one instance.  ws: riccati_smem_doubles<N,M,NC>() doubles of shared memory.
// LIE6: the first 6 state coordinates live on SE(3) (E-normalisation by T6); false for vector-space models (centroidal: T6 = I)
// SEEDED: solve the knots [io.k0, io.k1) only (see RiccatiIO).  dxs / dlams of knot k0 are written by leg 0 only, the terminal knot's
// rows by the last leg only; dphi receives the leg's partial.
template <int N, int M, int NC, bool LIE6 = true, bool SEEDED = false> HD void riccati_instance(const RiccatiIO &io, double *ws) {
  constexpr int NZ = N + M, NR = 1 + N, S = M + NC;
  const int T = io.T;
  const int K0 = SEEDED ? io.k0 : 0, K1 = SEEDED ? io.k1 : T;
  const bool seeded = SEEDED && io.seedP != nullptr, last = !SEEDED || K1 == T;
  const double mu = io.mu, mu_d = io.mu_d;
  // ---- carve shared memory
  double *H = ws;                       // NZ*NZ; its [0:N,0:N] block carries the value-function Hessian between knots
  double *U0 = H + NZ * NZ;             // union region
  double *P = U0, *G = P + N * N, *AB = G + N * N, *W = AB + N * NZ;                                       // phase 1
  double *CD = U0, *Sg = CD + NC * NZ, *Z = Sg + NC * NC, *Kv = Z + M * (NR + NC), *Rh = Kv + NC * NR;     // phase 2
  constexpr int phase1 = 2 * N * N + 2 * N * NZ;
  constexpr int phase2 = NC * NZ + NC * NC + M * (NR + NC) + NC * NR + M * M;
  double *vec = U0 + (phase1 > phase2 ? phase1 : phase2);
  double *p = vec, *pt = p + NZ, *gh = pt + NZ, *fb = gh + NZ, *tmp = fb + NZ, *dx = tmp + NZ, *z = dx + NZ, *dl = z + NZ;
  double *T6 = dl + NZ, *dbr = T6 + 36, *dva = dbr + NC, *red = dva + NC, *dinv = red + 512;
  ric_start_value<N, M, NC>(io, seeded, H, NZ, p);
  for (int k = K1 - 1; k >= K0; k--) {
    const double *gAB = io.AB + (size_t)k * N * NZ, *gH = io.H + (size_t)k * NZ * NZ;
    const int nca = io.nca[k];
    if (k >= 2) { // the loads below are on the knot's critical path: pull the blocks of knot k - 2 from HBM into L2 now
      PREFETCH_LINES(io.AB + (size_t)(k - 2) * N * NZ, N * NZ * 8); PREFETCH_LINES(io.H + (size_t)(k - 2) * NZ * NZ, NZ * NZ * 8);
      PREFETCH_LINES(io.g + (size_t)(k - 2) * NZ, NZ * 8); PREFETCH_LINES(io.fbar + (size_t)(k - 2) * N, N * 8);
    }
    // 1. load; P <- T' P T, p <- T' p
    PAR_FOR(e, N * N) { int i = e / N, j = e % N; P[e] = H[i * NZ + j]; }
    if (LIE6) PAR_FOR(e, 36) T6[e] = io.T6[(size_t)k * 36 + e];
    PAR_FOR(i, N) fb[i] = io.fbar[(size_t)k * N + i];
    PAR_FOR(e, N * NZ) AB[e] = gAB[e];
    SYNC();
    if (LIE6 && N >= 6) {
      PAR_FOR(e, N * 6) { int i = e / 6, j = e % 6; double s = 0; for (int l = 0; l < 6; l++) s += P[i * N + l] * T6[6 * l + j]; W[e] = s; }
      SYNC();
      PAR_FOR(e, N * 6) { int i = e / 6, j = e % 6; P[i * N + j] = W[e]; }
      SYNC();
      PAR_FOR(e, 6 * N) { int i = e / N, j = e % N; double s = 0; for (int l = 0; l < 6; l++) s += T6[6 * l + i] * P[l * N + j]; W[e] = s; }
      PAR_FOR(i, 6) { double s = 0; for (int l = 0; l < 6; l++) s += T6[6 * l + i] * p[l]; tmp[i] = s; }
      SYNC();
      PAR_FOR(e, 6 * N) P[e] = W[e];
      PAR_FOR(i, 6) p[i] = tmp[i];
      SYNC();
    }
    // 2. G = chol(I + mu_d P);  pt = G^-T G^-1 (p + P f);  P <- Pt = G^-T G^-1 P
    PAR_FOR(e, N * N) G[e] = mu_d * P[e] + ((e / N == e % N) ? 1.0 : 0.0);
    PAR_FOR(i, N) { double s = p[i]; for (int j = 0; j < N; j++) s += P[i * N + j] * fb[j]; pt[i] = s; }
    SYNC();
    if (N <= 12) small_spd_solve<(N <= 12 ? N : 1)>(G, N, P, N, N, pt, 1, 1);
    else {
      chol_blocked(G, N, N, dinv);
      trsm_blocked(G, N, N, dinv, P, N, N);
      trsm_blocked(G, N, N, dinv, pt, 1, 1);
    }
    // 3. W = Pt [A B];  H = H_k + [A B]' W;  gh = g + [A B]' pt
    PAR_FOR(e, NZ * NZ) H[e] = gH[e];
    gemm_par<false>(N, NZ, N, P, N, AB, NZ, W, NZ, 0.0);
    gemm_par<true>(NZ, NZ, N, AB, NZ, W, NZ, H, NZ, 1.0);
    PAR_FOR(i, NZ) { double s = io.g[(size_t)k * NZ + i]; for (int l = 0; l < N; l++) s += AB[l * NZ + i] * pt[l]; gh[i] = s; }
    PAR_FOR(e, N * NZ) io.W[(size_t)k * N * NZ + e] = W[e];
    PAR_FOR(i, N) io.pt[(size_t)k * N + i] = pt[i];
    SYNC();
    // 4. KKT by block elimination (phase-2 buffers alias P/G/AB/W, all dead now)
    const int ncol = NR + nca; // Z columns: [rh | Sh' | D']
    const double *gCD = io.CDact + (size_t)k * NC * NZ;
    const int32_t *ai = io.act_idx + (size_t)k * NC;
    PAR_FOR(e, nca * NZ) CD[e] = gCD[e];
    PAR_FOR(r, nca) dbr[r] = io.dbar[(size_t)k * NC + ai[r]];
    PAR_FOR(e, M * M) { int i = e / M, j = e % M; Rh[e] = 0.5 * (H[(N + i) * NZ + N + j] + H[(N + j) * NZ + N + i]); }
    SYNC();
    PAR_FOR(e, M * ncol) {
      int i = e / ncol, c = e % ncol;
      Z[i * ncol + c] = (c == 0) ? gh[N + i] : (c < NR ? H[(c - 1) * NZ + N + i] : CD[(c - NR) * NZ + N + i]);
    }
    SYNC();
    if (M <= 12) small_spd_solve<(M <= 12 ? M : 1)>(Rh, M, Z, ncol, ncol, nullptr, 0, 0);
    else {
      chol_blocked(Rh, M, M, dinv);
      trsm_blocked(Rh, M, M, dinv, Z, ncol, ncol);
    }
    ric_kkt_schur<N, M>(nca, 1, NR, mu, CD, dbr, Z, ncol, Sg, Kv);
    if (nca > 0) { chol_blocked(Sg, nca, nca, dinv); trsm_blocked(Sg, nca, nca, dinv, Kv, NR, NR); }
    ric_kkt_ku<M>(nca, NR, Z, ncol, Kv);
    ric_store_gains<N, M, NC>(io, k, Z, ncol, Kv, nca);
    // 5. P = Qh + Sh Ku + C' Kv, p = qh + Sh ku + C' kv : in place in H[0:N,0:N] / p, then symmetrise
    PAR_FOR(e, N * NR) {
      int i = e / NR, c = e % NR;
      double s = (c == 0) ? gh[i] : H[i * NZ + c - 1];
      for (int l = 0; l < M; l++) s += H[i * NZ + N + l] * Z[l * ncol + c];
      for (int r = 0; r < nca; r++) s += CD[r * NZ + i] * Kv[r * NR + c];
      if (c == 0) p[i] = s; else H[i * NZ + c - 1] = s;
    }
    SYNC();
    PAR_FOR(e, N * N) {
      int i = e / N, j = e % N;
      if (i < j) { double s = 0.5 * (H[i * NZ + j] + H[j * NZ + i]); H[i * NZ + j] = s; H[j * NZ + i] = s; }
    }
    SYNC();
  }
  // ---- forward sweep, dx0 = 0 (force_initial_condition, fulldynamic_talos.py:384)
  double acc = 0.0; // per-thread partial of the merit directional derivative
  ric_forward_start<N, SEEDED>(io, K0, p, dx);
  SYNC();
  for (int k = K0; k <= (last ? T : K1 - 1); k++) {
    const int nca = io.nca[k];
    const int32_t *ai = io.act_idx + (size_t)k * NC;
    const double *gdb = io.dbar + (size_t)k * NC, *gvp = io.vplus + (size_t)k * NC, *gv = io.v + (size_t)k * NC;
    double *gdv = io.dvs + (size_t)k * NC;
    if (k + 2 < T) {
      PREFETCH_LINES(io.K + (size_t)(k + 2) * S * NR, (M + io.nca[k + 2]) * NR * 8); PREFETCH_LINES(io.AB + (size_t)(k + 2) * N * NZ, N * NZ * 8);
      PREFETCH_LINES(io.W + (size_t)(k + 2) * N * NZ, N * NZ * 8);
    }
    if (k < T) {
      const double *gK = io.K + (size_t)k * S * NR;
      PAR_FOR(i, M + nca) {
        double s = gK[i * NR];
        for (int j = 0; j < N; j++) s += gK[i * NR + 1 + j] * dx[j];
        if (i < M) { z[N + i] = s; io.dus[(size_t)k * M + i] = s; } else dva[i - M] = s;
      }
      PAR_FOR(i, N) z[i] = dx[i];
      PAR_FOR(e, N * NZ) { AB[e] = io.AB[(size_t)k * N * NZ + e]; W[e] = io.W[(size_t)k * N * NZ + e]; }
      if (LIE6) PAR_FOR(e, 36) T6[e] = io.T6[(size_t)k * 36 + e];
    } else {
      const double *CT = io.CDact + (size_t)T * NC * NZ;
      PAR_FOR(r, nca) { double s = gdb[ai[r]]; for (int j = 0; j < N; j++) s += CT[r * NZ + j] * dx[j]; dva[r] = s / mu; }
      PAR_FOR(i, N) z[i] = dx[i];
    }
    PAR_FOR(r, NC) gdv[r] = gdb[r] / mu; // inactive rows; active ones overwritten below
    SYNC();
    PAR_FOR(r, nca) gdv[ai[r]] = dva[r];
    // directional derivative terms of this knot
    PAR_FOR(i, (k < T ? NZ : N)) acc += io.lxu[(size_t)k * NZ + i] * z[i];
    PAR_FOR(r, nca) { int row = ai[r]; acc += (2.0 * gvp[row] - gv[row]) * (mu * dva[r] - gdb[row]) - gdb[row] * dva[r]; }
    PAR_FOR(r, NC) { // inactive rows: -dbar * dv = -dbar^2/mu
      bool active = false;
      for (int q = 0; q < nca; q++) active |= (ai[q] == r);
      if (!active) acc -= gdb[r] * gdb[r] / mu;
    }
    if (k == T) break;
    PAR_FOR(i, N) {
      double s = io.pt[(size_t)k * N + i], a = io.fbar[(size_t)k * N + i];
      for (int j = 0; j < NZ; j++) { s += W[i * NZ + j] * z[j]; a += AB[i * NZ + j] * z[j]; }
      dl[i] = s; tmp[i] = a - mu_d * s;
      io.dlams[(size_t)(k + 1) * N + i] = s;
      double fbi = io.fbar[(size_t)k * N + i], lp = io.lplus[(size_t)(k + 1) * N + i], lm = io.lam[(size_t)(k + 1) * N + i];
      acc += (2.0 * lp - lm) * (mu_d * s - fbi) - fbi * s;
    }
    SYNC();
    PAR_FOR(i, N) {
      double s;
      if (LIE6 && N >= 6 && i < 6) { s = 0; for (int l = 0; l < 6; l++) s += T6[6 * i + l] * tmp[l]; } else s = tmp[i];
      dx[i] = s; io.dxs[(size_t)(k + 1) * N + i] = s;
    }
    SYNC();
  }
  red[TID] = acc;
  SYNC();
  ONE_THREAD { double s = 0; for (int t = 0; t < NTHREADS; t++) s += red[t]; io.dphi[0] = s; }
  SYNC();
}

} // namespace mpcdev
