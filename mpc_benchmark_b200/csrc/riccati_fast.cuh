// Proximal Riccati, tensor-core variant for state dimensions that are multiples of 8 (full / kinodynamic: n = 56).
// Same recursion and outputs as riccati_instance (riccati.cuh, SURVEY App. A6), plus the E normalisation by T6; what changes is
// HOW the dense work per knot is executed, all of it on the FP64 DMMA pipe out of shared memory (dmma.cuh):
//   Lambda = I + mu_d P = G G' (chol_mma),  [Pt | pt] = Lambda^-1 [P | pv] (trsm_mma, in place),  W = Pt [A B] (mma_tn_g),
//   H = H_k + [A B]' W (mma_sym_deferred),  and the value update P = H_xx + H_xu Ku (mma_tn)
// The padded control block of the KKT is factored and solved the same way (chol_mma, trsm_mma).  Leading dimensions are padded
// so that the DMMA fragment loads are bank-conflict free (RicFastLayout).
// Shared memory holds H, P and the factor; [A B]_k is bulk-copied into the H buffer while it is idle and W is staged behind it, so
// that both products read shared memory at a footprint (full dynamics: 114 KB per CTA) that lets TWO instances share an SM: one
// instance's serial pivot chains hide behind the other's products.
#pragma once
#include "dmma.cuh"
#include "riccati.cuh"

namespace mpcdev {

// optional per-phase cycle counters (thread 0 of the CTA handling instance 0), enabled with -DMPC_PHASE_TIMING
#if defined(MPC_PHASE_TIMING) && !defined(MPC_HOST_EMU)
#define PHASE_DECL long long ph_last = clock64(); long long ph_acc[32] = {0}
#define PHASE(i) do { SYNC(); if (threadIdx.x == 0) { long long t_ = clock64(); ph_acc[i] += t_ - ph_last; ph_last = t_; } } while (0)
#define PHASE_DUMP(ptr) do { if (threadIdx.x == 0 && (ptr)) for (int i_ = 0; i_ < 16; i_++) { (ptr)[i_] = (double)ph_acc[i_]; (ptr)[48 + i_] = (double)ph_acc[16 + i_]; } } while (0)
#else
#define PHASE_DECL
#define PHASE(i)
#define PHASE_DUMP(ptr)
#endif

template <int N, int M, int NC, int NCAP = NC> struct RicFastLayout {
  static constexpr int NZ = N + M, NR = 1 + N, S = M + NC;
  static constexpr int NBLK = N / 8;
  static constexpr int ZP = (NZ + 7) / 8 * 8;                       // padded n+m
  static constexpr int LDN = (N % 16 == 8) ? N : N + 8;             // ld of N x N buffers
  static constexpr int LDH = ZP;                                    // ld of the Hessian buffer
  static constexpr int LDW = ZP;                                    // ld of W in HBM: column NZ carries pt, the rest of the padding is zero
  static constexpr int LDZ = ZP + 4;                                // ld of [A B] and W staged in shared memory (over the idle H buffer): = 4 (mod 8) doubles, so the
                                                                    // 16 lanes of a half-warp fragment load (4 k-rows x 4 columns of 8 bytes) cover all 32 banks once
  static_assert(N * LDZ <= ZP * LDH && 2 * N * LDZ <= ZP * LDH + N * LDN, "[A B] must fit into the H buffer, W behind it up to the end of the factor");
  static constexpr int NQ_SYM = ((ZP / 8 + 1) / 2) * ((ZP / 8 + 1) / 2 + 1) / 2; // 16 x 16 blocks of the upper block triangle of H
  static constexpr int MAXQ = (NQ_SYM + 3) / 4;                    // per warp, for CTAs of at least 4 warps
  static constexpr int MR = (M + 7) / 8 * 8;                        // control block padded to whole 8 x 8 tiles (identity / zero padding)
  static constexpr int LDR = (MR % 16 == 8) ? MR : MR + 8;          // ld of the padded R^ buffer
  // phase-2 (KKT) buffers [Z | Kv | Rh | CD | Sg] are carved per knot for the knot's number of active rows
  static constexpr int even(int v) { return (v + 1) & ~1; }
  static constexpr int ldz_of(int nca) { return (NR + nca + 7) & ~7; }
  static constexpr int need2(int nca) { return MR * ldz_of(nca) + even(nca * NR) + MR * LDR + even(nca * NZ) + even(nca * nca); }
  // they alias P | G (dead by then) while the knot has at most NCAP active rows; knots with more run phase 2 out of a
  // per-instance scratch block in global memory (rare: iterates with most cone / box rows violated)
  static constexpr int un = (2 * N * LDN > need2(NCAP)) ? 2 * N * LDN : need2(NCAP);
  static constexpr int need2_all = need2(NC);
  static constexpr int scratch = need2_all + 64 * ((NC + 7) / 8);   // doubles per instance
  static constexpr int NDINV = (NBLK > MR / 8 ? NBLK : MR / 8) > (NCAP + 7) / 8 ? (NBLK > MR / 8 ? NBLK : MR / 8) : (NCAP + 7) / 8;
  static_assert(need2(NCAP) <= un && NCAP <= NC, "fast carving");
  static_assert(MR * ldz_of(0) <= N * LDN, "without active rows the value update reads nothing from U0 but Z, which stays clear of P");
  static_assert(un % 2 == 0 && (ZP * LDH) % 2 == 0 && ZP > NZ, "16-byte alignment of the bulk-copy destinations; spare padding column for pt");
  static constexpr int vecs = 5 * N + 2 * ZP + 36 + 2 * NC + 64 * NDINV + 8 * N + 32 + 16; // vectors, T6, dbr / dva, dinv, [pv | 0] tile, one reduction slot per warp, 8 mbarriers
  static constexpr int total = ZP * LDH + un + vecs;
};

// SEEDED: one leg [io.k0, io.k1) of the time-parallel solve, as riccati_instance<..., SEEDED> (riccati.cuh)
template <int N, int M, int NC, int NCAP = NC, bool SEEDED = false> HD void riccati_instance_fast(const RiccatiIO &io, double *ws) {
  using Lay = RicFastLayout<N, M, NC, NCAP>;
  constexpr int NZ = Lay::NZ, NR = Lay::NR, S = Lay::S, ZP = Lay::ZP, LDN = Lay::LDN, LDH = Lay::LDH, LDW = Lay::LDW, LDZ = Lay::LDZ, NBLK = Lay::NBLK, MR = Lay::MR, LDR = Lay::LDR;
  static_assert(N % 8 == 0, "fast Riccati needs n % 8 == 0");
  const int T = io.T;
  const int K0 = SEEDED ? io.k0 : 0, K1 = SEEDED ? io.k1 : T;
  const bool seeded = SEEDED && io.seedP != nullptr, last = !SEEDED || K1 == T;
  const double mu = io.mu, mu_d = io.mu_d;
  PHASE_DECL;
  // ---- carve shared memory
  double *H = ws;                              // ZP x LDH, zero padded; [0:N,0:N] carries the value-function Hessian between knots
  double *ABs = H;                             // ... and [A B]_k (N x LDZ) between the moment that Hessian is taken out and the Hessian update
  double *U0 = H + ZP * LDH;
  double *G = U0, *P = G + N * LDN;            // phase 1 (the factor first: W spills into its slot, see Ws)
  double *Ws = H + N * LDZ;                    // W (N x LDZ) between its product and the Hessian update: behind [A B], over the tail of the H buffer and the dead factor
  double *vec = U0 + Lay::un;
  double *p = vec, *pt = p + N, *gh = pt + N, *fb = gh + ZP, *tmp = fb + N, *dx = tmp + N, *z = dx + N; // gh, z: n + m entries, the others n
  double *T6 = z + ZP, *dbr = T6 + 36, *dva = dbr + NC, *dinv_s = dva + NC, *PV = dinv_s + 64 * Lay::NDINV, *red = PV + 8 * N; // (red: one slot per warp)
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(vec + Lay::vecs - 8); // mbarriers in the spare tail of vecs
  ONE_THREAD { for (int i_ = 0; i_ < 7; i_++) MBAR_INIT(mbar + i_, 1); } // 2: T6 / fbar, 3: [A B]; forward sweep: 4, 5: gain rows + vectors, 6: W + [A B]
  // ---- zero the padding of H once; terminal value function: P = H_T[xx] + C'C/mu, p = g_T[x] + C' d/mu
  PAR_FOR(e, ZP * LDH) H[e] = 0.0;
  PAR_FOR(e, N * 8) PV[e] = 0.0; // columns 1..7 of the [pv | 0] tile stay zero: the substitution solves each column on its own
  SYNC();
  ric_start_value<N, M, NC>(io, seeded, H, LDH, p);
  PAR_FOR(e, N * N) P[(e / N) * LDN + e % N] = H[(e / N) * LDH + e % N]; // the value update of every later knot writes P itself
  SYNC();
  // T6 and fbar of a knot arrive by bulk copies one knot ahead (mbar[2]); [A B]_k streams into the H buffer once the value Hessian
  // has been taken out of it (mbar[3]); [A B]_k and H_k are bulk-prefetched into L2 one knot ahead (H_k is read from there as
  // the initial value of the Hessian update's accumulators).
  static_assert((NZ * 8) % 16 == 0 && (LDH * 8) % 16 == 0 && (LDZ * 8) % 16 == 0 && (N * 8) % 16 == 0 && (N * NZ * 8) % 16 == 0 && (NZ * NZ * 8) % 16 == 0, "bulk copies need 16-byte rows");
  auto stage_small = [&](int kk) {
    ONE_THREAD {
      FENCE_PROXY_ASYNC();
      MBAR_EXPECT_TX(mbar + 2, (36 + N) * 8);
      BULK_G2S(T6, io.T6 + (size_t)kk * 36, 36 * 8, mbar + 2);
      BULK_G2S(fb, io.fbar + (size_t)kk * N, N * 8, mbar + 2);
    }
  };
  auto prefetch_knot = [&](int kk) {
    ONE_THREAD { PREFETCH_L2(io.AB + (size_t)kk * N * NZ, N * NZ * 8); PREFETCH_L2(io.H + (size_t)kk * NZ * NZ, NZ * NZ * 8); }
  };
  if (K1 > K0) { stage_small(K1 - 1); prefetch_knot(K1 - 1); }
  for (int k = K1 - 1; k >= K0; k--) {
    const double *gH = io.H + (size_t)k * NZ * NZ, *gAB = io.AB + (size_t)k * N * NZ;
    double *gW = io.W + (size_t)k * N * LDW;
    const int nca = io.nca[k];
    if (k > K0) prefetch_knot(k - 1);
    // 1. P <- T' H T (E normalisation: T = blockdiag(T6, I) touches the 6 base rows / columns only) and the normalised gradient
    //    tmp <- T' p.  Rows and columns >= 6 of P are already in place: the previous knot's value update stored them with H.
    MBAR_WAIT(mbar + 2, (K1 - 1 - k) & 1); // T6 and fbar of this knot (issued one knot ahead)
    PHASE(21);
    // the 6 base rows / columns, enumerated compactly so that no warp diverges over them: corner (36 terms), top edge, left edge
    PAR_FOR(s_, 36 + 12 * (N - 6)) {
      int i, j;
      double v = 0;
      if (s_ < 36) {
        i = s_ / 6; j = s_ % 6;
        for (int q = 0; q < 6; q++) {
          double r = 0;
          for (int m = 0; m < 6; m++) r += 0.5 * (H[q * LDH + m] + H[m * LDH + q]) * T6[6 * m + j];
          v += T6[6 * q + i] * r;
        }
      } else if (s_ < 36 + 6 * (N - 6)) {
        i = (s_ - 36) / (N - 6); j = 6 + (s_ - 36) % (N - 6);
        for (int q = 0; q < 6; q++) v += T6[6 * q + i] * H[q * LDH + j];
      } else {
        j = (s_ - 36 - 6 * (N - 6)) / (N - 6); i = 6 + (s_ - 36 - 6 * (N - 6)) % (N - 6);
        for (int q = 0; q < 6; q++) v += H[q * LDH + i] * T6[6 * q + j]; // (row q, column i: the same entries as the top edge, so P stays symmetric bit for bit there)
      }
      P[i * LDN + j] = v;
    }
    PAR_FOR(i, N) { double v = p[i]; if (i < 6) { v = 0; for (int q = 0; q < 6; q++) v += T6[6 * q + i] * p[q]; } tmp[i] = v; }
    SYNC(); // the base rows / columns of P and tmp are complete
    PHASE(16);
    // the H buffer is idle until the Hessian update: [A B]_k streams into it (one padded row per bulk copy; the products read columns
    // < ZP);  pv = tmp + P f into column 0 of the [pv | 0] tile and G <- I + mu_d P in the same pass over P
    ONE_THREAD MBAR_EXPECT_TX(mbar + 3, N * NZ * 8);
    PAR_FOR(i, N) { FENCE_PROXY_ASYNC(); BULK_G2S(ABs + i * LDZ, gAB + i * NZ, NZ * 8, mbar + 3); }
    PAR_FOR(e, N * (ZP - NZ)) { const int i = e / (ZP - NZ), j = NZ + e % (ZP - NZ); ABs[i * LDZ + j] = 0.0; }
    matvec_rows(P, LDN, N, N, fb, tmp, PV, 8, [&](int i, int j, double v) { G[i * LDN + j] = mu_d * v + ((i == j) ? 1.0 : 0.0); });
    SYNC(); // G and pv are complete
    if (k > K0) stage_small(k - 1); // T6 and fbar of this knot are consumed
    PHASE(1);
    // 2. G = chol(I + mu_d P)
    chol_mma<NBLK>(G, LDN, dinv_s);
    PHASE(2);
    // 3. [P | pv] <- Lambda^-1 [P | pv] in place: blocked forward / backward substitution, one warp per 8-column tile
    trsm_mma<NBLK>(G, LDN, dinv_s, P, LDN, NBLK, PV, 8, NBLK + 1);
    PHASE(4);
    // 4. W = Pt [A B] into shared memory (for the Hessian update) and straight from the accumulators to HBM (for the forward
    //    sweep); pt rides in the first padding column of W, so [A B]' pt falls out of the Hessian update
    MBAR_WAIT(mbar + 3, (K1 - 1 - k) & 1); // [A B]_k
    mma_tn_g<N>(NBLK, ZP / 8, P, LDN, ABs, LDZ, Ws, LDZ, nullptr, 0, 0, 0, false, gW, LDW, ZP);
    PHASE(17);
    PAR_FOR(i, N) { const double v = PV[8 * i]; pt[i] = v; Ws[i * LDZ + NZ] = v; gW[i * LDW + NZ] = v; io.pt[(size_t)k * N + i] = v; }
    SYNC();
    // 5. H = H_k + [A B]' W (symmetric: upper blocks computed, lower mirrored; H_k from L2, columns >= NZ read as zero).  The
    //    result overwrites the buffers [A B] and W sit in: accumulators stay in registers until every warp is done reading them.
    //    gh = g + [A B]' pt
    PHASE(22);
    mma_sym_deferred<N, Lay::MAXQ>(ZP / 8, ABs, LDZ, Ws, LDZ, H, LDH, gH, NZ, NZ, NZ);
    PHASE(18);
    // 8. KKT by block elimination.  Buffers [Z | Kv | Rh | CD | Sg] carved for this knot's active rows: over P | G (dead now), or
    //    in the instance's global scratch block when they do not fit
    const int ncol = NR + nca, ldz = (NR + nca + 7) & ~7; // Z columns: [rh | Sh' | D'], padded with zero columns to whole tiles
    const bool fits = nca <= NCAP;
    double *X2 = fits ? U0 : io.scratch;
    double *Z = X2, *Kv = Z + MR * ldz, *Rh = Kv + ((nca * NR + 1) & ~1), *CDs = Rh + MR * LDR, *Sg = CDs + ((nca * NZ + 1) & ~1); // = Lay::need2's carving
    double *dinv = fits ? dinv_s : io.scratch + Lay::need2_all;
    const double *gCD = io.CDact + (size_t)k * NC * NZ;
    const int32_t *ai = io.act_idx + (size_t)k * NC;
    const double *CD = fits ? CDs : gCD;
    PAR_FOR(i, N) gh[i] = io.g[(size_t)k * NZ + i] + H[i * LDH + NZ]; // (the control part goes straight into Z's column 0)
    if (fits) PAR_FOR(e, nca * NZ) CDs[e] = gCD[e];
    PAR_FOR(r, nca) dbr[r] = io.dbar[(size_t)k * NC + ai[r]];
    PAR_FOR(e, MR * MR) { // R^ = sym(H_uu), padded with the identity to MR x MR
      int i = e / MR, j = e % MR;
      Rh[i * LDR + j] = (i < M && j < M) ? 0.5 * (H[(N + i) * LDH + N + j] + H[(N + j) * LDH + N + i]) : ((i == j) ? 1.0 : 0.0);
    }
    PAR_FOR(e, MR * ldz) { // (reads the active rows from global memory: no barrier between the copy above and this loop)
      int i = e / ldz, c = e % ldz;
      Z[e] = (i >= M || c >= ncol) ? 0.0
           : ((c == 0) ? io.g[(size_t)k * NZ + N + i] + H[(N + i) * LDH + NZ] : (c < NR ? H[(N + i) * LDH + c - 1] : gCD[(c - NR) * NZ + N + i])); // H_ux row i (H is symmetric to rounding): conflict-free
    }
    SYNC(); // R^, Z, CD, dbar and gh are staged
    PHASE(6);
    // Z <- R^-1 Z on the tensor pipe: blocked Cholesky, then forward / backward substitution with one warp per 8-column tile of Z
    chol_mma<MR / 8>(Rh, LDR, dinv);
    PHASE(7);
    trsm_mma<MR / 8>(Rh, LDR, dinv, Z, ldz, ldz / 8, nullptr, 0, ldz / 8);
    PHASE(8);
    ric_kkt_schur<N, M>(nca, 1, NR, mu, CD, dbr, Z, ldz, Sg, Kv);
    PHASE(9);
    if (nca > 0) { chol_blocked(Sg, nca, nca, dinv); trsm_blocked(Sg, nca, nca, dinv, Kv, NR, NR); }
    PHASE(10);
    ric_kkt_ku<M>(nca, NR, Z, ldz, Kv, io.K + (size_t)k * S * NR, io.Kfb + (size_t)k * M * N);
    PHASE(11);
    // 9. P = Qh + Sh Ku + C' Kv, p = qh + Sh ku + C' kv : in place in H[0:N,0:N] / p, and the result also into the P buffer (its
    //    rows / columns >= 6 are the next knot's P as they stand).
    //    Sh Ku = H[N:, 0:N]' Z[:, 1:] runs on the DMMA pipe (K = MP, zero rows beyond M); the active-row part is usually empty.
    PAR_FOR(i, N) {
      double s = gh[i];
      for (int l = 0; l < M; l++) s += H[(N + l) * LDH + i] * Z[l * ldz]; // H_ux rows (as the DMMA update below): conflict-free
      for (int r = 0; r < nca; r++) s += CD[r * NZ + i] * Kv[r * NR];
      p[i] = s;
    }
    //    Without active rows the product is symmetric up to the rounding of well-scaled terms: upper blocks computed, lower mirrored.
    //    With active rows Ku and Kv carry 1/mu-sized entries that cancel in the sum, and the rounding of that cancellation must be
    //    averaged out as the oracle does: full product, then P <- (P + P') / 2.
    //    Without active rows the product stores P from its accumulators: the value update reads only Z of U0 then (Lay's static_assert).
    mma_tn(NBLK, NBLK, MR, H + N * LDH, LDH, Z + 1, ldz, H, LDH, H, LDH, N, N, nca == 0, nca == 0 ? P : nullptr, LDN);
    if (nca > 0) { // 2 x 4 register tiles over (row i, column c)
      constexpr int TC = N / 4;
      PAR_FOR(t, (N / 2) * TC) {
        const int i0 = (t / TC) * 2, c0 = (t % TC) * 4;
        double a[2][4];
#pragma unroll
        for (int r = 0; r < 2; r++)
#pragma unroll
          for (int q = 0; q < 4; q++) a[r][q] = H[(i0 + r) * LDH + c0 + q];
        for (int r = 0; r < nca; r++) {
          const double h0 = CD[r * NZ + i0], h1 = CD[r * NZ + i0 + 1];
          const double *kr = Kv + r * NR + 1 + c0;
#pragma unroll
          for (int q = 0; q < 4; q++) { a[0][q] += h0 * kr[q]; a[1][q] += h1 * kr[q]; }
        }
#pragma unroll
        for (int r = 0; r < 2; r++)
#pragma unroll
          for (int q = 0; q < 4; q++) H[(i0 + r) * LDH + c0 + q] = a[r][q];
      }
      SYNC(); // the rank-nca update is complete (and CD / Kv over P are consumed)
      PAR_FOR(e, N * N) { // lanes: 8 consecutive j x 4 consecutive i, which keeps the transposed access at 8-way bank conflicts
        const int blk = e >> 5, l = e & 31, i = (blk / (N / 8)) * 4 + (l >> 3), j = (blk % (N / 8)) * 8 + (l & 7);
        if (i < j) {
          const double v = 0.5 * (H[i * LDH + j] + H[j * LDH + i]);
          H[i * LDH + j] = v; H[j * LDH + i] = v; P[i * LDN + j] = v; P[j * LDN + i] = v;
        } else if (i == j) P[i * LDN + i] = H[i * LDH + i];
      }
      SYNC(); // H[0:N,0:N] and P are symmetric
    }
    PHASE(19);
    PHASE(12);
  }
  // ---- forward sweep, dx0 = 0 (force_initial_condition, fulldynamic_talos.py:384)
  PHASE(13);
  double acc = 0.0;
  ric_forward_start<N, SEEDED>(io, K0, p, dx);
  // everything that does not depend on the sequential chain is done for all knots at once: default multiplier steps
  // dv = dbar / mu of the inactive rows and their part of the directional derivative
  PAR_FOR(e_, ((last ? T + 1 : K1) - K0) * NC) {
    const int e = K0 * NC + e_;
    const int kk = e / NC, r = e % NC, na = io.nca[kk];
    const int32_t *ak = io.act_idx + (size_t)kk * NC;
    const double db = io.dbar[e];
    bool active = false;
    for (int q = 0; q < na; q++) active |= (ak[q] == r);
    io.dvs[e] = db / mu;
    if (!active) acc -= db * db / mu;
  }
  // W_k and [A B]_k (single stage), the first KROWS gain rows and the small per-knot vectors (two stages) go global -> shared by bulk
  // copies into the now dead H / P / G buffers: W / [A B] of knot k + 1 are requested as soon as knot k's mat-vecs are done, gain rows
  // and vectors two knots ahead; everything is bulk-prefetched from HBM into L2 PF knots ahead of the chain dx_k -> du_k -> dx_{k+1}
  // knots of HBM -> L2 prefetch ahead of the chain (resident instances x PF x 76 KB must stay well inside L2); distances 2 and 3 read
  // more from DRAM in the same kernel time
  constexpr int PF = 1;
  constexpr int FWA = N * LDW + N * NZ;    // W_k | [A B]_k
  constexpr int FX = 4 * N + NZ + 36;      // pt_k, fbar_k, lplus_{k+1}, lam_{k+1}, lxu_k, T6_k
  constexpr int KROWS = ((((ZP * LDH + Lay::un - FWA - 2 * FX) / 2) / NR) & ~1) < S ? ((((ZP * LDH + Lay::un - FWA - 2 * FX) / 2) / NR) & ~1) : (S & ~1);
  constexpr int FKX = KROWS * NR + FX;
  static_assert(KROWS >= M && FWA + 2 * FKX <= ZP * LDH + Lay::un && FWA % 2 == 0 && FKX % 2 == 0, "forward staging does not fit");
  static_assert((N * LDW * 8) % 16 == 0 && (N * NZ * 8) % 16 == 0 && (S * NR * 8) % 16 == 0 && (2 * NR * 8) % 16 == 0 && (N * 8) % 16 == 0 && (NZ * 8) % 16 == 0,
                "bulk copies need 16-byte sizes and offsets");
  auto prefetch_fwd = [&](int kk) {
    ONE_THREAD {
      const int rows = (M + io.nca[kk] + 1) & ~1;
      PREFETCH_L2(io.W + (size_t)kk * N * LDW, N * LDW * 8);
      PREFETCH_L2(io.AB + (size_t)kk * N * NZ, N * NZ * 8);
      PREFETCH_L2(io.K + (size_t)kk * S * NR, rows * NR * 8);
    }
  };
  auto stage_wa = [&](int kk) {
    ONE_THREAD {
      FENCE_PROXY_ASYNC(); // the buffer was last touched through the generic proxy
      MBAR_EXPECT_TX(mbar + 6, FWA * 8);
      BULK_G2S(ws, io.W + (size_t)kk * N * LDW, N * LDW * 8, mbar + 6);
      BULK_G2S(ws + N * LDW, io.AB + (size_t)kk * N * NZ, N * NZ * 8, mbar + 6);
    }
  };
  auto stage_kx = [&](int kk) {
    ONE_THREAD {
      double *bk = ws + FWA + ((kk - K0) & 1) * FKX, *bx = bk + KROWS * NR;
      unsigned long long *bar = mbar + 4 + ((kk - K0) & 1);
      int rows = M + io.nca[kk];
      if (rows > KROWS) rows = KROWS;
      rows = (rows + 1) & ~1; // whole 16-byte units (an extra row stays inside this knot's gain block)
      FENCE_PROXY_ASYNC();
      MBAR_EXPECT_TX(bar, (rows * NR + FX) * 8);
      BULK_G2S(bk, io.K + (size_t)kk * S * NR, rows * NR * 8, bar);
      BULK_G2S(bx, io.pt + (size_t)kk * N, N * 8, bar);
      BULK_G2S(bx + N, io.fbar + (size_t)kk * N, N * 8, bar);
      BULK_G2S(bx + 2 * N, io.lplus + (size_t)(kk + 1) * N, N * 8, bar);
      BULK_G2S(bx + 3 * N, io.lam + (size_t)(kk + 1) * N, N * 8, bar);
      BULK_G2S(bx + 4 * N, io.lxu + (size_t)kk * NZ, NZ * 8, bar);
      BULK_G2S(bx + 4 * N + NZ, io.T6 + (size_t)kk * 36, 36 * 8, bar);
    }
  };
  SYNC();
  for (int kk = K0; kk < K0 + PF && kk < K1; kk++) prefetch_fwd(kk);
  if (K1 > K0) { stage_kx(K0); stage_wa(K0); }
  if (K1 > K0 + 1) stage_kx(K0 + 1);
  for (int k = K0; k < K1; k++) {
    const int nca = io.nca[k];
    if (k + PF < K1) prefetch_fwd(k + PF);
    const double *sW = ws, *sAB = ws + N * LDW, *sK = ws + FWA + ((k - K0) & 1) * FKX, *sX = sK + KROWS * NR;
    const double *gK = io.K + (size_t)k * S * NR;
    MBAR_WAIT(mbar + 4 + ((k - K0) & 1), ((k - K0) >> 1) & 1); // gain rows and vectors of knot k (each barrier is used every other knot)
    // du, dv of the active rows: RA rows per warp at a time (independent reduction chains), columns over lanes
    constexpr int RA = 3;
    for (int base = WARP_ID * RA; base < M + nca; base += NWARPS * RA) {
      double sa[RA];
#pragma unroll
      for (int r = 0; r < RA; r++) sa[r] = 0.0;
      LANE_FOR(j, N) {
        const double dj = dx[j];
#pragma unroll
        for (int r = 0; r < RA; r++) {
          const int i = base + r;
          if (i < M + nca) sa[r] += ((i < KROWS) ? sK[i * NR + 1 + j] : LDCG(gK + i * NR + 1 + j)) * dj;
        }
      }
#pragma unroll
      for (int r = 0; r < RA; r++) sa[r] = WARP_SUM(sa[r]);
      if (LANE0) {
#pragma unroll
        for (int r = 0; r < RA; r++) {
          const int i = base + r;
          if (i >= M + nca) continue;
          const double v = sa[r] + ((i < KROWS) ? sK[i * NR] : LDCG(gK + i * NR));
          if (i < M) { z[N + i] = v; io.dus[(size_t)k * M + i] = v; } else dva[i - M] = v;
        }
      }
    }
    PAR_FOR(i, N) z[i] = dx[i];
    SYNC();
    if (nca > 0) {
      const int32_t *ai = io.act_idx + (size_t)k * NC;
      const double *gdb = io.dbar + (size_t)k * NC, *gvp = io.vplus + (size_t)k * NC, *gv = io.v + (size_t)k * NC;
      PAR_FOR(r, nca) {
        const int row = ai[r];
        io.dvs[(size_t)k * NC + row] = dva[r];
        acc += (2.0 * gvp[row] - gv[row]) * (mu * dva[r] - gdb[row]) - gdb[row] * dva[r];
      }
    }
    PAR_FOR(i, NZ) acc += sX[4 * N + i] * z[i];
    MBAR_WAIT(mbar + 6, (k - K0) & 1); // W_k, [A B]_k
    // dlam_{k+1} = pt + W z ; tmp = A dx + B du + fbar - mu_d dlam : RB rows per warp at a time
    constexpr int RB = 7;
    for (int base = WARP_ID * RB; base < N; base += NWARPS * RB) {
      double sl[RB], sa[RB];
#pragma unroll
      for (int r = 0; r < RB; r++) { sl[r] = 0.0; sa[r] = 0.0; }
      LANE_FOR(j, NZ) {
        const double zj = z[j];
#pragma unroll
        for (int r = 0; r < RB; r++)
          if (base + r < N) { sl[r] += sW[(base + r) * LDW + j] * zj; sa[r] += sAB[(base + r) * NZ + j] * zj; }
      }
#pragma unroll
      for (int r = 0; r < RB; r++) { sl[r] = WARP_SUM(sl[r]); sa[r] = WARP_SUM(sa[r]); }
      if (LANE0) {
#pragma unroll
        for (int r = 0; r < RB; r++) {
          const int i = base + r;
          if (i >= N) continue;
          const double fbi = sX[N + i], lp = sX[2 * N + i], lm = sX[3 * N + i], dl = sl[r] + sX[i];
          tmp[i] = sa[r] + fbi - mu_d * dl;
          io.dlams[(size_t)(k + 1) * N + i] = dl;
          acc += (2.0 * lp - lm) * (mu_d * dl - fbi) - fbi * dl;
        }
      }
    }
    SYNC();
    if (k + 1 < K1) stage_wa(k + 1); // the W / [A B] stage is free
    PAR_FOR(i, N) {
      double v;
      if (i < 6) { v = 0; for (int l = 0; l < 6; l++) v += sX[4 * N + NZ + 6 * i + l] * tmp[l]; } else v = tmp[i];
      dx[i] = v; io.dxs[(size_t)(k + 1) * N + i] = v;
    }
    PHASE(20);
    SYNC();
    if (k + 2 < K1) stage_kx(k + 2); // this knot's gain / vector stage is free
  }
  if (last) { // terminal knot: dv of the active terminal rows and the terminal cost gradient
    const int nca = io.nca[T];
    const int32_t *ai = io.act_idx + (size_t)T * NC;
    const double *gdb = io.dbar + (size_t)T * NC, *gvp = io.vplus + (size_t)T * NC, *gv = io.v + (size_t)T * NC;
    const double *CT = io.CDact + (size_t)T * NC * NZ;
    PAR_FOR(r, nca) {
      const int row = ai[r];
      double sv = gdb[row];
      for (int j = 0; j < N; j++) sv += CT[r * NZ + j] * dx[j];
      sv /= mu;
      io.dvs[(size_t)T * NC + row] = sv;
      acc += (2.0 * gvp[row] - gv[row]) * (mu * sv - gdb[row]) - gdb[row] * sv;
    }
    PAR_FOR(i, N) acc += io.lxu[(size_t)T * NZ + i] * dx[i];
  }
  PHASE(14);
  PHASE_DUMP(io.phase_out);
  acc = WARP_SUM(acc);
  if (LANE0) red[WARP_ID] = acc;
  SYNC();
  ONE_THREAD { double s = 0; for (int t = 0; t < NWARPS; t++) s += red[t]; io.dphi[0] = s; }
  SYNC();
}

} // namespace mpcdev
