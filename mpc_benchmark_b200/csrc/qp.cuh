// Batched dense QP solver (SURVEY 8f row f-3): ONE group of threads per QP, every matrix of the QP resident in shared memory.
// Boundary replaced: proxsuite.proxqp.dense.QP.solve() as driven by QP_utils.py:500-513,557-573 (IDSolver_ulim) and the other
// solver classes of that file.  Normative algorithm: oracle/qp.hpp (ProxQP restated: proximal augmented Lagrangian, semismooth
// Newton with an exact piecewise-quadratic linesearch, BCL outer loop); this file mirrors it step by step.
// Written in the group idiom of dev_common.cuh (PAR_FOR / SYNC / ONE_THREAD), so the same source runs serially under the
// test-only host emulation (tests/emu).
//
// Shared memory per QP (n = 62, n_eq = 40, n_in = 18: 103 KB, two QPs per SM): W = [A; C; H] stacked under one ODD leading
// dimension (row sweeps over lanes and column sweeps over threads are both free of bank conflicts; W v yields A v, C v, H v in one
// warp-cooperative pass), ONE n x n buffer with the Newton matrix K in its lower triangle and Q = H + rho I + A'A / mu_e — the part
// of K that only changes with the equality penalty — transposed in its upper triangle, and the vectors.  Scalars (norms, the
// linesearch's breakpoint search) are reduced by every warp redundantly, so they cost no block barrier.  (Three QPs per SM — H folded
// into the K buffer, K rebuilt from A in every Newton step — measured 16 % SLOWER: the third CTA takes the instruction-cache hit
// rate to 64 %.)
// HBM traffic = the QP data once in, (x, y, z, info) once out.
#pragma once
#include "../../include/mpcqp_b200.h"
#include "dev_common.cuh"
#include "dmma.cuh"

namespace mpcdev {

struct QPArgs {
  int n, ne, ni, box, batch;
  const double *H, *g, *A, *b, *C, *l, *u, *lb, *ub;
  long long sH, sg, sA, sb, sC, sl, su, slb, sub; // batch strides in doubles (0 = shared)
  double *x, *y, *z;
  mpc_qp_info_t *info;
  mpc_qp_settings_t st;
  long long *phase; // 8 cycle counters (builds with -DMPC_QP_PHASE_TIMING only), else unused
};

#if defined(MPC_QP_PHASE_TIMING) && !defined(MPC_HOST_EMU)
#define QP_T0() long long qt_ = clock64(); long long qacc_[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define QP_TICK(k) do { const long long n_ = clock64(); qacc_[k] += n_ - qt_; qt_ = n_; } while (0)
#define QP_TDUMP(inst) do { if (threadIdx.x == 0 && P.phase) for (int k_ = 0; k_ < 8; k_++) atomicAdd((unsigned long long *)P.phase + k_, (unsigned long long)qacc_[k_]); } while (0)
#else
#define QP_T0() ((void)0)
#define QP_TICK(k) ((void)0)
#define QP_TDUMP(inst) ((void)0)
#endif

// helpers with several call sites are NOT inlined: the solve kernel is one long loop whose body has to stay inside the instruction
// cache (12 k SASS instructions = 190 KB with everything inlined: "no instruction" was the second largest stall)
#ifdef MPC_HOST_EMU
#define QP_NOINLINE inline
#else
#define QP_NOINLINE __device__ __noinline__
#endif

HD int qp_ld(int n) { return n | 1; }
// doubles of shared memory one QP needs (host + device)
#ifdef MPC_HOST_EMU
#define QP_HOST_DEV inline
#else
#define QP_HOST_DEV inline __host__ __device__
#endif
QP_HOST_DEV int qp_smem_doubles(int n, int ne, int ni, int box) {
  const int ld = n | 1, nz = ni + (box ? n : 0), np = (n + CB - 1) / CB, nw = ne + ni + n, ldk = CB * np + 4;
  return nw * ld + 1 + CB * np * ldk + 2 * np * CB * CB + 8 * n + 4 * ne + 7 * nz + 2 * nw + ni + 32; // + 1: the K buffer starts on a 16-byte boundary
}

// NaN-propagating maximum (fmax drops NaNs; the non-finite status relies on them)
HD double qp_maxn(double a, double b) { return (b > a || b != b) ? b : a; }
// Warp-wide reductions.  Every warp of the group runs the small reductions of the solver REDUNDANTLY on the same shared-memory
// data (lanes over the items, butterfly), so all warps hold bitwise identical results and no block barrier is needed for a scalar.
HD double qp_wsum(double x) { return WARP_SUM(x); }
HD double qp_wmax(double x) {
#ifndef MPC_HOST_EMU
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = qp_maxn(x, __shfl_xor_sync(0xffffffffu, x, o));
#endif
  return x;
}
HD double qp_wmin(double x) {
#ifndef MPC_HOST_EMU
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = fmin(x, __shfl_xor_sync(0xffffffffu, x, o));
#endif
  return x;
}

HD bool qp_inf(double v) { return fabs(v) >= 1e20; }
QP_NOINLINE double qp_pow(double a, double b) { return pow(a, b); }

struct QPView { // carved shared memory of one QP
  int n, ne, ni, nz, nw, ld, box;
  int np8, ldk; // the Newton-matrix buffer is padded to whole 8 x 8 tiles (identity in the padding); its leading dimension = 4 (mod 8): conflict-free DMMA fragments
  double *W;    // [A (ne rows); C (ni rows); H (n rows)], one leading dimension: W v gives A v, C v and H v in ONE sweep
  double *As, *Cs, *Hs;
  double *KQ;   // np8 x np8: Newton matrix K in the lower triangle incl. diagonal (factored in place).  The factorisation touches the
                // lower BLOCK triangle and the diagonal 8 x 8 tiles only, so Q = H + rho I + A'A / mu_e lives transposed in the strictly
                // upper block triangle; its entries inside the diagonal tiles are in Qb, its diagonal in Qd
  double *Qb, *Qd, *Dinv, *act;
  double *x, *xe, *g, *grad, *dx, *hxg;            // n
  double *y, *ye, *re, *b;                         // ne
  double *z, *ze, *su, *sl, *lo, *up, *t;          // nz
  double *dual;                                    // n
  double *wx, *wd;                                 // nw = ne + ni + n: W x and W dx
  double *sc;
};
HD QPView qp_carve(double *m, int n, int ne, int ni, int box) {
  QPView v;
  v.n = n; v.ne = ne; v.ni = ni; v.box = box; v.nz = ni + (box ? n : 0); v.nw = ne + ni + n; v.ld = qp_ld(n);
  const int np = (n + CB - 1) / CB;
  v.W = m; v.As = m; v.Cs = m + ne * v.ld; v.Hs = m + (ne + ni) * v.ld; m += v.nw * v.ld;
  if ((v.nw * v.ld) & 1) m++; // the tensor-core routines store pairs of doubles into the K buffer: keep it 16-byte aligned
  v.np8 = CB * np; v.ldk = v.np8 + 4;
  v.KQ = m; m += v.np8 * v.ldk; v.Dinv = m; m += np * CB * CB; v.Qb = m; m += np * CB * CB;
  v.x = m; m += n; v.xe = m; m += n; v.g = m; m += n; v.grad = m; m += n; v.dx = m; m += n; v.hxg = m; m += n; v.Qd = m; m += n;
  v.y = m; m += ne; v.ye = m; m += ne; v.re = m; m += ne; v.b = m; m += ne;
  v.z = m; m += v.nz; v.ze = m; m += v.nz; v.su = m; m += v.nz; v.sl = m; m += v.nz; v.lo = m; m += v.nz; v.up = m; m += v.nz; v.t = m; m += v.nz;
  v.dual = m; m += n;
  v.wx = m; m += v.nw; v.wd = m; m += v.nw; v.act = m; m += ni; v.sc = m;
  return v;
}
enum { QS_PRI = 0, QS_DUA, QS_GAP, QS_OBJ, QS_PRIS, QS_DUAS, QS_GAPS, QS_NACT };

// Q(i, j), i > j: transposed in the strictly upper block triangle of KQ, or in Qb inside a diagonal 8 x 8 tile
HD double &qp_Q(const QPView &v, int i, int j) { return ((i >> 3) == (j >> 3)) ? v.Qb[(i >> 3) * 64 + (i & 7) * 8 + (j & 7)] : v.KQ[j * v.ldk + i]; }

// value of inequality row i (general rows, then the identity rows of the box) from a product W v stored in wv, v itself for the box
HD double qp_ineq(const QPView &v, const double *wv, const double *vec, int i) { return (i < v.ni) ? wv[v.ne + i] : vec[i - v.ni]; }

// out = W vec: rows over warps (7 at a time, independent reduction chains), columns over lanes (consecutive doubles: no bank
// conflicts), butterfly reduction.  Ends with the group barrier.
QP_NOINLINE void qp_wmatvec(const QPView &v, const double *vec, double *out) {
  matvec_rows<7>(v.W, v.ld, v.nw, v.n, vec, nullptr, out);
  SYNC();
}

// Residuals at (x, y, z) from wx = W x: every warp redundantly.  Needs v.dual[i] = (H x + g + A'y + C'z)_i from the column phase.
struct QPRes { double pri, dua, gap, obj, pris, duas, gaps; };
HD double qp_primal_residual(const QPView &v) { // max(|A x - b|, [s - u]+ + [s - l]-): lanes over the rows
  double pri = 0;
  LANE_FOR(w, v.ne + v.nz) {
    if (w < v.ne) pri = qp_maxn(pri, fabs(v.wx[w] - v.b[w]));
    else {
      const int i = w - v.ne;
      const double s = qp_ineq(v, v.wx, v.x, i);
      double viol = 0;
      if (!qp_inf(v.up[i])) viol += fmax(s - v.up[i], 0.0);
      if (!qp_inf(v.lo[i])) viol += fmin(s - v.lo[i], 0.0);
      pri = qp_maxn(pri, fabs(viol));
    }
  }
  return qp_wmax(pri);
}

// Q = H + rho I + A'A / mu_e (strict lower part stored transposed in the upper block triangle of KQ / in Qb, diagonal in Qd): formed
// once per value of mu_e (at the start and after a BCL penalty update), so that a Newton step only adds the few ACTIVE inequality rows
// to it.  A'A is a dense contraction: for the padded 64 x 64 case it runs on the FP64 tensor pipe (mma_tn, upper 16 x 16 blocks +
// mirror) straight into the K buffer, which is free at this point; then one pass adds H, scales and moves the entries to where Q lives.
// Other sizes: 2 x 2 register tiles.
QP_NOINLINE void qp_form_Q(const QPView &v, double rho, double mue) {
  const int n = v.n, ne = v.ne, ld = v.ld, ldk = v.ldk, th = (n + 1) / 2;
  const double ime = 1.0 / mue;
  if (v.np8 == 64 && ne >= 4 && ne % 4 == 0) {
    // columns n .. 63 of the operand read the first entries of the next row of W (finite): they only reach rows / columns >= n of the result
    mma_tn(8, 8, ne, v.As, ld, v.As, ld, v.KQ, ldk, nullptr, 0, 0, 0, true);
    PAR_FOR(e, n * n) {
      const int i = e / n, j = e % n;
      if (j > i) continue;
      const double q = v.Hs[i * ld + j] + v.KQ[i * ldk + j] * ime; // (A'A)(i, j) from the lower triangle; nobody writes there in this pass
      if (i == j) v.Qd[i] = q + rho; else qp_Q(v, i, j) = q;
    }
    PAR_FOR(e, (v.np8 - n) * v.np8) { // the product also wrote the padding rows of the Newton matrix: back to the identity
      const int r = n + e / v.np8, c = e % v.np8;
      if (c <= r) v.KQ[r * ldk + c] = (r == c) ? 1.0 : 0.0;
    }
    SYNC();
    return;
  }
  PAR_FOR(tile, th * th) {
    const int ti = tile / th, tj = tile % th;
    if (tj > ti) continue;
    const int i0 = 2 * ti, j0 = 2 * tj;
    const bool i1 = i0 + 1 < n, j1 = j0 + 1 < n;
    const int i1o = i1 ? 1 : 0, j1o = j1 ? 1 : 0;
    double a00 = 0, a01 = 0, a10 = 0, a11 = 0;
#pragma unroll 4
    for (int r = 0; r < ne; r++) {
      const double *ar = v.As + r * ld;
      const double x0 = ar[i0], x1 = ar[i0 + i1o], y0 = ar[j0], y1 = ar[j0 + j1o];
      a00 += x0 * y0; a01 += x0 * y1; a10 += x1 * y0; a11 += x1 * y1;
    }
    const double q00 = v.Hs[i0 * ld + j0] + a00 * ime, q01 = v.Hs[i0 * ld + j0 + j1o] + a01 * ime;
    const double q10 = v.Hs[(i0 + i1o) * ld + j0] + a10 * ime, q11 = v.Hs[(i0 + i1o) * ld + j0 + j1o] + a11 * ime;
    if (i0 == j0) {
      v.Qd[i0] = q00 + rho;
      if (i1) { v.Qd[i0 + 1] = q11 + rho; qp_Q(v, i0 + 1, i0) = q10; }
    } else {
      qp_Q(v, i0, j0) = q00;
      if (j1) qp_Q(v, i0, j0 + 1) = q01;
      if (i1) { qp_Q(v, i0 + 1, j0) = q10; if (j1) qp_Q(v, i0 + 1, j0 + 1) = q11; }
    }
  }
  SYNC();
}
// K = Q + C_act' C_act / mu_i (+ 1 / mu_i on the diagonal for active box rows), lower triangle incl. diagonal: 2 x 2 tiles, tile
// rows over warps, tile columns over lanes; the compacted list of active general rows (v.act, v.sc[QS_NACT]) comes from the
// gradient phase.
HD void qp_newton_matrix(const QPView &v, double mui) {
  const int n = v.n, ld = v.ld, ldk = v.ldk, th = (n + 1) / 2, nact = (int)v.sc[QS_NACT];
  const double imi = 1.0 / mui;
  WARP_TILE_FOR(ti, th) {
    LANE_FOR(tj, ti + 1) {
      const int i0 = 2 * ti, j0 = 2 * tj;
      const bool i1 = i0 + 1 < n, j1 = j0 + 1 < n;
      const int i1o = i1 ? 1 : 0, j1o = j1 ? 1 : 0;
      double c00 = 0, c01 = 0, c10 = 0, c11 = 0;
      for (int q = 0; q < nact; q++) {
        const double *cr = v.Cs + (int)v.act[q] * ld;
        const double x0 = cr[i0], x1 = cr[i0 + i1o], y0 = cr[j0], y1 = cr[j0 + j1o];
        c00 += x0 * y0; c01 += x0 * y1; c10 += x1 * y0; c11 += x1 * y1;
      }
      if (i0 == j0) {
        double d0 = v.Qd[i0] + c00 * imi, d1 = i1 ? v.Qd[i0 + 1] + c11 * imi : 0.0;
        if (v.box) {
          if (v.su[v.ni + i0] > 0 || v.sl[v.ni + i0] < 0) d0 += imi;
          if (i1 && (v.su[v.ni + i0 + 1] > 0 || v.sl[v.ni + i0 + 1] < 0)) d1 += imi;
        }
        v.KQ[i0 * ldk + i0] = d0;
        if (i1) { v.KQ[(i0 + 1) * ldk + i0] = qp_Q(v, i0 + 1, i0) + c10 * imi; v.KQ[(i0 + 1) * ldk + i0 + 1] = d1; }
      } else {
        v.KQ[i0 * ldk + j0] = qp_Q(v, i0, j0) + c00 * imi;
        if (j1) v.KQ[i0 * ldk + j0 + 1] = qp_Q(v, i0, j0 + 1) + c01 * imi;
        if (i1) {
          v.KQ[(i0 + 1) * ldk + j0] = qp_Q(v, i0 + 1, j0) + c10 * imi;
          if (j1) v.KQ[(i0 + 1) * ldk + j0 + 1] = qp_Q(v, i0 + 1, j0 + 1) + c11 * imi;
        }
      }
    }
  }
  SYNC();
}

// The whole solve of QP `inst` by the calling group.  smem: qp_smem_doubles(...) doubles of the group's shared memory.
HD void qp_solve_group(const QPArgs &P, int inst, double *smem) {
  const int n = P.n, ne = P.ne, ni = P.ni;
  const QPView v = qp_carve(smem, n, ne, ni, P.box);
  const int nz = v.nz, ld = v.ld;
  const mpc_qp_settings_t &st = P.st;
  QP_T0();
  // ---- load the QP
  {
    const double *H = P.H + inst * P.sH, *A = P.A + inst * P.sA, *Cm = P.C + inst * P.sC;
    PAR_FOR(e, n * n) v.Hs[(e / n) * ld + e % n] = H[e];
    PAR_FOR(e, ne * n) v.As[(e / n) * ld + e % n] = A[e];
    PAR_FOR(e, ni * n) v.Cs[(e / n) * ld + e % n] = Cm[e];
    PAR_FOR(e, (v.np8 - n) * v.np8) { // identity in the padding rows of the Newton matrix (never written again: the factor of I is I)
      const int r = n + e / v.np8, c = e % v.np8;
      if (c <= r) v.KQ[r * v.ldk + c] = (r == c) ? 1.0 : 0.0;
    }
    const double *g = P.g + inst * P.sg, *l = P.l + inst * P.sl, *u = P.u + inst * P.su;
    PAR_FOR(i, n) { v.g[i] = g[i]; v.x[i] = st.warm_start ? P.x[(long long)inst * n + i] : 0.0; }
    const double *bg = P.b + inst * P.sb;
    PAR_FOR(r, ne) { v.b[r] = bg[r]; v.y[r] = st.warm_start ? P.y[(long long)inst * ne + r] : 0.0; }
    PAR_FOR(i, nz) {
      v.lo[i] = (i < ni) ? l[i] : P.lb[inst * P.slb + i - ni];
      v.up[i] = (i < ni) ? u[i] : P.ub[inst * P.sub + i - ni];
      v.z[i] = st.warm_start ? P.z[(long long)inst * nz + i] : 0.0;
    }
  }
  SYNC();
  QP_TICK(0);
  double mue = st.mu_eq, mui = st.mu_in;
  const double eta_ext_init = qp_pow(0.1, st.alpha_bcl), eps_in_min = fmin(st.eps_abs, 1e-9);
  double eta_ext = eta_ext_init, eta_in = 1.0;
  int status = 1, it = 0, it_in = 0, mu_updates = 0;
  QPRes R = {0, 0, 0, 0, 0, 0, 0};
  qp_form_Q(v, st.rho, mue);
  QP_TICK(3);
  qp_wmatvec(v, v.x, v.wx); // wx = [A x; C x; H x]: computed once, then updated with every accepted step (wx += alpha W dx)
  for (;; it++) {
    // ---- residuals at (x, y, z)  (oracle/qp.hpp qp_residuals): column phase, then every warp reduces redundantly
    PAR_FOR(i, n) {
      double aty = 0, ctz = 0;
#pragma unroll 4
      for (int r = 0; r < ne; r++) aty += v.As[r * ld + i] * v.y[r];
#pragma unroll 4
      for (int k = 0; k < ni; k++) ctz += v.Cs[k * ld + i] * v.z[k];
      if (P.box) ctz += v.z[ni + i];
      v.dual[i] = v.wx[ne + ni + i] + v.g[i] + aty + ctz;
      v.grad[i] = fmax(fabs(aty), fabs(ctz)); // scale of the dual residual (scratch use of grad)
    }
    SYNC();
    {
      double pri = 0, nAC = 0, by = 0, bz = 0, xHx = 0, gx = 0, dua = 0, dsc = 0;
      LANE_FOR(w, ne + nz) {
        if (w < ne) { const double ax = v.wx[w]; pri = qp_maxn(pri, fabs(ax - v.b[w])); nAC = fmax(nAC, fabs(ax)); by += v.b[w] * v.y[w]; }
        else {
          const int i = w - ne;
          const double s = qp_ineq(v, v.wx, v.x, i), zi = v.z[i];
          nAC = fmax(nAC, fabs(s));
          double viol = 0;
          if (!qp_inf(v.up[i])) viol += fmax(s - v.up[i], 0.0);
          if (!qp_inf(v.lo[i])) viol += fmin(s - v.lo[i], 0.0);
          pri = qp_maxn(pri, fabs(viol));
          if (zi > 0 && !qp_inf(v.up[i])) bz += v.up[i] * zi;
          if (zi < 0 && !qp_inf(v.lo[i])) bz += v.lo[i] * zi;
        }
      }
      LANE_FOR(i, n) {
        const double hx = v.wx[ne + ni + i];
        xHx += v.x[i] * hx; gx += v.g[i] * v.x[i];
        dua = qp_maxn(dua, fabs(v.dual[i]));
        dsc = fmax(dsc, fmax(fmax(fabs(hx), fabs(v.g[i])), v.grad[i]));
      }
      by = qp_wsum(by); bz = qp_wsum(bz); xHx = qp_wsum(xHx); gx = qp_wsum(gx);
      R.pri = qp_wmax(pri); R.dua = qp_wmax(dua); R.pris = qp_wmax(nAC); R.duas = qp_wmax(dsc);
      R.gap = xHx + gx + by + bz; R.obj = 0.5 * xHx + gx;
      R.gaps = fmax(fmax(fabs(xHx), fabs(gx)), fmax(fabs(by), fabs(bz)));
    }
    QP_TICK(1);
    if (!isfinite(R.pri) || !isfinite(R.dua)) { status = 2; break; }
    const bool ok = R.pri <= st.eps_abs + st.eps_rel * R.pris && R.dua <= st.eps_abs + st.eps_rel * R.duas &&
                    (!st.check_duality_gap || fabs(R.gap) <= st.eps_abs + st.eps_rel * R.gaps);
    if (ok) { status = 0; break; }
    if (it >= st.max_iter) break;
    SYNC(); // (the grad scratch is rewritten below)
    PAR_FOR(i, n) v.xe[i] = v.x[i];
    PAR_FOR(r, ne) v.ye[r] = v.y[r];
    PAR_FOR(i, nz) v.ze[i] = v.z[i];
    SYNC();
    bool failed = false, stalled = false;
    const double ime = 1.0 / mue, imi = 1.0 / mui; // (the oracle divides: same value to one rounding)
    for (int in = 0;; in++) {
      // constraint residuals of the augmented Lagrangian from wx
      PAR_FOR(w, ne + nz) {
        if (w < ne) v.re[w] = v.wx[w] - v.b[w] + mue * v.ye[w];
        else {
          const int i = w - ne;
          const double s = qp_ineq(v, v.wx, v.x, i);
          const double su = qp_inf(v.up[i]) ? -1e300 : s - v.up[i] + mui * v.ze[i];
          const double sl = qp_inf(v.lo[i]) ? 1e300 : s - v.lo[i] + mui * v.ze[i];
          v.su[i] = su; v.sl[i] = sl;
          v.t[i] = (fmax(su, 0.0) + fmin(sl, 0.0)) * imi;
        }
      }
      SYNC();
      ONE_THREAD { // compacted list of the active general rows for the Newton matrix
        int c = 0;
        for (int k = 0; k < ni; k++) if (v.su[k] > 0 || v.sl[k] < 0) v.act[c++] = (double)k;
        v.sc[QS_NACT] = (double)c;
      }
      PAR_FOR(i, n) {
        const double hxg = v.g[i] + st.rho * (v.x[i] - v.xe[i]) + v.wx[ne + ni + i];
        double s = 0, c = 0;
#pragma unroll 4
        for (int r = 0; r < ne; r++) s += v.As[r * ld + i] * v.re[r];
#pragma unroll 4
        for (int k = 0; k < ni; k++) c += v.Cs[k * ld + i] * v.t[k];
        if (P.box) c += v.t[ni + i];
        v.hxg[i] = hxg;
        v.grad[i] = hxg + s * ime + c;
      }
      SYNC();
      double gn = 0;
      LANE_FOR(i, n) gn = qp_maxn(gn, fabs(v.grad[i]));
      gn = qp_wmax(gn);
      QP_TICK(2);
      if (!isfinite(gn)) { failed = true; break; }
      if (gn <= eta_in || in >= st.max_iter_in || stalled) break;
      // Newton step on the current active set
      qp_newton_matrix(v, mui);
      PAR_FOR(i, n) v.dx[i] = -v.grad[i];
      QP_TICK(3);
      // factorisation: tensor-core tiles with one-panel look-ahead for the reference's size (57 <= n <= 64), the SIMT panel routine otherwise
      if (v.np8 == 64) chol_mma<8>(v.KQ, v.ldk, v.Dinv); else chol_blocked(v.KQ, n, v.ldk, v.Dinv);
      QP_TICK(4);
      trsm_blocked(v.KQ, n, v.ldk, v.Dinv, v.dx, 1, 1);
      QP_TICK(5);
      it_in++;
      // exact linesearch on the piecewise quadratic: wd = [A dx; C dx; H dx], then every warp redundantly
      qp_wmatvec(v, v.dx, v.wd);
      double a0 = 0, b0 = 0;
      LANE_FOR(w, ne + n) {
        if (w < ne) { const double ad = v.wd[w] * ime; a0 += ad * v.wd[w]; b0 += ad * v.re[w]; }
        else { const int i = w - ne; a0 += v.dx[i] * (v.wd[ne + ni + i] + st.rho * v.dx[i]); b0 += v.dx[i] * v.hxg[i]; }
      }
      a0 = qp_wsum(a0); b0 = qp_wsum(b0);
      double lo = 0.0, hi = INFINITY;
      LANE_FOR(c, 2 * nz) {
        const int i = c >> 1;
        const double sv = (c & 1) ? v.sl[i] : v.su[i], cdi = qp_ineq(v, v.wd, v.dx, i);
        if (cdi == 0 || fabs(sv) >= 1e299) continue;
        const double t = -sv / cdi;
        if (!(t > 0)) continue;
        double d = b0 + a0 * t;
        for (int k = 0; k < nz; k++) { const double ck = qp_ineq(v, v.wd, v.dx, k); d += ck * imi * (fmax(v.su[k] + t * ck, 0.0) + fmin(v.sl[k] + t * ck, 0.0)); }
        if (d < 0) lo = fmax(lo, t); else hi = fmin(hi, t);
      }
      lo = qp_wmax(lo); hi = qp_wmin(hi);
      const double tm = isfinite(hi) ? 0.5 * (lo + hi) : lo + 1.0;
      double slope = 0, icpt = 0;
      LANE_FOR(i, nz) {
        const double cdi = qp_ineq(v, v.wd, v.dx, i);
        const double ci = cdi * imi;
        if (v.su[i] + tm * cdi > 0) { slope += ci * cdi; icpt += ci * v.su[i]; }
        if (v.sl[i] + tm * cdi < 0) { slope += ci * cdi; icpt += ci * v.sl[i]; }
      }
      slope = qp_wsum(slope); icpt = qp_wsum(icpt);
      double alpha = -(b0 + icpt) / (a0 + slope);
      alpha = fmin(fmax(alpha, lo), hi);
      if (!isfinite(alpha)) { failed = true; break; }
      double step = 0, xn = 1.0;
      LANE_FOR(i, n) { step = fmax(step, fabs(alpha * v.dx[i])); xn = fmax(xn, fabs(v.x[i])); }
      step = qp_wmax(step); xn = qp_wmax(xn);
      SYNC();
      PAR_FOR(i, n) v.x[i] += alpha * v.dx[i];
#ifdef QP_FRESH_WX
      SYNC();
      qp_wmatvec(v, v.x, v.wx);
#else
      PAR_FOR(w, v.nw) v.wx[w] += alpha * v.wd[w]; // W (x + alpha dx) = W x + alpha W dx: the products with dx are already there
      SYNC();
#endif
      QP_TICK(6);
      stalled = step <= 1e-14 * xn; // the Newton step is below the rounding level of x: leave after the next gradient evaluation
    }
    if (failed) { status = 2; break; }
    // ---- multiplier estimates at the inner solution (wx is W x for it), BCL test
    PAR_FOR(w, ne + nz) {
      if (w < ne) v.y[w] = v.ye[w] + (v.wx[w] - v.b[w]) / mue;
      else {
        const int i = w - ne;
        const double s = qp_ineq(v, v.wx, v.x, i);
        const double zu = qp_inf(v.up[i]) ? 0.0 : fmax(v.ze[i] + (s - v.up[i]) / mui, 0.0);
        const double zl = qp_inf(v.lo[i]) ? 0.0 : fmin(v.ze[i] + (s - v.lo[i]) / mui, 0.0);
        v.z[i] = zu + zl;
      }
    }
    SYNC();
    const double pri_new = qp_primal_residual(v);
    if (pri_new <= eta_ext) {
      eta_ext *= qp_pow(mui, st.beta_bcl);
      eta_in = fmax(eta_in * mui, eps_in_min);
    } else {
      SYNC();
      PAR_FOR(r, ne) v.y[r] = v.ye[r];
      PAR_FOR(i, nz) v.z[i] = v.ze[i];
      SYNC();
      const double nmui = fmax(mui * st.mu_update_factor, st.mu_min_in), nmue = fmax(mue * st.mu_update_factor, st.mu_min_eq);
      if (nmui != mui || nmue != mue) mu_updates++;
      if (nmue != mue) { qp_form_Q(v, st.rho, nmue); QP_TICK(3); }
      mui = nmui; mue = nmue;
      eta_ext = eta_ext_init * qp_pow(mui, st.alpha_bcl);
      eta_in = fmax(mui, eps_in_min);
    }
    QP_TICK(7);
  }
  QP_TDUMP(inst);
  SYNC();
  PAR_FOR(i, n) P.x[(long long)inst * n + i] = v.x[i];
  PAR_FOR(r, ne) P.y[(long long)inst * ne + r] = v.y[r];
  PAR_FOR(i, nz) P.z[(long long)inst * nz + i] = v.z[i];
  if (P.info) {
    ONE_THREAD {
      mpc_qp_info_t &o = P.info[inst];
      o.status = status; o.iter = it; o.iter_in = it_in; o.mu_updates = mu_updates;
      o.pri_res = R.pri; o.dua_res = R.dua; o.duality_gap = R.gap; o.objective = R.obj;
    }
  }
}

// IDSolver_ulim.computeMatrice (QP_utils.py:514-552) for one instance, nv = 28, nk = 2, 6-D contacts: fills A [40][62], b [40],
// C [18][62], l [18] of the handle from M, nle, Jc (LOCAL contact Jacobians, [12][28]), gamma [12], a [28], forces [12], cs [2].
HD void qp_assemble_id_group(const double *M, const double *nle, const double *Jc, const double *gamma, const double *a, const double *forces,
                             const int32_t *cs, double mu, double L, double W, double *A, double *b, double *C, double *l) {
  constexpr int nv = 28, nk = 2, fs = 6, nf = nk * fs, n = 2 * nv - 6 + nf, ne = nv + nf;
  PAR_FOR(e, ne * n) {
    const int r = e / n, c = e % n;
    double val = 0;
    if (r < nv) {
      if (c < nv) val = M[r * nv + c];
      else if (c < nv + nf) val = cs[(c - nv) / fs] ? -Jc[(c - nv) * nv + r] : 0.0;
      else val = (r >= 6 && c - nv - nf == r - 6) ? -1.0 : 0.0;
    } else if (c < nv) val = cs[(r - nv) / fs] ? Jc[(r - nv) * nv + c] : 0.0;
    A[e] = val;
  }
  PAR_FOR(r, ne) {
    double s;
    if (r < nv) {
      s = -nle[r];
      for (int j = 0; j < nv; j++) s -= M[r * nv + j] * a[j];
      for (int k = 0; k < nf; k++) if (cs[k / fs]) s += Jc[k * nv + r] * forces[k];
    } else {
      const int k = r - nv;
      s = 0;
      if (cs[k / fs]) { s = -gamma[k]; for (int j = 0; j < nv; j++) s -= Jc[k * nv + j] * a[j]; }
    }
    b[r] = s;
  }
  PAR_FOR(e, 9 * nk * n) {
    const int r = e / n, c = e % n, i = r / 9, rr = r % 9, cc = c - nv - i * fs;
    double val = 0;
    if (cs[i] && cc >= 0 && cc < fs) {
      // Cmin as written at QP_utils.py:474-484 (rows 2 and 3 repeat the x rows there)
      if (rr < 4) val = (cc == 0) ? ((rr & 1) ? 1.0 : -1.0) : (cc == 2 ? mu : 0.0);
      else if (rr == 4) val = (cc == 2) ? 1.0 : 0.0;
      else if (rr < 7) val = (cc == 2) ? W : (cc == 3 ? ((rr == 5) ? -1.0 : 1.0) : 0.0);
      else val = (cc == 2) ? L : (cc == 4 ? ((rr == 7) ? -1.0 : 1.0) : 0.0);
    }
    C[e] = val;
  }
  PAR_FOR(r, 9 * nk) {
    const int i = r / 9, rr = r % 9;
    const double *f = forces + i * fs;
    double val = 0;
    if (cs[i]) {
      switch (rr) { // QP_utils.py:538-548
      case 0: val = f[0] - f[2] * mu; break;
      case 1: val = -f[0] - f[2] * mu; break;
      case 2: val = f[1] - f[2] * mu; break;
      case 3: val = -f[1] - f[2] * mu; break;
      case 4: val = -f[2]; break;
      case 5: val = f[3] - f[2] * W; break;
      case 6: val = -f[3] - f[2] * W; break;
      case 7: val = f[4] - f[2] * L; break;
      default: val = -f[4] - f[2] * L; break;
      }
    }
    l[r] = val;
  }
}

// IKIDSolver_f6.computeMatrice (QP_utils.py:677-738) for one instance, nv = 28, two 6-D contacts: fills H [62][62], g [62] and, through
// qp_assemble_id_group with a = 0 and gamma = dJv on the active contacts, A, b, C, l.  Inputs per instance: M, nle, Jc, dJv, Ag [6][28],
// dAgv [6], Jang [2][3][28] (base, torso), dJang [2][3], task [98] (q_diff 28, dq_diff 28, LF 6, dLF 6, RF 6, dRF 6, base 3, dbase 3,
// torso 3, dtorso 3, dH 6), forces, cs; shared: weights [5], gains [1658] (Kp_q, Kd_q 28 x 28, Kp_f, Kd_f 6 x 6, Kp_b, Kd_b 3 x 3, row-major).
// sm: 24 * 28 + 24 + 12 + 28 doubles of the group's shared memory.
//   H[:28,:28] = w0 I + w1 (JL'JL + JR'JR) + w2 Ag'Ag + w3 (Jb'Jb + Jt'Jt),   H[28:40,28:40] = w4 I,   zeros elsewhere
//   g[:28] = -w0 (Kp_q q_diff + Kd_q dq_diff) + sum_k w_k r_k' J_k over the task rows J_k = (JL, JR, Ag, Jb, Jt) with
//            r = dJv_L - Kp_f LF - Kd_f dLF,  dJv_R - Kp_f RF - Kd_f dRF,  dAgv - dH,  dJv_b - Kp_b base - Kd_b dbase,  same for the torso
HD void qp_assemble_ikid_group(const double *M, const double *nle, const double *Jc, const double *dJv, const double *Ag, const double *dAgv, const double *Jang,
                               const double *dJang, const double *task, const double *forces, const int32_t *cs, const double *wt, const double *gains,
                               double mu, double L, double W, double *sm, double *H, double *g, double *A, double *b, double *C, double *l) {
  constexpr int nv = 28, n = 62, NR = 24;
  const double *Kpq = gains, *Kdq = Kpq + nv * nv, *Kpf = Kdq + nv * nv, *Kdf = Kpf + 36, *Kpb = Kdf + 36, *Kdb = Kpb + 9;
  double *J = sm, *r = J + NR * nv, *gamma = r + NR, *a = gamma + 12; // task rows JL, JR, Ag, Jb, Jt; their residuals; gamma; a = 0
  PAR_FOR(e, NR * nv) {
    const int k = e / nv, c = e % nv;
    J[e] = k < 12 ? Jc[e] : k < 18 ? Ag[(k - 12) * nv + c] : Jang[(k - 18) * nv + c];
  }
  PAR_FOR(k, NR) {
    double s;
    if (k < 12) { // contact rows: K_f is 6 x 6 over the rows of one foot
      const int f = k / 6, i = k % 6;
      const double *e = task + 56 + 12 * f, *de = e + 6;
      s = dJv[k];
      for (int j = 0; j < 6; j++) s -= Kpf[6 * i + j] * e[j] + Kdf[6 * i + j] * de[j];
    } else if (k < 18) s = dAgv[k - 12] - task[92 + k - 12];
    else { // base / torso rows: K_b is 3 x 3
      const int f = (k - 18) / 3, i = (k - 18) % 3;
      const double *e = task + 80 + 6 * f, *de = e + 3;
      s = dJang[k - 18];
      for (int j = 0; j < 3; j++) s -= Kpb[3 * i + j] * e[j] + Kdb[3 * i + j] * de[j];
    }
    r[k] = s;
  }
  PAR_FOR(k, 12) gamma[k] = cs[k / 6] ? dJv[k] : 0.0;
  PAR_FOR(j, nv) a[j] = 0.0;
  SYNC();
  PAR_FOR(e, n * n) {
    const int i = e / n, j = e % n;
    double v = 0;
    if (i < nv && j < nv) {
      double s1 = 0, s2 = 0, s3 = 0;
      for (int k = 0; k < 12; k++) s1 += J[k * nv + i] * J[k * nv + j];
      for (int k = 12; k < 18; k++) s2 += J[k * nv + i] * J[k * nv + j];
      for (int k = 18; k < NR; k++) s3 += J[k * nv + i] * J[k * nv + j];
      v = (i == j ? wt[0] : 0.0) + wt[1] * s1 + wt[2] * s2 + wt[3] * s3;
    } else if (i == j && i >= nv && i < nv + 12) v = wt[4];
    H[e] = v;
  }
  PAR_FOR(i, n) {
    double v = 0;
    if (i < nv) {
      double p = 0, s1 = 0, s2 = 0, s3 = 0;
      for (int j = 0; j < nv; j++) p += Kpq[i * nv + j] * task[j] + Kdq[i * nv + j] * task[nv + j];
      for (int k = 0; k < 12; k++) s1 += r[k] * J[k * nv + i];
      for (int k = 12; k < 18; k++) s2 += r[k] * J[k * nv + i];
      for (int k = 18; k < NR; k++) s3 += r[k] * J[k * nv + i];
      v = -wt[0] * p + wt[1] * s1 + wt[2] * s2 + wt[3] * s3;
    }
    g[i] = v;
  }
  qp_assemble_id_group(M, nle, Jc, gamma, a, forces, cs, mu, L, W, A, b, C, l);
}

} // namespace mpcdev
