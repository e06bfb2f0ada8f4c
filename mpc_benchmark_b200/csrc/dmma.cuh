// FP64 tensor-core GEMM on shared-memory operands (mma.sync.aligned.m8n8k4.f64 -> SASS DMMA.8x8x4).
//
// tcgen05/TMEM have no fp64 path on Blackwell, so dense fp64 contractions use the legacy DMMA pipe (same nominal
// peak as DFMA on B200, but 256 FMAs per warp instruction instead of 32: far lower issue and shared-memory
// pressure).  Used only where the stage matrices really are dense contractions (BASELINE north_star): Lambda^-1 P,
// Pt [A B] and [A B]' W in the proximal Riccati recursion.
//
// All products are in "TN" form C = A^T B with A stored [K][lda], B stored [K][ldb] (row-major), so both fragments
// read 8 consecutive doubles per k-row: conflict-free for leading dimensions = 8 (mod 16) doubles.
// Fragment layout (PTX ISA, m8n8k4 .f64): lane = 4*g + t;  a: A^T[row g][k t];  b: B[k t][col g];  c0,c1: C[row g][cols 2t, 2t+1].
#pragma once
#include "dev_common.cuh"
#ifdef MPC_HOST_EMU
#include <vector>
#endif

namespace mpcdev {

#ifdef MPC_HOST_EMU
// host reference of mma_tn and mma_tn_g
inline void mma_tn_ref(int mt, int nt, int K, const double *A, int lda, const double *B, int ldb, double *C, int ldc, const double *Cinit, int ldci,
                       int vr, int vc, bool upper_only, double *Cg, int ldcg, int vcg, double *C2 = nullptr, int ldc2 = 0) {
  for (int i = 0; i < 8 * mt; i++)
    for (int j = 0; j < 8 * nt; j++) {
      if (upper_only && (j / 16) < (i / 16)) continue;
      double s = (Cinit && i < vr && j < vc) ? Cinit[i * ldci + j] : 0.0;
      for (int k = 0; k < K; k++) s += A[k * lda + i] * B[k * ldb + j];
      C[i * ldc + j] = s;
      if (C2) C2[i * ldc2 + j] = s;
      if (Cg && j < vcg) Cg[i * ldcg + j] = s;
    }
  if (upper_only)
    for (int i = 0; i < 8 * mt; i++)
      for (int j = 0; j < 8 * nt; j++)
        if ((j / 16) < (i / 16) && i < (Cinit ? vc : 8 * nt)) {
          C[i * ldc + j] = C[j * ldc + i];
          if (C2) C2[i * ldc2 + j] = C[j * ldc + i];
        }
}
#else
__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Tile walk shared by the products: each warp takes 2 x 2 blocks of tiles, four independent accumulator chains c[a][b] (tile row
// ti + a, tile column tj + b) that share the A and B fragments.  r2 / c2: whether the second tile row / column exists.
struct TilePair {
  int bi, bj, ti, tj;
  bool r2, c2;
};
__device__ __forceinline__ int tile_pair_count(int mt, int nt, bool upper) {
  const int mtp = (mt + 1) / 2, ntp = (nt + 1) / 2;
  return upper ? mtp * (mtp + 1) / 2 : mtp * ntp;
}
// work item p: row-major over the block grid, or (upper: square, symmetric result) over the blocks on or above the block diagonal,
// enumerated compactly so that the warps stay balanced
__device__ __forceinline__ TilePair tile_pair(int p, int mt, int nt, bool upper) {
  const int mtp = (mt + 1) / 2, ntp = (nt + 1) / 2;
  TilePair w;
  if (upper) { w.bi = 0; int q = p; while (q >= mtp - w.bi) { q -= mtp - w.bi; w.bi++; } w.bj = w.bi + q; } else { w.bi = p / ntp; w.bj = p % ntp; }
  w.ti = w.bi * 2; w.tj = w.bj * 2;
  w.r2 = (w.ti + 1 < mt); w.c2 = (w.tj + 1 < nt);
  return w;
}
// one 4-row k-step of all four chains
__device__ __forceinline__ void dmma_2x2(double (&c)[2][2][2], double a0, double a1, double b0, double b1) {
  dmma_8x8x4(c[0][0][0], c[0][0][1], a0, b0);
  dmma_8x8x4(c[0][1][0], c[0][1][1], a0, b1);
  dmma_8x8x4(c[1][0][0], c[1][0][1], a1, b0);
  dmma_8x8x4(c[1][1][0], c[1][1][1], a1, b1);
}
// accumulators = Cinit (ldci) restricted to rows < vr and columns < vc, zero outside (all zero when Cinit == nullptr)
__device__ __forceinline__ void acc_init(double (&c)[2][2][2], const TilePair &w, int g, int t, const double *Cinit, int ldci, int vr, int vc) {
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) {
      c[a][b][0] = 0.0; c[a][b][1] = 0.0;
      const int row = (w.ti + a) * 8 + g, col = (w.tj + b) * 8 + 2 * t;
      if (Cinit && row < vr && (a == 0 || w.r2) && (b == 0 || w.c2)) {
        if (col < vc) c[a][b][0] = Cinit[row * ldci + col];
        if (col + 1 < vc) c[a][b][1] = Cinit[row * ldci + col + 1];
      }
    }
}
// store the existing tiles to C (and the same entries to the shared-memory copy C2, if any; ldc2 even), and their columns < vcg to
// the global mirror Cg (if any; vcg, ldcg even).  mirror: the block lies above the diagonal of a symmetric result and is also stored
// transposed (never a tile anyone reads as Cinit); columns >= vcm are scratch and stay out of the rows below
__device__ __forceinline__ void acc_store(const double (&c)[2][2][2], const TilePair &w, int g, int t, double *C, int ldc, double *Cg, int ldcg, int vcg,
                                          bool mirror, int vcm, double *C2 = nullptr, int ldc2 = 0) {
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) {
      if ((a == 1 && !w.r2) || (b == 1 && !w.c2)) continue;
      const int row = (w.ti + a) * 8 + g, col = (w.tj + b) * 8 + 2 * t;
      *reinterpret_cast<double2 *>(C + row * ldc + col) = make_double2(c[a][b][0], c[a][b][1]);
      if (C2) *reinterpret_cast<double2 *>(C2 + row * ldc2 + col) = make_double2(c[a][b][0], c[a][b][1]);
      if (Cg && col < vcg) *reinterpret_cast<double2 *>(Cg + row * ldcg + col) = make_double2(c[a][b][0], c[a][b][1]);
      if (mirror) {
        if (col < vcm) { C[col * ldc + row] = c[a][b][0]; if (C2) C2[col * ldc2 + row] = c[a][b][0]; }
        if (col + 1 < vcm) { C[(col + 1) * ldc + row] = c[a][b][1]; if (C2) C2[(col + 1) * ldc2 + row] = c[a][b][1]; }
      }
    }
}
#endif

// C (8*mt x 8*nt, ldc) = init + A^T B,  K multiple of 4.
//   init: 0 (Cinit == nullptr) or Cinit (ldci) restricted to rows < vr and cols < vc (zero outside) — lets the
//   Hessian update read H_k straight from global memory while keeping the shared copy zero-padded.
// upper_only: square symmetric result; only the 16 x 16 blocks on / above the block diagonal are computed, the rest is mirrored.
// C2 (optional, ldc2 even): a second copy of the result, stored from the accumulators with it.
HD void mma_tn(int mt, int nt, int K, const double *A, int lda, const double *B, int ldb, double *C, int ldc, const double *Cinit, int ldci,
               int vr, int vc, bool upper_only, double *C2 = nullptr, int ldc2 = 0) {
#ifdef MPC_HOST_EMU
  mma_tn_ref(mt, nt, K, A, lda, B, ldb, C, ldc, Cinit, ldci, vr, vc, upper_only, nullptr, 0, 0, C2, ldc2);
#else
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int nwork = tile_pair_count(mt, nt, upper_only), vcm = Cinit ? vc : 8 * nt;
  for (int p = warp; p < nwork; p += nwarps) {
    const TilePair w = tile_pair(p, mt, nt, upper_only);
    double c[2][2][2];
    acc_init(c, w, g, t, Cinit, ldci, vr, vc);
    const double *ap = A + t * lda + w.ti * 8 + g;
    const double *bp = B + t * ldb + w.tj * 8 + g;
    const int ao = w.r2 ? 8 : 0, bo = w.c2 ? 8 : 0; // out-of-range partner tiles recompute tile 0 (discarded)
#pragma unroll 2
    for (int k0 = 0; k0 < K; k0 += 4) {
      const double a0 = ap[k0 * lda], a1 = ap[k0 * lda + ao], b0 = bp[k0 * ldb], b1 = bp[k0 * ldb + bo];
      dmma_2x2(c, a0, a1, b0, b1);
    }
    acc_store(c, w, g, t, C, ldc, nullptr, 0, 0, upper_only && w.bi < w.bj, vcm, C2, ldc2);
  }
#endif
  SYNC();
}

// Same contraction as mma_tn with K fixed at compile time: the k-loop runs in two halves, and each half loads the fragments of its
// K/2 rows of both operands before its DMMAs, so that they are in flight together.  The result also goes to the global-memory
// mirror Cg (columns < vcg), straight from the accumulators.
template <int K>
HD void mma_tn_g(int mt, int nt, const double *A, int lda, const double *B, int ldb, double *C, int ldc, const double *Cinit, int ldci,
                 int vr, int vc, bool upper_only, double *Cg, int ldcg, int vcg) {
#ifdef MPC_HOST_EMU
  mma_tn_ref(mt, nt, K, A, lda, B, ldb, C, ldc, Cinit, ldci, vr, vc, upper_only, Cg, ldcg, vcg);
#else
  static_assert(K % 8 == 0, "k-loop is unrolled in two halves of whole 4-row steps");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int nwork = tile_pair_count(mt, nt, upper_only), vcm = Cinit ? vc : 8 * nt;
  for (int p = warp; p < nwork; p += nwarps) {
    const TilePair w = tile_pair(p, mt, nt, upper_only);
    double c[2][2][2];
    acc_init(c, w, g, t, Cinit, ldci, vr, vc);
    const int ao = w.r2 ? 8 : 0, bo = w.c2 ? 8 : 0; // out-of-range partner tiles recompute tile 0 (discarded)
    const double *ap = A + t * lda + w.ti * 8 + g;
    const double *bp = B + t * ldb + w.tj * 8 + g;
    constexpr int KH = K / 2, NS = KH / 4;
#pragma unroll 1
    for (int kc = 0; kc < K; kc += KH) {
      double a0[NS], a1[NS], b0[NS], b1[NS];
#pragma unroll
      for (int s = 0; s < NS; s++) {
        const int k0 = kc + 4 * s;
        a0[s] = ap[k0 * lda]; a1[s] = ap[k0 * lda + ao];
        b0[s] = bp[k0 * ldb]; b1[s] = bp[k0 * ldb + bo];
      }
#pragma unroll
      for (int s = 0; s < NS; s++) dmma_2x2(c, a0[s], a1[s], b0[s], b1[s]);
    }
    acc_store(c, w, g, t, C, ldc, Cg, ldcg, vcg, upper_only && w.bi < w.bj, vcm);
  }
#endif
  SYNC();
}

// Symmetric update C = Cinit + A^T B (C: 8 nt x 8 nt, result symmetric) whose OUTPUT BUFFER ALIASES THE A OPERAND: every warp keeps
// the accumulators of all its 16 x 16 blocks (upper block triangle, at most MAXQ per warp) in registers, the CTA synchronises once
// all operand reads are done, and only then the blocks and their mirrors are stored.  A, B: shared memory, [K][lda] / [K][ldb];
// Cinit: global, rows < vr / columns < vc (zero outside).  Mirrored entries whose source column is >= vc are written as zero (those
// columns are scratch: they must not reach the rows below).
template <int K, int MAXQ>
HD void mma_sym_deferred(int nt, const double *A, int lda, const double *B, int ldb, double *C, int ldc, const double *Cinit, int ldci, int vr, int vc) {
#ifdef MPC_HOST_EMU
  std::vector<double> out((size_t)64 * nt * nt);
  for (int i = 0; i < 8 * nt; i++)
    for (int j = 0; j < 8 * nt; j++) {
      if ((j / 16) < (i / 16)) continue;
      double s = (i < vr && j < vc) ? Cinit[i * ldci + j] : 0.0;
      for (int k = 0; k < K; k++) s += A[k * lda + i] * B[k * ldb + j];
      out[(size_t)i * 8 * nt + j] = s;
    }
  for (int i = 0; i < 8 * nt; i++)
    for (int j = 0; j < 8 * nt; j++) C[i * ldc + j] = ((j / 16) < (i / 16)) ? ((i < vc) ? out[(size_t)j * 8 * nt + i] : 0.0) : out[(size_t)i * 8 * nt + j];
#else
  static_assert(K % 4 == 0, "whole 4-row steps");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int nwork = tile_pair_count(nt, nt, true);
  double c[MAXQ][2][2][2];
#pragma unroll
  for (int q_ = 0; q_ < MAXQ; q_++) { // initial values of every block first: all L2 reads of this warp in flight together
    const int p = warp + q_ * nwarps;
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 2; b++) { c[q_][a][b][0] = 0.0; c[q_][a][b][1] = 0.0; }
    if (p < nwork) {
      const TilePair w = tile_pair(p, nt, nt, true);
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const int row = (w.ti + a) * 8 + g, col = (w.tj + b) * 8 + 2 * t;
          if (row < vr && (a == 0 || w.r2) && (b == 0 || w.c2)) {
            if (col + 1 < vc) { const double2 v = __ldcg(reinterpret_cast<const double2 *>(Cinit + row * ldci + col)); c[q_][a][b][0] = v.x; c[q_][a][b][1] = v.y; }
            else if (col < vc) c[q_][a][b][0] = __ldcg(Cinit + row * ldci + col);
          }
        }
    }
  }
#pragma unroll
  for (int q_ = 0; q_ < MAXQ; q_++) {
    const int p = warp + q_ * nwarps;
    if (p < nwork) {
      const TilePair w = tile_pair(p, nt, nt, true);
      const int ao = w.r2 ? 8 : 0, bo = w.c2 ? 8 : 0;
      const double *ap = A + t * lda + w.ti * 8 + g;
      const double *bp = B + t * ldb + w.tj * 8 + g;
#pragma unroll 2
      for (int s = 0; s < K / 4; s++) {
        const double a0 = ap[4 * s * lda], a1 = ap[4 * s * lda + ao], b0 = bp[4 * s * ldb], b1 = bp[4 * s * ldb + bo];
        dmma_2x2(c[q_], a0, a1, b0, b1);
      }
    }
  }
  SYNC(); // every read of A (and of anything else the output buffer aliases) is complete
#pragma unroll
  for (int q_ = 0; q_ < MAXQ; q_++) {
    const int p = warp + q_ * nwarps;
    if (p < nwork) {
      const TilePair w = tile_pair(p, nt, nt, true);
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          if ((a == 1 && !w.r2) || (b == 1 && !w.c2)) continue;
          const int row = (w.ti + a) * 8 + g, col = (w.tj + b) * 8 + 2 * t;
          *reinterpret_cast<double2 *>(C + row * ldc + col) = make_double2(c[q_][a][b][0], c[q_][a][b][1]);
          if (w.bi < w.bj) {
            C[col * ldc + row] = (col < vc) ? c[q_][a][b][0] : 0.0;
            C[(col + 1) * ldc + row] = (col + 1 < vc) ? c[q_][a][b][1] : 0.0;
          }
        }
    }
  }
#endif
  SYNC();
}

// ---- warp-level 8 x 8 tile kernels of the tensor-core Cholesky (all operands inside one row-major matrix A, leading dim ld)
// C(i0.., j0..) -= L(i0.., k0..k0+8) * L(j0.., k0..k0+8)^T
HD void tile_syrk(double *A, int ld, int i0, int j0, int k0) {
#ifdef MPC_HOST_EMU
  for (int r = 0; r < 8; r++)
    for (int c = 0; c < 8; c++) {
      double s = 0;
      for (int q = 0; q < 8; q++) s += A[(i0 + r) * ld + k0 + q] * A[(j0 + c) * ld + k0 + q];
      A[(i0 + r) * ld + j0 + c] -= s;
    }
#else
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const double *ar = A + (i0 + g) * ld + k0 + t, *br = A + (j0 + g) * ld + k0 + t;
  const double a0 = -ar[0], a1 = -ar[4], b0 = br[0], b1 = br[4];
  double2 *cp = reinterpret_cast<double2 *>(A + (i0 + g) * ld + j0 + 2 * t);
  double2 c = *cp;
  dmma_8x8x4(c.x, c.y, a0, b0);
  dmma_8x8x4(c.x, c.y, a1, b1);
  *cp = c;
#endif
}
// L(i0.., k0..k0+8) = A(i0.., k0..k0+8) * Di^T   (Di: 8 x 8 row-major inverse of the diagonal block's factor), in place
HD void tile_trsm(double *A, int ld, int i0, int k0, const double *Di) {
#ifdef MPC_HOST_EMU
  for (int r = 0; r < 8; r++) {
    double o[8];
    for (int c = 0; c < 8; c++) { double s = 0; for (int q = 0; q <= c; q++) s += A[(i0 + r) * ld + k0 + q] * Di[c * 8 + q]; o[c] = s; }
    for (int c = 0; c < 8; c++) A[(i0 + r) * ld + k0 + c] = o[c];
  }
#else
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const double *ar = A + (i0 + g) * ld + k0 + t;
  const double a0 = ar[0], a1 = ar[4], b0 = Di[g * 8 + t], b1 = Di[g * 8 + 4 + t];
  double2 c = make_double2(0.0, 0.0);
  dmma_8x8x4(c.x, c.y, a0, b0);
  dmma_8x8x4(c.x, c.y, a1, b1);
  __syncwarp();
  *reinterpret_cast<double2 *>(A + (i0 + g) * ld + k0 + 2 * t) = c;
#endif
}

#ifndef MPC_HOST_EMU
// One block row ib of trsm_mma's substitution on the column tiles zc (leading dimension lz) and, if two, zd (lw):
//   R_i = Z_i - sum_k L_ik Z_k (DMMA, two accumulator chains),  Z_i <- Dinv_i R_i (DMMA; the tile itself is the scratch that turns
// the accumulator layout into the B-fragment layout).  Forward: k < i.  BACK: the backward step, with L' and Dinv' and k > i.
template <int NB, bool BACK>
__device__ __forceinline__ void trsm_block_row(int ib, const double *A, int ld, const double *Dinv, double *zc, int lz, double *zd, int lw, bool two, int g, int t) {
  double2 *cp = reinterpret_cast<double2 *>(zc + (8 * ib + g) * lz + 2 * t), *dp = reinterpret_cast<double2 *>(zd + (8 * ib + g) * lw + 2 * t);
  double2 c = *cp, d = *dp;
  double e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0;
#pragma unroll
  for (int kb = BACK ? ib + 1 : 0; kb < (BACK ? NB : ib); kb++) {
    const double *pa = BACK ? A + (8 * kb + t) * ld + 8 * ib + g : A + (8 * ib + g) * ld + 8 * kb + t; // BACK: (L_ki)'[g][t] = L_ki[t][g]
    const double a0 = -pa[0], a1 = -pa[BACK ? 4 * ld : 4];
    const double *pb = zc + (8 * kb + t) * lz + g, *pd = zd + (8 * kb + t) * lw + g;
    dmma_8x8x4(c.x, c.y, a0, pb[0]);
    dmma_8x8x4(e0, e1, a1, pb[4 * lz]);
    if (two) { dmma_8x8x4(d.x, d.y, a0, pd[0]); dmma_8x8x4(f0, f1, a1, pd[4 * lw]); }
  }
  c.x += e0; c.y += e1; d.x += f0; d.y += f1;
  *cp = c;
  if (two) *dp = d;
  __syncwarp();
  const double b0 = zc[(8 * ib + t) * lz + g], b1 = zc[(8 * ib + 4 + t) * lz + g];
  const double h0 = zd[(8 * ib + t) * lw + g], h1 = zd[(8 * ib + 4 + t) * lw + g];
  __syncwarp();
  const double *Di = Dinv + 64 * ib;
  const double q0 = BACK ? Di[t * 8 + g] : Di[g * 8 + t], q1 = BACK ? Di[(4 + t) * 8 + g] : Di[g * 8 + 4 + t];
  double2 r = make_double2(0.0, 0.0), u = make_double2(0.0, 0.0);
  dmma_8x8x4(r.x, r.y, q0, b0);
  if (two) dmma_8x8x4(u.x, u.y, q0, h0);
  dmma_8x8x4(r.x, r.y, q1, b1);
  if (two) dmma_8x8x4(u.x, u.y, q1, h1);
  *cp = r;
  if (two) *dp = u;
  __syncwarp();
}
#endif

// In-place solve (L L')^-1 B on the tensor pipe, L = 8 NB x 8 NB factor left by chol_mma (strictly-lower tiles of A plus the
// inverses Dinv of its diagonal blocks).  B consists of `nt` column tiles of 8 columns: tile ct < nt_main lives in Bm (leading
// dimension ldb, columns 8 ct ..), the remaining tiles in Bx (leading dimension ldx).  ONE WARP PER COLUMN TILE runs the whole
// forward and backward substitution on its own 8 columns (trsm_block_row) — no block barriers, only warp-level ones: 2 NB short
// dependent steps per tile.
template <int NB> HD void trsm_mma(const double *A, int ld, const double *Dinv, double *Bm, int ldb, int nt_main, double *Bx, int ldx, int nt) {
#ifdef MPC_HOST_EMU
  trsm_blocked(A, 8 * NB, ld, Dinv, Bm, 8 * nt_main, ldb);
  if (nt > nt_main) trsm_blocked(A, 8 * NB, ld, Dinv, Bx, 8 * (nt - nt_main), ldx);
#else
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3, nw = blockDim.x >> 5;
  // a warp takes TWO column tiles per pass when there are enough of them (ct and ct + nw): two independent substitution chains
  // interleave in the same instruction stream and hide each other's DMMA / shared-memory latencies
  for (int ct = (threadIdx.x >> 5); ct < nt; ct += 2 * nw) {
    const int ct2 = ct + nw;
    const bool two = ct2 < nt;
    double *zc = (ct < nt_main) ? Bm + 8 * ct : Bx + 8 * (ct - nt_main);
    const int lz = (ct < nt_main) ? ldb : ldx;
    double *zd = !two ? zc : (ct2 < nt_main) ? Bm + 8 * ct2 : Bx + 8 * (ct2 - nt_main);
    const int lw = !two ? lz : (ct2 < nt_main) ? ldb : ldx;
#pragma unroll
    for (int ib = 0; ib < NB; ib++) trsm_block_row<NB, false>(ib, A, ld, Dinv, zc, lz, zd, lw, two, g, t); // Y_i = Dinv_i (B_i - sum_{k<i} L_ik Y_k)
#pragma unroll
    for (int ib = NB - 1; ib >= 0; ib--) trsm_block_row<NB, true>(ib, A, ld, Dinv, zc, lz, zd, lw, two, g, t); // X_i = Dinv_i' (Y_i - sum_{k>i} L_ki' X_k)
  }
#endif
  SYNC();
}

// Tensor-core blocked Cholesky (lower, in place) for n = 8 NB with a one-panel lookahead: per panel the tiles below the
// diagonal block are solved (one warp per tile), the next panel's column of tiles is updated, then thread 0 factors and
// inverts the next diagonal block in registers while warps 1.. update the remaining tiles of the trailing matrix.
// Only the lower triangle (and the full diagonal tiles) of A is referenced; Dinv receives the NB inverses of the diagonal blocks.
template <int NB> HD void chol_mma(double *A, int ld, double *Dinv) {
  DIAG_BLOCK(A, 0, 8, ld, Dinv);
  SYNC();
  for (int kb = 0; kb + 1 < NB; kb++) {
    const int k0 = 8 * kb, nt = NB - 1 - kb;
    const double *Di = Dinv + 64 * kb;
    WARP_TILE_FOR(p, nt) tile_trsm(A, ld, 8 * (kb + 1 + p), k0, Di);
    SYNC();
    // warp 0: the next diagonal tile's update, then its factorisation — the serial chain of the whole factorisation never leaves this warp
    // between two block barriers; the other warps: the rest of the next panel's column and of the trailing matrix
    if (IS_WARP0) tile_syrk(A, ld, 8 * (kb + 1), 8 * (kb + 1), k0);
    WARP_SYNC();
    DIAG_BLOCK(A, 8 * (kb + 1), 8, ld, Dinv + 64 * (kb + 1));
    const int m = nt - 1;
    WARP_TILE_FOR_REST(p, m + m * (m + 1) / 2) {
      if (p < m) tile_syrk(A, ld, 8 * (kb + 2 + p), 8 * (kb + 1), k0);
      else {
        const int q = p - m;
        int ti = 0;
        while ((ti + 1) * (ti + 2) / 2 <= q) ti++;
        const int tj = q - ti * (ti + 1) / 2;
        tile_syrk(A, ld, 8 * (kb + 2 + ti), 8 * (kb + 2 + tj), k0);
      }
    }
    SYNC();
  }
}

} // namespace mpcdev
