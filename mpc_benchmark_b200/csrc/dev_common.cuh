// Common device helpers for the sm_100a kernels.
//
// Kernel bodies are written as block-cooperative phases: `PAR_FOR(i, n)` distributes n independent work
// items over the threads of the CTA, `SYNC()` separates dependent phases, and every value that crosses a
// phase boundary lives in shared memory.  Under MPC_HOST_EMU (tests/_emu only — never part of the product
// library) the same source compiles with g++, PAR_FOR becomes a serial loop and SYNC a no-op, which lets the
// CPU test-suite check kernel logic against the oracle without a GPU.  The product path has NO CPU fallback.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef MPC_HOST_EMU
#define HD inline
#define PAR_FOR(i, n) for (int i = 0; i < (n); i++)
#define SYNC() ((void)0)
#define ONE_THREAD if (true)
#define TID 0
#define NTHREADS 1
#define IS_WARP0 true
#define WARP_FOR(i, n) for (int i = 0; i < (n); i++)
#define WARP_SYNC() ((void)0)
#define ATOMIC_INC(p) ((*(p))++)
#define WARP_TILE_FOR(p, n) for (int p = 0; p < (n); p++)
#define WARP_TILE_FOR_REST(p, n) for (int p = 0; p < (n); p++)
#define LANE_FOR(j, n) for (int j = 0; j < (n); j++)
#define WARP_SUM(x) (x)
#define LANE0 true
#define WARP_ID 0
#define NWARPS 1
#define MBAR_INIT(bar, count) ((void)0)
#define MBAR_EXPECT_TX(bar, bytes) ((void)0)
#define MBAR_WAIT(bar, parity) ((void)0)
#define FENCE_PROXY_ASYNC() ((void)0)
#define PREFETCH_L2(ptr, bytes) ((void)0)
#define PREFETCH_LINES(ptr, bytes) ((void)0)
#define LDCG(p) (*(p))
#define BULK_G2S(dst, src, bytes, bar) do { for (size_t i_ = 0; i_ < (size_t)(bytes) / 8; i_++) (dst)[i_] = (src)[i_]; } while (0)
struct double2 { double x, y; };
inline double2 make_double2(double x, double y) { return double2{x, y}; }
#else
#define HD __device__ __forceinline__
#define PAR_FOR(i, n) for (int i = threadIdx.x; i < (n); i += blockDim.x)
// A CTA holds blockDim.y independent GROUPS of blockDim.x threads (one work item each; evaluation kernels: one knot per
// group, several knots per CTA so that the groups run the same code side by side and share instruction fetches).  All
// cooperative phases are per group: work is spread over threadIdx.x and SYNC() is the group's own named barrier.
#define SYNC() asm volatile("bar.sync %0, %1;" ::"r"((int)threadIdx.y + 1), "r"((int)blockDim.x) : "memory")
#define ONE_THREAD if (threadIdx.x == 0)
#define TID ((int)threadIdx.x)
#define NTHREADS ((int)blockDim.x)
#define IS_WARP0 (threadIdx.x < 32)
#define WARP_FOR(i, n) for (int i = (threadIdx.x & 31); i < (n); i += 32)
#define WARP_SYNC() __syncwarp()
#define ATOMIC_INC(p) atomicAdd((p), 1)
// one 8 x 8 tile per warp: over all warps / over all warps except warp 0
#define WARP_TILE_FOR(p, n) for (int p = (threadIdx.x >> 5); p < (n); p += (blockDim.x >> 5))
#define WARP_TILE_FOR_REST(p, n) for (int p = (int)(threadIdx.x >> 5) - 1; p >= 0 && p < (n); p += (blockDim.x >> 5) - 1)
// matrix-vector pattern: rows over warps, columns over lanes (coalesced / conflict-free), butterfly reduction
#define LANE_FOR(j, n) for (int j = (threadIdx.x & 31); j < (n); j += 32)
#define WARP_SUM(x) mpcdev::warp_sum(x)
#define LANE0 ((threadIdx.x & 31) == 0)
#define WARP_ID ((int)(threadIdx.x >> 5))
#define NWARPS ((int)(blockDim.x >> 5))
// TMA-style bulk copies (cp.async.bulk, one instruction per contiguous block, completion counted in bytes on an mbarrier):
// ONE thread arms the barrier with the expected bytes and issues the copies; every consumer waits on the barrier's phase
// parity.  dst / src 16-byte aligned, bytes a multiple of 16.  FENCE_PROXY_ASYNC orders earlier generic-proxy accesses
// of a shared buffer before the async proxy overwrites it.
#define MBAR_INIT(bar, count) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"((unsigned)(count)) : "memory")
#define MBAR_EXPECT_TX(bar, bytes) \
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"((unsigned)(bytes)) : "memory")
#define BULK_G2S(dst, src, bytes, bar)                                                                                   \
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(          \
                   (unsigned)__cvta_generic_to_shared(dst)),                                                             \
               "l"(src), "r"((unsigned)(bytes)), "r"((unsigned)__cvta_generic_to_shared(bar))                            \
               : "memory")
#define MBAR_WAIT(bar, parity)                                                                                                           \
  asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}" ::"r"( \
                   (unsigned)__cvta_generic_to_shared(bar)),                                                                             \
               "r"((unsigned)(parity))                                                                                                   \
               : "memory")
#define FENCE_PROXY_ASYNC() asm volatile("fence.proxy.async.shared::cta;" ::: "memory")
// bulk prefetch of a contiguous global block into L2 (one instruction; address and size multiples of 16 bytes)
#define PREFETCH_L2(ptr, bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"((unsigned)(bytes)) : "memory")
#define LDCG(p) __ldcg(p)
// the same for blocks without 16-byte alignment: one prefetch.global.L2 per 128-byte line, spread over the threads of the group
#define PREFETCH_LINES(ptr, bytes) do { const char *p_ = reinterpret_cast<const char *>(ptr); for (int o_ = threadIdx.x * 128; o_ < (int)(bytes); o_ += blockDim.x * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p_ + o_)); } while (0)
#endif

namespace mpcdev {

#ifndef MPC_HOST_EMU
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
#endif


// Reciprocal / square root without the library routines' special-case code (hardware seed + two Newton steps, <= 2 ulp).  The
// library versions cost a single-lane dependency chain 80-130 cycles and dozens of (partly predicated) instructions per call; the
// serial sections of the kernels (pivot chains, Lie-group routines) are made of exactly such calls (tools/ubench/lat.cu, diag.cu):
// in a pivot chain rcp_ costs 56 cycles of dependent latency against 83 for a division.
// Arguments are positive and in the normal range at every call site; NaN / non-positive inputs still propagate as NaN.
#ifdef MPC_HOST_EMU
inline double rcp_(double a) { return 1.0 / a; }
inline double rsqrt_(double a) { return 1.0 / sqrt(a); }
inline double sqrt_(double a) { return sqrt(a); }
#else
__device__ __forceinline__ double rcp_(double a) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  double e = fma(-a, y, 1.0);
  y = fma(y, e, y);
  e = fma(-a, y, 1.0);
  return fma(y, e, y);
}
__device__ __forceinline__ double rsqrt_(double a) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  double t = a * y, e = fma(-t, y, 1.0);
  y = fma(0.5 * y, e, y);
  t = a * y; e = fma(-t, y, 1.0);
  return fma(0.5 * y, e, y);
}
__device__ __forceinline__ double sqrt_(double a) { return a * rsqrt_(a); } // a > 0
#endif

// ------------------------------------------------------------------ 3-vectors / 3x3 (row-major)
HD void cross3(const double *a, const double *b, double *c) {
  double c0 = a[1] * b[2] - a[2] * b[1], c1 = a[2] * b[0] - a[0] * b[2], c2 = a[0] * b[1] - a[1] * b[0];
  c[0] = c0; c[1] = c1; c[2] = c2;
}
HD double dot3(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
HD double dot6(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5]; }
HD void mat3_vec(const double *R, const double *x, double *y) {
  double y0 = R[0] * x[0] + R[1] * x[1] + R[2] * x[2], y1 = R[3] * x[0] + R[4] * x[1] + R[5] * x[2], y2 = R[6] * x[0] + R[7] * x[1] + R[8] * x[2];
  y[0] = y0; y[1] = y1; y[2] = y2;
}
HD void mat3T_vec(const double *R, const double *x, double *y) {
  double y0 = R[0] * x[0] + R[3] * x[1] + R[6] * x[2], y1 = R[1] * x[0] + R[4] * x[1] + R[7] * x[2], y2 = R[2] * x[0] + R[5] * x[1] + R[8] * x[2];
  y[0] = y0; y[1] = y1; y[2] = y2;
}
HD void mat3_mul(const double *A, const double *B, double *C) { // C = A B (C distinct from A,B)
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
HD void mat3_mulT(const double *A, const double *B, double *C) { // C = A^T B
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}
HD void skew3(const double *a, double *S) {
  S[0] = 0; S[1] = -a[2]; S[2] = a[1]; S[3] = a[2]; S[4] = 0; S[5] = -a[0]; S[6] = -a[1]; S[7] = a[0]; S[8] = 0;
}

// ------------------------------------------------------------------ SE3 (12 doubles: R row-major, p), spatial [lin; ang]
HD void se3_mul(const double *a, const double *b, double *c) { // c = a b
  double R[9], p[3];
  mat3_mul(a, b, R);
  mat3_vec(a, b + 9, p);
  for (int i = 0; i < 9; i++) c[i] = R[i];
  for (int i = 0; i < 3; i++) c[9 + i] = p[i] + a[9 + i];
}
HD void se3_inv_mul(const double *a, const double *b, double *c) { // c = a^-1 b
  double R[9], d[3], p[3];
  mat3_mulT(a, b, R);
  for (int i = 0; i < 3; i++) d[i] = b[9 + i] - a[9 + i];
  mat3T_vec(a, d, p);
  for (int i = 0; i < 9; i++) c[i] = R[i];
  for (int i = 0; i < 3; i++) c[9 + i] = p[i];
}
HD void se3_act_motion(const double *M, const double *m, double *o) { // local -> world
  double w[3], v[3], c[3];
  mat3_vec(M, m + 3, w); mat3_vec(M, m, v); cross3(M + 9, w, c);
  for (int i = 0; i < 3; i++) { o[i] = v[i] + c[i]; o[3 + i] = w[i]; }
}
HD void se3_actinv_motion(const double *M, const double *m, double *o) { // world -> local
  double c[3], t[3];
  cross3(M + 9, m + 3, c);
  for (int i = 0; i < 3; i++) t[i] = m[i] - c[i];
  double ol[3], oa[3];
  mat3T_vec(M, t, ol); mat3T_vec(M, m + 3, oa);
  for (int i = 0; i < 3; i++) { o[i] = ol[i]; o[3 + i] = oa[i]; }
}
HD void se3_act_force(const double *M, const double *f, double *o) { // local -> world
  double fl[3], fa[3], c[3];
  mat3_vec(M, f, fl); mat3_vec(M, f + 3, fa); cross3(M + 9, fl, c);
  for (int i = 0; i < 3; i++) { o[i] = fl[i]; o[3 + i] = fa[i] + c[i]; }
}
HD void cross_mm(const double *a, const double *b, double *o) { // motion x motion
  double t1[3], t2[3], t3[3];
  cross3(a + 3, b, t1); cross3(a, b + 3, t2); cross3(a + 3, b + 3, t3);
  for (int i = 0; i < 3; i++) { o[i] = t1[i] + t2[i]; o[3 + i] = t3[i]; }
}
HD void cross_mf(const double *a, const double *f, double *o) { // motion x* force
  double t1[3], t2[3], t3[3];
  cross3(a + 3, f, t1); cross3(a + 3, f + 3, t2); cross3(a, f, t3);
  for (int i = 0; i < 3; i++) { o[i] = t1[i]; o[3 + i] = t2[i] + t3[i]; }
}
// 6x6 motion action matrix of M (row-major 36)
HD void se3_action_matrix(const double *M, double *A) {
  double S[9], pR[9];
  skew3(M + 9, S); mat3_mul(S, M, pR);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      A[6 * i + j] = M[3 * i + j]; A[6 * i + 3 + j] = pR[3 * i + j];
      A[6 * (i + 3) + j] = 0; A[6 * (i + 3) + 3 + j] = M[3 * i + j];
    }
}
HD void mat6_vec(const double *A, const double *x, double *y) {
  double t[6];
  for (int i = 0; i < 6; i++) t[i] = A[6 * i] * x[0] + A[6 * i + 1] * x[1] + A[6 * i + 2] * x[2] + A[6 * i + 3] * x[3] + A[6 * i + 4] * x[4] + A[6 * i + 5] * x[5];
  for (int i = 0; i < 6; i++) y[i] = t[i];
}
HD void mat6_mul(const double *A, const double *B, double *C) { // C distinct
  for (int i = 0; i < 6; i++)
    for (int j = 0; j < 6; j++) { double s = 0; for (int k = 0; k < 6; k++) s += A[6 * i + k] * B[6 * k + j]; C[6 * i + j] = s; }
}

// Spatial inertia in 10-parameter form about the WORLD origin: I[0]=mass, I[1..3]=h=m*c, I[4..9]=Io (xx,xy,xz,yy,yz,zz)
HD void inertia_mul(const double *I, const double *m, double *f) { // f = I m
  double c1[3], c2[3];
  cross3(I + 1, m + 3, c1); // h x w
  cross3(I + 1, m, c2);     // h x v
  double w0 = m[3], w1 = m[4], w2 = m[5];
  double f0 = I[0] * m[0] - c1[0], f1 = I[0] * m[1] - c1[1], f2 = I[0] * m[2] - c1[2];
  double f3 = c2[0] + I[4] * w0 + I[5] * w1 + I[6] * w2;
  double f4 = c2[1] + I[5] * w0 + I[7] * w1 + I[8] * w2;
  double f5 = c2[2] + I[6] * w0 + I[8] * w1 + I[9] * w2;
  f[0] = f0; f[1] = f1; f[2] = f2; f[3] = f3; f[4] = f4; f[5] = f5;
}

// ------------------------------------------------------------------ SO3/SE3 exp, log and Jacobians
HD void so3_coeffs(double t2, double &a, double &b, double &c) {
  if (t2 < 1e-6) {
    a = 1.0 - t2 / 6 + t2 * t2 / 120; b = 0.5 - t2 / 24 + t2 * t2 / 720; c = 1.0 / 6 - t2 / 120 + t2 * t2 / 5040;
  } else {
    double t = sqrt_(t2), s, co;
    sincos(t, &s, &co);
    const double it = rcp_(t), it2 = it * it;
    a = s * it; b = (1.0 - co) * it2; c = (t - s) * (it2 * it);
  }
}
HD double vinv_coeff(double t2) {
  if (t2 < 1e-6) return 1.0 / 12 + t2 / 720 + t2 * t2 / 30240;
  double t = sqrt_(t2), s, co;
  sincos(t, &s, &co);
  return (1.0 - t * s * rcp_(2.0 * (1.0 - co))) * rcp_(t2);
}
HD void exp6(const double *xi, double *M) {
  const double *w = xi + 3;
  double t2 = dot3(w, w), a, b, c;
  so3_coeffs(t2, a, b, c);
  double W[9], W2[9], V[9];
  skew3(w, W); mat3_mul(W, W, W2);
  for (int i = 0; i < 9; i++) { double e = (i % 4 == 0) ? 1.0 : 0.0; M[i] = e + a * W[i] + b * W2[i]; V[i] = e + b * W[i] + c * W2[i]; }
  mat3_vec(V, xi, M + 9);
}
HD void log3(const double *R, double *w) {
  double s[3] = {(R[7] - R[5]) * 0.5, (R[2] - R[6]) * 0.5, (R[3] - R[1]) * 0.5};
  double ct = (R[0] + R[4] + R[8] - 1.0) * 0.5;
  double s2 = dot3(s, s), f;
  if (s2 < 1e-6 && ct > 0) f = 1.0 + s2 / 6 + s2 * s2 * (3.0 / 40.0) + s2 * s2 * s2 * (15.0 / 336.0);
  else { double sn = sqrt(s2); f = atan2(sn, ct) / sn; } // (s2 may be 0 at a half turn: library sqrt / division here)
  w[0] = s[0] * f; w[1] = s[1] * f; w[2] = s[2] * f;
}
HD void log6(const double *M, double *xi) {
  double w[3];
  log3(M, w);
  double t2 = dot3(w, w), cp = vinv_coeff(t2);
  double W[9], W2[9], Vi[9];
  skew3(w, W); mat3_mul(W, W, W2);
  for (int i = 0; i < 9; i++) Vi[i] = ((i % 4 == 0) ? 1.0 : 0.0) - 0.5 * W[i] + cp * W2[i];
  mat3_vec(Vi, M + 9, xi);
  xi[3] = w[0]; xi[4] = w[1]; xi[5] = w[2];
}
// Q block of the SE3 Jacobians (Barfoot 7.86) evaluated at (rho, phi)
HD void q_block(const double *rho, const double *phi, double *Q) {
  double t2 = dot3(phi, phi), c1, c2, c3;
  if (t2 < 1e-6) {
    c1 = 1.0 / 6 - t2 / 120 + t2 * t2 / 5040; c2 = 1.0 / 24 - t2 / 720 + t2 * t2 / 40320; c3 = 1.0 / 120 - t2 / 2520 + t2 * t2 / 120960;
  } else {
    double t = sqrt_(t2), s, c;
    sincos(t, &s, &c);
    const double it = rcp_(t), it2 = it * it, it4 = it2 * it2;
    c1 = (t - s) * (it2 * it); c2 = (t2 + 2 * c - 2) * (0.5 * it4); c3 = (2 * t - 3 * s + t * c) * (0.5 * it4 * it);
  }
  double P[9], Rr[9], PR[9], RP[9], PRP[9], PPR[9], RPP[9], PRPP[9], PPRP[9];
  skew3(phi, P); skew3(rho, Rr);
  mat3_mul(P, Rr, PR); mat3_mul(Rr, P, RP); mat3_mul(PR, P, PRP);
  mat3_mul(P, PR, PPR); mat3_mul(RP, P, RPP); mat3_mul(PRP, P, PRPP); mat3_mul(P, PRP, PPRP);
  for (int i = 0; i < 9; i++)
    Q[i] = 0.5 * Rr[i] + c1 * (PR[i] + RP[i] + PRP[i]) + c2 * (PPR[i] + RPP[i] - 3 * PRP[i]) + c3 * (PRPP[i] + PPRP[i]);
}
HD void Jexp6(const double *xi, double *J) { // right Jacobian of exp6 (6x6 row-major)
  double t2 = dot3(xi + 3, xi + 3), a, b, c;
  so3_coeffs(t2, a, b, c);
  double W[9], W2[9], J3[9], Q[9], nr[3] = {-xi[0], -xi[1], -xi[2]}, np[3] = {-xi[3], -xi[4], -xi[5]};
  skew3(xi + 3, W); mat3_mul(W, W, W2);
  for (int i = 0; i < 9; i++) J3[i] = ((i % 4 == 0) ? 1.0 : 0.0) - b * W[i] + c * W2[i];
  q_block(nr, np, Q);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) { J[6 * i + j] = J3[3 * i + j]; J[6 * i + 3 + j] = Q[3 * i + j]; J[6 * (i + 3) + j] = 0; J[6 * (i + 3) + 3 + j] = J3[3 * i + j]; }
}
HD void Jlog6_from_log(const double *xi, double *J) { // xi = log6(M)
  double t2 = dot3(xi + 3, xi + 3), cp = vinv_coeff(t2);
  double W[9], W2[9], J3i[9], Q[9], T1[9], B[9], nr[3] = {-xi[0], -xi[1], -xi[2]}, np[3] = {-xi[3], -xi[4], -xi[5]};
  skew3(xi + 3, W); mat3_mul(W, W, W2);
  for (int i = 0; i < 9; i++) J3i[i] = ((i % 4 == 0) ? 1.0 : 0.0) + 0.5 * W[i] + cp * W2[i];
  q_block(nr, np, Q);
  mat3_mul(J3i, Q, T1); mat3_mul(T1, J3i, B);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) { J[6 * i + j] = J3i[3 * i + j]; J[6 * i + 3 + j] = -B[3 * i + j]; J[6 * (i + 3) + j] = 0; J[6 * (i + 3) + 3 + j] = J3i[3 * i + j]; }
}
HD void quat_to_R(const double *q, double *R) {
  double x = q[0], y = q[1], z = q[2], w = q[3];
  double n = x * x + y * y + z * z + w * w, s = 2.0 * rcp_(n);
  R[0] = 1 - s * (y * y + z * z); R[1] = s * (x * y - z * w); R[2] = s * (x * z + y * w);
  R[3] = s * (x * y + z * w); R[4] = 1 - s * (x * x + z * z); R[5] = s * (y * z - x * w);
  R[6] = s * (x * z - y * w); R[7] = s * (y * z + x * w); R[8] = 1 - s * (x * x + y * y);
}
HD void quat_integrate(const double *q, const double *w, double *out) {
  double t2 = dot3(w, w), sh, ch;
  if (t2 < 1e-6) { sh = 0.5 - t2 / 48 + t2 * t2 / 3840; ch = 1.0 - t2 / 8 + t2 * t2 / 384; }
  else { double t = sqrt_(t2), s, c; sincos(0.5 * t, &s, &c); sh = s * rcp_(t); ch = c; }
  double dx = w[0] * sh, dy = w[1] * sh, dz = w[2] * sh, dw = ch;
  double x = q[0], y = q[1], z = q[2], ww = q[3];
  double ox = ww * dx + x * dw + y * dz - z * dy;
  double oy = ww * dy - x * dz + y * dw + z * dx;
  double oz = ww * dz + x * dy - y * dx + z * dw;
  double ow = ww * dw - x * dx - y * dy - z * dz;
  double n = rsqrt_(ox * ox + oy * oy + oz * oz + ow * ow);
  out[0] = ox * n; out[1] = oy * n; out[2] = oz * n; out[3] = ow * n;
}
// 6x6 inverse by Gauss-Jordan with partial pivoting (single thread)
HD void inv6(const double *A, double *Ai) {
  double M[6][12];
  for (int i = 0; i < 6; i++) for (int j = 0; j < 6; j++) { M[i][j] = A[6 * i + j]; M[i][6 + j] = (i == j) ? 1.0 : 0.0; }
  for (int c = 0; c < 6; c++) {
    int p = c;
    for (int r = c + 1; r < 6; r++) if (fabs(M[r][c]) > fabs(M[p][c])) p = r;
    if (p != c) for (int j = 0; j < 12; j++) { double t = M[p][j]; M[p][j] = M[c][j]; M[c][j] = t; }
    double d = rcp_(M[c][c]);
    for (int j = 0; j < 12; j++) M[c][j] *= d;
    for (int r = 0; r < 6; r++) if (r != c) { double f = M[r][c]; for (int j = 0; j < 12; j++) M[r][j] -= f * M[c][j]; }
  }
  for (int i = 0; i < 6; i++) for (int j = 0; j < 6; j++) Ai[6 * i + j] = M[i][6 + j];
}

// y[i * incy] = (y0 ? y0[i] : 0) + sum_j A[i * lda + j] x[j] for a matrix in shared memory: rows over warps (RB at a time, independent
// reduction chains), columns over lanes — consecutive lanes read consecutive doubles, so there are no bank conflicts whatever
// the leading dimension (a row per thread is a 16-way conflict for ld = 8 mod 16).  No barrier inside.  each(i, j, a) is called
// once for every entry a = A[i * lda + j] read, so that a caller can derive another matrix from A in the same pass.
struct NoEach {
  HD void operator()(int, int, double) const {}
};
template <int RB = 7, class Each = NoEach>
HD void matvec_rows(const double *A, int lda, int rows, int cols, const double *x, const double *y0, double *y, int incy = 1, Each each = Each()) {
  for (int base = WARP_ID * RB; base < rows; base += NWARPS * RB) {
    double acc[RB];
#pragma unroll
    for (int r = 0; r < RB; r++) acc[r] = 0.0;
    LANE_FOR(j, cols) {
      const double xj = x[j];
#pragma unroll
      for (int r = 0; r < RB; r++)
        if (base + r < rows) { const double a = A[(base + r) * lda + j]; acc[r] += a * xj; each(base + r, j, a); }
    }
#pragma unroll
    for (int r = 0; r < RB; r++) acc[r] = WARP_SUM(acc[r]);
    if (LANE0) {
#pragma unroll
      for (int r = 0; r < RB; r++)
        if (base + r < rows) y[(base + r) * incy] = acc[r] + (y0 ? y0[base + r] : 0.0);
    }
  }
}

// Group-wide reduction of four per-thread partials (two sums, two maxima): butterfly inside each warp, one slot per warp in
// `scratch` (>= 4 * warps doubles), combined by thread 0 into out[0..3] after the barrier.  Under emulation the single
// "thread" already holds the totals.
HD void reduce_sum2_max2(double s0, double s1, double m0, double m1, double *scratch, double *out) {
#ifdef MPC_HOST_EMU
  out[0] = s0; out[1] = s1; out[2] = m0; out[3] = m1;
#else
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    m0 = fmax(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
  }
  if (LANE0) { scratch[4 * WARP_ID] = s0; scratch[4 * WARP_ID + 1] = s1; scratch[4 * WARP_ID + 2] = m0; scratch[4 * WARP_ID + 3] = m1; }
  SYNC();
  ONE_THREAD {
    double a = 0, b = 0, c = 0, d = 0;
    for (int w = 0; w < NWARPS; w++) { a += scratch[4 * w]; b += scratch[4 * w + 1]; c = fmax(c, scratch[4 * w + 2]); d = fmax(d, scratch[4 * w + 3]); }
    out[0] = a; out[1] = b; out[2] = c; out[3] = d;
  }
#endif
  SYNC();
}
// Stable compaction of the indices r < n (n <= threads of the group) whose flag is set: idx[0..count) ascending, *count.
// Warp ballots + per-warp offsets through `scratch` (>= warps ints); serial under emulation.
HD void compact_flags(const int32_t *flags, int n, int32_t *idx, int32_t *count, int32_t *scratch) {
#ifdef MPC_HOST_EMU
  int c = 0;
  for (int r = 0; r < n; r++) if (flags[r]) idx[c++] = r;
  *count = c;
#else
  const int t = threadIdx.x, lane = t & 31;
  const bool f = (t < n) && flags[t] != 0;
  const unsigned mask = __ballot_sync(0xffffffffu, f);
  if (lane == 0) scratch[WARP_ID] = __popc(mask);
  SYNC();
  int off = 0;
  for (int w = 0; w < WARP_ID; w++) off += scratch[w];
  if (f) idx[off + __popc(mask & ((1u << lane) - 1u))] = t;
  if (t == NTHREADS - 1) *count = off + __popc(mask);
#endif
  SYNC();
}

// ------------------------------------------------------------------ blocked Cholesky / triangular solves (panel width 8)
// In-place lower Cholesky of A (n x n, ld) by 8-wide panels.  Dinv receives the inverses of the diagonal blocks (8 x 8
// lower, row-major, 64 doubles per panel), which turn the triangular solves below into small GEMMs.
constexpr int CB = 8;
#ifndef MPC_HOST_EMU
// Device version called by ALL lanes of the group's warp 0.  Lane 0 runs the pivot chain in registers as a square-root-free
// LDL' elimination (per column: reciprocal of the pivot -> scaled column -> update, 56 + 8.5 + 8.5 cycles of dependent
// latency; a Cholesky column costs a 77-cycle rsqrt more and the chain is what the whole blocked factorisation waits for).
// The eight lanes then finish side by side, one column each: r_i = rsqrt(d_i), the unit-triangular inverse by forward
// substitution (one FMA per dependent step), and the scaling  L = Lt diag(sqrt d),  L^-1 = diag(r) Lt^-1.
__device__ __forceinline__ void chol_diag_block_warp0(double *A, int k0, int bw, int ld, double *Di) {
  const int lane = threadIdx.x & 31;
  if (lane == 0) {
    double L[CB][CB];
#pragma unroll
    for (int r = 0; r < CB; r++)
#pragma unroll
      for (int c = 0; c < CB; c++) L[r][c] = (c <= r) ? ((r < bw) ? A[(k0 + r) * ld + k0 + c] : ((r == c) ? 1.0 : 0.0)) : 0.0;
#pragma unroll
    for (int j = 0; j < CB; j++) {
      const double rj = rcp_(L[j][j]);
      Di[j * CB + j] = L[j][j]; // pivot d_j (scratch for the finish below)
      double tcol[CB];
#pragma unroll
      for (int r = j + 1; r < CB; r++) { tcol[r] = L[r][j] * rj; Di[r * CB + j] = tcol[r]; } // unit-lower factor Lt
#pragma unroll
      for (int r = j + 1; r < CB; r++)
#pragma unroll
        for (int c = j + 1; c <= r; c++) L[r][c] -= tcol[r] * L[c][j];
    }
  }
  __syncwarp();
  double Lf[CB][CB], dd[CB], X[CB], lcol[CB];
  const int c = lane & 7;
  const double pc = Di[c * CB + c];
  const double rc = rsqrt_(pc); // one rsqrt per lane; the eight values are exchanged through the (free) first row of Di's upper triangle + slot 15
#pragma unroll
  for (int i = 0; i < CB; i++) {
    lcol[i] = Di[i * CB + c]; // own column of Lt (rows below the diagonal; the diagonal slot holds the pivot)
#pragma unroll
    for (int t = 0; t < CB; t++) Lf[i][t] = (t < i) ? Di[i * CB + t] : 0.0;
  }
  __syncwarp();
  if (lane < CB) Di[(c == 0) ? 15 : c] = rc; // slots (0,1..7) and (1,7): above the diagonal, never read as factor entries
  __syncwarp();
#pragma unroll
  for (int i = 0; i < CB; i++) dd[i] = Di[(i == 0) ? 15 : i];
  const double sc = pc * rc; // sqrt(d_c)
#pragma unroll
  for (int t = 0; t < CB; t++) X[t] = (t == c) ? 1.0 : 0.0;
#pragma unroll
  for (int t = 0; t < CB; t++) {
#pragma unroll
    for (int i = t + 1; i < CB; i++) X[i] -= Lf[i][t] * X[t]; // rows above the diagonal stay 0
  }
  __syncwarp();
  if (lane < CB) {
#pragma unroll
    for (int i = 0; i < CB; i++) {
      Di[i * CB + c] = (i < bw && c < bw) ? dd[i] * X[i] : 0.0;
      if (i < bw && c < bw && i >= c) A[(k0 + i) * ld + k0 + c] = (i == c) ? sc : lcol[i] * sc;
    }
  }
  __syncwarp();
}
#define DIAG_BLOCK(A, k0, bw, ld, Di) do { if (threadIdx.x < 32) mpcdev::chol_diag_block_warp0(A, k0, bw, ld, Di); } while (0)
#else
// Host-emulation version: the bw x bw diagonal block at k0 is factored (Cholesky) and inverted in place of the device's pivot
// chain (rows/cols >= bw are padded with the identity).
inline void chol_diag_block(double *A, int k0, int bw, int ld, double *Di) {
  double L[CB][CB], X[CB][CB], dd[CB];
#pragma unroll
  for (int r = 0; r < CB; r++)
#pragma unroll
    for (int c = 0; c < CB; c++) L[r][c] = (c <= r) ? ((r < bw) ? A[(k0 + r) * ld + k0 + c] : ((r == c) ? 1.0 : 0.0)) : 0.0;
#pragma unroll
  for (int j = 0; j < CB; j++) {
    const double d = rsqrt_(L[j][j]);
    dd[j] = d;
    L[j][j] = L[j][j] * d;
#pragma unroll
    for (int r = j + 1; r < CB; r++) L[r][j] *= d;
#pragma unroll
    for (int r = j + 1; r < CB; r++)
#pragma unroll
      for (int c = j + 1; c <= r; c++) L[r][c] -= L[r][j] * L[c][j];
  }
  // X = L^-1 column by column in right-looking order: as soon as X[t][c] is known it is folded into the partial sums of the
  // rows below, so the dependent chain per row is one multiply + one FMA (the 8 columns are independent chains)
#pragma unroll
  for (int c = 0; c < CB; c++) {
#pragma unroll
    for (int r = 0; r < CB; r++) X[r][c] = (r == c) ? 1.0 : 0.0;
#pragma unroll
    for (int t = c; t < CB; t++) {
      X[t][c] *= dd[t];
#pragma unroll
      for (int r = t + 1; r < CB; r++) X[r][c] -= L[r][t] * X[t][c];
    }
  }
#pragma unroll
  for (int r = 0; r < CB; r++)
#pragma unroll
    for (int c = 0; c < CB; c++) {
      if (r < bw && c <= r) A[(k0 + r) * ld + k0 + c] = L[r][c];
      Di[r * CB + c] = (r < bw && c < bw) ? X[r][c] : 0.0;
    }
}
#define DIAG_BLOCK(A, k0, bw, ld, Di) chol_diag_block(A, k0, bw, ld, Di)
#endif

// Small SPD systems (n <= 12: the centroidal model's 9 x 9 and 12 x 12 blocks): A X = B solved in place in B1 (n x n1, ld1) and
// B2 (n x n2, ld2).  ONE thread factors A = Lt D Lt' in registers (square-root-free pivot chain, as in the 8 x 8 diagonal blocks;
// a blocked factorisation would spend a whole padded 8 x 8 block on the ninth row) and leaves Lt (unit lower) / 1/d in A; then
// every right-hand-side column is one thread's forward / diagonal / backward substitution with broadcast loads of the factor.
// Two barriers instead of the ~10 of chol_blocked + trsm_blocked at this size.
template <int n> HD void small_spd_solve(double *A, int ld, double *B1, int n1, int ld1, double *B2, int n2, int ld2) {
  ONE_THREAD {
    double L[n][n];
#pragma unroll
    for (int r = 0; r < n; r++)
#pragma unroll
      for (int c = 0; c <= r; c++) L[r][c] = A[r * ld + c];
#pragma unroll
    for (int j = 0; j < n; j++) {
      const double rj = rcp_(L[j][j]);
      A[j * ld + j] = rj;
      double tcol[n];
#pragma unroll
      for (int r = j + 1; r < n; r++) { tcol[r] = L[r][j] * rj; A[r * ld + j] = tcol[r]; }
#pragma unroll
      for (int r = j + 1; r < n; r++)
#pragma unroll
        for (int c = j + 1; c <= r; c++) L[r][c] -= tcol[r] * L[c][j];
    }
  }
  SYNC();
  PAR_FOR(col, n1 + n2) {
    double *b = (col < n1) ? B1 + col : B2 + (col - n1);
    const int lb = (col < n1) ? ld1 : ld2;
    double y[n];
#pragma unroll
    for (int i = 0; i < n; i++) y[i] = b[i * lb];
#pragma unroll
    for (int j = 0; j < n; j++) {
#pragma unroll
      for (int i = j + 1; i < n; i++) y[i] -= A[i * ld + j] * y[j];
    }
#pragma unroll
    for (int j = 0; j < n; j++) y[j] *= A[j * ld + j];
#pragma unroll
    for (int j = n - 1; j >= 0; j--) {
#pragma unroll
      for (int i = 0; i < j; i++) y[i] -= A[j * ld + i] * y[j];
    }
#pragma unroll
    for (int i = 0; i < n; i++) b[i * lb] = y[i];
  }
  SYNC();
}

// Blocked Cholesky (lower, in place): per 8-wide panel, one thread factors + inverts the diagonal block, the panel below it
// is multiplied by the inverse, and the trailing matrix is updated on 2 x 2 register tiles.  (The 56 x 56 and padded control
// blocks of the Riccati kernel use the tensor-core version with look-ahead, chol_mma in dmma.cuh; a look-ahead variant of
// this SIMT routine was measured and lost on the small matrices / 128-thread groups of the evaluation kernels.)
HD void chol_blocked(double *A, int n, int ld, double *Dinv) {
  for (int k0 = 0; k0 < n; k0 += CB) {
    const int bw = (n - k0 < CB) ? n - k0 : CB;
    const double *Di = Dinv + (k0 / CB) * CB * CB;
    DIAG_BLOCK(A, k0, bw, ld, Dinv + (k0 / CB) * CB * CB);
    SYNC();
    // panel below the diagonal block: L[i, k0:k0+bw] = A[i, k0:k0+bw] * Dinv^T, one row per work item
    const int rem = n - k0 - bw, r0 = k0 + bw;
    if (rem <= 0) break;
    PAR_FOR(i, rem) {
      double *row = A + (r0 + i) * ld + k0;
      double v[CB], o[CB];
#pragma unroll
      for (int q = 0; q < CB; q++) v[q] = (q < bw) ? row[q] : 0.0;
#pragma unroll
      for (int c = 0; c < CB; c++) {
        double s = 0;
#pragma unroll
        for (int q = 0; q < CB; q++)
          if (q <= c) s += v[q] * Di[c * CB + q];
        o[c] = s;
      }
#pragma unroll
      for (int q = 0; q < CB; q++) if (q < bw) row[q] = o[q];
    }
    SYNC();
    // trailing update on 2 x 2 tiles of the lower triangle
    const int th = (rem + 1) / 2;
    PAR_FOR(t, th * th) {
      int ti = t / th, tj = t % th;
      if (tj > ti) continue;
      int i0 = r0 + 2 * ti, j0 = r0 + 2 * tj;
      double a00 = 0, a01 = 0, a10 = 0, a11 = 0;
      bool i1 = i0 + 1 < n, j1 = j0 + 1 < n;
      for (int q = 0; q < bw; q++) {
        double li0 = A[i0 * ld + k0 + q], li1 = i1 ? A[(i0 + 1) * ld + k0 + q] : 0.0;
        double lj0 = A[j0 * ld + k0 + q], lj1 = j1 ? A[(j0 + 1) * ld + k0 + q] : 0.0;
        a00 += li0 * lj0; a01 += li0 * lj1; a10 += li1 * lj0; a11 += li1 * lj1;
      }
      A[i0 * ld + j0] -= a00;
      if (j1 && j0 + 1 <= i0) A[i0 * ld + j0 + 1] -= a01;
      if (i1) { A[(i0 + 1) * ld + j0] -= a10; if (j1) A[(i0 + 1) * ld + j0 + 1] -= a11; }
    }
    SYNC();
  }
}
// In-place inverse of an SPD matrix A (n x n, ld; n even): blocked Cholesky, X = L^-1 by one warp per 8-wide block column
// (independent forward-substitution chains, warp-level barriers only), then A <- X' X on 2 x 2 register tiles (full symmetric
// result).  Turns every later solve with A into a barrier-free matrix product.  Dinv: 64 doubles per diagonal block;
// Ls: n * n + 64 * warps doubles of scratch.
HD void spd_inverse_blocked(double *A, int n, int ld, double *Dinv, double *Ls) {
  chol_blocked(A, n, ld, Dinv);
  const int nb = (n + CB - 1) / CB;
  double *tt = Ls + n * n + 64 * WARP_ID;
  for (int jb = WARP_ID; jb < nb; jb += NWARPS) {
    for (int ib = jb; ib < nb; ib++) {
      WARP_FOR(e, 64) { // tt = E_ij - sum_k L_ik X_kj
        const int r = e >> 3, c = e & 7, gi = CB * ib + r, gj = CB * jb + c;
        double s = 0.0;
        if (gi < n && gj < n) {
          s = (gi == gj) ? 1.0 : 0.0;
          for (int kb = jb; kb < ib; kb++)
            for (int q = 0; q < CB; q++) s -= A[gi * ld + CB * kb + q] * Ls[(CB * kb + q) * n + gj];
        }
        tt[e] = s;
      }
      WARP_SYNC();
      WARP_FOR(e, 64) { // X_ij = Dinv_i tt
        const int r = e >> 3, c = e & 7, gi = CB * ib + r, gj = CB * jb + c;
        if (gi < n && gj < n) {
          const double *Di = Dinv + 64 * ib;
          double s = 0.0;
          for (int q = 0; q <= r; q++) s += Di[r * CB + q] * tt[q * CB + c];
          Ls[gi * n + gj] = s;
        }
      }
      WARP_SYNC();
    }
  }
  SYNC();
  const int th = n / 2;
  PAR_FOR(t, th * th) {
    const int ti = t / th, tj = t % th;
    if (tj > ti) continue;
    const int i0 = 2 * ti, j0 = 2 * tj;
    double a00 = 0, a01 = 0, a10 = 0, a11 = 0;
    for (int k = i0; k < n; k++) { // X is lower triangular: rows k >= max(i, j)
      const double xi0 = Ls[k * n + i0], xi1 = Ls[k * n + i0 + 1], xj0 = Ls[k * n + j0], xj1 = Ls[k * n + j0 + 1];
      a00 += xi0 * xj0; a01 += xi0 * xj1; a10 += xi1 * xj0; a11 += xi1 * xj1;
    }
    A[i0 * ld + j0] = a00; A[j0 * ld + i0] = a00;
    A[i0 * ld + j0 + 1] = a01; A[(j0 + 1) * ld + i0] = a01;
    A[(i0 + 1) * ld + j0] = a10; A[j0 * ld + i0 + 1] = a10;
    A[(i0 + 1) * ld + j0 + 1] = a11; A[(j0 + 1) * ld + i0 + 1] = a11;
  }
  SYNC();
}
// Solve L L^T X = B in place (B: n x nrhs, ldb) with the diagonal-block inverses from chol_blocked.
HD void trsm_blocked(const double *L, int n, int ld, const double *Dinv, double *B, int nrhs, int ldb) {
  // forward: L Y = B
  for (int k0 = 0; k0 < n; k0 += CB) {
    const int bw = (n - k0 < CB) ? n - k0 : CB;
    const double *Di = Dinv + (k0 / CB) * CB * CB;
    PAR_FOR(c, nrhs) {
      double b[CB], x[CB];
#pragma unroll
      for (int r = 0; r < CB; r++) b[r] = (r < bw) ? B[(k0 + r) * ldb + c] : 0.0;
#pragma unroll
      for (int r = 0; r < CB; r++) {
        double s = 0;
#pragma unroll
        for (int t = 0; t < CB; t++)
          if (t <= r) s += Di[r * CB + t] * b[t];
        x[r] = s;
      }
#pragma unroll
      for (int r = 0; r < CB; r++) if (r < bw) B[(k0 + r) * ldb + c] = x[r];
    }
    SYNC();
    const int rem = n - k0 - bw, r0 = k0 + bw;
    const int tc = (nrhs + 3) / 4;
    PAR_FOR(t, rem * tc) {
      int i = r0 + t / tc, c0 = (t % tc) * 4;
      double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
      int nc4 = nrhs - c0 < 4 ? nrhs - c0 : 4;
      for (int q = 0; q < bw; q++) {
        double l = L[i * ld + k0 + q];
        const double *xr = B + (k0 + q) * ldb + c0;
        a0 += l * xr[0]; if (nc4 > 1) a1 += l * xr[1]; if (nc4 > 2) a2 += l * xr[2]; if (nc4 > 3) a3 += l * xr[3];
      }
      double *br = B + i * ldb + c0;
      br[0] -= a0; if (nc4 > 1) br[1] -= a1; if (nc4 > 2) br[2] -= a2; if (nc4 > 3) br[3] -= a3;
    }
    SYNC();
  }
  // backward: L^T X = Y
  const int nblk = (n + CB - 1) / CB;
  for (int kb = nblk - 1; kb >= 0; kb--) {
    const int k0 = kb * CB, bw = (n - k0 < CB) ? n - k0 : CB;
    const double *Di = Dinv + kb * CB * CB;
    PAR_FOR(c, nrhs) {
      double b[CB], x[CB];
#pragma unroll
      for (int r = 0; r < CB; r++) b[r] = (r < bw) ? B[(k0 + r) * ldb + c] : 0.0;
#pragma unroll
      for (int r = 0; r < CB; r++) {
        double s = 0;
#pragma unroll
        for (int t = 0; t < CB; t++)
          if (t >= r) s += Di[t * CB + r] * b[t];
        x[r] = s;
      }
#pragma unroll
      for (int r = 0; r < CB; r++) if (r < bw) B[(k0 + r) * ldb + c] = x[r];
    }
    SYNC();
    const int tc = (nrhs + 3) / 4;
    PAR_FOR(t, k0 * tc) {
      int i = t / tc, c0 = (t % tc) * 4;
      double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
      int nc4 = nrhs - c0 < 4 ? nrhs - c0 : 4;
      for (int q = 0; q < bw; q++) {
        double l = L[(k0 + q) * ld + i];
        const double *xr = B + (k0 + q) * ldb + c0;
        a0 += l * xr[0]; if (nc4 > 1) a1 += l * xr[1]; if (nc4 > 2) a2 += l * xr[2]; if (nc4 > 3) a3 += l * xr[3];
      }
      double *br = B + i * ldb + c0;
      br[0] -= a0; if (nc4 > 1) br[1] -= a1; if (nc4 > 2) br[2] -= a2; if (nc4 > 3) br[3] -= a3;
    }
    SYNC();
  }
}

} // namespace mpcdev
