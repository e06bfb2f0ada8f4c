// Isolated timing of the Riccati kernel's building blocks (one CTA alone on an SM; not product code).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I mpc_benchmark_b200/csrc -I include -o tools/ubench/phases tools/ubench/phases.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "dmma.cuh"
using namespace mpcdev;
constexpr int N = 56, NZ = 78, ZP = 80, LDN = 56, LDZ = 84, LDH = 80;
__global__ void __launch_bounds__(256) k(double *gW, const double *gH, long long *cyc, int reps) {
  extern __shared__ __align__(16) double sm[];
  double *H = sm, *G = H + ZP * LDH, *P = G + N * LDN, *vec = P + N * LDN, *dinv = vec, *PV = dinv + 64 * 8;
  double *ABs = H, *Ws = H + N * LDZ;
  for (int i = threadIdx.x; i < 14304; i += blockDim.x) sm[i] = 0.001 * ((i * 7) % 13);
  __syncthreads();
  long long t[8];
  // SPD matrix in G
  auto fillG = [&]() { for (int e = threadIdx.x; e < N * N; e += blockDim.x) { int i = e / N, j = e % N; G[i * LDN + j] = (i == j) ? 10.0 : 0.01 * ((i + j) % 5); } __syncthreads(); };
  fillG();
  t[0] = clock64();
  for (int r = 0; r < reps; r++) { chol_mma<7>(G, LDN, dinv); }
  t[1] = clock64();
  for (int r = 0; r < reps; r++) trsm_mma<7>(G, LDN, dinv, P, LDN, 7, PV, 8, 8);
  t[2] = clock64();
  for (int r = 0; r < reps; r++) mma_tn_g<N>(7, 10, P, LDN, ABs, LDZ, Ws, LDZ, nullptr, 0, 0, 0, false, gW, ZP, ZP);
  t[3] = clock64();
  for (int r = 0; r < reps; r++) mma_sym_deferred<N, 4>(10, ABs, LDZ, Ws, LDZ, H, LDH, gH, NZ, NZ, NZ);
  t[4] = clock64();
  for (int r = 0; r < reps; r++) mma_tn(7, 7, 24, H + N * LDH, LDH, P, LDN, H, LDH, H, LDH, N, N, true);
  t[5] = clock64();
  for (int r = 0; r < reps; r++) { chol_mma<3>(G, LDN, dinv); }
  t[6] = clock64();
  for (int r = 0; r < reps; r++) trsm_mma<3>(G, LDN, dinv, P, 64, 8, nullptr, 0, 8);
  t[7] = clock64();
  if (threadIdx.x == 0) for (int i = 0; i < 7; i++) cyc[blockIdx.x * 8 + i] = (t[i + 1] - t[i]) / reps;
}
int main() {
  double *gW, *gH; long long *cyc;
  cudaMalloc(&gW, 1 << 20); cudaMalloc(&gH, 1 << 20); cudaMalloc(&cyc, 4096); cudaMemset(gH, 0, 1 << 20);
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 114432);
  const char *names[] = {"chol_mma<7>", "trsm_mma<7> 8 tiles", "W gemm 7x10 K56", "H sym deferred 10x10 K56", "P update 7x7 K24 mirror", "chol_mma<3>", "trsm_mma<3> 8 tiles"};
  for (int thr : {128, 256}) for (int ctas : {1, 296}) {
    k<<<ctas, thr, 114432>>>(gW, gH, cyc, 20); cudaDeviceSynchronize();
    k<<<ctas, thr, 114432>>>(gW, gH, cyc, 20); cudaError_t e = cudaDeviceSynchronize();
    long long h[8]; cudaMemcpy(h, cyc, 64, cudaMemcpyDeviceToHost);
    printf("threads %d, %d CTAs (%s): %s\n", thr, ctas, ctas == 1 ? "alone" : "2 per SM", cudaGetErrorString(e));
    for (int i = 0; i < 7; i++) printf("   %-28s %8lld cycles\n", names[i], h[i]);
  }
  return 0;
}
