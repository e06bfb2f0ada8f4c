// Isolated timing of the 8 x 8 diagonal-block factorisation (not product code).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I mpc_benchmark_b200/csrc -I include -o tools/ubench/diag tools/ubench/diag.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "dmma.cuh"
using namespace mpcdev;
__global__ void k(long long *cyc, double *out, int reps) {
  __shared__ double A[64 * 8], Di[64];
  for (int e = threadIdx.x; e < 64 * 8; e += blockDim.x) { int i = (e / 8) % 8, j = e % 8; A[e] = (i == j) ? 10.0 + i : 0.1 * ((i + j) % 3); }
  __syncthreads();
  long long t0 = clock64();
  for (int r = 0; r < reps; r++) { DIAG_BLOCK(A + 64 * (r & 7), 0, 8, 8, Di); __syncwarp(); }
  long long t1 = clock64();
  // lane-0 chain only
  double acc = 0;
  for (int r = 0; r < reps; r++) {
    if (threadIdx.x == 0) {
      double L[8][8];
      const double *M = A + 64 * (r & 7);
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int c = 0; c < 8; c++) L[i][c] = (c <= i) ? fabs(M[i * 8 + c]) + (i == c ? 10.0 : 0.0) : 0.0;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const double rj = rcp_(L[j][j]);
        double tc[8];
#pragma unroll
        for (int i = j + 1; i < 8; i++) tc[i] = L[i][j] * rj;
#pragma unroll
        for (int i = j + 1; i < 8; i++)
#pragma unroll
          for (int c = j + 1; c <= i; c++) L[i][c] -= tc[i] * L[c][j];
        acc += rj;
      }
    }
  }
  long long t2 = clock64();
  if (threadIdx.x == 0) { cyc[0] = (t1 - t0) / reps; cyc[1] = (t2 - t1) / reps; out[0] = acc + Di[5]; }
}
int main() {
  long long *cyc; double *out;
  cudaMalloc(&cyc, 64); cudaMalloc(&out, 64);
  k<<<1, 128>>>(cyc, out, 50); cudaDeviceSynchronize();
  k<<<1, 128>>>(cyc, out, 50); cudaDeviceSynchronize();
  long long h[2]; cudaMemcpy(h, cyc, 16, cudaMemcpyDeviceToHost);
  printf("DIAG_BLOCK (chain + 8-lane finish, shared-memory in/out): %lld cycles; lane-0 LDL chain alone (loads + 8 pivots): %lld cycles\n", h[0], h[1]);
  return 0;
}
