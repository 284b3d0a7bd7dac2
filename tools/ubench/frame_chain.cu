// Micro-benchmark: latency of ONE lattice frame (csrc/lattice_fast.cuh: lattice_frame) when a single warp
// iterates it back to back (the recursion is a dependent chain: this is the floor of the per-frame time).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I include -I pytorch_end2end_speech_recognition_b200/csrc \
//        [-DSTORE_MODE=1|2] -o frame_chain tools/ubench/frame_chain.cu
#include <cstdio>
#include "lattice_fast.cuh"
using namespace b200ctc;

#ifndef STORE_MODE
#define STORE_MODE 0   // 0: recursion only   1: + phase-1 global stores (2 x STG.128 + STG.32)   2: + shared stores instead
#endif
__device__ unsigned char* g_scratch;

template <int SIDE>
__global__ void k(float* out, long long* cycles, int iters, int nwarps_active) {
  constexpr int NP = kLaneStates / 2;
  __shared__ __align__(16) unsigned char stage[16 * 32 * 48];
  __shared__ __align__(16) float row[4][64];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) row[i / 64][i % 64] = 0.3f + 0.001f * (i % 7);
  __syncthreads();
  if ((threadIdx.x >> 5) >= nwarps_active) return;
  const int lane = threadIdx.x & 31;
  LaneConst lc;
  lc.idxB_blank = 0;
  for (int m = 0; m < NP; ++m) { lc.idxB[m] = 4 * (1 + (lane * 3 + m * 5) % 29); lc.posB[m] = 0; }
  for (int u = 0; u < kLaneStates / 4; ++u) lc.Kf[u] = f2_pack(1.f, (lane & 1) ? 1.f : 0.f);
  lc.blankB = 0; lc.recB = 0; lc.expB = 0; lc.owned = true; lc.group = lane;
  LaneState st;
  for (int j = 0; j < NP; ++j) st.A[j] = f2_pack(1.0f + 0.01f * lane, 1.5f);
  st.e = 0;
  unsigned char* blk = g_scratch + ((size_t)(blockIdx.x * 16 + (threadIdx.x >> 5)) * 64 * 32 + lane) * 48;
  const int step = 32 * 48;
  unsigned char* sblk = stage + (threadIdx.x >> 5) * 32 * 48 + lane * 48;
  const long long t0 = clock64();
#pragma unroll 2
  for (int it = 0; it < iters; ++it) {
    f2 ACC[NP]; int E;
    lattice_frame<SIDE>(st, lc, row[it & 3], lane == 0, ACC, E);
    if (STORE_MODE == 1) {
      unsigned char* b = blk + (it & 63) * step;
      asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(b), "l"(ACC[3]), "l"(ACC[2]) : "memory");
      asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(b + 16), "l"(ACC[1]), "l"(ACC[0]) : "memory");
      *reinterpret_cast<int*>(b + 32) = E;
    }
    if (STORE_MODE == 2) {
      *reinterpret_cast<float4*>(sblk) = make_float4(f2_lo(ACC[3]), f2_hi(ACC[3]), f2_lo(ACC[2]), f2_hi(ACC[2]));
      *reinterpret_cast<float4*>(sblk + 16) = make_float4(f2_lo(ACC[1]), f2_hi(ACC[1]), f2_lo(ACC[0]), f2_hi(ACC[0]));
      *reinterpret_cast<int*>(sblk + 32) = E;
    }
  }
  const long long t1 = clock64();
  if (lane == 0) cycles[blockIdx.x * 32 + (threadIdx.x >> 5)] = t1 - t0;
  out[blockIdx.x * blockDim.x + threadIdx.x] = f2_lo(st.A[0]) + st.e;
}

int main() {
  float* out; long long* cyc;
  unsigned char* scr; cudaMalloc(&scr, (size_t)148 * 16 * 32 * 64 * 48); cudaMemcpyToSymbol(g_scratch, &scr, sizeof(scr));
  cudaMalloc(&out, 4 * 148 * 1024); cudaMalloc(&cyc, 8 * 148 * 32);
  const int iters = 20000;
  for (int nw : {1, 2, 4, 8, 16}) {
    k<0><<<148, 512>>>(out, cyc, iters, nw);
    k<0><<<148, 512>>>(out, cyc, iters, nw);
    cudaDeviceSynchronize();
    long long h[32]; cudaMemcpy(h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
    printf("STORE=%d  side 0: %2d warps/SM: %.1f cycles per frame (warp 0)\n", STORE_MODE, nw, (double)h[0] / iters);
  }
  k<1><<<148, 512>>>(out, cyc, iters, 1);
  cudaDeviceSynchronize();
  long long h1; cudaMemcpy(&h1, cyc, 8, cudaMemcpyDeviceToHost);
  printf("STORE=%d  side 1:  1 warp/SM : %.1f cycles per frame\n", STORE_MODE, (double)h1 / iters);
  printf("%s\n", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
