// Shared helpers for libb2nerf.so (sm_100a).  Error convention of include/b2nerf.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/b2nerf.h"
#include "../../include/b2nerf_debug.h"

namespace b2n {

extern thread_local char g_err[512];

inline int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
  snprintf(g_err, sizeof(g_err), fmt, a, b);
  return code;
}

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(B2N_ECUDA, "%s: %s", what, cudaGetErrorString(e));
  return B2N_OK;
}

#define B2N_REQUIRE(cond, msg)                                  \
  do {                                                          \
    if (!(cond)) return b2n::fail(B2N_EINVAL, "%s: %s", __func__, msg); \
  } while (0)

constexpr int kSMs = 148;  // B200

// Optional device-side row count (b2n_set_active_rows): while set, every entry point that takes a point count P
// treats rows >= *rows as absent -- its kernels clamp P on the device.  This is what lets a step behind an occupancy
// grid run without the host ever reading the number of active samples (fixed-capacity buffers, CUDA-graph capture).
extern thread_local const int* g_active_rows;
__device__ __forceinline__ int64_t clamp_rows(int64_t P, const int* __restrict__ rows) {
  if (!rows) return P;
  const int64_t n = (int64_t)__ldg(rows);
  return n < P ? (n < 0 ? 0 : n) : P;
}

inline unsigned grid_for(int64_t work_items, int per_block) {
  int64_t g = (work_items + per_block - 1) / per_block;
  if (g < 1) g = 1;
  return (unsigned)g;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Exclusive scan of one int per thread over the block; *total (shared) gets the block sum.  Every thread of the block
// must call it (it synchronises).
__device__ __forceinline__ int block_exclusive_scan(int v, int* total) {
  __shared__ int warp_tot[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    int t = lane < nw ? warp_tot[lane] : 0;
    int ti = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int q = __shfl_up_sync(0xffffffffu, ti, o);
      if (lane >= o) ti += q;
    }
    warp_tot[lane] = ti - t;  // exclusive prefix of the warp totals
    if (lane == 31) *total = ti;
  }
  __syncthreads();
  int res = inc - v + warp_tot[wid];
  __syncthreads();
  return res;
}

// streaming (read-once) loads/stores: keep L2 for the hash tables
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }

}  // namespace b2n
