// mma.sync (m16n8k16, 16-bit operands -> fp32) building blocks shared by the fused small-width MLP kernels
// (b2n_mlp64.cu: Instant decoder; b2n_fmlp.cu: deformation / time-modulation nets).
//
// Operand type ``op16``: bf16 by default; a translation unit that defines B2N_OP_F16 before including this header gets
// IEEE fp16 operands (the arithmetic of the reference's tinycudann FullyFusedMLP: 11 significant bits instead of 8 --
// the CPU error budget in tools/bf16_error_budget.py shows the 8-bit forward rounding, not the gradient rounding, is
// what puts the parameter gradients 3e-2 away from fp32).  fp16 conversions saturate (cvt.rn.satfinite) so that a
// large activation clamps to +-65504 instead of becoming inf; gradients are range-managed by the caller (a power-of-two
// scale on the incoming gradient, see k_instant_bwd_tc).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "b2n_common.cuh"

namespace b2n {

#ifdef B2N_OP_F16
typedef __half op16;
#else
typedef __nv_bfloat16 op16;
typedef op16 bf16;
#endif

constexpr int PAD = 8;       // 16-bit row padding: row stride = width + 8 keeps ldmatrix conflict-free

// ------------------------------------------------------------------------------ primitives
#ifdef B2N_OP_F16
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));     // first source -> upper half
  return r;
}
__device__ __forceinline__ float2 unpack2(uint32_t v) {
  return __half22float2(*reinterpret_cast<__half2*>(&v));
}
__device__ __forceinline__ op16 to_op16(float v) {
  const uint32_t r = pack2(v, 0.f);
  return __ushort_as_half((unsigned short)(r & 0xffffu));
}
__device__ __forceinline__ float from_op16(op16 v) { return __half2float(v); }
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
#else
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack2(uint32_t v) {
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&v);
  return __bfloat1622float2(b);
}
__device__ __forceinline__ op16 to_op16(float v) { return __float2bfloat16(v); }
__device__ __forceinline__ float from_op16(op16 v) { return __bfloat162float(v); }
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
#endif
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n" : "=r"(r[0]), "=r"(r[1]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}

// C[mt][j] (16 x 8 tiles) += A[mt][kt] * W^T ; W in smem as [n][k] bf16, row stride S.
// Loop order: k-pairs outer, n-tiles inner, and the two k-halves issued in separate sweeps, so that
// consecutive mma.sync never depend on each other's accumulator (NT*MT independent chains).
template <int MT, int NT, int KT>
__device__ __forceinline__ void gemm_fwd(float (&c)[MT][NT][4], const uint32_t (&a)[MT][KT][4], const op16* W, int S,
                                         int lane) {
  // n-tiles per sweep: G*MT independent accumulators in flight (8 when a warp owns a single 16-row slab)
  constexpr int G = (NT < 4) ? NT : ((MT == 1 && NT == 8) ? 8 : 4);
  const op16* base = W + (lane & 7) * S + 8 * (lane >> 3);
#pragma unroll
  for (int j0 = 0; j0 < NT; j0 += G) {
#pragma unroll
    for (int q = 0; q < KT / 2; ++q) {
      uint32_t b[G][4];
#pragma unroll
      for (int j = 0; j < G; ++j) {
        ldsm_x4(b[j], base + 8 * (j0 + j) * S + 32 * q);
#pragma unroll
        for (int m = 0; m < MT; ++m) mma16816(c[m][j0 + j], a[m][2 * q], b[j][0], b[j][1]);
      }
#pragma unroll
      for (int j = 0; j < G; ++j)
#pragma unroll
        for (int m = 0; m < MT; ++m) mma16816(c[m][j0 + j], a[m][2 * q + 1], b[j][2], b[j][3]);
    }
  }
  if (KT & 1) {
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      uint32_t b[2];
      ldsm_x2(b, W + (8 * j + (lane & 7)) * S + 16 * (KT - 1) + 8 * ((lane >> 3) & 1));
#pragma unroll
      for (int m = 0; m < MT; ++m) mma16816(c[m][j], a[m][KT - 1], b[0], b[1]);
    }
  }
}

// C[j] += (A_lo + A_hi) * W^T for one 16-row slab: the two products of the split first layer that share W_hi, with every
// weight fragment read from shared memory ONCE (lo term first).  KT even.
template <int NT, int KT>
__device__ __forceinline__ void gemm_fwd_hl(float (&c)[NT][4], const uint32_t (&a_hi)[KT][4], const uint32_t (&a_lo)[KT][4],
                                            const op16* W, int S, int lane) {
  static_assert(KT % 2 == 0, "k-tile pairs");
  const op16* base = W + (lane & 7) * S + 8 * (lane >> 3);
#pragma unroll
  for (int q = 0; q < KT / 2; ++q) {
    uint32_t b[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      ldsm_x4(b[j], base + 8 * j * S + 32 * q);
      mma16816(c[j], a_lo[2 * q], b[j][0], b[j][1]);
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) mma16816(c[j], a_lo[2 * q + 1], b[j][2], b[j][3]);
#pragma unroll
    for (int j = 0; j < NT; ++j) mma16816(c[j], a_hi[2 * q], b[j][0], b[j][1]);
#pragma unroll
    for (int j = 0; j < NT; ++j) mma16816(c[j], a_hi[2 * q + 1], b[j][2], b[j][3]);
  }
}

// dIn[16 x 8*NTo] += dZ[16 x 16*KTz] * W ; W in smem as [n][k] (n is the reduction index).
// Reduction index outer so that consecutive mma.sync hit different accumulators.
template <int NTo, int KTz>
__device__ __forceinline__ void gemm_dgrad(float (&c)[NTo][4], const uint32_t (&a)[KTz][4], const op16* W, int S,
                                           int lane) {
  static_assert(NTo % 2 == 0, "pairs of output tiles");
#pragma unroll
  for (int kt = 0; kt < KTz; ++kt) {
#pragma unroll
    for (int jp = 0; jp < NTo / 2; ++jp) {
      uint32_t b[4];
      ldsm_x4_t(b, W + (16 * kt + 8 * ((lane >> 3) & 1) + (lane & 7)) * S + 8 * (2 * jp + (lane >> 4)));
      mma16816(c[2 * jp], a[kt], b[0], b[1]);
      mma16816(c[2 * jp + 1], a[kt], b[2], b[3]);
    }
  }
}

// acc (16 rows of dW starting at n0, NTk*8 columns starting at k0) += dZ^T In over the 64 staged points.
template <int NTk>
__device__ __forceinline__ void wgrad_tile(float (&acc)[NTk][4], const op16* dZ, int Sz, int n0, const op16* In,
                                           int Si, int k0, int lane) {
  static_assert(NTk % 2 == 0, "pairs of tiles");
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    ldsm_x4_t(a, dZ + (16 * ks + 8 * (lane >> 4) + (lane & 7)) * Sz + n0 + 8 * ((lane >> 3) & 1));
#pragma unroll
    for (int jp = 0; jp < NTk / 2; ++jp) {
      uint32_t b[4];
      ldsm_x4_t(b, In + (16 * ks + 8 * ((lane >> 3) & 1) + (lane & 7)) * Si + k0 + 8 * (2 * jp + (lane >> 4)));
      mma16816(acc[2 * jp], a, b[0], b[1]);
      mma16816(acc[2 * jp + 1], a, b[2], b[3]);
    }
  }
}

// C tiles (fp32) -> A fragments (bf16) of the next layer, optional ReLU.
template <int NT, bool RELU>
__device__ __forceinline__ void c_to_a(const float (&c)[NT][4], uint32_t (&a)[NT / 2][4]) {
#pragma unroll
  for (int k = 0; k < NT / 2; ++k) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float* s = c[2 * k + h];
      float v0 = s[0], v1 = s[1], v2 = s[2], v3 = s[3];
      if (RELU) v0 = fmaxf(v0, 0.f), v1 = fmaxf(v1, 0.f), v2 = fmaxf(v2, 0.f), v3 = fmaxf(v3, 0.f);
      a[k][2 * h] = pack2(v0, v1);      // row g
      a[k][2 * h + 1] = pack2(v2, v3);  // row g + 8
    }
  }
}

// store A fragments of a 16-row slab into a [rows][width + PAD] bf16 tile (row0 = first row of the slab)
template <int KT>
__device__ __forceinline__ void store_a(const uint32_t (&a)[KT][4], op16* tile, int S, int row0, int col0, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    uint32_t* r0 = reinterpret_cast<uint32_t*>(tile + (row0 + g) * S + col0 + 16 * k + 2 * t);
    uint32_t* r1 = reinterpret_cast<uint32_t*>(tile + (row0 + g + 8) * S + col0 + 16 * k + 2 * t);
    r0[0] = a[k][0], r1[0] = a[k][1], r0[4] = a[k][2], r1[4] = a[k][3];
  }
}

// fp32 weight matrix [rows][src_cols] (row stride src_cols) -> bf16 smem [rows][cols + PAD]; columns
// src_cols..cols-1 (input padding the parameter vector does not store) are zero-filled
__device__ __forceinline__ void load_weights(const float* __restrict__ W, int rows, int cols, int src_cols, op16* dst) {
  const int S = cols + PAD;
  for (int i = threadIdx.x; i < rows * cols; i += blockDim.x) {
    const int r = i / cols, c = i - r * cols;
    dst[r * S + c] = to_op16(c < src_cols ? __ldg(W + (size_t)r * src_cols + c) : 0.f);
  }
}

}  // namespace b2n
