// Arithmetic of the fused Instant decoder that its forward (k_instant_fwd_tc, b2n_mlp64tc.cu) and the forward recompute
// of its backward (k_instant_bwd_tc, b2n_mlp64.cu) must compute identically -- the backward differentiates what the
// forward rendered: the density head, the output logistic and the view-direction features.
#pragma once
#ifndef B2N_OP_F16
#error "the Instant decoder has fp16 operands: define B2N_OP_F16 before including b2n_mlp64.cuh"
#endif
#include "b2n_mma.cuh"

namespace b2n {

// softplus(h0 - 5) and the logistic function on the MUFU units (ex2 / lg2 / rcp: ~1e-6 relative, two orders below the fp16
// operands around them) instead of libm's expf / log1pf and an IEEE division -- 110 of the ~1300 instructions a thread spent
// per forward tile.  Small e = exp(v): the series of log1p (relative error < e^3 / 4 < 8e-6 below 1/32)
__device__ __forceinline__ float softplus_m5(float h0) {
  const float v = h0 - 5.0f;
  const float e = __expf(fminf(v, 20.f));
  const float sp = e < 0.03125f ? e * (1.f - e * (0.5f - e * 0.33333334f)) : __logf(1.f + e);
  return v > 20.f ? v : sp;
}
__device__ __forceinline__ float sigmoidf(float v) { return __fdividef(1.f, 1.f + __expf(-v)); }

// view-direction Fourier features of one point as 32 fp16: store(i, v) receives 16-byte chunk i (features 8 i .. 8 i + 7)
// and writes it where the caller's tile layout puts it
template <class Store>
__device__ __forceinline__ void dir_features(const float (&d)[3], const float* __restrict__ bands, int L, float pad, Store&& store) {
  // columns [3 + 6 L, pad16(16 + 3 + 6 L) - 16) are the INPUT PADDING of color_net (43 -> 48 at L = 4): they hold `pad`
  // (0, or 1 for checkpoints of an upstream build whose padded inputs are ones: b2n.checkpoint), the rest zeros
  const int dd = 3 + 6 * L, dpad = ((16 + dd + 15) & ~15) - 16;
  float f[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = (i >= dd && i < dpad) ? pad : 0.f;
  f[0] = d[0], f[1] = d[1], f[2] = d[2];
  // band k+1 = 2 * band k (the reference's 2^k bands): double-angle recurrence instead of a fresh
  // sincosf (error grows ~2x per band from 1e-7: far below the fp16 rounding applied next)
  float ps[3], pc[3], prev = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < L) {
      const float fr = __ldg(bands + k);
      const bool dbl = (k > 0) && (fr == 2.f * prev);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        float s, c;
        if (dbl) {
          s = 2.f * ps[j] * pc[j];
          c = 1.f - 2.f * ps[j] * ps[j];
        } else {
          // view directions are unit vectors and the first band is 1: |arg| <= pi, where the MUFU sin/cos (abs.
          // error ~1e-6) is far inside the fp16 rounding applied below; larger arguments take the accurate path
          const float arg = __fmul_rn(__fmul_rn(d[j], fr), 3.14159274101257324f);
          // beyond +-pi (non-unit directions, custom bands): one fp32 reduction step to [-pi, pi] instead of libm's
          // Payne-Hanek path (hundreds of instructions and local memory in a kernel whose code must stay cache-resident)
          const float red = fabsf(arg) <= 3.2f ? arg : __fmaf_rn(-6.28318530717958648f, rintf(arg * 0.159154943091895336f), arg);
          __sincosf(red, &s, &c);
        }
        ps[j] = s, pc[j] = c;
        f[3 + 6 * k + j] = s;
        f[3 + 6 * k + 3 + j] = c;
      }
      prev = fr;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    store(i, make_uint4(pack2(f[8 * i], f[8 * i + 1]), pack2(f[8 * i + 2], f[8 * i + 3]), pack2(f[8 * i + 4], f[8 * i + 5]),
                        pack2(f[8 * i + 6], f[8 * i + 7])));
}

}  // namespace b2n
