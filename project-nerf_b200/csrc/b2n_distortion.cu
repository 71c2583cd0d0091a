// Distortion loss of mip-NeRF 360 (Barron et al. 2022, eq. 15) per ray, and its exact gradient w.r.t. sigma
// (b2n_distortion_* of include/b2nerf.h; DESIGN.md §5j).
//
// One warp per ray; lane l owns samples l, l+32, ... in the sample layouts of b2n_composite.cu (dense [B*N] or compact
// through mask words + ray offsets).  The weights are those of the composite (same per-sample arithmetic, warp
// product-scan per 32-sample chunk with a carried prefix).  In normalised distance s = (z - near) / (far - near),
// sample i owns [s_i, s_{i+1}] (s_N = 1), midpoint m_i and width d_i.  Because m is sorted the double sum is O(N):
//     L = 2 sum_i w_i (m_i W_{<i} - WM_{<i}) + 1/3 sum_i w_i^2 d_i,   W, WM = prefix sums of w and w*m
//     dL/dw_i = 2 (m_i W_{<i} - WM_{<i} + WM_{>i} - m_i W_{>i}) + 2/3 w_i d_i
// and dL/dw goes through the weights with the reverse affine scan of k_composite_bwd (no division by 1 - alpha + 1e-10).
// The backward recomputes the weights: pass 1 front to back (transmittance, offsets and prefix sums entering every
// chunk, totals), pass 2 back to front (gradients).
#include "b2n_common.cuh"

namespace b2n {
namespace {

__device__ __forceinline__ float incl_prod(float a, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, a, o);
    if (lane >= o) a *= t;
  }
  return a;
}

__device__ __forceinline__ float excl_sum(float v, int lane, float* total) {
  float inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  *total = __shfl_sync(0xffffffffu, inc, 31);
  const float ex = __shfl_up_sync(0xffffffffu, inc, 1);
  return lane == 0 ? 0.f : ex;
}

// One 32-sample chunk of a ray: everything but the transmittance, which needs the scan.
struct Chunk {
  bool act;      // an active sample (read from sigma, written to g_sigma)
  int64_t idx;   // its row
  float alpha, a, dl, e, mid, width;
  uint32_t word; // mask word of the chunk (all ones when dense)
};

__device__ __forceinline__ Chunk load_chunk(const float* __restrict__ sigma, const float* __restrict__ z,
                                            const uint32_t* __restrict__ mask_words, int64_t r, int N, int W, int k,
                                            int lane, int64_t off, int64_t lim, float dn, float near, float range) {
  Chunk c;
  const int s = (k << 5) + lane;
  const bool valid = s < N;
  const int64_t zb = r * N;
  c.word = mask_words ? mask_words[r * W + k] : 0xffffffffu;
  c.idx = mask_words ? off + __popc(c.word & ((1u << lane) - 1u)) : off + lane;
  c.act = valid && ((c.word >> lane) & 1u) && c.idx < lim;
  const float zs = valid ? z[zb + s] : 0.f;
  float zn = __shfl_down_sync(0xffffffffu, zs, 1);
  if (lane == 31 && s + 1 < N) zn = z[zb + s + 1];
  // compositing interval (b2n_composite_fwd): delta * |d|, 1e10 * |d| for the last sample
  c.dl = __fmul_rn((s == N - 1) ? 1e10f : __fsub_rn(zn, zs), dn);
  const float sg = c.act ? sigma[c.idx] : 0.f;
  c.e = expf(-__fmul_rn(sg, c.dl));
  c.alpha = valid ? __fsub_rn(1.0f, c.e) : 0.f;
  c.a = valid ? __fadd_rn(__fsub_rn(1.0f, c.alpha), 1e-10f) : 1.f;
  // distortion interval in normalised distance: [s_i, s_{i+1}], s_N = 1 (z_N = far)
  const float si = __fdiv_rn(__fsub_rn(zs, near), range);
  const float sn = (s == N - 1) ? 1.0f : __fdiv_rn(__fsub_rn(zn, near), range);
  c.mid = valid ? 0.5f * __fadd_rn(si, sn) : 0.f;
  c.width = valid ? __fsub_rn(sn, si) : 0.f;
  return c;
}

__device__ __forceinline__ int64_t row_limit(const int* __restrict__ rows) {
  if (!rows) return INT64_MAX;
  const int n = __ldg(rows);
  return n < 0 ? 0 : (int64_t)n;
}

}  // namespace

__global__ void __launch_bounds__(256)
k_distortion_fwd(const float* __restrict__ sigma, const float* __restrict__ z, const float* __restrict__ rays_d,
                 const uint32_t* __restrict__ mask_words, const int32_t* __restrict__ ray_offset, int64_t B, int N,
                 float near, float far, const int* __restrict__ rows, float* __restrict__ loss) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;
  const float range = far - near;
  const int64_t lim = row_limit(rows);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    float term = 0.f, quad = 0.f;
    if (!(mask_words && ray_offset[r + 1] == ray_offset[r])) {  // a ray without an active sample has zero weights
      const float d0 = __ldg(rays_d + 3 * r), d1 = __ldg(rays_d + 3 * r + 1), d2 = __ldg(rays_d + 3 * r + 2);
      const float dn = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);
      int64_t off = mask_words ? (int64_t)ray_offset[r] : r * N;
      float T0 = 1.f, Wc = 0.f, WMc = 0.f;
      for (int k = 0; k < W; ++k) {
        const Chunk c = load_chunk(sigma, z, mask_words, r, N, W, k, lane, off, lim, dn, near, range);
        const float incl = incl_prod(c.a, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.f;
        const float w = c.alpha * (T0 * excl);
        float tw, twm;
        const float Wex = Wc + excl_sum(w, lane, &tw);
        const float WMex = WMc + excl_sum(w * c.mid, lane, &twm);
        term += w * (c.mid * Wex - WMex);
        quad += w * w * c.width;
        Wc += tw, WMc += twm;
        T0 *= __shfl_sync(0xffffffffu, incl, 31);
        off += mask_words ? __popc(c.word) : 32;
      }
    }
    term = warp_sum(term), quad = warp_sum(quad);
    if (lane == 0) loss[r] = 2.0f * term + quad * (1.0f / 3.0f);
  }
}

__global__ void __launch_bounds__(256)
k_distortion_bwd(const float* __restrict__ sigma, const float* __restrict__ z, const float* __restrict__ rays_d,
                 const uint32_t* __restrict__ mask_words, const int32_t* __restrict__ ray_offset, int64_t B, int N,
                 float near, float far, const int* __restrict__ rows, const float* __restrict__ g_loss,
                 float* __restrict__ g_sigma) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;  // <= 32
  const float range = far - near;
  const int64_t lim = row_limit(rows);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    if (mask_words && ray_offset[r + 1] == ray_offset[r]) continue;  // no active sample: nothing to write
    const float d0 = __ldg(rays_d + 3 * r), d1 = __ldg(rays_d + 3 * r + 1), d2 = __ldg(rays_d + 3 * r + 2);
    const float dn = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);
    const int64_t off0 = mask_words ? (int64_t)ray_offset[r] : r * N;
    const float gL = g_loss[r];

    // pass 1 (front to back): transmittance, compact offset and prefix sums entering every chunk; lane k keeps those
    // of chunk k
    float T0 = 1.f, Wc = 0.f, WMc = 0.f, myT = 1.f, myW = 0.f, myWM = 0.f;
    int carryOff = 0, myOff = 0;
    for (int k = 0; k < W; ++k) {
      if (lane == k) myT = T0, myOff = carryOff, myW = Wc, myWM = WMc;
      const Chunk c = load_chunk(sigma, z, mask_words, r, N, W, k, lane, off0 + carryOff, lim, dn, near, range);
      const float incl = incl_prod(c.a, lane);
      float excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) excl = 1.f;
      const float w = c.alpha * (T0 * excl);
      float tw, twm;
      excl_sum(w, lane, &tw);
      excl_sum(w * c.mid, lane, &twm);
      Wc += tw, WMc += twm;
      T0 *= __shfl_sync(0xffffffffu, incl, 31);
      carryOff += mask_words ? __popc(c.word) : 32;
    }
    const float Wtot = Wc, WMtot = WMc;

    // pass 2 (back to front): dL/dw, then the reverse affine scan of the composite backward
    float Rend = 0.f;
    for (int k = W - 1; k >= 0; --k) {
      const int s = (k << 5) + lane;
      const bool valid = s < N;
      const float Tin = __shfl_sync(0xffffffffu, myT, k);
      const int offk = __shfl_sync(0xffffffffu, myOff, k);
      const float Win = __shfl_sync(0xffffffffu, myW, k), WMin = __shfl_sync(0xffffffffu, myWM, k);
      const Chunk c = load_chunk(sigma, z, mask_words, r, N, W, k, lane, off0 + offk, lim, dn, near, range);
      const float incl = incl_prod(c.a, lane);
      float excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) excl = 1.f;
      const float T = Tin * excl;
      const float w = c.alpha * T;
      float tw, twm;
      const float Wex = Win + excl_sum(w, lane, &tw);
      const float WMex = WMin + excl_sum(w * c.mid, lane, &twm);
      const float Wsuf = Wtot - (Wex + w), WMsuf = WMtot - (WMex + w * c.mid);
      const float v =
          gL * (2.0f * (c.mid * Wex - WMex + WMsuf - c.mid * Wsuf) + (2.0f / 3.0f) * w * c.width);
      // suffix composition of f_s(R) = b_s + a_s R over lanes s..31
      float fa = c.a, fb = valid ? c.alpha * v : 0.f;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float a2 = __shfl_down_sync(0xffffffffu, fa, o);
        const float b2 = __shfl_down_sync(0xffffffffu, fb, o);
        if (lane + o < 32) {
          fb = fb + fa * b2;
          fa = fa * a2;
        }
      }
      // R_s = (f_{s+1} o ... o f_31)(Rend)
      float na = __shfl_down_sync(0xffffffffu, fa, 1), nb = __shfl_down_sync(0xffffffffu, fb, 1);
      if (lane == 31) na = 1.f, nb = 0.f;
      const float Rs = nb + na * Rend;
      if (c.act) __stcs(g_sigma + c.idx, T * (v - Rs) * c.dl * c.e);
      const float A0 = __shfl_sync(0xffffffffu, fa, 0), B0 = __shfl_sync(0xffffffffu, fb, 0);
      Rend = B0 + A0 * Rend;
    }
  }
}

static inline unsigned ray_blocks(int64_t B) {  // 8 rays per 256-thread block, a few waves of resident blocks
  int64_t blocks = (B + 7) / 8;
  const int64_t cap = (int64_t)kSMs * 8 * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// checked before any launch, also for B == 0
#define B2N_DISTORTION_ARGS(B, N, near, far)                                                         \
  B2N_REQUIRE((B) >= 0, "negative B");                                                              \
  B2N_REQUIRE((N) >= 1 && (N) <= 1024, "need 1 <= N <= 1024");                                       \
  B2N_REQUIRE(isfinite(near) && isfinite(far) && (far) > (near) && isfinite((far) - (near)),         \
              "near and far must be finite with near < far")

}  // namespace b2n

using namespace b2n;

extern "C" int b2n_distortion_fwd(const float* sigma, const float* z, const float* rays_d, const uint32_t* mask_words,
                                  const int32_t* ray_offset, int64_t B, int N, float near, float far, float* loss,
                                  b2n_stream_t stream) {
  B2N_DISTORTION_ARGS(B, N, near, far);
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(sigma && z && rays_d && loss, "null pointer");
  B2N_REQUIRE(!mask_words == !ray_offset, "the compact layout needs both mask_words and ray_offset");
  k_distortion_fwd<<<ray_blocks(B), 256, 0, (cudaStream_t)stream>>>(sigma, z, rays_d, mask_words, ray_offset, B, N,
                                                                    near, far, g_active_rows, loss);
  return check_launch("b2n_distortion_fwd");
}

extern "C" int b2n_distortion_bwd(const float* sigma, const float* z, const float* rays_d, const uint32_t* mask_words,
                                  const int32_t* ray_offset, int64_t B, int N, float near, float far,
                                  const float* g_loss, float* g_sigma, b2n_stream_t stream) {
  B2N_DISTORTION_ARGS(B, N, near, far);
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(sigma && z && rays_d && g_loss && g_sigma, "null pointer");
  B2N_REQUIRE(!mask_words == !ray_offset, "the compact layout needs both mask_words and ray_offset");
  k_distortion_bwd<<<ray_blocks(B), 256, 0, (cudaStream_t)stream>>>(sigma, z, rays_d, mask_words, ray_offset, B, N,
                                                                    near, far, g_active_rows, g_loss, g_sigma);
  return check_launch("b2n_distortion_bwd");
}
