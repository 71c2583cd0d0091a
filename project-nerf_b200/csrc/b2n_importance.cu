// Hierarchical importance sampling (b2n_importance_sample of include/b2nerf.h, DESIGN.md §5h): coarse sigma ->
// compositing weights -> piecewise-constant pdf over the coarse midpoints -> inverse-CDF fine depths -> stable merge
// of the coarse and fine depths.  The rule is the sample_pdf of the original NeRF with sorted (linspace or stratified)
// u, so the fine depths come out sorted without a sort.
//
// One warp per ray.  The ray's coarse depths, its CDF and its fine depths are staged in the warp's slice of shared
// memory; the transmittance is the warp product-scan of b2n_composite_fwd, the CDF a
// warp sum-scan followed by a max-scan (exact), which keeps it non-decreasing whatever the association of the sums.
// searchsorted(c, u) and the merge ranks are binary searches in shared memory: every output is a pure function of the
// ray's inputs, with no atomics, so two runs give identical bits.
#include "b2n_common.cuh"

namespace b2n {

constexpr int kImpWarps = 8;  // rays (warps) per block

__device__ __forceinline__ float warp_incl_mul(float a, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, a, o);
    if (lane >= o) a *= t;
  }
  return a;
}

__device__ __forceinline__ float warp_incl_add(float a, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, a, o);
    if (lane >= o) a = __fadd_rn(a, t);
  }
  return a;
}

__device__ __forceinline__ float warp_incl_max(float a, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, a, o);
    if (lane >= o) a = fmaxf(a, t);
  }
  return a;
}

// number of entries of the sorted a[0..n) that are <= v (upper_bound) or < v (lower_bound); a NaN v counts nothing
__device__ __forceinline__ int upper_bound(const float* a, int n, float v) {
  int lo = 0;
  while (n > 0) {
    const int h = n >> 1;
    if (a[lo + h] <= v) lo += h + 1, n -= h + 1;
    else n = h;
  }
  return lo;
}

__device__ __forceinline__ int lower_bound(const float* a, int n, float v) {
  int lo = 0;
  while (n > 0) {
    const int h = n >> 1;
    if (a[lo + h] < v) lo += h + 1, n -= h + 1;
    else n = h;
  }
  return lo;
}

__device__ __forceinline__ float midpoint(const float* z, int i) { return __fmul_rn(0.5f, __fadd_rn(z[i], z[i + 1])); }

// shared memory of one warp: z [Nc], cdf [Nc-1] (the weights first), z_fine [Nf], merged z and source [Nc+Nf]
__host__ __device__ constexpr int imp_warp_floats(int Nc, int Nf) { return 2 * Nc + Nf + 2 * (Nc + Nf); }

__global__ void __launch_bounds__(kImpWarps * 32)
k_importance(const float* __restrict__ sigma, const float* __restrict__ z, const float* __restrict__ rays_d,
             const float* __restrict__ u_table, const float* __restrict__ u_jitter, int64_t B, int Nc, int Nf,
             float* __restrict__ z_fine, float* __restrict__ z_merged, int32_t* __restrict__ merge_src) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * kImpWarps + wid;
  if (r >= B) return;  // whole warps only: every shuffle below is warp-uniform
  const int M = Nc + Nf, nb = Nc - 1;  // nb = number of bins (midpoints) = CDF entries
  float* sz = smem + (size_t)wid * imp_warp_floats(Nc, Nf);
  float* sc = sz + Nc;
  float* sf = sc + Nc;
  float* smz = sf + Nf;
  int32_t* sms = (int32_t*)(smz + M);

  const float d0 = __ldg(rays_d + 3 * r), d1 = __ldg(rays_d + 3 * r + 1), d2 = __ldg(rays_d + 3 * r + 2);
  const float dn = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);
  const float* zr = z + r * Nc;
  const float* sr = sigma + r * Nc;
  for (int s = lane; s < Nc; s += 32) sz[s] = __ldcs(zr + s);
  __syncwarp();

  // weights w_s = alpha_s T_s with the transmittance scan of b2n_composite_fwd; sc[s] <- w_s + 1e-5 for s in
  // [1, Nc-2].  alpha = -expm1f(-sigma delta) rather than 1 - expf(.): the CDF of a nearly empty ray is made of small
  // weights, whose absolute error 1 - expf would hold at 2^-24 instead of relative to the weight
  float T0 = 1.f;
  for (int base = 0; base < Nc; base += 32) {
    const int s = base + lane;
    const bool valid = s < Nc;
    const float zs = valid ? sz[s] : 0.f;
    const float dl = (s == Nc - 1) ? __fmul_rn(1e10f, dn) : (valid ? __fmul_rn(__fsub_rn(sz[s + 1], zs), dn) : 0.f);
    const float sg = valid ? __ldcs(sr + s) : 0.f;
    const float alpha = valid ? -expm1f(-__fmul_rn(sg, dl)) : 0.f;
    const float a = valid ? __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f) : 1.f;
    const float incl = warp_incl_mul(a, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.f;
    const float wt = alpha * (T0 * excl);
    if (s >= 1 && s <= Nc - 2) sc[s] = __fadd_rn(wt, 1e-5f);
    T0 *= __shfl_sync(0xffffffffu, incl, 31);
  }
  __syncwarp();

  // unnormalised CDF: c[0] = 0, c[j] = sum_{i=1..j} (w_i + 1e-5), made non-decreasing by a running max (exact)
  float carry = 0.f;
  for (int base = 1; base < nb; base += 32) {
    const int j = base + lane;
    const float v = j < nb ? sc[j] : 0.f;
    float c = warp_incl_max(warp_incl_add(v, lane), lane);
    c = fmaxf(__fadd_rn(carry, c), carry);
    if (j < nb) sc[j] = c;
    carry = __shfl_sync(0xffffffffu, c, 31);
  }
  __syncwarp();
  const float total = sc[nb - 1];  // Nc >= 3: at least one bin's mass
  for (int j = lane; j < nb; j += 32) sc[j] = j == 0 ? 0.f : (j == nb - 1 ? 1.f : __fdiv_rn(sc[j], total));
  __syncwarp();

  // inverse CDF; u is non-decreasing in k, so are the fine depths
  float* zfr = z_fine + r * Nf;
  for (int k = lane; k < Nf; k += 32) {
    const float u = u_table ? __ldg(u_table + k)
                            : __fdiv_rn(__fadd_rn((float)k, __ldcs(u_jitter + r * Nf + k)), (float)Nf);
    const int i = upper_bound(sc, nb, u);
    const int below = max(i - 1, 0), above = min(i, nb - 1);
    const float cb = sc[below];
    float denom = __fsub_rn(sc[above], cb);
    if (denom < 1e-5f) denom = 1.f;
    const float t = __fdiv_rn(__fsub_rn(u, cb), denom);
    const float mb = midpoint(sz, below), ma = midpoint(sz, above);
    // the clamp to [m_below, m_above] only absorbs rounding: it keeps the depths sorted and inside the bins
    const float zf = fminf(fmaxf(__fadd_rn(mb, __fmul_rn(t, __fsub_rn(ma, mb))), mb), ma);
    sf[k] = zf;
    __stcs(zfr + k, zf);
  }
  __syncwarp();

  // stable merge, coarse first on ties: rank(coarse s) = s + #{fine < z_s}, rank(fine k) = k + #{coarse <= zf_k}
  for (int s = lane; s < Nc; s += 32) {
    const float v = sz[s];
    const int j = s + lower_bound(sf, Nf, v);
    smz[j] = v, sms[j] = s;
  }
  for (int k = lane; k < Nf; k += 32) {
    const float v = sf[k];
    const int j = k + upper_bound(sz, Nc, v);
    smz[j] = v, sms[j] = Nc + k;
  }
  __syncwarp();
  float* zmr = z_merged + r * M;
  int32_t* msr = merge_src + r * M;
  for (int j = lane; j < M; j += 32) __stcs(zmr + j, smz[j]), __stcs(msr + j, sms[j]);
}

}  // namespace b2n

using namespace b2n;

extern "C" int b2n_importance_sample(const float* sigma, const float* z, const float* rays_d, const float* u_table,
                                     const float* u_jitter, int64_t B, int Nc, int Nf, float* z_fine,
                                     float* z_merged, int32_t* merge_src, b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0, "negative B");
  B2N_REQUIRE(Nc >= 3, "need Nc >= 3 (at least one interior coarse weight)");
  B2N_REQUIRE(Nf >= 1, "need Nf >= 1");
  B2N_REQUIRE(Nc + Nf <= 1024, "need Nc + Nf <= 1024 (the compositing limit)");
  B2N_REQUIRE((u_table == nullptr) != (u_jitter == nullptr), "give exactly one of u_table and u_jitter");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(sigma && z && rays_d && z_fine && z_merged && merge_src, "null pointer");
  const size_t smem = (size_t)kImpWarps * imp_warp_floats(Nc, Nf) * sizeof(float);
  if (smem > 48 * 1024) {  // at most 8 warps x 16 KB (Nc + Nf = 1024)
    const cudaError_t e = cudaFuncSetAttribute(k_importance, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(B2N_ECUDA, "%s: %s", "b2n_importance_sample", cudaGetErrorString(e));
  }
  k_importance<<<grid_for(B, kImpWarps), kImpWarps * 32, smem, (cudaStream_t)stream>>>(
      sigma, z, rays_d, u_table, u_jitter, B, Nc, Nf, z_fine, z_merged, merge_src);
  return check_launch("b2n_importance_sample");
}
