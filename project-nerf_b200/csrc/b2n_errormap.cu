// Error-map ray sampling (b2n_errormap_* of include/b2nerf.h, DESIGN.md §5i): a per-view map of recent per-pixel loss
// over Hm x Wm cells, updated from each step's per-ray errors, and training pixels drawn in proportion to it (mixed
// with a uniform share), as in Instant-NGP.
//
// Determinism without float atomics: the per-ray errors are quantised to integers (2^-24) and summed with integer
// atomics, so a cell's sum does not depend on the order of the rays (nor on how they are split across ranks).  The CDF
// over the cells is an fp64 prefix in a fixed association, built of three sequential chains: 16 cells per thread, the
// 256 thread totals of a block (4096 cells), then the block totals.  Each chain carries the rounded sum forward, so the
// CDF is non-decreasing and a cell of weight 0 has a CDF step of exactly 0 (the map branch of the sampler never picks
// it).  tests/_errormap_oracle.py restates the same association in numpy, bit for bit.
#include "b2n_common.cuh"

namespace b2n {

constexpr int kEmPer = 16;                           // cells per thread of the CDF kernels
constexpr int kEmThreads = 256;                      // threads per CDF block
constexpr int kEmCells = kEmPer * kEmThreads;        // cells per CDF block
constexpr int kEmChainTile = 1024;                   // block totals staged per step of the cross-block chain
constexpr double kEmQ = 16777216.0;                  // 2^24: fixed-point scale of the accumulated errors

__device__ __forceinline__ int64_t clamp64(int64_t v, int64_t hi) { return v < 0 ? 0 : (v > hi ? hi : v); }

// the cell of pixel (y, x) of view v: (floor(y Hm / H), floor(x Wm / W)), in integers
__device__ __forceinline__ int64_t cell_of(int64_t v, int64_t y, int64_t x, int H, int W, int Hm, int Wm) {
  return (v * Hm + y * Hm / H) * Wm + x * Wm / W;
}

__device__ __forceinline__ double cell_weight(const float* e, int64_t c, int64_t n) {
  return c < n ? (double)fmaxf(__ldg(e + c), 0.f) : 0.0;   // fmaxf: a NaN cell weighs 0
}

__global__ void k_em_accumulate(const int64_t* __restrict__ img_idx, const int64_t* __restrict__ pix_y,
                                const int64_t* __restrict__ pix_x, const float* __restrict__ err, int64_t B, int V,
                                int H, int W, int Hm, int Wm, unsigned long long* __restrict__ acc_sum,
                                unsigned int* __restrict__ acc_cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int64_t v = clamp64(__ldg(img_idx + i), V - 1), y = clamp64(__ldg(pix_y + i), H - 1),
                x = clamp64(__ldg(pix_x + i), W - 1);
  const float r = __ldg(err + i);
  const float s = isfinite(r) ? fminf(fmaxf(r, 0.f), 1.f) : 0.f;
  const unsigned long long q = __float2ull_rn(__fmul_rn(s, 16777216.f));   // exact: a power-of-two scale
  const int64_t c = cell_of(v, y, x, H, W, Hm, Wm);
  atomicAdd(acc_sum + c, q);
  atomicAdd(acc_cnt + c, 1u);
}

__global__ void k_em_apply(float* __restrict__ e, unsigned long long* __restrict__ acc_sum,
                           unsigned int* __restrict__ acc_cnt, int64_t n, float beta) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const unsigned int cnt = acc_cnt[c];
  if (cnt == 0) return;                              // unobserved this step: the sum is 0 too
  const float m = __double2float_rn(__ddiv_rn(__dmul_rn((double)acc_sum[c], 1.0 / kEmQ), (double)cnt));
  const float old = e[c];
  e[c] = old < 0.f ? m : __fadd_rn(__fmul_rn(__fsub_rn(1.f, beta), old), __fmul_rn(beta, m));
  acc_sum[c] = 0ull;
  acc_cnt[c] = 0u;
}

// The block-local part of the CDF for the kEmCells cells of this block: l[j] = the thread's running sum of its 16
// cells (sequential), *excl = the sum of the totals of the threads before it (a sequential chain by thread 0), and the
// return value (the same in every thread) is the block total, excl(last thread) + its total.
__device__ __forceinline__ double em_block_prefix(const float* __restrict__ e, int64_t n, double (&l)[kEmPer],
                                                  double* excl) {
  __shared__ double s_tot[kEmThreads + 1];
  const int64_t base = (int64_t)blockIdx.x * kEmCells + (int64_t)threadIdx.x * kEmPer;
  double run = 0.0;
#pragma unroll
  for (int j = 0; j < kEmPer; ++j) {
    run = __dadd_rn(run, cell_weight(e, base + j, n));
    l[j] = run;
  }
  s_tot[threadIdx.x] = run;
  __syncthreads();
  if (threadIdx.x == 0) {
    double acc = 0.0;
    for (int k = 0; k < kEmThreads; ++k) {
      const double t = s_tot[k];
      s_tot[k] = acc;
      acc = __dadd_rn(acc, t);
    }
    s_tot[kEmThreads] = acc;
  }
  __syncthreads();
  *excl = s_tot[threadIdx.x];
  return s_tot[kEmThreads];
}

__global__ void __launch_bounds__(kEmThreads) k_em_cdf_totals(const float* __restrict__ e, int64_t n,
                                                              double* __restrict__ block_tot) {
  double l[kEmPer], excl;
  const double tot = em_block_prefix(e, n, l, &excl);
  if (threadIdx.x == 0) block_tot[blockIdx.x] = tot;
}

// block_tot[b] <- sum of block_tot[0..b) (a sequential chain by thread 0, one tile at a time); block_tot[nb] <- total
__global__ void __launch_bounds__(kEmChainTile) k_em_cdf_chain(double* __restrict__ block_tot, int64_t nb) {
  __shared__ double s[kEmChainTile];
  double acc = 0.0;
  for (int64_t t0 = 0; t0 < nb; t0 += kEmChainTile) {
    const int64_t i = t0 + threadIdx.x;
    if (i < nb) s[threadIdx.x] = block_tot[i];
    __syncthreads();
    if (threadIdx.x == 0) {
      const int m = nb - t0 < kEmChainTile ? (int)(nb - t0) : kEmChainTile;
      for (int k = 0; k < m; ++k) {
        const double t = s[k];
        s[k] = acc;
        acc = __dadd_rn(acc, t);
      }
    }
    __syncthreads();
    if (i < nb) block_tot[i] = s[threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.x == 0) block_tot[nb] = acc;
}

__global__ void __launch_bounds__(kEmThreads) k_em_cdf_write(const float* __restrict__ e, int64_t n,
                                                             const double* __restrict__ block_off,
                                                             double* __restrict__ cdf) {
  double l[kEmPer], excl;
  em_block_prefix(e, n, l, &excl);
  const double off = block_off[blockIdx.x];
  const int64_t base = (int64_t)blockIdx.x * kEmCells + (int64_t)threadIdx.x * kEmPer;
#pragma unroll
  for (int j = 0; j < kEmPer; ++j)
    if (base + j < n) cdf[base + j] = __dadd_rn(off, __dadd_rn(excl, l[j]));
}

// number of entries of the non-decreasing a[0..n) that are <= v (upper_bound) or < v (lower_bound)
__device__ __forceinline__ int64_t em_upper_bound(const double* a, int64_t n, double v) {
  int64_t lo = 0;
  while (n > 0) {
    const int64_t h = n >> 1;
    if (__ldg(a + lo + h) <= v) lo += h + 1, n -= h + 1;
    else n = h;
  }
  return lo;
}

__device__ __forceinline__ int64_t em_lower_bound(const double* a, int64_t n, double v) {
  int64_t lo = 0;
  while (n > 0) {
    const int64_t h = n >> 1;
    if (__ldg(a + lo + h) < v) lo += h + 1, n -= h + 1;
    else n = h;
  }
  return lo;
}

// floor(f * n) for an fp64 fraction f, clamped to [0, n-1]; NaN -> 0
__device__ __forceinline__ int64_t em_floor_index(double f, int64_t n) {
  const double x = floor(__dmul_rn(f, (double)n));
  if (!(x >= 0.0)) return 0;
  return x >= (double)(n - 1) ? n - 1 : (int64_t)x;
}

__global__ void k_em_sample(const float* __restrict__ e, const double* __restrict__ cdf, const float* __restrict__ u,
                            int64_t B, int V, int H, int W, int Hm, int Wm, float lam, int64_t* __restrict__ img_idx,
                            int64_t* __restrict__ pix_y, int64_t* __restrict__ pix_x, float* __restrict__ ratio) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int64_t n = (int64_t)V * Hm * Wm, HW = (int64_t)H * W, N = (int64_t)V * HW;
  const double S = __ldg(cdf + n - 1);
  const bool use_map = lam < 1.f && S > 0.0 && S < INFINITY;
  const double u0 = (double)__ldg(u + 3 * i), u1 = (double)__ldg(u + 3 * i + 1), u2 = (double)__ldg(u + 3 * i + 2);
  const double L = (double)lam;
  int64_t v, y, x;
  if (!use_map || u0 < L) {                            // uniform over all V*H*W pixels
    const int64_t k = em_floor_index(use_map ? __ddiv_rn(u0, L) : u0, N);
    v = k / HW;
    y = (k - v * HW) / W;
    x = k - v * HW - y * W;
  } else {                                             // a cell from the CDF, then a pixel inside it
    const double t = __dmul_rn(__ddiv_rn(__dsub_rn(u0, L), __dsub_rn(1.0, L)), S);
    // t < S for every u0 < 1; otherwise (u0 >= 1, NaN) the last cell of positive weight
    const int64_t c = t < S ? min(em_upper_bound(cdf, n, t), n - 1) : min(em_lower_bound(cdf, n, S), n - 1);
    v = c / ((int64_t)Hm * Wm);
    const int64_t ci = (c / Wm) % Hm, cj = c % Wm;
    const int64_t y_lo = (ci * H + Hm - 1) / Hm, y_hi = ((ci + 1) * H + Hm - 1) / Hm;
    const int64_t x_lo = (cj * W + Wm - 1) / Wm, x_hi = ((cj + 1) * W + Wm - 1) / Wm;
    y = y_lo + em_floor_index(u1, y_hi - y_lo);
    x = x_lo + em_floor_index(u2, x_hi - x_lo);
  }
  img_idx[i] = v, pix_y[i] = y, pix_x[i] = x;
  // ratio = 1 / (N p(v,y,x)) = 1 / (lam + (1 - lam) w_c N / (S n_y n_x)), p of the pixel whatever branch drew it
  double r = 1.0;
  if (use_map) {
    const int64_t ci = y * Hm / H, cj = x * Wm / W;
    const int64_t ny = ((ci + 1) * H + Hm - 1) / Hm - (ci * H + Hm - 1) / Hm;
    const int64_t nx = ((cj + 1) * W + Wm - 1) / Wm - (cj * W + Wm - 1) / Wm;
    const double w = cell_weight(e, cell_of(v, y, x, H, W, Hm, Wm), n);
    const double share = __ddiv_rn(__dmul_rn(w, (double)N), __dmul_rn(S, (double)(ny * nx)));
    r = __ddiv_rn(1.0, __dadd_rn(L, __dmul_rn(__dsub_rn(1.0, L), share)));
  }
  ratio[i] = __double2float_rn(r);
}

inline int64_t em_blocks(int64_t n) { return (n + kEmCells - 1) / kEmCells; }

}  // namespace b2n

using namespace b2n;

#define B2N_EM_REQUIRE_MAP(V, H, W, Hm, Wm)                                                                     \
  do {                                                                                                          \
    B2N_REQUIRE(V > 0 && H > 0 && W > 0, "need V, H, W >= 1");                                                  \
    B2N_REQUIRE(Hm >= 1 && Hm <= H && Wm >= 1 && Wm <= W, "need 1 <= Hm <= H and 1 <= Wm <= W");               \
    B2N_REQUIRE((int64_t)V * Hm * Wm < ((int64_t)1 << 31), "need V * Hm * Wm < 2^31");                          \
  } while (0)

extern "C" size_t b2n_errormap_scratch(int V, int Hm, int Wm) {
  if (V <= 0 || Hm <= 0 || Wm <= 0 || (int64_t)V * Hm * Wm >= ((int64_t)1 << 31)) return 0;
  return (size_t)(em_blocks((int64_t)V * Hm * Wm) + 1) * sizeof(double);
}

extern "C" int b2n_errormap_accumulate(const int64_t* img_idx, const int64_t* pix_y, const int64_t* pix_x,
                                       const float* err, int64_t B, int V, int H, int W, int Hm, int Wm,
                                       uint64_t* acc_sum, uint32_t* acc_cnt, b2n_stream_t stream) {
  B2N_EM_REQUIRE_MAP(V, H, W, Hm, Wm);
  B2N_REQUIRE(B >= 0 && B < ((int64_t)1 << 31), "need 0 <= B < 2^31");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(img_idx && pix_y && pix_x && err && acc_sum && acc_cnt, "null pointer");
  k_em_accumulate<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(
      img_idx, pix_y, pix_x, err, B, V, H, W, Hm, Wm, (unsigned long long*)acc_sum, (unsigned int*)acc_cnt);
  return check_launch("b2n_errormap_accumulate");
}

extern "C" int b2n_errormap_apply(float* e, uint64_t* acc_sum, uint32_t* acc_cnt, int V, int Hm, int Wm, float beta,
                                  b2n_stream_t stream) {
  B2N_REQUIRE(V > 0 && Hm >= 1 && Wm >= 1 && (int64_t)V * Hm * Wm < ((int64_t)1 << 31),
              "need V, Hm, Wm >= 1 and V * Hm * Wm < 2^31");
  B2N_REQUIRE(beta >= 0.f && beta <= 1.f, "need 0 <= beta <= 1");
  B2N_REQUIRE(e && acc_sum && acc_cnt, "null pointer");
  const int64_t n = (int64_t)V * Hm * Wm;
  k_em_apply<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(e, (unsigned long long*)acc_sum,
                                                                 (unsigned int*)acc_cnt, n, beta);
  return check_launch("b2n_errormap_apply");
}

extern "C" int b2n_errormap_cdf(const float* e, int V, int Hm, int Wm, double* cdf, void* scratch,
                                b2n_stream_t stream) {
  B2N_REQUIRE(V > 0 && Hm >= 1 && Wm >= 1 && (int64_t)V * Hm * Wm < ((int64_t)1 << 31),
              "need V, Hm, Wm >= 1 and V * Hm * Wm < 2^31");
  B2N_REQUIRE(e && cdf && scratch, "null pointer");
  const int64_t n = (int64_t)V * Hm * Wm, nb = em_blocks(n);
  double* block_tot = (double*)scratch;
  cudaStream_t s = (cudaStream_t)stream;
  k_em_cdf_totals<<<(unsigned)nb, kEmThreads, 0, s>>>(e, n, block_tot);
  k_em_cdf_chain<<<1, kEmChainTile, 0, s>>>(block_tot, nb);
  k_em_cdf_write<<<(unsigned)nb, kEmThreads, 0, s>>>(e, n, block_tot, cdf);
  return check_launch("b2n_errormap_cdf");
}

extern "C" int b2n_errormap_sample(const float* e, const double* cdf, const float* u, int64_t B, int V, int H, int W,
                                   int Hm, int Wm, float uniform_frac, int64_t* img_idx, int64_t* pix_y,
                                   int64_t* pix_x, float* ratio, b2n_stream_t stream) {
  B2N_EM_REQUIRE_MAP(V, H, W, Hm, Wm);
  B2N_REQUIRE((int64_t)V * H * W < ((int64_t)1 << 53), "need V * H * W < 2^53");
  B2N_REQUIRE(B >= 0, "negative B");
  B2N_REQUIRE(uniform_frac >= 0.f && uniform_frac <= 1.f, "need 0 <= uniform_frac <= 1");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(e && cdf && u && img_idx && pix_y && pix_x && ratio, "null pointer");
  k_em_sample<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(e, cdf, u, B, V, H, W, Hm, Wm, uniform_frac,
                                                                  img_idx, pix_y, pix_x, ratio);
  return check_launch("b2n_errormap_sample");
}
