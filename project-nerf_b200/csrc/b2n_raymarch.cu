// Ray marching front end: stratified depths, occupancy bitfield test, order-preserving
// compaction, occupancy-grid maintenance.  Replaces src/renderer.py:134-166, :186-201,
// :290-323 and the tail of DensityGrid.update (:119-131) of the reference.
//
// Bit-exactness: every expression that decides a sample depth, a sample position or a voxel
// index is written with __fmul_rn/__fadd_rn/__fsub_rn in the reference's operation order so
// that nvcc cannot contract it into an FMA (torch eager never fuses across ops).
#include "b2n_common.cuh"

namespace b2n {

// trunc((p + offset) * scale) with the reference's validity rule (0 <= idx < R).  Returns -1
// when out of range.  trunc(f) >= 0 <=> f > -1 and trunc(f) < R <=> f < R; NaN fails both.
__device__ __forceinline__ int voxel_axis(float p, float offset, float scale, int R) {
  float f = __fmul_rn(__fadd_rn(p, offset), scale);
  return (f > -1.0f && f < (float)R) ? (int)f : -1;
}

__device__ __forceinline__ bool voxel_active(float px, float py, float pz, const uint32_t* __restrict__ bits, int R,
                                             float offset, float scale) {
  int ix = voxel_axis(px, offset, scale, R);
  int iy = voxel_axis(py, offset, scale, R);
  int iz = voxel_axis(pz, offset, scale, R);
  if ((ix | iy | iz) < 0) return false;
  uint32_t v = ((uint32_t)ix * (uint32_t)R + (uint32_t)iy) * (uint32_t)R + (uint32_t)iz;
  return (__ldg(bits + (v >> 5)) >> (v & 31)) & 1u;
}

__global__ void k_pack_bits(const uint8_t* __restrict__ binary, int64_t n, uint32_t* __restrict__ bits) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool b = (v < n) && binary[v] != 0;
  uint32_t w = __ballot_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0 && v < n) bits[v >> 5] = w;
}

__global__ void k_active_mask(const float* __restrict__ pts, int64_t P, const uint32_t* __restrict__ bits, int R,
                              float offset, float scale, uint8_t* __restrict__ mask) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  mask[p] = voxel_active(pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], bits, R, offset, scale) ? 1 : 0;
}

__global__ void k_occ_update(const float* __restrict__ cur, float* __restrict__ grid, int64_t n, int dynamic,
                             float decay, float thr, uint8_t* __restrict__ binary, uint32_t* __restrict__ bits,
                             unsigned long long* __restrict__ n_active) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool b = false;
  if (v < n) {
    float g = cur[v];
    if (dynamic) g = fmaxf(__fmul_rn(grid[v], decay), g);
    grid[v] = g;
    b = g > thr;
    binary[v] = b ? 1 : 0;
  }
  uint32_t w = __ballot_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0 && v < n) {
    bits[v >> 5] = w;
    if (w) atomicAdd(n_active, (unsigned long long)__popc(w));
  }
}

// One warp per ray.  Lane l owns samples l, l+32, ...
__global__ void __launch_bounds__(256)
k_march_mask(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_base,
             const float* __restrict__ z_lo, const float* __restrict__ z_hi, const float* __restrict__ u,
             const uint32_t* __restrict__ bits, int R, float offset, float scale, int64_t B, int N,
             float* __restrict__ z_out, uint32_t* __restrict__ mask_words, int32_t* __restrict__ ray_count) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    const float ox = __ldg(rays_o + 3 * r), oy = __ldg(rays_o + 3 * r + 1), oz = __ldg(rays_o + 3 * r + 2);
    const float dx = __ldg(rays_d + 3 * r), dy = __ldg(rays_d + 3 * r + 1), dz = __ldg(rays_d + 3 * r + 2);
    int count = 0;
    for (int k = 0; k < W; ++k) {
      const int s = (k << 5) + lane;
      bool act = false;
      if (s < N) {
        float z;
        if (u) {
          const float lo = __ldg(z_lo + s), hi = __ldg(z_hi + s);
          z = __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), __ldcs(u + r * N + s)));
        } else {
          z = __ldg(z_base + s);
        }
        if (z_out) __stcs(z_out + r * N + s, z);
        if (bits) {
          const float px = __fadd_rn(ox, __fmul_rn(dx, z));
          const float py = __fadd_rn(oy, __fmul_rn(dy, z));
          const float pz = __fadd_rn(oz, __fmul_rn(dz, z));
          act = voxel_active(px, py, pz, bits, R, offset, scale);
        } else {
          act = true;
        }
      }
      const uint32_t w = __ballot_sync(0xffffffffu, act);
      if (lane == 0) mask_words[r * W + k] = w;
      count += __popc(w);
    }
    if (lane == 0) ray_count[r] = count;
  }
}

// The same for N <= 32 WC with the chunk loop unrolled: the WC jitter loads of a ray are issued before the first use, the WC
// voxel-bit gathers are independent, and the stratum bounds stay in registers across rays (the rolled loop had one 128-byte
// load in flight per warp: 0.144 ms for a 0.06 ms stream at 2^18 rays x 128 samples)
template <int WC>
__global__ void __launch_bounds__(256)
k_march_mask_u(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_base,
               const float* __restrict__ z_lo, const float* __restrict__ z_hi, const float* __restrict__ u,
               const uint32_t* __restrict__ bits, int R, float offset, float scale, int64_t B, int N,
               float* __restrict__ z_out, uint32_t* __restrict__ mask_words, int32_t* __restrict__ ray_count) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;
  float lo[WC], hi[WC];                      // stratum bounds (or the fixed depths) of this lane's samples: the same for every ray
#pragma unroll
  for (int k = 0; k < WC; ++k) {
    const int s = (k << 5) + lane;
    lo[k] = hi[k] = 0.f;
    if (s < N) {
      if (u) lo[k] = __ldg(z_lo + s), hi[k] = __ldg(z_hi + s);
      else lo[k] = __ldg(z_base + s);
    }
  }
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    float uu[WC];
#pragma unroll
    for (int k = 0; k < WC; ++k) {
      const int s = (k << 5) + lane;
      uu[k] = (u && s < N) ? __ldcs(u + r * N + s) : 0.f;
    }
    const float ox = __ldg(rays_o + 3 * r), oy = __ldg(rays_o + 3 * r + 1), oz = __ldg(rays_o + 3 * r + 2);
    const float dx = __ldg(rays_d + 3 * r), dy = __ldg(rays_d + 3 * r + 1), dz = __ldg(rays_d + 3 * r + 2);
    bool act[WC];
#pragma unroll
    for (int k = 0; k < WC; ++k) {
      const int s = (k << 5) + lane;
      act[k] = false;
      if (s < N) {
        const float z = u ? __fadd_rn(lo[k], __fmul_rn(__fsub_rn(hi[k], lo[k]), uu[k])) : lo[k];
        if (z_out) __stcs(z_out + r * N + s, z);
        if (bits) {
          const float px = __fadd_rn(ox, __fmul_rn(dx, z));
          const float py = __fadd_rn(oy, __fmul_rn(dy, z));
          const float pz = __fadd_rn(oz, __fmul_rn(dz, z));
          act[k] = voxel_active(px, py, pz, bits, R, offset, scale);
        } else {
          act[k] = true;
        }
      }
    }
    int count = 0;
#pragma unroll
    for (int k = 0; k < WC; ++k) {
      const uint32_t w = __ballot_sync(0xffffffffu, act[k]);
      if (k < W) {
        if (lane == 0) mask_words[r * W + k] = w;
        count += __popc(w);
      }
    }
    if (lane == 0) ray_count[r] = count;
  }
}

// ---- exclusive scan of ray_count (three small kernels) --------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 8;
constexpr int kScanChunk = kScanThreads * kScanPerThread;  // 2048 rays per block

__global__ void __launch_bounds__(kScanThreads) k_scan_block_sums(const int32_t* __restrict__ cnt, int64_t B,
                                                                  int32_t* __restrict__ block_sums) {
  __shared__ int tot;
  const int64_t base = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanPerThread;
  int s = 0;
#pragma unroll
  for (int i = 0; i < kScanPerThread; ++i)
    if (base + i < B) s += cnt[base + i];
  block_exclusive_scan(s, &tot);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

// single block: exclusive scan of the block sums in place; total + forced-first flag
__global__ void __launch_bounds__(1024) k_scan_top(int32_t* __restrict__ block_sums, int nb,
                                                   int32_t* __restrict__ total_out, int32_t* __restrict__ forced) {
  __shared__ int tot;
  int carry = 0;
  for (int base = 0; base < nb; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < nb ? block_sums[i] : 0;
    const int ex = block_exclusive_scan(v, &tot);
    if (i < nb) block_sums[i] = carry + ex;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *forced = (carry == 0) ? 1 : 0;
    *total_out = (carry == 0) ? 1 : carry;
  }
}

__global__ void __launch_bounds__(kScanThreads)
k_scan_final(int32_t* __restrict__ cnt, uint32_t* __restrict__ mask_words, int64_t B,
             const int32_t* __restrict__ block_sums, const int32_t* __restrict__ total,
             const int32_t* __restrict__ forced, int32_t* __restrict__ ray_offset) {
  __shared__ int tot;
  const int64_t base = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanPerThread;
  int v[kScanPerThread];
  int s = 0;
#pragma unroll
  for (int i = 0; i < kScanPerThread; ++i) {
    v[i] = (base + i < B) ? cnt[base + i] : 0;
    s += v[i];
  }
  int ex = block_exclusive_scan(s, &tot) + block_sums[blockIdx.x];
  const int f = *forced;  // no active sample anywhere: sample 0 of ray 0 is queried anyway
#pragma unroll
  for (int i = 0; i < kScanPerThread; ++i) {
    if (base + i < B) ray_offset[base + i] = f ? ((base + i) > 0 ? 1 : 0) : ex;
    ex += v[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ray_offset[B] = *total;
    if (f) {
      cnt[0] = 1;
      mask_words[0] |= 1u;
    }
  }
}

__global__ void __launch_bounds__(256)
k_march_compact(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ times,
                const float* __restrict__ z, const uint32_t* __restrict__ mask_words,
                const int32_t* __restrict__ ray_offset, int64_t B, int N, int32_t* __restrict__ sample_idx,
                float* __restrict__ pts, float* __restrict__ dirs, float* __restrict__ t_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    const float ox = __ldg(rays_o + 3 * r), oy = __ldg(rays_o + 3 * r + 1), oz = __ldg(rays_o + 3 * r + 2);
    const float dx = __ldg(rays_d + 3 * r), dy = __ldg(rays_d + 3 * r + 1), dz = __ldg(rays_d + 3 * r + 2);
    const float nrm = sqrtf(dx * dx + dy * dy + dz * dz);
    const float vx = __fdiv_rn(dx, nrm), vy = __fdiv_rn(dy, nrm), vz = __fdiv_rn(dz, nrm);
    const float tt = times ? __ldg(times + r) : 0.f;
    int64_t out = mask_words ? (int64_t)ray_offset[r] : r * N;
    for (int k = 0; k < W; ++k) {
      const int s = (k << 5) + lane;
      uint32_t w;
      if (mask_words) {
        w = mask_words[r * W + k];
      } else {
        const int rem = N - (k << 5);
        w = rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u);
      }
      if ((w >> lane) & 1u) {
        const int64_t j = out + __popc(w & ((1u << lane) - 1u));
        if (sample_idx) sample_idx[j] = (int32_t)(r * N + s);
        const float zz = z[r * N + s];
        if (pts) {
          pts[3 * j] = __fadd_rn(ox, __fmul_rn(dx, zz));
          pts[3 * j + 1] = __fadd_rn(oy, __fmul_rn(dy, zz));
          pts[3 * j + 2] = __fadd_rn(oz, __fmul_rn(dz, zz));
        }
        if (dirs) {
          dirs[3 * j] = vx;
          dirs[3 * j + 1] = vy;
          dirs[3 * j + 2] = vz;
        }
        if (t_out) t_out[j] = tt;
      }
      out += __popc(w);
    }
  }
}

// Backward of the points of k_march_compact, pts = o + d * z: g_o = sum_s g_pts, g_d = sum_s z_s g_pts over the ray's
// active samples.  One warp per ray, rows found as in k_march_compact (so rows behind a device-side count are never
// reached); each lane sums its own samples in order, then a fixed xor-butterfly: deterministic without atomics.
__global__ void __launch_bounds__(256)
k_march_points_bwd(const float* __restrict__ z, const uint32_t* __restrict__ mask_words,
                   const int32_t* __restrict__ ray_offset, const float* __restrict__ g_pts, int64_t B, int N,
                   float* __restrict__ g_o, float* __restrict__ g_d) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int W = (N + 31) >> 5;
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < B; r += warps) {
    float so[3] = {0.f, 0.f, 0.f}, sd[3] = {0.f, 0.f, 0.f};
    int64_t out = mask_words ? (int64_t)ray_offset[r] : r * N;
    for (int k = 0; k < W; ++k) {
      uint32_t w;
      if (mask_words) {
        w = mask_words[r * W + k];
      } else {
        const int rem = N - (k << 5);
        w = rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u);
      }
      if ((w >> lane) & 1u) {
        const int64_t j = out + __popc(w & ((1u << lane) - 1u));
        const float zz = __ldg(z + r * N + (k << 5) + lane);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float g = __ldcs(g_pts + 3 * j + c);
          so[c] += g;
          sd[c] = fmaf(zz, g, sd[c]);
        }
      }
      out += __popc(w);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      so[c] = warp_sum(so[c]);
      sd[c] = warp_sum(sd[c]);
    }
    if (lane < 3) {
      g_o[3 * r + lane] = lane == 0 ? so[0] : (lane == 1 ? so[1] : so[2]);
      g_d[3 * r + lane] = lane == 0 ? sd[0] : (lane == 1 ? sd[1] : sd[2]);
    }
  }
}

}  // namespace b2n

using namespace b2n;

extern "C" int b2n_occ_pack_bits(const uint8_t* binary, int64_t n_voxels, uint32_t* bits, b2n_stream_t stream) {
  B2N_REQUIRE(binary && bits && n_voxels >= 0, "null pointer or negative size");
  if (n_voxels == 0) return B2N_OK;
  k_pack_bits<<<grid_for(n_voxels, 256), 256, 0, (cudaStream_t)stream>>>(binary, n_voxels, bits);
  return check_launch("b2n_occ_pack_bits");
}

extern "C" int b2n_occ_active_mask(const float* pts, int64_t P, const uint32_t* bits, int R, float offset, float scale,
                                   uint8_t* mask, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && R > 0 && R <= 1024, "bad size");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(pts && bits && mask, "null pointer");
  k_active_mask<<<grid_for(P, 256), 256, 0, (cudaStream_t)stream>>>(pts, P, bits, R, offset, scale, mask);
  return check_launch("b2n_occ_active_mask");
}

extern "C" int b2n_occ_update(const float* cur_sigma, float* grid, int64_t n_voxels, int dynamic, float decay,
                              float threshold, uint8_t* binary, uint32_t* bits, int64_t* n_active,
                              b2n_stream_t stream) {
  B2N_REQUIRE(cur_sigma && grid && binary && bits && n_active && n_voxels > 0, "null pointer or bad size");
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(n_active, 0, sizeof(int64_t), st) != cudaSuccess) return check_launch("b2n_occ_update/memset");
  k_occ_update<<<grid_for(n_voxels, 256), 256, 0, st>>>(cur_sigma, grid, n_voxels, dynamic, decay, threshold, binary,
                                                       bits, (unsigned long long*)n_active);
  return check_launch("b2n_occ_update");
}

static inline unsigned ray_grid(int64_t B) {
  int64_t blocks = (B + 7) / 8;  // 8 warps (rays) per 256-thread block
  const int64_t cap = (int64_t)kSMs * 8 * 4;
  if (blocks > cap) blocks = cap;  // grid-stride beyond 4 waves of 8 resident blocks per SM
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

extern "C" int b2n_march_mask(const float* rays_o, const float* rays_d, const float* z_base, const float* z_lo,
                              const float* z_hi, const float* u, const uint32_t* bits, int R, float offset,
                              float scale, int64_t B, int N, float* z, uint32_t* mask_words, int32_t* ray_count,
                              b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0 && N > 0 && N <= 4096, "bad B or N");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(rays_o && rays_d && z_base && mask_words && ray_count, "null pointer");
  B2N_REQUIRE(!u || (z_lo && z_hi && z), "jitter needs the stratum bounds and z");
  B2N_REQUIRE(!bits || (R > 0 && R <= 1024), "bad grid resolution");
  B2N_REQUIRE(B * (int64_t)N < (int64_t)1 << 31, "B*N must fit int32");
  if (N <= 64)
    k_march_mask_u<2><<<ray_grid(B), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, z_base, z_lo, z_hi, u, bits, R, offset,
                                                                    scale, B, N, z, mask_words, ray_count);
  else if (N <= 128)
    k_march_mask_u<4><<<ray_grid(B), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, z_base, z_lo, z_hi, u, bits, R, offset,
                                                                    scale, B, N, z, mask_words, ray_count);
  else
    k_march_mask<<<ray_grid(B), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, z_base, z_lo, z_hi, u, bits, R, offset,
                                                               scale, B, N, z, mask_words, ray_count);
  return check_launch("b2n_march_mask");
}

extern "C" size_t b2n_march_scan_scratch(int64_t B) {
  int64_t nb = (B + kScanChunk - 1) / kScanChunk;
  if (nb < 1) nb = 1;
  return (size_t)(nb + 4) * sizeof(int32_t);
}

extern "C" int b2n_march_scan(int32_t* ray_count, uint32_t* mask_words, int W, int64_t B, int32_t* ray_offset,
                              int32_t* total_out, void* scratch, b2n_stream_t stream) {
  B2N_REQUIRE(B > 0 && W > 0, "bad size");
  B2N_REQUIRE(ray_count && mask_words && ray_offset && total_out && scratch, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int nb = (int)((B + kScanChunk - 1) / kScanChunk);
  int32_t* block_sums = (int32_t*)scratch;
  int32_t* forced = block_sums + nb;
  k_scan_block_sums<<<nb, kScanThreads, 0, st>>>(ray_count, B, block_sums);
  k_scan_top<<<1, 1024, 0, st>>>(block_sums, nb, total_out, forced);
  k_scan_final<<<nb, kScanThreads, 0, st>>>(ray_count, mask_words, B, block_sums, total_out, forced, ray_offset);
  return check_launch("b2n_march_scan");
}

extern "C" int b2n_march_compact(const float* rays_o, const float* rays_d, const float* times, const float* z,
                                 const uint32_t* mask_words, const int32_t* ray_offset, int64_t B, int N,
                                 int32_t* sample_idx, float* pts, float* dirs, float* t_out, b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0 && N > 0 && N <= 4096, "bad B or N");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(rays_o && rays_d && z, "null pointer");
  B2N_REQUIRE(!mask_words || ray_offset, "compact mode needs ray_offset");
  B2N_REQUIRE(!t_out || times, "t_out needs times");
  k_march_compact<<<ray_grid(B), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, times, z, mask_words, ray_offset, B,
                                                                N, sample_idx, pts, dirs, t_out);
  return check_launch("b2n_march_compact");
}

extern "C" int b2n_march_points_bwd(const float* z, const uint32_t* mask_words, const int32_t* ray_offset,
                                    const float* g_pts, int64_t B, int N, float* g_rays_o, float* g_rays_d,
                                    b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0 && N > 0 && N <= 4096, "bad B or N");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(z && g_pts && g_rays_o && g_rays_d, "null pointer");
  B2N_REQUIRE(!mask_words || ray_offset, "compact mode needs ray_offset");
  B2N_REQUIRE(B * (int64_t)N < (int64_t)1 << 31, "B*N must fit int32");
  k_march_points_bwd<<<ray_grid(B), 256, 0, (cudaStream_t)stream>>>(z, mask_words, ray_offset, g_pts, B, N, g_rays_o,
                                                                   g_rays_d);
  return check_launch("b2n_march_points_bwd");
}
