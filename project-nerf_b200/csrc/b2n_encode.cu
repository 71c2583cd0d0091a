// Input encodings: Fourier features (FourierRepresentation, src/embeddings.py:13-32) and the
// multiresolution hash grid that the reference obtains from tinycudann
// (HashRepresentation, src/embeddings.py:46-89).  Outputs are written at a column offset of a
// wider row-major buffer so the concatenations of src/core.py:276,348 and
// src/decoders.py:83,159 cost no extra pass.
#include "b2n_common.cuh"
#include "b2n_hash.cuh"
#include <cub/block/block_scan.cuh>

namespace b2n {

// ----------------------------------------------------------------------------- Fourier
// arg = (x * f) * pi in fp32, the reference's evaluation order; pi rounded to fp32 like the
// np.pi python scalar is by torch.  The argument reaches ~1e4 rad, so the accurate
// (range-reduced) sincosf is required, never __sinf.
#define B2N_PI_F 3.14159274101257324f

// one thread per (point, band slot): slot 0 copies the D inputs, slot k >= 1 writes the 2 D contiguous values
// [sin(x f_k pi) (D), cos(x f_k pi) (D)] of band k -- the threads of a point cover its output row contiguously.  A block
// owns 256 / (L + 1) whole points, so the index arithmetic is 32-bit and small (the first version spent more on a 64-bit
// division per output element than on the sincosf)
__global__ void __launch_bounds__(256) k_pe_fwd(const float* __restrict__ x, int64_t P, int D, const float* __restrict__ bands,
                                                int L, float* __restrict__ out, int ld, int col0, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  const int slots = L + 1, pts = 256 / slots;
  const int lp = threadIdx.x / slots, k = threadIdx.x - lp * slots;
  const int64_t p = (int64_t)blockIdx.x * pts + lp;
  if (lp >= pts || p >= P) return;
  const float* xp = x + p * D;
  float* row = out + p * ld + col0;
  if (k == 0) {
    for (int d = 0; d < D; ++d) row[d] = xp[d];
  } else {
    const float f = __ldg(bands + k - 1);
    float* dst = row + D + 2 * (k - 1) * D;
    for (int d = 0; d < D; ++d) {
      const float arg = __fmul_rn(__fmul_rn(xp[d], f), B2N_PI_F);
      float sn, cs;
      sincosf(arg, &sn, &cs);
      dst[d] = sn;
      dst[D + d] = cs;
    }
  }
}

__global__ void k_pe_bwd(const float* __restrict__ x, int64_t P, int D, const float* __restrict__ bands, int L,
                         const float* __restrict__ g, int ld, int col0, float* __restrict__ gx, int accumulate, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * D) return;
  const int64_t p = (P * D < (1LL << 31)) ? (int64_t)((uint32_t)i / (uint32_t)D) : i / D;      // 64-bit division only when needed
  const int d = (int)(i - p * D);
  const float xv = x[i];
  const float* row = g + p * ld + col0;
  float acc = row[d];
  for (int k = 0; k < L; ++k) {
    const float f = __ldg(bands + k);
    const float arg = __fmul_rn(__fmul_rn(xv, f), B2N_PI_F);
    float s, c;
    sincosf(arg, &s, &c);
    acc += (row[D + 2 * k * D + d] * c - row[D + (2 * k + 1) * D + d] * s) * (B2N_PI_F * f);
  }
  gx[i] = accumulate ? gx[i] + acc : acc;
}

template <int F>
__global__ void __launch_bounds__(256)
k_hash_fwd(const float* __restrict__ x, int64_t P, float bound, float two_bound, const float* __restrict__ table,
           const Levels lv, int nl, float* __restrict__ out, int ld, int col0, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  __shared__ SmemLevels sl;
  stage_levels(lv, nl, &sl);
  const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= P * nl) return;
  const int64_t p = item / nl;
  const int level = (int)(item - p * nl);
  const b2n_hash_level L = sl.l[level];
  bool in;
  float x01[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  const Cell c = locate(x01, L.scale);
  float vals[8][F];
  if (F == 2) {
    // The two x-neighbours of a corner pair are adjacent table entries half of the time (dense
    // levels: consecutive indices; hashed levels: x has hash prime 1, so for even gx the indices
    // differ only in bit 0).  An aligned pair is fetched with ONE 16-byte gather.
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t cy = c.g[1] + (k & 1), cz = c.g[2] + ((k >> 1) & 1);
      const uint32_t e0 = corner_entry(L, c.g[0], cy, cz), e1 = corner_entry(L, c.g[0] + 1, cy, cz);
      if ((e0 ^ e1) == 1u) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(table) + (e0 >> 1));
        const bool lo = (e0 & 1u) == 0u;
        vals[2 * k][0] = lo ? t.x : t.z, vals[2 * k][1] = lo ? t.y : t.w;
        vals[2 * k + 1][0] = lo ? t.z : t.x, vals[2 * k + 1][1] = lo ? t.w : t.y;
      } else {
        load_feat<F>(table, e0, vals[2 * k]);
        load_feat<F>(table, e1, vals[2 * k + 1]);
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k)
      load_feat<F>(table, corner_entry(L, c.g[0] + (k & 1), c.g[1] + ((k >> 1) & 1), c.g[2] + ((k >> 2) & 1)), vals[k]);
  }
  float acc[F];
#pragma unroll
  for (int f = 0; f < F; ++f) acc[f] = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float wt = ((k & 1) ? c.w[0] : 1.f - c.w[0]) * ((k & 2) ? c.w[1] : 1.f - c.w[1]) *
                     ((k & 4) ? c.w[2] : 1.f - c.w[2]);
#pragma unroll
    for (int f = 0; f < F; ++f) acc[f] += wt * vals[k][f];
  }
  float* o = out + p * ld + col0 + level * F;
  if (F == 2 && ((reinterpret_cast<uintptr_t>(o) & 7) == 0)) {
    __stcs(reinterpret_cast<float2*>(o), make_float2(acc[0], acc[1]));
  } else {
#pragma unroll
    for (int f = 0; f < F; ++f) __stcs(o + f, acc[f]);
  }
}

template <int F>
__global__ void __launch_bounds__(256)
k_hash_bwd_table(const float* __restrict__ x, int64_t P, float bound, float two_bound, const Levels lv, int nl,
                 int l0, const float* __restrict__ g, int ld, int col0, float* __restrict__ g_table, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  // items cover levels l0 .. nl-1 (the dense levels below l0 are handled by k_hash_bwd_table_dense)
  __shared__ SmemLevels sl;
  stage_levels(lv, nl, &sl);
  const int nli = nl - l0;
  const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= P * nli) return;
  const int64_t p = item / nli;
  const int level = l0 + (int)(item - p * nli);
  const b2n_hash_level L = sl.l[level];
  bool in;
  float x01[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  const Cell c = locate(x01, L.scale);
  float gv[F];
  const float* gi = g + p * ld + col0 + level * F;
  if (F == 2 && ((reinterpret_cast<uintptr_t>(gi) & 7) == 0)) {
    const float2 t = __ldcs(reinterpret_cast<const float2*>(gi));
    gv[0] = t.x, gv[1] = t.y;
  } else {
#pragma unroll
    for (int f = 0; f < F; ++f) gv[f] = __ldcs(gi + f);
  }
  bool any = false;
#pragma unroll
  for (int f = 0; f < F; ++f) any |= (gv[f] != 0.f);
  if (!any) return;  // nothing to scatter (e.g. samples that received no gradient)
  if (F == 2) {
    // aligned x-neighbour pairs (see k_hash_fwd) are reduced with ONE 16-byte red.global.add.v4.f32
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t cy = c.g[1] + (k & 1), cz = c.g[2] + ((k >> 1) & 1);
      const float wyz = ((k & 1) ? c.w[1] : 1.f - c.w[1]) * ((k & 2) ? c.w[2] : 1.f - c.w[2]);
      const float w0 = (1.f - c.w[0]) * wyz, w1 = c.w[0] * wyz;
      const uint32_t e0 = corner_entry(L, c.g[0], cy, cz), e1 = corner_entry(L, c.g[0] + 1, cy, cz);
      if ((e0 ^ e1) == 1u) {
        const bool lo = (e0 & 1u) == 0u;
        const float wa = lo ? w0 : w1, wb = lo ? w1 : w0;
        atomicAdd(reinterpret_cast<float4*>(g_table) + (e0 >> 1),
                  make_float4(wa * gv[0], wa * gv[1], wb * gv[0], wb * gv[1]));
      } else {
        atomicAdd(reinterpret_cast<float2*>(g_table) + e0, make_float2(w0 * gv[0], w0 * gv[1]));
        atomicAdd(reinterpret_cast<float2*>(g_table) + e1, make_float2(w1 * gv[0], w1 * gv[1]));
      }
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float wt = ((k & 1) ? c.w[0] : 1.f - c.w[0]) * ((k & 2) ? c.w[1] : 1.f - c.w[1]) *
                     ((k & 4) ? c.w[2] : 1.f - c.w[2]);
    const uint32_t e = corner_entry(L, c.g[0] + (k & 1), c.g[1] + ((k >> 1) & 1), c.g[2] + ((k >> 2) & 1));
    if (F == 2) {
      atomicAdd(reinterpret_cast<float2*>(g_table) + e, make_float2(wt * gv[0], wt * gv[1]));
    } else if (F == 4) {
      atomicAdd(reinterpret_cast<float4*>(g_table) + e, make_float4(wt * gv[0], wt * gv[1], wt * gv[2], wt * gv[3]));
    } else {
#pragma unroll
      for (int f = 0; f < F; ++f) atomicAdd(g_table + (size_t)e * F + f, wt * gv[f]);
    }
  }
}

// Coarse (dense, un-hashed) levels receive millions of reductions into a few thousand entries:
// with one red.global per (point, corner) they serialise in the L2 atomic units (measured: 1.5 ms
// per level against 0.6 ms for a hashed level at 24 M points).  Here one thread owns one POINT
// and loops over the dense levels; lanes are consecutive samples of a ray, which fall into the
// same cell in runs, so every corner is first reduced across each run of equal entries with a
// segmented warp scan and only the run head issues the red.global.
template <int F>
__global__ void __launch_bounds__(256)
k_hash_bwd_table_dense(const float* __restrict__ x, int64_t P, float bound, float two_bound, const Levels lv,
                       int n_dense, const float* __restrict__ g, int ld, int col0, float* __restrict__ g_table, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool live = p < P;
  float x01[3] = {0.f, 0.f, 0.f};
  if (live) {
    bool in;
#pragma unroll
    for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  }
  // the gradients of the first (up to) 8 dense-level features of a point are 32 contiguous bytes: two 16-byte loads
  // instead of one 4-byte load per feature (lanes are 128 B apart, so every load instruction costs 32 L1 wavefronts
  // whatever its width -- this kernel ran at 95 % L1TEX throughput)
  float gall[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const float* grow = g + p * ld + col0;
  const bool vec = live && ((reinterpret_cast<uintptr_t>(grow) & 15) == 0) && (ld - col0 >= 8);
  if (vec) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(grow));
    gall[0] = a.x, gall[1] = a.y, gall[2] = a.z, gall[3] = a.w;
    if (n_dense * F > 4) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(grow) + 1);
      gall[4] = b.x, gall[5] = b.y, gall[6] = b.z, gall[7] = b.w;
    }
  }
  for (int l = 0; l < n_dense; ++l) {
    const b2n_hash_level L = lv.l[l];      // warp-uniform index: constant-bank read
    const Cell c = locate(x01, L.scale);
    float gv[F];
#pragma unroll
    for (int f = 0; f < F; ++f) {
      const int j = l * F + f;
      if (vec && j < 8) {
        float v = gall[0];
#pragma unroll
        for (int q = 1; q < 8; ++q) v = (j == q) ? gall[q] : v;      // register select (l is warp-uniform)
        gv[f] = v;
      } else {
        gv[f] = live ? __ldg(grow + j) : 0.f;
      }
    }
    // Runs: consecutive lanes in the same cell share all 8 entries, so the run structure is computed once per
    // level from the cell index.  The segmented reduction stops after `steps` doubling steps (runs are a few
    // samples long: about res/12 lanes at the sample spacing of a ray): afterwards every lane whose offset inside
    // its run is a multiple of 2^steps holds the sum of up to 2^steps lanes and issues the red.  Fewer steps trade
    // shuffles (the kernel's bottleneck: 10 per corner and level for the full scan) against a few more atomics.
    const uint32_t cell = live ? (c.g[0] + c.g[1] * L.res + c.g[2] * L.res * L.res) : (0xffffffffu - (uint32_t)lane);
    const uint32_t cell_prev = __shfl_up_sync(0xffffffffu, cell, 1);
    const bool head = (lane == 0) || (cell != cell_prev);
    const uint32_t heads = __ballot_sync(0xffffffffu, head);
    const int steps = L.res <= 24 ? 3 : (L.res <= 64 ? 2 : 1);
    const int run_start = 31 - __clz((int)(heads & (0xffffffffu >> (31 - lane))));
    const bool issuer = live && (((lane - run_start) & ((1 << steps) - 1)) == 0);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float wt = ((k & 1) ? c.w[0] : 1.f - c.w[0]) * ((k & 2) ? c.w[1] : 1.f - c.w[1]) *
                       ((k & 4) ? c.w[2] : 1.f - c.w[2]);
      float v[F];
#pragma unroll
      for (int f = 0; f < F; ++f) v[f] = wt * gv[f];
      for (int s = 0; s < steps; ++s) {
        const int o = 1 << s;
        float t[F];
#pragma unroll
        for (int f = 0; f < F; ++f) t[f] = __shfl_down_sync(0xffffffffu, v[f], o);
        // lanes lane+1 .. lane+o all continue this lane's run <=> no head bit among them
        const bool same_run = (lane + o < 32) && (((heads >> (lane + 1)) & ((1u << o) - 1u)) == 0u);
        if (same_run) {
#pragma unroll
          for (int f = 0; f < F; ++f) v[f] += t[f];
        }
      }
      if (issuer) {
        const uint32_t e = corner_entry(L, c.g[0] + (k & 1), c.g[1] + ((k >> 1) & 1), c.g[2] + ((k >> 2) & 1));
        bool any = false;
#pragma unroll
        for (int f = 0; f < F; ++f) any |= (v[f] != 0.f);
        if (any) {
          if (F == 2) {
            atomicAdd(reinterpret_cast<float2*>(g_table) + e, make_float2(v[0], v[1]));
          } else if (F == 4) {
            atomicAdd(reinterpret_cast<float4*>(g_table) + e, make_float4(v[0], v[1], v[2], v[3]));
          } else {
#pragma unroll
            for (int f = 0; f < F; ++f) atomicAdd(g_table + (size_t)e * F + f, v[f]);
          }
        }
      }
    }
  }
}

// ----------------------------------------------------------------------------- pair-lane kernels (F == 2)
// The L1TEX unit retires one 128-byte line per load instruction per clock (the k_hash_fwd above ran at 97 % of that: its
// lanes are the 16 levels of two points, so every gather instruction touches 32 different lines).  Here lanes 2i / 2i+1
// of a warp share point i and take the x = 0 / x = 1 corner column of the cell; the level is warp-uniform and walked in a
// loop.  The two x-neighbours of a corner pair sit in the same 128-byte line (dense levels: adjacent entries; hashed
// levels: x carries hash prime 1, so the indices differ in the low bits only), hence one gather instruction costs 16 lines
// for 16 points instead of 32 lines for 32 (point, level) items at 1.5 instructions per corner pair: 4 instead of 6 line
// visits per (point, level) on the hashed levels, and on the coarse levels the 16 consecutive samples of a ray that a
// warp holds fall into a handful of cells that share their lines.  Level geometry comes from the constant bank.
__device__ __forceinline__ float pair_sum(float v) { return v + __shfl_xor_sync(0xffffffffu, v, 1); }

// Sum of (v0, v1) over the lanes of `peers` (the lanes of this one that hold the same key, __match_any_sync) in log2(|peers|)
// rounds of a tree over the ranks inside the group; the lowest lane of the group ends with the sum and gets true.  All 32
// lanes must call it.  (The warp-aggregation of E. Westphal, "Voting and Shuffling to Optimize Atomic Operations", 2015.)
__device__ __forceinline__ bool reduce_peers(uint32_t peers, float& v0, float& v1) {
  const int lane = threadIdx.x & 31;
  uint32_t rank = __popc(peers & ((1u << lane) - 1u));
  uint32_t above = peers & (0xfffffffeu << lane);              // the group's lanes above this one not yet summed
  const bool leader = rank == 0;
  while (__any_sync(0xffffffffu, above != 0u)) {
    const int next = __ffs(above);                              // nearest lane above still holding a partial sum (1-based)
    const float t0 = __shfl_sync(0xffffffffu, v0, next - 1), t1 = __shfl_sync(0xffffffffu, v1, next - 1);
    if (next) v0 += t0, v1 += t1;
    above &= __ballot_sync(0xffffffffu, !(rank & 1u));          // odd ranks have handed their partial sum down
    rank >>= 1;
  }
  return leader;
}

// Spatial order (b2n_hash_order): in ray order the 16 points of a warp are 16 samples of one ray and share cells only at
// the coarsest levels; in Morton order they share cells and table lines up to the middle levels.  The key is the Morton
// code of the point's cell on a 2^7 lattice over the box; within a bucket points keep the order in which the counting
// pass reached them (features do not depend on it, the table gradient is a sum of atomics anyway).
constexpr int kOrderBits = 7;
constexpr int kOrderBuckets = 1 << (3 * kOrderBits);      // 2 M counters: 8 MB of L2, beside the 52 MB C2 gradient table
constexpr int kOrderTile = 2048;                          // buckets per scan block (256 threads x 8)
constexpr int kOrderTiles = kOrderBuckets / kOrderTile;   // 1024: one block scans the tile sums
// Ordered input: the blocks resident at one time hold ~150 k consecutive points, a small stretch of the curve, and the
// coarse-level reductions of every SM would meet at the same few entries (scatter 7.5 -> 11.5 ms at 24 M points).  Block
// b takes the 128-point chunk (b mod kSpread) * R + b / kSpread of R * kSpread chunks: consecutive blocks sit 1/kSpread of
// the curve apart.  The ordered grid is padded to a multiple of kSpread blocks.
constexpr int kSpread = 2048;

__device__ __forceinline__ uint32_t spread3(uint32_t v) {     // 10 bits -> every third bit
  v = (v | (v << 16)) & 0x030000FFu;
  v = (v | (v << 8)) & 0x0300F00Fu;
  v = (v | (v << 4)) & 0x030C30C3u;
  return (v | (v << 2)) & 0x09249249u;
}

__device__ __forceinline__ uint32_t order_key(const float* __restrict__ x, int64_t p, float bound, float two_bound) {
  uint32_t q[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    bool in;
    const float u = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);      // clamped to [0, 1]; NaN -> 0
    q[d] = min((uint32_t)(u * (float)(1 << kOrderBits)), (uint32_t)((1 << kOrderBits) - 1));
  }
  return spread3(q[0]) | (spread3(q[1]) << 1) | (spread3(q[2]) << 2);
}

// first point of the 128-point chunk this block walks, or -1 (nothing to do)
__device__ __forceinline__ int64_t block_first_point(int64_t P, bool ordered) {
  if (!ordered) return (int64_t)blockIdx.x * 128;
  const int64_t nc = (P + 127) / 128, R = (nc + kSpread - 1) / kSpread, b = blockIdx.x;
  if (b / kSpread >= R) return -1;                      // padding of the grid: keeps the mapping one-to-one
  const int64_t c = (b % kSpread) * R + b / kSpread;
  return c < nc ? c * 128 : -1;
}

__global__ void __launch_bounds__(256)
k_order_count(const float* __restrict__ x, int64_t P, float bound, float two_bound, int* __restrict__ counts,
              int* __restrict__ rank, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) rank[p] = atomicAdd(counts + order_key(x, p, bound, two_bound), 1);
}

// exclusive scan of the bucket counts inside each tile of kOrderTile buckets (in place); tile totals to tile_sum
__global__ void __launch_bounds__(256) k_order_scan_tiles(int* __restrict__ counts, int* __restrict__ tile_sum) {
  using Scan = cub::BlockScan<int, 256>;
  __shared__ typename Scan::TempStorage tmp;
  int4* base = reinterpret_cast<int4*>(counts + (int64_t)blockIdx.x * kOrderTile) + 2 * threadIdx.x;
  const int4 a = base[0], b = base[1];
  int v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  int tot = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += v[i];
  int pre, all;
  Scan(tmp).ExclusiveSum(tot, pre, all);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int t = v[i];
    v[i] = pre;
    pre += t;
  }
  base[0] = make_int4(v[0], v[1], v[2], v[3]);
  base[1] = make_int4(v[4], v[5], v[6], v[7]);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = all;
}

__global__ void __launch_bounds__(kOrderTiles) k_order_scan_top(int* __restrict__ tile_sum) {
  using Scan = cub::BlockScan<int, kOrderTiles>;
  __shared__ typename Scan::TempStorage tmp;
  int v = tile_sum[threadIdx.x];
  Scan(tmp).ExclusiveSum(v, v);
  tile_sum[threadIdx.x] = v;
}

// only the 4-byte order entry is stored at the scattered position; x_sorted follows in k_order_gather with contiguous
// stores (three scattered 4-byte stores per point into the 288 MB x_sorted cost more than the whole sort otherwise)
__global__ void __launch_bounds__(256)
k_order_scatter(const float* __restrict__ x, int64_t P_cap, float bound, float two_bound, const int* __restrict__ counts,
                const int* __restrict__ tile_sum, const int* __restrict__ rank, int* __restrict__ order,
                const int* __restrict__ rows) {
  const int64_t P = clamp_rows(P_cap, rows);
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P_cap) return;
  int64_t pos = p;                                      // rows behind the device-side count keep their place
  if (p < P) {
    const uint32_t k = order_key(x, p, bound, two_bound);
    pos = (int64_t)__ldg(tile_sum + k / kOrderTile) + __ldg(counts + k) + rank[p];
  }
  order[pos] = (int)p;
}

__global__ void __launch_bounds__(256)
k_order_gather(const float* __restrict__ x, int64_t P_cap, const int* __restrict__ order, float* __restrict__ xs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P_cap) return;
  const int64_t p = __ldg(order + i);
#pragma unroll
  for (int d = 0; d < 3; ++d) xs[3 * i + d] = __ldg(x + 3 * p + d);
}

__global__ void __launch_bounds__(256)
k_hash_fwd_pair(const float* __restrict__ x, int64_t P, float bound, float two_bound, const float2* __restrict__ table,
                const Levels lv, int nl, float* __restrict__ out, int ld, int col0, const int* __restrict__ order,
                const int* __restrict__ rows) {
  // order != NULL: x is in sorted order and point i's feature row is row order[i] of out
  P = clamp_rows(P, rows);
  const int64_t p_block = block_first_point(P, order != nullptr);
  if (p_block < 0 || p_block >= P) return;                        // whole block behind the (device-side) row count
  const int64_t p = p_block + (threadIdx.x >> 1);
  const int s = threadIdx.x & 1;
  const bool live = p < P;
  float x01[3] = {0.f, 0.f, 0.f};
  if (live) {
    bool in;
#pragma unroll
    for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  }
  float* orow = out + (order && live ? (int64_t)__ldg(order + p) : p) * ld + col0;
  const bool vec = ((reinterpret_cast<uintptr_t>(out + col0) & 15) == 0) && ((ld & 3) == 0);
  // When the feature rows are contiguous (the plain [P, 2L] output, 2L <= 32) a warp's 16 rows are one contiguous block:
  // the levels are collected in shared memory and leave as fully coalesced 16-byte stores (4 lines per instruction instead
  // of 16: one L1 wavefront per point instead of four)
  __shared__ float4 stage[8][16 * 10];            // row stride 10 float4: (2 pi + s) mod 8 -- conflict-free 16-byte stores
  // (only while the table leaves room in the 126 MB L2: with the 94 MB table of T = 2^20 the full-line stores evict table
  // lines and the kernel gets 26 % slower -- measured, 24 M points)
  const bool contig = vec && col0 == 0 && ld == 2 * nl && ld <= 32 && (nl & 1) == 0 &&
                      (uint64_t)(lv.l[nl - 1].offset + lv.l[nl - 1].size) * 8u <= (64ull << 20);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, pi = lane >> 1;
  // 4 levels = 8 floats = one 32-byte sector of the point's feature row per chunk; lane s stores its 16-byte half
  for (int l0 = 0; l0 < nl; l0 += 4) {
    float keep0 = 0.f, keep1 = 0.f, keep2 = 0.f, keep3 = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = l0 + j;
      float a0 = 0.f, a1 = 0.f;
      if (l < nl) {                                   // warp-uniform
        const b2n_hash_level L = lv.l[l];
        const Cell c = locate(x01, L.scale);
        const uint32_t cx = c.g[0] + (uint32_t)s;
        const float wx = s ? c.w[0] : 1.f - c.w[0];
        float2 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t e = corner_entry(L, cx, c.g[1] + (k & 1), c.g[2] + (k >> 1));
          v[k] = live ? __ldg(table + e) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float w = wx * ((k & 1) ? c.w[1] : 1.f - c.w[1]) * ((k & 2) ? c.w[2] : 1.f - c.w[2]);
          a0 += w * v[k].x, a1 += w * v[k].y;
        }
      }
      a0 = pair_sum(a0), a1 = pair_sum(a1);
      if ((j >> 1) == s) {                             // lane 0 keeps levels l0, l0+1; lane 1 keeps l0+2, l0+3
        if (j & 1) keep2 = a0, keep3 = a1;
        else keep0 = a0, keep1 = a1;
      }
    }
    const int lf = l0 + 2 * s;                         // first level this lane stores
    if (contig) {
      if (lf + 1 < nl) stage[warp][pi * 10 + (lf >> 1)] = make_float4(keep0, keep1, keep2, keep3);
    } else if (live) {
      float* o = orow + 2 * lf;
      if (vec && lf + 1 < nl) {
        __stcs(reinterpret_cast<float4*>(o), make_float4(keep0, keep1, keep2, keep3));
      } else {
        if (lf < nl) __stcs(o, keep0), __stcs(o + 1, keep1);
        if (lf + 1 < nl) __stcs(o + 2, keep2), __stcs(o + 3, keep3);
      }
    }
  }
  if (contig) {
    __syncwarp();
    const int64_t p_warp = p_block + 16 * warp;                                         // first point of this warp
    const int per_row = ld >> 2;                                                        // float4 per feature row
    const int n4 = 16 * per_row;
    for (int i = lane; i < n4; i += 32) {
      const int row = i / per_row, col = i - row * per_row;
      const int64_t pr = p_warp + row;
      // ordered: the rows land at scattered addresses, but each is still one whole 128-byte line
      if (pr < P) __stcs(reinterpret_cast<float4*>(out + (order ? (int64_t)__ldg(order + pr) : pr) * ld) + col,
                         stage[warp][row * 10 + col]);
    }
  }
}

// Table gradient with the same lane mapping.  Ray order (dedup_res == 0): a level whose resolution is <= merge_res is
// reduced across the run of consecutive points (consecutive samples of a ray) that share a cell before the run head issues
// the red.global -- the coarse levels would otherwise serialise millions of reductions on a few thousand addresses.
// Spatial order (dedup_res > 0): the points of a warp are neighbours and reach the same vertices from different cells.  On a
// level whose resolution is <= dedup_res, instruction slot k takes the corner whose vertex has (y, z) parity k, so every
// occurrence of a vertex in the warp falls into the same slot; each slot is reduced over the lanes that hold the same
// entry and one of them issues the red.global.  The finer levels scatter plainly: there the match, the reduction rounds
// and the per-slot weights cost more issue slots than the fewer reductions save (DESIGN.md section 7b).
__global__ void __launch_bounds__(256)
k_hash_bwd_table_pair(const float* __restrict__ x, int64_t P, float bound, float two_bound, const Levels lv, int lbeg,
                      int nl, const float* __restrict__ g, int ld, int col0, float2* __restrict__ g_table,
                      uint32_t merge_res, uint32_t dedup_res, const int* __restrict__ order, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  // levels [lbeg, nl) of the table (lbeg a multiple of 4): a caller that overlaps the gradient all-reduce of the fine
  // levels with the scatter of the coarse ones launches this kernel once per level window.  order != NULL: x is in
  // sorted order and point i's gradient row is row order[i] of g
  const int64_t p_block = block_first_point(P, order != nullptr);
  if (p_block < 0 || p_block >= P) return;                        // whole block behind the (device-side) row count
  const int64_t p = p_block + (threadIdx.x >> 1);
  const int lane = threadIdx.x & 31, s = lane & 1, pi = lane >> 1;     // pi: point index inside the warp (0..15)
  const bool live = p < P;
  float x01[3] = {0.f, 0.f, 0.f};
  if (live) {
    bool in;
#pragma unroll
    for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  }
  const float* grow = g + (order && live ? (int64_t)__ldg(order + p) : p) * ld + col0;
  const bool vec = ((reinterpret_cast<uintptr_t>(g + col0) & 15) == 0) && ((ld & 3) == 0);
  for (int l0 = lbeg; l0 < nl; l0 += 4) {
    float gv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (live) {
      if (vec && l0 + 4 <= nl) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(grow + 2 * l0));
        const float4 b = __ldcs(reinterpret_cast<const float4*>(grow + 2 * l0) + 1);
        gv[0] = a.x, gv[1] = a.y, gv[2] = a.z, gv[3] = a.w, gv[4] = b.x, gv[5] = b.y, gv[6] = b.z, gv[7] = b.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (2 * l0 + j < 2 * nl) gv[j] = __ldcs(grow + 2 * l0 + j);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = l0 + j;
      if (l >= nl) break;                              // warp-uniform
      const b2n_hash_level L = lv.l[l];
      const Cell c = locate(x01, L.scale);
      const uint32_t cx = c.g[0] + (uint32_t)s;
      const float wx = s ? c.w[0] : 1.f - c.w[0];
      const float g0 = gv[2 * j], g1 = gv[2 * j + 1];
      if (L.res <= dedup_res) {
        // samples that received no gradient (and lanes behind the row count) leave the match with a key no entry has
        const bool act = live && (g0 != 0.f || g1 != 0.f);
        const uint32_t py = c.g[1] & 1u, pz = c.g[2] & 1u;
#pragma unroll 1
        for (int k = 0; k < 4; ++k) {
          const uint32_t dy = (k & 1) ^ py, dz = (k >> 1) ^ pz;
          const float w = wx * (dy ? c.w[1] : 1.f - c.w[1]) * (dz ? c.w[2] : 1.f - c.w[2]);
          const uint32_t e = corner_entry(L, cx, c.g[1] + dy, c.g[2] + dz);
          float v0 = w * g0, v1 = w * g1;
          if (reduce_peers(__match_any_sync(0xffffffffu, act ? e : 0xffffffffu), v0, v1) && act)
            atomicAdd(g_table + e, make_float2(v0, v1));
        }
        continue;
      }
      if (dedup_res > 0 || L.res > merge_res) {
        if (live && (g0 != 0.f || g1 != 0.f)) {        // samples that received no gradient scatter nothing
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float w = wx * ((k & 1) ? c.w[1] : 1.f - c.w[1]) * ((k & 2) ? c.w[2] : 1.f - c.w[2]);
            atomicAdd(g_table + corner_entry(L, cx, c.g[1] + (k & 1), c.g[2] + (k >> 1)), make_float2(w * g0, w * g1));
          }
        }
        continue;
      }
      // run structure from the cell index (identical in both lanes of a pair): head bits at the even lane positions
      const uint32_t cell = live ? (c.g[0] + c.g[1] * L.res + c.g[2] * L.res * L.res) : (0xffffffffu - (uint32_t)pi);
      const uint32_t cell_prev = __shfl_up_sync(0xffffffffu, cell, 2);
      const bool head = (pi == 0) || (cell != cell_prev);
      const uint32_t heads = __ballot_sync(0xffffffffu, head && s == 0);
      // merge depth (2^steps points): in ray order runs are about res / 12 samples long; in Morton order a warp's 16
      // points share a cell at the coarse levels and a few of them still do at res ~ 100 (measured at 24 M points)
      const int steps = order ? (L.res <= 54 ? 4 : (L.res <= 122 ? 3 : 2)) : (L.res <= 24 ? 3 : (L.res <= 64 ? 2 : 1));
      const int run_start = (31 - __clz((int)(heads & (0xffffffffu >> (31 - 2 * pi))))) >> 1;
      const bool issuer = live && (((pi - run_start) & ((1 << steps) - 1)) == 0);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float w = wx * ((k & 1) ? c.w[1] : 1.f - c.w[1]) * ((k & 2) ? c.w[2] : 1.f - c.w[2]);
        float v0 = w * g0, v1 = w * g1;
        for (int st = 0; st < steps; ++st) {
          const int o = 1 << st;
          const float t0 = __shfl_down_sync(0xffffffffu, v0, 2 * o), t1 = __shfl_down_sync(0xffffffffu, v1, 2 * o);
          // points pi+1 .. pi+o all continue this point's run <=> none of them is a head
          const uint32_t span = ((1u << (2 * o)) - 1u) & 0x55555555u;      // the even (head) bits of points pi+1 .. pi+o
          const bool same_run = (pi + o < 16) && (((heads >> (2 * (pi + 1))) & span) == 0u);
          if (same_run) v0 += t0, v1 += t1;
        }
        if (issuer && (v0 != 0.f || v1 != 0.f))
          atomicAdd(g_table + corner_entry(L, cx, c.g[1] + (k & 1), c.g[2] + (k >> 1)), make_float2(v0, v1));
      }
    }
  }
}

// dL/dx = sum_levels scale_l * sum_f g_f * d(trilinear)/dw, chained through clamp and the
// division by 2*bound.  One thread per point (the sum over levels stays in registers).
template <int F>
__global__ void __launch_bounds__(256)
k_hash_bwd_input(const float* __restrict__ x, int64_t P, float bound, float two_bound,
                 const float* __restrict__ table, const Levels lv, int nl, const float* __restrict__ g, int ld,
                 int col0, float* __restrict__ gx, int accumulate, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  bool in[3];
  float x01[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in[d]);
  float gsum[3] = {0.f, 0.f, 0.f};
  const float* gi = g + p * ld + col0;
  for (int l = 0; l < nl; ++l) {
    const b2n_hash_level L = lv.l[l];
    const Cell c = locate(x01, L.scale);
    float gv[F];
#pragma unroll
    for (int f = 0; f < F; ++f) gv[f] = gi[l * F + f];
    float dot[8];  // <g, table[corner]>
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v[F];
      load_feat<F>(table, corner_entry(L, c.g[0] + (k & 1), c.g[1] + ((k >> 1) & 1), c.g[2] + ((k >> 2) & 1)), v);
      float s = 0.f;
#pragma unroll
      for (int f = 0; f < F; ++f) s += gv[f] * v[f];
      dot[k] = s;
    }
    const float wx = c.w[0], wy = c.w[1], wz = c.w[2];
    // d/dwx: sum over (y,z) corners of weight_yz * (dot[x=1] - dot[x=0])
    const float ddx = (1.f - wy) * (1.f - wz) * (dot[1] - dot[0]) + wy * (1.f - wz) * (dot[3] - dot[2]) +
                      (1.f - wy) * wz * (dot[5] - dot[4]) + wy * wz * (dot[7] - dot[6]);
    const float ddy = (1.f - wx) * (1.f - wz) * (dot[2] - dot[0]) + wx * (1.f - wz) * (dot[3] - dot[1]) +
                      (1.f - wx) * wz * (dot[6] - dot[4]) + wx * wz * (dot[7] - dot[5]);
    const float ddz = (1.f - wx) * (1.f - wy) * (dot[4] - dot[0]) + wx * (1.f - wy) * (dot[5] - dot[1]) +
                      (1.f - wx) * wy * (dot[6] - dot[2]) + wx * wy * (dot[7] - dot[3]);
    gsum[0] += L.scale * ddx, gsum[1] += L.scale * ddy, gsum[2] += L.scale * ddz;
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const float v = in[d] ? (bound > 0.f ? gsum[d] / two_bound : gsum[d]) : 0.f;
    gx[3 * p + d] = accumulate ? gx[3 * p + d] + v : v;
  }
}

// The same with the pair-lane mapping of k_hash_fwd_pair (F == 2): lanes 2i / 2i+1 share point i and take the x = 0 / x = 1
// corner column, so the two 8-byte gathers of an x-neighbour pair ride in one instruction on one line / sector (4 instead of
// 8 line visits per (point, level)), and twice as many threads walk the levels.  Per lane: d/dx needs t_s = sum_k w_yz[k]
// <g, T[x_s, k]> of BOTH columns (ddx = t_1 - t_0), d/dy and d/dz are sums over the lane's own column weighted by w_x[s];
// all three are linear in the per-lane terms, so the pair is combined once, after the level loop.
__global__ void __launch_bounds__(256)
k_hash_bwd_input_pair(const float* __restrict__ x, int64_t P, float bound, float two_bound, const float2* __restrict__ table,
                      const Levels lv, int nl, const float* __restrict__ g, int ld, int col0, float* __restrict__ gx,
                      int accumulate, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  if ((int64_t)blockIdx.x * (blockDim.x >> 1) >= P) return;      // whole block behind the (device-side) row count
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t p = tid >> 1;
  const int s = threadIdx.x & 1;
  const bool live = p < P;
  bool in[3] = {false, false, false};
  float x01[3] = {0.f, 0.f, 0.f};
  if (live) {
#pragma unroll
    for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in[d]);
  }
  const float* gi = g + p * ld + col0;
  const bool gvec = ((reinterpret_cast<uintptr_t>(g + col0) & 7) == 0) && ((ld & 1) == 0);
  float gsx = 0.f, gsy = 0.f, gsz = 0.f;
  for (int l = 0; l < nl; ++l) {                       // warp-uniform
    const b2n_hash_level L = lv.l[l];
    const Cell c = locate(x01, L.scale);
    const uint32_t cx = c.g[0] + (uint32_t)s;
    float2 gv = make_float2(0.f, 0.f);
    if (live) gv = gvec ? __ldg(reinterpret_cast<const float2*>(gi + 2 * l)) : make_float2(__ldg(gi + 2 * l), __ldg(gi + 2 * l + 1));
    float dot[4];                                      // <g, table[x_s, y, z]>, k = y + 2 z
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t e = corner_entry(L, cx, c.g[1] + (k & 1), c.g[2] + (k >> 1));
      const float2 v = live ? __ldg(table + e) : make_float2(0.f, 0.f);
      dot[k] = gv.x * v.x + gv.y * v.y;
    }
    const float wx = s ? c.w[0] : 1.f - c.w[0], wy = c.w[1], wz = c.w[2];
    const float t = (1.f - wy) * (1.f - wz) * dot[0] + wy * (1.f - wz) * dot[1] + (1.f - wy) * wz * dot[2] + wy * wz * dot[3];
    gsx += L.scale * (s ? t : -t);
    gsy += L.scale * wx * ((1.f - wz) * (dot[1] - dot[0]) + wz * (dot[3] - dot[2]));
    gsz += L.scale * wx * ((1.f - wy) * (dot[2] - dot[0]) + wy * (dot[3] - dot[1]));
  }
  gsx = pair_sum(gsx), gsy = pair_sum(gsy), gsz = pair_sum(gsz);
  if (live && s == 0) {
    const float gs[3] = {gsx, gsy, gsz};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const float v = in[d] ? (bound > 0.f ? gs[d] / two_bound : gs[d]) : 0.f;
      gx[3 * p + d] = accumulate ? gx[3 * p + d] + v : v;
    }
  }
}

// ----------------------------------------------------------------------------- tri-grid temporal blend (Part 4)
// deform_feat = sum_i w_i(t) * HashGrid_i(x), i = start / mid / end anchors at t = 0, 0.5, 1 with tent weights of
// half-width 0.5, normalised (src/core.py:308-335).  The three grids share one geometry, so cell, corner indices and
// trilinear weights are computed once per (point, level) item; a grid whose weight is exactly zero (always at least
// one of the three) is neither gathered nor scattered to.  Replaces 3 encoder launches + ~25 elementwise launches
// (forward) and 3 scatter launches + their autograd glue (backward) by one kernel each way.
struct TriTables {
  const float* t[3];
};
struct TriGrads {
  float* t[3];
};

__device__ __forceinline__ void tri_weights(float tv, float (&w)[3]) {
  // clamp(1 - |t - a| / 0.5, 0, 1) for a in (0, 0.5, 1); / (w0 + w1 + w2 + 1e-8)   -- same fp32 operation order
  const float a[3] = {0.f, 0.5f, 1.f};
#pragma unroll
  for (int i = 0; i < 3; ++i)
    w[i] = fminf(fmaxf(__fsub_rn(1.0f, __fdiv_rn(fabsf(__fsub_rn(tv, a[i])), 0.5f)), 0.f), 1.f);
  const float tot = __fadd_rn(__fadd_rn(__fadd_rn(w[0], w[1]), w[2]), 1e-8f);
#pragma unroll
  for (int i = 0; i < 3; ++i) w[i] = __fdiv_rn(w[i], tot);
}

__global__ void __launch_bounds__(256)
k_hash_tri_fwd(const float* __restrict__ x, const float* __restrict__ tval, int64_t P, float bound, float two_bound,
               const TriTables tabs, const Levels lv, int nl, float* __restrict__ out, int ld, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  __shared__ SmemLevels sl;
  stage_levels(lv, nl, &sl);
  const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= P * nl) return;
  const int64_t p = item / nl;
  const int level = (int)(item - p * nl);
  const b2n_hash_level L = sl.l[level];
  bool in;
  float x01[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  float w[3];
  tri_weights(__ldg(tval + p), w);
  const Cell c = locate(x01, L.scale);
  uint32_t e[8];
  float wt[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    e[k] = corner_entry(L, c.g[0] + (k & 1), c.g[1] + ((k >> 1) & 1), c.g[2] + ((k >> 2) & 1));
    wt[k] = ((k & 1) ? c.w[0] : 1.f - c.w[0]) * ((k & 2) ? c.w[1] : 1.f - c.w[1]) * ((k & 4) ? c.w[2] : 1.f - c.w[2]);
  }
  float o0 = 0.f, o1 = 0.f;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (w[i] == 0.f) continue;          // 0 * f == 0 exactly: the inactive anchor grid is not read
    float vals[8][2];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {    // x-neighbour pair: one 16-byte gather when the two entries are an aligned pair
      if ((e[k] ^ e[k + 1]) == 1u) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(tabs.t[i]) + (e[k] >> 1));
        const bool lo = (e[k] & 1u) == 0u;
        vals[k][0] = lo ? q.x : q.z, vals[k][1] = lo ? q.y : q.w;
        vals[k + 1][0] = lo ? q.z : q.x, vals[k + 1][1] = lo ? q.w : q.y;
      } else {
        load_feat<2>(tabs.t[i], e[k], vals[k]);
        load_feat<2>(tabs.t[i], e[k + 1], vals[k + 1]);
      }
    }
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) a0 += wt[k] * vals[k][0], a1 += wt[k] * vals[k][1];
    o0 = __fadd_rn(o0, __fmul_rn(w[i], a0));
    o1 = __fadd_rn(o1, __fmul_rn(w[i], a1));
  }
  __stcs(reinterpret_cast<float2*>(out + p * ld + level * 2), make_float2(o0, o1));
}

__global__ void __launch_bounds__(256)
k_hash_tri_bwd(const float* __restrict__ x, const float* __restrict__ tval, int64_t P, float bound, float two_bound,
               const Levels lv, int nl, const float* __restrict__ g, int ld, const TriGrads grads, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  __shared__ SmemLevels sl;
  stage_levels(lv, nl, &sl);
  const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= P * nl) return;
  const int64_t p = item / nl;
  const int level = (int)(item - p * nl);
  const b2n_hash_level L = sl.l[level];
  const float2 gv = __ldcs(reinterpret_cast<const float2*>(g + p * ld + level * 2));
  if (gv.x == 0.f && gv.y == 0.f) return;
  bool in;
  float x01[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) x01[d] = to_unit(__ldg(x + 3 * p + d), bound, two_bound, &in);
  float w[3];
  tri_weights(__ldg(tval + p), w);
  const Cell c = locate(x01, L.scale);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t cy = c.g[1] + (k & 1), cz = c.g[2] + ((k >> 1) & 1);
    const float wyz = ((k & 1) ? c.w[1] : 1.f - c.w[1]) * ((k & 2) ? c.w[2] : 1.f - c.w[2]);
    const float w0 = (1.f - c.w[0]) * wyz, w1 = c.w[0] * wyz;
    const uint32_t e0 = corner_entry(L, c.g[0], cy, cz), e1 = corner_entry(L, c.g[0] + 1, cy, cz);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (w[i] == 0.f || !grads.t[i]) continue;
      const float g0 = __fmul_rn(w[i], gv.x), g1 = __fmul_rn(w[i], gv.y);     // d(w_i f_i)/d f_i, as autograd forms it
      if ((e0 ^ e1) == 1u) {
        const bool lo = (e0 & 1u) == 0u;
        const float wa = lo ? w0 : w1, wb = lo ? w1 : w0;
        atomicAdd(reinterpret_cast<float4*>(grads.t[i]) + (e0 >> 1), make_float4(wa * g0, wa * g1, wb * g0, wb * g1));
      } else {
        atomicAdd(reinterpret_cast<float2*>(grads.t[i]) + e0, make_float2(w0 * g0, w0 * g1));
        atomicAdd(reinterpret_cast<float2*>(grads.t[i]) + e1, make_float2(w1 * g0, w1 * g1));
      }
    }
  }
}

// A/B switch of the F == 2 kernels (b2nerf_debug.h: b2n_debug_hash_variant): bit 0 = pair-lane forward, bit 1 = pair-lane
// table gradient; g_merge_res = coarsest-level run merging threshold of the pair-lane table gradient in ray order.
// g_dedup_res (b2n_debug_hash_dedup): in spatial order the table gradient merges equal entries of a warp on the levels with
// res <= g_dedup_res; 0 = run merging up to g_merge_res, as in ray order.
static int g_hash_variant = 3;
static uint32_t g_merge_res = 128;      // measured on the C2 sample set: 64 -> 7.59 ms, 128 -> 7.49, 200 -> 7.44 (T = 2^20: 128 best)
static uint32_t g_dedup_res = 122;      // levels 0-5 of the C2 geometry: DESIGN.md section 7b

static int fill_levels(const b2n_hash_level* h, int L, Levels* out) {
  if (!h || L <= 0 || L > B2N_MAX_LEVELS) return -1;
  for (int i = 0; i < L; ++i) {
    out->l[i] = h[i];
    if (h[i].size == 0) return -1;
    if (h[i].hashed && (h[i].size & (h[i].size - 1))) return -1;
  }
  return 0;
}

}  // namespace b2n

using namespace b2n;

extern "C" int b2n_pe_fwd(const float* x, int64_t P, int D, const float* bands, int L, float* out, int ld_out,
                          int col0, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && D > 0 && D <= 4 && L >= 0 && L <= 32, "bad shape");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && out && (L == 0 || bands), "null pointer");
  B2N_REQUIRE(ld_out >= col0 + D + 2 * D * L && col0 >= 0, "output row too narrow");
  const int pts_per_block = 256 / (L + 1);
  const int64_t blocks = (P + pts_per_block - 1) / pts_per_block;
  B2N_REQUIRE(blocks <= 0x7fffffffLL, "too many points for one launch");
  k_pe_fwd<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, P, D, bands, L, out, ld_out, col0, g_active_rows);
  return check_launch("b2n_pe_fwd");
}

extern "C" int b2n_pe_bwd(const float* x, int64_t P, int D, const float* bands, int L, const float* g_out, int ld_g,
                          int col0, float* g_x, int accumulate, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && D > 0 && D <= 4 && L >= 0 && L <= 32, "bad shape");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && g_out && g_x && (L == 0 || bands), "null pointer");
  B2N_REQUIRE(ld_g >= col0 + D + 2 * D * L && col0 >= 0, "gradient row too narrow");
  k_pe_bwd<<<grid_for(P * D, 256), 256, 0, (cudaStream_t)stream>>>(x, P, D, bands, L, g_out, ld_g, col0, g_x,
                                                                  accumulate, g_active_rows);
  return check_launch("b2n_pe_bwd");
}

// grid of the pair-lane kernels: 128 points per block; ordered input pads it to a multiple of kSpread (block_first_point)
static unsigned pair_grid(int64_t P, const int* order) {
  const int64_t g = (P + 127) / 128;
  return (unsigned)(order ? (g + kSpread - 1) / kSpread * kSpread : (g < 1 ? 1 : g));
}

static int hash_fwd(const float* x, const int* order, int64_t P, float bound, const float* table,
                    const b2n_hash_level* levels_host, int L, int F, float* out, int ld_out, int col0, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && (F == 1 || F == 2 || F == 4) && bound >= 0.f, "bad shape (F in {1,2,4})");
  B2N_REQUIRE(!order || (F == 2 && (g_hash_variant & 1)), "an order needs F = 2 and the pair-lane forward");
  Levels lv;
  B2N_REQUIRE(fill_levels(levels_host, L, &lv) == 0, "bad level table");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && table && out, "null pointer");
  B2N_REQUIRE((reinterpret_cast<uintptr_t>(table) & 15) == 0, "table must be 16-byte aligned (vector gathers)");
  B2N_REQUIRE(ld_out >= col0 + L * F && col0 >= 0, "output row too narrow");
  const unsigned grid = grid_for(P * L, 256);
  const float tb = 2.0f * bound;
  cudaStream_t st = (cudaStream_t)stream;
  if (F == 2 && (g_hash_variant & 1))
    k_hash_fwd_pair<<<pair_grid(P, order), 256, 0, st>>>(x, P, bound, tb, reinterpret_cast<const float2*>(table), lv, L, out,
                                                       ld_out, col0, order, g_active_rows);
  else if (F == 2) k_hash_fwd<2><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, out, ld_out, col0, g_active_rows);
  else if (F == 4) k_hash_fwd<4><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, out, ld_out, col0, g_active_rows);
  else k_hash_fwd<1><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, out, ld_out, col0, g_active_rows);
  return check_launch("b2n_hash_fwd");
}

static int hash_bwd(const float* x, const int* order, int64_t P, float bound, const float* table,
                    const b2n_hash_level* levels_host, int L, int F, const float* g_out, int ld_g, int col0,
                    float* g_table, float* g_x, int accumulate_x, int level_begin, int level_end, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && (F == 1 || F == 2 || F == 4) && bound >= 0.f, "bad shape (F in {1,2,4})");
  if (level_end < 0) level_end = L;
  B2N_REQUIRE(level_begin >= 0 && level_begin <= level_end && level_end <= L, "bad level window");
  const bool windowed = level_begin != 0 || level_end != L;
  B2N_REQUIRE(!windowed || (F == 2 && (level_begin & 3) == 0), "a level window needs F = 2 and a start that is a multiple of 4");
  Levels lv;
  B2N_REQUIRE(fill_levels(levels_host, L, &lv) == 0, "bad level table");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && g_out, "null pointer");
  B2N_REQUIRE(ld_g >= col0 + L * F && col0 >= 0, "gradient row too narrow");
  B2N_REQUIRE(!g_x || table, "input gradient needs the table");
  B2N_REQUIRE((reinterpret_cast<uintptr_t>(g_table) & 15) == 0 && (reinterpret_cast<uintptr_t>(table) & 15) == 0,
              "table / g_table must be 16-byte aligned (vector reductions)");
  B2N_REQUIRE(!order || (!g_x && F == 2 && ((g_hash_variant & 2) || windowed)),
              "an order needs F = 2, the pair-lane table gradient and no input gradient");
  // the entry merge of the ordered scatter keys idle lanes with 0xffffffff, which no entry of the table may be
  B2N_REQUIRE(!order || (uint64_t)lv.l[L - 1].offset + lv.l[L - 1].size < 0xffffffffull, "table too large for the entry merge");
  const float tb = 2.0f * bound;
  cudaStream_t st = (cudaStream_t)stream;
  if (g_table && F == 2 && ((g_hash_variant & 2) || windowed)) {
    if (level_begin < level_end)
      k_hash_bwd_table_pair<<<pair_grid(P, order), 256, 0, st>>>(x, P, bound, tb, lv, level_begin, level_end, g_out, ld_g,
                                                               col0, reinterpret_cast<float2*>(g_table), g_merge_res,
                                                               order ? g_dedup_res : 0u, order,
                                                               g_active_rows);
  } else if (g_table) {
    int n_dense = 0;                      // leading run of un-hashed levels
    while (n_dense < L && !lv.l[n_dense].hashed) ++n_dense;
    if (n_dense > 0) {
      const unsigned gd = grid_for(P, 256);
      if (F == 2) k_hash_bwd_table_dense<2><<<gd, 256, 0, st>>>(x, P, bound, tb, lv, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
      else if (F == 4) k_hash_bwd_table_dense<4><<<gd, 256, 0, st>>>(x, P, bound, tb, lv, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
      else k_hash_bwd_table_dense<1><<<gd, 256, 0, st>>>(x, P, bound, tb, lv, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
    }
    if (n_dense < L) {
      const unsigned grid = grid_for(P * (L - n_dense), 256);
      if (F == 2) k_hash_bwd_table<2><<<grid, 256, 0, st>>>(x, P, bound, tb, lv, L, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
      else if (F == 4) k_hash_bwd_table<4><<<grid, 256, 0, st>>>(x, P, bound, tb, lv, L, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
      else k_hash_bwd_table<1><<<grid, 256, 0, st>>>(x, P, bound, tb, lv, L, n_dense, g_out, ld_g, col0, g_table, g_active_rows);
    }
  }
  if (g_x) {
    const unsigned grid = grid_for(P, 256);
    if (F == 2 && (g_hash_variant & 1))
      k_hash_bwd_input_pair<<<grid_for(2 * P, 256), 256, 0, st>>>(x, P, bound, tb, reinterpret_cast<const float2*>(table), lv, L, g_out,
                                                                ld_g, col0, g_x, accumulate_x, g_active_rows);
    else if (F == 2) k_hash_bwd_input<2><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, g_out, ld_g, col0, g_x, accumulate_x, g_active_rows);
    else if (F == 4) k_hash_bwd_input<4><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, g_out, ld_g, col0, g_x, accumulate_x, g_active_rows);
    else k_hash_bwd_input<1><<<grid, 256, 0, st>>>(x, P, bound, tb, table, lv, L, g_out, ld_g, col0, g_x, accumulate_x, g_active_rows);
  }
  return check_launch("b2n_hash_bwd");
}

extern "C" int b2n_hash_fwd(const float* x, int64_t P, float bound, const float* table,
                            const b2n_hash_level* levels_host, int L, int F, float* out, int ld_out, int col0,
                            b2n_stream_t stream) {
  return hash_fwd(x, nullptr, P, bound, table, levels_host, L, F, out, ld_out, col0, stream);
}

extern "C" int b2n_hash_fwd_ordered(const float* x_sorted, const int* order, int64_t P, float bound, const float* table,
                                    const b2n_hash_level* levels_host, int L, int F, float* out, int ld_out, int col0,
                                    b2n_stream_t stream) {
  B2N_REQUIRE(order, "null order");
  return hash_fwd(x_sorted, order, P, bound, table, levels_host, L, F, out, ld_out, col0, stream);
}

extern "C" int b2n_hash_bwd(const float* x, int64_t P, float bound, const float* table,
                            const b2n_hash_level* levels_host, int L, int F, const float* g_out, int ld_g, int col0,
                            float* g_table, float* g_x, int accumulate_x, int level_begin, int level_end,
                            b2n_stream_t stream) {
  return hash_bwd(x, nullptr, P, bound, table, levels_host, L, F, g_out, ld_g, col0, g_table, g_x, accumulate_x,
                  level_begin, level_end, stream);
}

extern "C" int b2n_hash_bwd_ordered(const float* x_sorted, const int* order, int64_t P, float bound, const float* table,
                                    const b2n_hash_level* levels_host, int L, int F, const float* g_out, int ld_g,
                                    int col0, float* g_table, int level_begin, int level_end, b2n_stream_t stream) {
  B2N_REQUIRE(order, "null order");
  return hash_bwd(x_sorted, order, P, bound, table, levels_host, L, F, g_out, ld_g, col0, g_table, nullptr, 0,
                  level_begin, level_end, stream);
}

extern "C" size_t b2n_hash_order_scratch(int64_t P) {
  return sizeof(int) * ((size_t)kOrderBuckets + kOrderTiles + (size_t)(P > 0 ? P : 0));
}

extern "C" int b2n_hash_order(const float* x, int64_t P, float bound, int* order, float* x_sorted, void* scratch,
                              b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && P < (1LL << 31) && bound >= 0.f, "bad shape (P < 2^31 rows)");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && order && x_sorted && scratch, "null pointer");
  B2N_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "scratch must be 16-byte aligned");
  int* counts = static_cast<int*>(scratch);
  int* tile_sum = counts + kOrderBuckets;
  int* rank = tile_sum + kOrderTiles;
  cudaStream_t st = (cudaStream_t)stream;
  const float tb = 2.0f * bound;
  if (cudaMemsetAsync(counts, 0, sizeof(int) * kOrderBuckets, st) != cudaSuccess) return check_launch("b2n_hash_order");
  k_order_count<<<grid_for(P, 256), 256, 0, st>>>(x, P, bound, tb, counts, rank, g_active_rows);
  k_order_scan_tiles<<<kOrderTiles, 256, 0, st>>>(counts, tile_sum);
  k_order_scan_top<<<1, kOrderTiles, 0, st>>>(tile_sum);
  k_order_scatter<<<grid_for(P, 256), 256, 0, st>>>(x, P, bound, tb, counts, tile_sum, rank, order, g_active_rows);
  k_order_gather<<<grid_for(P, 256), 256, 0, st>>>(x, P, order, x_sorted);
  return check_launch("b2n_hash_order");
}

extern "C" int b2n_hash_tri_fwd(const float* x, const float* t, int64_t P, float bound, const float* table_start,
                                const float* table_mid, const float* table_end, const b2n_hash_level* levels_host, int L,
                                float* out, int ld_out, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && bound >= 0.f, "bad shape");
  Levels lv;
  B2N_REQUIRE(fill_levels(levels_host, L, &lv) == 0, "bad level table");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && t && table_start && table_mid && table_end && out, "null pointer");
  B2N_REQUIRE(ld_out >= 2 * L && (ld_out & 1) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0, "output row too narrow / unaligned");
  const TriTables tabs{{table_start, table_mid, table_end}};
  k_hash_tri_fwd<<<grid_for(P * L, 256), 256, 0, (cudaStream_t)stream>>>(x, t, P, bound, 2.0f * bound, tabs, lv, L, out, ld_out, g_active_rows);
  return check_launch("b2n_hash_tri_fwd");
}

extern "C" int b2n_hash_tri_bwd(const float* x, const float* t, int64_t P, float bound, const b2n_hash_level* levels_host,
                                int L, const float* g_out, int ld_g, float* g_table_start, float* g_table_mid,
                                float* g_table_end, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0 && bound >= 0.f, "bad shape");
  Levels lv;
  B2N_REQUIRE(fill_levels(levels_host, L, &lv) == 0, "bad level table");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x && t && g_out, "null pointer");
  B2N_REQUIRE(ld_g >= 2 * L && (ld_g & 1) == 0 && (reinterpret_cast<uintptr_t>(g_out) & 7) == 0, "gradient row too narrow / unaligned");
  const TriGrads grads{{g_table_start, g_table_mid, g_table_end}};
  k_hash_tri_bwd<<<grid_for(P * L, 256), 256, 0, (cudaStream_t)stream>>>(x, t, P, bound, 2.0f * bound, lv, L, g_out, ld_g, grads, g_active_rows);
  return check_launch("b2n_hash_tri_bwd");
}

extern "C" int b2n_debug_hash_variant(int variant, int merge_res) {
  B2N_REQUIRE(variant >= 0 && variant <= 3, "variant must be in 0..3");
  // the run-merging path builds a uint32 cell id gx + gy res + gz res^2 of a level with res <= merge_res: res^3 must fit
  B2N_REQUIRE(merge_res <= 1625, "merge_res must be <= 1625 (1626^3 overflows the uint32 cell id)");
  g_hash_variant = variant;
  if (merge_res >= 0) g_merge_res = (uint32_t)merge_res;
  return B2N_OK;
}

extern "C" int b2n_debug_hash_config(int* variant, int* merge_res) {
  B2N_REQUIRE(variant && merge_res, "null pointer");
  *variant = g_hash_variant;
  *merge_res = (int)g_merge_res;
  return B2N_OK;
}

extern "C" int b2n_debug_hash_dedup(int dedup_res) {
  const int prev = (int)g_dedup_res;
  if (dedup_res >= 0) g_dedup_res = (uint32_t)dedup_res;
  return prev;
}
