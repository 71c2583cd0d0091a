// Surface extraction from a density lattice (b2n_mesh_*): marching tetrahedra over the Kuhn triangulation of the
// lattice, as a count -> scan -> emit chain without atomics.  The rules (lattice, padding ring, tetrahedra, vertex
// arithmetic, winding, order) are those of include/b2nerf.h and DESIGN.md §5f; tests/_mesh_oracle.py restates them in
// numpy float32 and the GPU tests compare against it bit for bit.
//
// Every pass walks the EXTENDED point lattice (R + 2 points per axis, the virtual sigma = 0 ring included) in tiles of
// kTile consecutive linear indices.  A point p doubles as the cell whose lowest corner it is: cells on the far faces
// (a coordinate of R + 1) have all corners in the ring and therefore no triangles, so one tiling and one scan serve both
// the per-point vertex counts and the per-cell triangle counts, and cell order = point order.
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "b2n_common.cuh"

namespace b2n {
namespace {

constexpr int kThreads = 256;
constexpr int kIters = 16;
constexpr int kTile = kThreads * kIters;     // 4096 points: tile sums stay below 2^16 (<= 7 vertices, <= 12 triangles each)
constexpr int kTopThreads = 256;
constexpr int kTopItems = 16;
constexpr int kMaxR = 1024;

// corner / direction codes: bit 0 = +x, bit 1 = +y, bit 2 = +z.  Direction classes in vertex order: x y z xy xz yz xyz.
__constant__ int8_t c_dir_code[7] = {1, 2, 4, 3, 5, 6, 7};
__constant__ int8_t c_dir_of_code[8] = {-1, 0, 1, 3, 2, 4, 5, 6};
// the 6 Kuhn tetrahedra {0, e_a, e_a + e_b, 1} for the permutations (a, b, c) in lexicographic order
// (xyz, xzy, yxz, yzx, zxy, zyx): codes of local vertices 1 and 2, and the permutation's parity (1 = odd: the
// tetrahedron (v0, v1, v2, v3) is negatively oriented and every triangle of the table is emitted reversed)
__constant__ int8_t c_tet_v1[6] = {1, 1, 2, 2, 4, 4};
__constant__ int8_t c_tet_v2[6] = {3, 5, 3, 6, 5, 6};
__constant__ int8_t c_tet_odd[6] = {0, 1, 1, 0, 0, 1};
// local edges (m, n), m < n: the edge runs from local vertex m (its lower end) to local vertex n
__constant__ int8_t c_edge_m[6] = {0, 0, 0, 1, 1, 2};
__constant__ int8_t c_edge_n[6] = {1, 2, 3, 2, 3, 3};
// case = bit m set when local vertex m is inside.  Triangles of a positively oriented tetrahedron, as local edges, wound
// so that the normal points from inside to outside.  1 inside (i): (ij, ik, il) with (i, j, k, l) an even permutation,
// j < k < l before the fix-up; 3 inside (outside o): (oa, oc, ob) likewise; 2 inside (i < j, outside k, l, (i, j, k, l)
// even): the quad (ik, il, jl, jk) split along the diagonal ik - jl.
__constant__ int8_t c_ntri[16] = {0, 1, 1, 2, 1, 2, 2, 1, 1, 2, 2, 1, 2, 1, 1, 0};
__constant__ int8_t c_tri[16][2][3] = {
    {{0, 0, 0}, {0, 0, 0}}, {{0, 1, 2}, {0, 0, 0}}, {{0, 4, 3}, {0, 0, 0}}, {{1, 2, 4}, {1, 4, 3}},
    {{1, 3, 5}, {0, 0, 0}}, {{2, 0, 3}, {2, 3, 5}}, {{0, 4, 5}, {0, 5, 1}}, {{2, 4, 5}, {0, 0, 0}},
    {{2, 5, 4}, {0, 0, 0}}, {{0, 1, 5}, {0, 5, 4}}, {{3, 0, 2}, {3, 2, 5}}, {{1, 5, 3}, {0, 0, 0}},
    {{1, 3, 4}, {1, 4, 2}}, {{0, 3, 4}, {0, 0, 0}}, {{0, 2, 1}, {0, 0, 0}}, {{0, 0, 0}, {0, 0, 0}}};

struct Lattice {
  const float* __restrict__ sigma;
  int R, N;          // N = R + 2
  int64_t M;         // N^3 points
  float tau;

  // sigma of the extended lattice: the virtual ring (and anything beyond it) is 0
  __device__ __forceinline__ float sig(int i, int j, int k) const {
    if ((unsigned)(i - 1) >= (unsigned)R || (unsigned)(j - 1) >= (unsigned)R || (unsigned)(k - 1) >= (unsigned)R)
      return 0.f;
    return __ldg(sigma + ((int64_t)(i - 1) * R + (j - 1)) * R + (k - 1));
  }
  __device__ __forceinline__ int64_t corner_delta(int code) const {
    return (code & 1 ? (int64_t)N * N : 0) + (code & 2 ? N : 0) + (code & 4 ? 1 : 0);
  }
  __device__ __forceinline__ void coords(int64_t p, int& i, int& j, int& k) const {
    const uint32_t q = (uint32_t)p, n = (uint32_t)N;
    k = (int)(q % n);
    const uint32_t r = q / n;
    j = (int)(r % n);
    i = (int)(r / n);
  }
};

// Per point: bits 0-6 = crossing mask of its 7 outgoing edges, bit 7 = inside, bits 8-11 = triangles of the cell it is the
// lowest corner of.  Per tile: (vertices | triangles << 16).
__global__ void __launch_bounds__(kThreads) k_mesh_count(Lattice L, uint16_t* __restrict__ code, uint32_t* __restrict__ tile_sum) {
  using Reduce = cub::BlockReduce<uint32_t, kThreads>;
  __shared__ typename Reduce::TempStorage tmp;
  const int64_t base = (int64_t)blockIdx.x * kTile;
  uint32_t acc = 0;
  for (int it = 0; it < kIters; ++it) {
    const int64_t p = base + it * kThreads + threadIdx.x;
    if (p >= L.M) break;
    int i, j, k;
    L.coords(p, i, j, k);
    uint32_t in8 = 0;                                   // bit c: corner with code c is inside
#pragma unroll
    for (int c = 0; c < 8; ++c) in8 |= (uint32_t)(L.sig(i + (c & 1), j + ((c >> 1) & 1), k + ((c >> 2) & 1)) > L.tau) << c;
    const uint32_t in0 = in8 & 1u;
    uint32_t mask = 0;
#pragma unroll
    for (int d = 0; d < 7; ++d) mask |= (((in8 >> c_dir_code[d]) & 1u) ^ in0) << d;
    uint32_t ntri = 0;
    if (in8 != 0 && in8 != 0xffu) {
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        const uint32_t cs = in0 | (((in8 >> c_tet_v1[q]) & 1u) << 1) | (((in8 >> c_tet_v2[q]) & 1u) << 2) | ((in8 >> 7) << 3);
        ntri += c_ntri[cs];
      }
    }
    code[p] = (uint16_t)(mask | (in0 << 7) | (ntri << 8));
    acc += __popc(mask) | (ntri << 16);
  }
  const uint32_t tot = Reduce(tmp).Sum(acc);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

// One block: exclusive int64 scans of the tile sums -> tile_off [T][2] (vertex, triangle) and the totals.
__global__ void __launch_bounds__(kTopThreads, 1) k_mesh_scan_top(const uint32_t* __restrict__ tile_sum, int64_t T,
                                                               long long* __restrict__ tile_off, long long* __restrict__ totals) {
  using Scan = cub::BlockScan<long long, kTopThreads>;
  __shared__ typename Scan::TempStorage tmp;
  long long carry_v = 0, carry_f = 0;
  for (int64_t b = 0; b < T; b += (int64_t)kTopThreads * kTopItems) {
    long long v[kTopItems], f[kTopItems];
#pragma unroll
    for (int u = 0; u < kTopItems; ++u) {
      const int64_t t = b + (int64_t)threadIdx.x * kTopItems + u;
      const uint32_t s = t < T ? tile_sum[t] : 0u;
      v[u] = s & 0xffffu;
      f[u] = s >> 16;
    }
    long long av, af;
    Scan(tmp).ExclusiveSum(v, v, av);
    __syncthreads();
    Scan(tmp).ExclusiveSum(f, f, af);
    __syncthreads();
#pragma unroll
    for (int u = 0; u < kTopItems; ++u) {
      const int64_t t = b + (int64_t)threadIdx.x * kTopItems + u;
      if (t < T) {
        tile_off[2 * t] = carry_v + v[u];
        tile_off[2 * t + 1] = carry_f + f[u];
      }
    }
    carry_v += av;
    carry_f += af;
  }
  if (threadIdx.x == 0) {
    totals[0] = carry_v;
    totals[1] = carry_f;
  }
}

// Vertices: per tile, the block scan of the vertex counts gives every point its first vertex id (stored for the face
// pass); vertex (p, d) is p + t (q - p) per coordinate, q = p + d, t = (tau - sigma_p) / (sigma_q - sigma_p), every
// operation rounded on its own (no contraction), so the result is the float32 expression evaluated step by step.
__global__ void __launch_bounds__(kThreads)
k_mesh_verts(Lattice L, const float* __restrict__ axis, const uint16_t* __restrict__ code, const long long* __restrict__ tile_off,
             int* __restrict__ vbase, float* __restrict__ verts) {
  using Scan = cub::BlockScan<int, kThreads>;
  __shared__ typename Scan::TempStorage tmp;
  const int64_t base = (int64_t)blockIdx.x * kTile;
  int carry = (int)tile_off[2 * blockIdx.x];
  for (int it = 0; it < kIters; ++it) {
    if (base + it * kThreads >= L.M) break;             // block-uniform
    const int64_t p = base + it * kThreads + threadIdx.x;
    const uint32_t mask = p < L.M ? (uint32_t)code[p] & 0x7fu : 0u;
    int ex, all;
    Scan(tmp).ExclusiveSum(__popc(mask), ex, all);
    const int vb = carry + ex;
    if (p < L.M) vbase[p] = vb;
    if (mask) {
      int i, j, k;
      L.coords(p, i, j, k);
      const float sa = L.sig(i, j, k);
      const float pa[3] = {__ldg(axis + i), __ldg(axis + j), __ldg(axis + k)};
      int r = 0;
#pragma unroll
      for (int d = 0; d < 7; ++d) {
        if (!((mask >> d) & 1u)) continue;
        const int c = c_dir_code[d];
        const int di = c & 1, dj = (c >> 1) & 1, dk = (c >> 2) & 1;
        const float sb = L.sig(i + di, j + dj, k + dk);
        const float pb[3] = {__ldg(axis + i + di), __ldg(axis + j + dj), __ldg(axis + k + dk)};
        const float t = __fdiv_rn(__fsub_rn(L.tau, sa), __fsub_rn(sb, sa));
        float* out = verts + 3 * (int64_t)(vb + r);
#pragma unroll
        for (int a = 0; a < 3; ++a) out[a] = __fadd_rn(pa[a], __fmul_rn(t, __fsub_rn(pb[a], pa[a])));
        ++r;
      }
    }
    carry += all;
    __syncthreads();
  }
}

// Faces: per tile, the block scan of the triangle counts gives every cell its first face id; the vertex on local edge
// (m, n) of a tetrahedron is (corner m, direction class of corner n - corner m) -> vbase + rank among the set mask bits.
__global__ void __launch_bounds__(kThreads)
k_mesh_faces(Lattice L, const uint16_t* __restrict__ code, const long long* __restrict__ tile_off,
             const int* __restrict__ vbase, int* __restrict__ faces) {
  using Scan = cub::BlockScan<int, kThreads>;
  __shared__ typename Scan::TempStorage tmp;
  const int64_t base = (int64_t)blockIdx.x * kTile;
  int carry = (int)tile_off[2 * blockIdx.x + 1];
  for (int it = 0; it < kIters; ++it) {
    if (base + it * kThreads >= L.M) break;
    const int64_t p = base + it * kThreads + threadIdx.x;
    const uint32_t ntri = p < L.M ? (uint32_t)code[p] >> 8 : 0u;
    int ex, all;
    Scan(tmp).ExclusiveSum((int)ntri, ex, all);
    if (ntri) {
      uint32_t cmask[8];                                // crossing masks of the 8 corners
      uint32_t in8 = 0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint32_t w = code[p + L.corner_delta(c)];
        cmask[c] = w & 0x7fu;
        in8 |= ((w >> 7) & 1u) << c;
      }
      int* out = faces + 3 * (int64_t)(carry + ex);
      for (int q = 0; q < 6; ++q) {
        const int lv[4] = {0, c_tet_v1[q], c_tet_v2[q], 7};
        const uint32_t cs = (in8 & 1u) | (((in8 >> lv[1]) & 1u) << 1) | (((in8 >> lv[2]) & 1u) << 2) | ((in8 >> 7) << 3);
        for (int s = 0; s < c_ntri[cs]; ++s) {
          int v[3];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            const int e = c_tri[cs][s][a];
            const int cm = lv[c_edge_m[e]], cn = lv[c_edge_n[e]];
            const int d = c_dir_of_code[cm ^ cn];
            v[a] = __ldg(vbase + p + L.corner_delta(cm)) + __popc(cmask[cm] & ((1u << d) - 1u));
          }
          if (c_tet_odd[q]) {
            const int w = v[1];
            v[1] = v[2];
            v[2] = w;
          }
          out[0] = v[0];
          out[1] = v[1];
          out[2] = v[2];
          out += 3;
        }
      }
    }
    carry += all;
    __syncthreads();
  }
}

inline size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

struct Layout {
  int64_t M, T;
  size_t code, vbase, tile_sum, tile_off, bytes;
};

inline Layout layout(int R) {
  Layout l;
  const int64_t N = R + 2;
  l.M = N * N * N;
  l.T = (l.M + kTile - 1) / kTile;
  l.code = 0;
  l.vbase = align256(sizeof(uint16_t) * l.M);
  l.tile_sum = l.vbase + align256(sizeof(int) * l.M);
  l.tile_off = l.tile_sum + align256(sizeof(uint32_t) * l.T);
  l.bytes = l.tile_off + sizeof(long long) * 2 * l.T;
  return l;
}

inline Lattice lattice(const float* sigma, int R, float tau) {
  Lattice L;
  L.sigma = sigma;
  L.R = R;
  L.N = R + 2;
  L.M = (int64_t)L.N * L.N * L.N;
  L.tau = tau;
  return L;
}

inline bool good_tau(float tau) { return tau > 0.f && tau <= 3.402823466e38f; }   // > 0, finite

}  // namespace
}  // namespace b2n

using namespace b2n;

extern "C" size_t b2n_mesh_scratch(int R) {
  if (R < 2 || R > kMaxR) return 0;
  return layout(R).bytes;
}

extern "C" int b2n_mesh_count(const float* sigma, int R, float threshold, void* scratch, int64_t* totals,
                              b2n_stream_t stream) {
  B2N_REQUIRE(R >= 2 && R <= kMaxR, "resolution R must be in [2, 1024]");
  B2N_REQUIRE(good_tau(threshold), "threshold must be finite and > 0");
  B2N_REQUIRE(sigma && scratch && totals, "null pointer");
  B2N_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "scratch must be 256-byte aligned");
  const Layout l = layout(R);
  char* s = static_cast<char*>(scratch);
  const Lattice L = lattice(sigma, R, threshold);
  cudaStream_t st = (cudaStream_t)stream;
  k_mesh_count<<<(unsigned)l.T, kThreads, 0, st>>>(L, reinterpret_cast<uint16_t*>(s + l.code),
                                                    reinterpret_cast<uint32_t*>(s + l.tile_sum));
  k_mesh_scan_top<<<1, kTopThreads, 0, st>>>(reinterpret_cast<const uint32_t*>(s + l.tile_sum), l.T,
                                             reinterpret_cast<long long*>(s + l.tile_off),
                                             reinterpret_cast<long long*>(totals));
  return check_launch("b2n_mesh_count");
}

extern "C" int b2n_mesh_emit(const float* sigma, const float* axis_ext, int R, float threshold, void* scratch,
                             int64_t n_verts, int64_t n_faces, float* verts, int32_t* faces, b2n_stream_t stream) {
  B2N_REQUIRE(R >= 2 && R <= kMaxR, "resolution R must be in [2, 1024]");
  B2N_REQUIRE(good_tau(threshold), "threshold must be finite and > 0");
  B2N_REQUIRE(n_verts >= 0 && n_faces >= 0, "negative vertex / face count");
  B2N_REQUIRE(n_verts < (1LL << 31) && n_faces < (1LL << 31),
              "the mesh has 2^31 or more vertices or faces: int32 face indices cannot address it");
  B2N_REQUIRE(n_verts > 0 || n_faces == 0, "faces without vertices");
  if (n_verts == 0) return B2N_OK;
  B2N_REQUIRE(sigma && axis_ext && scratch && verts && (faces || n_faces == 0), "null pointer");
  B2N_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "scratch must be 256-byte aligned");
  const Layout l = layout(R);
  char* s = static_cast<char*>(scratch);
  const Lattice L = lattice(sigma, R, threshold);
  cudaStream_t st = (cudaStream_t)stream;
  const uint16_t* code = reinterpret_cast<const uint16_t*>(s + l.code);
  const long long* tile_off = reinterpret_cast<const long long*>(s + l.tile_off);
  int* vbase = reinterpret_cast<int*>(s + l.vbase);
  k_mesh_verts<<<(unsigned)l.T, kThreads, 0, st>>>(L, axis_ext, code, tile_off, vbase, verts);
  if (n_faces > 0) k_mesh_faces<<<(unsigned)l.T, kThreads, 0, st>>>(L, code, tile_off, vbase, faces);
  return check_launch("b2n_mesh_emit");
}
