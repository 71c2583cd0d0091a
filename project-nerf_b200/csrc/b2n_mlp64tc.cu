// Forward of the fused 64-wide Instant decoder on tcgen05: InstantNeRFDecoder.forward (src/decoders.py:136-162; network
// and arithmetic in b2n_mlp64.cu's header -- fp16 operands, fp32 accumulation, sigma_net's first layer as a split hi/lo
// product) with the layer products on the 5th-generation tensor cores.
//
// Why: an earlier mma.sync forward kept activations in registers (C fragments re-packed as A fragments) and paid ~1500
// warp instructions per 32 points for fragment bookkeeping; at 255 registers it ran 8 warps per SM and was latency-bound
// (tensor pipe 40 %, IPC 0.29 per scheduler: profiles/r2a_kernels.md).  Here a CTA owns a 128-point tile = the 128 TMEM
// lanes: thread t owns point t.  Per layer ONE elected thread issues the K/16 tcgen05.mma (A = the activation tile in shared
// memory, K-major SWIZZLE_128B; B = the layer's weight tile, staged once per CTA; D = 128 x N fp32 in TMEM), commits to an
// mbarrier, and every thread then drains ITS accumulator row with tcgen05.ld, applies the activation, and writes the row
// back as the next layer's A operand -- in place: the MMA is done with the tile when the barrier fires.
//
// One layer step is a latency chain (issue -> MMA -> commit -> mbarrier -> tcgen05.ld -> pack -> st.shared ->
// fence.proxy.async -> bar.sync, ~1800 cycles measured with one CTA per SM), so throughput comes from co-resident CTAs:
// 52 KB of shared memory at pos_dim <= 32 (x_hi and x_lo share ONE 64-column tile) -> 4 CTAs per SM, 68 KB above -> 3.
// Measured, 4.2 M points (tools/kbench.py mlp64): 0.42 ms against 0.62 ms for that mma.sync kernel (pos_dim 32), 0.66
// against 0.86 ms (pos_dim 53); 1 / 2 / 3 / 4 CTAs per SM: 1.05 / 0.66 / 0.50 / 0.42 ms.
// cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for this kernel; the grid is sized from shared memory instead.
#define B2N_OP_F16
#include "b2n_mlp64.cuh"
#include "b2n_tc.cuh"

namespace b2n {
namespace itc {

constexpr int TILE = 128;                 // points per tile
constexpr int THREADS = 128;
constexpr uint32_t A_BYTES = 16384;       // [128 rows x 64 fp16] K-major, 128-byte rows, SWIZZLE_128B
constexpr uint32_t W64_BYTES = 8192;      // [64 x 64]
constexpr uint32_t W16_BYTES = 2048;      // [16 x 64]
// shared-memory map.  POS_K == 32: ONE activation tile -- x_hi in columns 0..31 and x_lo in columns 32..63 of the same
// 64-wide rows (the first layer multiplies it by [W1_hi | W1_hi] and by [W1_lo | 0]); POS_K == 64: x_lo has its own tile.
template <int POS_K, int NS>
struct Map {
  static constexpr uint32_t SLOT = POS_K == 64 ? 2 * A_BYTES : A_BYTES;      // activation tile(s) of one in-flight point tile
  static constexpr uint32_t A0 = 0;                          // x_hi (| x_lo) -> h1 -> c -> c1 -> c2 (in place)
  static constexpr uint32_t A1 = A0 + A_BYTES;               // x_lo (POS_K == 64 only)
  static constexpr uint32_t W1H = NS * SLOT;
  static constexpr uint32_t W1L = W1H + W64_BYTES;
  static constexpr uint32_t W2 = W1L + W64_BYTES;
  static constexpr uint32_t V1 = W2 + W16_BYTES;
  static constexpr uint32_t V2 = V1 + W64_BYTES;
  static constexpr uint32_t V3 = V2 + W64_BYTES;
  static constexpr uint32_t BAR = V3 + W16_BYTES;
  static constexpr uint32_t BYTES = BAR + 64 + 1024;         // + slack for the 1024-byte alignment of the base
};

using namespace b2n::tc;

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ float4 ldg_stream(const float* p) {      // read-once rows: non-coherent path, no L1 allocation
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// fp32 matrix [rows_valid][src_cols] (row stride src_cols) -> fp16 K-major SWIZZLE_128B tile [rows][64]; lo = the low half of the
// hi/lo split (w - fp16(w)); columns >= src_cols and rows >= rows_valid are zero
// dup32: columns 32..63 repeat columns 0..31 (the [W | W] operand of the merged x_hi | x_lo tile)
__device__ __forceinline__ void stage_weight(const float* __restrict__ W, int rows_valid, int src_cols, int rows,
                                             unsigned char* dst, bool lo, bool dup32 = false) {
  for (int i = threadIdx.x; i < rows * 8; i += blockDim.x) {
    const int r = i >> 3, c = i & 7;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int k = 8 * c + j;
      if (dup32) k &= 31;
      float w = (r < rows_valid && k < src_cols) ? __ldg(W + (size_t)r * src_cols + k) : 0.f;
      if (lo) w = w - __half2float(__float2half_rn(w));
      f[j] = w;
    }
    *reinterpret_cast<uint4*>(dst + swz(r, c)) = make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
}

// drain 16 * NCH accumulator columns of this thread's TMEM lane (all loads in flight, one wait), ReLU, pack to fp16 and write
// them as chunks c0.. of row r of the tile at shared address `tile`
template <int NCH, bool RELU>
__device__ __forceinline__ void drain_to_tile(uint32_t tmem_row, uint32_t tile, int r, int c0) {
  uint32_t v[NCH][16];
#pragma unroll
  for (int h = 0; h < NCH; ++h) tc_ld16(tmem_row + 16 * h, v[h]);
  tc_ld_wait();
#pragma unroll
  for (int h = 0; h < NCH; ++h) {
    uint32_t p[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      p[j] = pack2(__uint_as_float(v[h][2 * j]), __uint_as_float(v[h][2 * j + 1]));
      if (RELU) {              // on the packed pair: one HMNMX2 for two values (rounding is monotone, 0 exact)
        const __half2 r = __hmax2(*reinterpret_cast<__half2*>(&p[j]), __floats2half2_rn(0.f, 0.f));
        p[j] = *reinterpret_cast<const uint32_t*>(&r);
      }
    }
    sts128(tile + swz(r, c0 + 2 * h), p[0], p[1], p[2], p[3]);
    sts128(tile + swz(r, c0 + 2 * h + 1), p[4], p[5], p[6], p[7]);
  }
}

// POS_K: 32 or 64, the padded width of the sigma-net input held in the x tiles.  NS: point tiles a CTA keeps in flight -- with
// two, the CTA works on tile B's epilogue while the tensor core runs tile A's next layer (and vice versa): the MMA, its commit
// and the barrier wake-up leave the critical path.  NS = 2 costs one more activation tile (16 KB) and 32 prefetch registers
// (68 KB -> 3 CTAs = 6 tiles per SM instead of 4).  Measured after the instruction-count work (4.2 M points): 0.351 ms against
// 0.345 ms for NS = 1 with four CTAs per SM -- with four co-resident tiles the kernel is no longer waiting for its MMAs but
// bound by TMEM drain + packing + stores, so NS = 1 stays the default and NS = 2 an A/B variant (b2n_debug_instant_fwd_slots).
template <int POS_K, int NS>
__global__ void __launch_bounds__(THREADS, POS_K == 32 ? (NS == 1 ? 4 : 3) : 3)
k_instant_fwd_tc(const float* __restrict__ x, int ldx, int pos_dim, const float* __restrict__ dirs,
                 const float* __restrict__ bands, int L_dir, const float* __restrict__ sp, const float* __restrict__ cp,
                 int64_t P, float* __restrict__ rgb, float* __restrict__ sigma, const int* __restrict__ rows,
                 float in_pad_value, int* __restrict__ err) {
  P = clamp_rows(P, rows);
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  using M = Map<POS_K, NS>;
  constexpr bool MERGED = POS_K == 32;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + M::BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + NS);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int in_pad = (pos_dim + 15) & ~15;
  constexpr int KS1 = POS_K / 16;
  // ---- one-time set-up: weights as B operands, barriers, TMEM
  stage_weight(sp, 64, in_pad, 64, smem + M::W1H, false, MERGED);
  stage_weight(sp, 64, in_pad, 64, smem + M::W1L, true);
  stage_weight(sp + 64 * in_pad, 16, 64, 16, smem + M::W2, false);
  if (cp) {
    stage_weight(cp, 64, 48, 64, smem + M::V1, false);
    stage_weight(cp + 64 * 48, 64, 64, 64, smem + M::V2, false);
    stage_weight(cp + 64 * 48 + 64 * 64, 16, 64, 16, smem + M::V3, false);
  }
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) mbar_init(s32(bars + s), 1);
    mbar_init_fence();
  }
  if (warp == 0) tmem_alloc(s32(tmem_slot), 64 * NS);
  proxy_fence();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_row = tmem + ((uint32_t)(32 * warp) << 16);          // this thread's lane group
  const uint32_t a_base = s32(smem + M::A0), bar0 = s32(bars);
  const uint32_t w1h = s32(smem + M::W1H), w1l = s32(smem + M::W1L), w2 = s32(smem + M::W2);
  const uint32_t v1 = s32(smem + M::V1), v2 = s32(smem + M::V2), v3 = s32(smem + M::V3);
  const bool vec = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  uint32_t phase = 0;
  bool ok = true;

  const int64_t n_tiles = (P + TILE - 1) / TILE;
  const int64_t n_units = (n_tiles + NS - 1) / NS;
  // coalesced: consecutive threads read consecutive 16 bytes of a row
  constexpr int Q = POS_K / 4;
  float4 xr[NS][Q];
  const bool full_rows = vec && pos_dim == POS_K;       // every 16-byte piece of a row is a plain vector load
  auto load_rows = [&](int64_t t, float4 (&dst)[Q]) {
    if (full_rows && (t + 1) * TILE <= P) {              // interior tile: no per-element predicates
      const float* base = x + t * TILE * (int64_t)ldx;
#pragma unroll
      for (int it = 0; it < Q; ++it) {
        const int idx = it * THREADS + tid;
        dst[it] = ldg_stream(base + (int64_t)(idx / Q) * ldx + 4 * (idx % Q));
      }
      return;
    }
#pragma unroll
    for (int it = 0; it < Q; ++it) {
      const int idx = it * THREADS + tid;
      const int r = idx / Q, q = idx % Q;
      const int64_t pr = t * TILE + r;
      float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pr < P) {
        const float* src = x + pr * ldx + 4 * q;
        if (vec && 4 * q + 3 < pos_dim) {
          f = ldg_stream(src);
        } else {
          float e[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int k = 4 * q + j;
            e[j] = k < pos_dim ? __ldg(src + j) : (k < in_pad ? in_pad_value : 0.f);
          }
          f = make_float4(e[0], e[1], e[2], e[3]);
        }
      }
      dst[it] = f;
    }
  };
  // one elected thread issues a layer of slot s and commits to the slot's barrier
  auto issue = [&](int layer, int s) {
    const uint32_t a0 = a_base + s * M::SLOT, a1 = a0 + A_BYTES, acc = tmem + 64 * s;
    tc_fence_after();
    if (layer == 0) {            // sigma_net layer 1: split product, small terms first
      const uint32_t id = umma_idesc(Fmt::F16, Major::K, 64, 128);
      // x_lo W_hi: the merged tile holds x_lo in its upper 32 columns, facing the second copy of W_hi
#pragma unroll
      for (int k = 0; k < KS1; ++k)
        tc_mma(acc, umma_desc(MERGED ? a0 : a1) + 2 * (MERGED ? k + KS1 : k), umma_desc(w1h) + 2 * (MERGED ? k + KS1 : k), id, k > 0);
#pragma unroll
      for (int k = 0; k < KS1; ++k) tc_mma(acc, umma_desc(a0) + 2 * k, umma_desc(w1l) + 2 * k, id, 1u);
#pragma unroll
      for (int k = 0; k < KS1; ++k) tc_mma(acc, umma_desc(a0) + 2 * k, umma_desc(w1h) + 2 * k, id, 1u);
    } else {
      // 1: sigma_net layer 2 (64 -> 16)   2: color_net layer 1 (48 -> 64)   3: color_net layer 2   4: output layer (64 -> 3 of 16)
      const uint32_t w = layer == 1 ? w2 : (layer == 2 ? v1 : (layer == 3 ? v2 : v3));
      const uint32_t id = umma_idesc(Fmt::F16, Major::K, (layer == 1 || layer == 4) ? 16 : 64, 128);
      const int ks = layer == 2 ? 3 : 4;
      for (int k = 0; k < ks; ++k) tc_mma(acc, umma_desc(a0) + 2 * k, umma_desc(w) + 2 * k, id, k > 0);
    }
    tc_commit(bar0 + 8 * s);
  };

#pragma unroll
  for (int s = 0; s < NS; ++s) load_rows((int64_t)blockIdx.x * NS + s, xr[s]);
  for (int64_t unit = blockIdx.x; unit < n_units && ok; unit += gridDim.x) {
    float d[NS][3];
    // ---- input rows (fetched one unit ahead) -> x_hi / x_lo; only the POS_K columns the first layer reads
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const uint32_t a0 = a_base + s * M::SLOT, a1 = a0 + A_BYTES;
      const int64_t p = (unit * NS + s) * TILE + tid;
      // this point's view direction: needed after two layer steps -- loaded now, not a tile ahead (a prefetched value that
      // gets spilled makes the spill store wait for the load: 5 % of the stall samples, ncu)
      d[s][0] = d[s][1] = d[s][2] = 0.f;
      if (dirs && p < P) d[s][0] = __ldg(dirs + 3 * p), d[s][1] = __ldg(dirs + 3 * p + 1), d[s][2] = __ldg(dirs + 3 * p + 2);
#pragma unroll
      for (int it = 0; it < Q; ++it) {
        const int idx = it * THREADS + tid;
        const int r = idx / Q, q = idx % Q;
        const float4 f = xr[s][it];
        const uint32_t h0 = pack2(f.x, f.y), h1 = pack2(f.z, f.w);
        const float2 b0 = unpack2(h0), b1 = unpack2(h1);
        const uint32_t l0 = pack2(f.x - b0.x, f.y - b0.y), l1 = pack2(f.z - b1.x, f.w - b1.y);
        sts64(a0 + swz(r, q >> 1) + 8 * (q & 1), h0, h1);
        if (MERGED) sts64(a0 + swz(r, 4 + (q >> 1)) + 8 * (q & 1), l0, l1);
        else sts64(a1 + swz(r, q >> 1) + 8 * (q & 1), l0, l1);
      }
      load_rows((unit + gridDim.x) * NS + s, xr[s]);            // lands during the layer phases below
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
#pragma unroll
      for (int s = 0; s < NS; ++s) issue(0, s);
    }
    // ---- h1 = relu(layer 1) over x_hi; then layer 2
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      ok = ok && mbar_wait(bar0 + 8 * s, phase, err);
      tc_fence_after();
      drain_to_tile<4, true>(tmem_row + 64 * s, a_base + s * M::SLOT, tid, 0);
      proxy_fence();
      tc_fence_before();
      __syncthreads();
      if (tid == 0) issue(1, s);
    }
    phase ^= 1;
    // ---- h (16): density head; colour-net input = [h | direction features]
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const uint32_t a0 = a_base + s * M::SLOT;
      const int64_t p = (unit * NS + s) * TILE + tid;
      ok = ok && mbar_wait(bar0 + 8 * s, phase, err);
      tc_fence_after();
      uint32_t v[16];
      tc_ld16(tmem_row + 64 * s, v);
      tc_ld_wait();
      if (p < P) __stcs(sigma + p, softplus_m5(__uint_as_float(v[0])));
      if (rgb) {
        uint32_t q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) q[j] = pack2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        sts128(a0 + swz(tid, 0), q[0], q[1], q[2], q[3]);
        sts128(a0 + swz(tid, 1), q[4], q[5], q[6], q[7]);
        uint4 df[4];             // all four chunks first, then the stores (storing each chunk as it is packed reschedules NS = 2)
        dir_features(d[s], bands, L_dir, in_pad_value, [&](int i, uint4 v) { df[i] = v; });
#pragma unroll
        for (int i = 0; i < 4; ++i) sts128(a0 + swz(tid, 2 + i), df[i].x, df[i].y, df[i].z, df[i].w);      // layer 1 of color_net reads K = 48 only
        proxy_fence();
      }
      tc_fence_before();
      __syncthreads();
      if (rgb && tid == 0) issue(2, s);
    }
    phase ^= 1;
    if (!rgb) continue;           // density sweep: the colour network is skipped
    // ---- color_net hidden layers
#pragma unroll
    for (int layer = 3; layer <= 4; ++layer) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        ok = ok && mbar_wait(bar0 + 8 * s, phase, err);
        tc_fence_after();
        drain_to_tile<4, true>(tmem_row + 64 * s, a_base + s * M::SLOT, tid, 0);
        proxy_fence();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) issue(layer, s);
      }
      phase ^= 1;
    }
    // ---- output layer + sigmoid
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const int64_t p = (unit * NS + s) * TILE + tid;
      ok = ok && mbar_wait(bar0 + 8 * s, phase, err);
      tc_fence_after();
      uint32_t v[16];
      tc_ld16(tmem_row + 64 * s, v);
      tc_ld_wait();
      if (p < P) {
        rgb[3 * p] = sigmoidf(__uint_as_float(v[0]));
        rgb[3 * p + 1] = sigmoidf(__uint_as_float(v[1]));
        rgb[3 * p + 2] = sigmoidf(__uint_as_float(v[2]));
      }
    }
    phase ^= 1;
    tc_fence_before();
    __syncthreads();              // the accumulators are free for the next unit
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64 * NS);
}

}  // namespace itc
}  // namespace b2n

using namespace b2n;

// point tiles in flight per CTA of k_instant_fwd_tc at pos_dim <= 32 (b2n_debug_instant_fwd_slots): see the kernel
static int g_fwd_slots = 1;
extern "C" int b2n_debug_instant_fwd_slots(int slots) {
  const int prev = g_fwd_slots;
  if (slots == 1 || slots == 2) g_fwd_slots = slots;
  return prev;
}

// rgb == NULL: density only -- dirs / dir_bands / color_params are not read and may be NULL; err_flag: device int, set
// non-zero if a stalled barrier aborted a tile.
extern "C" int b2n_instant_mlp_fwd_tc(const float* x_enc, int ldx, int pos_dim, const float* dirs, const float* dir_bands,
                                      int L_dir, const float* sigma_params, const float* color_params, int64_t P,
                                      float* rgb, float* sigma, float in_pad_value, int* err_flag, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(pos_dim > 0 && pos_dim <= 64 && ldx >= pos_dim, "pos_dim must be in [1, 64]");
  B2N_REQUIRE(L_dir >= 0 && L_dir <= 4, "direction encoding must have at most 4 bands (27 features)");
  B2N_REQUIRE(x_enc && sigma_params && sigma && err_flag, "null pointer");
  B2N_REQUIRE(!rgb || (dirs && color_params && (L_dir == 0 || dir_bands)), "null pointer");
  if (!rgb) dirs = nullptr, dir_bands = nullptr, L_dir = 0, color_params = nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tiles = (P + itc::TILE - 1) / itc::TILE;
  auto launch = [&](auto kern, uint32_t smem_bytes, int ns) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    // CTAs per SM by shared memory (227 KB, 1 KB reserved per CTA); cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1
    // for this kernel although the hardware co-schedules 3-4 (measured: 1.05 -> 0.49 ms with three per SM); registers
    // (<= 168 x 128) and TMEM (64 * ns of 512 columns) allow more than shared memory does
    int per_sm = (int)(232448u / (smem_bytes + 1024u));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8 / ns) per_sm = 8 / ns;        // 512 TMEM columns per SM
    const int64_t units = (tiles + ns - 1) / ns;
    int64_t grid = (int64_t)kSMs * per_sm;
    if (grid > units) grid = units;
    kern<<<(unsigned)grid, itc::THREADS, smem_bytes, st>>>(x_enc, ldx, pos_dim, dirs, dir_bands, L_dir, sigma_params,
                                                          color_params, P, rgb, sigma, g_active_rows, in_pad_value,
                                                          err_flag);
  };
  if (pos_dim <= 32 && g_fwd_slots == 2) launch(itc::k_instant_fwd_tc<32, 2>, itc::Map<32, 2>::BYTES, 2);
  else if (pos_dim <= 32) launch(itc::k_instant_fwd_tc<32, 1>, itc::Map<32, 1>::BYTES, 1);
  else launch(itc::k_instant_fwd_tc<64, 1>, itc::Map<64, 1>::BYTES, 1);
  return check_launch("b2n_instant_mlp_fwd_tc");
}
