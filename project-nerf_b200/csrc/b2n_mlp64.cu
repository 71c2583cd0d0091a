// Backward of the fused 64-wide decoder of the hash-grid configs: InstantNeRFDecoder.forward (src/decoders.py:136-162),
// i.e. the two tinycudann FullyFusedMLPs of the reference plus the direction Fourier features (src/embeddings.py:22-32 on
// view dirs), the softplus(h0-5) density head, the concat and the sigmoid.  The forward is k_instant_fwd_tc
// (b2n_mlp64tc.cu); the arithmetic both must compute identically is in b2n_mlp64.cuh.
//
//   sigma_net : x[pos] -> 64 (ReLU) -> 16            (no biases, widths padded to 16)
//   sigma     = softplus(h[0] - 5)
//   color_net : cat[h(16), gamma(d)(27 -> 32)] -> 64 (ReLU) -> 64 (ReLU) -> 3 (sigmoid)
//
// Arithmetic: IEEE fp16 operands (what the reference's tinycudann FullyFusedMLP uses), fp32 accumulation on the tensor
// cores.  Two departures from plain fp16, both measured on the CPU error budget
// (tools/bf16_error_budget.py) as what decides the distance of the parameter gradients from an fp32 evaluation:
//   * sigma_net's FIRST layer -- the product with the hash-grid features, whose pre-activations decide 64 ReLU masks and
//     the density -- is a split product x_hi W_hi + x_lo W_hi + x_hi W_lo (x = x_hi + x_lo in fp16): ~21 significant bits;
//   * the gradient chain runs on S * dL/dy with S a power of two that puts the largest incoming gradient at 2^7..2^8
//     (found by a one-pass |.|-max reduction, k_grad_absmax), so fp16's narrow exponent range never clips it; outputs are
//     divided by S.
#define B2N_OP_F16
#include "b2n_mlp64.cuh"
#include "b2n_tc.cuh"

namespace b2n {

constexpr int HID = 64;      // hidden width
constexpr int GEO = 16;      // sigma_net output width
constexpr int CIN = 48;      // color_net padded input width (16 + 27 -> 48)
constexpr int MLP_THREADS = 128;

// view direction of point p (zeros beyond P): loaded long before dir_features needs it (ncu showed long-scoreboard stalls
// on the small per-tile loads as the top stall reason of the decoder kernels)
__device__ __forceinline__ void load_dir(const float* __restrict__ dirs, int64_t p, int64_t P, float (&d)[3]) {
  d[0] = d[1] = d[2] = 0.f;
  if (dirs && p < P) d[0] = __ldg(dirs + 3 * p), d[1] = __ldg(dirs + 3 * p + 1), d[2] = __ldg(dirs + 3 * p + 2);
}
// A-fragment elements of 16 rows of x_enc [P, pos_dim] as fp32 pairs (`pad` in the input padding, zero beyond it and
// beyond P), for software pipelining: issue the loads now, split into hi / lo (and stall) later
template <int KT>
__device__ __forceinline__ void load_x_raw(const float* __restrict__ x, int ldx, int pos_dim, int64_t p0, int64_t P,
                                           float2 (&raw)[KT][4], int lane, float pad = 0.f) {
  const int g = lane >> 2, t = lane & 3;
  const int in_pad = (pos_dim + 15) & ~15;      // columns [pos_dim, in_pad) are sigma_net's input padding: value `pad`
  const bool vec = ((ldx & 1) == 0) && ((reinterpret_cast<uintptr_t>(x) & 7) == 0);
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int64_t p = p0 + g + 8 * r;
        const int c = 16 * k + 8 * h + 2 * t;
        float2 v = make_float2(0.f, 0.f);
        if (p < P) {
          const float* src = x + p * ldx + c;
          if (vec && c + 1 < pos_dim) {
            v = __ldcs(reinterpret_cast<const float2*>(src));
          } else {
            if (c < pos_dim) v.x = __ldcs(src);
            else if (c < in_pad) v.x = pad;
            if (c + 1 < pos_dim) v.y = __ldcs(src + 1);
            else if (c + 1 < in_pad) v.y = pad;
          }
        }
        raw[k][2 * h + r] = v;
      }
}
// interior tiles of a full-width, 8-byte aligned input: the same loads without the per-element predicates
template <int KT>
__device__ __forceinline__ void load_x_raw_full(const float* __restrict__ x, int ldx, int64_t p0, float2 (&raw)[KT][4], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float* r0 = x + (p0 + g) * ldx + 2 * t;
  const float* r1 = r0 + 8 * (int64_t)ldx;
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      raw[k][2 * h] = __ldcs(reinterpret_cast<const float2*>(r0 + 16 * k + 8 * h));
      raw[k][2 * h + 1] = __ldcs(reinterpret_cast<const float2*>(r1 + 16 * k + 8 * h));
    }
}
// x = hi + lo with hi = fp16(x), lo = fp16(x - hi): the operands of the split first-layer product
__device__ __forceinline__ void pack_hl(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  hi = pack2(v0, v1);
  const float2 h = unpack2(hi);
  lo = pack2(v0 - h.x, v1 - h.y);
}
template <int KT>
__device__ __forceinline__ void pack_x_hl(const float2 (&raw)[KT][4], uint32_t (&hi)[KT][4], uint32_t (&lo)[KT][4]) {
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int i = 0; i < 4; ++i) pack_hl(raw[k][i].x, raw[k][i].y, hi[k][i], lo[k][i]);
}

struct MlpSmem {
  // offsets (in bf16 elements) of the weight matrices inside dynamic shared memory
  int w1, w2, v1, v2, v3, w1lo, end;
};
template <int POS_K>
__host__ __device__ constexpr MlpSmem weight_layout() {
  MlpSmem m{};
  m.w1 = 0;
  m.w2 = m.w1 + HID * (POS_K + PAD);
  m.v1 = m.w2 + GEO * (HID + PAD);
  m.v2 = m.v1 + HID * (CIN + PAD);
  m.v3 = m.v2 + HID * (HID + PAD);
  m.w1lo = m.v3 + 16 * (HID + PAD);            // low half of the split first-layer weights
  m.end = m.w1lo + HID * (POS_K + PAD);
  return m;
}

// in_pad = pad16(pos_dim): the stored width of sigma_net's first matrix (16, 32, 48 or 64 <= POS_K)
template <int POS_K>
__device__ __forceinline__ void load_all_weights(const float* __restrict__ sp, const float* __restrict__ cp, int in_pad,
                                                 op16* sm) {
  constexpr MlpSmem L = weight_layout<POS_K>();
  load_weights(sp, HID, POS_K, in_pad, sm + L.w1);
  {   // W1_lo = fp16(W1 - fp16(W1))
    constexpr int S = POS_K + PAD;
    for (int i = threadIdx.x; i < HID * POS_K; i += blockDim.x) {
      const int r = i / POS_K, c = i - r * POS_K;
      const float w = c < in_pad ? __ldg(sp + (size_t)r * in_pad + c) : 0.f;
      sm[L.w1lo + r * S + c] = to_op16(w - from_op16(to_op16(w)));
    }
  }
  load_weights(sp + HID * in_pad, GEO, HID, HID, sm + L.w2);
  if (!cp) return;                       // density only: no colour network
  load_weights(cp, HID, CIN, CIN, sm + L.v1);
  load_weights(cp + HID * CIN, HID, HID, HID, sm + L.v2);
  load_weights(cp + HID * CIN + HID * HID, 16, HID, HID, sm + L.v3);
}

// max |g| over the incoming gradients as float bits (non-negative floats order like unsigned integers; a NaN has the
// largest bit pattern, so a non-finite gradient anywhere is visible in the result)
__global__ void __launch_bounds__(256) k_grad_absmax(const float* __restrict__ a, const float* __restrict__ b, int64_t P,
                                                     unsigned int* __restrict__ out, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  const int64_t na = 3 * P, nb = P;              // a = g_rgb [P,3], b = g_sigma [P]
  unsigned int m = 0u;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
  auto scan = [&](const float* __restrict__ v, int64_t n) {
    // 16-byte loads over the aligned body (the first version read 4 bytes per thread per step: 2.3 TB/s), scalars at the ends
    const int64_t head = min(n, (int64_t)((16 - (reinterpret_cast<uintptr_t>(v) & 15)) & 15) >> 2);
    const int64_t n4 = (n - head) >> 2;
    const float4* v4 = reinterpret_cast<const float4*>(v + head);
    for (int64_t i = t0; i < n4; i += nt) {
      const float4 q = __ldcs(v4 + i);
      m = max(max(m, __float_as_uint(q.x) & 0x7fffffffu), __float_as_uint(q.y) & 0x7fffffffu);
      m = max(max(m, __float_as_uint(q.z) & 0x7fffffffu), __float_as_uint(q.w) & 0x7fffffffu);
    }
    for (int64_t i = t0; i < head; i += nt) m = max(m, __float_as_uint(__ldg(v + i)) & 0x7fffffffu);
    for (int64_t i = head + 4 * n4 + t0; i < n; i += nt) m = max(m, __float_as_uint(__ldg(v + i)) & 0x7fffffffu);
  };
  scan(a, na);
  scan(b, nb);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// power-of-two gradient scale S from the |.|-max bits: S * max in [2^7, 2^8); 1 for an all-zero gradient; NaN when the
// incoming gradient holds an inf / NaN (GradScaler overflow step: every output must be non-finite too, never a clamped
// finite value that would be applied as a step)
__device__ __forceinline__ float grad_scale_from(unsigned int bits) {
  if (bits == 0u) return 1.f;
  if (bits >= 0x7f800000u) return __uint_as_float(0x7fc00000u);
  int e = (int)(bits >> 23) - 127;                      // max in [2^e, 2^(e+1))   (subnormal max: e = -127)
  int se = 7 - e;                                       // S = 2^se
  se = se > 120 ? 120 : (se < -120 ? -120 : se);
  return __uint_as_float((unsigned int)(se + 127) << 23);
}

// ------------------------------------------------------------------------------ backward, weight gradients on tcgen05
// A warp owns 16 points of a 64-point tile.  It recomputes the forward (split first layer) and runs the data-gradient
// chain on mma.sync: activations and gradients as fragments in registers, weights in padded shared-memory rows read with
// ldmatrix / ldmatrix.trans.  Every layer input and pre-activation gradient is staged in shared memory, and the five
// weight gradients dW = dZ^T In -- a third of the kernel's tensor work, the part that would need BOTH operands from
// shared memory through ldmatrix.trans, and 88 accumulator registers per thread -- go to the 5th-generation tensor cores:
// the staged tiles are written in the SWIZZLE_128B layout (64 points x 128 B, 16-byte chunk c of row r at c ^ (r & 7)),
// which read with the point as the contraction index is exactly tcgen05's MN-major operand form (b2n_wgrad256.cu), and
// per tile 12 MMAs (M = 128, K = 16 points each) accumulate into fp32 accumulators that live in TMEM for the whole
// persistent loop.  The MMAs run asynchronously under the next tile's first layer.
//
// pos_dim <= 32 (MERGED map, 8 slots of 8 KB; x, dz5 and dz2 share one 64-column tile X = [x | dz5 | dz2]):
//   0 dz3 | 1 dz4 | 2 c | 3 c1 | 4 dz1 | 5 h1 | 6 c2 | 7 X
//   D1 [128 x 128] = [dz3; dz4]^T [c | c1] -> rows 0..63 x cols 0..47 = dV1,       rows 64..127 x cols 64..127 = dV2
//   D2 [128 x 64]  = [c2; X]^T    X        -> rows 0..63 x cols 32..34 = dV3^T
//   D3 [128 x 64]  = [dz1; h1]^T  X        -> rows 0..63 x cols 0..in_pad-1 = dW1, rows 64..127 x cols 48..63 = dW2^T
// wider inputs (9 slots):
//   0 dz3 | 1 dz4 | 2 c | 3 c1 | 4 c2 | 5 h1 | 6 dz5 (cols 0..15), dz2 (cols 16..31) | 7 dz1 | 8 x
//   D1 as above;  D2 = [c2; h1]^T [dz5, dz2] -> rows 0..63 x cols 0..2 = dV3^T, rows 64..127 x cols 16..31 = dW2^T;
//   D3 = [dz1; x]^T [x] -> rows 0..63 x cols 0..in_pad-1 = dW1
// (the off-diagonal blocks are by-products nobody reads; an M = 64 MMA costs the same tensor time as M = 128).
//
// GROUPS == 1: a CTA is one 4-warp group (two CTAs per SM: 8 warps); its thread 0 issues the MMAs after a __syncthreads.
// GROUPS == 3 (pos_dim <= 32): ONE CTA per SM holds three 4-warp groups, each with its own tile slots and 168 registers
// per thread -- 12 warps per SM for the latency-bound mma.sync chain -- that share the weights and ONE set of TMEM
// accumulators; one thread of a fourth warpgroup (which hands its registers to the workers: setmaxnreg) is the only MMA
// issuer (tcgen05.mma is ordered per issuing thread: one issuer keeps the read-modify-write of the shared accumulators
// in order).  A group hands a staged tile over through an mbarrier
// (128 arrivals) and gets it back through the issuer's tcgen05.commit.
namespace bwtc {
constexpr int SLOT = 8192;
constexpr int D1 = 0, D2 = 128, D3 = 192, TMEM_COLS = 256;
template <int POS_K>
struct Slots {
  static constexpr bool MERGED = POS_K == 32;
  static constexpr int N = MERGED ? 8 : 9;
  static constexpr int DZ3 = 0, DZ4 = 1, C = 2, C1 = 3;
  static constexpr int DZ1 = MERGED ? 4 : 7, H1 = 5, C2 = MERGED ? 6 : 4, X = MERGED ? 7 : 8;
  static constexpr int DZ25 = MERGED ? 7 : 6;            // tile holding dz5 / dz2 ...
  static constexpr int COL_DZ5 = MERGED ? 32 : 0;        // ... and their first columns
  static constexpr int COL_DZ2 = MERGED ? 48 : 16;
  static constexpr int A2 = C2;                          // A operand of D2: [c2; next slot]
  static constexpr int B2 = DZ25;
  static constexpr int A3 = DZ1;                         // A operand of D3: [dz1; next slot]
  static constexpr int B3 = X;
};
// element offset of (row, col) inside a 64 x 64 swizzled tile
__device__ __forceinline__ int sw(int r, int c) { return r * 64 + ((((c >> 3) ^ r) & 7) << 3) + (c & 7); }
// A fragments of a 16-row slab -> swizzled tile: one stmatrix per 16 x 16 block (the four 8 x 8 matrices of an A fragment
// are rows g / g+8 x columns 0..7 / 8..15; lane i supplies the address of row i % 8 of matrix i / 8)
template <int KT>
__device__ __forceinline__ void store_a_sw(const uint32_t (&a)[KT][4], op16* tile, int row0, int col0, int lane) {
  const int r = row0 + (lane & 7) + 8 * ((lane >> 3) & 1);
  const int cb = col0 + 8 * (lane >> 4);
#pragma unroll
  for (int k = 0; k < KT; ++k)
    asm volatile("stmatrix.sync.aligned.m8n8.x4.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(tile + sw(r, cb + 16 * k))),
                 "r"(a[k][0]), "r"(a[k][1]), "r"(a[k][2]), "r"(a[k][3]) : "memory");
}
template <int POS_K, int GROUPS>
constexpr size_t smem_bytes() {
  return (size_t)GROUPS * Slots<POS_K>::N * SLOT + (size_t)weight_layout<POS_K>().end * sizeof(op16) + 128;
}
template <int GROUPS>
constexpr int threads() { return GROUPS == 1 ? MLP_THREADS : (GROUPS + 1) * MLP_THREADS; }
}  // namespace bwtc

// ReLU gate of a packed gradient fragment by the packed ACTIVATION fragment of the same layer (forward A fragments and
// c_to_a outputs share one (row, column) layout): 2 instructions per 2 elements, no shared-memory re-read
template <int KT>
__device__ __forceinline__ void relu_gate(uint32_t (&dz)[KT][4], const uint32_t (&act)[KT][4]) {
  const __half2 zero = __floats2half2_rn(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int i = 0; i < 4; ++i) dz[k][i] &= __hgt2_mask(*reinterpret_cast<const __half2*>(&act[k][i]), zero);
}

template <int POS_K, int GROUPS>
__global__ void __launch_bounds__(bwtc::threads<GROUPS>(), GROUPS == 1 ? 2 : 1)
k_instant_bwd_tc(const float* __restrict__ x, int ldx, int pos_dim, const float* __restrict__ dirs,
                 const float* __restrict__ bands, int L_dir, const float* __restrict__ sp, const float* __restrict__ cp,
                 int64_t P, const float* __restrict__ g_rgb, const float* __restrict__ g_sigma, float* __restrict__ g_x,
                 int ldg, float* __restrict__ g_sp, float* __restrict__ g_cp, const unsigned int* __restrict__ absmax,
                 const int* __restrict__ rows, float in_pad_value, int* __restrict__ err) {
  using namespace bwtc;
  using namespace tc;
  using SL = Slots<POS_K>;
  // the ReLU gates of the gradient chain use the forward's A fragments, kept live in registers (HSET2 + LOP3 per pair;
  // re-reading the staged tiles with ldmatrix was measured: 1.11 against 1.085 ms per 4.2 M points)
  P = clamp_rows(P, rows);
  // the operand tiles need a 1024-byte aligned base: dynamic shared memory starts on one when the kernel has no static
  // shared memory (checked: a misaligned base raises the error flag instead of computing garbage)
  extern __shared__ __align__(1024) unsigned char smem[];
  if ((s32(smem) & 1023u) != 0u) {
    if (threadIdx.x == 0) atomicCAS(err, 0, 8);
    return;
  }
  const float gscale = grad_scale_from(__ldg(absmax));
  const float inv_s = 1.f / gscale;
  op16* sm = reinterpret_cast<op16*>(smem + GROUPS * SL::N * SLOT);          // weights, padded rows (mma.sync B operands)
  constexpr MlpSmem L = weight_layout<POS_K>();
  constexpr int SX = POS_K + PAD, SH = HID + PAD, SC = CIN + PAD;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + L.end);                  // done[GROUPS], full[GROUPS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * GROUPS);
  constexpr int KT1 = POS_K / 16;
  const int in_pad = (pos_dim + 15) & ~15;
  const int group = threadIdx.x / MLP_THREADS;                               // GROUPS: the issuer warp
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & 3, g = lane >> 2, t = lane & 3;
  const int row0 = 16 * warp;  // this warp's slab inside the 64-point tile
  load_all_weights<POS_K>(sp, cp, in_pad, sm);
  for (int i = threadIdx.x; i < GROUPS * SL::N * SLOT / 16; i += blockDim.x)      // unused tile columns are operands too: finite
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (threadIdx.x == 0) {
    for (int i = 0; i < GROUPS; ++i) {
      mbar_init(s32(bars + i), 1);
      mbar_init(s32(bars + GROUPS + i), MLP_THREADS);
    }
    mbar_init_fence();
  }
  if (threadIdx.x < 32) tmem_alloc(s32(tmem_slot), TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const bool gx_vec = g_x && ((ldg & 1) == 0) && ((pos_dim & 1) == 0) && ((reinterpret_cast<uintptr_t>(g_x) & 7) == 0);
  const int64_t n_tiles = (P + 63) / 64;
  const int64_t tile_first = (int64_t)blockIdx.x * GROUPS, tile_step = (int64_t)gridDim.x * GROUPS;

  // the 12 weight-gradient MMAs of one staged tile group + the commit that hands the slots back
  auto issue_wgrad = [&](int grp, uint32_t acc_first) {
    const uint32_t base = s32(smem) + grp * SL::N * SLOT;
    const uint32_t id128 = umma_idesc(Fmt::F16, Major::MN, 128, 128), id64 = umma_idesc(Fmt::F16, Major::MN, 64, 128);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const uint32_t o = base + kk * 2048;
      const uint32_t acc = (acc_first | (uint32_t)kk) ? 1u : 0u;
      tc_mma(tmem + D1, umma_desc_mn(o + SL::DZ3 * SLOT, SLOT), umma_desc_mn(o + SL::C * SLOT, SLOT), id128, acc);
      tc_mma(tmem + D2, umma_desc_mn(o + SL::A2 * SLOT, SLOT), umma_desc_mn(o + SL::B2 * SLOT, SLOT), id64, acc);
      tc_mma(tmem + D3, umma_desc_mn(o + SL::A3 * SLOT, SLOT), umma_desc_mn(o + SL::B3 * SLOT, SLOT), id64, acc);
    }
    tc_commit(s32(bars + grp));
  };

  bool ok = true;
  if (GROUPS > 1 && group == GROUPS) {
    // ================================ MMA issuer (one thread of the fourth warpgroup) ================================
    // registers are allocated per warpgroup: the kernel starts at 128 per thread (512 threads), the issuer's warpgroup
    // gives back all but 32 and the three worker groups grow to 160
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (threadIdx.x == GROUPS * MLP_THREADS) {
      // groups are served IN ORDER: a group that is early waits for its neighbours (ncu: ~11 try_wait rounds per tile in the
      // workers' wait for their slots), which keeps the three groups a third of a tile period apart -- their HMMA-heavy and
      // LSU-heavy phases interleave.  Serving whichever group is ready first was measured three ways (test_wait polling with a
      // 100 ns back-off, the same with an initial stagger of the groups, try_wait with a 200 ns suspend hint rotating over the
      // groups): 1.44-1.45 ms against 1.12 ms per 4.2 M points -- it is the enforced round-robin that pays
      uint32_t issued = 0u;
      for (int64_t base_tile = tile_first, it = 0; base_tile < n_tiles && ok; base_tile += tile_step, ++it) {
        for (int grp = 0; grp < GROUPS && ok; ++grp) {
          if (base_tile + grp >= n_tiles) break;
          ok = mbar_wait(s32(bars + GROUPS + grp), (uint32_t)(it & 1), err);
          tc_fence_after();
          issue_wgrad(grp, issued);
          issued = 1u;
        }
      }
    }
  } else {
    // ================================ worker groups ================================
    if (GROUPS > 1) asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
    op16* tiles = reinterpret_cast<op16*>(smem) + group * SL::N * (SLOT / 2);
    auto T = [&](int slot) { return tiles + slot * (SLOT / 2); };
    const uint32_t bar_done = s32(bars + group), bar_full = s32(bars + GROUPS + group);
    float2 xraw[KT1][4];       // this tile's x_enc rows as fp32: fetched one tile ahead, split into hi / lo at the top of the tile
    const bool x_full = pos_dim == POS_K && ((ldx & 1) == 0) && ((reinterpret_cast<uintptr_t>(x) & 7) == 0);
    auto fetch_x = [&](int64_t t) {
      if (x_full && (t + 1) * 64 <= P) load_x_raw_full<KT1>(x, ldx, t * 64 + row0, xraw, lane);
      else load_x_raw<KT1>(x, ldx, pos_dim, t * 64 + row0, P, xraw, lane, in_pad_value);
    };
    fetch_x(tile_first + group);
    uint32_t phase = 0;
    bool pending = false;
    for (int64_t tile = tile_first + group; tile < n_tiles && ok; tile += tile_step) {
      const int64_t p0 = tile * 64 + row0;
      // ---------------- forward recompute (staging every layer input)
      uint32_t ax[1][KT1][4], axl[1][KT1][4];
      pack_x_hl<KT1>(xraw, ax[0], axl[0]);
      float dcur[3];
      load_dir(dirs, p0 + (lane & 15), P, dcur);
      float grgb[4] = {0.f, 0.f, 0.f, 0.f}, gsig[2] = {0.f, 0.f};
      {
        const int64_t pa = p0 + g, pb = pa + 8;
        const int col = 2 * t;
        if (col < 3) {
          if (pa < P) {
            grgb[0] = __ldcs(g_rgb + 3 * pa + col);
            if (col + 1 < 3) grgb[1] = __ldcs(g_rgb + 3 * pa + col + 1);
          }
          if (pb < P) {
            grgb[2] = __ldcs(g_rgb + 3 * pb + col);
            if (col + 1 < 3) grgb[3] = __ldcs(g_rgb + 3 * pb + col + 1);
          }
        }
        if (t == 0) {
          if (pa < P) gsig[0] = __ldcs(g_sigma + pa);
          if (pb < P) gsig[1] = __ldcs(g_sigma + pb);
        }
      }                            // (scaled by S where they are used: the loads have the whole forward to land)
      uint32_t ah[1][4][4];
      {
        float c[1][8][4] = {};
        gemm_fwd<1, 8, KT1>(c, ax, sm + L.w1lo, SX, lane);             // split product: x_hi W_lo, then (x_lo + x_hi) W_hi with
        gemm_fwd_hl<8, KT1>(c[0], ax[0], axl[0], sm + L.w1, SX, lane);  // every W_hi fragment read from shared memory once
        c_to_a<8, true>(c[0], ah[0]);
      }
      // the previous tile's weight-gradient MMAs have had the first layer to finish reading the staged tiles
      if (pending) {
        ok = mbar_wait(bar_done, phase, err);
        phase ^= 1;
        tc_fence_after();
      }
      store_a_sw<KT1>(ax[0], T(SL::X), row0, 0, lane);
      store_a_sw<4>(ah[0], T(SL::H1), row0, 0, lane);
      // next tile's inputs: the fragments are dead from here on
      fetch_x(tile + tile_step);
      float hs0 = 0.f, hs1 = 0.f;  // h[.,0] of rows g and g+8 (threads with t == 0)
      uint32_t ac[1][3][4];
      {
        float c[1][2][4] = {};
        gemm_fwd<1, 2, 4>(c, ah, sm + L.w2, SH, lane);
        hs0 = c[0][0][0], hs1 = c[0][0][2];
        uint32_t tmp[1][4];
        c_to_a<2, false>(c[0], tmp);
        ac[0][0][0] = tmp[0][0], ac[0][0][1] = tmp[0][1], ac[0][0][2] = tmp[0][2], ac[0][0][3] = tmp[0][3];
        store_a_sw<1>(tmp, T(SL::C), row0, 0, lane);
      }
      if (lane < 16) {             // chunks 2..5 (columns 16..47) of swizzled row row0 + lane: the colour net's direction input
        op16* row = T(SL::C) + (row0 + lane) * 64;
        const int xr = (row0 + lane) & 7;
        dir_features(dcur, bands, L_dir, in_pad_value,
                     [&](int i, uint4 v) { *reinterpret_cast<uint4*>(row + 8 * ((2 + i) ^ xr)) = v; });
      }
      __syncwarp();
      {
        const int r = row0 + (lane & 7) + 8 * ((lane >> 3) & 1);
        ldsm_x4(ac[0][1], T(SL::C) + sw(r, 16 + 8 * (lane >> 4)));
        ldsm_x4(ac[0][2], T(SL::C) + sw(r, 32 + 8 * (lane >> 4)));
      }
      uint32_t a1[1][4][4], a2[1][4][4];
      {
        float c[1][8][4] = {};
        gemm_fwd<1, 8, 3>(c, ac, sm + L.v1, SC, lane);
        c_to_a<8, true>(c[0], a1[0]);
        store_a_sw<4>(a1[0], T(SL::C1), row0, 0, lane);
      }
      {
        float c[1][8][4] = {};
        gemm_fwd<1, 8, 4>(c, a1, sm + L.v2, SH, lane);
        c_to_a<8, true>(c[0], a2[0]);
        store_a_sw<4>(a2[0], T(SL::C2), row0, 0, lane);
      }
      // ---------------- output layer + its gradient
      uint32_t dz5[1][4];
      {
        float c[1][1][4] = {};
        gemm_fwd<1, 1, 4>(c, a2, sm + L.v3, SH, lane);
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        const int64_t pa = p0 + g, pb = pa + 8;
        const int col = 2 * t;
        if (col < 3) {
          if (pa < P) {
            const float y = sigmoidf(c[0][0][0]);
            d[0] = grgb[0] * gscale * y * (1.f - y);
            if (col + 1 < 3) {
              const float y1 = sigmoidf(c[0][0][1]);
              d[1] = grgb[1] * gscale * y1 * (1.f - y1);
            }
          }
          if (pb < P) {
            const float y = sigmoidf(c[0][0][2]);
            d[2] = grgb[2] * gscale * y * (1.f - y);
            if (col + 1 < 3) {
              const float y1 = sigmoidf(c[0][0][3]);
              d[3] = grgb[3] * gscale * y1 * (1.f - y1);
            }
          }
        }
        dz5[0][0] = pack2(d[0], d[1]), dz5[0][1] = pack2(d[2], d[3]), dz5[0][2] = 0u, dz5[0][3] = 0u;
        store_a_sw<1>(dz5, T(SL::DZ25), row0, SL::COL_DZ5, lane);
      }
      // ---------------- data-gradient chain
      uint32_t dz[1][4][4];
      {
        float c[8][4] = {};
        gemm_dgrad<8, 1>(c, dz5, sm + L.v3, SH, lane);          // d c2
        c_to_a<8, false>(c, dz[0]);
        relu_gate<4>(dz[0], a2[0]);            // c2's fragments are still live here in every variant (the output layer just read them)
        store_a_sw<4>(dz[0], T(SL::DZ4), row0, 0, lane);
      }
      {
        float c[8][4] = {};
        gemm_dgrad<8, 4>(c, dz[0], sm + L.v2, SH, lane);        // d c1
        c_to_a<8, false>(c, dz[0]);
        relu_gate<4>(dz[0], a1[0]);            // c1's fragments kept live across four stages: 16 registers against 4 ldmatrix + a warp sync
        store_a_sw<4>(dz[0], T(SL::DZ3), row0, 0, lane);
      }
      uint32_t dz2[1][4];
      {
        float c[2][4] = {};
        gemm_dgrad<2, 4>(c, dz[0], sm + L.v1, SC, lane);        // d h (first 16 inputs of color_net)
        if (t == 0) {                                           // density head: softplus'(h0 - 5)
          const int64_t pa = p0 + g, pb = pa + 8;
          if (pa < P) {
            const float v = hs0 - 5.f;
            c[0][0] += gsig[0] * gscale * (v > 20.f ? 1.f : sigmoidf(v));
          }
          if (pb < P) {
            const float v = hs1 - 5.f;
            c[0][2] += gsig[1] * gscale * (v > 20.f ? 1.f : sigmoidf(v));
          }
        }
        c_to_a<2, false>(c, dz2);
        store_a_sw<1>(dz2, T(SL::DZ25), row0, SL::COL_DZ2, lane);
      }
      {
        float c[8][4] = {};
        gemm_dgrad<8, 1>(c, dz2, sm + L.w2, SH, lane);          // d hidden1
        c_to_a<8, false>(c, dz[0]);
        relu_gate<4>(dz[0], ah[0]);
        store_a_sw<4>(dz[0], T(SL::DZ1), row0, 0, lane);
      }
      // ---------------- weight gradients over the 64 staged points: 12 asynchronous MMAs
      proxy_fence();               // the staged tiles are read by the tensor cores (async proxy)
      if (GROUPS == 1) {
        tc_fence_before();
        __syncthreads();
        if (threadIdx.x == 0) {
          tc_fence_after();
          issue_wgrad(0, pending ? 1u : 0u);
        }
      } else {
        mbar_arrive(bar_full);      // release: the issuer acquires
      }
      pending = true;
      if (g_x) {                   // d x_enc: registers + weights only, overlaps the MMAs
        float c[POS_K / 8][4] = {};
        gemm_dgrad<POS_K / 8, 4>(c, dz[0], sm + L.w1, SX, lane);
        const int64_t pa = p0 + g, pb = pa + 8;
        float* ra = g_x + pa * ldg + 2 * t;
        float* rb = g_x + pb * ldg + 2 * t;
        if (gx_vec && pos_dim == POS_K && (tile + 1) * 64 <= P) {      // interior tile, full width: no predicates
#pragma unroll
          for (int j = 0; j < POS_K / 8; ++j) {
            __stcs(reinterpret_cast<float2*>(ra + 8 * j), make_float2(c[j][0] * inv_s, c[j][1] * inv_s));
            __stcs(reinterpret_cast<float2*>(rb + 8 * j), make_float2(c[j][2] * inv_s, c[j][3] * inv_s));
          }
        } else if (gx_vec) {       // column pairs are contiguous and 8-byte aligned: one full 32-byte sector per row and store
#pragma unroll
          for (int j = 0; j < POS_K / 8; ++j) {
            if (8 * j + 2 * t < pos_dim) {
              if (pa < P) __stcs(reinterpret_cast<float2*>(ra + 8 * j), make_float2(c[j][0] * inv_s, c[j][1] * inv_s));
              if (pb < P) __stcs(reinterpret_cast<float2*>(rb + 8 * j), make_float2(c[j][2] * inv_s, c[j][3] * inv_s));
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < POS_K / 8; ++j) {
            const int col = 8 * j + 2 * t;
            if (pa < P) {
              if (col < pos_dim) ra[8 * j] = c[j][0] * inv_s;
              if (col + 1 < pos_dim) ra[8 * j + 1] = c[j][1] * inv_s;
            }
            if (pb < P) {
              if (col < pos_dim) rb[8 * j] = c[j][2] * inv_s;
              if (col + 1 < pos_dim) rb[8 * j + 1] = c[j][3] * inv_s;
            }
          }
        }
      }
    }
    if (pending && ok) ok = mbar_wait(bar_done, phase, err);      // this group's last MMAs are complete
  }
  // ---------------- flush: TMEM accumulators -> one red per weight per CTA
  tc_fence_before();
  __syncthreads();                 // every group's MMAs are complete (each group waited for its own)
  tc_fence_after();
  if (group == 0 && ok && tile_first < n_tiles) {
    const uint32_t lane_base = tmem + ((uint32_t)(32 * warp) << 16);
    const int f = 32 * (warp & 1) + lane;                   // feature index of this TMEM lane within its 64-row block
    const bool upper = warp >= 2;
    auto drain = [&](int col0, int ncols, float* dst, int stride_col, int n_valid) {
      // accumulator columns [col0, col0 + ncols): element j < n_valid goes to dst[j * stride_col]
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        uint32_t v[16];
        tc_ld16(lane_base + col0 + c0, v);
        tc_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (c0 + j < n_valid) atomicAdd(dst + (size_t)(c0 + j) * stride_col, __uint_as_float(v[j]) * inv_s);
      }
    };
    float* gV1 = g_cp;
    float* gV2 = g_cp + HID * CIN;
    float* gV3 = g_cp + HID * CIN + HID * HID;
    float* gW1 = g_sp;
    float* gW2 = g_sp + HID * in_pad;
    if (!upper) {
      drain(D1, 48, gV1 + f * CIN, 1, CIN);                          // dV1[f][k]
      drain(D2 + SL::COL_DZ5, 16, gV3 + f, HID, 3);                  // dV3[o][f], o < 3 (rows 3..15 are padding)
      drain(D3, POS_K, gW1 + f * in_pad, 1, in_pad);                 // dW1[f][k]
    } else {
      drain(D1 + 64, 64, gV2 + f * HID, 1, HID);                     // dV2[f][k]
      drain((SL::MERGED ? D3 : D2) + SL::COL_DZ2, 16, gW2 + f, HID, GEO);      // dW2[o][f]
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace b2n

using namespace b2n;

static int check_mlp_args(const float* x, int ldx, int pos_dim, const float* dirs, const float* bands, int L_dir,
                          const float* sp, const float* cp) {
  B2N_REQUIRE(pos_dim > 0 && pos_dim <= 64 && ldx >= pos_dim, "pos_dim must be in [1, 64]");
  B2N_REQUIRE(L_dir >= 0 && L_dir <= 4, "direction encoding must have at most 4 bands (27 features)");
  B2N_REQUIRE(x && dirs && sp && cp && (L_dir == 0 || bands), "null pointer");
  return B2N_OK;
}

// groups per CTA of k_instant_bwd_tc at pos_dim <= 32: 3 (default: one CTA per SM with 12 worker warps + the issuer) or
// 1 (two 4-warp CTAs per SM).  Measured at 4.2 M points (tools/kbench.py mlp64): 1.37 ms against 1.44 ms (a former
// all-mma.sync backward: 1.70 ms).  The 12-warp schedule only paid off once the d x_enc stores were vectorised (the LSU
// was the shared limit: 1.55 ms both before); ncu: `wait` (fixed-latency dependencies) is the top stall of both schedules
static int g_bwd_groups = 3;
extern "C" int b2n_debug_instant_bwd_groups(int groups) {
  const int prev = g_bwd_groups;
  if (groups == 1 || groups == 3 || groups == 4) g_bwd_groups = groups;      // 4: groups = 1 with ONE CTA per SM (overlap experiments)
  return prev;
}

// |g|-max pre-pass + k_instant_bwd_tc; err_flag as in b2n_instant_mlp_fwd_tc.
extern "C" int b2n_instant_mlp_bwd_tc(const float* x_enc, int ldx, int pos_dim, const float* dirs, const float* dir_bands,
                                      int L_dir, const float* sigma_params, const float* color_params, int64_t P,
                                      const float* g_rgb, const float* g_sigma, float* g_x_enc, int ldg,
                                      float* g_sigma_params, float* g_color_params, void* work4, float in_pad_value,
                                      int* err_flag, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  int rc = check_mlp_args(x_enc, ldx, pos_dim, dirs, dir_bands, L_dir, sigma_params, color_params);
  if (rc) return rc;
  B2N_REQUIRE(g_rgb && g_sigma && g_sigma_params && g_color_params && work4 && err_flag, "null pointer");
  B2N_REQUIRE(!g_x_enc || ldg >= pos_dim, "gradient row too narrow");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tiles = (P + 63) / 64;
  unsigned int* absmax = (unsigned int*)work4;
  if (cudaMemsetAsync(absmax, 0, 4, st) != cudaSuccess) return check_launch("b2n_instant_mlp_bwd_tc (memset)");
  {
    const int64_t n = 4 * P;
    const unsigned grid = (unsigned)((n + 1023) / 1024 < (int64_t)kSMs * 8 ? (n + 1023) / 1024 : (int64_t)kSMs * 8);
    k_grad_absmax<<<grid, 256, 0, st>>>(g_rgb, g_sigma, P, absmax, g_active_rows);
  }
  auto launch = [&](auto kern, size_t smem, int groups) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    // CTAs per SM by construction: two 4-warp CTAs (shared memory <= 113 KB, 256 of the 512 TMEM columns each) or one
    // CTA of three groups; the occupancy API reports 1 for tcgen05 kernels (see b2n_instant_mlp_fwd_tc)
    const int64_t units = groups == 1 ? tiles : (tiles + groups - 1) / groups;
    int64_t grid = groups == 1 && g_bwd_groups != 4 ? (int64_t)kSMs * 2 : (int64_t)kSMs;
    if (grid > units) grid = units;
    kern<<<(unsigned)grid, groups == 1 ? MLP_THREADS : (groups + 1) * MLP_THREADS, smem, st>>>(
        x_enc, ldx, pos_dim, dirs, dir_bands, L_dir, sigma_params, color_params, P, g_rgb, g_sigma, g_x_enc, ldg,
        g_sigma_params, g_color_params, absmax, g_active_rows, in_pad_value, err_flag);
  };
  if (pos_dim <= 32) {
    if (g_bwd_groups == 3) launch(k_instant_bwd_tc<32, 3>, bwtc::smem_bytes<32, 3>(), 3);
    else launch(k_instant_bwd_tc<32, 1>, bwtc::smem_bytes<32, 1>(), 1);
  } else {
    launch(k_instant_bwd_tc<64, 1>, bwtc::smem_bytes<64, 1>(), 1);
  }
  return check_launch("b2n_instant_mlp_bwd_tc");
}
