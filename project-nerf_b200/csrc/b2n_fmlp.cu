// Fused small-width ReLU MLPs of the dynamic configs, one kernel forward and one kernel backward:
//   DeformationNetwork        cat[gamma(x'), gamma(t')](84) -> 128 -> 128 -> 128 -> 3   (src/decoders.py:171-195)
//   HashDeformationDecoder    cat[hash feat(24), time mod(64)](88) -> 64 -> 64 -> 3     (src/decoders.py:285-316,
//                                                                      tinycudann FullyFusedMLP replaced)
//   TimeModulationNetwork     gamma(t')(21) -> 64 -> 64, sigmoid                        (src/decoders.py:340-371)
// and any other ReLU MLP of that family: 1..3 hidden layers of width 64 or 128, up to 96 inputs taken
// from one or two row-major fp32 sources (the concat is never materialised), up to 64 outputs, optional
// biases, linear or sigmoid output.
//
// Arithmetic: op16 operands, fp32 accumulation on the tensor cores (mma.sync m16n8k16) -- the
// reference runs these nets in fp16 (tinycudann) or under torch.amp.autocast (nn.Linear).
//   forward : each warp owns 16*MT points; the C fragments of a layer are re-packed in registers as
//             the A fragments of the next layer; weights are op16 in shared memory (ldmatrix), biases
//             initialise the accumulators.  When training, the op16 input row and every hidden
//             activation are also written to HBM ("planes").
//   backward: each warp owns 16 points; the data-gradient chain runs in registers (ldmatrix.trans on
//             the same weight tiles), ReLU gates come from the saved planes, every pre-activation
//             gradient dZ_l is written to HBM in op16 and the input gradient in fp32.
//   wgrad   : dW_l = dZ_l^T In_l and db_l = colsum(dZ_l) for all layers of the network in one launch
//             (k_fmlp_wgrad): split over P, tensor-core accumulators per CTA, one atomicAdd per weight.
#define B2N_OP_F16
#include "b2n_mma.cuh"

namespace b2n {
namespace fm {

constexpr int THREADS = 128;
constexpr int MAX_HID = 3;

struct Args {
  const float* x0; int ld0, d0;
  const float* x1; int ld1, d1;
  const float* W[MAX_HID + 1]; int ldw[MAX_HID + 1];   // W[0..n_hidden-1] hidden layers, W[n_hidden] output layer
  const float* b[MAX_HID + 1];
  int n_hidden, out_dim, out_act;
  int64_t P;
  float* y; int ldy;
  op16* xin;       // [P][IN_PAD]  op16 copy of the concatenated input (training) or null
  op16* hplanes;   // [n_hidden][P][H] hidden activations (training) or null
  // backward only
  const float* g_y; int ldgy;
  const float* y_out;   // forward outputs (sigmoid derivative)
  op16* dz_out;    // [P][OUT_PAD16]
  op16* dz_h;      // [n_hidden][P][H]
  float* g_x0; int ldg0;
  float* g_x1; int ldg1;
  unsigned int* work;   // [0] |g_y|-max bits (pre-pass), [1] the gradient scale S as a float (written by the kernel)
  const int* rows;      // optional device-side row count (b2n_set_active_rows)
};

template <int H, int KT_IN, int NT_OUT>
struct Layout {
  static constexpr int IN_PAD = 16 * KT_IN;
  static constexpr int OUT_ROWS = (8 * NT_OUT + 15) / 16 * 16;   // rows of the output matrix kept in smem
  static constexpr int S0 = IN_PAD + PAD, SH = H + PAD;
  static constexpr int w0 = 0;
  static constexpr int wh = w0 + H * S0;                          // hidden matrices 1 .. MAX_HID-1
  static constexpr int wo = wh + (MAX_HID - 1) * H * SH;
  static constexpr int end_op16 = wo + OUT_ROWS * SH;
  static constexpr int bias_floats = MAX_HID * H + OUT_ROWS;
  static constexpr size_t bytes = (size_t)end_op16 * sizeof(op16) + (size_t)bias_floats * sizeof(float);
};

// fp32 matrix [rows_valid][cols_valid] (row stride ldw) -> op16 smem [rows][cols + PAD], zero filled elsewhere
__device__ __forceinline__ void load_w(const float* __restrict__ W, int ldw, int rows_valid, int cols_valid, int rows,
                                       int cols, op16* dst) {
  const int S = cols + PAD;
  for (int i = threadIdx.x; i < rows * cols; i += blockDim.x) {
    const int r = i / cols, c = i - r * cols;
    dst[r * S + c] = to_op16((r < rows_valid && c < cols_valid) ? __ldg(W + (size_t)r * ldw + c) : 0.f);
  }
}

// skip_w0: the backward without input gradients never touches the first matrix -- it is not staged and every later
// offset moves down by its size (26 KB at H = 128: 3 CTAs per SM instead of 2)
template <int H, int KT_IN, int NT_OUT>
__device__ __forceinline__ float* stage_weights(const Args& a, op16* sm, bool skip_w0 = false) {
  using LY = Layout<H, KT_IN, NT_OUT>;
  if (!skip_w0) load_w(a.W[0], a.ldw[0], H, a.d0 + a.d1, H, LY::IN_PAD, sm + LY::w0);
  else sm -= LY::wh;
  for (int l = 1; l < a.n_hidden; ++l) load_w(a.W[l], a.ldw[l], H, H, H, H, sm + LY::wh + (l - 1) * H * LY::SH);
  load_w(a.W[a.n_hidden], a.ldw[a.n_hidden], a.out_dim, H, LY::OUT_ROWS, H, sm + LY::wo);
  float* bias = reinterpret_cast<float*>(sm + LY::end_op16);
  for (int i = threadIdx.x; i < LY::bias_floats; i += blockDim.x) {
    float v = 0.f;
    if (i < MAX_HID * H) {
      const int l = i / H, c = i - l * H;
      if (l < a.n_hidden && a.b[l]) v = __ldg(a.b[l] + c);
    } else {
      const int c = i - MAX_HID * H;
      if (c < a.out_dim && a.b[a.n_hidden]) v = __ldg(a.b[a.n_hidden] + c);
    }
    bias[i] = v;
  }
  return bias;
}

// A fragments of 16 rows of the (virtually concatenated) input [x0 | x1 | 0]
template <int KT>
__device__ __forceinline__ void load_in(const Args& a, int64_t P, int64_t p0, uint32_t (&f)[KT][4], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const int din = a.d0 + a.d1;
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int64_t p = p0 + g + 8 * r;
        const int c = 16 * k + 8 * h + 2 * t;
        float v[2] = {0.f, 0.f};
        if (p < P) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int cc = c + j;
            if (cc < a.d0) v[j] = __ldcs(a.x0 + p * a.ld0 + cc);
            else if (cc < din) v[j] = __ldcs(a.x1 + p * a.ld1 + (cc - a.d0));
          }
        }
        f[k][2 * h + r] = pack2(v[0], v[1]);
      }
}

// split version for software pipelining: issue the loads of a tile now, pack (and wait for them) one tile later
template <int KT>
__device__ __forceinline__ void load_in_raw(const Args& a, int64_t P, int64_t p0, float (&raw)[KT][4][2], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const int din = a.d0 + a.d1;
#pragma unroll
  for (int k = 0; k < KT; ++k)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int64_t p = p0 + g + 8 * r;
        const int c = 16 * k + 8 * h + 2 * t;
        raw[k][2 * h + r][0] = raw[k][2 * h + r][1] = 0.f;
        if (p < P) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int cc = c + j;
            if (cc < a.d0) raw[k][2 * h + r][j] = __ldcs(a.x0 + p * a.ld0 + cc);
            else if (cc < din) raw[k][2 * h + r][j] = __ldcs(a.x1 + p * a.ld1 + (cc - a.d0));
          }
        }
      }
}

// A fragments of a 16-row slab -> rows p0.. of a row-major op16 plane (row stride ld, even)
// rows [P, Ppad) are written as zeros (see Args::Ppad)
template <int KT>
__device__ __forceinline__ void store_plane(const uint32_t (&f)[KT][4], op16* plane, int ld, int64_t p0, int64_t P,
                                            int lane, int64_t Ppad = 0) {
  const int g = lane >> 2, t = lane & 3;
  const int64_t pa = p0 + g, pb = pa + 8;
  if (Ppad < P) Ppad = P;
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (pa < Ppad) {
      uint32_t* r0 = reinterpret_cast<uint32_t*>(plane + pa * ld + 16 * k + 2 * t);
      const bool v = pa < P;
      r0[0] = v ? f[k][0] : 0u, r0[4] = v ? f[k][2] : 0u;
    }
    if (pb < Ppad) {
      uint32_t* r1 = reinterpret_cast<uint32_t*>(plane + pb * ld + 16 * k + 2 * t);
      const bool v = pb < P;
      r1[0] = v ? f[k][1] : 0u, r1[4] = v ? f[k][3] : 0u;
    }
  }
}

template <int NT>
__device__ __forceinline__ void init_bias(float (&c)[NT][4], const float* bias, int lane) {
  const int t = lane & 3;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const float b0 = bias[8 * j + 2 * t], b1 = bias[8 * j + 2 * t + 1];
    c[j][0] = b0, c[j][1] = b1, c[j][2] = b0, c[j][3] = b1;
  }
}

// zero the gradient where the saved (post-ReLU) activation is not positive
template <int NT>
__device__ __forceinline__ void relu_gate(float (&c)[NT][4], const op16* plane, int ld, int64_t p0, int64_t P, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const int64_t pa = p0 + g, pb = pa + 8;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const uint32_t ra = pa < P ? __ldcs(reinterpret_cast<const uint32_t*>(plane + pa * ld + 8 * j + 2 * t)) : 0u;
    const uint32_t rb = pb < P ? __ldcs(reinterpret_cast<const uint32_t*>(plane + pb * ld + 8 * j + 2 * t)) : 0u;
    const float2 lo = unpack2(ra), hi = unpack2(rb);
    if (!(lo.x > 0.f)) c[j][0] = 0.f;
    if (!(lo.y > 0.f)) c[j][1] = 0.f;
    if (!(hi.x > 0.f)) c[j][2] = 0.f;
    if (!(hi.y > 0.f)) c[j][3] = 0.f;
  }
}

// split version: the gate words of a layer are fetched one GEMM ahead of their use
template <int NT>
__device__ __forceinline__ void load_gate(const op16* plane, int ld, int64_t p0, int64_t P, uint32_t (&ga)[NT],
                                          uint32_t (&gb)[NT], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const int64_t pa = p0 + g, pb = pa + 8;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    ga[j] = pa < P ? __ldcs(reinterpret_cast<const uint32_t*>(plane + pa * ld + 8 * j + 2 * t)) : 0u;
    gb[j] = pb < P ? __ldcs(reinterpret_cast<const uint32_t*>(plane + pb * ld + 8 * j + 2 * t)) : 0u;
  }
}
template <int NT>
__device__ __forceinline__ void apply_gate(float (&c)[NT][4], const uint32_t (&ga)[NT], const uint32_t (&gb)[NT]) {
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const float2 lo = unpack2(ga[j]), hi = unpack2(gb[j]);
    if (!(lo.x > 0.f)) c[j][0] = 0.f;
    if (!(lo.y > 0.f)) c[j][1] = 0.f;
    if (!(hi.x > 0.f)) c[j][2] = 0.f;
    if (!(hi.y > 0.f)) c[j][3] = 0.f;
  }
}

__device__ __forceinline__ float sigm(float v) { return 1.f / (1.f + expf(-v)); }

// max |g_y| as float bits (see k_grad_absmax in b2n_mlp64.cu: same convention, NaN sorts above everything)
__global__ void __launch_bounds__(256) k_fmlp_absmax(const float* __restrict__ g, int ld, int cols, int64_t P,
                                                     unsigned int* __restrict__ out, const int* __restrict__ rows) {
  P = clamp_rows(P, rows);
  unsigned int m = 0u;
  const int64_t n = P * cols;
  if (ld == cols && (n & 3) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0) {       // contiguous rows: flat 16-byte loads
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n >> 2); i += (int64_t)gridDim.x * blockDim.x) {
      const float4 v = __ldg(g4 + i);
      m = max(max(m, __float_as_uint(v.x) & 0x7fffffffu), __float_as_uint(v.y) & 0x7fffffffu);
      m = max(max(m, __float_as_uint(v.z) & 0x7fffffffu), __float_as_uint(v.w) & 0x7fffffffu);
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      const int64_t p = i / cols;
      m = max(m, __float_as_uint(__ldg(g + p * ld + (i - p * cols))) & 0x7fffffffu);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}
__device__ __forceinline__ float fmlp_scale_from(unsigned int bits) {
  if (bits == 0u) return 1.f;
  if (bits >= 0x7f800000u) return __uint_as_float(0x7fc00000u);      // non-finite gradient in -> non-finite out
  int se = 7 - ((int)(bits >> 23) - 127);
  se = se > 120 ? 120 : (se < -120 ? -120 : se);
  return __uint_as_float((unsigned int)(se + 127) << 23);
}

// ------------------------------------------------------------------------------ forward
template <int H, int KT_IN, int NT_OUT, int MT>
__global__ void __launch_bounds__(THREADS) k_fmlp_fwd(const Args a) {
  // NOT a local copy of `a`: the layer arrays are indexed dynamically, and a modified copy of a kernel parameter lives in
  // local memory (272-byte stack frame, every a.* an LDL); the row counts are plain locals instead
  const int64_t P = clamp_rows(a.P, a.rows);              // valid rows (device-side count, b2n_set_active_rows)
  const int64_t Pcap = a.P;                               // rows the planes were allocated for: stride between layer planes
  const int64_t Ppad = min(a.P, (P + 63) & ~(int64_t)63);    // rows [P, Ppad) of the saved planes are zero-filled (the tcgen05
                                                          // weight-gradient kernel streams whole 64-row tiles)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  op16* sm = reinterpret_cast<op16*>(smem_raw);
  using LY = Layout<H, KT_IN, NT_OUT>;
  const float* bias = stage_weights<H, KT_IN, NT_OUT>(a, sm);
  __syncthreads();
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  constexpr int ROWS = 16 * MT;
  const int64_t n_tiles = (Ppad + ROWS - 1) / ROWS;
  const int64_t wstride = (int64_t)gridDim.x * (THREADS / 32);
  // single-slab variants (H = 128) have registers to spare: the next tile's input rows are fetched one tile ahead
  constexpr bool PF = (MT == 1);
  constexpr int KTP = PF ? KT_IN : 1;
  float raw[KTP][4][2];
  const int64_t tile0 = (int64_t)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5);
  if (PF) load_in_raw<KTP>(a, P, tile0 * ROWS, raw, lane);
  for (int64_t tile = tile0; tile < n_tiles; tile += wstride) {
    const int64_t p0 = tile * ROWS;
    uint32_t ah[MT][H / 16][4];
    {
      uint32_t ax[MT][KT_IN][4];
      if (PF) {
#pragma unroll
        for (int k = 0; k < KT_IN; ++k)
#pragma unroll
          for (int i = 0; i < 4; ++i) ax[0][k][i] = pack2(raw[k % KTP][i][0], raw[k % KTP][i][1]);
        load_in_raw<KTP>(a, P, (tile + wstride) * ROWS, raw, lane);
        if (a.xin) store_plane<KT_IN>(ax[0], a.xin, LY::IN_PAD, p0, P, lane, Ppad);
      } else {
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          load_in<KT_IN>(a, P, p0 + 16 * m, ax[m], lane);
          if (a.xin) store_plane<KT_IN>(ax[m], a.xin, LY::IN_PAD, p0 + 16 * m, P, lane, Ppad);
        }
      }
      float c[MT][H / 8][4];
#pragma unroll
      for (int m = 0; m < MT; ++m) init_bias<H / 8>(c[m], bias, lane);
      gemm_fwd<MT, H / 8, KT_IN>(c, ax, sm + LY::w0, LY::S0, lane);
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        c_to_a<H / 8, true>(c[m], ah[m]);
        if (a.hplanes) store_plane<H / 16>(ah[m], a.hplanes, H, p0 + 16 * m, P, lane, Ppad);
      }
    }
#pragma unroll 1
    for (int l = 1; l < a.n_hidden; ++l) {
      float c[MT][H / 8][4];
#pragma unroll
      for (int m = 0; m < MT; ++m) init_bias<H / 8>(c[m], bias + l * H, lane);
      gemm_fwd<MT, H / 8, H / 16>(c, ah, sm + LY::wh + (l - 1) * H * LY::SH, LY::SH, lane);
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        c_to_a<H / 8, true>(c[m], ah[m]);
        if (a.hplanes) store_plane<H / 16>(ah[m], a.hplanes + (size_t)l * Pcap * H, H, p0 + 16 * m, P, lane, Ppad);
      }
    }
    {
      float c[MT][NT_OUT][4];
#pragma unroll
      for (int m = 0; m < MT; ++m) init_bias<NT_OUT>(c[m], bias + MAX_HID * H, lane);
      gemm_fwd<MT, NT_OUT, H / 16>(c, ah, sm + LY::wo, LY::SH, lane);
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const int64_t pa = p0 + 16 * m + g, pb = pa + 8;
#pragma unroll
        for (int j = 0; j < NT_OUT; ++j) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int col = 8 * j + 2 * t + (i & 1);
            const int64_t p = (i & 2) ? pb : pa;
            if (col < a.out_dim && p < P) {
              float v = c[m][j][i];
              if (a.out_act == B2N_ACT_SIGMOID) v = sigm(v);
              else if (a.out_act == B2N_ACT_RELU) v = fmaxf(v, 0.f);
              a.y[p * a.ldy + col] = v;
            }
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------ backward (data gradients)
template <int H, int KT_IN, int NT_OUT>
__global__ void __launch_bounds__(THREADS) k_fmlp_bwd(const Args a) {
  // NOT a local copy of `a`: the layer arrays are indexed dynamically, and a modified copy of a kernel parameter lives in
  // local memory (272-byte stack frame, every a.* an LDL); the row counts are plain locals instead
  const int64_t P = clamp_rows(a.P, a.rows);              // valid rows (device-side count, b2n_set_active_rows)
  const int64_t Pcap = a.P;                               // rows the planes were allocated for: stride between layer planes
  const int64_t Ppad = min(a.P, (P + 63) & ~(int64_t)63);    // rows [P, Ppad) of the saved planes are zero-filled
  extern __shared__ __align__(16) unsigned char smem_raw[];
  op16* sm = reinterpret_cast<op16*>(smem_raw);
  using LY = Layout<H, KT_IN, NT_OUT>;
  const bool need_x = a.g_x0 || a.g_x1;
  const float gscale = fmlp_scale_from(__ldg(a.work));
  const float inv_s = 1.f / gscale;
  if (blockIdx.x == 0 && threadIdx.x == 0) reinterpret_cast<float*>(a.work)[1] = gscale;    // for the weight-gradient pass
  stage_weights<H, KT_IN, NT_OUT>(a, sm, !need_x);
  if (!need_x) sm -= LY::wh;          // all offsets below are relative to the (unstaged) first matrix
  __syncthreads();
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  constexpr int KTO = LY::OUT_ROWS / 16;
  const int64_t n_tiles = (Ppad + 15) / 16;
  const int64_t wstride = (int64_t)gridDim.x * (THREADS / 32);
  for (int64_t tile = (int64_t)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5); tile < n_tiles; tile += wstride) {
    const int64_t p0 = tile * 16;
    uint32_t ga[H / 8], gb[H / 8];      // ReLU gate words of the layer about to be gated
    load_gate<H / 8>(a.hplanes + (size_t)(a.n_hidden - 1) * Pcap * H, H, p0, P, ga, gb, lane);
    // ---- dZ of the output layer
    uint32_t dzo[KTO][4];
#pragma unroll
    for (int k = 0; k < KTO; ++k)
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const int64_t p = p0 + g + 8 * r;
          const int c = 16 * k + 8 * h + 2 * t;
          float v[2] = {0.f, 0.f};
          if (p < P) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              if (c + j < a.out_dim) {
                float gy = __ldcs(a.g_y + p * a.ldgy + c + j);
                if (a.out_act != B2N_ACT_NONE) {
                  const float y = __ldcs(a.y_out + p * a.ldy + c + j);
                  gy = (a.out_act == B2N_ACT_SIGMOID) ? gy * y * (1.f - y) : (y > 0.f ? gy : 0.f);
                }
                v[j] = gy * gscale;
              }
            }
          }
          dzo[k][2 * h + r] = pack2(v[0], v[1]);
        }
    store_plane<KTO>(dzo, a.dz_out, LY::OUT_ROWS, p0, P, lane, Ppad);
    // ---- last hidden layer
    uint32_t dz[H / 16][4];
    {
      float c[H / 8][4] = {};
      gemm_dgrad<H / 8, KTO>(c, dzo, sm + LY::wo, LY::SH, lane);
      apply_gate<H / 8>(c, ga, gb);
      if (a.n_hidden > 1) load_gate<H / 8>(a.hplanes + (size_t)(a.n_hidden - 2) * Pcap * H, H, p0, P, ga, gb, lane);
      c_to_a<H / 8, false>(c, dz);
      store_plane<H / 16>(dz, a.dz_h + (size_t)(a.n_hidden - 1) * Pcap * H, H, p0, P, lane, Ppad);
    }
#pragma unroll 1
    for (int l = a.n_hidden - 1; l >= 1; --l) {
      float c[H / 8][4] = {};
      gemm_dgrad<H / 8, H / 16>(c, dz, sm + LY::wh + (l - 1) * H * LY::SH, LY::SH, lane);
      apply_gate<H / 8>(c, ga, gb);
      if (l > 1) load_gate<H / 8>(a.hplanes + (size_t)(l - 2) * Pcap * H, H, p0, P, ga, gb, lane);
      c_to_a<H / 8, false>(c, dz);
      store_plane<H / 16>(dz, a.dz_h + (size_t)(l - 1) * Pcap * H, H, p0, P, lane, Ppad);
    }
    if (a.g_x0 || a.g_x1) {
      float c[2 * KT_IN][4] = {};
      gemm_dgrad<2 * KT_IN, H / 16>(c, dz, sm + LY::w0, LY::S0, lane);
      const int din = a.d0 + a.d1;
#pragma unroll
      for (int j = 0; j < 2 * KT_IN; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int col = 8 * j + 2 * t + (i & 1);
          const int64_t p = p0 + g + ((i & 2) ? 8 : 0);
          if (p < P) {
            if (col < a.d0) {
              if (a.g_x0) a.g_x0[p * a.ldg0 + col] = c[j][i] * inv_s;
            } else if (col < din) {
              if (a.g_x1) a.g_x1[p * a.ldg1 + (col - a.d0)] = c[j][i] * inv_s;
            }
          }
        }
    }
  }
}


// ------------------------------------------------------------------------------ weight / bias gradients
// dW_l[rows, k] += dZ_l^T In_l and db_l[rows] += colsum(dZ_l) over all P points, for every layer of one
// network in a single launch (blockIdx.y = layer).  A CTA streams 64-point tiles of the two op16 planes
// into shared memory (cp.async, double buffered); each warp owns one 16-row x (up to) 64-column tile of
// dW in tensor-core accumulators for the whole persistent loop and flushes it with one atomicAdd per
// weight at the end.  (cuBLAS was tried first: for these skinny [<=128 x P] x [P x <=128] shapes with P
// changing every step its host-side heuristics cost ~6 ms of CPU time per call.)
constexpr int WG_THREADS = 512;
constexpr int WG_TILE = 64;
constexpr int WG_MAXW = 128;                       // widest plane
constexpr int WG_S = WG_MAXW + PAD;                // smem row stride of both tiles
constexpr size_t WG_SMEM = (size_t)2 * 2 * WG_TILE * WG_S * sizeof(op16);

struct WgLayer {
  const op16* dz; int ldz, rows;       // [P][ldz], rows = plane width (multiple of 16)
  const op16* in; int ldi, k;          // [P][ldi], k = plane width (multiple of 16)
  float* dW; int lddw, rows_valid, k_valid;
  float* db;                           // [rows_valid] or null
};
struct WgArgs {
  WgLayer L[MAX_HID + 1];
  int64_t P;
  const float* scale;                  // device: the dZ planes hold S * dZ (b2n_fmlp_bwd); results are divided by S.  null: 1
  const int* rows;                     // optional device-side row count
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
  const int n = valid ? 16 : 0;        // src-size 0: the 16 bytes are zero filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(n) : "memory");
}

__device__ __forceinline__ void wg_load_tile(const WgLayer& L, int64_t p0, int64_t P, op16* dzs, op16* ins) {
  const int cz = L.rows >> 3, ci = L.k >> 3;       // 16-byte chunks per row
  for (int i = threadIdx.x; i < WG_TILE * (cz + ci); i += WG_THREADS) {
    const bool is_z = i < WG_TILE * cz;
    const int j = is_z ? i : i - WG_TILE * cz;
    const int w = is_z ? cz : ci;
    const int r = j / w, c = j - r * w;
    const int64_t p = p0 + r;
    const bool ok = p < P;
    const op16* src = is_z ? L.dz + (ok ? p : 0) * L.ldz + 8 * c : L.in + (ok ? p : 0) * L.ldi + 8 * c;
    cp_async16((is_z ? dzs : ins) + r * WG_S + 8 * c, src, ok);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

__global__ void __launch_bounds__(WG_THREADS) k_fmlp_wgrad(const WgArgs a) {
  const int64_t P = clamp_rows(a.P, a.rows);        // (no local copy of `a`: see k_fmlp_fwd)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  op16* sm = reinterpret_cast<op16*>(smem_raw);
  const WgLayer& L = a.L[blockIdx.y];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int n_row_tiles = L.rows >> 4, n_col_tiles = (L.k + 63) >> 6;
  const bool active = warp < n_row_tiles * n_col_tiles;
  const int n0 = 16 * (warp % n_row_tiles), k0 = 64 * (warp / n_row_tiles);
  const int npairs = active ? min(L.k - k0, 64) >> 4 : 0;      // pairs of 8-column tiles this warp owns
  float acc[8][4] = {};
  float bsum = 0.f;
  const float inv_s = a.scale ? 1.f / __ldg(a.scale) : 1.f;
  const int64_t n_tiles = (P + WG_TILE - 1) / WG_TILE;
  int buf = 0;
  if ((int64_t)blockIdx.x < n_tiles) wg_load_tile(L, (int64_t)blockIdx.x * WG_TILE, P, sm, sm + WG_TILE * WG_S);
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    op16* dzs = sm + buf * 2 * WG_TILE * WG_S;
    op16* ins = dzs + WG_TILE * WG_S;
    const int64_t next = tile + gridDim.x;
    if (next < n_tiles) {
      op16* nz = sm + (buf ^ 1) * 2 * WG_TILE * WG_S;
      wg_load_tile(L, next * WG_TILE, P, nz, nz + WG_TILE * WG_S);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    if (active) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t af[4];
        ldsm_x4_t(af, dzs + (16 * ks + 8 * (lane >> 4) + (lane & 7)) * WG_S + n0 + 8 * ((lane >> 3) & 1));
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) {
          if (jp < npairs) {
            uint32_t b[4];
            ldsm_x4_t(b, ins + (16 * ks + 8 * ((lane >> 3) & 1) + (lane & 7)) * WG_S + k0 + 8 * (2 * jp + (lane >> 4)));
            mma16816(acc[2 * jp], af, b[0], b[1]);
            mma16816(acc[2 * jp + 1], af, b[2], b[3]);
          }
        }
      }
    }
    if (L.db && threadIdx.x < L.rows) {
      float s = 0.f;
#pragma unroll 8
      for (int r = 0; r < WG_TILE; ++r) s += from_op16(dzs[r * WG_S + threadIdx.x]);
      bsum += s;
    }
    __syncthreads();
    buf ^= 1;
  }
  if (active) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < 2 * npairs) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = n0 + g + ((i & 2) ? 8 : 0), col = k0 + 8 * j + 2 * t + (i & 1);
          if (row < L.rows_valid && col < L.k_valid && acc[j][i] != 0.f)
            atomicAdd(L.dW + (size_t)row * L.lddw + col, acc[j][i] * inv_s);
        }
      }
    }
  }
  if (L.db && threadIdx.x < L.rows_valid) atomicAdd(L.db + threadIdx.x, bsum * inv_s);
}

static int persistent_grid(const void* kernel, size_t smem, int64_t warp_tiles) {
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, THREADS, smem);
  if (per_sm < 1) per_sm = 1;
  int64_t g = (int64_t)kSMs * per_sm;
  const int64_t blocks = (warp_tiles + THREADS / 32 - 1) / (THREADS / 32);
  if (g > blocks) g = blocks;
  if (g < 1) g = 1;
  return (int)g;
}


template <int H, int KT_IN, int NT_OUT, int MT>
static int launch_fwd(const Args& a, cudaStream_t st) {
  constexpr size_t smem = Layout<H, KT_IN, NT_OUT>::bytes;
  auto k = k_fmlp_fwd<H, KT_IN, NT_OUT, MT>;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int grid = persistent_grid((const void*)k, smem, (a.P + 16 * MT - 1) / (16 * MT));
  k<<<grid, THREADS, smem, st>>>(a);
  return check_launch("b2n_fmlp_fwd");
}
template <int H, int KT_IN, int NT_OUT>
static int launch_bwd(const Args& a, cudaStream_t st) {
  using LY = Layout<H, KT_IN, NT_OUT>;
  const size_t smem = LY::bytes - ((a.g_x0 || a.g_x1) ? 0 : (size_t)LY::wh * sizeof(op16));
  auto k = k_fmlp_bwd<H, KT_IN, NT_OUT>;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int grid = persistent_grid((const void*)k, smem, (a.P + 15) / 16);
  k<<<grid, THREADS, smem, st>>>(a);
  return check_launch("b2n_fmlp_bwd");
}

}  // namespace fm
}  // namespace b2n

using namespace b2n;
using namespace b2n::fm;

// need_inputs: the forward reads x0 / x1; the backward only needs their widths
static int fill_args(Args* a, bool need_inputs, const float* x0, int ld0, int d0, const float* x1, int ld1, int d1,
                     int hidden, int n_hidden, const float* const* W, const int* ldw, const float* const* b, int out_dim,
                     int out_act, int64_t P) {
  B2N_REQUIRE(hidden == 64 || hidden == 128, "hidden width must be 64 or 128");
  B2N_REQUIRE(n_hidden >= 1 && n_hidden <= MAX_HID, "1..3 hidden layers");
  B2N_REQUIRE(d0 > 0 && d1 >= 0, "bad input widths");
  B2N_REQUIRE(!need_inputs || (x0 && ld0 >= d0 && (d1 == 0 || (x1 && ld1 >= d1))), "bad input sources");
  B2N_REQUIRE(d0 + d1 <= 96, "at most 96 inputs");
  B2N_REQUIRE(out_dim >= 1 && out_dim <= 64, "1..64 outputs");
  B2N_REQUIRE(out_act == B2N_ACT_NONE || out_act == B2N_ACT_RELU || out_act == B2N_ACT_SIGMOID, "bad activation");
  B2N_REQUIRE(W && ldw && (b || !need_inputs), "null pointer");
  a->x0 = x0, a->ld0 = ld0, a->d0 = d0, a->x1 = x1, a->ld1 = ld1, a->d1 = d1;
  for (int l = 0; l <= n_hidden; ++l) {
    B2N_REQUIRE(W[l], "null weight");
    const int k = (l == 0) ? d0 + d1 : hidden;
    B2N_REQUIRE(ldw[l] >= k, "weight row shorter than the layer input");
    a->W[l] = W[l], a->ldw[l] = ldw[l], a->b[l] = b ? b[l] : nullptr;
  }
  a->n_hidden = n_hidden, a->out_dim = out_dim, a->out_act = out_act, a->P = P;
  a->rows = g_active_rows;
  return B2N_OK;
}

extern "C" int b2n_fmlp_in_pad(int d_in) { return d_in <= 32 ? 32 : 96; }
extern "C" int b2n_fmlp_out_pad(int out_dim) { return out_dim <= 16 ? 16 : 64; }

extern "C" int b2n_fmlp_fwd(const float* x0, int ld0, int d0, const float* x1, int ld1, int d1, int hidden, int n_hidden,
                            const float* const* W, const int* ldw, const float* const* b, int out_dim, int out_act,
                            int64_t P, float* y, int ldy, void* xin_plane, void* h_planes, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  Args a{};
  int rc = fill_args(&a, true, x0, ld0, d0, x1, ld1, d1, hidden, n_hidden, W, ldw, b, out_dim, out_act, P);
  if (rc) return rc;
  B2N_REQUIRE(y && ldy >= out_dim, "bad output");
  a.y = y, a.ldy = ldy, a.xin = (op16*)xin_plane, a.hplanes = (op16*)h_planes;
  cudaStream_t st = (cudaStream_t)stream;
  const bool small_in = d0 + d1 <= 32, small_out = out_dim <= 16;
  if (hidden == 64) {
    if (small_in) return small_out ? launch_fwd<64, 2, 2, 2>(a, st) : launch_fwd<64, 2, 8, 2>(a, st);
    return small_out ? launch_fwd<64, 6, 2, 2>(a, st) : launch_fwd<64, 6, 8, 2>(a, st);
  }
  if (small_in) return small_out ? launch_fwd<128, 2, 2, 1>(a, st) : launch_fwd<128, 2, 8, 1>(a, st);
  return small_out ? launch_fwd<128, 6, 2, 1>(a, st) : launch_fwd<128, 6, 8, 1>(a, st);
}

extern "C" int b2n_fmlp_bwd(int d0, int d1, int hidden, int n_hidden, const float* const* W, const int* ldw, int out_dim,
                            int out_act, int64_t P, const float* y, int ldy, const float* g_y, int ldgy,
                            const void* h_planes, void* dz_out, void* dz_h, float* g_x0, int ldg0, float* g_x1, int ldg1,
                            void* work8, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  Args a{};
  int rc = fill_args(&a, false, nullptr, 0, d0, nullptr, 0, d1, hidden, n_hidden, W, ldw, nullptr, out_dim, out_act, P);
  if (rc) return rc;
  B2N_REQUIRE(g_y && ldgy >= out_dim && h_planes && dz_out && dz_h && work8, "null pointer");
  B2N_REQUIRE(out_act == B2N_ACT_NONE || (y && ldy >= out_dim), "activation derivative needs the forward output");
  B2N_REQUIRE((!g_x0 || ldg0 >= d0) && (!g_x1 || ldg1 >= d1), "gradient row too narrow");
  a.y_out = y, a.ldy = ldy, a.g_y = g_y, a.ldgy = ldgy, a.hplanes = (op16*)h_planes;
  a.dz_out = (op16*)dz_out, a.dz_h = (op16*)dz_h, a.g_x0 = g_x0, a.ldg0 = ldg0, a.g_x1 = g_x1, a.ldg1 = ldg1;
  a.work = (unsigned int*)work8;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(a.work, 0, 8, st) != cudaSuccess) return check_launch("b2n_fmlp_bwd (memset)");
  {
    const int64_t n = P * out_dim;
    const unsigned grid = (unsigned)((n + 1023) / 1024 < (int64_t)kSMs * 8 ? (n + 1023) / 1024 : (int64_t)kSMs * 8);
    k_fmlp_absmax<<<grid, 256, 0, st>>>(g_y, ldgy, out_dim, P, a.work, g_active_rows);
  }
  const bool small_in = d0 + d1 <= 32, small_out = out_dim <= 16;
  if (hidden == 64) {
    if (small_in) return small_out ? launch_bwd<64, 2, 2>(a, st) : launch_bwd<64, 2, 8>(a, st);
    return small_out ? launch_bwd<64, 6, 2>(a, st) : launch_bwd<64, 6, 8>(a, st);
  }
  if (small_in) return small_out ? launch_bwd<128, 2, 2>(a, st) : launch_bwd<128, 2, 8>(a, st);
  return small_out ? launch_bwd<128, 6, 2>(a, st) : launch_bwd<128, 6, 8>(a, st);
}

extern "C" int b2n_fmlp_wgrad(int n_layers, const void* const* dz, const int* ldz, const int* rows, const void* const* in,
                              const int* ldi, const int* k, float* const* dW, const int* lddw, const int* rows_valid,
                              const int* k_valid, float* const* db, int64_t P, const float* scale, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  B2N_REQUIRE(n_layers >= 1 && n_layers <= MAX_HID + 1, "1..4 layers");
  B2N_REQUIRE(dz && ldz && rows && in && ldi && k && dW && lddw && rows_valid && k_valid && db, "null pointer");
  if (P == 0) return B2N_OK;
  WgArgs a{};
  for (int l = 0; l < n_layers; ++l) {
    B2N_REQUIRE(dz[l] && in[l] && dW[l], "null plane");
    B2N_REQUIRE(rows[l] % 16 == 0 && rows[l] >= 16 && rows[l] <= WG_MAXW && k[l] % 16 == 0 && k[l] >= 16 && k[l] <= WG_MAXW,
                "plane widths must be multiples of 16 in [16, 128]");
    B2N_REQUIRE((rows[l] / 16) * ((k[l] + 63) / 64) <= WG_THREADS / 32, "tile count exceeds the CTA");
    B2N_REQUIRE(ldz[l] >= rows[l] && ldi[l] >= k[l] && ldz[l] % 8 == 0 && ldi[l] % 8 == 0, "plane rows must be 16-byte aligned");
    B2N_REQUIRE(rows_valid[l] <= rows[l] && k_valid[l] <= k[l] && lddw[l] >= k_valid[l], "bad gradient shape");
    a.L[l] = WgLayer{(const op16*)dz[l], ldz[l], rows[l], (const op16*)in[l], ldi[l], k[l], dW[l], lddw[l], rows_valid[l],
                     k_valid[l], db[l]};
  }
  a.P = P, a.scale = scale, a.rows = g_active_rows;
  cudaFuncSetAttribute(k_fmlp_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM);
  const int64_t n_tiles = (P + WG_TILE - 1) / WG_TILE;
  dim3 grid((unsigned)(n_tiles < kSMs ? n_tiles : kSMs), (unsigned)n_layers);
  k_fmlp_wgrad<<<grid, WG_THREADS, WG_SMEM, (cudaStream_t)stream>>>(a);
  return check_launch("b2n_fmlp_wgrad");
}

