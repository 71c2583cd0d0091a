// Weight / bias gradients of the 256-wide vanilla NeRF decoder on tcgen05 (autograd of NeRFDecoder.forward,
// src/decoders.py:68-87, w.r.t. the nn.Linear parameters):
//     dW_l[256 x 256] = dZ_l^T H_{l-1}   (contraction over all P points),   db_l = column sums of dZ_l
// for the eight 256 x 256 layers (trunk layers 1..7 and the feature layer) in ONE launch.  dZ_l / H_l are the bf16
// [P][256] planes written by b2n_nerf_mlp_bwd / b2n_nerf_mlp_fwd, i.e. POINT-major: the contraction index is the row.
// That is the MN-major operand form of tcgen05.mma (DESIGN.md 7c): a TMA box {64 columns, 64 points} with
// SWIZZLE_128B is already a valid operand block, so there is no transpose anywhere.
//
// grid = (splits of P, jobs).  A CTA owns one (job, P-slice): it streams 64-point stages (dZ tile 64 x 256 and H tile
// 64 x 256 = 64 KB, 3-stage TMA/mbarrier ring), issues 8 MMAs per stage (M = 128 per dZ column half, N = 256, K = 16)
// into a 256 x 256 fp32 accumulator that fills the 512 TMEM columns, and at the end adds it to dW with red.global.
// The eight warps that drain TMEM at the end spend the main loop summing the columns of the dZ tiles (bias gradients),
// so the dZ planes are read exactly once.  Jobs without a GEMM (the view-layer and layer-0 planes, whose weight
// gradients have other shapes) only do the column sums.
// The work is HBM-bound (115 FLOP/B): 2.15 GB at P = 262 144.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <string.h>
#include "b2n_common.cuh"
#include "b2n_tc.cuh"

namespace b2n {
namespace wg256 {

using namespace tc;

constexpr int TP = 64;                         // points per stage
constexpr int BLK = TP * 128;                  // one 64-column operand block: 64 rows x 128 B
constexpr int STAGE_BYTES = 8 * BLK;           // dZ: 4 blocks, H: 4 blocks
constexpr int N_STAGES = 3;
constexpr int OFF_BAR = N_STAGES * STAGE_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 128;
constexpr int N_THREADS = 320;                 // warp 0 TMA producer, warp 1 MMA issuer, warps 2..9 column sums + drain
constexpr int MAX_JOBS = 12;

// D[128 * m_halves][n_cols] += A^T B over the points, A / B = planes (tensor map index, slot)
struct Job {
  int a_map, a_slot;        // A operand (its columns become the rows of D): 128 * m_halves columns
  int m_halves;             // 2: 256 columns of A, 1: the first 128
  int b_map, b_slot;        // B operand; b_map < 0: column sums only
  int n_cols;               // columns of B taken: 64, 128 or 256 (beyond the tensor width the TMA zero-fills)
  float* dW;                // [128 * m_halves][n_cols] fp32 or null
  float* db;                // fp32 [bias_cols] or null: column sums of the A plane
  int bias_cols;
};
struct Args {
  Job job[MAX_JOBS];
  int64_t P;
  int64_t rows_per_split;   // multiple of TP
  int* err;
  int fp16;                 // operand planes are IEEE fp16 (the fused 128-wide MLPs) instead of bf16 (the 256-wide decoder)
  const float* scale;       // device scalar S: the dZ planes hold S * dZ, results are divided by S (null: 1)
  const int* rows;          // optional device-side row count; rows up to the next multiple of 64 behind it are zero in the planes
};

__global__ void __launch_bounds__(N_THREADS, 1)
k_wgrad256(const Args a, const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
           const __grid_constant__ CUtensorMap tm2, const __grid_constant__ CUtensorMap tm3) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  const uint32_t bar_full = s32(bars + 0), bar_empty = s32(bars + 3), bar_done = s32(bars + 6);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(bars + 8);
  const Job job = a.job[blockIdx.y];
  const bool gemm = job.b_map >= 0;
  const int dz_blocks = 2 * job.m_halves, in_blocks = gemm ? job.n_cols >> 6 : 0;
  const int64_t P_eff = clamp_rows(a.P, a.rows);
  const int64_t row_begin = (int64_t)blockIdx.x * a.rows_per_split;
  int64_t row_end = row_begin + a.rows_per_split;
  if (row_end > P_eff) row_end = P_eff;
  const int n_steps = row_begin < P_eff ? (int)((row_end - row_begin + TP - 1) / TP) : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < N_STAGES; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, gemm ? 9 : 8);
    }
    mbar_init(bar_done, 1);
    *abort_flag = 0;
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(s32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      for (int it = 0; it < n_steps; ++it) {
        const int st = it % N_STAGES;
        if (!mbar_wait(bar_empty + 8 * st, ((it / N_STAGES) & 1) ^ 1, abort_flag, a.err, 1)) break;
        const uint32_t bytes = (uint32_t)(dz_blocks + in_blocks) * BLK;
        mbar_expect_tx(bar_full + 8 * st, bytes);
        const int r0 = (int)(row_begin + (int64_t)it * TP);
        const uint32_t base = s32(smem + st * STAGE_BYTES);
        auto pick = [&](int i) { return i == 0 ? &tm0 : (i == 1 ? &tm1 : (i == 2 ? &tm2 : &tm3)); };
        const CUtensorMap* ta = pick(job.a_map);
        for (int b = 0; b < dz_blocks; ++b) tma_load_3d(base + b * BLK, ta, 64 * b, r0, job.a_slot, bar_full + 8 * st);
        if (gemm) {
          const CUtensorMap* tb = pick(job.b_map);
          for (int b = 0; b < in_blocks; ++b) tma_load_3d(base + (4 + b) * BLK, tb, 64 * b, r0, job.b_slot, bar_full + 8 * st);
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (gemm) {
      const uint32_t idesc = umma_idesc(a.fp16 ? Fmt::F16 : Fmt::BF16, Major::MN, job.n_cols, 128);
      for (int it = 0; it < n_steps; ++it) {
        const int st = it % N_STAGES;
        if (!mbar_wait(bar_full + 8 * st, (it / N_STAGES) & 1, abort_flag, a.err, 2)) break;
        tc_fence_after();
        if (lane == 0) {
          const uint32_t base = s32(smem + st * STAGE_BYTES);
#pragma unroll
          for (int kk = 0; kk < TP / 16; ++kk) {
            for (int mh = 0; mh < job.m_halves; ++mh) {
              const uint64_t ad = umma_desc_mn(base + mh * 2 * BLK + kk * 2048, BLK);      // dZ columns 128*mh .. +127
              const uint64_t bd = umma_desc_mn(base + 4 * BLK + kk * 2048, BLK);           // input columns 0 .. n_cols-1
              tc_mma(tmem + mh * 256, ad, bd, idesc, (it > 0 || kk > 0) ? 1u : 0u);
            }
          }
          tc_commit(bar_empty + 8 * st);
          if (it + 1 == n_steps) tc_commit(bar_done);
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ column sums (main loop) + accumulator drain ================================
    const int c = threadIdx.x - 64;             // 0..255: the dZ column this thread sums
    float colsum = 0.f;
    const float inv_s = a.scale ? 1.f / __ldg(a.scale) : 1.f;
    for (int it = 0; it < n_steps; ++it) {
      const int st = it % N_STAGES;
      if (!mbar_wait(bar_full + 8 * st, (it / N_STAGES) & 1, abort_flag, a.err, 3)) break;
      if (job.db && c < job.bias_cols) {
        const unsigned char* blk = smem + st * STAGE_BYTES + (c >> 6) * BLK + (c & 7) * 2;
        const int ch = (c & 63) >> 3;
        float s = 0.f;
#pragma unroll 8
        if (a.fp16) {
#pragma unroll 8
          for (int r = 0; r < TP; ++r) s += __half2float(*reinterpret_cast<const __half*>(blk + r * 128 + ((ch ^ (r & 7)) << 4)));
        } else {
#pragma unroll 8
          for (int r = 0; r < TP; ++r)
            s += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(blk + r * 128 + ((ch ^ (r & 7)) << 4)));
        }
        colsum += s;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty + 8 * st);
    }
    if (job.db && n_steps > 0 && c < job.bias_cols) atomicAdd(job.db + c, colsum * inv_s);
    if (gemm && n_steps > 0 && mbar_wait(bar_done, 0, abort_flag, a.err, 4)) {
      tc_fence_after();
      const int q = warp & 3;                   // TMEM lane quarter this warp may read
      const int mh = (warp - 2) >> 2;           // which dZ column half (accumulator columns 256*mh ..)
      const int n = 128 * mh + 32 * q + lane;   // output neuron = dW row
      float* drow = job.dW + (size_t)n * job.n_cols;
      for (int c0 = 0; mh < job.m_halves && c0 < job.n_cols; c0 += 32) {
        uint32_t v[32];
        tc_ld32(tmem + ((uint32_t)(32 * q) << 16) + 256 * mh + c0, v);
        tc_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          atomicAdd(reinterpret_cast<float4*>(drow + c0 + j),
                    make_float4(__uint_as_float(v[j]) * inv_s, __uint_as_float(v[j + 1]) * inv_s,
                                __uint_as_float(v[j + 2]) * inv_s, __uint_as_float(v[j + 3]) * inv_s));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
static bool make_map(CUtensorMap* m, const void* planes, int64_t P, int n_slots, int width = 256, bool fp16 = false) {
  if (!planes) return true;             // unused map slot
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)width, (cuuint64_t)P, (cuuint64_t)n_slots};
  const cuuint64_t strides[2] = {(cuuint64_t)width * 2, (cuuint64_t)P * width * 2};
  const cuuint32_t box[3] = {64, TP, 1};   // planes narrower than a 64-column block: the TMA zero-fills the rest
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(planes), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace wg256
}  // namespace b2n

using namespace b2n;
using namespace b2n::wg256;

// dz_planes / fwd_planes: bf16 [10][P][256] as written by b2n_nerf_mlp_bwd / b2n_nerf_mlp_fwd; x_bf16: bf16 [P][kx]
// (encoded positions zero-padded to kx = 64 or 128 columns), d_bf16: bf16 [P][64] (encoded directions, zero-padded).
// All outputs fp32 and ACCUMULATED (zero them first):
//   dW    [8][256][256]  dW[l-1] = dZ_l^T H_{l-1} for trunk layers l = 1..7 (skip layer 4: its first 256 input columns),
//                        dW[7] = dZ_feat^T H_7 (feature layer)
//   dW0   [256][kx]      dZ_0^T x           dW4x [256][kx]   dZ_4^T x  (x part of the skip layer)
//   dWv_h [128][256]     dZ_view^T H_8      dWv_d [128][64]  dZ_view^T d
//   db    [10][256]      column sums of every dZ plane by slot (0 view, 1 feature, 2..9 = trunk layers 7..0)
// x_bf16 / d_bf16 (and their outputs) may be NULL: those products are then left to the caller.
extern "C" int b2n_nerf_mlp_wgrad(const void* dz_planes, const void* fwd_planes, const void* x_bf16, int kx,
                                  const void* d_bf16, int64_t P, float* dW, float* dW0, float* dW4x, float* dWv_h,
                                  float* dWv_d, float* db, int* err_flag, b2n_stream_t stream) {
  B2N_REQUIRE(dz_planes && fwd_planes && dW && db && err_flag, "null pointer");
  B2N_REQUIRE(P >= TP, "needs at least 64 points");
  B2N_REQUIRE(!x_bf16 || ((kx == 64 || kx == 128) && dW0 && dW4x), "x operand: kx must be 64 or 128, outputs required");
  B2N_REQUIRE(!d_bf16 || (dWv_h && dWv_d), "d operand: outputs required");
  alignas(64) CUtensorMap tm_dz, tm_in, tm_x, tm_d;
  memset(&tm_dz, 0, sizeof(tm_dz)), memset(&tm_in, 0, sizeof(tm_in)), memset(&tm_x, 0, sizeof(tm_x)), memset(&tm_d, 0, sizeof(tm_d));
  B2N_REQUIRE(make_map(&tm_dz, dz_planes, P, 10) && make_map(&tm_in, fwd_planes, P, 10), "cuTensorMapEncodeTiled failed");
  B2N_REQUIRE(!x_bf16 || make_map(&tm_x, x_bf16, P, 1, kx), "cuTensorMapEncodeTiled failed (x)");
  B2N_REQUIRE(!d_bf16 || make_map(&tm_d, d_bf16, P, 1, 64), "cuTensorMapEncodeTiled failed (d)");
  Args a{};
  int n = 0;
  // tensor maps: 0 = dZ planes, 1 = forward planes, 2 = x, 3 = d
  for (int l = 1; l <= 7; ++l)
    a.job[n++] = Job{0, 9 - l, 2, 1, l - 1, 256, dW + (size_t)(l - 1) * 65536, db + (size_t)(9 - l) * 256, 256};
  a.job[n++] = Job{0, 1, 2, 1, 7, 256, dW + (size_t)7 * 65536, db + 256, 256};
  if (x_bf16) {
    a.job[n++] = Job{0, 9, 2, 2, 0, kx, dW0, db + (size_t)9 * 256, 256};
    a.job[n++] = Job{0, 5, 2, 2, 0, kx, dW4x, nullptr, 0};
  } else {
    a.job[n++] = Job{0, 9, 2, -1, 0, 256, nullptr, db + (size_t)9 * 256, 256};   // layer-0 plane: bias sums only
  }
  if (d_bf16) {
    a.job[n++] = Job{0, 0, 1, 1, 8, 256, dWv_h, db, 128};
    a.job[n++] = Job{0, 0, 1, 3, 0, 64, dWv_d, nullptr, 0};
  } else {
    a.job[n++] = Job{0, 0, 1, -1, 0, 256, nullptr, db, 128};                     // view-layer plane: bias sums only
  }
  a.P = P, a.err = err_flag;
  int splits = (2 * kSMs) / n;                             // ~2 CTAs' worth of jobs per SM (the narrow jobs are short)
  const int64_t max_splits = (P + TP - 1) / TP;
  if (splits > max_splits) splits = (int)max_splits;
  if (splits < 1) splits = 1;
  a.rows_per_split = ((P + splits - 1) / splits + TP - 1) / TP * TP;
  cudaFuncSetAttribute(k_wgrad256, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  k_wgrad256<<<dim3((unsigned)splits, (unsigned)n), N_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a, tm_dz, tm_in, tm_x, tm_d);
  return check_launch("b2n_nerf_mlp_wgrad");
}

// Weight / bias gradients of the 128-wide fused MLPs (DeformationNetwork: b2n_fmlp_*) through the same kernel.
// dz_h fp16 [n_hidden][P][128], dz_out fp16 [P][out_pad], h_planes fp16 [n_hidden][P][128], xin fp16 [P][in_pad] as written
// by b2n_fmlp_fwd / b2n_fmlp_bwd.  ACCUMULATES (fp32): dW0 [128][128] = dZ_0^T xin (columns >= in_pad stay 0),
// dWh [n_hidden-1][128][128] = dZ_l^T H_{l-1}, dWoT [128][64] = H_last^T dZ_out (the TRANSPOSED output-layer gradient,
// columns >= out_pad stay 0), db_h [n_hidden][128] = column sums of the hidden dZ planes.
extern "C" int b2n_fmlp_wgrad_tc(const void* dz_h, const void* dz_out, const void* h_planes, const void* xin, int64_t P,
                                 int n_hidden, int in_pad, int out_pad, float* dW0, float* dWh, float* dWoT, float* db_h,
                                 int* err_flag, const float* scale, b2n_stream_t stream) {
  B2N_REQUIRE(dz_h && dz_out && h_planes && xin && dW0 && dWoT && db_h && err_flag, "null pointer");
  B2N_REQUIRE(n_hidden >= 1 && n_hidden <= 3 && (n_hidden == 1 || dWh), "1..3 hidden layers");
  B2N_REQUIRE(P >= TP && (in_pad == 32 || in_pad == 96) && (out_pad == 16 || out_pad == 64), "bad plane widths");
  alignas(64) CUtensorMap tm[4];
  memset(tm, 0, sizeof(tm));
  B2N_REQUIRE(make_map(&tm[0], dz_h, P, n_hidden, 128, true) && make_map(&tm[1], h_planes, P, n_hidden, 128, true) &&
                  make_map(&tm[2], xin, P, 1, in_pad, true) && make_map(&tm[3], dz_out, P, 1, out_pad, true),
              "cuTensorMapEncodeTiled failed");
  Args a{};
  int n = 0;
  a.job[n++] = Job{0, 0, 1, 2, 0, in_pad <= 64 ? 64 : 128, dW0, db_h, 128};
  for (int l = 1; l < n_hidden; ++l)
    a.job[n++] = Job{0, l, 1, 1, l - 1, 128, dWh + (size_t)(l - 1) * 16384, db_h + (size_t)l * 128, 128};
  a.job[n++] = Job{1, n_hidden - 1, 1, 3, 0, 64, dWoT, nullptr, 0};
  a.P = P, a.err = err_flag, a.fp16 = 1, a.scale = scale, a.rows = g_active_rows;
  int splits = (2 * kSMs) / n;
  const int64_t max_splits = (P + TP - 1) / TP;
  if (splits > max_splits) splits = (int)max_splits;
  if (splits < 1) splits = 1;
  a.rows_per_split = ((P + splits - 1) / splits + TP - 1) / TP * TP;
  cudaFuncSetAttribute(k_wgrad256, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  k_wgrad256<<<dim3((unsigned)splits, (unsigned)n), N_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a, tm[0], tm[1], tm[2], tm[3]);
  return check_launch("b2n_fmlp_wgrad_tc");
}
