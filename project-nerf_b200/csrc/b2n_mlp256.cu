// 256-wide vanilla NeRF decoder (NeRFDecoder.forward / backward, src/decoders.py:68-87) on the
// 5th-gen tensor cores: tcgen05.mma (cta_group::1, M=128, N=128, K=16, bf16 x bf16 -> fp32 in TMEM).
//
//   h = x; for i in 0..7: (i == 4: h = [h, x]); h = relu(W_i h + b_i)
//   sigma = relu(w_s h + b_s); feat = W_f h + b_f; hv = relu(W_v [feat, d] + b_v); rgb = sigmoid(W_c hv + b_c)
//
// One persistent CTA per SM works on PAIRS of 128-point tiles whose activations never leave the
// SM: they sit in shared memory as bf16 in the canonical K-major SWIZZLE_128B UMMA layout (4
// k-blocks of 128 rows x 128 B per tile) and are the A operand of the next layer.
//
// Schedule (measured: reading a 128 x 256 fp32 accumulator out of TMEM costs about as many cycles
// as the MMAs that produced it, so the two must overlap): the tiles are processed in LOCK-STEP
// BUT ALTERNATING -- while the tensor core runs layer l of tile B, all eight epilogue warps drain
// layer l of tile A (TMEM -> +bias/ReLU -> bf16 -> swizzled st.shared), and vice versa:
//       tensor : MMA(A,l)  MMA(B,l)  MMA(A,l+1)  MMA(B,l+1) ...
//       epilog :           EPI(A,l)  EPI(B,l)    EPI(A,l+1) ...
// Accumulators: tile A in TMEM columns 0..255, tile B in 256..511 (all 512 columns).
//
// Weights are pre-packed once per optimizer step (b2n_nerf_mlp_pack*) into a stream of 16 KB
// chunks that are byte images of B operand tiles ([128 n-rows x 64 k] bf16, same swizzle), so
// the producer needs no tensor map: one elected thread issues one 1-D bulk copy (cp.async.bulk
// -> mbarrier complete_tx) per chunk into a 4-stage ring (the layer is streamed once per tile;
// L2 serves it, measured L2 throughput < 20 %).
//
// Warp roles (11 warps): warp 0 = weight producer, warp 1 = TMEM allocator + MMA issuer (one
// elected thread), warps 2..9 = epilogue: warp_id % 4 selects the TMEM lane quarter (rows), warps
// 2-5 take accumulator columns 0..127 and warps 6-9 columns 128..255 of the tile being drained,
// warp 10 = plane store (training: TMA tensor stores of the finished activation tiles).
// The 256->1 density head and the 128->3 colour head are dot products inside the epilogue.
//
// DEFAULT SCHEDULE = CTA PAIRS (template parameter CTA2, b2n_debug_mlp256_set_pair): the kernel is launched as clusters
// of two CTAs on an SM pair and every MMA is a cta_group::2 instruction (M = 256: this CTA's 128-row tile + the
// peer's; N = the layer width) issued by the leader.  Each CTA stages only ITS 128 output rows of every weight
// chunk (TMA tile loads whose bytes are credited to the leader's barrier), a layer whose k-chunks fit in the ring is
// streamed ONCE per tile pair (tile 1 re-reads the slots tile 0 used), commits multicast to both CTAs, and the
// peer's idle MMA warp relays "my tile is in place" to the leader with a single remote arrive.  Weight traffic per
// CTA drops 4x, results are bit-identical to the single-CTA schedule (tests).  Measured at P = 262 144 (C1, kernel
// times inside a training loop): training forward 0.57 -> 0.44 ms, backward chain 0.56 -> 0.335 ms (869 TFLOP/s = 62 %
// of the sustained cuBLAS bf16 rate), inference forward 0.49 -> 0.37 ms (60 %).
// What the B2N_TRACE timeline (tools/kbench.py mlp256t) shows is left: each tile runs the serial chain
//   MMAs of the step (act ready -> accumulator seen by the epilogue: ~2900 cycles, 2048 of them tensor time)
//   -> drain (TMEM reads at 64 B/cycle: >= 2000 cycles) -> slower of the two CTAs' epilogues + relay (300..2600)
// = ~7400 cycles per step with two tiles in flight, i.e. the tensor pipe is busy 55 % of a steady-state step.  The next
// step is ONE tile per CTA with a double-buffered accumulator and the act tile handed over per 64-column k-block, so
// that the MMAs of layer l+1 start a quarter of a drain after layer l's accumulator completes (DESIGN.md).
//
// The notes below describe the single-CTA schedule (B2N_MLP256_PAIR=0), kept for A/B timing:
//
// Measured on B200 (tools/kbench.py mlp256, P = 2^20): 727 TFLOP/s = 52 % of the sustained cuBLAS bf16
// peak.  Per layer and tile pair: tensor work 4096 cycles, epilogue 5300 cycles (TMEM drain ~64 B/cycle
// plus 64 KB of swizzled stores), period 8800 cycles, independent of the number of CTAs (not L2 bound).
// The binding resource is SHARED-MEMORY BANDWIDTH: with both operands in smem an M=128,N=128,K=16 MMA
// reads 8 KB per 64 cycles (= the 128 B/cycle limit) while the weight ring and the epilogue write another
// 192 KB per tile and layer.  Next step (round 2): cta_group::2 (each CTA supplies half of B) or the A
// operand in TMEM.
//
// Every mbarrier wait is bounded; on time-out the CTA raises an abort flag, stores an error code
// and drains, so a protocol bug cannot hang the GPU.
#include <cuda.h>
#pragma nv_diag_suppress 128   // "loop is not reachable": the single-CTA MMA loop in the CTA-pair instantiations
#include <stdlib.h>
#include <string.h>
#include <cuda_bf16.h>
#include "b2n_common.cuh"
#include "b2n_tc.cuh"

namespace b2n {
namespace m256 {

using namespace tc;

constexpr int HID = 256;
constexpr int KBLK_BYTES = 128 * 128;          // one k-block of one tile: 128 rows x 64 bf16
constexpr int ACT_BYTES = 4 * KBLK_BYTES;      // 128 x 256 bf16
constexpr int CHUNK_BYTES = 128 * 128;         // one weight chunk: 128 n-rows x 64 k bf16
constexpr int N_STAGES = 4;
constexpr int OFF_ACT = 0;                     // [2 tiles][ACT_BYTES]
constexpr int OFF_AUX = OFF_ACT + 2 * ACT_BYTES;       // [2 tiles][KBLK_BYTES]   x_enc, later d_enc
constexpr int OFF_RING = OFF_AUX + 2 * KBLK_BYTES;     // [N_STAGES][CHUNK_BYTES]
constexpr int OFF_VEC = OFF_RING + N_STAGES * CHUNK_BYTES;   // 256 floats bias + 384 floats head weights / scratch
constexpr int OFF_BAR = OFF_VEC + (256 + 384) * 4;
constexpr int SMEM_BYTES = OFF_BAR + 208;
static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");

constexpr int N_THREADS = 352;          // 11 warps: producer, MMA, 8 x epilogue, plane store
constexpr int EPI_THREADS = 256;
constexpr int MAX_STEPS = 14, MAX_CHUNKS = 96;

enum { EPI_RELU = 0, EPI_RELU_SIGMA = 1, EPI_LINEAR = 2, EPI_VIEW_RGB = 3,
       EPI_B_LINEAR = 4, EPI_B_MASK = 5, EPI_B_MASK_SIGMA = 6 };

struct Step {
  int n_act;     // k-chunks taken from the activation buffer (0, 2 or 4)
  int aux_k16;   // k16 sub-steps taken from the aux buffer (0 = none, 4 = 64 columns, 2 = 32 columns)
  int n;         // output width of the step (256 or 128)
  int epi;       // epilogue kind
  int bias_off;  // fwd: offset into the bias vector; bwd: index of the gating forward plane
  int save_slot; // index of the saved plane (or -1)
  int acc_in;    // 1: the MMAs accumulate onto what the previous (partial) step left in TMEM
  int partial;   // 1: no drain -- the epilogue only re-stages the aux block for the next step
  int restage;   // aux block content for the NEXT step: 0 keep, 1 x_enc[:, 0:64], 2 x_enc[:, 64:128], 3 d_enc
  int tma;       // 1: the saved plane of this step is written by a TMA tensor store of the activation tile
                 //    (issued by the MMA warp at the next step) instead of st.global from the epilogue registers
};
struct Plan {
  int n_steps;
  Step s[MAX_STEPS];
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// stage 4 of the 8 sixteen-byte chunks (c0 .. c0+3) of one fp32 input row as bf16 into an aux k-block
__device__ __forceinline__ void stage_row(const float* __restrict__ src, int width, bool valid, unsigned char* blk,
                                          int r, int c0) {
#pragma unroll 1
  for (int c = c0; c < c0 + 4; ++c) {
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = 8 * c + j;
      f[j] = (valid && col < width) ? __ldg(src + col) : 0.f;
    }
    *reinterpret_cast<uint4*>(blk + swz(r, c)) =
        make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
  }
}

// timeline of the third tile pair of CTA 0 (CTA 1 = the peer of CTA 0 with debug flag 32) (debug): prof[8 + (step * 2 + tile) * 16 + k] = clock64() at event k
#define B2N_TRACE(step, tile, k)                                                                     \
  do {                                                                                               \
    if (a.prof && blockIdx.x == ((a.dbg >> 5) & 1) && pair == pair_first + 2 * pair_step)             \
      a.prof[8 + ((step) * 2 + (tile)) * 16 + (k)] = clock64();                                       \
  } while (0)

struct FwdArgs {
  const float* x_enc; int pos_dim;
  const float* d_enc; int dir_dim;
  const unsigned char* packed;      // weight chunk stream
  const float* bias;                // concatenated biases, Step::bias_off indexes it
  const float* w_sigma;
  const float* w_rgb;
  const float* head_bias;           // device float[4]: b_sigma, b_rgb[0..2]
  int64_t P;
  float* rgb; float* sigma;
  __nv_bfloat16* save;              // [n_slots][P][256] or nullptr
  int* err;
  // backward only
  uint32_t* mask_out;               // fwd (training): [10][P][8] ReLU bit masks of the saved planes (bit c = plane[c] > 0)
  const uint32_t* mask_in;          // bwd: the same buffer (gates of the data-gradient chain)
  const float* g_rgb; const float* g_sigma;   // [P,3], [P]
  const float* rgb_out; const float* sigma_out;
  float* dz_small;                  // [P,4]: d(pre-sigmoid rgb)[3], d(pre-relu sigma)
  long long* prof;                  // optional [8] cycle counters of CTA 0 (b2n_debug_mlp256_prof)
  Plan plan;
  int use_tma;                      // the planes are written through the TMA tensor map passed next to this struct
  int dbg;                          // timing experiments (b2n_debug_mlp256_flags): 1 = epilogue skips the drain,
                                    // 2 = no MMAs are issued (weights still stream), 4 = no weight loads, 8 = no row loads / stores: results are garbage;
                                    // 16 = accumulate the role counters prof[0..7] (each costs a global read-modify-write on the role's
                                    // serial path: the B2N_TRACE timeline is only trustworthy without them)
};

// one out-of-line copy: the three call sites are off the hot loop, and inlining them grew the forward kernel
// by 850 instructions (measured: -8 % throughput, the epilogue is instruction-cache sensitive)
__device__ __noinline__ void restage_aux(const FwdArgs& a, int what, int64_t p, bool valid, unsigned char* aux, int r,
                                         int c0) {
  const float* src;
  int width;
  if (what == 1) src = a.x_enc + p * a.pos_dim, width = a.pos_dim < 64 ? a.pos_dim : 64;
  else if (what == 2) src = a.x_enc + p * a.pos_dim + 64, width = a.pos_dim - 64;
  else if (what == 3) src = a.d_enc + p * a.dir_dim, width = a.dir_dim;
  else return;
  stage_row(src, width, valid, aux, r, c0);
}

// WIDE: forward with 64 < pos_dim <= 96 (partial steps / aux swaps); the common instantiation carries none of that code
// CTA2: launched as clusters of two CTAs (one SM pair).  Every MMA is a cta_group::2 instruction issued by the
// leader (cluster rank 0) over BOTH CTAs' tiles: M = 256 (this CTA's 128 rows + the peer's), N = the whole layer
// width, each CTA staging only ITS half of every weight chunk (output rows 128*rank .. +127) -- per CTA that halves
// the weight-ring traffic and the B-operand reads, which is what bounds the single-CTA kernel (file header).
template <bool BWD, bool WIDE = false, bool CTA2 = false>
__global__ void __launch_bounds__(N_THREADS, 1) k_mlp256(const __grid_constant__ FwdArgs a, const __grid_constant__ CUtensorMap tmap_save,
                                                         const __grid_constant__ CUtensorMap tmap_w) {
  // tmap_save: 3-D map of the saved planes (cols, rows, slot), box 64 x 128 x 1, SWIZZLE_128B
  // tmap_w (CTA2 only): the packed weight stream, no swizzle (the stream
  //                     is already a byte image of the swizzled operand tiles): [bytes / 512][256 bf16], box 256 x 16
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  // The backward chain never uses the aux blocks (its steps read activations only): as a CTA pair it runs a 6-slot
  // weight ring over [aux | ring], so the first chunks of the next step are fetched while tile 1 still reads this one's
  constexpr int NST = (CTA2 && BWD) ? 6 : N_STAGES;
  constexpr int RING = (CTA2 && BWD) ? OFF_AUX : OFF_RING;
  const uint32_t bar_full = s32(bars + 0);     // [NST <= 8]
  const uint32_t bar_empty = s32(bars + 8);    // [NST <= 8]
  const uint32_t bar_acc = s32(bars + 16);     // [2] MMA -> epilogue: accumulators of tile t complete
  const uint32_t bar_act = s32(bars + 18);     // [2] epilogue -> MMA: A operand of tile t written, accumulator drained
  const uint32_t bar_st = s32(bars + 20);      // [2] store warp -> epilogue: the plane store has read tile t (it may be overwritten)
  const uint32_t bar_tail = s32(bars + 24);    // [2] epilogue -> store warp: the LAST step's output of tile t is in the act tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(bars + 23);
  float* vec = reinterpret_cast<float*>(smem + OFF_VEC);
  const uint32_t rank = CTA2 ? cluster_ctarank() : 0u;      // 0 = leader (issues the MMAs)

  if ((s32(smem) & 1023u) != 0) {  // SWIZZLE_128B operands need 1024-byte aligned tiles
    if (threadIdx.x == 0) atomicCAS(a.err, 0, 100);
    return;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < NST; ++i) mbar_init(bar_full + 8 * i, 1), mbar_init(bar_empty + 8 * i, 1);
    // CTA2: the leader's bar_act also collects ONE arrival from the peer CTA: the peer's (otherwise idle) MMA warp
    // waits for its own epilogue and relays.  (Cluster-scope release arrivals by the epilogue threads themselves
    // lagged the local ones by ~2500 cycles in the B2N_TRACE timeline.)
    for (int t = 0; t < 2; ++t) {
      mbar_init(bar_acc + 8 * t, 1);
      mbar_init(bar_act + 8 * t, (CTA2 && rank == 0) ? EPI_THREADS + 1 : EPI_THREADS);
      mbar_init(bar_st + 8 * t, 1);
      mbar_init(bar_tail + 8 * t, EPI_THREADS);
    }
    *abort_flag = 0;
    mbar_init_fence();
  }
  if (CTA2) {
    cluster_sync_all();                         // both CTAs resident, barriers initialised, before anything crosses over
    if (warp == 1) tmem_alloc2(s32(tmem_slot), 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
  } else {
    if (warp == 1) tmem_alloc(s32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  const uint32_t tmem = *tmem_slot;
  // tile pairs: a CTA owns pairs pair_first, pair_first + pair_step, ...; the two CTAs of a cluster walk the
  // consecutive pairs 2q, 2q+1 in lock-step (n_pairs is rounded up to even so both run the same number of rounds;
  // rows >= P are masked like the ragged tail of the last pair)
  const int64_t n_pairs = CTA2 ? 2 * ((a.P + 511) / 512) : (a.P + 255) / 256;
  const int64_t pair_first = CTA2 ? 2 * (int64_t)cluster_idx() + rank : (int64_t)blockIdx.x;
  const int64_t pair_step = CTA2 ? 2 * (int64_t)cluster_count() : (int64_t)gridDim.x;
  const Plan& plan = a.plan;

  if (warp == 0) {
    // ================================ weight producer ================================
    if (CTA2 && lane == 0) {
      // one ring slot per k-chunk: this CTA's 128 (64 for the 128-wide view layer) output rows of it; the bytes of
      // both CTAs are credited to the LEADER's bar_full, which its MMA thread waits on
      uint32_t use = 0;
      const uint32_t full_leader = mapa(bar_full, 0);
      for (int64_t pair = pair_first; pair < n_pairs; pair += pair_step) {
        int chunk0 = 0;                                           // first 16 KB chunk of the step in the packed stream
        for (int s = 0; s < plan.n_steps; ++s) {
          const int nkc = plan.s[s].n_act + (plan.s[s].aux_k16 ? 1 : 0), halves = plan.s[s].n / 128;
          const uint32_t bytes = halves == 2 ? CHUNK_BYTES : CHUNK_BYTES / 2;
          // a step whose k-chunks all fit in the ring is streamed ONCE: tile 1 re-uses the slots tile 0 read (the MMA
          // warp frees them after tile 1's pass), which halves the L2 traffic again and gives every load the time of
          // a whole tile pass to land; longer steps (skip layer, view layer) are streamed once per tile
          const int passes = nkc <= NST ? 1 : 2;
          for (int t = 0; t < passes; ++t) {
            for (int c = 0; c < nkc; ++c, ++use) {
              const uint32_t st = use % NST, ph = (use / NST) & 1;
              if (!mbar_wait(bar_empty + 8 * st, ph ^ 1, abort_flag, a.err, 1)) goto prod_done;
              if (a.dbg & 4) {
                if (rank == 0) mbar_arrive(bar_full + 8 * st);
                continue;
              }
              if (rank == 0) mbar_expect_tx(bar_full + 8 * st, 2 * bytes);
              const uint32_t dst = s32(smem + RING + st * CHUNK_BYTES);
              // tensor-map rows are 512 B: a 16 KB chunk = 32 rows, one box = 16 rows = 8 KB
              const int row = halves == 2 ? (chunk0 + 2 * c + (int)rank) * 32 : (chunk0 + c) * 32 + 16 * (int)rank;
              tma_load_2d_pair(dst, &tmap_w, 0, row, full_leader + 8 * st);
              if (halves == 2) tma_load_2d_pair(dst + CHUNK_BYTES / 2, &tmap_w, 0, row + 16, full_leader + 8 * st);
            }
          }
          chunk0 += nkc * halves;
        }
      }
    } else if (!CTA2 && lane == 0) {
      uint32_t use = 0;  // running chunk counter (ring position)
      for (int64_t pair = pair_first; pair < n_pairs; pair += pair_step) {
        const unsigned char* step_src = a.packed;
        for (int s = 0; s < plan.n_steps; ++s) {
          const int nch = (plan.s[s].n_act + (plan.s[s].aux_k16 ? 1 : 0)) * (plan.s[s].n / 128);
          for (int t = 0; t < 2; ++t) {        // the layer is streamed once per tile
            const unsigned char* src = step_src;
            for (int c = 0; c < nch; ++c, ++use) {
              const uint32_t st = use % NST, ph = (use / NST) & 1;
              if (!mbar_wait(bar_empty + 8 * st, ph ^ 1, abort_flag, a.err, 1)) goto prod_done;
              if (a.dbg & 4) {
                mbar_arrive(bar_full + 8 * st);
                src += CHUNK_BYTES;
                continue;
              }
              mbar_expect_tx(bar_full + 8 * st, CHUNK_BYTES);
              bulk_g2s(s32(smem + RING + st * CHUNK_BYTES), src, CHUNK_BYTES, bar_full + 8 * st);
              src += CHUNK_BYTES;
            }
          }
          step_src += (size_t)nch * CHUNK_BYTES;
        }
      }
    }
  prod_done:;
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    // The whole warp walks the (warp-uniform) schedule; one elected lane issues the tcgen05 ops.
    {
      uint32_t use = 0, act_phase[2] = {0, 0};
      const uint32_t idesc = umma_idesc(Fmt::BF16, Major::K, 128, 128);
      const uint32_t ring0 = s32(smem + RING), act0 = s32(smem + OFF_ACT), aux0 = s32(smem + OFF_AUX);
      for (int64_t pair = pair_first; pair < n_pairs; pair += pair_step) {
        for (int s = 0; s < plan.n_steps; ++s) {
          const int n_act = plan.s[s].n_act, aux_k16 = plan.s[s].aux_k16;
          const int nkc = n_act + (aux_k16 ? 1 : 0), halves = plan.s[s].n / 128;
          const bool acc_in = WIDE && plan.s[s].acc_in != 0;
          for (int t = 0; t < 2; ++t) {
            long long t0 = clock64();
            if (lane == 0) B2N_TRACE(s, t, 3);
            if (!mbar_wait(bar_act + 8 * t, act_phase[t] & 1, abort_flag, a.err, 2)) goto mma_done;
            if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && lane == 0) a.prof[0] += clock64() - t0;   // waiting for the epilogue
            if (lane == 0) B2N_TRACE(s, t, 4);
            ++act_phase[t];
            tc_fence_after();
            const uint32_t d_tmem = tmem + t * 256;
            if (lane == 0) B2N_TRACE(s, t, 13);
            if (CTA2) {
              // leader: one M = 256 x N = layer-width MMA per k16 over both CTAs' tiles; the peer's warp only does the
              // plane stores of its own tile
              if (rank == 0) {
                const uint32_t idesc2 = umma_idesc(Fmt::BF16, Major::K, plan.s[s].n, 256);
                const bool shared = nkc <= NST;      // both tiles read the same ring slots (see the producer)
                const uint32_t use0 = use;
                for (int c = 0; c < nkc; ++c) {
                  const bool from_aux = c >= n_act;
                  const int nk = from_aux ? aux_k16 : 4;
                  const uint64_t adesc = umma_desc(from_aux ? aux0 + t * KBLK_BYTES : act0 + t * ACT_BYTES + c * KBLK_BYTES);
                  const uint32_t st = (use0 + c) % NST, ph = ((use0 + c) / NST) & 1;
                  // tile 1 of a shared step reads the slots tile 0 has already waited for
                  if (!(shared && t == 1)) {
                    if (!mbar_wait(bar_full + 8 * st, ph, abort_flag, a.err, 3)) goto mma_done;
                    tc_fence_after();
                  }
                  if (lane == 0 && c == 0) B2N_TRACE(s, t, 5);
                  const uint64_t bdesc = umma_desc(ring0 + st * CHUNK_BYTES);
                  if (elect_one()) {
                    if (a.dbg & 2) {
                    } else if (nk == 4) {
#pragma unroll
                      for (int k = 0; k < 4; ++k)
                        tc_mma2(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc2, (acc_in || c > 0 || k > 0) ? 1u : 0u);
                    } else {
#pragma unroll
                      for (int k = 0; k < 2; ++k)
                        tc_mma2(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc2, (acc_in || c > 0 || k > 0) ? 1u : 0u);
                    }
                    if (!shared || t == 1) tc_commit2(bar_empty + 8 * st);   // frees the slot in BOTH CTAs
                  }
                  __syncwarp();
                }
                if (!shared || t == 1) use = use0 + nkc;
                if (lane == 0) B2N_TRACE(s, t, 6);
                if (elect_one()) tc_commit2(bar_acc + 8 * t);
                __syncwarp();
              } else {
                // peer: its tile is in place (acquired above); tell the leader, whose MMAs read both CTAs' tiles
                if (elect_one()) mbar_arrive_cluster(mapa(bar_act, 0) + 8 * t);
                __syncwarp();
              }
              continue;
            }
            for (int c = 0; c < nkc; ++c) {
              const bool from_aux = c >= n_act;
              const int nk = from_aux ? aux_k16 : 4;
              const uint64_t adesc = umma_desc(from_aux ? aux0 + t * KBLK_BYTES : act0 + t * ACT_BYTES + c * KBLK_BYTES);
              for (int h = 0; h < halves; ++h, ++use) {
                const uint32_t st = use % NST, ph = (use / NST) & 1;
                t0 = clock64();
                if (!mbar_wait(bar_full + 8 * st, ph, abort_flag, a.err, 3)) goto mma_done;
                if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && lane == 0) a.prof[1] += clock64() - t0;   // waiting for weights
                if (lane == 0 && c == 0 && h == 0) B2N_TRACE(s, t, 5);
                tc_fence_after();
                const uint64_t bdesc = umma_desc(ring0 + st * CHUNK_BYTES);
                if (elect_one()) {
                  if (a.dbg & 2) {
                  } else if (nk == 4) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                      tc_mma(d_tmem + h * 128, adesc + 2 * k, bdesc + 2 * k, idesc, (acc_in || c > 0 || k > 0) ? 1u : 0u);
                  } else {
#pragma unroll
                    for (int k = 0; k < 2; ++k)
                      tc_mma(d_tmem + h * 128, adesc + 2 * k, bdesc + 2 * k, idesc, (acc_in || c > 0 || k > 0) ? 1u : 0u);
                  }
                  tc_commit(bar_empty + 8 * st);   // frees the ring slot once these MMAs have read it
                }
                __syncwarp();
              }
            }
            if (lane == 0) B2N_TRACE(s, t, 6);
            if (elect_one()) tc_commit(bar_acc + 8 * t);
            __syncwarp();
          }
        }
      }
    }
  mma_done:;
  } else if (warp == 10) {
    // ================================ plane store ================================
    // The activation tile the epilogue has just finished is also a saved plane: this warp sends it to HBM with TMA
    // tensor stores while the MMAs of the next step read it (both only read), and tells the epilogue through bar_st
    // when the store engine has read the tile, i.e. when the next epilogue may overwrite it.  (These stores used to be
    // issued by the MMA warp: ~800 cycles of issue + the read wait on the serial path of every tile and step.)
    if (a.use_tma) {
      uint32_t act_phase[2] = {0, 0}, tail_phase = 0;
      const uint32_t act0 = s32(smem + OFF_ACT);
      for (int64_t pair = pair_first; pair < n_pairs; pair += pair_step) {
        for (int s = 0; s < plan.n_steps; ++s) {
          for (int t = 0; t < 2; ++t) {
            if (!mbar_wait(bar_act + 8 * t, act_phase[t] & 1, abort_flag, a.err, 6)) goto store_done;
            ++act_phase[t];
            if (elect_one()) {
              if (s > 0 && plan.s[s - 1].tma) {
                const int row0 = (int)(pair * 256 + t * 128);
                for (int kb = 0; kb < plan.s[s - 1].n / 64; ++kb)
                  tma_store_3d(&tmap_save, act0 + t * ACT_BYTES + kb * KBLK_BYTES, 64 * kb, row0, plan.s[s - 1].save_slot);
                bulk_commit();
                bulk_wait_read0();
              }
              mbar_arrive(bar_st + 8 * t);
            }
            __syncwarp();
          }
        }
        // the last step's plane: nothing reads that tile after it, so the epilogue announces it on bar_tail; the extra
        // bar_st arrival is what the NEXT pair's pre-step waits for before it writes into the tile again
        if (plan.s[plan.n_steps - 1].tma) {
          for (int t = 0; t < 2; ++t) {
            if (!mbar_wait(bar_tail + 8 * t, tail_phase & 1, abort_flag, a.err, 7)) goto store_done;
            if (elect_one()) {
              const Step& lp = plan.s[plan.n_steps - 1];
              const int row0 = (int)(pair * 256 + t * 128);
              for (int kb = 0; kb < lp.n / 64; ++kb)
                tma_store_3d(&tmap_save, act0 + t * ACT_BYTES + kb * KBLK_BYTES, 64 * kb, row0, lp.save_slot);
              bulk_commit();
              bulk_wait_read0();
              mbar_arrive(bar_st + 8 * t);
            }
            __syncwarp();
          }
          ++tail_phase;
        }
      }
      if (elect_one()) bulk_wait0();                 // all plane stores complete before the CTA exits
      __syncwarp();
    }
  store_done:;
  } else {
    // ================================ epilogue (8 warps, all on the tile being drained) ================
    const int e = threadIdx.x - 64;            // 0..255
    const int q = warp & 3;                    // TMEM lane quarter this warp may touch
    const int half = (warp - 2) >> 2;          // accumulator column half this warp drains
    const int r = 32 * q + lane;               // row inside the tile
    const int c0 = 128 * half;                 // first accumulator column of this thread
    uint32_t acc_phase[2] = {0, 0}, st_phase[2] = {0, 0};
    const bool tail_store = a.use_tma && plan.s[plan.n_steps - 1].tma;   // the last step's plane goes through the act tile too
    if (BWD) {  // head weights are needed by every pair: stage them once
      vec[e] = __ldg(a.w_sigma + e);
      vec[256 + e] = __ldg(a.w_rgb + e);
      if (e < 128) vec[512 + e] = __ldg(a.w_rgb + 256 + e);
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    // "A operand of tile t is in place" (this CTA's MMA / store warps wait for it)
    auto arrive_act = [&](int t) { mbar_arrive(bar_act + 8 * t); };
    // forward: the bias row (and head weights) of a step are fetched into registers one step ahead, so the staging
    // between two steps is bar.sync / st.shared / bar.sync without a global-load latency in the critical path
    float pf0 = 0.f, pf1 = 0.f, pf2 = 0.f;
    auto prefetch_step = [&](int s_from) {
      if (BWD) return;
      int ns = s_from;
      while (ns < plan.n_steps && WIDE && plan.s[ns].partial) ++ns;
      if (ns >= plan.n_steps) return;
      const Step& np = plan.s[ns];
      if (e < np.n) pf0 = __ldg(a.bias + np.bias_off + e);
      if (np.epi == EPI_RELU_SIGMA) pf1 = __ldg(a.w_sigma + e);
      if (np.epi == EPI_VIEW_RGB) {
        pf1 = __ldg(a.w_rgb + e);
        if (e < 128) pf2 = __ldg(a.w_rgb + 256 + e);
      }
    };
    for (int64_t pair = pair_first; pair < n_pairs; pair += pair_step) {
      const long long tp0 = clock64();
      prefetch_step(0);
      float row_scalar[2] = {0.f, 0.f};   // fwd: unused; bwd: d(pre-relu sigma) of this thread's row in tile t
      // ---- pre-step: first A operand of both tiles
      for (int t = 0; t < 2; ++t) {
        unsigned char* act = smem + OFF_ACT + t * ACT_BYTES;
        unsigned char* aux = smem + OFF_AUX + t * KBLK_BYTES;
        const int64_t p = pair * 256 + t * 128 + r;
        const bool valid = p < a.P && !(a.dbg & 8);
        // the previous pair's last plane must have left the tile (its store is announced with one more bar_st phase)
        if (tail_store && pair != pair_first && !mbar_wait(bar_st + 8 * t, st_phase[t]++ & 1, abort_flag, a.err, 8)) goto epi_done;
        if (!BWD) {
          stage_row(a.x_enc + p * a.pos_dim, a.pos_dim < 64 ? a.pos_dim : 64, valid, aux, r, 4 * half);
        } else {
          // colour head backward -> dZ_view (128 wide; this thread covers 64 of its columns)
          float dzr[3] = {0.f, 0.f, 0.f};
          if (valid) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              const float y = __ldg(a.rgb_out + 3 * p + j);
              dzr[j] = __ldg(a.g_rgb + 3 * p + j) * y * (1.f - y);
            }
            row_scalar[t] = __ldg(a.sigma_out + p) > 0.f ? __ldg(a.g_sigma + p) : 0.f;
            if (half == 0) *reinterpret_cast<float4*>(a.dz_small + 4 * p) = make_float4(dzr[0], dzr[1], dzr[2], row_scalar[t]);
          }
          // gate of the view layer: bits 64*half .. 64*half+63 of the hv plane's mask row
          uint2 hvm = make_uint2(0u, 0u);
          if (valid) hvm = __ldcs(reinterpret_cast<const uint2*>(a.mask_in + ((size_t)9 * a.P + p) * 8 + 2 * half));
          __nv_bfloat16* srow = (a.save && valid) ? a.save + ((size_t)0 * a.P + p) * HID : nullptr;
#pragma unroll 2
          for (int c = 8 * half; c < 8 * half + 8; ++c) {
            const int cl = c - 8 * half;                                  // 0..7: byte cl of this thread's 64 gate bits
            const uint32_t hb = ((cl < 4 ? hvm.x : hvm.y) >> (8 * (cl & 3))) & 0xffu;
            float f[8];
            const float4* w0 = reinterpret_cast<const float4*>(vec + 256 + 8 * c);        // 16-byte broadcast loads
            const float4* w1 = reinterpret_cast<const float4*>(vec + 256 + 128 + 8 * c);
            const float4* w2 = reinterpret_cast<const float4*>(vec + 256 + 256 + 8 * c);
#pragma unroll
            for (int j4 = 0; j4 < 2; ++j4) {
              const float4 a0 = w0[j4], a1 = w1[j4], a2 = w2[j4];
              const float g[4] = {dzr[0] * a0.x + dzr[1] * a1.x + dzr[2] * a2.x, dzr[0] * a0.y + dzr[1] * a1.y + dzr[2] * a2.y,
                                  dzr[0] * a0.z + dzr[1] * a1.z + dzr[2] * a2.z, dzr[0] * a0.w + dzr[1] * a1.w + dzr[2] * a2.w};
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) f[4 * j4 + jj] = ((hb >> (4 * j4 + jj)) & 1u) ? g[jj] : 0.f;
            }
            const uint4 pk = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
            *reinterpret_cast<uint4*>(act + ((8 * c) >> 6) * KBLK_BYTES + swz(r, ((8 * c) & 63) >> 3)) = pk;
            if (srow) __stcs(reinterpret_cast<uint4*>(srow + 8 * c), pk);
          }
        }
        proxy_fence();
        arrive_act(t);
      }
      if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && e == 0) a.prof[4] += 1, a.prof[5] += clock64() - tp0;   // pairs of CTA 0; pre-step
      for (int s = 0; s < plan.n_steps; ++s) {
        const Step& sp = plan.s[s];
        const bool last = (s + 1 == plan.n_steps);
        if (!BWD && WIDE && sp.partial) {
          // the MMAs of this step only add a k-slice to the accumulators: when they have read the aux
          // block, swap in the next slice of the input row; nothing is drained
          for (int t = 0; t < 2; ++t) {
            unsigned char* aux = smem + OFF_AUX + t * KBLK_BYTES;
            const int64_t p = pair * 256 + t * 128 + r;
            const bool valid = p < a.P && !(a.dbg & 8);
            if (!mbar_wait(bar_acc + 8 * t, acc_phase[t] & 1, abort_flag, a.err, 4)) goto epi_done;
            if (a.use_tma && !mbar_wait(bar_st + 8 * t, st_phase[t]++ & 1, abort_flag, a.err, 5)) goto epi_done;
            ++acc_phase[t];
            tc_fence_after();
            restage_aux(a, sp.restage, p, valid, aux, r, 4 * half);
            tc_fence_before();
            proxy_fence();
            arrive_act(t);
          }
          continue;
        }
        if (!BWD) {
          // stage this step's bias (and the head weights) for broadcast reads
          const long long ts0 = clock64();
          if (e == 0) B2N_TRACE(s, 0, 7);
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (e < sp.n) vec[e] = pf0;
          if (sp.epi == EPI_RELU_SIGMA) vec[256 + e] = pf1;
          if (sp.epi == EPI_VIEW_RGB) {
            vec[256 + e] = pf1;
            if (e < 128) vec[512 + e] = pf2;
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          prefetch_step(s + 1);
          if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && e == 0) a.prof[6] += clock64() - ts0;   // bias staging
        }
        const bool works = c0 < sp.n;            // a 128-wide step is drained by the column-half-0 warps only
        for (int t = 0; t < 2; ++t) {
          unsigned char* act = smem + OFF_ACT + t * ACT_BYTES;
          unsigned char* aux = smem + OFF_AUX + t * KBLK_BYTES;
          const int64_t p = pair * 256 + t * 128 + r;
          const bool valid = p < a.P && !(a.dbg & 8);
          const uint32_t trow = tmem + ((uint32_t)(32 * q) << 16) + t * 256 + c0;
          // bwd: the ReLU gate of this step = 128 mask bits of the forward plane named in bias_off, fetched before
          // the wait so that the load overlaps the MMAs
          const bool gated = BWD && sp.epi != EPI_B_LINEAR;
          uint4 gate = make_uint4(0u, 0u, 0u, 0u);
          if (gated && valid)
            gate = __ldcs(reinterpret_cast<const uint4*>(a.mask_in + ((size_t)sp.bias_off * a.P + p) * 8 + 4 * half));
          long long t0 = clock64();
          if (e == 0) B2N_TRACE(s, t, 0);
          if (!mbar_wait(bar_acc + 8 * t, acc_phase[t] & 1, abort_flag, a.err, 4)) goto epi_done;
          if (a.use_tma && !mbar_wait(bar_st + 8 * t, st_phase[t]++ & 1, abort_flag, a.err, 5)) goto epi_done;
          long long t1 = clock64();
          if (e == 0) B2N_TRACE(s, t, 1);
          if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && e == 0) a.prof[2] += t1 - t0;    // epilogue waiting for the MMAs
          ++acc_phase[t];
          tc_fence_after();
          float sig_acc = 0.f, rgb_acc[3] = {0.f, 0.f, 0.f};
          const bool relu = sp.epi != EPI_LINEAR;
          __nv_bfloat16* save_row = (a.save && sp.save_slot >= 0 && valid && !(a.use_tma && sp.tma))
                                        ? a.save + ((size_t)sp.save_slot * a.P + p) * HID : nullptr;
          uint32_t mbits[4] = {0u, 0u, 0u, 0u};   // fwd: ReLU bits of this thread's 128 columns; bwd: the gate bits
          if (works && !(a.dbg & 1)) {
            // TMEM reads are the scarce resource of this epilogue (~64 B/cycle/SM): keep one 32-column
            // load in flight while the previous block is converted and stored (double-buffered registers)
            uint32_t vbuf[2][32];
            tc_ld32(trow, vbuf[0]);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
              const int colb = c0 + 32 * cb;           // first accumulator column of this block of 32
              tc_ld_wait();
              if (cb + 1 < 4) tc_ld32(trow + 32 * (cb + 1), vbuf[(cb + 1) & 1]);
              const uint32_t (&v)[32] = vbuf[cb & 1];
              float f[32];
              if (!BWD) {
                const float4* bias4 = reinterpret_cast<const float4*>(vec + colb);   // 16-byte broadcast loads
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                  const float4 b = bias4[j4];
                  const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                  for (int jj = 0; jj < 4; ++jj) {
                    const int j = 4 * j4 + jj;
                    float x = __uint_as_float(v[j]) + bb[jj];
                    f[j] = relu ? fmaxf(x, 0.f) : x;
                  }
                }
                if (a.mask_out) {      // training: 1 bit per activation replaces a 512-byte row read in the backward
                  // bit j = (f[j] > 0): for f >= +0 (ReLU output) the integer negation of the float's bits has its sign
                  // bit set exactly when f > 0; two instructions per bit (negate, funnel-shift the sign in).  For the
                  // linear step the bits of negative values are garbage, and nothing reads that slot's mask.
                  // Four independent 8-bit chains (a single 32-long dependent chain costs its full latency here:
                  // there are only two epilogue warps per scheduler to hide it), merged by byte permutes.
                  uint32_t mq[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                  for (int j = 7; j >= 0; --j) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) mq[k] = __funnelshift_l(0u - __float_as_uint(f[8 * k + j]), mq[k], 1);
                  }
                  mbits[cb] = __byte_perm(__byte_perm(mq[0], mq[1], 0x0040), __byte_perm(mq[2], mq[3], 0x0040), 0x5410);
                }
                if (sp.epi == EPI_RELU_SIGMA) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) sig_acc = fmaf(f[j], vec[256 + colb + j], sig_acc);
                } else if (sp.epi == EPI_VIEW_RGB) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) {
                    rgb_acc[0] = fmaf(f[j], vec[256 + colb + j], rgb_acc[0]);
                    rgb_acc[1] = fmaf(f[j], vec[256 + 128 + colb + j], rgb_acc[1]);
                    rgb_acc[2] = fmaf(f[j], vec[256 + 256 + colb + j], rgb_acc[2]);
                  }
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                if (sp.epi == EPI_B_MASK_SIGMA) {   // + d(sigma_pre) * w_sigma  (density head, rank-1)
#pragma unroll
                  for (int j = 0; j < 32; ++j) f[j] = fmaf(row_scalar[t], vec[colb + j], f[j]);
                }
                if (gated) {
                  const uint32_t m = gate.x * (cb == 0) + gate.y * (cb == 1) + gate.z * (cb == 2) + gate.w * (cb == 3);
#pragma unroll
                  for (int j = 0; j < 32; ++j)
                    if (!((m >> j) & 1u)) f[j] = 0.f;
                }
              }
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                const uint4 pk = make_uint4(pack_bf16(f[8 * c4], f[8 * c4 + 1]), pack_bf16(f[8 * c4 + 2], f[8 * c4 + 3]),
                                            pack_bf16(f[8 * c4 + 4], f[8 * c4 + 5]), pack_bf16(f[8 * c4 + 6], f[8 * c4 + 7]));
                const int col = colb + 8 * c4;            // first column of this 16-byte chunk
                if (!last || tail_store)
                  *reinterpret_cast<uint4*>(act + (col >> 6) * KBLK_BYTES + swz(r, (col & 63) >> 3)) = pk;
                if (save_row) __stcs(reinterpret_cast<uint4*>(save_row + col), pk);
              }
            }
          }
          if (!BWD && a.mask_out && works && valid && sp.save_slot >= 0)
            __stcs(reinterpret_cast<uint4*>(a.mask_out + ((size_t)sp.save_slot * a.P + p) * 8 + 4 * half),
                   make_uint4(mbits[0], mbits[1], mbits[2], mbits[3]));
          if (!BWD) {
            if (sp.epi == EPI_RELU_SIGMA) {
              // the density dot product is split over the two column halves: combine through smem
              if (half == 1) vec[512 + r] = sig_acc;
              asm volatile("bar.sync 1, 256;" ::: "memory");
              if (half == 0 && valid) a.sigma[p] = fmaxf(sig_acc + vec[512 + r] + __ldg(a.head_bias), 0.f);
              asm volatile("bar.sync 1, 256;" ::: "memory");
            }
            if (sp.epi == EPI_VIEW_RGB && works && valid) {
#pragma unroll
              for (int j = 0; j < 3; ++j) a.rgb[3 * p + j] = 1.f / (1.f + expf(-(rgb_acc[j] + __ldg(a.head_bias + 1 + j))));
            }
            // the aux block is re-used: next slice of x (pos_dim > 64), or the encoded view direction once
            // the skip layer has consumed x
            if (WIDE) restage_aux(a, sp.restage, p, valid, aux, r, 4 * half);
            else if (sp.restage == 3) stage_row(a.d_enc + p * a.dir_dim, a.dir_dim, valid, aux, r, 4 * half);
          }
          tc_fence_before();
          proxy_fence();
          if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && e == 0) a.prof[3] += clock64() - t1;   // epilogue body
          if (e == 0) B2N_TRACE(s, t, 2);
          if (!last) arrive_act(t);
          else if (tail_store) mbar_arrive(bar_tail + 8 * t);
        }
      }
      if (a.prof && (a.dbg & 16) && blockIdx.x == 0 && e == 0) a.prof[7] += clock64() - tp0;     // whole pair
    }
  epi_done:;
  }
  if (CTA2) {
    tc_fence_before();
    cluster_sync_all();       // nothing of this CTA (barriers, TMEM, tiles) is touched by the peer after this point
    if (warp == 1) tmem_dealloc2(tmem, 512);
    return;
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------------------- weight packing
struct PackChunk {
  const float* W;   // source matrix, row-major, leading dimension ldw
  // forward (trans = 0): tile row i <- source row n0+i (< n_real), tile k <- source column k0 + k (< k_real)
  // backward (trans = 1): tile row i <- source column n0+i (< n_real), tile k <- source row k0 + k (< k_real)
  int ldw, n0, n_real, k0, k_real, trans;
};
struct PackArgs {
  int n_chunks;
  PackChunk c[MAX_CHUNKS];
  unsigned char* dst;
};

__global__ void k_mlp256_pack(const PackArgs a) {
  const PackChunk& c = a.c[blockIdx.x];
  unsigned char* dst = a.dst + (size_t)blockIdx.x * CHUNK_BYTES;
  for (int i = threadIdx.x; i < 128 * 8; i += blockDim.x) {
    const int row = i >> 3, ch = i & 7;
    const int n = c.n0 + row;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = c.k0 + 8 * ch + j;
      const bool ok = n < c.n_real && k < c.k_real;
      f[j] = ok ? __ldg(c.trans ? c.W + (size_t)k * c.ldw + n : c.W + (size_t)n * c.ldw + k) : 0.f;
    }
    *reinterpret_cast<uint4*>(dst + swz(row, ch)) =
        make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
  }
}

}  // namespace m256
}  // namespace b2n

using namespace b2n;
using namespace b2n::m256;

// Forward plan of the reference architecture (8 x 256, skip at 4, view 128); dir_dim <= 32.
// pos_dim <= 64: x is one 64-column aux block.  64 < pos_dim <= 96 (Part 3: 63 canonical + 21 time
// features): the layers that read x (0 and 4) run as two accumulating steps, x[:, 0:64] then x[:, 64:96],
// with the epilogue warps swapping the aux block in between.
static void build_fwd_plan(Plan* pl, int pos_dim) {
  int n = 0;
  auto add = [&](int n_act, int aux_k16, int width, int epi, int bias_off, int slot, int acc_in = 0, int partial = 0,
                 int restage = 0) {
    pl->s[n++] = Step{n_act, aux_k16, width, epi, bias_off, slot, acc_in, partial, restage};
  };
  const bool wide = pos_dim > 64;
  if (!wide) {
    add(0, 4, 256, EPI_RELU, 0, 0);
  } else {
    add(0, 4, 256, EPI_RELU, 0, -1, 0, 1, 2);     // x[:, 0:64]   -> swap in x[:, 64:]
    add(0, 2, 256, EPI_RELU, 0, 0, 1, 0, 1);      // + x[:, 64:96] -> drain, swap x[:, 0:64] back for the skip layer
  }
  add(4, 0, 256, EPI_RELU, 256, 1);
  add(4, 0, 256, EPI_RELU, 512, 2);
  add(4, 0, 256, EPI_RELU, 768, 3);
  if (!wide) {
    add(4, 4, 256, EPI_RELU, 1024, 4, 0, 0, 3);   // skip layer: [h, x]; afterwards the aux block takes d_enc
  } else {
    add(4, 4, 256, EPI_RELU, 1024, -1, 0, 1, 2);
    add(0, 2, 256, EPI_RELU, 1024, 4, 1, 0, 3);
  }
  add(4, 0, 256, EPI_RELU, 1280, 5);
  add(4, 0, 256, EPI_RELU, 1536, 6);
  add(4, 0, 256, EPI_RELU_SIGMA, 1792, 7);  // + density head
  add(4, 0, 256, EPI_LINEAR, 2048, 8);      // feature layer (no activation)
  add(4, 2, 128, EPI_VIEW_RGB, 2304, 9);    // view layer [feat, d] + colour head
  pl->n_steps = n;
}

// ---------------------------------------------------------------------------------------- TMA tensor map of the planes
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
// planes: bf16 [n_slots][P][256]; box = one swizzled k-block of an activation tile (64 columns x 128 rows).
// Returns false when the map cannot be built (the kernel then stores the planes from registers).
static bool make_plane_map(CUtensorMap* m, void* planes, int64_t P, int n_slots) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || !planes || P < 128) return false;
  const cuuint64_t dims[3] = {256, (cuuint64_t)P, (cuuint64_t)n_slots};
  const cuuint64_t strides[2] = {512, (cuuint64_t)P * 512};
  const cuuint32_t box[3] = {64, 128, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, planes, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// packed weight stream as a 2-D tensor [bytes / 512 rows][256 bf16]; box = 16 rows = 8 KB (half a chunk), no swizzle
static bool make_weight_map(CUtensorMap* m, const void* packed, size_t bytes) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || !packed || bytes < (size_t)CHUNK_BYTES) return false;
  const cuuint64_t dims[2] = {256, (cuuint64_t)(bytes / 512)};
  const cuuint64_t strides[1] = {512};
  const cuuint32_t box[2] = {256, 16};
  const cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(packed), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// CTA-pair schedule on/off (-1 = not decided yet: environment variable B2N_MLP256_PAIR, default on)
static int g_pair_mode = -1;
extern "C" int b2n_debug_mlp256_set_pair(int on) {
  g_pair_mode = on ? 1 : 0;
  return B2N_OK;
}
static bool pair_mode() {
  if (g_pair_mode < 0) {
    const char* e = getenv("B2N_MLP256_PAIR");
    g_pair_mode = (e && e[0] == '0') ? 0 : 1;
  }
  return g_pair_mode == 1;
}

// launches `kernel` as clusters of two CTAs, one cluster per SM pair (persistent); returns false when the device
// cannot co-schedule a pair (the caller then uses the single-CTA kernel)
template <typename K>
static bool launch_pairs(K kernel, const FwdArgs& a, const CUtensorMap& tmap_save, const CUtensorMap& tmap_w, cudaStream_t stream) {
  static int max_clusters = -1;          // same resources for every instantiation (one CTA per SM)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(N_THREADS), cfg.dynamicSmemBytes = SMEM_BYTES, cfg.stream = stream, cfg.attrs = attr, cfg.numAttrs = 1;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  if (max_clusters < 0) {
    cfg.gridDim = dim3(kSMs);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess) n = 0, cudaGetLastError();
    max_clusters = n;
  }
  if (max_clusters < 1) return false;
  const int64_t n_quads = (a.P + 511) / 512;
  int n_clusters = max_clusters < kSMs / 2 ? max_clusters : kSMs / 2;
  if (n_quads < n_clusters) n_clusters = (int)n_quads;
  cfg.gridDim = dim3(2 * n_clusters);
  if (cudaLaunchKernelEx(&cfg, kernel, a, tmap_save, tmap_w) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return true;
}

// every step that saves a plane leaves its output in the activation tile and the store warp sends it by TMA (the last
// step of a pair included: bar_tail)
static void mark_tma_steps(Plan* pl) {
  for (int i = 0; i < pl->n_steps; ++i) pl->s[i].tma = (pl->s[i].save_slot >= 0 && !pl->s[i].partial) ? 1 : 0;
}

static long long* g_prof = nullptr;
static int g_dbg = 0;
extern "C" int b2n_debug_mlp256_flags(int flags) {
  g_dbg = flags;
  return B2N_OK;
}
// debug aid: cycle counters of CTA 0 ([0] MMA waits epilogue, [1] MMA waits weights, [2] epilogue waits MMA,
// [3] epilogue body, [4] tile pairs); pass a device int64[8 + 14 * 2 * 16] (zeroed) or NULL to disable; entries from 8 on = B2N_TRACE timeline
extern "C" int b2n_debug_mlp256_prof(void* device_int64x8) {
  g_prof = (long long*)device_int64x8;
  return B2N_OK;
}

// chunks: (1 + 3*4 + 5 + 3*4 + 4) k-chunks x 2 halves for the 256-wide steps, 5 x 1 for the view layer,
// plus 2 more k-chunks x 2 halves when pos_dim > 64 (the buffer is always sized for that case)
extern "C" size_t b2n_nerf_mlp_packed_bytes(void) { return (size_t)((1 + 12 + 5 + 12 + 4 + 2) * 2 + 5) * CHUNK_BYTES; }

// weights: the nn.Linear weight matrices of NeRFDecoder: pts_layers[0..7], feature_layer, view_layer
extern "C" int b2n_nerf_mlp_pack(const float* const* pts_w, const float* feature_w, const float* view_w, int pos_dim,
                                 int dir_dim, void* packed, b2n_stream_t stream) {
  B2N_REQUIRE(pts_w && feature_w && view_w && packed, "null pointer");
  B2N_REQUIRE(pos_dim > 0 && pos_dim <= 96 && dir_dim > 0 && dir_dim <= 32, "pos_dim <= 96 and dir_dim <= 32 required");
  PackArgs pa{};
  int n = 0;
  const int x_lo = pos_dim < 64 ? pos_dim : 64;      // columns of the first x block
  // one k-chunk of a layer = `halves` chunks of 128 output rows each, in [k-chunk][half] order
  auto add = [&](const float* W, int ldw, int n_real, int halves, int k0, int k_real) {
    for (int h = 0; h < halves; ++h) pa.c[n++] = PackChunk{W, ldw, 128 * h, n_real, k0, k_real, 0};
  };
  for (int l = 0; l < 8; ++l) {
    B2N_REQUIRE(pts_w[l], "null weight");
    if (l == 0) {
      add(pts_w[0], pos_dim, 256, 2, 0, x_lo);
      if (pos_dim > 64) add(pts_w[0], pos_dim, 256, 2, 64, pos_dim);
    } else {
      const int ld = (l == 4) ? 256 + pos_dim : 256;
      for (int c = 0; c < 4; ++c) add(pts_w[l], ld, 256, 2, 64 * c, 256);
      if (l == 4) {
        add(pts_w[4], ld, 256, 2, 256, 256 + x_lo);
        if (pos_dim > 64) add(pts_w[4], ld, 256, 2, 256 + 64, ld);
      }
    }
  }
  for (int c = 0; c < 4; ++c) add(feature_w, 256, 256, 2, 64 * c, 256);
  for (int c = 0; c < 4; ++c) add(view_w, 256 + dir_dim, 128, 1, 64 * c, 256);
  add(view_w, 256 + dir_dim, 128, 1, 256, 256 + dir_dim);
  pa.n_chunks = n;
  pa.dst = (unsigned char*)packed;
  B2N_REQUIRE((size_t)n * CHUNK_BYTES <= b2n_nerf_mlp_packed_bytes() && n <= MAX_CHUNKS, "internal: packed size mismatch");
  k_mlp256_pack<<<n, 256, 0, (cudaStream_t)stream>>>(pa);
  return check_launch("b2n_nerf_mlp_pack");
}

extern "C" int b2n_nerf_mlp_fwd(const float* x_enc, int pos_dim, const float* d_enc, int dir_dim, const void* packed,
                                const float* bias, const float* w_sigma, const float* w_rgb, const float* head_bias,
                                int64_t P, float* rgb, float* sigma, void* save, void* relu_masks, int* err_flag,
                                b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(x_enc && d_enc && packed && bias && w_sigma && w_rgb && head_bias && rgb && sigma && err_flag,
              "null pointer");
  B2N_REQUIRE(pos_dim > 0 && pos_dim <= 96 && dir_dim > 0 && dir_dim <= 32, "pos_dim <= 96 and dir_dim <= 32 required");
  FwdArgs a{};
  a.x_enc = x_enc, a.pos_dim = pos_dim, a.d_enc = d_enc, a.dir_dim = dir_dim;
  a.packed = (const unsigned char*)packed, a.bias = bias, a.w_sigma = w_sigma, a.w_rgb = w_rgb;
  a.head_bias = head_bias;
  a.P = P, a.rgb = rgb, a.sigma = sigma, a.save = (__nv_bfloat16*)save, a.err = err_flag;
  B2N_REQUIRE(!save == !relu_masks, "save planes and relu_masks go together");
  a.mask_out = (uint32_t*)relu_masks;
  build_fwd_plan(&a.plan, pos_dim);
  mark_tma_steps(&a.plan);
  alignas(64) CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  a.use_tma = (a.save && make_plane_map(&tmap, save, P, 10)) ? 1 : 0;
  a.prof = g_prof, a.dbg = g_dbg;
  alignas(64) CUtensorMap tmap_w;
  memset(&tmap_w, 0, sizeof(tmap_w));
  if (pair_mode() && make_weight_map(&tmap_w, packed, b2n_nerf_mlp_packed_bytes())) {
    const bool ok = pos_dim > 64 ? launch_pairs(k_mlp256<false, true, true>, a, tmap, tmap_w, (cudaStream_t)stream)
                                 : launch_pairs(k_mlp256<false, false, true>, a, tmap, tmap_w, (cudaStream_t)stream);
    if (ok) return check_launch("b2n_nerf_mlp_fwd");
  }
  const int64_t n_pairs = (P + 255) / 256;
  const int grid = (int)(n_pairs < kSMs ? n_pairs : kSMs);
  if (pos_dim > 64) {
    cudaFuncSetAttribute(k_mlp256<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    k_mlp256<false, true><<<grid, N_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a, tmap, tmap_w);
  } else {
    cudaFuncSetAttribute(k_mlp256<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    k_mlp256<false, false><<<grid, N_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a, tmap, tmap_w);
  }
  return check_launch("b2n_nerf_mlp_fwd");
}

// ---------------------------------------------------------------------------------------- backward (data gradients)
// Chain (all on the tensor cores, same schedule as the forward):
//   pre : dZ_view = (d rgb_pre * W_rgb) (.) [hv > 0]                       (epilogue warps, 128 wide)
//   B1  : d feat  = dZ_view  * W_view[:, :256]            K = 128   -> dZ_feat (linear)
//   B2  : d h7    = dZ_feat  * W_feat + d sigma_pre * w_sigma, gated by H7  -> dZ7
//   B3..: d h_{l-1} = dZ_l * W_l[:, :256], gated by H_{l-1}    (l = 7 .. 1)  -> dZ_{l-1}
// Every dZ plane is written to HBM in bf16: the weight gradients dW_l = dZ_l^T In_l are plain
// [256 x P] x [P x 256] GEMMs done outside this kernel.  Step::bias_off holds the index of the
// forward plane that gates the step.
static void build_bwd_plan(Plan* pl) {
  int n = 0;
  auto add = [&](int n_act, int epi, int gate_plane, int slot) { pl->s[n++] = Step{n_act, 0, 256, epi, gate_plane, slot}; };
  add(2, EPI_B_LINEAR, 0, 1);        // d feat
  add(4, EPI_B_MASK_SIGMA, 7, 2);    // dZ7
  for (int l = 7; l >= 1; --l) add(4, EPI_B_MASK, l - 1, 2 + (8 - l));   // dZ6 .. dZ0 -> slots 3..9
  pl->n_steps = n;
}

extern "C" size_t b2n_nerf_mlp_packed_bwd_bytes(void) { return (size_t)(2 + 4 * 8) * 2 * CHUNK_BYTES; }

extern "C" int b2n_nerf_mlp_pack_bwd(const float* const* pts_w, const float* feature_w, const float* view_w, int pos_dim,
                                     int dir_dim, void* packed, b2n_stream_t stream) {
  B2N_REQUIRE(pts_w && feature_w && view_w && packed, "null pointer");
  B2N_REQUIRE(pos_dim > 0 && pos_dim <= 96 && dir_dim > 0 && dir_dim <= 32, "pos_dim <= 96 and dir_dim <= 32 required");
  PackArgs pa{};
  int n = 0;
  // tile rows = input index of the layer (first 256 inputs, two halves), tile k = output index of the layer
  auto add = [&](const float* W, int ldw, int n_out, int k0) {
    for (int h = 0; h < 2; ++h) pa.c[n++] = PackChunk{W, ldw, 128 * h, 256, k0, n_out, 1};
  };
  for (int c = 0; c < 2; ++c) add(view_w, 256 + dir_dim, 128, 64 * c);
  for (int c = 0; c < 4; ++c) add(feature_w, 256, 256, 64 * c);
  for (int l = 7; l >= 1; --l) {
    B2N_REQUIRE(pts_w[l], "null weight");
    const int ld = (l == 4) ? 256 + pos_dim : 256;
    for (int c = 0; c < 4; ++c) add(pts_w[l], ld, 256, 64 * c);
  }
  pa.n_chunks = n;
  pa.dst = (unsigned char*)packed;
  B2N_REQUIRE((size_t)n * CHUNK_BYTES == b2n_nerf_mlp_packed_bwd_bytes(), "internal: packed size mismatch");
  k_mlp256_pack<<<n, 256, 0, (cudaStream_t)stream>>>(pa);
  return check_launch("b2n_nerf_mlp_pack_bwd");
}

extern "C" int b2n_nerf_mlp_bwd(const void* packed_bwd, const float* w_sigma, const float* w_rgb, const void* relu_masks,
                                const float* rgb, const float* sigma, const float* g_rgb, const float* g_sigma,
                                int64_t P, void* dz_planes, float* dz_small, int* err_flag, b2n_stream_t stream) {
  B2N_REQUIRE(P >= 0, "negative size");
  if (P == 0) return B2N_OK;
  B2N_REQUIRE(packed_bwd && w_sigma && w_rgb && relu_masks && rgb && sigma && g_rgb && g_sigma && dz_planes &&
                  dz_small && err_flag, "null pointer");
  FwdArgs a{};
  a.packed = (const unsigned char*)packed_bwd, a.w_sigma = w_sigma, a.w_rgb = w_rgb;
  a.mask_in = (const uint32_t*)relu_masks, a.rgb_out = rgb, a.sigma_out = sigma, a.g_rgb = g_rgb;
  a.g_sigma = g_sigma, a.P = P, a.save = (__nv_bfloat16*)dz_planes, a.dz_small = dz_small, a.err = err_flag;
  build_bwd_plan(&a.plan);
  mark_tma_steps(&a.plan);
  alignas(64) CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  a.use_tma = make_plane_map(&tmap, dz_planes, P, 10) ? 1 : 0;
  a.prof = g_prof, a.dbg = g_dbg;
  alignas(64) CUtensorMap tmap_w;
  memset(&tmap_w, 0, sizeof(tmap_w));
  if (pair_mode() && make_weight_map(&tmap_w, packed_bwd, b2n_nerf_mlp_packed_bwd_bytes()) &&
      launch_pairs(k_mlp256<true, false, true>, a, tmap, tmap_w, (cudaStream_t)stream))
    return check_launch("b2n_nerf_mlp_bwd");
  cudaFuncSetAttribute(k_mlp256<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  const int64_t n_pairs = (P + 255) / 256;
  const int grid = (int)(n_pairs < kSMs ? n_pairs : kSMs);
  k_mlp256<true><<<grid, N_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a, tmap, tmap_w);
  return check_launch("b2n_nerf_mlp_bwd");
}
