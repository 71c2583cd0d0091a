/* b2nerf.h -- C ABI of libb2nerf.so: the B200 (sm_100a) ray-marching hot path
 * of Project-NeRF (encode -> MLP -> sample/mask/composite, forward + backward).
 *
 * The reference (CV-Project2025/Project-NeRF) is pure Python; its hot path is
 * bound through torch ops and the external tiny-cuda-nn extension.  This header
 * is what a maintainer binds instead (ctypes stub: INTEGRATION.md).  Each entry
 * point cites the reference code it replaces (paths relative to the reference
 * repository root).
 *
 * Conventions
 *  - every function returns 0 on success or a negative B2N_E* code; it never
 *    throws, never exits, never synchronises the stream, allocates nothing;
 *  - all pointers are DEVICE pointers to contiguous row-major fp32 unless
 *    stated; the caller owns every buffer; `stream` is a cudaStream_t;
 *  - sizes are element counts; empty inputs (P == 0, B == 0) are a no-op;
 *  - functions are stateless and re-entrant; device = current device.
 */
#ifndef B2NERF_H_
#define B2NERF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2N_ABI_VERSION 19

#define B2N_OK 0
#define B2N_EINVAL (-1)  /* bad argument (null pointer, size, unsupported shape) */
#define B2N_ECUDA (-2)   /* CUDA launch/runtime error; see b2n_last_error()      */

typedef void* b2n_stream_t; /* cudaStream_t */

int b2n_abi_version(void);
/* thread-local, valid until the next failing call on this thread */
const char* b2n_last_error(void);

/* Optional DEVICE-side row count.  While set (non-NULL; host-side, per thread), every entry point below that takes a
 * point count P treats rows >= *rows_device of its point-indexed arguments as absent: they are neither read nor written
 * (the clamp happens inside the kernels, so the host never has to know the number).  This is how a ray-marching step
 * behind an occupancy grid runs with fixed-capacity buffers and no device->host read of the active-sample count
 * (the reference reads it three times per call: src/renderer.py:309-323), which makes the step CUDA-graph capturable.
 * Honoured by: b2n_pe_*, b2n_hash_*, b2n_instant_mlp_*, b2n_fmlp_* (the saved planes get zero rows up to the next
 * multiple of 64 behind the count).  NOT honoured by the fp32 b2n_linear_* / b2n_sigma_head_* and the 256-wide
 * b2n_nerf_mlp_* entry points; b2n_composite_* / b2n_march_* index samples through ray offsets and do not need it. */
int b2n_set_active_rows(const int* rows_device);

/* activation codes shared by the linear / fused-MLP entry points */
enum { B2N_ACT_NONE = 0, B2N_ACT_RELU = 1, B2N_ACT_SIGMOID = 2 };

/* ------------------------------------------------------------------------
 * Ray marching: stratified depths, occupancy test, compaction
 * ---------------------------------------------------------------------- */

/* Packs a bool occupancy grid (torch.bool [R,R,R], 1 byte/voxel, x slowest;
 * src/renderer.py:29) into a bitfield of n_voxels/32 words (bit v%32 of word
 * v/32).  n_voxels must be a multiple of 32. */
int b2n_occ_pack_bits(const uint8_t* binary, int64_t n_voxels, uint32_t* bits, b2n_stream_t stream);

/* DensityGrid.get_active_mask (src/renderer.py:134-166): voxel index =
 * trunc((p + offset) * scale) per axis, valid iff 0 <= idx < R on all axes,
 * mask = valid && grid bit.  pts [P,3] -> mask [P] (1 byte each, 0/1). */
int b2n_occ_active_mask(const float* pts, int64_t P, const uint32_t* bits, int R, float offset, float scale,
                        uint8_t* mask, b2n_stream_t stream);

/* DensityGrid.update tail (src/renderer.py:119-131): grid = dynamic ?
 * max(grid*decay, cur) : cur; binary = grid > threshold; also emits the packed
 * bitfield and the number of active voxels (device int64 counter, zeroed by
 * the call). */
int b2n_occ_update(const float* cur_sigma, float* grid, int64_t n_voxels, int dynamic, float decay, float threshold,
                   uint8_t* binary, uint32_t* bits, int64_t* n_active, b2n_stream_t stream);

/* sample_stratified + point generation + occupancy test in one pass
 * (src/renderer.py:186-201, :290-291, :305).
 *   z_base/z_lo/z_hi [N]  unperturbed depths and the stratum bounds (host-built
 *                         once with torch so they are bit-identical to the
 *                         reference's linspace arithmetic);
 *   u [B,N] or NULL       the U[0,1) jitter (torch.rand) -- NULL = no perturb;
 *   bits or NULL          occupancy bitfield; NULL = every sample active;
 * outputs
 *   z [B,N]               z = lo + (hi - lo) * u   (or z_base); may be NULL
 *                         when u is NULL (the depths are then z_base itself)
 *   mask_words [B,W]      W = (N+31)/32, bit s%32 of word s/32 = sample active
 *   ray_count [B]         active samples of the ray (int32)                  */
int b2n_march_mask(const float* rays_o, const float* rays_d, const float* z_base, const float* z_lo,
                   const float* z_hi, const float* u, const uint32_t* bits, int R, float offset, float scale,
                   int64_t B, int N, float* z, uint32_t* mask_words, int32_t* ray_count, b2n_stream_t stream);

/* Exclusive scan of ray_count -> ray_offset [B+1] (int32; last = total).  If
 * no sample is active the reference forces sample 0 of ray 0
 * (src/renderer.py:309-311): the scan then sets bit 0 of mask_words[0],
 * ray_count[0] = 1 and total = 1.  `total_out` is a device int32 (copy it to
 * the host to size the compact buffers).  scratch: b2n_march_scan_scratch(B)
 * bytes. */
size_t b2n_march_scan_scratch(int64_t B);
int b2n_march_scan(int32_t* ray_count, uint32_t* mask_words, int W, int64_t B, int32_t* ray_offset,
                   int32_t* total_out, void* scratch, b2n_stream_t stream);

/* Order-preserving compaction (the boolean-mask gathers of
 * src/renderer.py:315-323): for every active sample, in (ray, sample) order,
 * writes sample_idx (= ray*N + s), the point o + d*z, the normalised view
 * direction d/|d| (src/renderer.py:294) and, if times != NULL, the ray's time.
 * Any output pointer may be NULL.  mask_words == NULL means dense (all B*N). */
int b2n_march_compact(const float* rays_o, const float* rays_d, const float* times, const float* z,
                      const uint32_t* mask_words, const int32_t* ray_offset, int64_t B, int N,
                      int32_t* sample_idx, float* pts, float* dirs, float* t_out, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Alpha compositing (volume_render, src/renderer.py:204-237; mean_delta_x,
 * src/renderer.py:363-380)
 *   rgb [P,3], sigma [P], dx [P,3] or NULL: per-sample fields, either dense
 *   (P = B*N, mask_words == NULL) or compact (active samples only, in
 *   (ray, sample) order; inactive samples count as rgb = sigma = dx = 0).
 *   bg: [3] (bg_per_ray = 0) or [B,3] (bg_per_ray = 1) or NULL (no background).
 * forward  -> color [B,3], depth [B], acc [B], mean_dx [B,3] (if dx)
 * backward -> g_rgb [P,3], g_sigma [P], g_dx [P,3] (same layout as inputs)
 * ---------------------------------------------------------------------- */
int b2n_composite_fwd(const float* rgb, const float* sigma, const float* dx, const float* z, const float* rays_d,
                      const float* bg, int bg_per_ray, const uint32_t* mask_words, const int32_t* ray_offset,
                      int64_t B, int N, float* color, float* depth, float* acc, float* mean_dx,
                      b2n_stream_t stream);
int b2n_composite_bwd(const float* rgb, const float* sigma, const float* dx, const float* z, const float* rays_d,
                      const float* bg, int bg_per_ray, const uint32_t* mask_words, const int32_t* ray_offset,
                      int64_t B, int N, const float* g_color, const float* g_depth, const float* g_acc,
                      const float* g_mean_dx, float* g_rgb, float* g_sigma, float* g_dx, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Fourier positional encoding (FourierRepresentation.forward,
 * src/embeddings.py:22-32): out row = [x, sin((x*f0)*pi), cos(..), ...];
 * written at column `col0` of a row-major buffer with leading dimension ld_out
 * so that concatenations (src/core.py:276, src/decoders.py:83,159) need no
 * extra pass.  bands: device [L].  D <= 4.
 * backward accumulates (+=) into g_x [P,D] when accumulate != 0.
 * ---------------------------------------------------------------------- */
int b2n_pe_fwd(const float* x, int64_t P, int D, const float* bands, int L, float* out, int ld_out, int col0,
               b2n_stream_t stream);
int b2n_pe_bwd(const float* x, int64_t P, int D, const float* bands, int L, const float* g_out, int ld_g, int col0,
               float* g_x, int accumulate, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Multiresolution hash grid (HashRepresentation.forward,
 * src/embeddings.py:75-89 -> tinycudann HashGrid, 3-D, linear interpolation)
 * ---------------------------------------------------------------------- */
#define B2N_MAX_LEVELS 32
typedef struct {
  float scale;     /* exp2f(l*log2f(per_level_scale))*base - 1              */
  uint32_t res;    /* ceil(scale) + 1                                        */
  uint32_t size;   /* entries in this level                                  */
  uint32_t offset; /* first entry of this level in the flat table            */
  uint32_t hashed; /* 1: spatial hash, 0: dense x + y*res + z*res^2          */
} b2n_hash_level;

/* x [P,3] world coordinates; x01 = clamp((x + bound) / (2*bound), 0, 1);
 * table: flat fp32 [n_entries * F] (F = 1, 2 or 4); out [P, L*F] written at col0 of ld_out. */
int b2n_hash_fwd(const float* x, int64_t P, float bound, const float* table, const b2n_hash_level* levels_host,
                 int L, int F, float* out, int ld_out, int col0, b2n_stream_t stream);
/* g_table (fp32, same shape as table) is ACCUMULATED into (atomics); g_x [P,3]
 * is overwritten (or accumulated when accumulate_x != 0); either may be NULL.
 * [level_begin, level_end) restricts the TABLE gradient to a window of levels (0, -1 = all; a proper window needs
 * F = 2 and level_begin % 4 == 0): the data-parallel path scatters the fine levels first and all-reduces their slice
 * of the flat table while the coarse levels are still being scattered (b2n/dp.py).  g_x always covers all levels. */
int b2n_hash_bwd(const float* x, int64_t P, float bound, const float* table, const b2n_hash_level* levels_host,
                 int L, int F, const float* g_out, int ld_g, int col0, float* g_table, float* g_x, int accumulate_x,
                 int level_begin, int level_end, b2n_stream_t stream);

/* Spatial order of the points, so that the 16 points a warp of the pair-lane kernels holds share cells and table lines:
 * order int32 [P] is a permutation, sorted position -> original row, by the Morton code of the point's cell on a 2^7
 * lattice over the box (within a cell, in no particular order); x_sorted [P,3] = x[order].  Rows behind the device-side
 * row count (b2n_set_active_rows) keep their place.  scratch: b2n_hash_order_scratch(P) bytes, 16-byte aligned.  Five
 * kernels, no host synchronisation. */
size_t b2n_hash_order_scratch(int64_t P);
int b2n_hash_order(const float* x, int64_t P, float bound, int* order, float* x_sorted, void* scratch,
                   b2n_stream_t stream);
/* b2n_hash_fwd / b2n_hash_bwd (table gradient only) over points in that order: point i is x_sorted[i], its feature row
 * (gradient row) is row order[i] of out (g_out), so the results are those of the plain entries on x.  F = 2 and the
 * pair-lane kernels only (b2nerf_debug.h variant 3); anything else is refused. */
int b2n_hash_fwd_ordered(const float* x_sorted, const int* order, int64_t P, float bound, const float* table,
                         const b2n_hash_level* levels_host, int L, int F, float* out, int ld_out, int col0,
                         b2n_stream_t stream);
int b2n_hash_bwd_ordered(const float* x_sorted, const int* order, int64_t P, float bound, const float* table,
                         const b2n_hash_level* levels_host, int L, int F, const float* g_out, int ld_g, int col0,
                         float* g_table, int level_begin, int level_end, b2n_stream_t stream);

/* Tri-grid temporal blend of Part 4 (src/core.py:308-335): out[P, 2L] = sum_i w_i(t) * HashGrid_i(x) for the
 * start / mid / end deformation grids (one shared geometry, F = 2), w_i = clamp(1 - |t - a_i| / 0.5, 0, 1) with
 * a = (0, 0.5, 1), normalised by (w0 + w1 + w2 + 1e-8).  t [P] (one time per point).  One kernel each way; a grid
 * whose weight is zero is neither read nor scattered to.  backward: g_out [P, 2L] -> ACCUMULATES w_i-weighted table
 * gradients into g_table_* (fp32, zero-initialised by the caller; any may be NULL).  No gradient w.r.t. x or t. */
int b2n_hash_tri_fwd(const float* x, const float* t, int64_t P, float bound, const float* table_start,
                     const float* table_mid, const float* table_end, const b2n_hash_level* levels_host, int L,
                     float* out, int ld_out, b2n_stream_t stream);
int b2n_hash_tri_bwd(const float* x, const float* t, int64_t P, float bound, const b2n_hash_level* levels_host, int L,
                     const float* g_out, int ld_g, float* g_table_start, float* g_table_mid, float* g_table_end,
                     b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * fp32 dense layers (torch.nn.Linear of NeRFDecoder / DeformationNetwork /
 * TimeModulationNetwork, src/decoders.py:55-66,176-189,347, and the bias-free
 * matrices of the tinycudann FullyFusedMLPs, src/decoders.py:111-134,285-295)
 *   fwd   : Y[P,N]   = act(X[P,K] * W[N,K]^T + b)       b may be NULL
 *   dgrad : dX[P,K]  = (dY[P,N] * W[N,K]) (.) act'(Xact)  Xact = the activation
 *           output that produced X (NULL / B2N_ACT_NONE: no mask);
 *           accumulate != 0: dX += ...
 *   wgrad : dW[N,K] += dY^T X ; db[N] += colsum(dY)      (db may be NULL)
 *   act_bwd: dZ = dY (.) act'(Y) in place on dY (Y = activation OUTPUT)
 * ld* are leading dimensions (row strides, in elements).
 * ---------------------------------------------------------------------- */
int b2n_linear_fwd(const float* X, int ldx, const float* W, int ldw, const float* b, float* Y, int ldy, int64_t P,
                   int K, int N, int act, b2n_stream_t stream);
int b2n_linear_dgrad(const float* dY, int lddy, const float* W, int ldw, const float* Xact, int ldxa, int act,
                     float* dX, int lddx, int64_t P, int K, int N, int accumulate, b2n_stream_t stream);
int b2n_linear_wgrad(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, float* db, int64_t P,
                     int K, int N, b2n_stream_t stream);
int b2n_act_bwd(float* dY, int lddy, const float* Y, int ldy, int64_t P, int N, int act, b2n_stream_t stream);

/* sigma head of InstantNeRFDecoder (src/decoders.py:153):
 * sigma[p] = softplus(h[p*ld + 0] - 5); backward: g_h0 += g_sigma * sigmoid(h0 - 5). */
int b2n_sigma_head_fwd(const float* h, int ldh, int64_t P, float* sigma, b2n_stream_t stream);
int b2n_sigma_head_bwd(const float* h, int ldh, int64_t P, const float* g_sigma, float* g_h, int ldg,
                       b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Fused InstantNeRFDecoder (src/decoders.py:136-162: two tinycudann
 * FullyFusedMLPs + softplus density head + concat + sigmoid) including the
 * view-direction Fourier features (src/embeddings.py:22-32 applied to d,
 * src/core.py:358).  IEEE fp16 tensor-core operands (tinycudann's arithmetic),
 * fp32 accumulation; sigma_net's first layer as a split (hi + lo) product; the
 * backward chain runs on a power-of-two multiple of the incoming gradient
 * (found by an |.|-max pre-pass into work4: 4 device bytes owned by the caller)
 * and a non-finite incoming gradient makes every output non-finite.  Hidden
 * width 64; pos_dim <= 64 (padded with zeros); L_dir <= 4 bands.
 *   x_enc [P, pos_dim] (row stride ldx), dirs [P,3] unit view directions,
 *   sigma_params flat [64*pad16(pos_dim) + 16*64], color_params flat
 *   [64*48 + 64*64 + 16*64] (row-major [out,in] matrices, reference layout).
 * forward  -> rgb [P,3], sigma [P]
 * backward -> g_x_enc [P,pos_dim] (row stride ldg; may be NULL), and
 *             ACCUMULATES into g_sigma_params / g_color_params (fp32).
 * The backward recomputes the forward; nothing but the inputs is saved.
 * ---------------------------------------------------------------------- */
/* in_pad_value: what the PADDED input columns of the two FullyFusedMLPs hold (pos_dim .. pad16(pos_dim) of sigma_net,
 * 16 + dir_dim .. pad16(16 + dir_dim) of color_net): 0 (this package, the oracle) or 1 (checkpoints of an upstream
 * tiny-cuda-nn whose Network pads its inputs with ones, which makes those weight columns a bias: b2n.checkpoint). */
/* Forward: the layer products run on tcgen05; a CTA owns 128 points = the 128 TMEM lanes, activations round-trip
 * TMEM -> registers -> shared memory between layers.  rgb == NULL computes sigma alone (dirs, dir_bands and
 * color_params are then not read and may be NULL).  err_flag: a device int the kernel sets non-zero if it had to abort
 * a stalled mbarrier wait (outputs are then invalid); it is never cleared by the kernel. */
int b2n_instant_mlp_fwd_tc(const float* x_enc, int ldx, int pos_dim, const float* dirs, const float* dir_bands,
                           int L_dir, const float* sigma_params, const float* color_params, int64_t P, float* rgb,
                           float* sigma, float in_pad_value, int* err_flag, b2n_stream_t stream);
/* Backward: the forward recompute and the data-gradient chain run on mma.sync, the five weight gradients dW = dZ^T In
 * on tcgen05: the staged 64-point tiles are MN-major SWIZZLE_128B operands, the fp32 accumulators live in TMEM for the
 * whole persistent loop.  err_flag as in b2n_instant_mlp_fwd_tc. */
int b2n_instant_mlp_bwd_tc(const float* x_enc, int ldx, int pos_dim, const float* dirs, const float* dir_bands,
                           int L_dir, const float* sigma_params, const float* color_params, int64_t P,
                           const float* g_rgb, const float* g_sigma, float* g_x_enc, int ldg, float* g_sigma_params,
                           float* g_color_params, void* work4, float in_pad_value, int* err_flag, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Fused small-width ReLU MLPs of the dynamic configs, bf16 tensor-core
 * operands, fp32 accumulation:
 *   DeformationNetwork     cat[gamma(x'),gamma(t')](84)->128->128->128->3  (src/decoders.py:171-195)
 *   HashDeformationDecoder cat[hash feat(24), time mod(64)](88)->64->64->3 (src/decoders.py:285-316)
 *   TimeModulationNetwork  gamma(t')(21)->64->64 sigmoid                   (src/decoders.py:340-371)
 * General form: input = [x0 | x1] (two row-major fp32 sources, d0 + d1 <= 96,
 * x1 may be NULL with d1 = 0; the concat is never materialised), n_hidden
 * (1..3) ReLU layers of width `hidden` (64 or 128), then an output layer to
 * out_dim (<= 64) with activation out_act.  W[l] (l = 0..n_hidden) are row-major
 * [out,in] fp32 matrices with row stride ldw[l] (torch.nn.Linear.weight, or the
 * slices of a tinycudann flat `params`); b[l] may be NULL (no bias).
 * forward : y [P,out_dim] (row stride ldy); when xin_plane / h_planes are given
 *           (training) also writes the fp16 input rows [P][b2n_fmlp_in_pad(d0+d1)]
 *           and the hidden activations [n_hidden][P][hidden].
 * backward: from g_y, the forward output y (needed for sigmoid/relu outputs) and
 *           h_planes: writes dz_out fp16 [P][b2n_fmlp_out_pad(out_dim)], dz_h fp16
 *           [n_hidden][P][hidden] (pre-activation gradients TIMES the power-of-two
 *           scale S the kernel derives from max|g_y| and leaves as a float at
 *           work8 + 4; work8 = 8 device bytes owned by the caller) and the fp32 input
 *           gradients g_x0 [P,d0] / g_x1 [P,d1] (either may be NULL).  Weight and
 *           bias gradients are dZ_l^T * In_l GEMMs / column sums over the planes
 *           (plain GEMMs, done by the caller).
 * ---------------------------------------------------------------------- */
int b2n_fmlp_in_pad(int d_in);
int b2n_fmlp_out_pad(int out_dim);
int b2n_fmlp_fwd(const float* x0, int ld0, int d0, const float* x1, int ld1, int d1, int hidden, int n_hidden,
                 const float* const* W, const int* ldw, const float* const* b, int out_dim, int out_act, int64_t P,
                 float* y, int ldy, void* xin_plane, void* h_planes, b2n_stream_t stream);
/* dW_l[rows_valid, k_valid] (row stride lddw) += dZ_l^T In_l ; db_l[rows_valid] += colsum(dZ_l) for
 * l < n_layers in one launch: dz[l] fp16 [P][ldz] of width rows[l], in[l] fp16 [P][ldi] of width k[l]
 * (widths multiples of 16, <= 128).  ACCUMULATES into fp32 dW / db (db[l] may be NULL).  scale: device float S (work8 + 4
 * of b2n_fmlp_bwd: its dZ planes hold S * dZ) -- results are divided by it; NULL = 1. */
int b2n_fmlp_wgrad(int n_layers, const void* const* dz, const int* ldz, const int* rows, const void* const* in,
                   const int* ldi, const int* k, float* const* dW, const int* lddw, const int* rows_valid,
                   const int* k_valid, float* const* db, int64_t P, const float* scale, b2n_stream_t stream);
/* The same gradients for hidden = 128 through the tcgen05 plane-GEMM kernel of b2n_nerf_mlp_wgrad (TMA-loaded planes,
 * MN-major operands, HBM-bound): dz_h fp16 [n_hidden][P][128], dz_out fp16 [P][out_pad], h_planes fp16 [n_hidden][P][128],
 * xin fp16 [P][in_pad]; scale as in b2n_fmlp_wgrad.  ACCUMULATES fp32: dW0 [128][128] = dZ_0^T xin (columns >= in_pad stay 0), dWh
 * [n_hidden-1][128][128] = dZ_l^T H_{l-1}, dWoT [128][64] = H_last^T dZ_out (the TRANSPOSED output-layer gradient),
 * db_h [n_hidden][128] = column sums of the hidden dZ planes.  P >= 64. */
int b2n_fmlp_wgrad_tc(const void* dz_h, const void* dz_out, const void* h_planes, const void* xin, int64_t P, int n_hidden,
                      int in_pad, int out_pad, float* dW0, float* dWh, float* dWoT, float* db_h, int* err_flag,
                      const float* scale, b2n_stream_t stream);
int b2n_fmlp_bwd(int d0, int d1, int hidden, int n_hidden, const float* const* W, const int* ldw, int out_dim,
                 int out_act, int64_t P, const float* y, int ldy, const float* g_y, int ldgy, const void* h_planes,
                 void* dz_out, void* dz_h, float* g_x0, int ldg0, float* g_x1, int ldg1, void* work8,
                 b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * 256-wide vanilla NeRF decoder (NeRFDecoder.forward, src/decoders.py:68-87)
 * on tcgen05 tensor cores (bf16 operands, fp32 accumulation in TMEM).  Fixed
 * architecture of the reference configs: 8 x 256 trunk, skip [h, x] at layer 4,
 * 128-wide view layer; pos_dim <= 96 (above 64 the layers reading x run as two
 * accumulating MMA steps), dir_dim <= 32.
 *   b2n_nerf_mlp_pack: converts the fp32 nn.Linear weights (pts_layers[0..7],
 *     feature_layer, view_layer) into the bf16 operand-tile stream the kernel
 *     consumes (b2n_nerf_mlp_packed_bytes() bytes); call once per weight update.
 *   b2n_nerf_mlp_fwd: x_enc [P,pos_dim], d_enc [P,dir_dim] -> rgb [P,3], sigma [P].
 *     bias: concatenated [8*256 + 256 + 128]; w_sigma [256]; w_rgb [3*128];
 *     head_bias: device float[4] = {b_sigma, b_rgb[3]}; save: optional bf16
 *     [10][P][256] planes of the layer outputs (training), written by TMA tensor
 *     stores of the activation tiles; relu_masks: uint32 [10][P][8], bit c of a row
 *     = (plane[c] > 0) for the ReLU layers (slots 0..7 and 9; slot 8, the linear feature
 *     layer, is written but unspecified: nothing gates with it), given exactly when `save`
 *     is (the backward gates with these 32-byte rows instead of re-reading the 512-byte
 *     plane rows); err_flag: device int
 *     (0 = ok; non-zero = the kernel aborted a stalled pipeline instead of hanging).
 * ---------------------------------------------------------------------- */
size_t b2n_nerf_mlp_packed_bytes(void);
int b2n_nerf_mlp_pack(const float* const* pts_w, const float* feature_w, const float* view_w, int pos_dim, int dir_dim,
                      void* packed, b2n_stream_t stream);
int b2n_nerf_mlp_fwd(const float* x_enc, int pos_dim, const float* d_enc, int dir_dim, const void* packed,
                     const float* bias, const float* w_sigma, const float* w_rgb, const float* head_bias, int64_t P,
                     float* rgb, float* sigma, void* save, void* relu_masks, int* err_flag, b2n_stream_t stream);

/* Backward data-gradient chain of the same decoder on tcgen05 (autograd of
 * src/decoders.py:68-87 w.r.t. the activations).  relu_masks = the bit masks written
 * by b2n_nerf_mlp_fwd; rgb/sigma = its outputs; g_rgb [P,3], g_sigma [P] = incoming
 * gradients.  Writes dz_planes (bf16 [10][P][256]: dZ_view(128 wide), dZ_feat,
 * dZ7 .. dZ0 = pre-activation gradients of every layer) and dz_small (fp32 [P,4]:
 * d rgb_pre[3], d sigma_pre).  Weight/bias gradients are dZ^T * layer-input GEMMs
 * over those planes (plain GEMMs, done by the caller). */
/* Input gradient of the same decoder from the planes of b2n_nerf_mlp_bwd:
 * g_x [P,pos_dim] = dZ0 * W0 + dZ4 * W4[:, 256:256+pos_dim] (x feeds layer 0 and the skip concat of
 * layer 4).  dz0 / dz4: bf16 [P][256] planes (dz_planes[9] / dz_planes[5]); W0 = pts_layers[0].weight
 * (row stride ldw0), W4x = pts_layers[4].weight + 256 (row stride ldw4).  Needed by Part 3
 * (src/core.py:268-277: the decoder input depends on the trainable deformation). */
int b2n_nerf_mlp_dx(const void* dz0, const void* dz4, const float* W0, int ldw0, const float* W4x, int ldw4, int pos_dim,
                    int64_t P, float* g_x, int ldg, b2n_stream_t stream);
/* Weight / bias gradients of the same decoder on tcgen05 (MN-major operands: the point-major planes are consumed as
 * they lie, TMA-loaded; one launch).  dz_planes / fwd_planes = bf16 [10][P][256] of b2n_nerf_mlp_bwd / _fwd; x_bf16 = bf16
 * [P][kx] encoded positions zero-padded to kx = 64 or 128 columns; d_bf16 = bf16 [P][64] encoded directions, zero-padded.
 * All outputs fp32 and ACCUMULATED: dW [8][256][256]: dW[l-1] = dZ_l^T H_{l-1} for trunk layers l = 1..7 (skip layer 4:
 * its first 256 input columns), dW[7] = dZ_feat^T H_7; dW0 [256][kx] = dZ_0^T x; dW4x [256][kx] = dZ_4^T x; dWv_h
 * [128][256] = dZ_view^T H_8; dWv_d [128][64] = dZ_view^T d; db [10][256] = column sums of every dZ plane (slot 0 view
 * layer, 1 feature layer, 2..9 = trunk layers 7..0).  x_bf16 / d_bf16 and their outputs may be NULL.  P >= 64.  The two
 * 1- and 3-row heads stay with the caller. */
/* out[p, 0:kpad] (bf16) = x[p, 0:width] (fp32) zero-padded; kpad a multiple of 8.  Builds x_bf16 / d_bf16 of
 * b2n_nerf_mlp_wgrad in one pass. */
int b2n_pad_bf16(const float* x, int64_t P, int width, int kpad, void* out, b2n_stream_t stream);
/* The two small heads of the same decoder (sigma_layer 1 x 256 on H_7, rgb_layer 3 x 128 on hv), one streaming pass:
 * dz_small [P,4] fp32 of b2n_nerf_mlp_bwd, h7 / hv = planes 7 and 9 of b2n_nerf_mlp_fwd (bf16 [P][256]).  ACCUMULATES
 * gw_sigma [256], gw_rgb [3][128], gb [4] (rgb biases, then the sigma bias). */
int b2n_nerf_mlp_head_wgrad(const float* dz_small, const void* h7_plane, const void* hv_plane, int64_t P, float* gw_sigma,
                            float* gw_rgb, float* gb, b2n_stream_t stream);
int b2n_nerf_mlp_wgrad(const void* dz_planes, const void* fwd_planes, const void* x_bf16, int kx, const void* d_bf16,
                       int64_t P, float* dW, float* dW0, float* dW4x, float* dWv_h, float* dWv_d, float* db,
                       int* err_flag, b2n_stream_t stream);
size_t b2n_nerf_mlp_packed_bwd_bytes(void);
int b2n_nerf_mlp_pack_bwd(const float* const* pts_w, const float* feature_w, const float* view_w, int pos_dim,
                          int dir_dim, void* packed, b2n_stream_t stream);
int b2n_nerf_mlp_bwd(const void* packed_bwd, const float* w_sigma, const float* w_rgb, const void* relu_masks,
                     const float* rgb, const float* sigma, const float* g_rgb, const float* g_sigma, int64_t P,
                     void* dz_planes, float* dz_small, int* err_flag, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * GPU-resident training-ray sampler (sample_random_rays, src/dataset.py:147-171,
 * :268-294): poses [V,4,4] fp32, images [V,H,W,4] uint8 RGBA, times [V] or NULL;
 * img_idx / pix_y / pix_x: int64 [B] pixel picks (drawn by the caller, on the CPU
 * generator for reference-identical streams or on the device) -> rays_o [B,3],
 * rays_d [B,3] (unit), target_rgba [B,4] in [0,1], t_out [B] (optional).
 * ---------------------------------------------------------------------- */
int b2n_sample_rays(const float* poses, const uint8_t* images_rgba8, const float* times, const int64_t* img_idx,
                    const int64_t* pix_y, const int64_t* pix_x, int64_t B, int V, int H, int W, float focal,
                    float scene_scale, float* rays_o, float* rays_d, float* target_rgba, float* t_out,
                    b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Per-step parameter update (SURVEY 8f-2): what run.py:611-630, :1112-1120 + :1167-1178, :1840-1859 + :1940-1949 do with
 * ~100 torch launches per step -- TV loss over the flat hash tables, GradScaler.unscale_, clip_grad_norm_, AdamW -- as two
 * passes.  Tensors are contiguous fp32 device buffers; the descriptor array lives on the HOST.
 *   b2n_opt_prepare: g <- g / *grad_scale (if given) + tv_scale * (sign(p[i]-p[i-1]) - sign(p[i+1]-p[i]))
 *                    (tv_scale = tv_weight / (n - 1): the gradient of tv_weight * mean|p[1:] - p[:-1]|, run.py:614-616);
 *                    norm2[clip_group] += sum g^2 (norm2: device float[B2N_OPT_MAX_GROUPS], zeroed by the caller).
 *   b2n_opt_adamw  : g * min(1, max_norm[group] / (sqrt(norm2[group]) + 1e-6)) (clip_grad_norm_; max_norm < 0 or norm2 NULL:
 *                    no clipping), then torch.optim.AdamW's update with the descriptor's hyper-parameters
 *                    (bias_corr = 1 - beta^step from the descriptor, or from the device scalar step_dev when given: a
 *                    step skipped for an inf must not advance it); nothing is written when *found_inf != 0.
 *                    already_unscaled = b2n_opt_prepare ran with the same grad_scale. */
#define B2N_OPT_MAX_TENSORS 40
#define B2N_OPT_MAX_GROUPS 8
typedef struct {
  float* p; float* g; float* m; float* v;
  int64_t n;
  float lr, weight_decay, beta1, beta2, eps, bias_corr1, bias_corr2, tv_scale;
  int clip_group;    /* -1: not part of any norm */
  int reserved;      /* set by the library (16-byte alignment of the four buffers); callers pass 0 */
} b2n_opt_tensor;
int b2n_opt_prepare(const b2n_opt_tensor* tensors, int n_tensors, const float* grad_scale, float* norm2,
                    b2n_stream_t stream);
int b2n_opt_adamw(const b2n_opt_tensor* tensors, int n_tensors, const float* grad_scale, int already_unscaled,
                  const float* found_inf, const float* step_dev, const float* norm2, const float* max_norm_host,
                  b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Surface extraction (marching tetrahedra) from a density lattice: the closed triangle mesh of the region sigma > tau,
 * e.g. of the lattice that DensityGrid.update sweeps (src/renderer.py:49-116), at any resolution 2 <= R <= 1024.
 *   sigma [R,R,R] fp32, index [ix,iy,iz] (x slowest) = the point (axis[ix], axis[iy], axis[iz]) of a 1-D axis (torch's
 *     linspace(-bound, bound, R) in the Python API).  A point is INSIDE when sigma > tau (strict, as `grid > threshold`);
 *     tau > 0 and finite.
 *   The lattice is padded with a virtual ring of points where sigma = 0, so every surface is closed: the EXTENDED axis
 *     axis_ext [R+2] = {axis[0] - h, axis[0..R-1], axis[R-1] + h}, h = axis[1] - axis[0] (fp32), is what the vertex
 *     coordinates come from.  Points of the extended lattice are numbered p = (i*(R+2) + j)*(R+2) + k.
 *   Every cell is split into the 6 Kuhn tetrahedra {0, e_a, e_a+e_b, e_a+e_b+e_c} for the permutations (a,b,c) of the
 *     axes in lexicographic order xyz, xzy, yxz, yzx, zxy, zyx.  Their edges run from a point p to p + d, d one of 7
 *     direction classes in the order x, y, z, xy, xz, yz, xyz.  Each edge whose ends lie on different sides of tau
 *     carries ONE vertex shared by every face around it: a = p, b = p + d, t = (tau - sigma_a) / (sigma_b - sigma_a),
 *     vertex = a + t*(b - a) per coordinate, each operation rounded separately (fp32, no fused multiply-add).
 *   A tetrahedron with 1 or 3 corners inside gives one triangle, with 2 inside a quad (ik, il, jl, jk) (i < j inside,
 *     k, l outside ordered so that (i,j,k,l) is an even permutation of the corners 0..3), split along ik - jl.  Every
 *     triangle is wound so that its normal points from inside to outside (derived from the case and the tetrahedron's
 *     parity, never from coordinates).
 *   Order (deterministic, no atomics): vertices by point p, then direction class; faces by cell (= its lowest point p),
 *     then tetrahedron, then triangle.
 * b2n_mesh_count: sigma -> totals (device int64 [2]: number of vertices V, faces F; exact, even when they exceed int32)
 *   and the per-point counts in scratch (b2n_mesh_scratch(R) bytes, 256-byte aligned; 0 for an unsupported R).
 * b2n_mesh_emit: with the same sigma, tau and scratch, and V / F read back from totals -> verts [V,3] fp32 (world
 *   coordinates), faces [F,3] int32 vertex ids.  Refuses V or F >= 2^31.  Two kernels; V == 0 is a no-op.
 * The host read of the totals between the two calls is the only synchronisation of an extraction. */
size_t b2n_mesh_scratch(int R);
int b2n_mesh_count(const float* sigma, int R, float threshold, void* scratch, int64_t* totals, b2n_stream_t stream);
int b2n_mesh_emit(const float* sigma, const float* axis_ext, int R, float threshold, void* scratch, int64_t n_verts,
                  int64_t n_faces, float* verts, int32_t* faces, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Inference rendering with early ray termination (b2n.render; DESIGN.md §5g).  Not the reference's render_rays: a
 * separate contract that equals the masked render_rays(perturb=False, density_grid) at eps = 0.
 *   Samples: depth z_s = z_base[s] (s < N <= 1024), point o + d*z_s with separately rounded fp32 operations (bitwise
 *     the points of b2n_march_compact), active iff bit s of the ray's mask_words (b2n_march_mask with u = z = NULL,
 *     then b2n_march_scan when a grid is used, which keeps the forced sample 0 of ray 0 of an all-empty mask).
 *   Compositing: the active samples of a ray, front to back, one at a time, with the per-sample arithmetic of
 *     b2n_composite_fwd: delta_s = (z_base[s+1] - z_base[s]) * |d| (1e10 * |d| for s = N-1; z_base[s+1] is the next
 *     depth of the full grid, active or not), alpha = 1 - expf(-sigma * delta), w = alpha * T, T <- T * (1 - alpha +
 *     1e-10), color += w * rgb, depth += w * z_s, acc += w, each operation rounded separately.  After a sample, T < eps
 *     ends the ray: none of its later samples count (eps = 0: never).  N == 1 composites nothing (pure background).
 *   Only the order of the transmittance product differs from b2n_composite_fwd (a sequential chain instead of a warp
 *   scan).  The per-ray state lives in fp32 across waves, so the result does not depend on how the samples of a ray
 *   are grouped into waves.  For eps > 0 and colours, bg in [0, 1], color and acc lie within T_stop <= eps of the
 *   eps = 0 result and depth within eps * far (plus fp32 rounding).
 * A render is a loop of waves over the ALIVE rays (int32 ray ids, ascending):
 *   b2n_render_begin: state [B] (32 bytes per ray: T, colour, depth, acc, cursor) initialised, alive = the rays with at
 *     least one active sample, *n_alive (device int32) = their number.  3 kernels.
 *   b2n_render_emit: for alive[0..n_alive), the next (up to) K active samples after each ray's cursor, compacted in
 *     (alive slot, sample) order: sample_idx (s), pts [P,3], dirs [P,3] (d/|d|, as b2n_march_compact), t_out [P]
 *     (the ray's time; NULL when times is NULL), and *total (device int32) = P.  3 kernels (count, scan, write).
 *   b2n_render_composite: rgb [P,3], sigma [P] of those samples (the model's output) folded into the state of every
 *     alive ray; the rays that are not done (T >= eps and an active sample left) go, in order, to alive_next, and
 *     *n_alive_next (device int32) = their number.  Takes the alive list, n_alive and scratch of the emit before it;
 *     alive_next must not alias alive.  3 kernels (fold, scan, write).
 *   b2n_render_finish: color [B,3] = colour + (1 - acc) * bg, depth [B], acc [B] of every ray; bg [3] (bg_per_ray = 0)
 *     or [B,3] (bg_per_ray = 1).
 * scratch: b2n_render_scratch(B) bytes, shared by begin / emit / composite.  The host reads *n_alive (to size the next
 * wave) and *total (to size the model call): two 4-byte reads per wave and no other synchronisation.  Those reads make
 * a render impossible to capture in a CUDA graph, by design.  B * N < 2^31 and n_alive * K < 2^31. */
size_t b2n_render_scratch(int64_t B);
int b2n_render_begin(const uint32_t* mask_words, int64_t B, int N, void* state, int32_t* alive, int32_t* n_alive,
                     void* scratch, b2n_stream_t stream);
int b2n_render_emit(const float* rays_o, const float* rays_d, const float* times, const float* z_base,
                    const uint32_t* mask_words, int64_t B, int N, const void* state, const int32_t* alive,
                    int64_t n_alive, int K, int32_t* sample_idx, float* pts, float* dirs, float* t_out, int32_t* total,
                    void* scratch, b2n_stream_t stream);
int b2n_render_composite(const float* rgb, const float* sigma, const float* z_base, const float* rays_d, int64_t B,
                         int N, float eps, void* state, const int32_t* alive, int64_t n_alive,
                         const int32_t* sample_idx, int32_t* alive_next, int32_t* n_alive_next, void* scratch,
                         b2n_stream_t stream);
int b2n_render_finish(const void* state, int64_t B, const float* bg, int bg_per_ray, float* color, float* depth,
                      float* acc, b2n_stream_t stream);

/* ------------------------------------------------------------------------
 * Hierarchical importance sampling (b2n.importance; DESIGN.md §5h): NeRF's sample_pdf (Mildenhall et al. 2020) on the
 * GPU.  Not part of the reference, which samples one stratified pass; an extension that is off unless asked for.
 * Per ray r < B, with sorted coarse depths z [B,Nc] (jittered or not) and coarse densities sigma [B,Nc]:
 *   Weights, with the arithmetic of b2n_composite_fwd: delta_s = (z_{s+1} - z_s) * |d| (1e10 * |d| for s = Nc-1),
 *     alpha_s = 1 - exp(-sigma_s * delta_s), T_0 = 1, T_{s+1} = T_s * (1 - alpha_s + 1e-10), w_s = alpha_s * T_s;
 *     alpha is computed as -expm1f(-sigma * delta), which keeps the small weights of a nearly empty ray accurate.
 *   Bins: the Nc-1 midpoints m_i = (z_i + z_{i+1}) / 2.  PDF: w_1 .. w_{Nc-2} (first and last dropped), each + 1e-5,
 *     normalised; CDF c [Nc-1] = [0, cumsum(pdf)] (c[Nc-2] = 1; kept non-decreasing in fp32 by a running max).
 *   Fine positions u_k, k < Nf: u_table [Nf] (deterministic: torch.linspace(0, 1, Nf), built on the host), or
 *     u_k = (k + U[r,k]) / Nf from u_jitter U [B,Nf] in [0,1) (stratified).  Exactly one of the two must be given.
 *   Inverse CDF: i = searchsorted(c, u, right=True), below = max(i-1, 0), above = min(i, Nc-2),
 *     denom = c[above] - c[below] (1 if < 1e-5), t = (u - c[below]) / denom,
 *     z_fine[r,k] = m[below] + t * (m[above] - m[below]), clamped to [m[below], m[above]] (which only absorbs rounding).
 *     Every index is clamped: no input, a non-finite sigma included, reads out of range.  u non-decreasing in k makes
 *     z_fine non-decreasing in k, inside [m_0, m_{Nc-2}].
 *   Merge: z_merged [B,Nc+Nf] = the coarse and fine depths merged, non-decreasing, coarse before fine on ties;
 *     merge_src [B,Nc+Nf] int32 = the source of each slot: s for coarse slot s, Nc + k for fine slot k.  z_merged is
 *     bitwise the source value.
 * Limits: Nc >= 3, Nf >= 1, Nc + Nf <= 1024 (b2n_composite_*'s limit); refused before any launch.  One kernel, one warp
 * per ray, no atomics, no host synchronisation (capturable in a CUDA graph), deterministic.  Reads 8*Nc bytes per ray
 * (+ 4*Nf with u_jitter), writes 4*Nf + 8*(Nc + Nf). */
int b2n_importance_sample(const float* sigma, const float* z, const float* rays_d, const float* u_table,
                          const float* u_jitter, int64_t B, int Nc, int Nf, float* z_fine, float* z_merged,
                          int32_t* merge_src, b2n_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B2NERF_H_ */
