/* b2nerf_debug.h -- development / measurement entry points of libb2nerf.so.
 *
 * NOT part of the drop-in boundary (include/b2nerf.h): nothing in project-nerf_b200/src or b2n/ops.py calls these on a
 * product path.  They exist for tools/kbench.py, tools/mnmajor_probe.py, the A/B parity tests of kernel schedules and
 * bench.py's L2 gather peak.  Same conventions as b2nerf.h (int return code, b2n_last_error()).
 */
#ifndef B2NERF_DEBUG_H_
#define B2NERF_DEBUG_H_
#include "b2nerf.h"
#ifdef __cplusplus
extern "C" {
#endif

/* per-role cycle counters of CTA 0 of the next b2n_nerf_mlp_* launches (device int64[8 + 448]: 8 counters, then a
 * clock64 timeline of CTA 0's third tile pair, [step][tile][16 events]; or NULL) */
int b2n_debug_mlp256_prof(void* device_int64x8);
/* timing experiments only (results become garbage): 1 = the epilogue skips the accumulator drain,
 * 2 = no MMAs are issued (weights still stream); 0 = normal */
int b2n_debug_mlp256_flags(int flags);
/* schedule of b2n_nerf_mlp_fwd / _bwd: 1 (default; environment B2N_MLP256_PAIR=0 turns it off) = clusters of two CTAs
 * issuing cta_group::2 MMAs (M = 256 over an SM pair, each CTA staging half of every weight chunk); 0 = one CTA per SM.
 * Both produce the same results; the switch exists for A/B timing and parity tests. */
int b2n_debug_mlp256_set_pair(int on);

/* point tiles a CTA of b2n_instant_mlp_fwd_tc keeps in flight at pos_dim <= 32: 1 (default: 4 CTAs = 4 tiles per SM) or 2 (the
 * epilogue of one tile runs under the MMAs of the other; 3 CTAs = 6 tiles per SM; measured equal).  Same results.  Returns the previous
 * value. */
int b2n_debug_instant_fwd_slots(int slots);

/* schedule of b2n_instant_mlp_bwd_tc at pos_dim <= 32: 3 (default) = one CTA per SM with three 4-warp groups and a
 * single MMA issuer, 1 = two 4-warp CTAs per SM.  Same results up to the order of the fp32 accumulation.  Returns the
 * previous value. */
int b2n_debug_instant_bwd_groups(int groups);

/* A/B switch of the F = 2 hash-grid kernels: variant bit 0 = pair-lane forward (default on), bit 1 = pair-lane table
 * gradient (default on); 0 = the (point, level)-per-lane kernels.  merge_res >= 0 sets the coarsest-level run-merging
 * threshold of the pair-lane table gradient (levels with res <= merge_res are reduced across runs of equal cells).
 * B2N_EINVAL, and nothing changes, for a variant outside 0..3 or merge_res > 1625 (the merge path's uint32 cell id of a
 * level holds res^3). */
int b2n_debug_hash_variant(int variant, int merge_res);
/* the current variant and merge threshold (host ints), so that a caller can restore what it found */
int b2n_debug_hash_config(int* variant, int* merge_res);
/* table gradient of the spatially ordered F = 2 hash grid (b2n_hash_bwd_ordered): dedup_res > 0 takes the corners by
 * vertex parity and reduces equal table entries across the warp before the reductions on the levels with res <= dedup_res
 * (default 122); 0 = run merging up to merge_res, as in ray order.  Same table gradient up to the order of the fp32 sums.
 * dedup_res < 0 changes nothing.  Returns the previous value. */
int b2n_debug_hash_dedup(int dedup_res);

/* random 8-byte gathers over a float2[n_entries] table (n_entries = 2^k): the L2 gather peak the hash-grid kernels are
 * compared against (tools/kbench.py l2, bench.py hash_vs_l2) */
int b2n_debug_gather_bench(const float* table, int64_t n_entries, int blocks, int per_thread, float* sink,
                           b2n_stream_t stream);
/* random red.global.add over a float2[n_entries] table.  mode 0: every lane its own random entry (v2.f32); 1: lane pairs
 * on adjacent entries of one 16-byte pair; 2: groups of 4 lanes on the 4 entries of one 32-byte sector; 3: v4.f32 on a
 * random aligned entry pair, all lanes; 4: as 3, even lanes only; 5: as 0, even lanes only; 6: groups of 16 lanes on the
 * 16 entries of one 128-byte line */
int b2n_debug_red_bench(float* table, int64_t n_entries, int blocks, int per_thread, int mode, b2n_stream_t stream);

/* D[128x128] = A^T B through tcgen05.mma with MN-major shared-memory operands (A, B: bf16 [64][128], row = contraction
 * index); lbo / sbo / kadv (bytes) and extra instruction-descriptor bits are arguments */
int b2n_debug_mnmajor_probe(const void* A, const void* B, float* D, int lbo, int sbo, int kadv, int idesc_extra,
                            b2n_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B2NERF_DEBUG_H_ */
