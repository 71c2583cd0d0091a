// Inference rendering with early ray termination (b2n_render_* of include/b2nerf.h, DESIGN.md §5g).
//
// A render is a loop of waves over the alive rays.  Each wave emits the next K active samples of every alive ray
// (count -> scan -> write, order-preserving), the host runs the model on them, and the compositor folds them into the
// per-ray fp32 state one sample at a time, then compacts the rays that are not done into the next alive list
// (flag -> scan -> write).  One thread per alive ray everywhere; no atomics, so every output is deterministic.
//
// Bit-exactness: the points are o + d*z with __fadd_rn/__fmul_rn as in b2n_march_compact, and every compositing
// operation is rounded separately (no contraction into FMA), so a ray's result depends only on its samples, never on
// how they were grouped into waves.
#include "b2n_common.cuh"

namespace b2n {

struct RayState {
  float T, c0, c1, c2, depth, acc;
  int cursor;  // first active sample not yet composited (N: none left)
  int pad;
};
static_assert(sizeof(RayState) == 32, "RayState is 32 bytes per ray");

constexpr int kRT = 256;  // threads (= alive rays) per block of every kernel below

struct Scratch {
  int32_t *cnt, *ncur, *off, *flag, *block_sums;
};

__host__ __device__ inline int64_t render_blocks(int64_t B) { return (B + kRT - 1) / kRT; }

inline Scratch scratch_of(void* p, int64_t B) {
  int32_t* q = (int32_t*)p;
  return Scratch{q, q + B, q + 2 * B, q + 3 * B, q + 4 * B};
}

// first active sample at or after s (N if none).  Bits at or beyond N are never set in mask words.
__device__ __forceinline__ int next_active(const uint32_t* __restrict__ words, int W, int N, int s) {
  if (s >= N) return N;
  int k = s >> 5;
  uint32_t w = __ldg(words + k) & (0xffffffffu << (s & 31));
  while (!w) {
    if (++k >= W) return N;
    w = __ldg(words + k);
  }
  return (k << 5) + __ffs(w) - 1;
}

// exclusive scan of block sums in place, the grand total to *total (single block)
__global__ void __launch_bounds__(1024) k_render_scan_top(int32_t* __restrict__ block_sums, int nb,
                                                          int32_t* __restrict__ total) {
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
  if (threadIdx.x == 0) *total = carry;
}

// alive_next[pos] = alive[i] (or i when alive is NULL) for every flagged slot, in slot order
__global__ void __launch_bounds__(kRT) k_render_compact(const int32_t* __restrict__ alive, int64_t n,
                                                        const int32_t* __restrict__ flag,
                                                        const int32_t* __restrict__ block_sums,
                                                        int32_t* __restrict__ alive_next) {
  __shared__ int tot;
  const int64_t i = (int64_t)blockIdx.x * kRT + threadIdx.x;
  const int f = i < n ? flag[i] : 0;
  const int pos = block_exclusive_scan(f, &tot) + block_sums[blockIdx.x];
  if (f) alive_next[pos] = alive ? alive[i] : (int32_t)i;
}

__global__ void __launch_bounds__(kRT) k_render_begin(const uint32_t* __restrict__ words, int64_t B, int N,
                                                      RayState* __restrict__ state, int32_t* __restrict__ flag,
                                                      int32_t* __restrict__ block_sums) {
  __shared__ int tot;
  const int64_t r = (int64_t)blockIdx.x * kRT + threadIdx.x;
  const int W = (N + 31) >> 5;
  int f = 0;
  if (r < B) {
    const int cur = next_active(words + r * W, W, N, 0);
    state[r] = RayState{1.f, 0.f, 0.f, 0.f, 0.f, 0.f, cur, 0};
    f = cur < N;
    flag[r] = f;
  }
  block_exclusive_scan(f, &tot);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

// count: up to K active samples from the cursor on, and the first active sample after them
__global__ void __launch_bounds__(kRT) k_render_emit_count(const uint32_t* __restrict__ words, int N,
                                                           const RayState* __restrict__ state,
                                                           const int32_t* __restrict__ alive, int64_t n, int K,
                                                           int32_t* __restrict__ cnt, int32_t* __restrict__ ncur,
                                                           int32_t* __restrict__ block_sums) {
  __shared__ int tot;
  const int64_t i = (int64_t)blockIdx.x * kRT + threadIdx.x;
  const int W = (N + 31) >> 5;
  int c = 0;
  if (i < n) {
    const int64_t r = alive[i];
    const uint32_t* wr = words + r * W;
    const int cur = state[r].cursor;
    int k = cur >> 5, next = N;
    uint32_t w = __ldg(wr + k) & (0xffffffffu << (cur & 31));
    for (;;) {
      const int pc = __popc(w);
      if (c + pc >= K) {
        for (; c < K; ++c) w &= w - 1u;  // drop the samples this wave takes
        next = w ? (k << 5) + __ffs(w) - 1 : next_active(wr, W, N, (k + 1) << 5);
        break;
      }
      c += pc;
      if (++k >= W) break;
      w = __ldg(wr + k);
    }
    cnt[i] = c;
    ncur[i] = next;
  }
  block_exclusive_scan(c, &tot);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(kRT)
k_render_emit_write(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ times,
                    const float* __restrict__ z_base, const uint32_t* __restrict__ words, int N,
                    const RayState* __restrict__ state, const int32_t* __restrict__ alive, int64_t n,
                    const int32_t* __restrict__ cnt, const int32_t* __restrict__ block_sums, int32_t* __restrict__ off,
                    int32_t* __restrict__ sample_idx, float* __restrict__ pts, float* __restrict__ dirs,
                    float* __restrict__ t_out) {
  __shared__ int tot;
  const int64_t i = (int64_t)blockIdx.x * kRT + threadIdx.x;
  const int W = (N + 31) >> 5;
  const int c = i < n ? cnt[i] : 0;
  const int o0 = block_exclusive_scan(c, &tot) + block_sums[blockIdx.x];
  if (i >= n) return;
  off[i] = o0;
  const int64_t r = alive[i];
  const float ox = __ldg(rays_o + 3 * r), oy = __ldg(rays_o + 3 * r + 1), oz = __ldg(rays_o + 3 * r + 2);
  const float dx = __ldg(rays_d + 3 * r), dy = __ldg(rays_d + 3 * r + 1), dz = __ldg(rays_d + 3 * r + 2);
  const float nrm = sqrtf(dx * dx + dy * dy + dz * dz);  // the expression of b2n_march_compact
  const float vx = __fdiv_rn(dx, nrm), vy = __fdiv_rn(dy, nrm), vz = __fdiv_rn(dz, nrm);
  const float tt = times ? __ldg(times + r) : 0.f;
  const uint32_t* wr = words + r * W;
  const int cur = state[r].cursor;
  int k = cur >> 5;
  uint32_t w = __ldg(wr + k) & (0xffffffffu << (cur & 31));
  for (int64_t j = o0; j < (int64_t)o0 + c;) {
    if (!w) {
      w = __ldg(wr + ++k);
      continue;
    }
    const int s = (k << 5) + __ffs(w) - 1;
    w &= w - 1u;
    const float z = __ldg(z_base + s);
    sample_idx[j] = s;
    pts[3 * j] = __fadd_rn(ox, __fmul_rn(dx, z));
    pts[3 * j + 1] = __fadd_rn(oy, __fmul_rn(dy, z));
    pts[3 * j + 2] = __fadd_rn(oz, __fmul_rn(dz, z));
    dirs[3 * j] = vx, dirs[3 * j + 1] = vy, dirs[3 * j + 2] = vz;
    if (t_out) t_out[j] = tt;
    ++j;
  }
}

__global__ void __launch_bounds__(kRT)
k_render_fold(const float* __restrict__ rgb, const float* __restrict__ sigma, const float* __restrict__ z_base,
              const float* __restrict__ rays_d, int N, float eps, RayState* __restrict__ state,
              const int32_t* __restrict__ alive, int64_t n, const int32_t* __restrict__ sample_idx,
              const int32_t* __restrict__ cnt, const int32_t* __restrict__ ncur, const int32_t* __restrict__ off,
              int32_t* __restrict__ flag, int32_t* __restrict__ block_sums) {
  __shared__ int tot;
  const int64_t i = (int64_t)blockIdx.x * kRT + threadIdx.x;
  int f = 0;
  if (i < n) {
    const int64_t r = alive[i];
    RayState st = state[r];
    const float d0 = __ldg(rays_d + 3 * r), d1 = __ldg(rays_d + 3 * r + 1), d2 = __ldg(rays_d + 3 * r + 2);
    const float dn = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);  // the expression of b2n_composite_fwd
    const int64_t o0 = off[i], o1 = o0 + cnt[i];
    bool done = false;
    if (N > 1) {  // N == 1: the reference composites nothing
      for (int64_t j = o0; j < o1; ++j) {
        const int s = __ldcs(sample_idx + j);
        const float zs = __ldg(z_base + s);
        const float dl = __fmul_rn(s == N - 1 ? 1e10f : __fsub_rn(__ldg(z_base + s + 1), zs), dn);
        const float alpha = __fsub_rn(1.0f, expf(-__fmul_rn(__ldcs(sigma + j), dl)));
        const float wt = __fmul_rn(alpha, st.T);
        st.T = __fmul_rn(st.T, __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f));
        st.c0 = __fadd_rn(st.c0, __fmul_rn(wt, __ldcs(rgb + 3 * j)));
        st.c1 = __fadd_rn(st.c1, __fmul_rn(wt, __ldcs(rgb + 3 * j + 1)));
        st.c2 = __fadd_rn(st.c2, __fmul_rn(wt, __ldcs(rgb + 3 * j + 2)));
        st.depth = __fadd_rn(st.depth, __fmul_rn(wt, zs));
        st.acc = __fadd_rn(st.acc, wt);
        if (st.T < eps) {
          done = true;
          break;
        }
      }
    }
    st.cursor = done ? N : ncur[i];
    state[r] = st;
    f = st.cursor < N;
    flag[i] = f;
  }
  block_exclusive_scan(f, &tot);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(kRT) k_render_finish(const RayState* __restrict__ state, int64_t B,
                                                       const float* __restrict__ bg, int bg_per_ray,
                                                       float* __restrict__ color, float* __restrict__ depth,
                                                       float* __restrict__ acc) {
  const int64_t r = (int64_t)blockIdx.x * kRT + threadIdx.x;
  if (r >= B) return;
  const RayState st = state[r];
  float c0 = st.c0, c1 = st.c1, c2 = st.c2;
  const float* b = bg + (bg_per_ray ? 3 * r : 0);
  const float rem = 1.0f - st.acc;  // the background term of b2n_composite_fwd
  c0 += rem * b[0], c1 += rem * b[1], c2 += rem * b[2];
  color[3 * r] = c0, color[3 * r + 1] = c1, color[3 * r + 2] = c2;
  depth[r] = st.depth;
  acc[r] = st.acc;
}

}  // namespace b2n

using namespace b2n;

extern "C" size_t b2n_render_scratch(int64_t B) {
  if (B < 0) return 0;
  return (size_t)(4 * B + render_blocks(B) + 1) * sizeof(int32_t);
}

#define B2N_RENDER_SIZES(B, N)                                                   \
  B2N_REQUIRE((B) > 0 && (N) > 0 && (N) <= 1024, "need B > 0 and 0 < N <= 1024"); \
  B2N_REQUIRE((B) * (int64_t)(N) < (int64_t)1 << 31, "B*N must fit int32")

extern "C" int b2n_render_begin(const uint32_t* mask_words, int64_t B, int N, void* state, int32_t* alive,
                                int32_t* n_alive, void* scratch, b2n_stream_t stream) {
  B2N_RENDER_SIZES(B, N);
  B2N_REQUIRE(mask_words && state && alive && n_alive && scratch, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const Scratch sc = scratch_of(scratch, B);
  const int nb = (int)render_blocks(B);
  k_render_begin<<<nb, kRT, 0, st>>>(mask_words, B, N, (RayState*)state, sc.flag, sc.block_sums);
  k_render_scan_top<<<1, 1024, 0, st>>>(sc.block_sums, nb, n_alive);
  k_render_compact<<<nb, kRT, 0, st>>>(nullptr, B, sc.flag, sc.block_sums, alive);
  return check_launch("b2n_render_begin");
}

extern "C" int b2n_render_emit(const float* rays_o, const float* rays_d, const float* times, const float* z_base,
                               const uint32_t* mask_words, int64_t B, int N, const void* state, const int32_t* alive,
                               int64_t n_alive, int K, int32_t* sample_idx, float* pts, float* dirs, float* t_out,
                               int32_t* total, void* scratch, b2n_stream_t stream) {
  B2N_RENDER_SIZES(B, N);
  B2N_REQUIRE(n_alive >= 0 && n_alive <= B, "need 0 <= n_alive <= B");
  B2N_REQUIRE(K >= 1 && K <= N, "need 1 <= K <= N");
  B2N_REQUIRE(n_alive * (int64_t)K < (int64_t)1 << 31, "n_alive*K must fit int32");
  B2N_REQUIRE(rays_o && rays_d && z_base && mask_words && state && alive && sample_idx && pts && dirs && total &&
                  scratch,
              "null pointer");
  B2N_REQUIRE(!t_out || times, "t_out needs times");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_alive == 0) {
    if (cudaMemsetAsync(total, 0, sizeof(int32_t), st) != cudaSuccess) return check_launch("b2n_render_emit/memset");
    return B2N_OK;
  }
  const Scratch sc = scratch_of(scratch, B);
  const int nb = (int)render_blocks(n_alive);
  const RayState* s = (const RayState*)state;
  k_render_emit_count<<<nb, kRT, 0, st>>>(mask_words, N, s, alive, n_alive, K, sc.cnt, sc.ncur, sc.block_sums);
  k_render_scan_top<<<1, 1024, 0, st>>>(sc.block_sums, nb, total);
  k_render_emit_write<<<nb, kRT, 0, st>>>(rays_o, rays_d, times, z_base, mask_words, N, s, alive, n_alive, sc.cnt,
                                          sc.block_sums, sc.off, sample_idx, pts, dirs, t_out);
  return check_launch("b2n_render_emit");
}

extern "C" int b2n_render_composite(const float* rgb, const float* sigma, const float* z_base, const float* rays_d,
                                    int64_t B, int N, float eps, void* state, const int32_t* alive, int64_t n_alive,
                                    const int32_t* sample_idx, int32_t* alive_next, int32_t* n_alive_next,
                                    void* scratch, b2n_stream_t stream) {
  B2N_RENDER_SIZES(B, N);
  B2N_REQUIRE(n_alive >= 0 && n_alive <= B, "need 0 <= n_alive <= B");
  B2N_REQUIRE(eps >= 0.f && eps < 1.f, "need 0 <= eps < 1 (finite)");  // NaN fails both
  B2N_REQUIRE(rgb && sigma && z_base && rays_d && state && alive && sample_idx && alive_next && n_alive_next &&
                  scratch,
              "null pointer");
  B2N_REQUIRE(alive_next != alive, "alive_next must not alias alive");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_alive == 0) {
    if (cudaMemsetAsync(n_alive_next, 0, sizeof(int32_t), st) != cudaSuccess)
      return check_launch("b2n_render_composite/memset");
    return B2N_OK;
  }
  const Scratch sc = scratch_of(scratch, B);
  const int nb = (int)render_blocks(n_alive);
  k_render_fold<<<nb, kRT, 0, st>>>(rgb, sigma, z_base, rays_d, N, eps, (RayState*)state, alive, n_alive, sample_idx,
                                    sc.cnt, sc.ncur, sc.off, sc.flag, sc.block_sums);
  k_render_scan_top<<<1, 1024, 0, st>>>(sc.block_sums, nb, n_alive_next);
  k_render_compact<<<nb, kRT, 0, st>>>(alive, n_alive, sc.flag, sc.block_sums, alive_next);
  return check_launch("b2n_render_composite");
}

extern "C" int b2n_render_finish(const void* state, int64_t B, const float* bg, int bg_per_ray, float* color,
                                 float* depth, float* acc, b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0, "negative B");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(state && bg && color && depth && acc, "null pointer");
  k_render_finish<<<(unsigned)render_blocks(B), kRT, 0, (cudaStream_t)stream>>>((const RayState*)state, B, bg,
                                                                               bg_per_ray ? 1 : 0, color, depth, acc);
  return check_launch("b2n_render_finish");
}
