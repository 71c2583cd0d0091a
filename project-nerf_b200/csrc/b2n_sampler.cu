// GPU-resident training-ray sampler (SURVEY.md 8f-1): replaces the CPU fancy-index gather + three
// H2D copies of BlenderDataset / DynamicDataset.sample_random_rays (src/dataset.py:147-171,
// :268-294).  The image stack lives in HBM as 8-bit RGBA (lossless: the PNGs are 8-bit and the
// reference's float conversion is v / 255), poses as fp32 4x4.  One thread per ray: pinhole
// direction ((x - W/2)/f, -(y - H/2)/f, -1), rotate by c2w[:3,:3], normalise, origin = c2w[:3,3]
// * scene_scale, target = rgba / 255, time = times[img].
#include <cub/device/device_radix_sort.cuh>

#include "b2n_common.cuh"

namespace b2n {

__global__ void k_sample_rays(const float* __restrict__ poses, const uint8_t* __restrict__ images,
                              const float* __restrict__ times, const int64_t* __restrict__ img_idx,
                              const int64_t* __restrict__ pix_y, const int64_t* __restrict__ pix_x, int64_t B, int V,
                              int H, int W, float focal, float scene_scale, float* __restrict__ rays_o,
                              float* __restrict__ rays_d, float* __restrict__ target, float* __restrict__ t_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int64_t v = img_idx[i], y = pix_y[i], x = pix_x[i];
  const float* M = poses + 16 * v;
  // same fp32 expression order as the reference: (pix - W*0.5) / focal
  const float dx = __fdiv_rn(__fsub_rn((float)x, (float)W * 0.5f), focal);
  const float dy = -__fdiv_rn(__fsub_rn((float)y, (float)H * 0.5f), focal);
  const float dz = -1.0f;
  float d[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) d[r] = M[4 * r] * dx + M[4 * r + 1] * dy + M[4 * r + 2] * dz;
  const float n = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    rays_d[3 * i + r] = __fdiv_rn(d[r], n);
    const float o = M[4 * r + 3];
    rays_o[3 * i + r] = scene_scale != 1.0f ? __fmul_rn(o, scene_scale) : o;
  }
  const uchar4 px = *reinterpret_cast<const uchar4*>(images + (((size_t)v * H + y) * W + x) * 4);
  float4 t;
  t.x = __fdiv_rn((float)px.x, 255.0f), t.y = __fdiv_rn((float)px.y, 255.0f);
  t.z = __fdiv_rn((float)px.z, 255.0f), t.w = __fdiv_rn((float)px.w, 255.0f);
  *reinterpret_cast<float4*>(target + 4 * i) = t;
  if (t_out) t_out[i] = times[v];
}

// ---- backward to the poses (pose refinement, DESIGN.md §5k) --------------------------------------------------------
// Rays are grouped by view with a stable radix sort of (view, ray index); one block per view then sums its rays in
// sorted order in fp64 and combines its warps in a fixed order.  No float atomics: the same inputs give the same bits.
constexpr int kPoseThreads = 256;

// sort key: the view id, or V (sorted last, never summed) for an id outside [0, V)
__global__ void k_pose_keys(const int64_t* __restrict__ img_idx, int64_t B, int V, uint32_t* __restrict__ keys,
                            int32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int64_t v = img_idx[i];
  keys[i] = (v >= 0 && v < V) ? (uint32_t)v : (uint32_t)V;
  vals[i] = (int32_t)i;
}

// [start[v], end[v]) = the sorted positions of view v (both left 0 for a view without rays)
__global__ void k_pose_bounds(const uint32_t* __restrict__ keys, int64_t B, int V, int32_t* __restrict__ start,
                              int32_t* __restrict__ end) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= B) return;
  const uint32_t k = keys[p];
  if (k >= (uint32_t)V) return;
  if (p == 0 || keys[p - 1] != k) start[k] = (int32_t)p;
  if (p == B - 1 || keys[p + 1] != k) end[k] = (int32_t)(p + 1);
}

__global__ void __launch_bounds__(kPoseThreads)
k_pose_reduce(const float* __restrict__ poses, const int64_t* __restrict__ pix_y, const int64_t* __restrict__ pix_x,
              const int32_t* __restrict__ order, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
              int H, int W, float focal, float scene_scale, const float* __restrict__ g_o,
              const float* __restrict__ g_d, float* __restrict__ g_poses) {
  __shared__ double part[kPoseThreads / 32][12];
  const int v = blockIdx.x;
  const float* M = poses + 16 * (int64_t)v;
  double R[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) R[3 * r + c] = (double)M[4 * r + c];
  double acc[12];                                    // g_R row-major [0, 9), g_t [9, 12)
#pragma unroll
  for (int k = 0; k < 12; ++k) acc[k] = 0.0;
  for (int p = start[v] + threadIdx.x; p < end[v]; p += kPoseThreads) {
    const int64_t i = order[p];
    // the camera direction of k_sample_rays, bit for bit
    const float cx = __fdiv_rn(__fsub_rn((float)pix_x[i], (float)W * 0.5f), focal);
    const float cy = -__fdiv_rn(__fsub_rn((float)pix_y[i], (float)H * 0.5f), focal);
    const double c[3] = {(double)cx, (double)cy, -1.0};
    double d[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) d[r] = R[3 * r] * c[0] + R[3 * r + 1] * c[1] + R[3 * r + 2] * c[2];
    const double n = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    double g[3], dot = 0.0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      d[r] /= n;
      g[r] = (double)__ldg(g_d + 3 * i + r);
      dot += d[r] * g[r];
    }
    // d(d/|d|)/dd = (I - dh dh^T) / |d|;  dd/dR = . (x) c
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const double gr = (g[r] - d[r] * dot) / n;
#pragma unroll
      for (int k = 0; k < 3; ++k) acc[3 * r + k] += gr * c[k];
      acc[9 + r] += (double)scene_scale * (double)__ldg(g_o + 3 * i + r);
    }
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 12; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 12; ++k) part[wid][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    const int r = threadIdx.x >> 2, c = threadIdx.x & 3;
    float out = 0.f;
    if (r < 3) {
      const int k = c < 3 ? 3 * r + c : 9 + r;
      double s = 0.0;
      for (int w = 0; w < kPoseThreads / 32; ++w) s += part[w][k];
      out = (float)s;
    }
    g_poses[16 * (int64_t)v + threadIdx.x] = out;
  }
}

struct PoseScratch {
  uint32_t *keys, *keys_sorted;
  int32_t *vals, *order, *start, *end;
  void* sort_tmp;
  size_t sort_bytes, bytes;
};

static int pose_key_bits(int V) { return 32 - __builtin_clz((unsigned)V); }   // keys 0 .. V

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// layout of the scratch of b2n_sample_rays_bwd; base == NULL only sizes it
static cudaError_t pose_scratch(void* base, int64_t B, int V, PoseScratch* s) {
  s->sort_bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, s->sort_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)B, 0,
                                                  pose_key_bits(V));
  if (e != cudaSuccess) return e;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t n) { void* q = p ? p + off : nullptr; off += align256(n); return q; };
  s->keys = (uint32_t*)take(4 * (size_t)B);
  s->keys_sorted = (uint32_t*)take(4 * (size_t)B);
  s->vals = (int32_t*)take(4 * (size_t)B);
  s->order = (int32_t*)take(4 * (size_t)B);
  s->start = (int32_t*)take(8 * (size_t)V);        // start [V] and end [V], one memset
  s->end = s->start ? s->start + V : nullptr;
  s->sort_tmp = take(s->sort_bytes);
  s->bytes = off;
  return cudaSuccess;
}

}  // namespace b2n

using namespace b2n;

extern "C" size_t b2n_sample_rays_bwd_scratch(int64_t B, int V) {
  if (B < 0 || B >= ((int64_t)1 << 31) || V <= 0) return 0;
  PoseScratch s;
  if (pose_scratch(nullptr, B > 0 ? B : 1, V, &s) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return s.bytes;
}

extern "C" int b2n_sample_rays_bwd(const float* poses, const int64_t* img_idx, const int64_t* pix_y,
                                   const int64_t* pix_x, int64_t B, int V, int H, int W, float focal, float scene_scale,
                                   const float* g_rays_o, const float* g_rays_d, float* g_poses, void* scratch,
                                   b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0 && B < ((int64_t)1 << 31) && V > 0 && H > 0 && W > 0 && focal > 0.f, "bad shape");
  B2N_REQUIRE(poses && g_poses, "null pointer");
  B2N_REQUIRE(B == 0 || (img_idx && pix_y && pix_x && g_rays_o && g_rays_d && scratch), "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {
    if (cudaMemsetAsync(g_poses, 0, 64 * (size_t)V, st) != cudaSuccess) return check_launch("b2n_sample_rays_bwd");
    return B2N_OK;
  }
  PoseScratch s;
  if (pose_scratch(scratch, B, V, &s) != cudaSuccess) return check_launch("b2n_sample_rays_bwd/scratch");
  k_pose_keys<<<grid_for(B, 256), 256, 0, st>>>(img_idx, B, V, s.keys, s.vals);
  if (cudaMemsetAsync(s.start, 0, 8 * (size_t)V, st) != cudaSuccess) return check_launch("b2n_sample_rays_bwd/memset");
  if (cub::DeviceRadixSort::SortPairs(s.sort_tmp, s.sort_bytes, s.keys, s.keys_sorted, s.vals, s.order, (int)B, 0,
                                      pose_key_bits(V), st) != cudaSuccess)
    return check_launch("b2n_sample_rays_bwd/sort");
  k_pose_bounds<<<grid_for(B, 256), 256, 0, st>>>(s.keys_sorted, B, V, s.start, s.end);
  k_pose_reduce<<<V, kPoseThreads, 0, st>>>(poses, pix_y, pix_x, s.order, s.start, s.end, H, W, focal, scene_scale,
                                            g_rays_o, g_rays_d, g_poses);
  return check_launch("b2n_sample_rays_bwd");
}

extern "C" int b2n_sample_rays(const float* poses, const uint8_t* images_rgba8, const float* times,
                               const int64_t* img_idx, const int64_t* pix_y, const int64_t* pix_x, int64_t B, int V,
                               int H, int W, float focal, float scene_scale, float* rays_o, float* rays_d,
                               float* target_rgba, float* t_out, b2n_stream_t stream) {
  B2N_REQUIRE(B >= 0 && V > 0 && H > 0 && W > 0 && focal > 0.f, "bad shape");
  if (B == 0) return B2N_OK;
  B2N_REQUIRE(poses && images_rgba8 && img_idx && pix_y && pix_x && rays_o && rays_d && target_rgba, "null pointer");
  B2N_REQUIRE(!t_out || times, "t_out needs times");
  k_sample_rays<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(poses, images_rgba8, times, img_idx, pix_y, pix_x, B,
                                                                   V, H, W, focal, scene_scale, rays_o, rays_d,
                                                                   target_rgba, t_out);
  return check_launch("b2n_sample_rays");
}
