// get_lidar_coor on the GPU: frustum points -> ego/lidar frame.
//
// Reference behaviour: LSSViewTransformer.get_lidar_coor,
// mmdet3d/models/necks/view_transformer.py:114-152 (view_transformer_raw.py:121-158):
// nine ATen launches, two batched torch.inverse calls and ~3 passes over the
// [B,N,D,H,W,3] tensor.  Here: one tiny kernel folds the per-camera 3x3 algebra
// (inverse of post_rots, sensor2ego[:3,:3] * inverse(cam2imgs), in float64 then
// rounded once), one streaming kernel applies it to every frustum point in the
// reference's operation order:
//     p = frustum - post_trans;  p = inv(post_rots) p;  p.xy *= p.z;
//     p = (R K^-1) p + t;        p = bda p
// Float results agree with the reference to rounding (it is upstream of the
// bit-exact op boundary; the ranks are defined on whatever `coor` is passed to
// voxel_pooling_prepare_v2).
#include "geometry.cuh"

namespace veon {

__device__ inline void inv3(const double* m, double* o) {
  const double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7],
               i = m[8];
  const double A = e * i - f * h, B = -(d * i - f * g), C = d * h - e * g;
  const double det = a * A + b * B + c * C;
  const double r = 1.0 / det;
  o[0] = A * r; o[1] = -(b * i - c * h) * r; o[2] = (b * f - c * e) * r;
  o[3] = B * r; o[4] = (a * i - c * g) * r;  o[5] = -(a * f - c * d) * r;
  o[6] = C * r; o[7] = -(a * h - b * g) * r; o[8] = (a * e - b * d) * r;
}

__global__ void k_cam_xforms(const float* __restrict__ sensor2ego,
                             const float* __restrict__ cam2imgs,
                             const float* __restrict__ post_rots,
                             const float* __restrict__ post_trans,
                             const float* __restrict__ bda, int B, int N,
                             CamXform* __restrict__ out) {
  pdl_launch_dependents();  // k_lidar_coor may be scheduled behind this grid (common.cuh)
  const int bn = blockIdx.x * blockDim.x + threadIdx.x;
  if (bn >= B * N) return;
  double pr[9], k[9], ipr[9], ik[9];
  for (int j = 0; j < 9; ++j) { pr[j] = post_rots[bn * 9 + j]; k[j] = cam2imgs[bn * 9 + j]; }
  inv3(pr, ipr);
  inv3(k, ik);
  CamXform x;
  const float* s = sensor2ego + (int64_t)bn * 16;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) {
      x.undo[r * 3 + c] = (float)ipr[r * 3 + c];
      double acc = 0.0;
      for (int j = 0; j < 3; ++j) acc += (double)s[r * 4 + j] * ik[j * 3 + c];
      x.c2e[r * 3 + c] = (float)acc;
    }
    x.pt[r] = post_trans[bn * 3 + r];
    x.t[r] = s[r * 4 + 3];
  }
  const float* bd = bda + (int64_t)(bn / N) * 9;
  for (int j = 0; j < 9; ++j) x.bda[j] = bd[j];
  out[bn] = x;
}

__global__ void __launch_bounds__(256)
k_lidar_coor(const float* __restrict__ frustum, const CamXform* __restrict__ xf, int64_t DHW,
             int64_t total, float* __restrict__ coor) {
  pdl_wait();
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int64_t bn = p / DHW, f = p - bn * DHW;
  float* o = coor + 3 * p;
  lidar_point(frustum + 3 * f, xf[bn], o[0], o[1], o[2]);
}

int launch_cam_xforms(const float* sensor2ego, const float* cam2imgs, const float* post_rots,
                      const float* post_trans, const float* bda, int B, int N, CamXform* xf,
                      cudaStream_t stream) {
  k_cam_xforms<<<(B * N + 63) / 64, 64, 0, stream>>>(sensor2ego, cam2imgs, post_rots, post_trans,
                                                     bda, B, N, xf);
  VEON_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------- layout change
// feat arrives as [B*N, C, H*W] (the network's channels-first maps,
// view_transformer.py:279-285 views + permutes it) and the pooling kernels gather
// channel-contiguous rows; the reference lets `.contiguous()` do the copy
// (bev_pool.py:88).  Batched tiled transpose [batch][R][S] -> [batch][S][R], used in
// both directions (feat forward, feat_grad backward).  E = uint16_t moves bfloat16 maps and
// gradients as bits: nothing is rounded.
template <typename E>
__global__ void __launch_bounds__(256)
k_transpose(const E* __restrict__ src, int R, int S, E* __restrict__ dst) {
  __shared__ E t[32][33];
  const int64_t base = (int64_t)blockIdx.z * R * S;
  const int s0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + 8 * i, c = s0 + tx;
    if (r < R && c < S) t[ty + 8 * i][tx] = __ldg(src + base + (int64_t)r * S + c);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = s0 + ty + 8 * i, r = r0 + tx;
    if (r < R && c < S) dst[base + (int64_t)c * R + r] = t[tx][ty + 8 * i];
  }
}

}  // namespace veon

using namespace veon;

extern "C" size_t veon_lidar_coor_workspace_bytes(int B, int N) {
  return (B > 0 && N > 0) ? sizeof(CamXform) * (size_t)B * N : 0;
}

extern "C" int veon_lidar_coor(const float* frustum, const float* sensor2ego,
                               const float* cam2imgs, const float* post_rots,
                               const float* post_trans, const float* bda, int B, int N, int D,
                               int H, int W, float* coor, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!frustum || !sensor2ego || !cam2imgs || !post_rots || !post_trans || !bda || !coor ||
      !workspace || B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0)
    return VEON_E_BADARG;
  if (workspace_bytes < sizeof(CamXform) * (size_t)B * N) return VEON_E_WORKSPACE;
  CamXform* xf = (CamXform*)workspace;
  int rc = launch_cam_xforms(sensor2ego, cam2imgs, post_rots, post_trans, bda, B, N, xf, stream);
  if (rc) return rc;
  const int64_t DHW = (int64_t)D * H * W, total = DHW * B * N;
  VEON_CUDA_TRY(launch_pdl(k_lidar_coor, dim3((unsigned)ceil_div64(total, 256)), dim3(256), 0, stream,
                           frustum, (const CamXform*)xf, DHW, total, coor));
  VEON_LAUNCH_CHECK();
  return 0;
}

template <typename E>
static int transpose_batched(const E* src, int64_t batch, int R, int S, E* dst,
                             cudaStream_t stream) {
  if (!src || !dst || batch <= 0 || R <= 0 || S <= 0) return VEON_E_BADARG;
  if (batch > 65535) return VEON_E_RANGE;
  const dim3 grid((unsigned)((S + 31) / 32), (unsigned)((R + 31) / 32), (unsigned)batch);
  k_transpose<<<grid, 256, 0, stream>>>(src, R, S, dst);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_transpose_batched(const float* src, int64_t batch, int R, int S, float* dst,
                                      void* stream) {
  return transpose_batched(src, batch, R, S, dst, (cudaStream_t)stream);
}

extern "C" int veon_transpose_batched_u16(const uint16_t* src, int64_t batch, int R, int S,
                                          uint16_t* dst, void* stream) {
  return transpose_batched(src, batch, R, S, dst, (cudaStream_t)stream);
}

// ---- calibration hash (SURVEY 8f-3: rank cache keyed on the calibration) ------------------------
// The reference's `accelerate` cache (view_transformer.py:154-173) assumes the calibration never
// changes.  A 64-bit hash of the five calibration tensors' BITS lets a caller keep the prepared
// ranks of every rig it has seen and re-use them whenever the same calibration comes back -- one
// tiny kernel and an 8-byte read instead of the whole index preparation.
namespace veon {
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {   // splitmix64 finaliser
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}
struct HashSpan { const float* p; int n; };
struct HashJobs { HashSpan s[5]; };

__global__ void __launch_bounds__(256)
k_calib_hash(HashJobs jobs, unsigned long long seed, unsigned long long* __restrict__ out) {
  __shared__ unsigned long long part[8];
  unsigned long long h = 0;
  unsigned long long base = 0;
  for (int j = 0; j < 5; ++j) {
    for (int i = threadIdx.x; i < jobs.s[j].n; i += blockDim.x)
      h += mix64((unsigned long long)__float_as_uint(jobs.s[j].p[i]) ^ ((base + i + 1) * 0x9e3779b97f4a7c15ull));
    base += (unsigned long long)jobs.s[j].n + 0x10000ull;   // position AND tensor matter
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = seed;
    for (int w = 0; w < 8; ++w) t += part[w];
    *out = mix64(t);
    __threadfence_system();
  }
}
}  // namespace veon

extern "C" int veon_calib_hash(const float* sensor2ego, const float* cam2imgs,
                               const float* post_rots, const float* post_trans, const float* bda,
                               int B, int N, uint64_t* out, void* stream) {
  if (!sensor2ego || !cam2imgs || !post_rots || !post_trans || !bda || !out || B <= 0 || N <= 0)
    return VEON_E_BADARG;
  veon::HashJobs jobs;
  jobs.s[0] = {sensor2ego, B * N * 16};
  jobs.s[1] = {cam2imgs, B * N * 9};
  jobs.s[2] = {post_rots, B * N * 9};
  jobs.s[3] = {post_trans, B * N * 3};
  jobs.s[4] = {bda, B * 9};
  veon::k_calib_hash<<<1, 256, 0, (cudaStream_t)stream>>>(
      jobs, ((unsigned long long)(unsigned)B << 32) | (unsigned)N,
      reinterpret_cast<unsigned long long*>(out));
  VEON_LAUNCH_CHECK();
  return 0;
}
