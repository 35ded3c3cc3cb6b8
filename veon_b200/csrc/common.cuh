// Shared helpers for libveonlift (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/veon_lift.h"

#define VEON_CUDA_TRY(expr)                         \
  do {                                              \
    cudaError_t _e = (expr);                        \
    if (_e != cudaSuccess) return (int)_e;          \
  } while (0)

// every kernel launch of this library goes through here (counted for bench.py)
#define VEON_LAUNCH_CHECK()                         \
  do {                                              \
    cudaError_t _e = cudaGetLastError();            \
    if (_e != cudaSuccess) return (int)_e;          \
    veon_count_launch();                            \
  } while (0)

extern "C" void veon_count_launch(void);

namespace veon {

// ---- programmatic dependent launch --------------------------------------------------
// Chains of short kernels (the index preparation is seven of them) lose ~4-6 us per link
// to launch latency.  A kernel launched with launch_pdl() may be scheduled as soon as every
// CTA of its predecessor has executed pdl_launch_dependents(); it must call pdl_wait()
// before touching anything the predecessor (or, transitively, anything earlier in the
// stream) produced.  Both are no-ops for a normally launched grid.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// every kernel of a chain starts with this
__device__ __forceinline__ void pdl_prologue() {
  pdl_wait();
  pdl_launch_dependents();
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

constexpr int kTileVoxels = 32;  // one warp-wide x-run of the output volume

// A tile holding at least this many points is "heavy": one warp would serialise
// on it for longer than a whole average work share, so the plan lists such tiles
// and the forward hands each of them to a whole CTA (pool_fwd.cu).  The list
// capacity assumes the threshold never goes below kHeavyMinThreshold.
constexpr int kHeavyMinThreshold = 32;
#ifndef VEON_HEAVY_THR
#define VEON_HEAVY_THR 96
#endif
constexpr int kHeavyDefaultThreshold = VEON_HEAVY_THR;
inline int heavy_threshold() { return kHeavyDefaultThreshold; }
inline int64_t heavy_capacity(int64_t n_points, int64_t n_tiles) {
  const int64_t by_points = n_points / kHeavyMinThreshold;
  return by_points < n_tiles ? by_points : n_tiles;
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Launch configuration that depends on the device (opt-in shared-memory sizes, occupancy,
// SM count) is cached PER DEVICE: one process may drive several GPUs.
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}
inline int sm_count_total() {
  static int n[kMaxDevices] = {};
  const int dev = current_device();
  if (n[dev] == 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}
// SMs the caller wants left free (veon_reserve_sms): a collective running beside the path on
// another stream (NCCL) needs somewhere to put its CTAs -- persistent grids that fill every SM
// make it wait for a kernel boundary.
inline int& reserved_sms() {
  static int r = 0;
  return r;
}
// what the persistent grids size themselves by
inline int sm_count() {
  const int n = sm_count_total() - reserved_sms();
  return n < 1 ? 1 : n;
}

// Streaming stores/loads: the feature volume is written once and never re-read
// by the same kernel, so keep it from evicting the (L2-resident) rank / depth /
// feature inputs.
__device__ __forceinline__ void st_stream(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 v;
  asm volatile("ld.global.cs.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream(const float* p) {
  float v;
  asm volatile("ld.global.cs.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// bfloat16 volumes and gradients.  Sums stay float32; a stored value is rounded once, to nearest
// even (cvt.rn.bf16.f32, as torch's device-side cast), and a loaded one is widened exactly.  The
// overloads take the float32 helpers' element counts: st_stream4 / ld_stream4 move four elements,
// which for bfloat16 is one 8-byte access (8-byte aligned).
using bf16 = __nv_bfloat16;
__device__ __forceinline__ uint32_t bf16x2_bits(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);   // .x = lo at the lower address
  return (uint32_t)__bfloat16_as_ushort(h.x) | ((uint32_t)__bfloat16_as_ushort(h.y) << 16);
}
__device__ __forceinline__ void st_stream(bf16* p, float v) {
  asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"(__bfloat16_as_ushort(__float2bfloat16_rn(v)))
               : "memory");
}
__device__ __forceinline__ void st_stream4(bf16* p, float4 v) {
  asm volatile("st.global.cs.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(bf16x2_bits(v.x, v.y)),
               "r"(bf16x2_bits(v.z, v.w))
               : "memory");
}
__device__ __forceinline__ float widen(float v) { return v; }
__device__ __forceinline__ float widen(bf16 v) {
  return __uint_as_float((uint32_t)__bfloat16_as_ushort(v) << 16);
}
__device__ __forceinline__ float4 ld_stream4(const bf16* p) {
  uint32_t a, b;
  asm volatile("ld.global.cs.v2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
  // (not make_float4: another caller of it changes how the float kernels around it are inlined,
  //  and their code must stay as it is)
  float4 r;
  r.x = __uint_as_float(a << 16);
  r.y = __uint_as_float(a & 0xffff0000u);
  r.z = __uint_as_float(b << 16);
  r.w = __uint_as_float(b & 0xffff0000u);
  return r;
}
__device__ __forceinline__ float ld_stream(const bf16* p) {
  unsigned short h;
  asm volatile("ld.global.cs.b16 %0, [%1];" : "=h"(h) : "l"(p));
  return __uint_as_float((uint32_t)h << 16);
}
// read-only path, widened
__device__ __forceinline__ float ldg_widen(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_widen(const bf16* p) {
  return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}

// bfloat16 feature rows (the pooling's input under autocast): four channels are one 16-byte
// (float) or 8-byte (bf16, 8-byte aligned) read-only load, widened exactly in registers; a
// feature gradient stored as bf16 is rounded once, to nearest even.
__device__ __forceinline__ float4 ldg_widen4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float4 ldg_widen4(const bf16* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  float4 r;
  r.x = __uint_as_float(u.x << 16);
  r.y = __uint_as_float(u.x & 0xffff0000u);
  r.z = __uint_as_float(u.y << 16);
  r.w = __uint_as_float(u.y & 0xffff0000u);
  return r;
}
__device__ __forceinline__ void store_rn(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_rn(bf16* p, float v) { *p = __float2bfloat16_rn(v); }

// four elements of a row or a channel plane into shared memory: 16 bytes of float, 8 of bf16
// (cp.async.cg copies 16 bytes only)
__device__ __forceinline__ void cp_async_4(float* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_4(bf16* smem_dst, const bf16* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// _merge_classes_prob + the label rule for one voxel (san_in_veon_entry_temporal.py:273-297,
// veon_temporal.py:223-229,240); shared by the classify kernels and the fused lift + classify.
struct ClassMerge {  // running per-class max over prompt rows + first-index arg-max over classes
  float best = 0.f, cur = 0.f;
  int best_cls = -1, cur_cls = -1;
  bool bad = false;
  __device__ __forceinline__ void push(int cls, float logit) {
    bad |= !(logit < INFINITY);  // NaN / +inf => the softmax score is NaN => free
    if (cls != cur_cls) {
      if (cur_cls >= 0 && (best_cls < 0 || cur > best)) { best = cur; best_cls = cur_cls; }
      cur_cls = cls;
      cur = logit;
    } else {
      cur = fmaxf(cur, logit);
    }
  }
  __device__ __forceinline__ int label(float b0, float b1, int free_label) {
    if (cur_cls >= 0 && (best_cls < 0 || cur > best)) { best = cur; best_cls = cur_cls; }
    bad |= (best == -INFINITY);
    const float m = fmaxf(b0, b1);  // softmax(bin_occ)[0] > 0.5, evaluated like torch.softmax
    const float e0 = expf(b0 - m), e1 = expf(b1 - m);
    const bool occupied = (e0 / (e0 + e1)) > 0.5f;
    return (occupied && !bad) ? best_cls : free_label;
  }
};

}  // namespace veon
