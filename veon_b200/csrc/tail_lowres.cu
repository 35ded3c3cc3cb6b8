// Open-vocabulary tail at the decoder's resolution (SURVEY.md 8f-4).
//
// The reference up-samples the decoder's feature volume to the Occ3D grid and classifies there:
//   feat_occ = F.interpolate(occ_preds["feat_occ"], size=occ_size, mode="trilinear",
//                            align_corners=False)             san_in_veon_temporal.py:196-201
//   bin_occ  = F.interpolate(occ_preds["bin_occ"], ...)        san_in_veon_temporal.py:202-207
//   sem_occ  = einsum("qc,bczhw->bqzhw", W, feat_occ)          san_in_veon_temporal.py:208,257-259
// Trilinear interpolation and the classifier are both linear and the interpolation weights do
// not depend on the channel, so  W . interp(feat) == interp(W . feat):  the contraction runs on
// the low-resolution volume (8x fewer voxels for 8x100x100 -> 16x200x200, on tcgen05 through
// veon_semantic_inference_3d) and only the Q logit channels are interpolated.  The up-sampled
// C-channel volume (1.31 GB per sample at C = 512) is never produced.
//
// This file: interpolation of the Q + 2 channels fused with the class merge, arg-max, gate and
// uint8 emission (san_in_veon_entry_temporal.py:273-297, veon_temporal.py:223-229,240).
// Source index and weights follow ATen's upsample_trilinear3d for align_corners=False:
//   src = max(scale * (dst + 0.5) - 0.5, 0), scale = in / out (float); i0 = (int)src;
//   i1 = i0 + (i0 < in - 1); l1 = src - i0; l0 = 1 - l1;
//   value = lz0 * (ly0 * (lx0 * a + lx1 * b) + ly1 * (lx0 * c + lx1 * d)) + lz1 * (same at z1).
#include <math.h>

#include "common.cuh"

namespace veon {

struct Axis {
  int i0, i1;
  float l0, l1;
};
__host__ __device__ __forceinline__ Axis axis_source(int dst, float scale, int in_size) {
  float src = scale * ((float)dst + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  Axis a;
  a.i0 = (int)src;
  if (a.i0 > in_size - 1) a.i0 = in_size - 1;
  a.i1 = a.i0 + (a.i0 < in_size - 1 ? 1 : 0);
  a.l1 = src - (float)a.i0;
  a.l0 = 1.f - a.l1;
  return a;
}


// The same for the ZO outputs of one (x, y) column: the prompt's class is the same for all of
// them, so the run bookkeeping is scalar and only the two maxima and the winner are per output.
template <int ZO>
struct ColumnMerge {
  float best[ZO], cur[ZO];
  int best_cls[ZO];
  uint32_t bad = 0;  // bit z: NaN / +inf seen => the softmax score is NaN => free
  int cur_cls = -1;
  bool have_best = false;
  __device__ __forceinline__ ColumnMerge() {
#pragma unroll
    for (int z = 0; z < ZO; ++z) { best[z] = 0.f; cur[z] = 0.f; best_cls[z] = -1; }
  }
  __device__ __forceinline__ void close_run() {
    if (cur_cls < 0) return;
#pragma unroll
    for (int z = 0; z < ZO; ++z)
      if (!have_best || cur[z] > best[z]) { best[z] = cur[z]; best_cls[z] = cur_cls; }
    have_best = true;
  }
  __device__ __forceinline__ void push(int cls, const float* v) {
    if (cls != cur_cls) {
      close_run();
      cur_cls = cls;
#pragma unroll
      for (int z = 0; z < ZO; ++z) cur[z] = v[z];
    } else {
#pragma unroll
      for (int z = 0; z < ZO; ++z) cur[z] = fmaxf(cur[z], v[z]);
    }
#pragma unroll
    for (int z = 0; z < ZO; ++z) bad |= (uint32_t)(!(v[z] < INFINITY)) << z;
  }
  // after the last push + close_run(): labels of the column, stored as [.., Z] bytes
  __device__ __forceinline__ void store(const float* b0, const float* b1, int free_label,
                                        uint8_t* dst) const {
    auto label = [&](int z) -> uint32_t {
      const bool is_bad = ((bad >> z) & 1u) || best[z] == -INFINITY;
      const float mx = fmaxf(b0[z], b1[z]);  // softmax(bin_occ)[0] > 0.5 as torch.softmax does it
      const float e0 = expf(b0[z] - mx), e1 = expf(b1[z] - mx);
      const bool occupied = (e0 / (e0 + e1)) > 0.5f;
      return (uint32_t)(uint8_t)((occupied && !is_bad) ? best_cls[z] : free_label);
    };
    if constexpr (ZO % 16 == 0) {
#pragma unroll
      for (int z0 = 0; z0 < ZO; z0 += 16) {
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          w[k] = 0;
#pragma unroll
          for (int i = 0; i < 4; ++i) w[k] |= label(z0 + 4 * k + i) << (8 * i);
        }
        *reinterpret_cast<uint4*>(dst + z0) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    } else {
#pragma unroll
      for (int z = 0; z < ZO; ++z) dst[z] = (uint8_t)label(z);
    }
  }
};

constexpr int kColThreads = 128;

// Fast path: one thread per output (x, y) column, all ZO outputs of the column in registers.
// Per prompt row the thread reads the 4 x ZI low-resolution neighbours once (2*ZI/ZO loads per
// output instead of 8), interpolates in-plane, then along z with compile-time z weights.
// Threads run along x, so a warp's loads fall into 1-3 sectors per (row, y, z).
#ifndef VEON_COLS_MINBLOCKS
#define VEON_COLS_MINBLOCKS 1
#endif
template <int ZI, int ZO>
__global__ void __launch_bounds__(kColThreads, VEON_COLS_MINBLOCKS)
k_upsample_classify_cols(const float* __restrict__ logits, const float* __restrict__ bin_occ,
                         const int32_t* __restrict__ class_of_prompt, int Q, int Yi, int Xi,
                         int Y, int X, float sy, float sx, int free_label,
                         uint8_t* __restrict__ labels) {
  const int b = blockIdx.y;
  const int idx = blockIdx.x * kColThreads + threadIdx.x;
  if (idx >= X * Y) return;
  const int x = idx % X, y = idx / X;
  const Axis ax = axis_source(x, sx, Xi), ay = axis_source(y, sy, Yi);
  const int o00 = ay.i0 * Xi + ax.i0, o01 = ay.i0 * Xi + ax.i1;
  const int o10 = ay.i1 * Xi + ax.i0, o11 = ay.i1 * Xi + ax.i1;
  const int64_t plane = (int64_t)Yi * Xi;
  const int64_t Vi = plane * ZI;
  constexpr float sz = (float)ZI / (float)ZO;

  auto column = [&](const float* __restrict__ src, float* out) {
    float col[ZI];
#pragma unroll
    for (int z = 0; z < ZI; ++z) {
      const float* p = src + z * plane;
      const float a = __ldg(p + o00), bb = __ldg(p + o01), c = __ldg(p + o10), d = __ldg(p + o11);
      col[z] = ay.l0 * (ax.l0 * a + ax.l1 * bb) + ay.l1 * (ax.l0 * c + ax.l1 * d);
    }
#pragma unroll
    for (int z = 0; z < ZO; ++z) {
      const Axis az = axis_source(z, sz, ZI);  // folded at compile time
      out[z] = az.l0 * col[az.i0] + az.l1 * col[az.i1];
    }
  };

  ColumnMerge<ZO> m;
  const float* lg = logits + (int64_t)b * Q * Vi;
  for (int q = 0; q < Q; ++q) {
    float v[ZO];
    column(lg + (int64_t)q * Vi, v);
    m.push(__ldg(class_of_prompt + q), v);
  }
  m.close_run();
  float b0[ZO], b1[ZO];
  column(bin_occ + ((int64_t)b * 2 + 0) * Vi, b0);
  column(bin_occ + ((int64_t)b * 2 + 1) * Vi, b1);
  m.store(b0, b1, free_label, labels + (((int64_t)b * X + x) * Y + y) * ZO);  // [B,X,Y,Z]
}

// Any other pair of sizes: one thread per output voxel, 8 neighbours per channel.
__global__ void __launch_bounds__(kColThreads)
k_upsample_classify_any(const float* __restrict__ logits, const float* __restrict__ bin_occ,
                        const int32_t* __restrict__ class_of_prompt, int Q, int Zi, int Yi, int Xi,
                        int Z, int Y, int X, float sz, float sy, float sx, int free_label,
                        uint8_t* __restrict__ labels) {
  const int b = blockIdx.y;
  const int64_t V = (int64_t)Z * Y * X;
  const int64_t v = (int64_t)blockIdx.x * kColThreads + threadIdx.x;
  if (v >= V) return;
  const int x = (int)(v % X), y = (int)((v / X) % Y), z = (int)(v / ((int64_t)X * Y));
  const Axis ax = axis_source(x, sx, Xi), ay = axis_source(y, sy, Yi), az = axis_source(z, sz, Zi);
  const int64_t plane = (int64_t)Yi * Xi, Vi = plane * Zi;
  const int o00 = ay.i0 * Xi + ax.i0, o01 = ay.i0 * Xi + ax.i1;
  const int o10 = ay.i1 * Xi + ax.i0, o11 = ay.i1 * Xi + ax.i1;
  auto sample = [&](const float* __restrict__ src) {
    const float* p0 = src + az.i0 * plane;
    const float* p1 = src + az.i1 * plane;
    const float lo = ay.l0 * (ax.l0 * __ldg(p0 + o00) + ax.l1 * __ldg(p0 + o01)) +
                     ay.l1 * (ax.l0 * __ldg(p0 + o10) + ax.l1 * __ldg(p0 + o11));
    const float hi = ay.l0 * (ax.l0 * __ldg(p1 + o00) + ax.l1 * __ldg(p1 + o01)) +
                     ay.l1 * (ax.l0 * __ldg(p1 + o10) + ax.l1 * __ldg(p1 + o11));
    return az.l0 * lo + az.l1 * hi;
  };
  ClassMerge m;
  const float* lg = logits + (int64_t)b * Q * Vi;
  for (int q = 0; q < Q; ++q) m.push(__ldg(class_of_prompt + q), sample(lg + (int64_t)q * Vi));
  const float b0 = sample(bin_occ + ((int64_t)b * 2 + 0) * Vi);
  const float b1 = sample(bin_occ + ((int64_t)b * 2 + 1) * Vi);
  labels[(((int64_t)b * X + x) * Y + y) * Z + z] = (uint8_t)m.label(b0, b1, free_label);
}

// ---- merge + arg-max + gate of ready-made logits (no interpolation) ---------------------------
// _merge_classes_prob (san_in_veon_entry_temporal.py:273-297) + the label rule
// (veon_temporal.py:223-229,240) on sem_occ [B,Q,Z,Y,X] / bin_occ [B,2,Z,Y,X]; the batch strides
// are free so that both may be channel slices of one pooled volume (lift_classify).
template <int ZO>
__global__ void __launch_bounds__(kColThreads)
k_classify_cols(const float* __restrict__ sem_occ, int64_t sem_bstride,
                const float* __restrict__ bin_occ, int64_t bin_bstride,
                const int32_t* __restrict__ class_of_prompt, int Q, int Y, int X, int free_label,
                uint8_t* __restrict__ labels) {
  const int b = blockIdx.y;
  const int idx = blockIdx.x * kColThreads + threadIdx.x;
  const int plane = X * Y;
  if (idx >= plane) return;
  const int x = idx % X, y = idx / X;
  const int64_t V = (int64_t)plane * ZO;
  auto column = [&](const float* __restrict__ src, float* out) {
#pragma unroll
    for (int z = 0; z < ZO; ++z) out[z] = ld_stream(src + (int64_t)z * plane + idx);
  };
  ColumnMerge<ZO> m;
  const float* lg = sem_occ + (int64_t)b * sem_bstride;
  for (int q = 0; q < Q; ++q) {
    float v[ZO];
    column(lg + (int64_t)q * V, v);
    m.push(__ldg(class_of_prompt + q), v);
  }
  m.close_run();
  float b0[ZO], b1[ZO];
  column(bin_occ + (int64_t)b * bin_bstride, b0);
  column(bin_occ + (int64_t)b * bin_bstride + V, b1);
  m.store(b0, b1, free_label, labels + (((int64_t)b * X + x) * Y + y) * ZO);
}

__global__ void __launch_bounds__(kColThreads)
k_classify_any(const float* __restrict__ sem_occ, int64_t sem_bstride,
               const float* __restrict__ bin_occ, int64_t bin_bstride,
               const int32_t* __restrict__ class_of_prompt, int Q, int Z, int Y, int X,
               int free_label, uint8_t* __restrict__ labels) {
  const int b = blockIdx.y;
  const int64_t V = (int64_t)Z * Y * X;
  const int64_t v = (int64_t)blockIdx.x * kColThreads + threadIdx.x;
  if (v >= V) return;
  ClassMerge m;
  const float* lg = sem_occ + (int64_t)b * sem_bstride + v;
  for (int q = 0; q < Q; ++q) m.push(__ldg(class_of_prompt + q), ld_stream(lg + (int64_t)q * V));
  const float b0 = ld_stream(bin_occ + (int64_t)b * bin_bstride + v);
  const float b1 = ld_stream(bin_occ + (int64_t)b * bin_bstride + V + v);
  const int x = (int)(v % X), y = (int)((v / X) % Y), z = (int)(v / ((int64_t)X * Y));
  labels[(((int64_t)b * X + x) * Y + y) * Z + z] = (uint8_t)m.label(b0, b1, free_label);
}

}  // namespace veon

using namespace veon;

extern "C" int veon_classify_logits(const float* sem_occ, int64_t sem_batch_stride,
                                    const float* bin_occ, int64_t bin_batch_stride,
                                    const int32_t* class_of_prompt, int B, int Q, int Z, int Y,
                                    int X, int free_label, uint8_t* labels, void* stream) {
  if (!sem_occ || !bin_occ || !class_of_prompt || !labels || B <= 0 || Q <= 0 || Z <= 0 ||
      Y <= 0 || X <= 0 || B > 65535 || sem_batch_stride < 0 || bin_batch_stride < 0)
    return VEON_E_BADARG;
  if ((int64_t)X * Y > INT32_MAX) return VEON_E_RANGE;
  cudaStream_t st = (cudaStream_t)stream;
  if (Z == 16 && (((uintptr_t)labels) & 15) == 0) {
    dim3 grid((unsigned)ceil_div64((int64_t)X * Y, kColThreads), (unsigned)B);
    k_classify_cols<16><<<grid, kColThreads, 0, st>>>(sem_occ, sem_batch_stride, bin_occ,
                                                      bin_batch_stride, class_of_prompt, Q, Y, X,
                                                      free_label, labels);
  } else {
    dim3 grid((unsigned)ceil_div64((int64_t)Z * Y * X, kColThreads), (unsigned)B);
    k_classify_any<<<grid, kColThreads, 0, st>>>(sem_occ, sem_batch_stride, bin_occ,
                                                 bin_batch_stride, class_of_prompt, Q, Z, Y, X,
                                                 free_label, labels);
  }
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_upsample_classify(const float* sem_occ_lr, const float* bin_occ_lr,
                                      const int32_t* class_of_prompt, int B, int Q, int Zi, int Yi,
                                      int Xi, int Z, int Y, int X, int free_label,
                                      uint8_t* labels, void* stream) {
  if (!sem_occ_lr || !bin_occ_lr || !class_of_prompt || !labels || B <= 0 || Q <= 0 || Zi <= 0 ||
      Yi <= 0 || Xi <= 0 || Z <= 0 || Y <= 0 || X <= 0 || B > 65535)
    return VEON_E_BADARG;
  if ((int64_t)Yi * Xi * Zi > INT32_MAX || (int64_t)X * Y > INT32_MAX) return VEON_E_RANGE;
  const float sz = (float)Zi / (float)Z, sy = (float)Yi / (float)Y, sx = (float)Xi / (float)X;
  cudaStream_t st = (cudaStream_t)stream;
  if (Zi == 8 && Z == 16 && (((uintptr_t)labels) & 15) == 0) {
    dim3 grid((unsigned)ceil_div64((int64_t)X * Y, kColThreads), (unsigned)B);
    k_upsample_classify_cols<8, 16><<<grid, kColThreads, 0, st>>>(
        sem_occ_lr, bin_occ_lr, class_of_prompt, Q, Yi, Xi, Y, X, sy, sx, free_label, labels);
  } else {
    dim3 grid((unsigned)ceil_div64((int64_t)Z * Y * X, kColThreads), (unsigned)B);
    k_upsample_classify_any<<<grid, kColThreads, 0, st>>>(sem_occ_lr, bin_occ_lr, class_of_prompt,
                                                          Q, Zi, Yi, Xi, Z, Y, X, sz, sy, sx,
                                                          free_label, labels);
  }
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t veon_voxel_text_argmax_lowres_workspace_bytes(int B, int Q, int Zi, int Yi,
                                                                int Xi) {
  if (B <= 0 || Q <= 0 || Zi <= 0 || Yi <= 0 || Xi <= 0) return 0;
  return sizeof(float) * (size_t)B * Q * Zi * Yi * Xi;
}

// T = float or uint16_t (bfloat16), CL = channels-last [B,Zi,Yi,Xi,C]: the logits pass of that
// element type and layout, then the same interpolation and classification of the float32 logits
template <bool CL = false, typename T>
static int voxel_text_argmax_lowres(const T* feat_occ_lr, const float* text_w,
                                    const int32_t* class_of_prompt, const float* bin_occ_lr, int B,
                                    int C, int Q, int Zi, int Yi, int Xi, int Z, int Y, int X,
                                    int free_label, uint8_t* labels, void* workspace,
                                    size_t ws_bytes, const void* w_image, void* stream) {
  if (!workspace) return VEON_E_BADARG;
  if (ws_bytes < veon_voxel_text_argmax_lowres_workspace_bytes(B, Q, Zi, Yi, Xi))
    return VEON_E_WORKSPACE;
  float* sem_lr = static_cast<float*>(workspace);
  int rc;
  if constexpr (CL && sizeof(T) == 4)
    rc = veon_semantic_inference_3d_cl(text_w, feat_occ_lr, B, C, Q, Zi, Yi, Xi, sem_lr, w_image,
                                       stream);
  else if constexpr (CL)
    rc = veon_semantic_inference_3d_cl_bf16(text_w, feat_occ_lr, B, C, Q, Zi, Yi, Xi, sem_lr,
                                            w_image, stream);
  else if constexpr (sizeof(T) == 4)
    rc = veon_semantic_inference_3d(text_w, feat_occ_lr, B, C, Q, Zi, Yi, Xi, sem_lr, w_image, stream);
  else
    rc = veon_semantic_inference_3d_bf16(text_w, feat_occ_lr, B, C, Q, Zi, Yi, Xi, sem_lr, w_image,
                                         stream);
  if (rc != 0) return rc;
  return veon_upsample_classify(sem_lr, bin_occ_lr, class_of_prompt, B, Q, Zi, Yi, Xi, Z, Y, X,
                                free_label, labels, stream);
}

extern "C" int veon_voxel_text_argmax_lowres(const float* feat_occ_lr, const float* text_w,
                                             const int32_t* class_of_prompt,
                                             const float* bin_occ_lr, int B, int C, int Q, int Zi,
                                             int Yi, int Xi, int Z, int Y, int X, int free_label,
                                             uint8_t* labels, void* workspace, size_t ws_bytes,
                                             const void* w_image, void* stream) {
  return voxel_text_argmax_lowres(feat_occ_lr, text_w, class_of_prompt, bin_occ_lr, B, C, Q, Zi,
                                  Yi, Xi, Z, Y, X, free_label, labels, workspace, ws_bytes,
                                  w_image, stream);
}

extern "C" int veon_voxel_text_argmax_lowres_bf16(const uint16_t* feat_occ_lr, const float* text_w,
                                                  const int32_t* class_of_prompt,
                                                  const float* bin_occ_lr, int B, int C, int Q,
                                                  int Zi, int Yi, int Xi, int Z, int Y, int X,
                                                  int free_label, uint8_t* labels, void* workspace,
                                                  size_t ws_bytes, const void* w_image,
                                                  void* stream) {
  return voxel_text_argmax_lowres(feat_occ_lr, text_w, class_of_prompt, bin_occ_lr, B, C, Q, Zi,
                                  Yi, Xi, Z, Y, X, free_label, labels, workspace, ws_bytes,
                                  w_image, stream);
}

extern "C" int veon_voxel_text_argmax_lowres_cl(const float* feat_occ_lr, const float* text_w,
                                                const int32_t* class_of_prompt,
                                                const float* bin_occ_lr, int B, int C, int Q,
                                                int Zi, int Yi, int Xi, int Z, int Y, int X,
                                                int free_label, uint8_t* labels, void* workspace,
                                                size_t ws_bytes, const void* w_image,
                                                void* stream) {
  return voxel_text_argmax_lowres<true>(feat_occ_lr, text_w, class_of_prompt, bin_occ_lr, B, C, Q,
                                        Zi, Yi, Xi, Z, Y, X, free_label, labels, workspace,
                                        ws_bytes, w_image, stream);
}

extern "C" int veon_voxel_text_argmax_lowres_cl_bf16(const uint16_t* feat_occ_lr,
                                                     const float* text_w,
                                                     const int32_t* class_of_prompt,
                                                     const float* bin_occ_lr, int B, int C, int Q,
                                                     int Zi, int Yi, int Xi, int Z, int Y, int X,
                                                     int free_label, uint8_t* labels,
                                                     void* workspace, size_t ws_bytes,
                                                     const void* w_image, void* stream) {
  return voxel_text_argmax_lowres<true>(feat_occ_lr, text_w, class_of_prompt, bin_occ_lr, B, C, Q,
                                        Zi, Yi, Xi, Z, Y, X, free_label, labels, workspace,
                                        ws_bytes, w_image, stream);
}
