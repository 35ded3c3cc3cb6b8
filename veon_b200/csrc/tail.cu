// Open-vocabulary tail: voxel-feature x text-embedding logits with fused
// per-class max, argmax, occupancy gate and uint8 label emission.
//
// Reference behaviour (three separate stages, ~25 launches, the [B,Q,Z,Y,X]
// logits and [B,18,Z,Y,X] merged tensor both materialised):
//   semantic_inference_3d  einsum "qc,bczhw->bqzhw"   san_in_veon_temporal.py:257-259
//   _merge_classes_prob    max over each class's prompts   san_in_veon_entry_temporal.py:273-297
//   label rule             softmax/max/gate/where/permute/uint8   veon_temporal.py:223-229,240
//
// This file: the entry point and the fp32 FFMA kernel used for shapes the tensor-core
// path (tail_tc.cu: tcgen05 3xTF32, TMEM accumulators) does not take (C % 32 != 0,
// V % 4 != 0, more than 128 prompt rows) -- one thread per voxel, text rows staged in
// shared memory per prompt tile, everything after the dot products fused in registers.
// Features are float32 or bfloat16 (T); a bfloat16 value is widened exactly on load, so the
// bfloat16 instances give the float32 ones' bits on x.float().  Channels-last volumes
// ([B,Z,Y,X,C], the _cl entries) take the tensor-core path alone.
#include <math.h>

#include "common.cuh"

namespace veon {

constexpr int kTailThreads = 128;
constexpr int kTailQT = 24;  // prompts held in registers per pass

// LOGITS: store sem_occ [B,Q,V] (semantic_inference_3d alone) instead of the labels.
template <bool LOGITS, typename T>
__global__ void __launch_bounds__(kTailThreads)
k_voxel_text_argmax(const T* __restrict__ feat_occ, const float* __restrict__ text_w,
                    const int32_t* __restrict__ class_of_prompt,
                    const float* __restrict__ bin_occ, int C, int Q, int Z, int Y, int X,
                    int free_label, uint8_t* __restrict__ labels, float* __restrict__ logits) {
  extern __shared__ float w_s[];  // [kTailQT][C] of the current prompt tile
  const int64_t V = (int64_t)Z * Y * X;
  const int b = blockIdx.y;
  const int64_t v = (int64_t)blockIdx.x * kTailThreads + threadIdx.x;
  const bool live = v < V;
  const T* f = feat_occ + (int64_t)b * C * V + (live ? v : 0);

  float best = 0.f, cur = 0.f;
  int best_cls = -1, cur_cls = -1;
  bool bad = false;  // NaN / +inf anywhere => softmax score is NaN => free

  for (int q0 = 0; q0 < Q; q0 += kTailQT) {
    const int nq = min(kTailQT, Q - q0);
    __syncthreads();
    for (int i = threadIdx.x; i < nq * C; i += kTailThreads) w_s[i] = text_w[(int64_t)q0 * C + i];
    __syncthreads();
    float acc[kTailQT];
#pragma unroll
    for (int q = 0; q < kTailQT; ++q) acc[q] = 0.f;
    int c = 0;
    for (; c + 4 <= C; c += 4) {
      const float f0 = ldg_widen(f + (int64_t)(c + 0) * V), f1 = ldg_widen(f + (int64_t)(c + 1) * V);
      const float f2 = ldg_widen(f + (int64_t)(c + 2) * V), f3 = ldg_widen(f + (int64_t)(c + 3) * V);
#pragma unroll
      for (int q = 0; q < kTailQT; ++q) {
        if (q < nq) {
          const float* w = w_s + q * C + c;
          acc[q] = fmaf(w[0], f0, acc[q]);
          acc[q] = fmaf(w[1], f1, acc[q]);
          acc[q] = fmaf(w[2], f2, acc[q]);
          acc[q] = fmaf(w[3], f3, acc[q]);
        }
      }
    }
    for (; c < C; ++c) {
      const float f0 = ldg_widen(f + (int64_t)c * V);
#pragma unroll
      for (int q = 0; q < kTailQT; ++q)
        if (q < nq) acc[q] = fmaf(w_s[q * C + c], f0, acc[q]);
    }
    if constexpr (LOGITS) {
#pragma unroll
      for (int q = 0; q < kTailQT; ++q)
        if (q < nq && live) logits[((int64_t)b * Q + q0 + q) * V + v] = acc[q];
      continue;
    }
    // group-max over prompts of one class, then first-index argmax over classes
#pragma unroll
    for (int q = 0; q < kTailQT; ++q) {
      if (q < nq) {
        const int cls = class_of_prompt[q0 + q];
        const float x = acc[q];
        bad |= !(x < INFINITY);  // NaN or +inf
        if (cls != cur_cls) {
          if (cur_cls >= 0 && (best_cls < 0 || cur > best)) { best = cur; best_cls = cur_cls; }
          cur_cls = cls;
          cur = x;
        } else {
          cur = fmaxf(cur, x);
        }
      }
    }
  }
  if constexpr (LOGITS) return;
  if (cur_cls >= 0 && (best_cls < 0 || cur > best)) { best = cur; best_cls = cur_cls; }
  if (!live) return;
  bad |= (best == -INFINITY);  // all logits -inf => softmax NaN
  const float b0 = bin_occ[((int64_t)b * 2 + 0) * V + v];
  const float b1 = bin_occ[((int64_t)b * 2 + 1) * V + v];
  // softmax(bin_occ)[0] > 0.5, evaluated like torch.softmax
  const float m = fmaxf(b0, b1);
  const float e0 = expf(b0 - m), e1 = expf(b1 - m);
  const bool occupied = (e0 / (e0 + e1)) > 0.5f;
  const int label = (occupied && !bad) ? best_cls : free_label;
  // [B,Z,Y,X] -> permute(0,3,2,1) -> [B,X,Y,Z]
  const int x = (int)(v % X);
  const int y = (int)((v / X) % Y);
  const int z = (int)(v / ((int64_t)X * Y));
  labels[(((int64_t)b * X + x) * Y + y) * Z + z] = (uint8_t)label;
}

}  // namespace veon

using namespace veon;

// tensor-core path (tail_tc.cu); VEON_E_UNSUPPORTED when the shape does not fit it.
// CL: feat_occ is channels-last [B,Z,Y,X,C].
bool veon_tail_tc_takes(int C, int Q, int64_t V, const float* text_w);
template <typename T, bool CL>
int veon_tail_tc_launch(const T* feat_occ, const float* text_w, const int32_t* cls,
                        const float* bin_occ, int B, int C, int Q, int Z, int Y, int X,
                        int free_label, uint8_t* labels, float* logits, const void* w_image,
                        cudaStream_t stream);

// labels (logits == nullptr) or raw logits (labels == nullptr) of B volumes.  bfloat16 features
// take the route the float32 call would take on x.float(): the FFMA kernel where it takes that,
// else tcgen05 -- and VEON_E_UNSUPPORTED where its bfloat16 loader cannot (V % 8 == 4 or an
// 8- but not 16-byte aligned feat_occ), so that the caller widens instead of getting other bits.
template <typename T>
static int tail_dispatch(const T* feat_occ, const float* text_w,
                         const int32_t* class_of_prompt, const float* bin_occ, int B, int C,
                         int Q, int Z, int Y, int X, int free_label, uint8_t* labels,
                         float* logits, const void* w_image, cudaStream_t stream) {
  {  // tcgen05 path unless the shape does not fit it (C % 32, V % 4, Q > 128)
    const int rc = veon_tail_tc_launch<T, false>(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y,
                                          X, free_label, labels, logits, w_image, stream);
    if (rc != VEON_E_UNSUPPORTED) return rc;
    if (sizeof(T) == 2 && veon_tail_tc_takes(C, Q, (int64_t)Z * Y * X, text_w)) return rc;
  }
  const size_t smem = sizeof(float) * (size_t)kTailQT * C;
  if (smem > 200 * 1024) return VEON_E_UNSUPPORTED;
  static size_t attr_smem_dev[kMaxDevices] = {};
  size_t& attr_smem = attr_smem_dev[current_device()];
  if (attr_smem == 0) attr_smem = 48 * 1024;
  if (smem > attr_smem) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_voxel_text_argmax<false, T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_voxel_text_argmax<true, T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem = smem;
  }
  const int64_t V = (int64_t)Z * Y * X;
  dim3 grid((unsigned)ceil_div64(V, kTailThreads), (unsigned)B);
  if (logits)
    k_voxel_text_argmax<true, T><<<grid, kTailThreads, smem, stream>>>(
        feat_occ, text_w, class_of_prompt, bin_occ, C, Q, Z, Y, X, free_label, labels, logits);
  else
    k_voxel_text_argmax<false, T><<<grid, kTailThreads, smem, stream>>>(
        feat_occ, text_w, class_of_prompt, bin_occ, C, Q, Z, Y, X, free_label, labels, logits);
  VEON_LAUNCH_CHECK();
  return 0;
}

// A channels-last volume (CL) takes tcgen05 exactly where the channels-first call on its
// contiguous copy does, so both give the same bits; everywhere else (C % 32 != 0, V % 4 != 0,
// Q > 128, a feat_occ that is not 16-byte aligned) VEON_E_UNSUPPORTED, and the caller makes the
// volume contiguous.  There is no channels-last FFMA kernel.
template <bool CL, typename T>
static int tail_route(const T* feat_occ, const float* text_w, const int32_t* class_of_prompt,
                      const float* bin_occ, int B, int C, int Q, int Z, int Y, int X,
                      int free_label, uint8_t* labels, float* logits, const void* w_image,
                      cudaStream_t stream) {
  if constexpr (CL)
    return veon_tail_tc_launch<T, true>(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y,
                                        X, free_label, labels, logits, w_image, stream);
  else
    return tail_dispatch(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y, X, free_label,
                         labels, logits, w_image, stream);
}

template <bool CL = false, typename T>
static int voxel_text_argmax(const T* feat_occ, const float* text_w,
                             const int32_t* class_of_prompt, const float* bin_occ, int B, int C,
                             int Q, int Z, int Y, int X, int free_label, uint8_t* labels,
                             const void* w_image, void* stream) {
  if (!feat_occ || !text_w || !class_of_prompt || !bin_occ || !labels || B <= 0 || C <= 0 ||
      Q <= 0 || Z <= 0 || Y <= 0 || X <= 0 || B > 65535)
    return VEON_E_BADARG;
  return tail_route<CL>(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y, X, free_label,
                        labels, nullptr, w_image, (cudaStream_t)stream);
}

template <bool CL = false, typename T>
static int semantic_inference_3d(const float* text_w, const T* feat_occ, int B, int C, int Q,
                                 int Z, int Y, int X, float* sem_occ, const void* w_image,
                                 void* stream) {
  if (!feat_occ || !text_w || !sem_occ || B <= 0 || C <= 0 || Q <= 0 || Z <= 0 || Y <= 0 ||
      X <= 0 || B > 65535)
    return VEON_E_BADARG;
  return tail_route<CL>(feat_occ, text_w, nullptr, nullptr, B, C, Q, Z, Y, X, 0, nullptr, sem_occ,
                        w_image, (cudaStream_t)stream);
}

extern "C" int veon_voxel_text_argmax(const float* feat_occ, const float* text_w,
                                      const int32_t* class_of_prompt, const float* bin_occ,
                                      int B, int C, int Q, int Z, int Y, int X, int free_label,
                                      uint8_t* labels, const void* w_image, void* stream) {
  return voxel_text_argmax(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y, X,
                           free_label, labels, w_image, stream);
}

extern "C" int veon_voxel_text_argmax_bf16(const uint16_t* feat_occ, const float* text_w,
                                           const int32_t* class_of_prompt, const float* bin_occ,
                                           int B, int C, int Q, int Z, int Y, int X,
                                           int free_label, uint8_t* labels, const void* w_image,
                                           void* stream) {
  return voxel_text_argmax(reinterpret_cast<const bf16*>(feat_occ), text_w, class_of_prompt,
                           bin_occ, B, C, Q, Z, Y, X, free_label, labels, w_image, stream);
}

extern "C" int veon_semantic_inference_3d(const float* text_w, const float* feat_occ, int B, int C,
                                          int Q, int Z, int Y, int X, float* sem_occ,
                                          const void* w_image, void* stream) {
  return semantic_inference_3d(text_w, feat_occ, B, C, Q, Z, Y, X, sem_occ, w_image, stream);
}

extern "C" int veon_semantic_inference_3d_bf16(const float* text_w, const uint16_t* feat_occ,
                                               int B, int C, int Q, int Z, int Y, int X,
                                               float* sem_occ, const void* w_image, void* stream) {
  return semantic_inference_3d(text_w, reinterpret_cast<const bf16*>(feat_occ), B, C, Q, Z, Y, X,
                               sem_occ, w_image, stream);
}

// channels-last feat_occ [B,Z,Y,X,C]
extern "C" int veon_voxel_text_argmax_cl(const float* feat_occ, const float* text_w,
                                         const int32_t* class_of_prompt, const float* bin_occ,
                                         int B, int C, int Q, int Z, int Y, int X, int free_label,
                                         uint8_t* labels, const void* w_image, void* stream) {
  return voxel_text_argmax<true>(feat_occ, text_w, class_of_prompt, bin_occ, B, C, Q, Z, Y, X,
                                 free_label, labels, w_image, stream);
}

extern "C" int veon_voxel_text_argmax_cl_bf16(const uint16_t* feat_occ, const float* text_w,
                                              const int32_t* class_of_prompt, const float* bin_occ,
                                              int B, int C, int Q, int Z, int Y, int X,
                                              int free_label, uint8_t* labels,
                                              const void* w_image, void* stream) {
  return voxel_text_argmax<true>(reinterpret_cast<const bf16*>(feat_occ), text_w, class_of_prompt,
                                 bin_occ, B, C, Q, Z, Y, X, free_label, labels, w_image, stream);
}

extern "C" int veon_semantic_inference_3d_cl(const float* text_w, const float* feat_occ, int B,
                                             int C, int Q, int Z, int Y, int X, float* sem_occ,
                                             const void* w_image, void* stream) {
  return semantic_inference_3d<true>(text_w, feat_occ, B, C, Q, Z, Y, X, sem_occ, w_image, stream);
}

extern "C" int veon_semantic_inference_3d_cl_bf16(const float* text_w, const uint16_t* feat_occ,
                                                  int B, int C, int Q, int Z, int Y, int X,
                                                  float* sem_occ, const void* w_image,
                                                  void* stream) {
  return semantic_inference_3d<true>(text_w, reinterpret_cast<const bf16*>(feat_occ), B, C, Q, Z,
                                     Y, X, sem_occ, w_image, stream);
}

// ---- training-time voxel x text arg-max over a POINT LIST (SURVEY 8f-4) ----------------------
// Proj2Dto3DLoss, loss/occ_loss_utils/occ3d_nuscenes.py:472-482: for the N selected voxels
//   pred_probs    = einsum('nc,dc->nd', feat[N,C], W[:-1])          (no background row)
//   pred_indices  = max(pred_probs, dim=1).indices                  best PROMPT
//   pred_class    = max over the prompts of each class (_merge_classes_prob, :249-265), then
//   pred_class_idx = max(., dim=1).indices                          best merged CLASS
// Here: logits [Q, ldn] (row q = prompt q over the points, as veon_semantic_inference_3d writes
// them for a [C, N] operand), one thread per point walks the Q rows once: coalesced reads, both
// arg-maxes with first-index ties (torch.max(dim) returns the first maximum).
__global__ void __launch_bounds__(256)
k_point_argmax(const float* __restrict__ logits, const int32_t* __restrict__ class_of_prompt, int Q,
               int64_t N, int64_t ldn, int64_t* __restrict__ prompt_idx,
               int64_t* __restrict__ class_idx) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float best_p = 0.f, best_c = 0.f, run = 0.f;
  int arg_p = -1, arg_c = -1, run_cls = -1;
  for (int q = 0; q < Q; ++q) {
    const float x = __ldg(logits + (int64_t)q * ldn + n);
    const int cq = __ldg(class_of_prompt + q);
    if (arg_p < 0 || x > best_p) { best_p = x; arg_p = q; }
    if (cq != run_cls) {           // a new class starts: close the previous one
      if (run_cls >= 0 && (arg_c < 0 || run > best_c)) { best_c = run; arg_c = run_cls; }
      run_cls = cq;
      run = x;
    } else if (x > run) {
      run = x;
    }
  }
  if (run_cls >= 0 && (arg_c < 0 || run > best_c)) arg_c = run_cls;
  prompt_idx[n] = arg_p;
  class_idx[n] = arg_c;
}

extern "C" int veon_point_text_argmax(const float* logits, const int32_t* class_of_prompt, int Q,
                                      int64_t N, int64_t ldn, int64_t* prompt_idx,
                                      int64_t* class_idx, void* stream) {
  if (!logits || !class_of_prompt || !prompt_idx || !class_idx || Q <= 0 || N < 0 || ldn < N)
    return VEON_E_BADARG;
  if (N == 0) return 0;
  k_point_argmax<<<(unsigned)ceil_div64(N, 256), 256, 0, (cudaStream_t)stream>>>(
      logits, class_of_prompt, Q, N, ldn, prompt_idx, class_idx);
  VEON_LAUNCH_CHECK();
  return 0;
}
