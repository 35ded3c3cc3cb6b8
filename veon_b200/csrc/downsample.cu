// 2x2x2 max-downsample of the pooled volume and its gradient.
//
// Reference: LSSViewTransformerRaw.forward (view_transformer_raw.py:549-553)
//   rearrange(bev_feat, 'b c (z dz) (h dh) (w dw) -> b c z h w (dz dh dw)', dz=2, dh=2, dw=2)
//   torch.max(bev_feat, dim=-1).values
// i.e. a strided gather + reduction in ATen (2.8 ms for the 1.31 GB volume of C2 on B200) and,
// in training, the backward of max(dim): the WHOLE gradient goes to the one arg-max element,
// the first one in (dz, dh, dw) order on ties.  (Ties are structural here: empty voxels are
// exactly 0.0.)  Both are plain streaming passes: a thread owns two neighbouring outputs = one
// 16-byte load from each of the four input x-rows, so every access is a full coalesced line.
// NaN propagates like torch.max (a NaN input makes the output NaN; the first NaN takes the
// gradient).
#include "common.cuh"

namespace veon {

__device__ __forceinline__ float max_nan(float a, float b) { return (b > a || b != b) ? b : a; }

// volumes: in [BC][Z][Y][X], out [BC][Z/2][Y/2][X/2]; X % 4 == 0, Z and Y even
// MASK: also store, per output, WHICH of its 8 inputs is the arg-max (one bit set, bit index
// (dz*2+dy)*2+dx = the position in the reference's trailing (dz dh dw) axis, first maximum on
// ties): all the backward needs, so the volume need not be kept for it.
__device__ __forceinline__ bool is_max(float v, float m) { return v == m || (m != m && v != v); }
template <bool MASK>
__global__ void __launch_bounds__(256)
k_maxdown2_fwd(const float* __restrict__ in, int64_t n_quads, int Zh, int Yh, int X4, int Y, int X,
               float* __restrict__ out, uint8_t* __restrict__ mask) {
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_quads;
       q += (int64_t)gridDim.x * blockDim.x) {
    const int x4 = (int)(q % X4);
    int64_t r = q / X4;
    const int yo = (int)(r % Yh);
    r /= Yh;
    const int zo = (int)(r % Zh);
    const int64_t bc = r / Zh;
    const float* p = in + ((bc * (2 * Zh) + 2 * zo) * Y + 2 * yo) * (int64_t)X + 4 * x4;
    const float4 a = ld_stream4(p), b = ld_stream4(p + X);
    const float4 c = ld_stream4(p + (int64_t)Y * X), d = ld_stream4(p + (int64_t)Y * X + X);
    float2 o;
    o.x = max_nan(max_nan(max_nan(a.x, a.y), max_nan(b.x, b.y)),
                  max_nan(max_nan(c.x, c.y), max_nan(d.x, d.y)));
    o.y = max_nan(max_nan(max_nan(a.z, a.w), max_nan(b.z, b.w)),
                  max_nan(max_nan(c.z, c.w), max_nan(d.z, d.w)));
    const int64_t oi = ((bc * Zh + zo) * Yh + yo) * (int64_t)(X / 2) + 2 * x4;
    *reinterpret_cast<float2*>(out + oi) = o;
    if (MASK) {
      uint32_t m0 = is_max(a.x, o.x) | is_max(a.y, o.x) << 1 | is_max(b.x, o.x) << 2 |
                    is_max(b.y, o.x) << 3 | is_max(c.x, o.x) << 4 | is_max(c.y, o.x) << 5 |
                    is_max(d.x, o.x) << 6 | is_max(d.y, o.x) << 7;
      uint32_t m1 = is_max(a.z, o.y) | is_max(a.w, o.y) << 1 | is_max(b.z, o.y) << 2 |
                    is_max(b.w, o.y) << 3 | is_max(c.z, o.y) << 4 | is_max(c.w, o.y) << 5 |
                    is_max(d.z, o.y) << 6 | is_max(d.w, o.y) << 7;
      m0 &= 0u - m0;   // the first maximum only
      m1 &= 0u - m1;
      *reinterpret_cast<uchar2*>(mask + oi) = make_uchar2((unsigned char)m0, (unsigned char)m1);
    }
  }
}

__global__ void __launch_bounds__(256)
k_maxdown2_bwd(const float* __restrict__ in, const float* __restrict__ out,
               const float* __restrict__ grad_out, int64_t n_quads, int Zh, int Yh, int X4, int Y,
               int X, float* __restrict__ grad_in) {
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_quads;
       q += (int64_t)gridDim.x * blockDim.x) {
    const int x4 = (int)(q % X4);
    int64_t r = q / X4;
    const int yo = (int)(r % Yh);
    r /= Yh;
    const int zo = (int)(r % Zh);
    const int64_t bc = r / Zh;
    const int64_t ibase = ((bc * (2 * Zh) + 2 * zo) * Y + 2 * yo) * (int64_t)X + 4 * x4;
    const int64_t obase = ((bc * Zh + zo) * Yh + yo) * (int64_t)(X / 2) + 2 * x4;
    const int64_t step[4] = {0, X, (int64_t)Y * X, (int64_t)Y * X + X};
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = ld_stream4(in + ibase + step[k]);
    const float2 m = *reinterpret_cast<const float2*>(out + obase);
    const float2 g = *reinterpret_cast<const float2*>(grad_out + obase);
    // the whole gradient to the FIRST maximum in (dz, dy, dx) order = k-major, then x
    // (the backward of torch.max(dim).values: index_put of the arg-max)
    bool open0 = true, open1 = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float4 w;
      w.x = (open0 && is_max(v[k].x, m.x)) ? g.x : 0.f;
      open0 = open0 && !is_max(v[k].x, m.x);
      w.y = (open0 && is_max(v[k].y, m.x)) ? g.x : 0.f;
      open0 = open0 && !is_max(v[k].y, m.x);
      w.z = (open1 && is_max(v[k].z, m.y)) ? g.y : 0.f;
      open1 = open1 && !is_max(v[k].z, m.y);
      w.w = (open1 && is_max(v[k].w, m.y)) ? g.y : 0.f;
      open1 = open1 && !is_max(v[k].w, m.y);
      st_stream4(grad_in + ibase + step[k], w);
    }
  }
}

// ---- channels-last volumes: in [B][Z][Y][X][C], out [B][Z/2][Y/2][X/2][C] ----------------------
// A thread owns one output element (b, zo, yo, xo, c); consecutive threads are consecutive
// channels, so each of its eight loads is a full coalesced line across the warp.  The same
// reduction tree, NaN rule and first-arg-max order (dz, dy, dx) as the channels-first kernels.
__device__ __forceinline__ void cl_block(int64_t e, int C, int Zh, int Yh, int Xh, int Y, int X,
                                         int64_t& ibase, int64_t step[4]) {
  const int64_t vo = e / C;
  const int c = (int)(e - vo * C);
  uint32_t r = (uint32_t)vo;   // output voxels < 2^32 (checked by the launcher)
  const int xo = (int)(r % (uint32_t)Xh);
  r /= (uint32_t)Xh;
  const int yo = (int)(r % (uint32_t)Yh);
  r /= (uint32_t)Yh;
  const int zo = (int)(r % (uint32_t)Zh);
  const int64_t b = r / (uint32_t)Zh;
  const int64_t row = (int64_t)X * C;   // one y step
  ibase = (((b * (2 * Zh) + 2 * zo) * Y + 2 * yo) * (int64_t)X + 2 * xo) * C + c;
  step[0] = 0;
  step[1] = row;
  step[2] = (int64_t)Y * row;
  step[3] = (int64_t)Y * row + row;
}

__global__ void __launch_bounds__(256)
k_maxdown2_cl_fwd(const float* __restrict__ in, int64_t n_out, int C, int Zh, int Yh, int Xh, int Y,
                  int X, float* __restrict__ out) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_out;
       e += (int64_t)gridDim.x * blockDim.x) {
    int64_t ib, st[4];
    cl_block(e, C, Zh, Yh, Xh, Y, X, ib, st);
    float a[4][2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      a[k][0] = __ldcs(in + ib + st[k]);
      a[k][1] = __ldcs(in + ib + st[k] + C);
    }
    out[e] = max_nan(max_nan(max_nan(a[0][0], a[0][1]), max_nan(a[1][0], a[1][1])),
                     max_nan(max_nan(a[2][0], a[2][1]), max_nan(a[3][0], a[3][1])));
  }
}

__global__ void __launch_bounds__(256)
k_maxdown2_cl_bwd(const float* __restrict__ in, const float* __restrict__ out,
                  const float* __restrict__ grad_out, int64_t n_out, int C, int Zh, int Yh, int Xh,
                  int Y, int X, float* __restrict__ grad_in) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_out;
       e += (int64_t)gridDim.x * blockDim.x) {
    int64_t ib, st[4];
    cl_block(e, C, Zh, Yh, Xh, Y, X, ib, st);
    float v[4][2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[k][0] = __ldcs(in + ib + st[k]);
      v[k][1] = __ldcs(in + ib + st[k] + C);
    }
    const float m = out[e], g = grad_out[e];
    bool open = true;   // the whole gradient to the FIRST maximum in (dz, dy, dx) order
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const bool hit = open && is_max(v[k][dx], m);
        open = open && !is_max(v[k][dx], m);
        st_stream(grad_in + ib + st[k] + dx * C, hit ? g : 0.f);
      }
    }
  }
}

static int check_cl(const void* a, const void* b, int B, int C, int Z, int Y, int X) {
  if (!a || !b || B <= 0 || C <= 0 || Z <= 0 || Y <= 0 || X <= 0) return VEON_E_BADARG;
  if ((Z & 1) || (Y & 1) || (X & 1)) return VEON_E_UNSUPPORTED;
  if ((int64_t)B * (Z / 2) * (Y / 2) * (X / 2) > 0xffffffffLL) return VEON_E_RANGE;
  return 0;
}

static int check(const void* a, const void* b, int64_t BC, int Z, int Y, int X) {
  if (!a || !b || BC <= 0 || Z <= 0 || Y <= 0 || X <= 0) return VEON_E_BADARG;
  if ((Z & 1) || (Y & 1) || (X & 3) || ((uintptr_t)a & 15) || ((uintptr_t)b & 7))
    return VEON_E_UNSUPPORTED;
  return 0;
}

}  // namespace veon

using namespace veon;

extern "C" int veon_maxdown2_fwd(const float* in, int64_t BC, int Z, int Y, int X, float* out,
                                 void* stream_) {
  int rc = check(in, out, BC, Z, Y, X);
  if (rc) return rc;
  const int64_t n_quads = BC * (Z / 2) * (Y / 2) * (X / 4);
  int64_t blocks = ceil_div64(n_quads, 256);
  if (blocks > 148 * 64) blocks = 148 * 64;
  k_maxdown2_fwd<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(
      in, n_quads, Z / 2, Y / 2, X / 4, Y, X, out, nullptr);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_maxdown2_fwd_mask(const float* in, int64_t BC, int Z, int Y, int X, float* out,
                                      uint8_t* mask, void* stream_) {
  int rc = check(in, out, BC, Z, Y, X);
  if (rc) return rc;
  if (!mask) return VEON_E_BADARG;
  if ((uintptr_t)mask & 1) return VEON_E_UNSUPPORTED;
  const int64_t n_quads = BC * (Z / 2) * (Y / 2) * (X / 4);
  int64_t blocks = ceil_div64(n_quads, 256);
  if (blocks > 148 * 64) blocks = 148 * 64;
  k_maxdown2_fwd<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(
      in, n_quads, Z / 2, Y / 2, X / 4, Y, X, out, mask);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_maxdown2_bwd(const float* in, const float* out, const float* grad_out,
                                 int64_t BC, int Z, int Y, int X, float* grad_in, void* stream_) {
  int rc = check(in, out, BC, Z, Y, X);
  if (rc) return rc;
  if (!grad_out || !grad_in) return VEON_E_BADARG;
  if (((uintptr_t)grad_in & 15) || ((uintptr_t)grad_out & 7)) return VEON_E_UNSUPPORTED;
  const int64_t n_quads = BC * (Z / 2) * (Y / 2) * (X / 4);
  int64_t blocks = ceil_div64(n_quads, 256);
  if (blocks > 148 * 64) blocks = 148 * 64;
  k_maxdown2_bwd<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(
      in, out, grad_out, n_quads, Z / 2, Y / 2, X / 4, Y, X, grad_in);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_maxdown2_cl_fwd(const float* in, int B, int C, int Z, int Y, int X, float* out,
                                    void* stream_) {
  int rc = check_cl(in, out, B, C, Z, Y, X);
  if (rc) return rc;
  const int64_t n_out = (int64_t)B * (Z / 2) * (Y / 2) * (X / 2) * C;
  int64_t blocks = ceil_div64(n_out, 256);
  if (blocks > 148 * 64) blocks = 148 * 64;
  k_maxdown2_cl_fwd<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(
      in, n_out, C, Z / 2, Y / 2, X / 2, Y, X, out);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_maxdown2_cl_bwd(const float* in, const float* out, const float* grad_out,
                                    int B, int C, int Z, int Y, int X, float* grad_in,
                                    void* stream_) {
  int rc = check_cl(in, out, B, C, Z, Y, X);
  if (rc) return rc;
  if (!grad_out || !grad_in) return VEON_E_BADARG;
  const int64_t n_out = (int64_t)B * (Z / 2) * (Y / 2) * (X / 2) * C;
  int64_t blocks = ceil_div64(n_out, 256);
  if (blocks > 148 * 64) blocks = 148 * 64;
  k_maxdown2_cl_bwd<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(
      in, out, grad_out, n_out, C, Z / 2, Y / 2, X / 2, Y, X, grad_in);
  VEON_LAUNCH_CHECK();
  return 0;
}
