// bev_pool_v2 backward for a channels-first [B,C,Z,Y,X] out_grad.
//
// Reference behaviour: QuickCumsumCuda.backward (bev_pool.py:43-83): argsort by
// ranks_feat + interval rebuild on every call, `out_grad.contiguous()` (a full
// transpose back to channels-last, :69), then bev_pool_grad_kernel
// (bev_pool_cuda.cu:67-121) with ONE THREAD per feature pixel walking all its
// points and all channels twice, stride-C uncoalesced.
//
// Here, two atomic-free passes:
//   k_bwd_rows    one warp per occupied 32-voxel tile (occupancy mask and first
//                 interval come from the plan: one load latency), reads the
//                 tile's out_grad lines (only the 32-byte sectors that hold an
//                 occupied voxel, all loads in flight together), transposes
//                 through shared memory and emits
//                 one compact channel-contiguous row per interval
//                 (rows[interval, C]).  Empty tiles are never read.
//   k_bwd_pixels  one warp per feature pixel (the reference's by-ranks_feat
//                 interval): its kept points come from the pixel-major
//                 point->interval table the prepare step emitted (no sort),
//                 the pixel's feature row lives in registers, each point costs
//                 one row read:  depth_grad[p] = <row, feat>,
//                 feat_grad += depth[p] * row.  Both outputs are written
//                 densely (zeros for dropped points), so no memset either.
// Every output element has exactly one writer and a fixed summation order
// (ascending depth bin) => bitwise run-to-run deterministic.
// A channels-last out_grad [B,Z,Y,X,C] already holds every occupied voxel's gradient as one
// contiguous row: k_bwd_pixels<KCH, true> reads those rows in place (no row pass, no scratch).
// A bfloat16 out_grad (template parameter T = bf16) is widened exactly where it is read: into the
// float compact rows (row pass) or into registers (single pass); all arithmetic stays float.
#include "common.cuh"

namespace veon {

constexpr int kBwdWarps = 8;   // pixel pass: 8 consecutive pixels per CTA
#ifndef VEON_ROW_WARPS
#define VEON_ROW_WARPS 4
#endif
constexpr int kRowWarps = VEON_ROW_WARPS;   // row pass
constexpr int kPitch = kTileVoxels + 1;

// one warp: tile t, channel chunk starting at cbase -> compact rows
template <int KCH, typename T>
__device__ __forceinline__ void rows_tile(float* tile, int lane, const T* __restrict__ out_grad,
                                          const int32_t* __restrict__ tile_istart,
                                          const uint32_t* __restrict__ tile_occ, int64_t t,
                                          int cbase, int64_t tiles_per_sample, int64_t V, int C,
                                          int vec_ok, float* __restrict__ rows) {
  constexpr int CC = 32 * KCH;
  const uint32_t occ = __ldg(tile_occ + t);  // one independent load each: a single latency
  const int32_t i0 = __ldg(tile_istart + t);
  if (occ == 0u) return;                     // empty tile: nothing read (warp-uniform)
  const int64_t b = t / tiles_per_sample;
  const int64_t v0 = (t - b * tiles_per_sample) * kTileVoxels;

  // fetch only 32-byte sectors (8 voxels) that contain an occupied voxel.
  // lane (r = lane/8, q = lane%8) loads voxels 4q..4q+3 of channel 4*it + r with
  // one 16-byte load; the 4 scalar smem stores hit banks (c + 4q + i) mod 32.
  const int cmax = min(CC, C - cbase);
  const int q4 = (lane & 7) * 4, r = lane >> 3;
  const bool want = ((occ >> (q4 & 24)) & 0xffu) != 0u;
  if (vec_ok && v0 + kTileVoxels <= V) {
    const T* g = out_grad + ((int64_t)b * C + cbase + r) * V + v0 + q4;
    float* trow = tile + r * kPitch + q4;
    if (cmax == CC) {  // all CC/4 loads of the lane in flight at once
      float4 v[CC / 4];
#pragma unroll
      for (int it = 0; it < CC / 4; ++it)
        v[it] = want ? ld_stream4(g + (int64_t)it * 4 * V) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int it = 0; it < CC / 4; ++it) {
        float* tr = trow + it * 4 * kPitch;
        tr[0] = v[it].x; tr[1] = v[it].y; tr[2] = v[it].z; tr[3] = v[it].w;
      }
    } else {
      for (int c = r; c < cmax; c += 4, g += 4 * V, trow += 4 * kPitch) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (want) v = ld_stream4(g);
        trow[0] = v.x; trow[1] = v.y; trow[2] = v.z; trow[3] = v.w;
      }
    }
  } else {
    const bool wants = ((occ >> (lane & 24)) & 0xffu) != 0u && (v0 + lane < V);
    const T* g = out_grad + ((int64_t)b * C + cbase) * V + v0 + lane;
    for (int cl = 0; cl < cmax; ++cl)
      tile[cl * kPitch + lane] = wants ? ld_stream(g + (int64_t)cl * V) : 0.f;
  }
  __syncwarp();
  // j-th occupied voxel of the tile -> interval i0 + j
  uint32_t rest = occ;
  float* row = rows + (int64_t)i0 * C + cbase + lane;
  while (rest) {
    const int vj = __ffs(rest) - 1;
    rest &= rest - 1;
#pragma unroll
    for (int k = 0; k < KCH; ++k)
      if (lane + 32 * k < cmax) row[32 * k] = tile[(lane + 32 * k) * kPitch + vj];
    row += C;
  }
}

template <int KCH, typename T = float>
__global__ void __launch_bounds__(kRowWarps * 32)
k_bwd_rows(const T* __restrict__ out_grad, const int32_t* __restrict__ tile_istart,
           const uint32_t* __restrict__ tile_occ, int64_t tile_begin, int64_t tile_end,
           int64_t tiles_per_sample, int64_t V, int C, int n_chunks, int vec_ok,
           float* __restrict__ rows) {
  constexpr int CC = 32 * KCH;
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t group = blockIdx.x / n_chunks;
  const int cbase = (int)(blockIdx.x - group * n_chunks) * CC;
  const int64_t t = tile_begin + group * kRowWarps + warp;
  if (t >= tile_end) return;
  rows_tile<KCH>(smem + warp * (CC * kPitch), lane, out_grad, tile_istart, tile_occ, t, cbase,
                 tiles_per_sample, V, C, vec_ok, rows);
}


// Persistent variant of the row pass (aligned volumes): every warp strides over the
// (tile, channel chunk) items, keeps the NEXT occupied tile's 8 KB of out_grad in flight
// (16-byte cp.async into the second half of a double-buffered shared tile, no registers
// held) while it extracts the rows of the current one, and reads the plan's occupancy /
// first-interval words 32 items at a time, one table ahead -- so neither the plan lookup
// nor the transposition/row write sits between two tiles' loads.
constexpr int kRowPitchP = kTileVoxels + 4;  // 16-byte aligned rows for cp.async

// T = bf16: the shared tiles hold the gradient's own bf16 values, widened as the rows are extracted.
template <int KCH, typename T = float>
__global__ void __launch_bounds__(kRowWarps * 32)
k_bwd_rows_persistent(const T* __restrict__ out_grad, const int32_t* __restrict__ tile_istart,
                      const uint32_t* __restrict__ tile_occ, int64_t n_items,
                      int64_t tiles_per_sample, int64_t V, int C, int n_chunks,
                      float* __restrict__ rows) {
  constexpr int CC = 32 * KCH;
  constexpr int kBuf = CC * kRowPitchP;
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T* buf = reinterpret_cast<T*>(smem) + warp * 2 * kBuf;
  const int64_t TW = (int64_t)gridDim.x * kRowWarps;
  const int64_t first = (int64_t)blockIdx.x * kRowWarps + warp;
  if (first >= n_items) return;
  const int64_t mine = (n_items - first + TW - 1) / TW;
  const int q4 = (lane & 7) * 4, r = lane >> 3;

  auto load_table = [&](int64_t k0, uint32_t& occ, int32_t& i0) {
    const int64_t k = k0 + lane;
    occ = 0u;
    i0 = 0;
    if (k < mine) {
      const int64_t t = (first + k * TW) / n_chunks;
      occ = __ldg(tile_occ + t);
      i0 = __ldg(tile_istart + t);
    }
  };
  // rows of the tile sitting in `tile`: j-th occupied voxel -> interval i0 + j
  auto extract = [&](const T* tile, uint32_t occ, int32_t i0, int cbase) {
    const int cmax = min(CC, C - cbase);
    float* row = rows + (int64_t)i0 * C + cbase + lane;
    uint32_t rest = occ;
    while (rest) {
      const int vj = __ffs(rest) - 1;
      rest &= rest - 1;
#pragma unroll
      for (int k = 0; k < KCH; ++k)
        if (lane + 32 * k < cmax) row[32 * k] = widen(tile[(lane + 32 * k) * kRowPitchP + vj]);
      row += C;
    }
  };

  uint32_t occ_tab, occ_nxt = 0u, p_occ = 0u;
  int32_t i0_tab, i0_nxt = 0, p_i0 = 0;
  int p_cbase = 0, cur = 0;
  load_table(0, occ_tab, i0_tab);
  for (int64_t k0 = 0; k0 < mine; k0 += 32) {
    if (k0 + 32 < mine) load_table(k0 + 32, occ_nxt, i0_nxt);
    const int nj = (int)min((int64_t)32, mine - k0);
    for (int j = 0; j < nj; ++j) {
      const uint32_t occ = __shfl_sync(0xffffffffu, occ_tab, j);
      if (occ == 0u) continue;  // empty tile: nothing read (warp-uniform)
      const int32_t i0 = __shfl_sync(0xffffffffu, i0_tab, j);
      const int64_t item = first + (k0 + j) * TW;
      const int64_t t = item / n_chunks;
      const int cbase = (int)(item - t * n_chunks) * CC;
      const int64_t b = t / tiles_per_sample;
      const int64_t v0 = (t - b * tiles_per_sample) * kTileVoxels;
      const int cmax = min(CC, C - cbase);
      // only the 32-byte sectors (8 voxels) that contain an occupied voxel
      if (((occ >> (q4 & 24)) & 0xffu) != 0u) {
        const T* g = out_grad + ((int64_t)b * C + cbase + r) * V + v0 + q4;
        T* dst = buf + cur * kBuf + r * kRowPitchP + q4;
#pragma unroll
        for (int it = 0; it < CC / 4; ++it)
          if (4 * it + r < cmax) cp_async_4(dst + it * 4 * kRowPitchP, g + (int64_t)it * 4 * V);
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      if (p_occ) {
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncwarp();
        extract(buf + (cur ^ 1) * kBuf, p_occ, p_i0, p_cbase);
        __syncwarp();  // the other half is refilled next
      }
      p_occ = occ;
      p_i0 = i0;
      p_cbase = cbase;
      cur ^= 1;
    }
    occ_tab = occ_nxt;
    i0_tab = i0_nxt;
  }
  if (p_occ) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    extract(buf + (cur ^ 1) * kBuf, p_occ, p_i0, p_cbase);
  }
}


// ---- row pass for a gradient that arrives behind the 2x2x2 max-downsample ---------------
// (LSSViewTransformerRaw: pool -> rearrange + torch.max(dim), view_transformer_raw.py:549-553.)
// The gradient of max(dim) goes to the arg-max alone; the forward kept that as an 8-bit mask
// with ONE bit set per output (k_maxdown2_fwd<true>: the first maximum of the block), so the
// gradient row of an occupied voxel is
//   rows[i, c] = bit(mask[c, block], pos) ? grad_ds[c, block] : 0       (popc(mask) == 1)
// and neither the full-resolution gradient nor the volume itself is ever read: 0.2 GB instead
// of 2.9 + 1.2 GB for the down-sample backward followed by the plain row pass.
// One warp per occupied tile, lanes = channels, four voxels' loads in flight.
// A bfloat16 grad_ds (TG = bf16) is widened exactly where it is loaded; the rows stay float.
// ptxas gives either instance 64 registers; asked for 4 CTAs per SM (the same 64), it allocates
// the bf16 one without the 20-byte spill the float one has.  (0 = no minimum: the float kernel
// compiles as it did.)
template <typename TG>
__global__ void __launch_bounds__(256, sizeof(TG) == 2 ? 4 : 0)
k_bwd_rows_ds(const TG* __restrict__ grad_ds, const uint8_t* __restrict__ mask,
              const int32_t* __restrict__ tile_istart, const uint32_t* __restrict__ tile_occ,
              int64_t n_tiles, int64_t tiles_per_sample, int Z, int Y, int X, int C,
              float* __restrict__ rows) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int Zh = Z / 2, Yh = Y / 2, Xh = X / 2;
  const int64_t plane = (int64_t)Zh * Yh * Xh;
  for (int64_t t = warp0; t < n_tiles; t += n_warps) {
    const uint32_t occ = __ldg(tile_occ + t);
    if (occ == 0u) continue;
    const int32_t i0 = __ldg(tile_istart + t);
    const int64_t b = t / tiles_per_sample;
    const int32_t v0 = (int32_t)(t - b * tiles_per_sample) * kTileVoxels;
    uint32_t rest = occ;
    int j = 0;                                   // j-th occupied voxel -> interval i0 + j
    while (rest) {
      int64_t blk[4];
      int pos[4], nv = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        blk[q] = 0;
        pos[q] = 0;
        if (rest) {
          const int v = v0 + __ffs(rest) - 1;
          rest &= rest - 1;
          const int x = v % X, y = (v / X) % Y, z = v / (X * Y);
          blk[q] = ((int64_t)(z >> 1) * Yh + (y >> 1)) * Xh + (x >> 1);
          pos[q] = ((z & 1) * 2 + (y & 1)) * 2 + (x & 1);
          nv = q + 1;
        }
      }
      for (int c = lane; c < C; c += 32) {
        const int64_t base = ((int64_t)b * C + c) * plane;
        float g[4];
        uint32_t m[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          g[q] = 0.f;
          m[q] = 0u;
          if (q < nv) {
            g[q] = ldg_widen(grad_ds + base + blk[q]);
            m[q] = __ldg(mask + base + blk[q]);
          }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < nv)
            rows[(int64_t)(i0 + j + q) * C + c] =
                ((m[q] >> pos[q]) & 1u) ? g[q] / (float)__popc(m[q]) : 0.f;
      }
      j += nv;
    }
  }
}

// Same result with full-sector accesses and no shared memory (X % 8 == 0): tile starts and row
// lengths are then multiples of 8, so every aligned group of 8 voxels of a tile lies in one
// x-row = 4 consecutive blocks of one (z/2, y/2) row of the down-sampled volume.  Lane
// (cs = lane / 4, q = lane % 4) owns voxels 8q..8q+7 of the tile for channels cs, cs + 8, ...:
// one 16-byte (bf16: 8-byte) load of grad_ds and one 4-byte load of the mask per channel, then up
// to 8 predicated 4-byte row stores; the 8 lanes of a q write 32 consecutive bytes of a row.
template <typename TG>
__global__ void __launch_bounds__(256)
k_bwd_rows_ds_direct(const TG* __restrict__ grad_ds, const uint8_t* __restrict__ mask,
                     const int32_t* __restrict__ tile_istart,
                     const uint32_t* __restrict__ tile_occ, int64_t n_tiles,
                     int64_t tiles_per_sample, int Z, int Y, int X, int C,
                     float* __restrict__ rows) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int Zh = Z / 2, Yh = Y / 2, Xh = X / 2;
  const int64_t plane = (int64_t)Zh * Yh * Xh;
  const int cs = lane >> 2, q = lane & 3;
  for (int64_t t = warp0; t < n_tiles; t += n_warps) {
    const uint32_t occ = __ldg(tile_occ + t);
    const uint32_t bits = (occ >> (8 * q)) & 0xffu;       // this lane's 8 voxels
    if (occ == 0u) continue;
    const int32_t i0 = __ldg(tile_istart + t);
    if (bits == 0u) continue;
    const int64_t b = t / tiles_per_sample;
    const int32_t v = (int32_t)(t - b * tiles_per_sample) * kTileVoxels + 8 * q;  // first voxel
    const int row = v / X, x = v - row * X;               // (x is a multiple of 8)
    const int z = row / Y, y = row - z * Y;
    const int64_t blk0 = ((int64_t)(z >> 1) * Yh + (y >> 1)) * Xh + (x >> 1);
    const int pos0 = ((z & 1) * 2 + (y & 1)) * 2;
    const int ibase = i0 + __popc(occ & ((1u << (8 * q)) - 1u));   // interval of the first set bit
    for (int c = cs; c < C; c += 8) {
      const int64_t src = ((int64_t)b * C + c) * plane + blk0;
      const float4 g4 = ldg_widen4(grad_ds + src);
      const uchar4 m4 = __ldg(reinterpret_cast<const uchar4*>(mask + src));
      const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
      const uint32_t mv[4] = {m4.x, m4.y, m4.z, m4.w};
      float* r = rows + (int64_t)ibase * C + c;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float share = gv[i] / (float)__popc(mv[i]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          if ((bits >> (2 * i + e)) & 1u) {
            *r = ((mv[i] >> (pos0 + e)) & 1u) ? share : 0.f;
            r += C;
          }
        }
      }
    }
  }
}

// Sum U per-lane partials over the warp, for U values at once: after log2(U) exchange
// steps every lane holds ONE value (the one selected by its upper lane bits), which is
// then reduced over the remaining lane bits.  U + log2(32/U) - 1 shuffles instead of 5*U.
// Returns the sum for value index `which` (valid in every lane).
template <int U>
__device__ __forceinline__ float reduce_many(float (&d)[U], int lane, int& which) {
  static_assert(U == 4 || U == 8, "U must be 4 or 8");
  int idx = 0;
  if constexpr (U == 8) {
    const bool hi = lane & 16;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float keep = hi ? d[4 + i] : d[i], send = hi ? d[i] : d[4 + i];
      d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
    idx = hi ? 4 : 0;
    const bool h8 = lane & 8;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float keep = h8 ? d[2 + i] : d[i], send = h8 ? d[i] : d[2 + i];
      d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    idx += h8 ? 2 : 0;
    const bool h4 = lane & 4;
    const float keep = h4 ? d[1] : d[0], send = h4 ? d[0] : d[1];
    float v = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    idx += h4 ? 1 : 0;
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    which = idx;
    return v;
  } else {
    const bool hi = lane & 16;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float keep = hi ? d[2 + i] : d[i], send = hi ? d[i] : d[2 + i];
      d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
    idx = hi ? 2 : 0;
    const bool h8 = lane & 8;
    const float keep = h8 ? d[1] : d[0], send = h8 ? d[0] : d[1];
    float v = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    idx += h8 ? 1 : 0;
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    which = idx;
    return v;
  }
}

// One warp per feature pixel; a CTA's 8 warps are 8 consecutive pixels so that
// their strided depth / depth_grad accesses share 32-byte sectors.
// one warp: feature pixel `pix`; wsm = 4*D floats of per-warp shared memory.
// COHERENT: true when `rows` was written earlier in the SAME kernel (fused path): the
// read-only (.nc) path may then not be used.
// CL: `rows` is a channels-last out_grad [B*V, C] itself; a kept point's row is that of its
// voxel, ranks_bev[interval_starts[interval]] (only intervals a kept point names are read, so a
// capacity-sized interval_starts is never read past the device-side interval count).
// T = bf16 (CL only): the gradient rows are bf16, widened in registers.
// TF = bf16: the pixel's feature row is read as bf16 and widened; feat_grad is stored as bf16,
// each float sum rounded once.
template <int KCH, bool COHERENT, bool CL = false, typename T = float, typename TF = float>
__device__ __forceinline__ void pixel_warp(float* wsm, int lane, const T* __restrict__ rows,
                                           const float* __restrict__ depth,
                                           const TF* __restrict__ feat,
                                           const int32_t* __restrict__ point_interval,
                                           const int32_t* __restrict__ ranks_bev,
                                           const int32_t* __restrict__ interval_starts,
                                           int64_t pix, int D, int HW, int C,
                                           float* __restrict__ depth_grad,
                                           TF* __restrict__ feat_grad) {
  constexpr int CC = 32 * KCH;
  constexpr int U = (KCH <= 2) ? 8 : 4;  // gradient rows in flight per warp
  // per warp: dots[D] | dep[D] | iis[D] (row index: interval, CL: voxel) | kd[D]
  float* dots = wsm;
  float* dep = dots + D;
  int* iis = reinterpret_cast<int*>(dep + D);
  int* kd = iis + D;
  const int64_t bn = pix / HW;
  const int hw = (int)(pix - bn * HW);
  const int64_t dbase = bn * (int64_t)D * HW + hw;

  int nk = 0;
  for (int d0 = 0; d0 < D; d0 += 32) {
    const int d = d0 + lane;
    int ii = -1;
    float dv = 0.f;
    if (d < D) {
      ii = __ldg(point_interval + pix * D + d);
      dv = __ldg(depth + dbase + (int64_t)d * HW);
      if (CL && ii >= 0) ii = __ldg(ranks_bev + __ldg(interval_starts + ii));
      dots[d] = 0.f;
    }
    const uint32_t m = __ballot_sync(0xffffffffu, ii >= 0);
    if (ii >= 0) {
      const int pos = nk + __popc(m & ((1u << lane) - 1u));
      kd[pos] = d;
      iis[pos] = ii;
      dep[pos] = dv;
    }
    nk += __popc(m);
  }
  __syncwarp();

  const int n_chunks = (C + CC - 1) / CC;
  for (int ch = 0; ch < n_chunks; ++ch) {
    const int cbase = ch * CC;
    float f[KCH], acc[KCH];
#pragma unroll
    for (int k = 0; k < KCH; ++k) {
      const int c = cbase + lane + 32 * k;
      f[k] = c < C ? ldg_widen(feat + pix * C + c) : 0.f;
      acc[k] = 0.f;
    }
    for (int j0 = 0; j0 < nk; j0 += U) {
      float g[U][KCH];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = min(j0 + u, nk - 1);
        const T* row = rows + (int64_t)iis[j] * C + cbase + lane;
#pragma unroll
        for (int k = 0; k < KCH; ++k) {
          if constexpr (COHERENT)
            g[u][k] = (cbase + lane + 32 * k < C) ? __ldcg(row + 32 * k) : 0.f;
          else
            g[u][k] = (cbase + lane + 32 * k < C) ? ldg_widen(row + 32 * k) : 0.f;
        }
      }
      float dot[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        dot[u] = 0.f;
        if (j0 + u < nk) {
          const float dv = dep[j0 + u];
#pragma unroll
          for (int k = 0; k < KCH; ++k) {
            dot[u] = fmaf(g[u][k], f[k], dot[u]);
            acc[k] = fmaf(dv, g[u][k], acc[k]);
          }
        }
      }
      int which;
      const float total = reduce_many<U>(dot, lane, which);
      // one lane per point (the lanes whose low bits are zero) owns the result
      if ((lane & (32 / U - 1)) == 0 && j0 + which < nk) dots[kd[j0 + which]] += total;
    }
#pragma unroll
    for (int k = 0; k < KCH; ++k) {
      const int c = cbase + lane + 32 * k;
      if (c < C) store_rn(feat_grad + pix * C + c, acc[k]);
    }
  }
  __syncwarp();
  // dense depth_grad column: dots[] is zero for dropped bins
  for (int d = lane; d < D; d += 32) depth_grad[dbase + (int64_t)d * HW] = dots[d];
}

// CL: the single-pass channels-last backward (rows = out_grad [B,Z,Y,X,C], no row pass).  (Its
// KCH = 8 instance spills 24 bytes at the register count ptxas picks on its own; the minimum of
// one CTA per SM lets it keep everything in registers.)
template <int KCH, bool CL = false, typename T = float, typename TF = float>
__global__ void __launch_bounds__(kBwdWarps * 32, CL ? 1 : 0)
k_bwd_pixels(const T* __restrict__ rows, const float* __restrict__ depth,
             const TF* __restrict__ feat, const int32_t* __restrict__ point_interval,
             const int32_t* __restrict__ ranks_bev, const int32_t* __restrict__ interval_starts,
             int64_t pix_begin, int64_t pix_end, int D, int HW, int C,
             float* __restrict__ depth_grad, TF* __restrict__ feat_grad) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t pix = pix_begin + (int64_t)blockIdx.x * kBwdWarps + warp;
  if (pix >= pix_end) return;
  pixel_warp<KCH, false, CL, T, TF>(smem + (size_t)warp * 4 * D, lane, rows, depth, feat, point_interval,
                             ranks_bev, interval_starts, pix, D, HW, C, depth_grad, feat_grad);
}

// (Round 2 measured a single-launch variant of this -- one persistent cooperative kernel whose row
// role and pixel role meet in L2 through two sample-sized slots -- and dropped it: bit-identical,
// but at C2 the pixel role needs the whole SM's warp slots to hide its gather latency (65 us per
// sample with 16 warps per SM against 12 us as its own kernel) and 35 MB of rows do not survive
// in L2 next to the 120 MB of out_grad a sample streams, evict-first / evict-last hints or not:
// 491 us against 324 us for the two launches below.  profiles/README.md has the role timeline.)

template <int KCH, typename T>
static int launch_rows(const T* out_grad, const int32_t* tile_istart, const uint32_t* tile_occ,
                       int64_t tile_begin, int64_t tile_end, int64_t tps, int64_t V, int C,
                       float* rows, cudaStream_t stream) {
  constexpr int CC = 32 * KCH;
  const size_t smem = sizeof(float) * kRowWarps * CC * kPitch;
  const size_t psmem = sizeof(T) * kRowWarps * 2 * CC * kRowPitchP;
  static int ctas_per_sm[kMaxDevices] = {};
  const int dev = current_device();
  if (ctas_per_sm[dev] == 0) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_bwd_rows<KCH, T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_bwd_rows_persistent<KCH, T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
    int n = 0;
    VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        &n, k_bwd_rows_persistent<KCH, T>, kRowWarps * 32, psmem));
    ctas_per_sm[dev] = n < 1 ? 1 : n;
  }
  const int n_chunks = (C + CC - 1) / CC;
  const int vec_ok = ((V & 3) == 0) && (((uintptr_t)out_grad & (4 * sizeof(T) - 1)) == 0);
  if (vec_ok && (V % kTileVoxels) == 0 && tile_begin == 0) {
    const int64_t n_items = tile_end * n_chunks;
    if (n_items <= 0) return 0;
    int64_t pblocks = (int64_t)ctas_per_sm[dev] * sm_count();
    if (pblocks > ceil_div64(n_items, kRowWarps)) pblocks = ceil_div64(n_items, kRowWarps);
    k_bwd_rows_persistent<KCH, T><<<(unsigned)pblocks, kRowWarps * 32, psmem, stream>>>(
        out_grad, tile_istart, tile_occ, n_items, tps, V, C, n_chunks, rows);
    VEON_LAUNCH_CHECK();
    return 0;
  }
  const int64_t blocks = ceil_div64(tile_end - tile_begin, kRowWarps) * n_chunks;
  if (blocks <= 0) return 0;
  if (blocks > 0x7fffffffLL) return VEON_E_RANGE;
  k_bwd_rows<KCH, T><<<(unsigned)blocks, kRowWarps * 32, smem, stream>>>(
      out_grad, tile_istart, tile_occ, tile_begin, tile_end, tps, V, C, n_chunks, vec_ok, rows);
  VEON_LAUNCH_CHECK();
  return 0;
}

template <int KCH, bool CL, typename T, typename TF>
static int launch_pixels(const T* rows, const float* depth, const TF* feat,
                         const int32_t* point_interval, const int32_t* ranks_bev,
                         const int32_t* interval_starts, int64_t pix_begin, int64_t pix_end,
                         int D, int HW, int C, float* depth_grad, TF* feat_grad,
                         cudaStream_t stream) {
  const size_t smem = sizeof(float) * kBwdWarps * 4 * (size_t)D;
  if (smem > 200 * 1024) return VEON_E_UNSUPPORTED;
  static size_t attr_smem[kMaxDevices] = {};
  const int dev = current_device();
  if (attr_smem[dev] == 0) attr_smem[dev] = 48 * 1024;
  if (smem > attr_smem[dev]) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_bwd_pixels<KCH, CL, T, TF>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem[dev] = smem;
  }
  const int64_t blocks = ceil_div64(pix_end - pix_begin, kBwdWarps);
  if (blocks <= 0) return 0;
  if (blocks > 0x7fffffffLL) return VEON_E_RANGE;
  k_bwd_pixels<KCH, CL, T, TF><<<(unsigned)blocks, kBwdWarps * 32, smem, stream>>>(
      rows, depth, feat, point_interval, ranks_bev, interval_starts, pix_begin, pix_end, D, HW, C,
      depth_grad, feat_grad);
  VEON_LAUNCH_CHECK();
  return 0;
}

// the compact rows of tiles [0, n_tiles)
template <typename T>
static int row_pass(const T* out_grad, const int32_t* tile_istart, const uint32_t* tile_occ,
                    int64_t n_tiles, int64_t tps, int64_t V, int C, float* rows,
                    cudaStream_t stream) {
  return C <= 32 ? launch_rows<1>(out_grad, tile_istart, tile_occ, 0, n_tiles, tps, V, C, rows, stream)
                 : launch_rows<2>(out_grad, tile_istart, tile_occ, 0, n_tiles, tps, V, C, rows, stream);
}

// ranks_bev / interval_starts: the channels-last pass (rows = out_grad), else NULL
template <bool CL = false, typename T = float, typename TF = float>
static int pixel_pass(const T* rows, const float* depth, const TF* feat,
                      const int32_t* point_interval, int64_t pixels, int D, int HW, int C,
                      float* depth_grad, TF* feat_grad, cudaStream_t stream,
                      const int32_t* ranks_bev = nullptr, const int32_t* interval_starts = nullptr) {
#define VEON_PIX(K_) launch_pixels<K_, CL, T, TF>(rows, depth, feat, point_interval, ranks_bev, interval_starts, 0, pixels, D, HW, C, depth_grad, feat_grad, stream)
  switch (C <= 32 ? 1 : (C <= 64 ? 2 : (C <= 256 ? 4 : 8))) {   // channels per lane
    case 1: return VEON_PIX(1);
    case 2: return VEON_PIX(2);
    case 4: return VEON_PIX(4);
    default: return VEON_PIX(8);
  }
#undef VEON_PIX
}

}  // namespace veon

using namespace veon;

extern "C" size_t veon_bev_pool_v2_bwd_workspace_floats(int64_t n_intervals, int B, int N, int D,
                                                        int H, int W, int C,
                                                        int64_t voxels_per_sample) {
  if (n_intervals < 0 || B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0 || C <= 0 ||
      voxels_per_sample <= 0)
    return 0;
  // one compact row per interval
  return (size_t)(n_intervals > 0 ? n_intervals : 1) * (size_t)C;
}

// The two passes on a channels-first out_grad of float or bf16 elements T (the rows are float),
// for feature rows (and their gradient) of float or bf16 elements TF.
template <typename T, typename TF = float>
static int bwd_planar(const T* out_grad, const float* depth, const TF* feat,
                      const int32_t* tile_istart, const uint32_t* tile_occ,
                      const int32_t* point_interval, int64_t n_intervals, int B, int N, int D,
                      int H, int W, int C, int64_t V, float* rows_ws, int64_t rows_ws_floats,
                      float* depth_grad, TF* feat_grad, cudaStream_t stream) {
  if (!out_grad || !depth || !feat || !tile_istart || !tile_occ || !point_interval || !rows_ws ||
      !depth_grad || !feat_grad || B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0 || C <= 0 ||
      V <= 0 || n_intervals < 0)
    return VEON_E_BADARG;
  if (rows_ws_floats < n_intervals * (int64_t)C) return VEON_E_WORKSPACE;
  const int64_t tps = ceil_div64(V, kTileVoxels);
  const int HW = H * W;
  const int64_t pix_per_sample = (int64_t)N * HW;
  // general route: one row launch + one pixel launch over all samples (launch ramps cost more
  // than keeping the rows L2-resident by sample groups saves: 456 vs 593 us at C2, round 1)
  const int rc = row_pass(out_grad, tile_istart, tile_occ, B * tps, tps, V, C, rows_ws, stream);
  if (rc) return rc;
  return pixel_pass(rows_ws, depth, feat, point_interval, B * pix_per_sample, D, HW, C,
                    depth_grad, feat_grad, stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar(
    const float* out_grad, const float* depth, const float* feat, const int32_t* tile_istart,
    const uint32_t* tile_occ, const int32_t* point_interval, int64_t n_intervals, int B, int N,
    int D, int H, int W, int C, int64_t V, float* rows_ws, int64_t rows_ws_floats,
    float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar(out_grad, depth, feat, tile_istart, tile_occ, point_interval, n_intervals, B,
                    N, D, H, W, C, V, rows_ws, rows_ws_floats, depth_grad, feat_grad,
                    (cudaStream_t)stream);
}

// bf16 out_grad: the row pass widens it into the same float rows, the pixel pass is unchanged.
extern "C" int veon_bev_pool_v2_bwd_planar_bf16(
    const uint16_t* out_grad, const float* depth, const float* feat, const int32_t* tile_istart,
    const uint32_t* tile_occ, const int32_t* point_interval, int64_t n_intervals, int B, int N,
    int D, int H, int W, int C, int64_t V, float* rows_ws, int64_t rows_ws_floats,
    float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar(reinterpret_cast<const bf16*>(out_grad), depth, feat, tile_istart, tile_occ,
                    point_interval, n_intervals, B, N, D, H, W, C, V, rows_ws, rows_ws_floats,
                    depth_grad, feat_grad, (cudaStream_t)stream);
}

// Single pass for a channels-last out_grad [B,Z,Y,X,C]: its occupied rows are already contiguous,
// so the pixel pass reads them in place -- no row pass, no scratch.  Same rows, same order of
// operations: the same bits as veon_bev_pool_v2_bwd_planar on the channels-first copy.
template <typename T, typename TF = float>
static int bwd_planar_cl(const T* out_grad, const float* depth, const TF* feat,
                         const int32_t* ranks_bev, const int32_t* interval_starts,
                         const int32_t* point_interval, int B, int N, int D, int H, int W, int C,
                         int64_t V, float* depth_grad, TF* feat_grad, void* stream_) {
  if (!out_grad || !depth || !feat || !ranks_bev || !interval_starts || !point_interval ||
      !depth_grad || !feat_grad || B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0 || C <= 0 ||
      V <= 0)
    return VEON_E_BADARG;
  if ((int64_t)B * V > 0x7fffffffLL) return VEON_E_RANGE;
  return pixel_pass<true>(out_grad, depth, feat, point_interval, (int64_t)B * N * H * W, D, H * W,
                          C, depth_grad, feat_grad, (cudaStream_t)stream_, ranks_bev,
                          interval_starts);
}

extern "C" int veon_bev_pool_v2_bwd_planar_cl(
    const float* out_grad, const float* depth, const float* feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* point_interval, int B, int N, int D, int H,
    int W, int C, int64_t V, float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar_cl(out_grad, depth, feat, ranks_bev, interval_starts, point_interval, B, N, D,
                       H, W, C, V, depth_grad, feat_grad, stream);
}

// bf16 out_grad rows, read in place and widened in registers: the same float fma chain.
extern "C" int veon_bev_pool_v2_bwd_planar_cl_bf16(
    const uint16_t* out_grad, const float* depth, const float* feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* point_interval, int B, int N, int D, int H,
    int W, int C, int64_t V, float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar_cl(reinterpret_cast<const bf16*>(out_grad), depth, feat, ranks_bev,
                       interval_starts, point_interval, B, N, D, H, W, C, V, depth_grad,
                       feat_grad, stream);
}

template <typename TG, typename TF>
static int bwd_planar_ds(
    const TG* grad_ds, const uint8_t* mask, const float* depth, const TF* feat,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* point_interval,
    int64_t n_intervals, int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
    float* rows_ws, float* depth_grad, TF* feat_grad, cudaStream_t stream) {
  if (!grad_ds || !mask || !depth || !feat || !tile_istart || !tile_occ || !point_interval ||
      !rows_ws || !depth_grad || !feat_grad || B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0 ||
      C <= 0 || Z <= 0 || Y <= 0 || X <= 0 || n_intervals < 0)
    return VEON_E_BADARG;
  if ((Z | Y | X) & 1) return VEON_E_UNSUPPORTED;
  const int64_t V = (int64_t)Z * Y * X;
  const int64_t tps = ceil_div64(V, kTileVoxels), n_tiles = (int64_t)B * tps;
  if ((int64_t)B * V > 0x7fffffffLL) return VEON_E_RANGE;
  const int sms = sm_count();
  const int64_t plane = (int64_t)(Z / 2) * (Y / 2) * (X / 2);
  const bool direct = (X % 8) == 0 && (plane % 4) == 0 &&
                      ((uintptr_t)grad_ds & (4 * sizeof(TG) - 1)) == 0 &&
                      ((uintptr_t)mask & 3) == 0;
  int64_t blocks = ceil_div64(n_tiles, 8);
  if (blocks > (int64_t)sms * 8) blocks = (int64_t)sms * 8;
  if (direct)
    k_bwd_rows_ds_direct<TG><<<(unsigned)blocks, 256, 0, stream>>>(
        grad_ds, mask, tile_istart, tile_occ, n_tiles, tps, Z, Y, X, C, rows_ws);
  else
    k_bwd_rows_ds<TG><<<(unsigned)blocks, 256, 0, stream>>>(grad_ds, mask, tile_istart, tile_occ,
                                                            n_tiles, tps, Z, Y, X, C, rows_ws);
  VEON_LAUNCH_CHECK();
  return pixel_pass(rows_ws, depth, feat, point_interval, (int64_t)B * N * H * W, D, H * W, C,
                    depth_grad, feat_grad, stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_ds(
    const float* grad_ds, const uint8_t* mask, const float* depth, const float* feat,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* point_interval,
    int64_t n_intervals, int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
    float* rows_ws, float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar_ds(grad_ds, mask, depth, feat, tile_istart, tile_occ, point_interval,
                       n_intervals, B, N, D, H, W, C, Z, Y, X, rows_ws, depth_grad, feat_grad,
                       (cudaStream_t)stream);
}

// bfloat16 feature rows [B*N*H*W, C] and their gradient: the pixel pass reads each pixel's row as
// bf16 (widened exactly) and stores feat_grad as bf16 (the float sums rounded once, to nearest
// even); depth_grad and the row passes are those of the float twins, bit for bit.  Arguments,
// checks and error codes are the twins'.
extern "C" int veon_bev_pool_v2_bwd_planar_bf16feat(
    const float* out_grad, const float* depth, const uint16_t* feat, const int32_t* tile_istart,
    const uint32_t* tile_occ, const int32_t* point_interval, int64_t n_intervals, int B, int N,
    int D, int H, int W, int C, int64_t V, float* rows_ws, int64_t rows_ws_floats,
    float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar(out_grad, depth, reinterpret_cast<const bf16*>(feat), tile_istart, tile_occ,
                    point_interval, n_intervals, B, N, D, H, W, C, V, rows_ws, rows_ws_floats,
                    depth_grad, reinterpret_cast<bf16*>(feat_grad), (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_bf16_bf16feat(
    const uint16_t* out_grad, const float* depth, const uint16_t* feat, const int32_t* tile_istart,
    const uint32_t* tile_occ, const int32_t* point_interval, int64_t n_intervals, int B, int N,
    int D, int H, int W, int C, int64_t V, float* rows_ws, int64_t rows_ws_floats,
    float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar(reinterpret_cast<const bf16*>(out_grad), depth,
                    reinterpret_cast<const bf16*>(feat), tile_istart, tile_occ, point_interval,
                    n_intervals, B, N, D, H, W, C, V, rows_ws, rows_ws_floats, depth_grad,
                    reinterpret_cast<bf16*>(feat_grad), (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_cl_bf16feat(
    const float* out_grad, const float* depth, const uint16_t* feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* point_interval, int B, int N, int D, int H,
    int W, int C, int64_t V, float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar_cl(out_grad, depth, reinterpret_cast<const bf16*>(feat), ranks_bev,
                       interval_starts, point_interval, B, N, D, H, W, C, V, depth_grad,
                       reinterpret_cast<bf16*>(feat_grad), stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_cl_bf16_bf16feat(
    const uint16_t* out_grad, const float* depth, const uint16_t* feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* point_interval, int B, int N, int D, int H,
    int W, int C, int64_t V, float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar_cl(reinterpret_cast<const bf16*>(out_grad), depth,
                       reinterpret_cast<const bf16*>(feat), ranks_bev, interval_starts,
                       point_interval, B, N, D, H, W, C, V, depth_grad,
                       reinterpret_cast<bf16*>(feat_grad), stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_ds_bf16feat(
    const float* grad_ds, const uint8_t* mask, const float* depth, const uint16_t* feat,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* point_interval,
    int64_t n_intervals, int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
    float* rows_ws, float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar_ds(grad_ds, mask, depth, reinterpret_cast<const bf16*>(feat), tile_istart,
                       tile_occ, point_interval, n_intervals, B, N, D, H, W, C, Z, Y, X, rows_ws,
                       depth_grad, reinterpret_cast<bf16*>(feat_grad), (cudaStream_t)stream);
}

// bfloat16 grad_ds [B,C,Z/2,Y/2,X/2] (the reduced volume of veon_maxdown2_fwd_mask_bf16): widened
// exactly where the row pass loads it, everything after is the float32 twin's.
extern "C" int veon_bev_pool_v2_bwd_planar_ds_bf16(
    const uint16_t* grad_ds, const uint8_t* mask, const float* depth, const float* feat,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* point_interval,
    int64_t n_intervals, int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
    float* rows_ws, float* depth_grad, float* feat_grad, void* stream) {
  return bwd_planar_ds(reinterpret_cast<const bf16*>(grad_ds), mask, depth, feat, tile_istart,
                       tile_occ, point_interval, n_intervals, B, N, D, H, W, C, Z, Y, X, rows_ws,
                       depth_grad, feat_grad, (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_bwd_planar_ds_bf16_bf16feat(
    const uint16_t* grad_ds, const uint8_t* mask, const float* depth, const uint16_t* feat,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* point_interval,
    int64_t n_intervals, int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
    float* rows_ws, float* depth_grad, uint16_t* feat_grad, void* stream) {
  return bwd_planar_ds(reinterpret_cast<const bf16*>(grad_ds), mask, depth,
                       reinterpret_cast<const bf16*>(feat), tile_istart, tile_occ, point_interval,
                       n_intervals, B, N, D, H, W, C, Z, Y, X, rows_ws, depth_grad,
                       reinterpret_cast<bf16*>(feat_grad), (cudaStream_t)stream);
}

#ifdef VEON_TOOLS   // tools/build_variant.sh NAME "-DVEON_TOOLS": never in the shipped library
// ---- experiment hooks (not part of include/veon_lift.h; used by tools/bwd_pipeline.py) -------------
// the two passes on their own, and an L2 access-policy window for a stream
extern "C" int veon_internal_bwd_rows(const float* out_grad, const int32_t* tile_istart,
                                      const uint32_t* tile_occ, int64_t n_tiles, int64_t tps,
                                      int64_t V, int C, float* rows, void* stream) {
  return row_pass(out_grad, tile_istart, tile_occ, n_tiles, tps, V, C, rows, (cudaStream_t)stream);
}
extern "C" int veon_internal_bwd_pixels(const float* rows, const float* depth, const float* feat,
                                        const int32_t* point_interval, int64_t pixels, int D, int HW,
                                        int C, float* depth_grad, float* feat_grad, void* stream) {
  return pixel_pass(rows, depth, feat, point_interval, pixels, D, HW, C, depth_grad, feat_grad,
                    (cudaStream_t)stream);
}
extern "C" int veon_internal_l2_window(void* stream, void* base, size_t bytes, float hit_ratio,
                                       size_t set_aside_bytes) {
  if (set_aside_bytes) {
    cudaError_t e = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside_bytes);
    if (e != cudaSuccess) return (int)e;
  }
  cudaStreamAttrValue a = {};
  a.accessPolicyWindow.base_ptr = base;
  a.accessPolicyWindow.num_bytes = bytes;
  a.accessPolicyWindow.hitRatio = hit_ratio;
  a.accessPolicyWindow.hitProp = bytes ? cudaAccessPropertyPersisting : cudaAccessPropertyNormal;
  a.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  return (int)cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &a);
}
#endif  // VEON_TOOLS
