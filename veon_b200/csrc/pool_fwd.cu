// bev_pool_v2 forward, fused with the reference's memset and transpose.
//
// Reference behaviour: QuickCumsumCuda.forward (bev_pool.py:17-41: new_zeros
// + bev_pool_v2_kernel, bev_pool_cuda.cu:21-48) followed by
// `.permute(0,4,1,2,3).contiguous()` (bev_pool.py:91).  The reference runs one
// thread per (interval, channel), writes only occupied voxels of a
// channels-last volume, and needs a memset before and a full transpose after.
//
// Here one warp handles one 32-voxel x-run of the output ("tile") for a chunk of
// 32*KCH channels at a time (persistent grid, warps stride over the tiles).
// Because points are sorted by voxel, the tile's points are one contiguous
// slice [tile_start[t], tile_start[t+1]) of the rank arrays.  Lanes run over
// CHANNELS while gathering (feature rows are read as full 128-byte lines, the
// per-voxel sum lives in registers) and over VOXELS while storing (one 16-byte
// store per lane = four full 128-byte lines of four channel planes per
// instruction); a padded, zero-filled shared tile [c][33] does the transposition.
// Empty voxels come out as zeros, so the volume is touched exactly once: no
// memset, no permute pass, no atomics.  Accumulation order inside a voxel is the
// rank order, fma(feat, depth, acc) starting from 0 -- the same sequence of
// roundings as the reference kernel's `psum += feat * depth`.
//
// Kernels in this file:
//   k_pool_fwd         the warp-per-tile kernel above: the general route (any C, ragged volumes,
//                      no workspace).  Aligned volumes with C % 64 == 0 take the two-role
//                      streaming kernel of pool_fwd_stream.cu instead (see there).
//   k_pool_fwd_heavy   a CTA per heavy tile (rows staged by cp.async), queued behind the main grid
//   k_pool_fwd_narrow  C <= 32 (C % 4 == 0): a LANE per voxel instead of a lane per channel, all
//                      channels of the voxel in registers, same fma order; heavy grid first
//   k_pool_ds_fwd      opt-in: pooling fused with the neck's 2x2x2 max-downsample
// The first three also write channels-last volumes out[B,Z,Y,X,C] (template flag CL,
// veon_bev_pool_v2_fwd_planar_cl): same sums, rows instead of channel planes.
#include <type_traits>

#include "common.cuh"
#include "pool_fwd.cuh"

#ifndef VEON_FWD_WARPS
#define VEON_FWD_WARPS 8
#endif

namespace veon {

// x 2 CTAs/SM.  Keep it at 8: the 8 consecutive tiles of a CTA then cover an aligned 1 KB
// of every channel plane; 7-warp CTAs (896 B) write the same volume 19 % slower
// (tools/micro/store_pattern.cu: 266 vs 224 us).
constexpr int kFwdWarps = VEON_FWD_WARPS;
// Row pitch of the [channel][voxel] shared tiles.  Odd: the per-voxel store of a channel column
// (lane = channel, address lane * pitch + v) and the write-out reads (4 rows x 8 voxel quads)
// are then both conflict-free.  (36 kept the rows 16-byte aligned for LDS.128 but made every
// voxel store a 4-way bank conflict: 65 M of 117 M shared-memory wavefronts at C3, ncu.)
constexpr int kRowPitch = kTileVoxels + 1;

// ---- per-warp prefetch ring in shared memory (cp.async, no registers held) ----
// slot (ints): [0]=s [1]=e [2]=tile [3]=cbase, then one int4 per point (lane j):
//   landing   {ranks_bev, ranks_feat, ranks_depth, depth}
//   fixed up  {ranks_bev, row offset (floats), voxel | first<<8, depth}
#ifndef VEON_FWD_DIST
#define VEON_FWD_DIST 2
#endif
constexpr int kDist = VEON_FWD_DIST;         // prefetch distance in items per stage
constexpr int kRingSlots = 4 * kDist;        // bounds run 3*kDist ahead
constexpr int kSlotInts = 4 + 4 * 32;

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// every group except the (kDist-1) most recent ones has landed
__device__ __forceinline__ void cp_async_wait_dist() {
  asm volatile("cp.async.wait_group %0;" ::"n"(kDist - 1) : "memory");
}

// Channels-last zeros: voxels [va, vb) of the tile whose first voxel has the global index g0,
// channels [c0, c0 + cw) of each row.  Whole rows are one contiguous span (16-byte stores when
// aligned); a channel chunk of a row is one span per voxel.  Warp-wide.
template <typename T>
__device__ __forceinline__ void zero_rows_cl(T* __restrict__ out, int64_t g0, int va, int vb,
                                             int c0, int cw, int C, int lane) {
  auto span = [&](T* p, int64_t n) {
    if ((((uintptr_t)p | (uintptr_t)(n * (int64_t)sizeof(T))) & (4 * sizeof(T) - 1)) == 0) {
      for (int64_t i = 4 * lane; i < n; i += 128) st_stream4(p + i, make_float4(0.f, 0.f, 0.f, 0.f));
    } else {
      for (int64_t i = lane; i < n; i += 32) st_stream(p + i, 0.f);
    }
  };
  if (va >= vb) return;
  if (cw == C) {
    span(out + (g0 + va) * C, (int64_t)(vb - va) * C);
  } else {
    for (int v = va; v < vb; ++v) span(out + (g0 + v) * C + c0, cw);
  }
}

// A feature element as the lane-per-channel gather carries it: a float as it is, a bf16 as its raw
// bits, widened only at the fma (a widened copy next to each of the rows in flight made the
// kernel spill).
__device__ __forceinline__ float ld_feat(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_feat(const bf16* p) {
  return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)));
}
template <typename TF>
__device__ __forceinline__ float feat_value(float v) {
  if constexpr (std::is_same<TF, float>::value) return v;
  else return __uint_as_float(__float_as_uint(v) << 16);
}

// Persistent: every warp strides over (tile, channel-chunk) items.
//  * index prefetch: tile bounds -> rank triple -> depth value run 3 / 2 / 1 x kDist
//    items ahead as 4-byte cp.async copies into a per-warp ring (no registers held;
//    `wait_group kDist-1` leaves the youngest group in flight, so short items do not
//    expose the latency); a lanes=points fix-up turns the landed ranks into
//    (row byte offset, voxel | first-of-voxel) so that the gather loop needs ONE
//    broadcast LDS.128 per point.  The (tile, chunk, sample) of the next item is kept
//    as running counters: no integer division in the loop;
//  * gather: lanes = channels, up to 16 points' rows in flight (issued in groups of 4,
//    groups past the tile's last point are skipped), per-voxel sums in registers
//    (fma(feat, depth, acc) in rank order), one store per occupied voxel into the
//    zero-filled [c][33] shared tile;
//  * write-out: lanes = voxels, LDS.128 + one 16-byte streaming store covers
//    4 channel planes x 128 B per instruction.
// (A TMA tensor-store write-out was measured slower here: ~17 B/clk/SM for boxes
//  of 128-byte rows vs ~23 B/clk/SM for st.global.v4; see profiles/README.md.)
// Slot header: [0]=s [1]=e [2]=g0 (global voxel index of the tile's first voxel)
//              [3]=sample<<16 | chunk
// FULLC: C is a multiple of the chunk width, so no channel predicate anywhere.
// LOOPC (rows wider than one chunk): an item is a whole TILE and the channel chunks are looped
// inside it -- the index work (ring, fix-up, the records of the points past the first 32, kept
// in `ext`) is done once per tile instead of once per (tile, chunk).
// CL: channels-last output out[B,Z,Y,X,C].  The shared tile is then ROW-major, [voxel][CC + 4]:
// a finished voxel sum (lanes = channels) is one conflict-free row store, and the write-out
// moves the tile's rows -- one contiguous 32 * C * 4-byte block when a chunk holds every
// channel -- with 16-byte loads and stores (vec_ok: C % 4 == 0 and a 16-byte aligned volume).
// Nothing is transposed.  (Storing the rows straight from the registers, with zeros for the
// empty voxels between them, was measured at 578 us at C2: short scattered stores.)
// T: the volume's element type, float or bf16 (rounded once, at the store; the tiles stay float).
// TF: the feature rows' element type, float or bf16: a lane loads its channel's 2 or 4 bytes and
// widens them exactly; the point records' byte offsets scale by sizeof(TF).
template <int KCH, bool FULLC, bool LOOPC = false, bool CL = false, typename T = float,
          typename TF = float>
__global__ void __launch_bounds__(kFwdWarps * 32)
k_pool_fwd(const float* __restrict__ depth, const TF* __restrict__ feat,
           const int32_t* __restrict__ ranks_depth, const int32_t* __restrict__ ranks_feat,
           const int32_t* __restrict__ ranks_bev, const int32_t* __restrict__ tile_start,
           const int32_t* __restrict__ heavy, uint32_t n_items, uint32_t tiles_per_sample,
           int64_t V, int C, uint32_t n_chunks, int vec_ok, T* __restrict__ out,
           uint32_t loop_chunks) {
  constexpr int CC = 32 * KCH;
  constexpr int U = (KCH <= 2) ? 16 : 8;  // feature rows in flight per warp
  constexpr int kClPitch = CC + 4;   // CL: row pitch of the [voxel][channel] tile
  constexpr int kTileFloats = CL ? kTileVoxels * kClPitch : CC * kRowPitch;
  // records of the points past the first 32 of a tile (a tile of the main grid has fewer points
  // than the plan's heavy threshold)
  constexpr int kExtInts = LOOPC ? ((kHeavyDefaultThreshold + 31) / 32 - 1) * 128 : 0;
  constexpr int kWarpFloats = kTileFloats + kRingSlots * kSlotInts + kExtInts;
  extern __shared__ __align__(16) float smem[];
  pdl_launch_dependents();  // the heavy-tile grid may be queued behind this one
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* tile = smem + warp * kWarpFloats;
  int32_t* ring = reinterpret_cast<int32_t*>(tile + kTileFloats);
  int32_t* ext = ring + kRingSlots * kSlotInts;
  (void)ext;
  const uint32_t TW = gridDim.x * kFwdWarps;
  const uint32_t first_item = blockIdx.x * kFwdWarps + warp;
  if (first_item >= n_items) return;
  const uint32_t my_items = (n_items - first_item + TW - 1) / TW;
  // tiles with at least this many points belong to k_pool_fwd_heavy
  const int32_t heavy_thr = heavy ? __ldg(heavy + 1) : 0x7fffffff;
  const uint32_t Vu = (uint32_t)V;                    // B*V < 2^31 (checked by the launcher)
  const bool whole_tiles = (Vu % kTileVoxels) == 0;   // no ragged tile at a sample's end

  // running decode of the next item to enter the ring (advanced by TW items per call)
  uint32_t nx_t = first_item / n_chunks;
  uint32_t nx_chunk = first_item - nx_t * n_chunks;
  uint32_t nx_b = nx_t / tiles_per_sample;
  uint32_t nx_vt = nx_t - nx_b * tiles_per_sample;
  const uint32_t step_t = TW / n_chunks, step_c = TW - step_t * n_chunks;

  auto slot_of = [&](uint32_t m) { return ring + (m & (kRingSlots - 1)) * kSlotInts; };
  auto issue_bounds = [&](uint32_t m) {  // header of item m; must be called for m = 0, 1, 2, ...
    int32_t* sl = slot_of(m);
    if (m < my_items) {
      if (lane < 2) cp_async4(sl + lane, tile_start + nx_t + lane);
      if (lane == 0) {
        const int32_t g0 = (int32_t)(nx_b * Vu + nx_vt * kTileVoxels);
        *reinterpret_cast<int2*>(sl + 2) = make_int2(g0, (int)((nx_b << 16) | nx_chunk));
      }
      uint32_t dt = step_t;
      nx_chunk += step_c;
      if (nx_chunk >= n_chunks) {
        nx_chunk -= n_chunks;
        ++dt;
      }
      nx_t += dt;
      nx_vt += dt;
      while (nx_vt >= tiles_per_sample) {
        nx_vt -= tiles_per_sample;
        ++nx_b;
      }
    } else if (lane < 2) {
      sl[lane] = 0;
    }
  };
  auto issue_ranks = [&](uint32_t m) {  // needs bounds(m)
    int32_t* sl = slot_of(m);
    int32_t* pt = sl + 4 + 4 * lane;
    const int2 se = *reinterpret_cast<const int2*>(sl);
    const int32_t i = se.x + lane;
    if (i < se.y) {
      cp_async4(pt + 0, ranks_bev + i);
      cp_async4(pt + 1, ranks_feat + i);
      cp_async4(pt + 2, ranks_depth + i);
    } else {
      pt[0] = -1;
    }
  };
  // needs ranks(m): depth gather + fix-up of the landed ranks (lanes = points)
  auto issue_depth = [&](uint32_t m) {
    int32_t* sl = slot_of(m);
    int32_t* pt = sl + 4 + 4 * lane;
    const int32_t rb = pt[0];
    if (rb >= 0) {
      cp_async4(pt + 3, depth + pt[2]);
      const int2 h = *reinterpret_cast<const int2*>(sl + 2);
      const int32_t up = lane ? pt[-4] : -1;
      // byte offset of this channel chunk of the point's feature row (< 2^32, checked)
      pt[1] = (int32_t)(((uint32_t)pt[1] * (uint32_t)C + (uint32_t)(h.y & 0xffff) * CC) *
                        (uint32_t)sizeof(TF));
      pt[2] = (rb - h.x) | ((rb != up) ? 0x100 : 0);  // voxel | first-of-voxel
    }
  };

  // prologue: fill the pipeline (three serialized latencies, once per warp)
#pragma unroll
  for (int i = 0; i < 3 * kDist; ++i) issue_bounds(i);
  cp_async_commit(); cp_async_wait_all(); __syncwarp();
#pragma unroll
  for (int i = 0; i < 2 * kDist; ++i) issue_ranks(i);
  cp_async_commit(); cp_async_wait_all(); __syncwarp();
#pragma unroll
  for (int i = 0; i < kDist; ++i) issue_depth(i);
  cp_async_commit(); cp_async_wait_all(); __syncwarp();

  const int q4 = (lane & 7) * 4, r = lane >> 3;  // write-out role of this lane
  float* const tlane = tile + lane * kRowPitch;   // flush base: channel = lane (+32k)
  const char* const feat_lane = reinterpret_cast<const char*>(feat) + lane * (int)sizeof(TF);
  const int64_t ostep = 4 * V;

  for (uint32_t m = 0; m < my_items; ++m) {
    cp_async_wait_dist();
    __syncwarp();
    int32_t* sl = slot_of(m);
    const int4 h = *reinterpret_cast<const int4*>(sl);  // s, e, g0, sample<<16 | chunk
    issue_bounds(m + 3 * kDist);  // lands in the slot item m-kDist used
    issue_ranks(m + 2 * kDist);
    issue_depth(m + kDist);
    cp_async_commit();
    const int32_t s0 = h.x, e0 = h.y, g0 = h.z;
    if (e0 - s0 >= heavy_thr) continue;

    const uint32_t b = (uint32_t)h.w >> 16;
    const bool fast = vec_ok && (whole_tiles || (uint32_t)g0 - b * Vu + kTileVoxels <= Vu);
    const uint32_t n_loop = LOOPC ? loop_chunks : 1u;
    // CL: voxels of this tile inside the volume (a ragged sample end has fewer than 32)
    const int v_end = CL ? (int)min((uint32_t)kTileVoxels, Vu - ((uint32_t)g0 - b * Vu)) : 0;

    if (CL && e0 <= s0) {  // empty tile
      const int c_lo = LOOPC ? 0 : (h.w & 0xffff) * CC;
      zero_rows_cl(out, g0, 0, v_end, c_lo, LOOPC ? C : min(CC, C - c_lo), C, lane);
      continue;
    }
    if (!CL && e0 <= s0 && fast) {  // empty tile
      const int c_lo = LOOPC ? 0 : (h.w & 0xffff) * CC;
      const int c_hi = LOOPC ? C : min(c_lo + CC, C);
      T* o = out + (int64_t)(b * (uint32_t)(C - 1) + (uint32_t)(c_lo + r)) * V + g0 + q4;
#ifndef VEON_FWD_X_NOSTORE
#pragma unroll 4
      for (int c = c_lo + r; c < c_hi; c += 4, o += ostep) st_stream4(o, make_float4(0.f, 0.f, 0.f, 0.f));
#endif
      continue;
    }

    // records of the points past the first 32 (a tile of the main grid has < heavy_thr <= 96):
    // fetched synchronously; LOOPC keeps them in `ext` for all channel chunks of the tile
    auto fetch_block = [&](int32_t base, int32_t* dst, int32_t last_rb, int cb) {
      const int32_t i = base + lane;
      int32_t rb = -1, rf = 0;
      float d = 0.f;
      if (i < e0) {
        rb = __ldg(ranks_bev + i);
        rf = __ldg(ranks_feat + i);
        d = __ldg(depth + __ldg(ranks_depth + i));
      }
      int32_t up = __shfl_up_sync(0xffffffffu, rb, 1);
      if (lane == 0) up = last_rb;   // first point of the block: new voxel iff it differs
      int32_t* pt = dst + 4 * lane;
      pt[0] = rb;
      pt[1] = (int32_t)(((uint32_t)rf * (uint32_t)C + (uint32_t)cb) * (uint32_t)sizeof(TF));
      pt[2] = (rb - g0) | ((rb != up) ? 0x100 : 0);
      pt[3] = __float_as_int(d);
      return __shfl_sync(0xffffffffu, rb, 31);
    };
    if constexpr (LOOPC) {
      int32_t last = sl[4 + 4 * 31 + 0];
      int blk = 0;
      for (int32_t base = s0 + 32; base < e0; base += 32, ++blk)
        last = fetch_block(base, ext + 128 * blk, last, 0);
      __syncwarp();
    }

    for (uint32_t ch = 0; ch < n_loop; ++ch) {
      const int cbase = LOOPC ? (int)ch * CC : (h.w & 0xffff) * CC;
      const int cmax = FULLC ? CC : min(CC, C - cbase);
      // (b*C + cbase + r)*V + v0 + q4  with  v0 = g0 - b*V
      T* o = out + (int64_t)(b * (uint32_t)(C - 1) + (uint32_t)(cbase + r)) * V + g0 + q4;
      const char* const feat_ch = feat_lane + (LOOPC ? (uint32_t)cbase * (uint32_t)sizeof(TF) : 0u);

      __syncwarp();
      {  // zero the tile (empty voxels must read as 0)
        float4* t4 = reinterpret_cast<float4*>(tile);
#pragma unroll
        for (int i = 0; i < (kTileFloats / 4 + 31) / 32; ++i)
          if (lane + 32 * i < kTileFloats / 4) t4[lane + 32 * i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      __syncwarp();

      float acc[KCH];
      int acc_vl = -1;
      const bool full_chunk = FULLC || (cmax == CC);
      // one finished voxel into the tile: CL row acc_vl, else column acc_vl
      auto flush = [&]() {
#pragma unroll
        for (int k = 0; k < KCH; ++k) {
          if constexpr (CL) tile[acc_vl * kClPitch + lane + 32 * k] = acc[k];
          else tlane[32 * k * kRowPitch + acc_vl] = acc[k];
        }
      };
      int blk = 0;
      for (int32_t base = s0; base < e0; base += 32, ++blk) {
        const int cnt = min(32, e0 - base);
        const int4* pts = reinterpret_cast<const int4*>(sl + 4);
        if (base != s0) {
          if constexpr (LOOPC) {
            pts = reinterpret_cast<const int4*>(ext + 128 * (blk - 1));
          } else {  // one chunk per item: the later blocks go through the slot
            __syncwarp();
            const int32_t last = sl[4 + 4 * 31 + 0];
            __syncwarp();
            fetch_block(base, sl + 4, last, cbase);
            __syncwarp();
          }
        }
        for (int j0 = 0; j0 < cnt; j0 += U) {
          int4 p[U];
          float f[U][KCH];
#pragma unroll
          for (int g = 0; g < U / 4; ++g) {
            if (j0 + 4 * g < cnt) {  // warp-uniform: skip the groups past the last point
#pragma unroll
              for (int uu = 0; uu < 4; ++uu) {
                const int u = 4 * g + uu;
                p[u] = pts[min(j0 + u, cnt - 1)];
                const TF* row = reinterpret_cast<const TF*>(feat_ch + (uint32_t)p[u].y);
#pragma unroll
                for (int k = 0; k < KCH; ++k)
#ifdef VEON_FWD_X_NOGATHER   // tools only: elimination timing
                  f[u][k] = (float)p[u].y;
#else
                  f[u][k] = (FULLC || full_chunk || lane + 32 * k < cmax) ? ld_feat(row + 32 * k) : 0.f;
#endif
              }
            }
          }
#pragma unroll
          for (int g = 0; g < U / 4; ++g) {
            if (j0 + 4 * g < cnt) {
#pragma unroll
              for (int uu = 0; uu < 4; ++uu) {
                const int u = 4 * g + uu;
                if (j0 + u < cnt) {
                  const float dj = __int_as_float(p[u].w);
                  if (p[u].z & 0x100) {  // first point of its voxel (warp-uniform)
                    if (acc_vl >= 0) flush();
                    acc_vl = p[u].z & 0xff;
#pragma unroll
                    for (int k = 0; k < KCH; ++k) acc[k] = fmaf(feat_value<TF>(f[u][k]), dj, 0.f);
                  } else {
#pragma unroll
                    for (int k = 0; k < KCH; ++k) acc[k] = fmaf(feat_value<TF>(f[u][k]), dj, acc[k]);
                  }
                }
              }
            }
          }
        }
      }
      if (acc_vl >= 0) flush();
      __syncwarp();

      if constexpr (CL) {
        // rows v < v_end, channels [cbase, cbase + cmax): element (or 16-byte piece) j of the
        // flat [v][q] index space per lane and step, (v, q) advanced without a division
        const int w = vec_ok ? 4 : 1;
        const int per_row = cmax / w;
        int v = 0, q = lane;
        while (q >= per_row) { q -= per_row; ++v; }
        T* const obase = out + (int64_t)g0 * C + cbase;
        for (; v < v_end;) {
          const float* t = tile + v * kClPitch + q * w;
          T* o = obase + (int64_t)v * C + q * w;
          if (vec_ok) st_stream4(o, *reinterpret_cast<const float4*>(t));
          else st_stream(o, *t);
          q += 32;
          while (q >= per_row) { q -= per_row; ++v; }
        }
        continue;   // (the __syncwarp before the next zero-fill protects the tile reuse)
      }

      // Write-out: lane (r = lane/8, q = lane%8) moves voxels 4q..4q+3 of channel
      // 4*it + r with four LDS.32 + one 16-byte streaming store.
      const float* trow = tile + r * kRowPitch + q4;
      if (fast) {
#pragma unroll 4
        for (int c = r; c < cmax; c += 4, o += ostep, trow += 4 * kRowPitch) {
#ifdef VEON_FWD_X_NOSTORE
          if (trow[0] == 123.456f) st_stream4(o, make_float4(trow[0], trow[1], trow[2], trow[3]));
#else
          st_stream4(o, make_float4(trow[0], trow[1], trow[2], trow[3]));
#endif
        }
      } else {  // ragged volume edge / unaligned volume: scalar, bounds-checked
        const int v0 = (int)((uint32_t)g0 - b * Vu);
        for (int c = r; c < cmax; c += 4, o += ostep, trow += 4 * kRowPitch)
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (v0 + q4 + i < V) st_stream(o + i, trow[i]);
      }
      // (the __syncwarp before the next zero-fill protects the tile reuse)
    }
    // (the __syncwarp before the next zero-fill protects the tile reuse)
  }
  cp_async_wait_all();
}

// ---- heavy tiles -------------------------------------------------------------
// A tile with hundreds of points (voxels next to the cameras collect a whole
// frustum column each) would keep ONE warp of the kernel above busy for longer
// than an average warp's entire share of the volume, one exposed load latency per
// 16 points.  The plan lists such tiles and the kernel above skips them; here a
// whole CTA takes one: 128 points per round, ALL their feature rows in flight at
// once (cp.async into shared memory, the index records of the next two rounds
// prefetched in registers), then each warp runs the fma chains of its voxels out
// of shared memory.  Only the loads are parallelised -- every (voxel, channel) sum
// is still accumulated point by point in rank order (partial sums are carried in
// the shared tile between rounds), so the result stays bit-identical.
constexpr int kHeavyThreads = 256;
constexpr int kHeavyChunk = 128;  // points per round; one index record per thread < 128

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}

// Fused lift + classify (veon_lift_classify_fwd): the pooled channels are
// [gate 0, gate 1, logit 0 .. Q-1, padding] and a tile ends as 32 labels instead of C planes.
struct ClsArgs {
  const int32_t* cls;   // [Q] merged class of every prompt row
  uint8_t* labels;      // [B,X,Y,Z]
  int Q, X, Y, Z, free_label;
};
__device__ __forceinline__ void store_label(const ClsArgs& ca, uint32_t b, uint32_t v, int label) {
  const uint32_t row = v / (uint32_t)ca.X, x = v - row * (uint32_t)ca.X;
  const uint32_t z = row / (uint32_t)ca.Y, y = row - z * (uint32_t)ca.Y;
  ca.labels[(((int64_t)b * ca.X + x) * ca.Y + y) * ca.Z + z] = (uint8_t)label;
}

// CL: channels-last write-out (warp = voxel, lanes = channels), see k_pool_fwd
// TF = bf16: rows are staged as they are (8-byte copies of 4-channel pieces, half the shared
// memory) and widened in the fma chains.
template <int KCH, bool CLS = false, bool CL = false, typename T = float, typename TF = float>
__global__ void __launch_bounds__(kHeavyThreads)
k_pool_fwd_heavy(const float* __restrict__ depth, const TF* __restrict__ feat,
                 const int32_t* __restrict__ ranks_depth, const int32_t* __restrict__ ranks_feat,
                 const int32_t* __restrict__ ranks_bev, const int32_t* __restrict__ tile_start,
                 const int32_t* __restrict__ heavy, int heavy_cap, uint32_t tiles_per_sample,
                 int64_t V, int C, uint32_t n_chunks, int vec_ok, T* __restrict__ out,
                 int join, int min_points, ClsArgs ca = ClsArgs()) {
  constexpr int CC = 32 * KCH;
  constexpr int kSegs = CC / 4;  // 16-byte segments per staged row
  extern __shared__ __align__(16) float hsm[];
  TF* rows = reinterpret_cast<TF*>(hsm);                        // [kHeavyChunk][CC]
  float* tile = reinterpret_cast<float*>(rows + kHeavyChunk * CC);  // [CC][kRowPitch]
  float* dep = tile + CC * kRowPitch;                           // [kHeavyChunk]
  uint32_t* off = reinterpret_cast<uint32_t*>(dep + kHeavyChunk);  // [kHeavyChunk]
  int32_t* bounds = reinterpret_cast<int32_t*>(off + kHeavyChunk); // [2][start 32 | end 32]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // no griddepcontrol.wait up front: this grid and the main grid write disjoint tiles and read
  // only what earlier, normally launched work produced; it joins at the end (below)
  pdl_launch_dependents();
  const uint32_t n_heavy = (uint32_t)min(__ldg(heavy), heavy_cap);
  const uint32_t n_work = n_heavy * n_chunks;

  for (uint32_t w = blockIdx.x; w < n_work; w += gridDim.x) {
    const uint32_t hi = w / n_chunks;
    const int cbase = (int)(w - hi * n_chunks) * CC;
    const uint32_t t = (uint32_t)__ldg(heavy + 2 + hi);
    const int32_t s = __ldg(tile_start + t);
    const int32_t n = __ldg(tile_start + t + 1) - s;
    if (n < min_points) continue;  // left to the main grid (k_pool_fwd_narrow takes more)
    const uint32_t b = t / tiles_per_sample;
    const int v0 = (int)(t - b * tiles_per_sample) * kTileVoxels;
    const int32_t g0 = (int32_t)((int64_t)b * V) + v0;
    const int cmax = min(CC, C - cbase);
    const int n_rounds = (n + kHeavyChunk - 1) / kHeavyChunk;

    // index records, one point per thread < kHeavyChunk, two rounds deep in registers:
    //   stage A(k): ranks of round k            (rf, rb, previous point's rb, rd)
    //   stage B(k): depth[rd] of round k        (needs A(k))
    int32_t rf1 = 0, rb1 = -1, rp1 = -1, rd1 = 0, rf2 = 0, rb2 = -1, rp2 = -1, rd2 = 0;
    float d1 = 0.f;
    auto stage_a = [&](int k, int32_t& rf, int32_t& rb, int32_t& rp, int32_t& rd) {
      const int32_t i = k * kHeavyChunk + tid;
      rb = -1;
      if (tid < kHeavyChunk && i < n) {
        rf = __ldg(ranks_feat + s + i);
        rd = __ldg(ranks_depth + s + i);
        rb = __ldg(ranks_bev + s + i);
        rp = i ? __ldg(ranks_bev + s + i - 1) : -1;
      }
    };
    stage_a(0, rf1, rb1, rp1, rd1);
    if (n_rounds > 1) stage_a(1, rf2, rb2, rp2, rd2);
    if (rb1 >= 0) d1 = __ldg(depth + rd1);

    {  // clear the tile and both boundary tables
      float4* t4 = reinterpret_cast<float4*>(tile);
      for (int i = tid; i < CC * kRowPitch / 4; i += kHeavyThreads)
        t4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (tid < 128) bounds[tid] = 0;
    }
    __syncthreads();

    for (int k = 0; k < n_rounds; ++k) {
      const int cnt = min(kHeavyChunk, n - k * kHeavyChunk);
      int32_t* cstart = bounds + (k & 1) * 64;
      int32_t* cend = cstart + 32;
      // publish round k's records and the [start, end) of every voxel inside the round
      if (rb1 >= 0) {
        const int vox = rb1 - g0, voxp = rp1 - g0;
        off[tid] = (uint32_t)rf1 * (uint32_t)C;
        dep[tid] = d1;
        const bool first = (tid == 0) || (rb1 != rp1);
        if (first) cstart[vox] = tid;
        if (first && tid > 0) cend[voxp] = tid;
        if (tid == cnt - 1) cend[vox] = cnt;
      }
      // advance the register pipeline: B(k+1) and A(k+2) fly during this round's row copy
      rf1 = rf2; rb1 = rb2; rp1 = rp2; rd1 = rd2;
      d1 = 0.f;
      if (rb1 >= 0) d1 = __ldg(depth + rd1);
      rb2 = -1;
      if (k + 2 < n_rounds) stage_a(k + 2, rf2, rb2, rp2, rd2);
      // the other table is free now (last read in round k-1): clear it for round k+1
      if (tid >= 128 && tid < 192) bounds[((k + 1) & 1) * 64 + tid - 128] = 0;
      __syncthreads();

      // every feature row of the round in flight at once
#pragma unroll
      for (int i = 0; i < kHeavyChunk * kSegs / kHeavyThreads; ++i) {
        const int idx = tid + kHeavyThreads * i;
        const int r = idx / kSegs, seg = (idx % kSegs) * 4;
#ifndef VEON_FWD_X_HEAVY_NOCOPY   // tools only: elimination timing
        if (r < cnt && seg < cmax) cp_async_4(rows + r * CC + seg, feat + off[r] + cbase + seg);
#endif
      }
      cp_async_commit();
      cp_async_wait_all();
      __syncthreads();

      // fma chains: warp w owns voxels w, w+8, w+16, w+24; lanes = channels
#pragma unroll 1
      for (int v = warp; v < kTileVoxels; v += kHeavyThreads / 32) {
        const int a = cstart[v], e = cend[v];
        if (e <= a) continue;
        float acc[KCH];
#pragma unroll
        for (int c = 0; c < KCH; ++c) acc[c] = tile[(lane + 32 * c) * kRowPitch + v];
#ifndef VEON_FWD_X_HEAVY_NOFMA
#pragma unroll 4
        for (int j = a; j < e; ++j) {
          const float dj = dep[j];
#pragma unroll
          for (int c = 0; c < KCH; ++c) acc[c] = fmaf(widen(rows[j * CC + lane + 32 * c]), dj, acc[c]);
        }
#endif
#pragma unroll
        for (int c = 0; c < KCH; ++c) tile[(lane + 32 * c) * kRowPitch + v] = acc[c];
      }
      __syncthreads();
    }

    if constexpr (CLS) {  // one chunk holds every channel: lanes = voxels, classify from the tile
      if (warp == 0 && v0 + lane < V) {
        ClassMerge m;
        for (int q = 0; q < ca.Q; ++q) m.push(__ldg(ca.cls + q), tile[(2 + q) * kRowPitch + lane]);
        store_label(ca, b, (uint32_t)(v0 + lane),
                    m.label(tile[lane], tile[kRowPitch + lane], ca.free_label));
      }
    } else if constexpr (CL) {  // rows of the empty voxels are the tile's zeros
      for (int v = warp; v < kTileVoxels && v0 + v < V; v += kHeavyThreads / 32) {
        T* o = out + ((int64_t)g0 + v) * C + cbase;
        for (int c = lane; c < cmax; c += 32) st_stream(o + c, tile[c * kRowPitch + v]);
      }
    } else {  // write-out: thread (row = tid/8, q = tid%8) moves voxels 4q..4q+3 of channel row (+32j)
      const int q4 = (tid & 7) * 4;
      const bool fast = vec_ok && (v0 + kTileVoxels <= V);
      for (int c = tid >> 3; c < cmax; c += kHeavyThreads / 8) {
        T* o = out + ((int64_t)b * C + cbase + c) * V + v0 + q4;
        const float* trow = tile + c * kRowPitch + q4;
        if (fast) {
          st_stream4(o, make_float4(trow[0], trow[1], trow[2], trow[3]));
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (v0 + q4 + i < V) st_stream(o + i, trow[i]);
        }
      }
    }
    __syncthreads();
  }
  // join != 0 (always, when this grid was launched as a programmatic dependent): do not
  // COMPLETE before the grid it depends on has completed and flushed -- whatever is launched
  // next on the stream, a programmatic dependent or a graph node included, then sees the whole
  // volume (PTX: a dependent of a grid that triggers launch_dependents must execute
  // griddepcontrol.wait).
  if (join) pdl_wait();
}


// ---- fused pooling + 2x2x2 max-downsample, forward (SURVEY 8f-1) ------------------------
// VEON's neck reduces the pooled volume 8x right away (view_transformer_raw.py:549-553:
// rearrange to [..., (dz dh dw)] + torch.max(dim=-1).values).  Here the full-resolution volume is never written: a CTA
// takes one output row (b, z/2, y/2), pools its four input x-rows one after the other into a
// shared [c][X] tile -- points of a row are one contiguous slice of the sorted rank arrays,
// found through the per-voxel prefix `voxel_start` the preparation leaves in its workspace;
// rows staged by cp.async, rank-ordered fma chains as in k_pool_fwd_heavy -- and folds each
// into a running [c][X/2] maximum.  Sums are the same bits as the unfused kernel's and max is
// exact, so the result equals pool + that reduction bit for bit.  Forward only (inference path).
__device__ __forceinline__ float ds_max(float a, float b) { return (b > a || b != b) ? b : a; }
constexpr int kDsThreads = 256;
constexpr int kDsRound = 96;   // points staged per round (thread per point)

template <int KCH>
__global__ void __launch_bounds__(kDsThreads)
k_pool_ds_fwd(const float* __restrict__ depth, const float* __restrict__ feat,
              const int32_t* __restrict__ ranks_depth, const int32_t* __restrict__ ranks_feat,
              const int32_t* __restrict__ ranks_bev, const int32_t* __restrict__ voxel_start,
              uint32_t n_items, uint32_t n_chunks, int Z, int Y, int Xfull, int xsplit,
              int C, float* __restrict__ out) {
  constexpr int CC = 32 * KCH;
  constexpr int kSegs = CC / 4;
  const int X = Xfull / xsplit;              // voxels of the x-run one item covers
  const int Xp = (X + 3) / 4 * 4 + 4;        // pitch of the full-resolution row tile
  const int Xh = X / 2, Xhp = Xh + 1;        // pitch of the running maximum
  extern __shared__ __align__(16) float dsm[];
  float* rows = dsm;                                                // [kDsRound][CC]
  float* stage = rows + kDsRound * CC;                              // [CC][Xp]
  float* outb = stage + CC * Xp;                                    // [CC][Xhp]
  float* dep = outb + CC * Xhp;                                     // [kDsRound]
  uint32_t* off = reinterpret_cast<uint32_t*>(dep + kDsRound);      // [kDsRound]
  int32_t* bounds = reinterpret_cast<int32_t*>(off + kDsRound);     // [2][start Xp | end Xp]
  int32_t* rs = bounds + 4 * Xp;                                    // [4] first point of a row
  int32_t* rn = rs + 4;                                             // [4] points in the row
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Zh = Z / 2, Yh = Y / 2;
  const int64_t V = (int64_t)Z * Y * Xfull;

  struct Rec { int32_t rb, rp, rf, rd; float d; };
  struct Rnd { int sub, base; };
  auto first_round = [&]() -> Rnd {
    for (int q = 0; q < 4; ++q) if (rn[q] > 0) return Rnd{q, 0};
    return Rnd{4, 0};
  };
  auto next_round = [&](Rnd r) -> Rnd {
    if (r.base + kDsRound < rn[r.sub]) return Rnd{r.sub, r.base + kDsRound};
    for (int q = r.sub + 1; q < 4; ++q) if (rn[q] > 0) return Rnd{q, 0};
    return Rnd{4, 0};
  };
  auto stage_a = [&](Rnd r, Rec& c) {
    c.rb = -1;
    c.rp = -1;
    const int q = r.base + tid;
    if (tid < kDsRound && q < rn[r.sub]) {
      const int32_t i = rs[r.sub] + q;
      c.rb = __ldg(ranks_bev + i);
      c.rf = __ldg(ranks_feat + i);
      c.rd = __ldg(ranks_depth + i);
      if (q > 0) c.rp = __ldg(ranks_bev + i - 1);
    }
  };
  auto stage_b = [&](Rec& c) {
    c.d = 0.f;
    if (c.rb >= 0) c.d = __ldg(depth + c.rd);
  };

  for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const uint32_t piece = item / n_chunks, chunk = item - piece * n_chunks;
    const uint32_t cell = piece / (uint32_t)xsplit;
    const int x0 = (int)(piece - cell * (uint32_t)xsplit) * X;   // first input voxel of the run
    const int yo = (int)(cell % (uint32_t)Yh);
    const int zo = (int)((cell / (uint32_t)Yh) % (uint32_t)Zh);
    const int64_t b = cell / ((uint32_t)Yh * (uint32_t)Zh);
    const int cbase = (int)chunk * CC;
    __syncthreads();   // previous item fully written out
    if (tid < 4) {
      const int64_t g = b * V + ((int64_t)(2 * zo + (tid >> 1)) * Y + 2 * yo + (tid & 1)) * Xfull + x0;
      const int32_t s0 = __ldg(voxel_start + g);
      rs[tid] = s0;
      rn[tid] = __ldg(voxel_start + g + X) - s0;
    }
    for (int i = tid; i < 4 * Xp; i += kDsThreads) bounds[i] = 0;
    __syncthreads();

    Rnd cur = first_round();
    Rec rec;
    rec.rb = -1;
    if (cur.sub < 4) {
      stage_a(cur, rec);
      stage_b(rec);
    }
    int parity = 0;
    for (int sub = 0; sub < 4; ++sub) {
      if (rn[sub] == 0) {   // empty input row: contributes zeros
        for (int c = warp; c < CC; c += kDsThreads / 32)
          for (int xo = lane; xo < Xh; xo += 32)
            outb[c * Xhp + xo] = sub == 0 ? 0.f : ds_max(outb[c * Xhp + xo], 0.f);
        continue;
      }
      const int32_t g_row = (int32_t)(b * V + ((int64_t)(2 * zo + (sub >> 1)) * Y + 2 * yo + (sub & 1)) * Xfull + x0);
      {
        float4* s4 = reinterpret_cast<float4*>(stage);
        for (int i = tid; i < CC * Xp / 4; i += kDsThreads) s4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      while (cur.sub == sub) {
        const int cnt = min(kDsRound, rn[sub] - cur.base);
        int32_t* cstart = bounds + parity * 2 * Xp;
        int32_t* cend = cstart + Xp;
        if (rec.rb >= 0) {   // publish the round's records and voxel [start, end) ranges
          const int vox = rec.rb - g_row;
          off[tid] = ((uint32_t)rec.rf * (uint32_t)C + chunk * CC) * 4u;
          dep[tid] = rec.d;
          const bool starts = (tid == 0) || (rec.rb != rec.rp);
          if (starts) cstart[vox] = tid;
          if (tid > 0 && rec.rb != rec.rp) cend[rec.rp - g_row] = tid;
          if (tid == cnt - 1) cend[vox] = cnt;
        }
        const Rnd nx = next_round(cur);
        __syncthreads();
        {
          const char* fbase = reinterpret_cast<const char*>(feat);
#pragma unroll
          for (int i = 0; i < kDsRound * kSegs / kDsThreads; ++i) {
            const int idx = tid + kDsThreads * i;
            const int r = idx / kSegs, seg = (idx % kSegs) * 4;
            if (r < cnt) cp_async16(rows + r * CC + seg, fbase + off[r] + seg * 4);
          }
          cp_async_commit();
        }
        Rec nrec;
        nrec.rb = -1;
        if (nx.sub < 4) stage_a(nx, nrec);
        for (int i = tid; i < 2 * Xp; i += kDsThreads) bounds[(parity ^ 1) * 2 * Xp + i] = 0;
        cp_async_wait_all();
        __syncthreads();
        if (nx.sub < 4) stage_b(nrec);
        // fma chains: voxel block k (32 voxels) belongs to warp k % 8; lanes = channels
        for (int vb = warp * 32; vb < X; vb += kDsThreads) {
          const int vv = vb + lane;
          const int a_l = vv < X ? cstart[vv] : 0, e_l = vv < X ? cend[vv] : 0;
          uint32_t m = __ballot_sync(0xffffffffu, e_l > a_l);
          while (m) {
            const int v = __ffs(m) - 1;
            m &= m - 1;
            const int a = __shfl_sync(0xffffffffu, a_l, v), e = __shfl_sync(0xffffffffu, e_l, v);
            float* sp = stage + lane * Xp + vb + v;
            float acc[KCH];
#pragma unroll
            for (int c = 0; c < KCH; ++c) acc[c] = sp[32 * c * Xp];
#pragma unroll 4
            for (int j = a; j < e; ++j) {
              const float dj = dep[j];
#pragma unroll
              for (int c = 0; c < KCH; ++c) acc[c] = fmaf(rows[j * CC + lane + 32 * c], dj, acc[c]);
            }
#pragma unroll
            for (int c = 0; c < KCH; ++c) sp[32 * c * Xp] = acc[c];
          }
        }
        parity ^= 1;
        rec = nrec;
        cur = nx;
        __syncthreads();
      }
      // fold the finished row into the running maximum (pairs along x)
      // (warp w: channels w, w+8, ...; lanes along x -- the same element-to-thread map in
      //  every fold and in the write-out, so outb needs no barrier of its own)
      for (int c = warp; c < CC; c += kDsThreads / 32)
        for (int xo = lane; xo < Xh; xo += 32) {
          const float2 p2 = *reinterpret_cast<const float2*>(stage + c * Xp + 2 * xo);
          const float m2 = ds_max(p2.x, p2.y);
          outb[c * Xhp + xo] = sub == 0 ? m2 : ds_max(outb[c * Xhp + xo], m2);
        }
      __syncthreads();
    }
    // out[b, cbase + c, zo, yo, :]
    for (int c = warp; c < CC; c += kDsThreads / 32) {
      float* o = out + (((b * C + cbase + c) * Zh + zo) * Yh + yo) * (int64_t)(Xfull / 2) + x0 / 2;
      for (int xo = lane; xo < Xh; xo += 32) o[xo] = outb[c * Xhp + xo];
    }
  }
}

// ---- narrow rows (C <= 32): lane = voxel ---------------------------------------------------
// With few channels a lane-per-channel warp leaves lanes idle and pays one row-load latency
// per point (the logit-space lift pools Q + 2 = 20 channels over 4x the points of C2:
// 437 us for 410 MB).  Here a warp still owns a 32-voxel tile, but a LANE owns a voxel: it
// walks its own contiguous slice of the sorted points, two points per trip with all their
// loads (ranks, depth, the 16-byte pieces of both rows) in flight together, and accumulates
// every channel of its voxel in registers with the same fma(feat, depth, acc) chain in rank
// order, so the result is the same bits as k_pool_fwd's.  The write-out needs no transposition:
// for each channel plane the 32 lanes store one aligned 128-byte run (zeros for empty voxels).
// Segment bounds come from ranks_bev itself (head flags over the tile's points, 32 at a time).
// A lane walks two points per load latency, so this kernel keeps every tile below
// kNarrowHeavyMin points (at C3 density the plan's threshold of 96 would hand half of all
// points to the CTA-per-tile kernel: 252 us of a 437 us call); k_pool_fwd_heavy skips those.
constexpr int kNarrowWarps = 8;
constexpr int kNarrowHeavyMin = 512;
// Fused lift + classify (CLS): NP passes of 4*NV channels each over the tile's points; the
// class-merge state lives in registers between the passes (the merge is a scan over the prompt
// rows in order), so Q + 2 <= 96 channels need no more registers than 32 do.
// CL: channels-last output; a lane's voxel row is NV 16-byte stores and the warp's 32 rows are one
// contiguous 32 * C * 4-byte block.
// TF = bf16: a 4-channel piece is one 8-byte load, widened in registers.
template <int NV, bool CLS = false, int NP = 1, bool CL = false, typename T = float,
          typename TF = float>  // 4-channel pieces per pass: C = 4 * NV * NP
__global__ void __launch_bounds__(kNarrowWarps * 32, (NV <= 5) ? 3 : 2)
k_pool_fwd_narrow(const float* __restrict__ depth, const TF* __restrict__ feat,
                  const int32_t* __restrict__ ranks_depth, const int32_t* __restrict__ ranks_feat,
                  const int32_t* __restrict__ ranks_bev, const int32_t* __restrict__ tile_start,
                  const int32_t* __restrict__ heavy, uint32_t n_tiles, uint32_t tiles_per_sample,
                  int64_t V, T* __restrict__ out, uint32_t zero, int heavy_min, int join,
                  ClsArgs ca) {
  static_assert(CLS || NP == 1, "several passes only make sense when the sums are consumed here");
  constexpr int CP = 4 * NV;        // channels per pass
  constexpr int C = CP * NP;        // row length
  __shared__ int32_t seg_s[kNarrowWarps][32];
  pdl_launch_dependents();  // the heavy-tile grid may be queued behind this one
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t* seg = seg_s[warp];
  uint32_t heads[3] = {0u, 0u, 0u};   // CLS: bit q = prompt row q starts a class (Q <= 94)
  if constexpr (CLS) {
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      const int q = 32 * w + lane;
      const bool h = q < ca.Q && (q == 0 || __ldg(ca.cls + q) != __ldg(ca.cls + q - 1));
      heads[w] = __ballot_sync(0xffffffffu, h);
    }
  }
  const int32_t heavy_thr = heavy ? max(__ldg(heavy + 1), heavy_min) : 0x7fffffff;
  const uint32_t TW = gridDim.x * kNarrowWarps;
  // The per-tile chain (bounds -> ranks_bev -> segment table -> ranks -> rows -> stores) is a
  // string of dependent load latencies, so the head of the chain runs ahead: bounds are read
  // two tiles early, the first 32 ranks_bev of a tile one tile early.
  const uint32_t first = blockIdx.x * kNarrowWarps + warp;
  int32_t ns = 0, ne = 0, as = 0, ae = 0, nrb = 0;  // next tile, the one after; next tile's ranks
  if (first < n_tiles) {
    ns = __ldg(tile_start + first);
    ne = __ldg(tile_start + first + 1);
    if (ns + lane < ne) nrb = __ldg(ranks_bev + ns + lane);
  }
  if (first + TW < n_tiles) {
    as = __ldg(tile_start + first + TW);
    ae = __ldg(tile_start + first + TW + 1);
  }
  for (uint32_t t = first; t < n_tiles; t += TW) {
    const int32_t s0 = ns, e0 = ne, rb_first = nrb;
    ns = as;
    ne = ae;
    as = ae = 0;
    if (t + 2 * TW < n_tiles) {
      as = __ldg(tile_start + t + 2 * TW);
      ae = __ldg(tile_start + t + 2 * TW + 1);
    }
    nrb = (ns + lane < ne) ? __ldg(ranks_bev + ns + lane) : 0;
    if (e0 - s0 >= heavy_thr) continue;  // k_pool_fwd_heavy's
    const uint32_t b = t / tiles_per_sample;
    const uint32_t v0 = (t - b * tiles_per_sample) * kTileVoxels;
    const int32_t g0 = (int32_t)((int64_t)b * V) + (int32_t)v0;  // rank of the tile's first voxel
    int32_t st = -1, en = 0;   // this lane's voxel: its points are [st, en)
    if (e0 > s0) {
      // first point of every occupied voxel
      seg[lane] = -1;
      __syncwarp();
      int32_t prev;
      {
        const int32_t vox = (s0 + lane < e0) ? rb_first - g0 : -2;
        const int32_t up = __shfl_up_sync(0xffffffffu, vox, 1);
        if (s0 + lane < e0 && (lane == 0 || vox != up) && (uint32_t)vox < 32u) seg[vox] = s0 + lane;
        prev = __shfl_sync(0xffffffffu, vox, 31);
      }
      for (int32_t p0 = s0 + 32; p0 < e0; p0 += 128) {  // four rounds' loads in flight together
        int32_t vx[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int32_t i = p0 + 32 * r + lane;
          vx[r] = (i < e0) ? __ldg(ranks_bev + i) - g0 : -2;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int32_t i = p0 + 32 * r + lane;
          int32_t up = __shfl_up_sync(0xffffffffu, vx[r], 1);
          if (lane == 0) up = prev;
          if (i < e0 && vx[r] != up && (uint32_t)vx[r] < 32u) seg[vx[r]] = i;
          prev = __shfl_sync(0xffffffffu, vx[r], 31);
        }
      }
      __syncwarp();
      st = seg[lane];
      const uint32_t occ = __ballot_sync(0xffffffffu, st >= 0);
      const uint32_t higher = (lane == 31) ? 0u : (occ >> (lane + 1));
      const int nxt = higher ? lane + __ffs(higher) : 0;
      const int32_t nst = __shfl_sync(0xffffffffu, st, nxt);
      en = higher ? nst : e0;
      __syncwarp();  // seg is rewritten for the next tile
    }
    // CLS: class-wise max over the prompt rows, first-index arg-max over the classes -- the
    // branch-free form of ClassMerge -- carried from pass to pass
    float best = -INFINITY, cur = -INFINITY, gate0 = 0.f, gate1 = 0.f;
    int best_q = 0, cur_q = 0;
    bool bad = false;
#pragma unroll 1
    for (int pass = 0; pass < NP; ++pass) {
      float acc[CP];
#pragma unroll
      for (int c = 0; c < CP; ++c) acc[c] = 0.f;
      if (st >= 0) {
        const TF* fbase = feat + pass * CP;
        int32_t i = st;
        bool two = i + 1 < en;
        int32_t r0 = __ldg(ranks_depth + i), f0 = __ldg(ranks_feat + i);
        int32_t r1 = two ? __ldg(ranks_depth + i + 1) : r0;
        int32_t f1 = two ? __ldg(ranks_feat + i + 1) : f0;
        while (true) {
          // A trip always runs both fma chains (no branch for the scheduler to sink the second
          // point's loads into); a missing second point is (+0) * (-0): acc + (-0) == acc bit for
          // bit, whatever acc is.
          const float d0 = __ldg(depth + r0), d1 = two ? __ldg(depth + r1) : -0.f;
          const TF* row0 = fbase + (int64_t)f0 * C;
          const TF* row1 = fbase + (int64_t)f1 * C;
          float4 a[NV], q[NV];
#pragma unroll
          for (int k = 0; k < NV; ++k) a[k] = ldg_widen4(row0 + 4 * k);
#pragma unroll
          for (int k = 0; k < NV; ++k) q[k] = two ? ldg_widen4(row1 + 4 * k) : make_float4(0.f, 0.f, 0.f, 0.f);
          // `zero` is a kernel argument that is always 0: making the first depth value depend
          // on every piece of the second row keeps the assembler from re-using the first row's
          // registers for the second row's loads (it otherwise issues them only after the first
          // chain has consumed its operands: two exposed latencies per trip instead of one).
          uint32_t tie = 0;
#pragma unroll
          for (int k = 0; k < NV; ++k) tie |= __float_as_uint(q[k].x);
          const float d0t = __uint_as_float(__float_as_uint(d0) | (tie & zero));
          i += 2;  // the next trip's ranks travel with this trip's rows
          const bool more = i < en;
          if (more) {
            two = i + 1 < en;
            r0 = __ldg(ranks_depth + i);
            f0 = __ldg(ranks_feat + i);
            r1 = two ? __ldg(ranks_depth + i + 1) : r0;
            f1 = two ? __ldg(ranks_feat + i + 1) : f0;
          }
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            acc[4 * k + 0] = fmaf(a[k].x, d0t, acc[4 * k + 0]);
            acc[4 * k + 1] = fmaf(a[k].y, d0t, acc[4 * k + 1]);
            acc[4 * k + 2] = fmaf(a[k].z, d0t, acc[4 * k + 2]);
            acc[4 * k + 3] = fmaf(a[k].w, d0t, acc[4 * k + 3]);
          }
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            acc[4 * k + 0] = fmaf(q[k].x, d1, acc[4 * k + 0]);
            acc[4 * k + 1] = fmaf(q[k].y, d1, acc[4 * k + 1]);
            acc[4 * k + 2] = fmaf(q[k].z, d1, acc[4 * k + 2]);
            acc[4 * k + 3] = fmaf(q[k].w, d1, acc[4 * k + 3]);
          }
          if (!more) break;
        }
      }
      if constexpr (CLS) {
        // rows are [gate 0, gate 1, logit 0 .. Q-1, padding]: channel c of pass p is prompt
        // p * CP + c - 2; padding enters as -inf and changes nothing
        if (pass == 0) { gate0 = acc[0]; gate1 = acc[1]; }
#pragma unroll
        for (int c = 0; c < CP; ++c) {
          const int q = pass * CP + c - 2;
          const bool real = q >= 0 && q < ca.Q;
          const float logit = real ? acc[c] : -INFINITY;
          bad |= !(logit < INFINITY);
          const uint32_t word = q < 32 ? heads[0] : (q < 64 ? heads[1] : heads[2]);
          const bool head = real && ((word >> (q & 31)) & 1u);
          const bool take = head && (cur > best);
          best = take ? cur : best;
          best_q = take ? cur_q : best_q;
          cur = head ? logit : fmaxf(cur, logit);
          cur_q = head ? q : cur_q;
        }
      } else if constexpr (CL) {
        T* o = out + ((int64_t)g0 + lane) * C;
#pragma unroll
        for (int k = 0; k < NV; ++k)
          st_stream4(o + 4 * k, make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]));
      } else {
        T* o = out + (int64_t)b * C * V + v0 + lane;
#pragma unroll
        for (int c = 0; c < CP; ++c) st_stream(o + (int64_t)c * V, acc[c]);
      }
    }
    if constexpr (CLS) {
      if (cur > best) { best = cur; best_q = cur_q; }
      bad |= (best == -INFINITY);
      const float mx = fmaxf(gate0, gate1);
      const float e0g = expf(gate0 - mx), e1g = expf(gate1 - mx);
      const bool occupied = (e0g / (e0g + e1g)) > 0.5f;
      store_label(ca, b, v0 + lane, (occupied && !bad) ? __ldg(ca.cls + best_q) : ca.free_label);
    }
  }
  if (join) pdl_wait();   // launched behind the heavy grid: complete after it (see k_pool_fwd_heavy)
}


// ---- launchers ---------------------------------------------------------------------------------
template <int KCH, bool CLS = false, bool CL = false, typename T = float, typename TF = float>
static int heavy_config(size_t& smem, int& ctas_per_sm) {
  constexpr int CC = 32 * KCH;
  smem = sizeof(TF) * kHeavyChunk * CC + sizeof(float) * (CC * kRowPitch + 2 * kHeavyChunk + 128);
  static int cached[kMaxDevices] = {};
  const int dev = current_device();
  if (cached[dev] == 0) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_pool_fwd_heavy<KCH, CLS, CL, T, TF>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int n = 0;
    VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_pool_fwd_heavy<KCH, CLS, CL, T, TF>,
                                                                kHeavyThreads, smem));
    cached[dev] = n < 1 ? 1 : (n > 8 ? 8 : n);
  }
  ctas_per_sm = cached[dev];
  return 0;
}

// the heavy-tile grid; pdl: queued as a programmatic dependent of the previous launch (joins it)
template <int KCH, bool CLS = false, bool CL = false, typename T = float, typename TF = float>
static int launch_heavy(const float* depth, const TF* feat, const int32_t* rd, const int32_t* rf,
                        const int32_t* rb, const int32_t* tile_start, const int32_t* heavy,
                        int64_t heavy_ints, int B, int C, int64_t V, T* out, bool pdl,
                        int min_points, cudaStream_t stream, ClsArgs ca = ClsArgs()) {
  constexpr int CC = 32 * KCH;
  size_t smem;
  int per_sm;
  int rc = heavy_config<KCH, CLS, CL, T, TF>(smem, per_sm);
  if (rc) return rc;
  const int64_t tps = ceil_div64(V, kTileVoxels);
  const int n_chunks = (C + CC - 1) / CC;
  const int vec_ok = ((V & 3) == 0) && (((uintptr_t)out & (4 * sizeof(T) - 1)) == 0);
  const int heavy_cap = (int)(heavy_ints - 2);
  int64_t blocks = (int64_t)heavy_cap * n_chunks;
  if (blocks > (int64_t)per_sm * sm_count()) blocks = (int64_t)per_sm * sm_count();
  if (blocks <= 0) return 0;
  if (pdl) {
    VEON_CUDA_TRY(launch_pdl(k_pool_fwd_heavy<KCH, CLS, CL, T, TF>, dim3((unsigned)blocks), dim3(kHeavyThreads),
                             smem, stream, depth, feat, rd, rf, rb, tile_start, heavy, heavy_cap,
                             (uint32_t)tps, V, C, (uint32_t)n_chunks, vec_ok, out, 1, min_points, ca));
  } else {
    k_pool_fwd_heavy<KCH, CLS, CL, T, TF><<<(unsigned)blocks, kHeavyThreads, smem, stream>>>(
        depth, feat, rd, rf, rb, tile_start, heavy, heavy_cap, (uint32_t)tps, V, C,
        (uint32_t)n_chunks, vec_ok, out, 0, min_points, ca);
  }
  VEON_LAUNCH_CHECK();
  return 0;
}

int launch_heavy_behind(const float* depth, const float* feat, const int32_t* rd,
                        const int32_t* rf, const int32_t* rb, const int32_t* tile_start,
                        const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                        float* out, int min_points, cudaStream_t stream) {
  if (!heavy || heavy_ints < 2 || (C & 3) != 0 || ((uintptr_t)feat & 15) != 0)
    return VEON_E_BADARG;
  return C <= 32 ? launch_heavy<1>(depth, feat, rd, rf, rb, tile_start, heavy, heavy_ints, B, C, V,
                                   out, true, min_points, stream)
                 : launch_heavy<2>(depth, feat, rd, rf, rb, tile_start, heavy, heavy_ints, B, C, V,
                                   out, true, min_points, stream);
}

// general route: k_pool_fwd over every (tile, channel chunk), the heavy tiles queued behind it
template <int KCH, bool FULLC, bool LOOPC, bool CL, typename T, typename TF>
static int launch_fwd_impl(const float* depth, const TF* feat, const int32_t* rd,
                           const int32_t* rf, const int32_t* rb, const int32_t* tile_start,
                           const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                           bool feat_rows_fit_32bit, T* out, cudaStream_t stream) {
  constexpr int CC = 32 * KCH;
  constexpr int kExtInts = LOOPC ? ((kHeavyDefaultThreshold + 31) / 32 - 1) * 128 : 0;
  const size_t smem = sizeof(float) * kFwdWarps *
                      ((CL ? kTileVoxels * (CC + 4) : CC * kRowPitch) + kRingSlots * kSlotInts + kExtInts);
  static int ctas_per_sm[kMaxDevices] = {};
  const int dev = current_device();
  if (ctas_per_sm[dev] == 0) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_pool_fwd<KCH, FULLC, LOOPC, CL, T, TF>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int n = 0;
    VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_pool_fwd<KCH, FULLC, LOOPC, CL, T, TF>,
                                                                kFwdWarps * 32, smem));
    ctas_per_sm[dev] = n < 1 ? 1 : n;
  }
  const int64_t tps = ceil_div64(V, kTileVoxels), n_tiles = (int64_t)B * tps;
  const int n_chunks = (C + CC - 1) / CC;
  if (n_tiles * n_chunks > 0x7fffffffLL || (int64_t)B * V > 0x7fffffffLL) return VEON_E_RANGE;
  if (!feat_rows_fit_32bit) return VEON_E_RANGE;   // the gather uses 32-bit byte offsets
  // 4-element (16-byte float, 8-byte bf16) stores: channel planes of 4-voxel pieces
  // (channels-first) or rows of 4-channel pieces (channels-last)
  const int vec_ok = (((CL ? C : V) & 3) == 0) && (((uintptr_t)out & (4 * sizeof(T) - 1)) == 0);
  const int64_t n_items = LOOPC ? n_tiles : n_tiles * n_chunks;   // LOOPC: chunks looped per tile
  int64_t blocks = ceil_div64(n_items, kFwdWarps);
  const int64_t resident = (int64_t)ctas_per_sm[dev] * sm_count();  // persistent grid
  if (blocks > resident) blocks = resident;
  // the heavy-tile kernel stages feature rows with 4-element (16- or 8-byte) copies
  if (heavy && ((C & 3) != 0 || ((uintptr_t)feat & (4 * sizeof(TF) - 1)) != 0)) heavy = nullptr;
  k_pool_fwd<KCH, FULLC, LOOPC, CL, T, TF><<<(unsigned)blocks, kFwdWarps * 32, smem, stream>>>(
      depth, feat, rd, rf, rb, tile_start, heavy, (uint32_t)n_items, (uint32_t)tps,
      V, C, (uint32_t)(LOOPC ? 1 : n_chunks), vec_ok, out, (uint32_t)n_chunks);
  VEON_LAUNCH_CHECK();
  // Heavy-tile CTAs behind the main grid (both trigger launch_dependents at their first
  // instruction): they fill the SMs as the persistent CTAs finish one by one, and join the main
  // grid before they complete.
#ifndef VEON_FWD_X_NOHEAVY
  if (heavy)
    return launch_heavy<(KCH > 2 ? 2 : KCH), false, CL, T, TF>(depth, feat, rd, rf, rb, tile_start, heavy, heavy_ints,
                                             B, C, V, out, true, 0, stream);
#endif
  return 0;
}

template <int KCH, bool CL, typename T, typename TF>
static int launch_fwd(const float* depth, const TF* feat, const int32_t* rd,
                      const int32_t* rf, const int32_t* rb, const int32_t* tile_start,
                      const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                      bool feat_rows_fit_32bit, T* out, cudaStream_t stream) {
  // rows of several chunks: one item per tile (needs the heavy list: it bounds a tile's points)
#ifndef VEON_FWD_X_NOLOOPC
  const bool loopc =
      heavy && C > 32 * KCH && (C & 3) == 0 && ((uintptr_t)feat & (4 * sizeof(TF) - 1)) == 0;
#else
  const bool loopc = false;
#endif
#define VEON_FWD_GO(FULLC_, LOOPC_)                                                            \
  return launch_fwd_impl<KCH, FULLC_, LOOPC_, CL, T, TF>(depth, feat, rd, rf, rb, tile_start, heavy,      \
                                              heavy_ints, B, C, V, feat_rows_fit_32bit, out, stream)
  if (C % (32 * KCH) == 0) {
    if (loopc) VEON_FWD_GO(true, true);
    VEON_FWD_GO(true, false);
  }
  if (loopc) VEON_FWD_GO(false, true);
  VEON_FWD_GO(false, false);
#undef VEON_FWD_GO
}

// narrow rows: the heavy tiles (from kNarrowHeavyMin points) first, as a normal launch (a heavy
// CTA works ~100 us on one 1 000-point tile at C3 density: behind the persistent main grid the
// two nearly serialise, 344 vs 295 us); k_pool_fwd_narrow moves in beside it as its programmatic
// dependent and joins it at the end
template <int NV, bool CLS = false, int NP = 1, bool CL = false, typename T = float,
          typename TF = float>
static int launch_fwd_narrow(const float* depth, const TF* feat, const int32_t* rd,
                             const int32_t* rf, const int32_t* rb, const int32_t* tile_start,
                             const int32_t* heavy, int64_t heavy_ints, int B, int64_t V,
                             T* out, cudaStream_t stream, ClsArgs ca = ClsArgs()) {
  constexpr int C = 4 * NV * NP;
  constexpr int KCH = (C + 31) / 32;   // the heavy CTA holds every channel of its tile
  const int64_t tps = V / kTileVoxels, n_tiles = (int64_t)B * tps;
  static int ctas_per_sm[kMaxDevices] = {};
  const int dev = current_device();
  if (ctas_per_sm[dev] == 0) {
    int n = 0;
    VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_pool_fwd_narrow<NV, CLS, NP, CL, T, TF>,
                                                                kNarrowWarps * 32, 0));
    ctas_per_sm[dev] = n < 1 ? 1 : n;
  }
  int64_t blocks = ceil_div64(n_tiles, kNarrowWarps);
  if (blocks > (int64_t)ctas_per_sm[dev] * sm_count()) blocks = (int64_t)ctas_per_sm[dev] * sm_count();
  int rc = launch_heavy<KCH, CLS, CL, T, TF>(depth, feat, rd, rf, rb, tile_start, heavy, heavy_ints, B, C, V,
                                  out, false, kNarrowHeavyMin, stream, ca);
  if (rc) return rc;
  VEON_CUDA_TRY(launch_pdl(k_pool_fwd_narrow<NV, CLS, NP, CL, T, TF>, dim3((unsigned)blocks),
                           dim3(kNarrowWarps * 32), 0, stream, depth, feat, rd, rf, rb, tile_start,
                           heavy, (uint32_t)n_tiles, (uint32_t)tps, V, out, 0u, kNarrowHeavyMin, 1,
                           ca));
  VEON_LAUNCH_CHECK();
  return 0;
}

}  // namespace veon

using namespace veon;

// Not part of the ABI in include/veon_lift.h: lets tools/fwd_check.py push wide rows through the
// streaming kernel for its parity sweep and timing comparison.
extern "C" void veon_internal_fwd_stream_force(int on) { stream_force = on != 0; }

extern "C" size_t veon_bev_pool_v2_fwd_workspace_bytes(int B, int C, int64_t V) {
  if (B <= 0 || C <= 0 || V <= 0) return 0;
  // the ring of compact rows (a few slots per SM; only their occupied prefix is ever touched,
  // so the part that lives in L2 is a fraction of this)
  return fwd_stream_workspace_bytes(C);
}

// All planar entry points: out is [B,C,Z,Y,X], or [B,Z,Y,X,C] with CL (the same kernels with a
// row write-out: same sums, same bits, another layout), of float or bf16 elements T, from feature
// rows of float or bf16 elements TF.  Routes in order: narrow rows, the streaming kernel
// (channels-first float volumes from float rows only; needs tile_occ and a workspace), the general
// kernel.
template <bool CL, typename T, typename TF = float>
static int fwd_planar(const float* depth, const TF* feat, const int32_t* ranks_depth,
                      const int32_t* ranks_feat, const int32_t* ranks_bev,
                      const int32_t* tile_start, const uint32_t* tile_occ,
                      const int32_t* tile_heavy, int64_t tile_heavy_ints, int B, int C, int64_t V,
                      int64_t n_feat_rows, T* out, void* workspace, size_t workspace_bytes,
                      cudaStream_t stream) {
  if (!depth || !feat || !ranks_depth || !ranks_feat || !ranks_bev || !tile_start || !out ||
      B <= 0 || C <= 0 || V <= 0 || n_feat_rows <= 0 || (tile_heavy && tile_heavy_ints < 2))
    return VEON_E_BADARG;
  // the gather addresses feature rows with 32-bit BYTE offsets; the ring header packs
  // sample<<16 | chunk
  const bool fit32 = n_feat_rows * (int64_t)C <= 0x3fffffffLL && B < 65536 &&
                     (int64_t)C <= 65535LL * 32;
  {  // narrow rows: lane-per-voxel kernel.  Without a heavy list a single lane would walk
     // arbitrarily long voxels; rank arithmetic is exact only while B*V <= 2^24
    const bool ok = C <= 32 && (C & 3) == 0 && tile_heavy && fit32 && V % kTileVoxels == 0 &&
                    (int64_t)B * V <= (1 << 24) &&
                    ((uintptr_t)feat & (4 * sizeof(TF) - 1)) == 0 &&
                    ((uintptr_t)out & (4 * sizeof(T) - 1)) == 0;
    if (ok) {
#define VEON_NARROW_CASE(NV_) case NV_: return launch_fwd_narrow<NV_, false, 1, CL, T, TF>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start, tile_heavy, tile_heavy_ints, B, V, out, stream);
      switch (C / 4) {
        VEON_NARROW_CASE(1) VEON_NARROW_CASE(2) VEON_NARROW_CASE(3) VEON_NARROW_CASE(4)
        VEON_NARROW_CASE(5) VEON_NARROW_CASE(6) VEON_NARROW_CASE(7) VEON_NARROW_CASE(8)
        default: break;
      }
#undef VEON_NARROW_CASE
    }
  }
  // aligned volumes, whole 64-channel chunks: the two-role streaming kernel.  It has no bf16-row
  // form: where it would run on float rows, bf16 rows are refused (VEON_E_UNSUPPORTED), and the
  // caller widens them into a fresh -- aligned -- float copy and calls the float entry.
  if constexpr (!CL && std::is_same<T, float>::value && !std::is_same<TF, float>::value) {
    if (workspace && tile_occ && tile_heavy &&
        fwd_stream_supported(B, C, V, out, out, n_feat_rows))
      return VEON_E_UNSUPPORTED;
  }
  if constexpr (!CL && std::is_same<T, float>::value && std::is_same<TF, float>::value) {
    if (workspace && tile_occ && tile_heavy &&
        fwd_stream_supported(B, C, V, feat, out, n_feat_rows)) {
      const int rc = launch_fwd_stream(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                                       tile_start, tile_occ, tile_heavy, tile_heavy_ints, B, C, V,
                                       out, workspace, workspace_bytes, stream);
      if (rc != VEON_E_UNSUPPORTED && rc != VEON_E_WORKSPACE) return rc;
    }
  }
  if (C <= 32)
    return launch_fwd<1, CL, T, TF>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start,
                             tile_heavy, tile_heavy_ints, B, C, V, fit32, out, stream);
  return launch_fwd<2, CL, T, TF>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start,
                           tile_heavy, tile_heavy_ints, B, C, V, fit32, out, stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar(const float* depth, const float* feat,
                                           const int32_t* ranks_depth,
                                           const int32_t* ranks_feat,
                                           const int32_t* ranks_bev,
                                           const int32_t* tile_start,
                                           const int32_t* tile_istart,
                                           const uint32_t* tile_occ,
                                           const int32_t* tile_heavy, int64_t tile_heavy_ints,
                                           int B, int C, int64_t V, int64_t n_feat_rows,
                                           float* out, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  return fwd_planar<false>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start, tile_occ,
                           tile_heavy, tile_heavy_ints, B, C, V, n_feat_rows, out, workspace,
                           workspace_bytes, (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar_cl(const float* depth, const float* feat,
                                              const int32_t* ranks_depth,
                                              const int32_t* ranks_feat,
                                              const int32_t* ranks_bev,
                                              const int32_t* tile_start,
                                              const int32_t* tile_heavy, int64_t tile_heavy_ints,
                                              int B, int C, int64_t V, int64_t n_feat_rows,
                                              float* out, void* stream) {
  return fwd_planar<true>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start, nullptr,
                          tile_heavy, tile_heavy_ints, B, C, V, n_feat_rows, out, nullptr, 0,
                          (cudaStream_t)stream);
}

// bfloat16 volumes: the same kernels with a bf16 write-out (float sums, one rounding per element
// at the store).  The channels-first one never takes the streaming kernel, so it needs no
// workspace; it accepts the float twin's arguments all the same.
extern "C" int veon_bev_pool_v2_fwd_planar_bf16(const float* depth, const float* feat,
                                                const int32_t* ranks_depth,
                                                const int32_t* ranks_feat,
                                                const int32_t* ranks_bev,
                                                const int32_t* tile_start,
                                                const int32_t* tile_istart,
                                                const uint32_t* tile_occ,
                                                const int32_t* tile_heavy, int64_t tile_heavy_ints,
                                                int B, int C, int64_t V, int64_t n_feat_rows,
                                                uint16_t* out, void* workspace,
                                                size_t workspace_bytes, void* stream) {
  return fwd_planar<false>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start, tile_occ,
                           tile_heavy, tile_heavy_ints, B, C, V, n_feat_rows,
                           reinterpret_cast<bf16*>(out), workspace, workspace_bytes,
                           (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar_cl_bf16(const float* depth, const float* feat,
                                                   const int32_t* ranks_depth,
                                                   const int32_t* ranks_feat,
                                                   const int32_t* ranks_bev,
                                                   const int32_t* tile_start,
                                                   const int32_t* tile_heavy,
                                                   int64_t tile_heavy_ints, int B, int C, int64_t V,
                                                   int64_t n_feat_rows, uint16_t* out,
                                                   void* stream) {
  return fwd_planar<true>(depth, feat, ranks_depth, ranks_feat, ranks_bev, tile_start, nullptr,
                          tile_heavy, tile_heavy_ints, B, C, V, n_feat_rows,
                          reinterpret_cast<bf16*>(out), nullptr, 0, (cudaStream_t)stream);
}

// bfloat16 feature rows [n_feat_rows, C]: the same kernels reading 2-byte channels, widened exactly,
// so every volume is the bits of the float twin on the widened rows.  Arguments, checks and error
// codes are the twins'; the channels-first float-volume entry returns VEON_E_UNSUPPORTED where its
// twin would take the streaming kernel (see fwd_planar).
extern "C" int veon_bev_pool_v2_fwd_planar_bf16feat(
    const float* depth, const uint16_t* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev, const int32_t* tile_start,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* tile_heavy,
    int64_t tile_heavy_ints, int B, int C, int64_t V, int64_t n_feat_rows, float* out,
    void* workspace, size_t workspace_bytes, void* stream) {
  return fwd_planar<false>(depth, reinterpret_cast<const bf16*>(feat), ranks_depth, ranks_feat,
                           ranks_bev, tile_start, tile_occ, tile_heavy, tile_heavy_ints, B, C, V,
                           n_feat_rows, out, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar_bf16_bf16feat(
    const float* depth, const uint16_t* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev, const int32_t* tile_start,
    const int32_t* tile_istart, const uint32_t* tile_occ, const int32_t* tile_heavy,
    int64_t tile_heavy_ints, int B, int C, int64_t V, int64_t n_feat_rows, uint16_t* out,
    void* workspace, size_t workspace_bytes, void* stream) {
  return fwd_planar<false>(depth, reinterpret_cast<const bf16*>(feat), ranks_depth, ranks_feat,
                           ranks_bev, tile_start, tile_occ, tile_heavy, tile_heavy_ints, B, C, V,
                           n_feat_rows, reinterpret_cast<bf16*>(out), workspace, workspace_bytes,
                           (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar_cl_bf16feat(
    const float* depth, const uint16_t* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev, const int32_t* tile_start,
    const int32_t* tile_heavy, int64_t tile_heavy_ints, int B, int C, int64_t V,
    int64_t n_feat_rows, float* out, void* stream) {
  return fwd_planar<true>(depth, reinterpret_cast<const bf16*>(feat), ranks_depth, ranks_feat,
                          ranks_bev, tile_start, nullptr, tile_heavy, tile_heavy_ints, B, C, V,
                          n_feat_rows, out, nullptr, 0, (cudaStream_t)stream);
}

extern "C" int veon_bev_pool_v2_fwd_planar_cl_bf16_bf16feat(
    const float* depth, const uint16_t* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev, const int32_t* tile_start,
    const int32_t* tile_heavy, int64_t tile_heavy_ints, int B, int C, int64_t V,
    int64_t n_feat_rows, uint16_t* out, void* stream) {
  return fwd_planar<true>(depth, reinterpret_cast<const bf16*>(feat), ranks_depth, ranks_feat,
                          ranks_bev, tile_start, nullptr, tile_heavy, tile_heavy_ints, B, C, V,
                          n_feat_rows, reinterpret_cast<bf16*>(out), nullptr, 0,
                          (cudaStream_t)stream);
}

// Fused lift + classify: pools the [gate 0, gate 1, logit 0..Q-1, pad] rows and ends every tile
// as 32 labels -- the pooled logit volume is never written (SURVEY 8f-4).
extern "C" int veon_lift_classify_fwd(const float* depth, const float* pix,
                                      const int32_t* ranks_depth, const int32_t* ranks_feat,
                                      const int32_t* ranks_bev, const int32_t* tile_start,
                                      const int32_t* tile_heavy, int64_t tile_heavy_ints, int B,
                                      int C, int Q, int Z, int Y, int X, int64_t n_pix_rows,
                                      const int32_t* class_of_prompt, int free_label,
                                      uint8_t* labels, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!depth || !pix || !ranks_depth || !ranks_feat || !ranks_bev || !tile_start || !tile_heavy ||
      tile_heavy_ints < 2 || !class_of_prompt || !labels || B <= 0 || C <= 0 || Q <= 0 ||
      Z <= 0 || Y <= 0 || X <= 0 || n_pix_rows <= 0)
    return VEON_E_BADARG;
  const int64_t V = (int64_t)Z * Y * X;
  if ((C & 3) != 0 || Q + 2 > C || C > 96 || Q > 94 || V % kTileVoxels != 0 ||
      ((uintptr_t)pix & 15) != 0)
    return VEON_E_UNSUPPORTED;
  // 32-bit row offsets; rank arithmetic is exact only while B*V <= 2^24
  if (n_pix_rows * (int64_t)C > 0x3fffffffLL || B >= 65536 || (int64_t)B * V > (1 << 24))
    return VEON_E_RANGE;
  ClsArgs ca;
  ca.cls = class_of_prompt; ca.labels = labels; ca.Q = Q; ca.X = X; ca.Y = Y; ca.Z = Z;
  ca.free_label = free_label;
  // Cp = 4 * NV * NP: one pass up to 32 channels, two up to 64, three up to 96
#define VEON_CLS_CASE(NV_, NP_)                                                                   \
  if (C == 4 * NV_ * NP_)                                                                         \
    return launch_fwd_narrow<NV_, true, NP_>(depth, pix, ranks_depth, ranks_feat, ranks_bev,      \
                                             tile_start, tile_heavy, tile_heavy_ints, B, V,       \
                                             (float*)nullptr, stream, ca);
  if (C <= 32) {
    VEON_CLS_CASE(1, 1) VEON_CLS_CASE(2, 1) VEON_CLS_CASE(3, 1) VEON_CLS_CASE(4, 1)
    VEON_CLS_CASE(5, 1) VEON_CLS_CASE(6, 1) VEON_CLS_CASE(7, 1) VEON_CLS_CASE(8, 1)
  } else if (C <= 64) {
    VEON_CLS_CASE(5, 2) VEON_CLS_CASE(6, 2) VEON_CLS_CASE(7, 2) VEON_CLS_CASE(8, 2)
  } else {
    VEON_CLS_CASE(6, 3) VEON_CLS_CASE(7, 3) VEON_CLS_CASE(8, 3)
  }
#undef VEON_CLS_CASE
  return VEON_E_UNSUPPORTED;
}

extern "C" int veon_bev_pool_v2_ds_fwd(const float* depth, const float* feat,
                                       const int32_t* ranks_depth, const int32_t* ranks_feat,
                                       const int32_t* ranks_bev, const int32_t* voxel_start,
                                       int B, int C, int Z, int Y, int X, int64_t n_feat_rows,
                                       float* out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!depth || !feat || !ranks_depth || !ranks_feat || !ranks_bev || !voxel_start || !out ||
      B <= 0 || C <= 0 || Z <= 0 || Y <= 0 || X <= 0 || n_feat_rows <= 0)
    return VEON_E_BADARG;
  constexpr int KCH = 2, CC = 64;
  // even grid, whole 64-channel chunks, 16-byte feature rows, exact float32 voxel ranks
  if ((Z | Y | X) & 1 || C % CC != 0 || ((uintptr_t)feat & 15) != 0) return VEON_E_UNSUPPORTED;
  const int64_t V = (int64_t)Z * Y * X;
  if ((int64_t)B * V >= (1 << 24) || n_feat_rows * (int64_t)C > 0x3fffffffLL) return VEON_E_RANGE;
  const int xsplit = 1;   // (halving the x-rows per item was measured slower: per-item overheads)
  const int Xs = X / xsplit;
  const int Xp = (Xs + 3) / 4 * 4 + 4, Xhp = Xs / 2 + 1;
  const size_t smem = sizeof(float) * ((size_t)kDsRound * CC + (size_t)CC * Xp + (size_t)CC * Xhp +
                                       2 * kDsRound + 4 * (size_t)Xp + 8);
  if (smem > 220 * 1024) return VEON_E_UNSUPPORTED;
  static size_t attr_smem[kMaxDevices] = {};
  const int dev = current_device();
  if (smem > attr_smem[dev]) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_pool_ds_fwd<KCH>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem[dev] = smem;
  }
  int per_sm = 1;
  VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pool_ds_fwd<KCH>,
                                                              kDsThreads, smem));
  if (per_sm < 1) per_sm = 1;
  const int n_chunks = C / CC;
  const int64_t n_items = (int64_t)B * (Z / 2) * (Y / 2) * xsplit * n_chunks;
  if (n_items > 0x7fffffffLL) return VEON_E_RANGE;
  int64_t blocks = (int64_t)per_sm * sm_count();
  if (blocks > n_items) blocks = n_items;
  k_pool_ds_fwd<KCH><<<(unsigned)blocks, kDsThreads, smem, stream>>>(
      depth, feat, ranks_depth, ranks_feat, ranks_bev, voxel_start, (uint32_t)n_items,
      (uint32_t)n_chunks, Z, Y, X, xsplit, C, out);
  VEON_LAUNCH_CHECK();
  return 0;
}
