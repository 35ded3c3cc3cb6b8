// voxel_pooling_prepare_v2 on the GPU: frustum points -> (ranks, intervals).
//
// Reference behaviour: mmdet3d/models/necks/view_transformer.py:202-260
// (identical copy at view_transformer_raw.py:244-302).  This is NOT a port of
// its ~25 ATen launches.  The voxel rank is a bounded integer key, so the
// "argsort" is a single-digit radix (counting) sort over a dense per-voxel
// histogram:
//
//   k_classify   coor -> key (float32 rank arithmetic, bit-exact), histogram
//                via one returning atomic per kept point (gives an arrival
//                slot inside the voxel)
//   k_scan       single-pass decoupled-look-back scan of the histogram: point
//                offsets AND interval numbering in one 64-bit packed scan;
//                emits interval_starts / interval_lengths directly
//   k_tiles      tile tables for the pooling kernels (by-product)
//   k_scatter    point -> its voxel segment (arrival order), writes ranks_bev
//   k_rank       segmented rank-by-counting: puts every segment into ascending
//                ranks_depth order (= what a stable sort would give), writes
//                ranks_depth / ranks_feat and the point->interval table
//   k_sort_long  bitonic fallback for pathological segments (> kLongSeg)
//
// The dense histogram doubles as the voxel->points map the pooling kernels
// need, so no separate pass builds it.
#include "geometry.cuh"

namespace veon {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;  // 2048 bins per CTA
constexpr int kLongSeg = 2048;                         // rank-by-counting limit

struct GridF {
  float lo[3], iv[3], gs[3];
  float gyx;   // fl(gs.y * gs.x)
  float gzyx;  // fl(fl(gs.z * gs.y) * gs.x)
};

// view_transformer.py:241-244 evaluated in float32 exactly as torch does:
//   r  = b * (gs2*gs1*gs0);  r += z * (gs1*gs0);  r += y*gs0 + x
__host__ __device__ __forceinline__ float rank_f32(float b, float z, float y, float x,
                                                   const GridF& g) {
#ifdef __CUDA_ARCH__
  float r = __fmul_rn(b, g.gzyx);
  r = __fadd_rn(r, __fmul_rn(z, g.gyx));
  float t = __fadd_rn(__fmul_rn(y, g.gs[0]), x);
  return __fadd_rn(r, t);
#else
  volatile float r = b * g.gzyx;
  volatile float zz = z * g.gyx;
  r = r + zz;
  volatile float t = y * g.gs[0];
  t = t + x;
  r = r + t;
  return r;
#endif
}

static GridF make_grid(const float* lower, const float* interval, const float* gs) {
  GridF g;
  for (int i = 0; i < 3; ++i) { g.lo[i] = lower[i]; g.iv[i] = interval[i]; g.gs[i] = gs[i]; }
  volatile float a = gs[1] * gs[0];
  g.gyx = a;
  volatile float zy = gs[2] * gs[1];
  volatile float zyx = zy * gs[0];
  g.gzyx = zyx;
  return g;
}

// number of histogram bins = largest reachable key + 1 (rank_f32 is monotone in
// every argument because float32 rounding is monotone)
static int64_t num_bins(int B, const GridF& g) {
  float mx[3];
  for (int i = 0; i < 3; ++i) {
    // largest integer-valued t with t < gs[i]
    float t = floorf(g.gs[i]);
    if (t >= g.gs[i]) t -= 1.0f;
    if (t < 0.0f) t = 0.0f;
    mx[i] = t;
  }
  float r = rank_f32((float)(B - 1), mx[2], mx[1], mx[0], g);
  if (!(r >= 0.0f)) return 1;
  if (r > 2.0e9f) return -1;
  return (int64_t)r + 1;
}

struct PrepWs {
  int32_t *key, *slot, *tmp, *count, *offset, *iidx, *long_list;
  unsigned long long* desc;
  uint32_t* ctrl;  // [0] scan ticket, [1] number of long segments
  int64_t nbins_pad, scan_tiles, long_cap;
  size_t zero_begin, zero_bytes, total;
};

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static PrepWs carve(void* base, int64_t P, int64_t nbins, int64_t BV) {
  PrepWs w;
  int64_t need = (nbins > BV ? nbins : BV) + 1;  // offset[v + 1] must exist for every key
  w.nbins_pad = (need + kScanTile - 1) / kScanTile * kScanTile;
  w.scan_tiles = w.nbins_pad / kScanTile;
  w.long_cap = P / kLongSeg + 2;
  size_t off = 0;
  char* b = (char*)base;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  size_t o_key = take(sizeof(int32_t) * P);
  size_t o_slot = take(sizeof(int32_t) * P);
  size_t o_tmp = take(sizeof(int32_t) * P);
  size_t o_off = take(sizeof(int32_t) * w.nbins_pad);
  size_t o_iidx = take(sizeof(int32_t) * w.nbins_pad);
  size_t o_long = take(sizeof(int32_t) * w.long_cap);
  // zero-initialised region: histogram, look-back descriptors, control words
  w.zero_begin = off;
  size_t o_count = take(sizeof(int32_t) * w.nbins_pad);
  size_t o_desc = take(sizeof(unsigned long long) * w.scan_tiles);
  size_t o_ctrl = take(sizeof(uint32_t) * 16);
  w.zero_bytes = off - w.zero_begin;
  w.total = off;
  w.key = (int32_t*)(b + o_key);
  w.slot = (int32_t*)(b + o_slot);
  w.tmp = (int32_t*)(b + o_tmp);
  w.offset = (int32_t*)(b + o_off);
  w.iidx = (int32_t*)(b + o_iidx);
  w.long_list = (int32_t*)(b + o_long);
  w.count = (int32_t*)(b + o_count);
  w.desc = (unsigned long long*)(b + o_desc);
  w.ctrl = (uint32_t*)(b + o_ctrl);
  return w;
}

// ---------------------------------------------------------------- k_classify
// One thread per frustum point.  (coor - lower) / interval with IEEE sub/div
// (no contraction), truncation toward zero like `.long()` (:227), bounds test
// against the FLOAT grid_size (:233-235), float32 rank (:241-244).
// FUSED: the coordinates are not read but computed from the frustum and the per-camera
// transforms (the formula of k_lidar_coor, geometry.cuh): `coor` never exists in memory.
template <bool FUSED>
__global__ void __launch_bounds__(256)
k_classify(const float* __restrict__ coor, const float* __restrict__ frustum,
           const CamXform* __restrict__ xf, int64_t DHW, int64_t P, int64_t pts_per_sample,
           GridF g, int64_t nbins, int32_t* __restrict__ key, int32_t* __restrict__ slot,
           int32_t* __restrict__ count, const float* __restrict__ depth_w, float depth_eps) {
  pdl_prologue();
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float cx, cy, cz;
  if (FUSED) {
    const int64_t bn = p / DHW;
    lidar_point(frustum + 3 * (p - bn * DHW), xf[bn], cx, cy, cz);
  } else {
    const float* c = coor + 3 * p;
    cx = __ldg(c + 0);
    cy = __ldg(c + 1);
    cz = __ldg(c + 2);
  }
  float fx = __fdiv_rn(__fsub_rn(cx, g.lo[0]), g.iv[0]);
  float fy = __fdiv_rn(__fsub_rn(cy, g.lo[1]), g.iv[1]);
  float fz = __fdiv_rn(__fsub_rn(cz, g.lo[2]), g.iv[2]);
  float tx = truncf(fx), ty = truncf(fy), tz = truncf(fz);
  // NaN compares false everywhere -> dropped (the CPU reference drops it too:
  // cvttss2si yields INT64_MIN).  (-1,0) truncates to -0.0 which IS kept.
  bool kept = (tx >= 0.0f) && (tx < g.gs[0]) && (ty >= 0.0f) && (ty < g.gs[1]) &&
              (tz >= 0.0f) && (tz < g.gs[2]);
  // opt-in (inference): a point whose depth weight is negligible is dropped like an out-of-grid
  // one -- VEON's two-hot depth leaves ~90 % of the bins at the e^-16 clamp (SURVEY 8f-2)
  if (depth_w != nullptr && kept) kept = __ldg(depth_w + p) > depth_eps;
  int32_t k = -1, s = 0;
  if (kept) {
    float b = (float)(p / pts_per_sample);
    float r = rank_f32(b, tz, ty, tx, g);
    int64_t ki = (int64_t)r;  // .int() truncation; r >= 0 here
    if (ki >= 0 && ki < nbins) {
      k = (int32_t)ki;
      s = atomicAdd(count + k, 1);
    }
  }
  key[p] = k;
  slot[p] = s;
}

// -------------------------------------------------------------------- k_scan
// packed 64-bit scan element: bits 0..30 points, bits 31..61 occupied voxels,
// bits 62..63 look-back status
__device__ __forceinline__ unsigned long long pack_count(int c) {
  return (unsigned long long)(uint32_t)c | ((unsigned long long)(c > 0) << 31);
}
constexpr unsigned long long kFlagAgg = 1ull << 62;
constexpr unsigned long long kFlagIncl = 2ull << 62;
constexpr unsigned long long kValMask = (1ull << 62) - 1;

__device__ __forceinline__ unsigned long long ld_relaxed(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(kScanThreads)
k_scan(const int32_t* __restrict__ count, int32_t* __restrict__ offset,
       int32_t* __restrict__ iidx, int32_t* __restrict__ istarts,
       int32_t* __restrict__ ilens, unsigned long long* desc, uint32_t* ctrl,
       int32_t* __restrict__ long_list, int long_cap, int64_t* counts_out,
       int64_t* counts_mirror, int num_tiles,
       int32_t* __restrict__ tile_start, int32_t* __restrict__ tile_istart,
       uint32_t* __restrict__ tile_occ, int64_t n_pool_tiles) {
  pdl_prologue();
  __shared__ uint32_t s_tile;
  __shared__ unsigned long long s_warp[kScanThreads / 32];
  __shared__ unsigned long long s_excl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ctrl, 1u);  // ticket => predecessors are running/finished
  __syncthreads();
  const uint32_t tile = s_tile;
  const int64_t base = (int64_t)tile * kScanTile + (int64_t)tid * kScanItems;
  int c[kScanItems];
  {
    const int4* src = reinterpret_cast<const int4*>(count + base);
    int4 a = src[0], b = src[1];
    c[0] = a.x; c[1] = a.y; c[2] = a.z; c[3] = a.w;
    c[4] = b.x; c[5] = b.y; c[6] = b.z; c[7] = b.w;
  }
  unsigned long long tsum = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) tsum += pack_count(c[i]);
  unsigned long long incl = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  unsigned long long wprefix = 0, btotal = 0;
#pragma unroll
  for (int w = 0; w < kScanThreads / 32; ++w) {
    unsigned long long v = s_warp[w];
    if (w < warp) wprefix += v;
    btotal += v;
  }
  // decoupled look-back, one warp wide: lane l inspects predecessor tile-1-l;
  // the window slides back 32 tiles at a time until an inclusive prefix is seen
  if (warp == 0) {
    unsigned long long excl = 0;
    if (tile == 0) {
      if (lane == 0) st_relaxed(desc, kFlagIncl | btotal);
    } else {
      if (lane == 0) st_relaxed(desc + tile, kFlagAgg | btotal);
      int64_t hi = (int64_t)tile - 1;  // newest predecessor of the window
      while (true) {
        const int64_t j = hi - lane;
        unsigned long long d = kFlagIncl;  // virtual tile -1: inclusive prefix 0
        if (j >= 0) {
          do { d = ld_relaxed(desc + j); } while ((d >> 62) == 0);
        }
        const uint32_t incl_mask = __ballot_sync(0xffffffffu, (d & kFlagIncl) != 0);
        // lanes nearer than (and including) the first inclusive one contribute
        const int stop = incl_mask ? __ffs(incl_mask) - 1 : 31;
        unsigned long long v = (lane <= stop) ? (d & kValMask) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        excl += v;
        if (incl_mask) break;
        hi -= 32;
      }
      if (lane == 0) st_relaxed(desc + tile, kFlagIncl | (excl + btotal));
    }
    if (lane == 0) s_excl = excl;
  }
  __syncthreads();
  unsigned long long run = s_excl + wprefix + (incl - tsum);
  int32_t off8[kScanItems], idx8[kScanItems];
  uint32_t occ8 = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    const int32_t pts = (int32_t)(run & 0x7fffffffull);
    const int32_t ints = (int32_t)((run >> 31) & 0x7fffffffull);
    off8[i] = pts;
    idx8[i] = ints;
    if (c[i] > 0) {
      occ8 |= 1u << i;
      istarts[ints] = pts;
      ilens[ints] = c[i];
      if (c[i] > kLongSeg) {
        uint32_t q = atomicAdd(ctrl + 1, 1u);
        if ((int)q < long_cap) long_list[q] = (int32_t)(base + i);
      }
    }
    run += pack_count(c[i]);
  }
  {  // one full 32-byte sector per thread and array
    int4* o4 = reinterpret_cast<int4*>(offset + base);
    int4* i4 = reinterpret_cast<int4*>(iidx + base);
    o4[0] = make_int4(off8[0], off8[1], off8[2], off8[3]);
    o4[1] = make_int4(off8[4], off8[5], off8[6], off8[7]);
    i4[0] = make_int4(idx8[0], idx8[1], idx8[2], idx8[3]);
    i4[1] = make_int4(idx8[4], idx8[5], idx8[6], idx8[7]);
  }
  // pooling-tile tables (V % 32 == 0: bin g starts tile g/32).  Four consecutive
  // threads hold one 32-voxel tile; combine their 8-bit occupancy masks.
  if (tile_start) {
    uint32_t m = occ8 << (8 * (tid & 3));
    m |= __shfl_xor_sync(0xffffffffu, m, 1);
    m |= __shfl_xor_sync(0xffffffffu, m, 2);
    const int64_t pt = base >> 5;
    if ((tid & 3) == 0 && pt <= n_pool_tiles) {
      tile_start[pt] = off8[0];
      tile_istart[pt] = idx8[0];
      tile_occ[pt] = m;
    }
  }
  if ((int)tile == num_tiles - 1 && tid == kScanThreads - 1) {
    counts_out[0] = (int64_t)(run & 0x7fffffffull);
    counts_out[1] = (int64_t)((run >> 31) & 0x7fffffffull);
    if (counts_mirror) {  // pinned host memory: the host reads it after an event, no copy queued
      counts_mirror[0] = counts_out[0];
      counts_mirror[1] = counts_out[1];
      __threadfence_system();
    }
  }
}

// ------------------------------------------------------------------- k_tiles
// tile tables when V is not a multiple of 32 (otherwise k_scan emits them)
__global__ void k_tiles(const int32_t* __restrict__ count, const int32_t* __restrict__ offset,
                        const int32_t* __restrict__ iidx, int64_t n_tiles,
                        int64_t tiles_per_sample, int64_t V, int32_t* __restrict__ tile_start,
                        int32_t* __restrict__ tile_istart, uint32_t* __restrict__ tile_occ) {
  pdl_prologue();
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  int64_t b = t / tiles_per_sample, vt = t % tiles_per_sample;
  int64_t g = b * V + vt * kTileVoxels;  // t == n_tiles -> g == B*V (sentinel)
  tile_start[t] = offset[g];
  tile_istart[t] = iidx[g];
  uint32_t m = 0;
  if (t < n_tiles)
    for (int i = 0; i < kTileVoxels && vt * kTileVoxels + i < V; ++i)
      if (count[g + i] > 0) m |= 1u << i;
  tile_occ[t] = m;
}

// -------------------------------------------------------------------- k_fill
// Clears the scratch regions with a kernel instead of cudaMemsetAsync: memsets and the
// caller's bulk host<->device copies share the copy engines, and a step's first launch
// must not queue behind a 20 MB transfer of the previous step's results.
struct FillJob {
  uint32_t* p;
  int64_t n;   // 32-bit words
  uint32_t v;
};
struct FillJobs {
  FillJob j[3];
};
__global__ void __launch_bounds__(256) k_fill(FillJobs jobs) {
  pdl_launch_dependents();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    uint32_t* p = jobs.j[q].p;
    const int64_t n = jobs.j[q].n;
    const uint32_t v = jobs.j[q].v;
    if (n <= 0) continue;
    // 16-byte stores over the aligned middle, scalar head and tail
    const int64_t head = min(n, (int64_t)((16 - ((uintptr_t)p & 15)) & 15) / 4);
    const int64_t n4 = (n - head) / 4;
    uint4* p4 = reinterpret_cast<uint4*>(p + head);
    for (int64_t i = t0; i < n4; i += stride) p4[i] = make_uint4(v, v, v, v);
    if (t0 < head) p[t0] = v;
    const int64_t tail0 = head + 4 * n4;
    if (t0 < n - tail0) p[tail0 + t0] = v;
  }
}

static int launch_fill(const FillJobs& jobs, cudaStream_t stream) {
  int64_t words = 0;
  for (int q = 0; q < 3; ++q) words += jobs.j[q].n > 0 ? jobs.j[q].n : 0;
  if (words == 0) return 0;
  int64_t blocks = ceil_div64(ceil_div64(words, 4), 256 * 4);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  k_fill<<<(unsigned)blocks, 256, 0, stream>>>(jobs);
  VEON_LAUNCH_CHECK();
  return 0;
}

// -------------------------------------------------------------- k_heavy_list
// heavy[0] = number of listed tiles (zeroed by the caller's k_fill), heavy[1] = threshold,
// heavy[2..] = tile ids in arbitrary order (the order only affects scheduling)
__global__ void k_heavy_list(const int32_t* __restrict__ tile_start, int64_t n_tiles, int thr,
                             int cap, int32_t* __restrict__ heavy) {
  pdl_prologue();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t == 0) heavy[1] = thr;
  if (t >= n_tiles) return;
  if (tile_start[t + 1] - tile_start[t] >= thr) {
    const int i = atomicAdd(heavy, 1);
    if (i < cap) heavy[2 + i] = (int32_t)t;
  }
}

static int build_heavy_list(const int32_t* tile_start, int64_t n_tiles, int64_t n_points_cap,
                            int32_t* heavy, cudaStream_t stream) {
  // heavy[0] was cleared by the caller's k_fill
  VEON_CUDA_TRY(launch_pdl(k_heavy_list, dim3((unsigned)ceil_div64(n_tiles, 256)), dim3(256), 0, stream,
                           tile_start, n_tiles, heavy_threshold(),
                           (int)heavy_capacity(n_points_cap, n_tiles), heavy));
  VEON_LAUNCH_CHECK();
  return 0;
}

// ----------------------------------------------------------------- k_scatter
__global__ void __launch_bounds__(256)
k_scatter(const int32_t* __restrict__ key, const int32_t* __restrict__ slot,
          const int32_t* __restrict__ offset, int64_t P, int32_t* __restrict__ tmp,
          int32_t* __restrict__ ranks_bev) {
  pdl_prologue();
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int32_t k = key[p];
  if (k < 0) return;
  int32_t pos = offset[k] + slot[p];
  tmp[pos] = (int32_t)p;
  ranks_bev[pos] = k;
}

struct PointDims {
  int D, HW, DHW;  // DHW <= P < 2^31
};
__device__ __forceinline__ void split_point(int32_t p, const PointDims& d, int32_t& pix,
                                            int32_t& dd) {
  int32_t bn = p / d.DHW;
  int32_t rem = p - bn * d.DHW;
  dd = rem / d.HW;
  pix = bn * d.HW + (rem - dd * d.HW);
}

// -------------------------------------------------------------------- k_rank
// One thread per sorted slot i.  Its point id p ranks inside its voxel segment
// by counting smaller ids (segments are short: mean 1.5-2.5, p99 <= 20).
__global__ void __launch_bounds__(256)
k_rank(const int32_t* __restrict__ tmp, const int32_t* __restrict__ ranks_bev,
       const int32_t* __restrict__ offset, const int32_t* __restrict__ iidx,
       const int64_t* __restrict__ counts, PointDims dims,
       int32_t* __restrict__ ranks_depth, int32_t* __restrict__ ranks_feat,
       int32_t* __restrict__ point_interval) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= counts[0]) return;
  const int32_t v = ranks_bev[i];
  const int32_t s = offset[v], e = offset[v + 1];
  if (e - s > kLongSeg) return;  // k_sort_long owns it
  const int32_t p = tmp[i];
  int32_t r = 0;
  for (int32_t j = s; j < e; ++j) r += (tmp[j] < p);
  int32_t pix, dd;
  split_point(p, dims, pix, dd);
  ranks_depth[s + r] = p;
  ranks_feat[s + r] = pix;
  if (point_interval) point_interval[(int64_t)pix * dims.D + dd] = iidx[v];
}

// --------------------------------------------------------------- k_sort_long
// Pathological segments (thousands of points in one voxel): one CTA sorts the
// segment in place with a same-direction bitonic network (virtual +inf padding
// never moves), then emits it.
__global__ void __launch_bounds__(1024)
k_sort_long(int32_t* tmp, const int32_t* __restrict__ offset, const int32_t* __restrict__ iidx,
            const int32_t* __restrict__ long_list, const uint32_t* __restrict__ ctrl,
            int long_cap, PointDims dims, int32_t* __restrict__ ranks_depth,
            int32_t* __restrict__ ranks_feat, int32_t* __restrict__ point_interval) {
  pdl_prologue();
  uint32_t n_long = ctrl[1];
  if ((int)n_long > long_cap) n_long = long_cap;
  for (uint32_t q = blockIdx.x; q < n_long; q += gridDim.x) {
    const int32_t v = long_list[q];
    const int32_t s = offset[v], len = offset[v + 1] - s;
    int32_t* a = tmp + s;
    int64_t n2 = 1;
    while (n2 < len) n2 <<= 1;
    for (int64_t k = 2; k <= n2; k <<= 1) {
      for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
        int64_t l = i ^ (k - 1);
        if (l > i && l < len) {
          int32_t x = a[i], y = a[l];
          if (x > y) { a[i] = y; a[l] = x; }
        }
      }
      __syncthreads();
      for (int64_t j = k >> 2; j > 0; j >>= 1) {
        for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
          int64_t l = i ^ j;
          if (l > i && l < len) {
            int32_t x = a[i], y = a[l];
            if (x > y) { a[i] = y; a[l] = x; }
          }
        }
        __syncthreads();
      }
    }
    const int32_t ii = iidx[v];
    for (int32_t i = threadIdx.x; i < len; i += blockDim.x) {
      int32_t p = a[i], pix, dd;
      split_point(p, dims, pix, dd);
      ranks_depth[s + i] = p;
      ranks_feat[s + i] = pix;
      if (point_interval) point_interval[(int64_t)pix * dims.D + dd] = ii;
    }
    __syncthreads();
  }
}

// ============================================================ plan from ranks
// For rank arrays the caller already holds (accelerate cache or user input):
// validate that they are what prepare would have produced, and build the tile
// tables + point->interval table.
__device__ __forceinline__ int64_t lower_bound_i32(const int32_t* a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)a[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void k_plan_tiles(const int32_t* __restrict__ ranks_bev, int64_t n_points,
                             const int32_t* __restrict__ istarts, int64_t n_int,
                             int64_t n_tiles, int64_t tiles_per_sample, int64_t V,
                             int32_t* __restrict__ tile_start,
                             int32_t* __restrict__ tile_istart,
                             uint32_t* __restrict__ tile_occ) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  int64_t b = t / tiles_per_sample, vt = t % tiles_per_sample;
  int64_t g = b * V + vt * kTileVoxels;
  int64_t ps = lower_bound_i32(ranks_bev, n_points, g);
  tile_start[t] = (int32_t)ps;
  tile_istart[t] = (int32_t)lower_bound_i32(istarts, n_int, ps);
  uint32_t m = 0;
  if (t < n_tiles) {
    const int64_t gend = min(g + kTileVoxels, (b + 1) * V);
    for (int64_t i = ps; i < n_points; ++i) {
      const int64_t rbv = ranks_bev[i];
      if (rbv >= gend || rbv < g) break;
      m |= 1u << (int)(rbv - g);
    }
  }
  tile_occ[t] = m;
}

__global__ void k_plan_points(const int32_t* __restrict__ ranks_depth,
                              const int32_t* __restrict__ ranks_feat,
                              const int32_t* __restrict__ ranks_bev, int64_t n_points,
                              int64_t P, int64_t n_feat_rows, int64_t BV, PointDims dims,
                              int32_t* flags) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_points) return;
  int32_t f = 0;
  const int32_t rb = ranks_bev[i], rd = ranks_depth[i], rf = ranks_feat[i];
  if (i > 0 && ranks_bev[i - 1] > rb) f |= VEON_PLAN_UNSORTED;
  if (rb < 0 || rb >= BV || rd < 0 || rd >= P || rf < 0 || rf >= n_feat_rows) {
    f |= VEON_PLAN_OUT_OF_RANGE;
  } else {
    int32_t pix, dd;
    split_point(rd, dims, pix, dd);
    if (pix != rf) f |= VEON_PLAN_NONCANONICAL;
  }
  if (f) atomicOr(flags, f);
}

__global__ void k_plan_intervals(const int32_t* __restrict__ ranks_depth,
                                 const int32_t* __restrict__ ranks_bev, int64_t n_points,
                                 const int32_t* __restrict__ istarts,
                                 const int32_t* __restrict__ ilens, int64_t n_int, int64_t P,
                                 PointDims dims, int32_t* __restrict__ point_interval,
                                 int32_t* flags) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_int) return;
  const int64_t s = istarts[k], l = ilens[k];
  int32_t f = 0;
  const int64_t expect = (k == 0) ? 0 : (int64_t)istarts[k - 1] + ilens[k - 1];
  if (l <= 0 || s != expect || s + l > n_points || (k == n_int - 1 && s + l != n_points)) {
    atomicOr(flags, VEON_PLAN_BAD_INTERVALS);
    return;
  }
  const int32_t rb = ranks_bev[s];
  if (s > 0 && ranks_bev[s - 1] == rb) f |= VEON_PLAN_BAD_INTERVALS;
  for (int64_t i = s; i < s + l; ++i) {
    if (ranks_bev[i] != rb) f |= VEON_PLAN_BAD_INTERVALS;
    const int32_t rd = ranks_depth[i];
    if (rd >= 0 && rd < P) {
      int32_t pix, dd;
      split_point(rd, dims, pix, dd);
      int32_t old = atomicCAS(point_interval + (int64_t)pix * dims.D + dd, -1, (int32_t)k);
      if (old != -1) f |= VEON_PLAN_DUPLICATE;
    }
  }
  if (f) atomicOr(flags, f);
}

}  // namespace veon

using namespace veon;

extern "C" int64_t veon_pool_num_tiles(int B, int64_t V) {
  return (int64_t)B * ceil_div64(V, kTileVoxels);
}

extern "C" int64_t veon_pool_heavy_list_ints(int64_t n_points, int64_t n_tiles) {
  if (n_points < 0 || n_tiles < 0) return 0;
  return 2 + heavy_capacity(n_points, n_tiles);
}

static int check_dims(int B, int N, int D, int H, int W, int64_t* P) {
  if (B <= 0 || N <= 0 || D <= 0 || H <= 0 || W <= 0) return VEON_E_BADARG;
  int64_t p = (int64_t)B * N * D * H * W;
  if (p > 0x7fffffffLL - 2 * kScanTile) return VEON_E_RANGE;
  *P = p;
  return 0;
}

static int64_t voxels_of(const float* gs) {
  return (int64_t)gs[0] * (int64_t)gs[1] * (int64_t)gs[2];  // int(grid_size[i]), :190-193
}

extern "C" size_t veon_prepare_v2_workspace_bytes(int B, int N, int D, int H, int W,
                                                  const float* grid_size) {
  int64_t P;
  if (!grid_size || check_dims(B, N, D, H, W, &P)) return 0;
  const float one[3] = {1.f, 1.f, 1.f}, zero[3] = {0.f, 0.f, 0.f};
  GridF g = make_grid(zero, one, grid_size);
  int64_t nbins = num_bins(B, g);
  if (nbins < 0) return 0;
  PrepWs w = carve(nullptr, P, nbins, (int64_t)B * voxels_of(grid_size));
  return w.total;
}

static int prepare_impl(const float* coor, const float* frustum, const CamXform* xf, int B, int N,
                        int D, int H, int W, const float* lower, const float* interval,
                               const float* grid_size, int32_t* ranks_bev,
                               int32_t* ranks_depth, int32_t* ranks_feat,
                               int32_t* interval_starts, int32_t* interval_lengths,
                               int64_t* counts, int64_t* counts_host, int32_t* tile_start,
                               int32_t* tile_istart, uint32_t* tile_occ, int32_t* tile_heavy,
                               int32_t* point_interval, void* workspace,
                               size_t workspace_bytes, void* stream_,
                               const float* depth_w = nullptr, float depth_eps = 0.f) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int64_t P;
  int rc = check_dims(B, N, D, H, W, &P);
  if (rc) return rc;
  if ((!coor && !(frustum && xf)) || !lower || !interval || !grid_size || !ranks_bev ||
      !ranks_depth || !ranks_feat || !interval_starts || !interval_lengths || !counts || !workspace)
    return VEON_E_BADARG;
  GridF g = make_grid(lower, interval, grid_size);
  const int64_t nbins = num_bins(B, g);
  const int64_t V = voxels_of(grid_size);
  if (nbins < 0 || V <= 0 || (int64_t)B * V > 0x7fffffffLL - 2 * kScanTile) return VEON_E_RANGE;
  PrepWs w = carve(workspace, P, nbins, (int64_t)B * V);
  if (workspace_bytes < w.total) return VEON_E_WORKSPACE;
  if (((uintptr_t)workspace & 15) != 0) return VEON_E_BADARG;

  {
    FillJobs jobs = {};
    jobs.j[0] = {reinterpret_cast<uint32_t*>((char*)workspace + w.zero_begin),
                 (int64_t)(w.zero_bytes / 4), 0u};
    if (point_interval) jobs.j[1] = {reinterpret_cast<uint32_t*>(point_interval), P, 0xffffffffu};
    if (tile_start && tile_istart && tile_occ && tile_heavy)
      jobs.j[2] = {reinterpret_cast<uint32_t*>(tile_heavy), 2, 0u};
    rc = launch_fill(jobs, stream);
    if (rc) return rc;
  }

  const int64_t pts_per_sample = (int64_t)N * D * H * W;
  const unsigned pblocks = (unsigned)ceil_div64(P, 256);
  // from here on every kernel is a programmatic dependent of the one before (common.cuh)
  const int64_t DHW = (int64_t)D * H * W;
  if (coor) {
    VEON_CUDA_TRY(launch_pdl(k_classify<false>, dim3(pblocks), dim3(256), 0, stream, coor,
                             (const float*)nullptr, (const CamXform*)nullptr, DHW, P,
                             pts_per_sample, g, nbins, w.key, w.slot, w.count, depth_w, depth_eps));
  } else {
    VEON_CUDA_TRY(launch_pdl(k_classify<true>, dim3(pblocks), dim3(256), 0, stream,
                             (const float*)nullptr, frustum, xf, DHW, P, pts_per_sample, g, nbins,
                             w.key, w.slot, w.count, depth_w, depth_eps));
  }
  VEON_LAUNCH_CHECK();
  const bool want_tiles = tile_start && tile_istart && tile_occ;
  const int64_t tps = ceil_div64(V, kTileVoxels), n_tiles = (int64_t)B * tps;
  const bool fused_tiles = want_tiles && (V % kTileVoxels == 0);
  VEON_CUDA_TRY(launch_pdl(k_scan, dim3((unsigned)w.scan_tiles), dim3(kScanThreads), 0, stream,
                           w.count, w.offset, w.iidx, interval_starts, interval_lengths, w.desc,
                           w.ctrl, w.long_list, (int)w.long_cap, counts, counts_host,
                           (int)w.scan_tiles, fused_tiles ? tile_start : nullptr, tile_istart,
                           tile_occ, n_tiles));
  VEON_LAUNCH_CHECK();
  if (want_tiles && !fused_tiles) {
    VEON_CUDA_TRY(launch_pdl(k_tiles, dim3((unsigned)ceil_div64(n_tiles + 1, 256)), dim3(256), 0,
                             stream, w.count, w.offset, w.iidx, n_tiles, tps, V, tile_start,
                             tile_istart, tile_occ));
    VEON_LAUNCH_CHECK();
  }
  if (want_tiles && tile_heavy) {
    rc = build_heavy_list(tile_start, n_tiles, P, tile_heavy, stream);
    if (rc) return rc;
  }
  VEON_CUDA_TRY(launch_pdl(k_scatter, dim3(pblocks), dim3(256), 0, stream, w.key, w.slot, w.offset,
                           P, w.tmp, ranks_bev));
  VEON_LAUNCH_CHECK();
  PointDims dims{D, H * W, D * H * W};
  VEON_CUDA_TRY(launch_pdl(k_rank, dim3(pblocks), dim3(256), 0, stream, w.tmp, ranks_bev, w.offset,
                           w.iidx, counts, dims, ranks_depth, ranks_feat, point_interval));
  VEON_LAUNCH_CHECK();
  VEON_CUDA_TRY(launch_pdl(k_sort_long, dim3(64), dim3(1024), 0, stream, w.tmp, w.offset, w.iidx,
                           w.long_list, w.ctrl, (int)w.long_cap, dims, ranks_depth, ranks_feat,
                           point_interval));
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" int veon_prepare_v2(const float* coor, int B, int N, int D, int H, int W,
                               const float* lower, const float* interval,
                               const float* grid_size, int32_t* ranks_bev,
                               int32_t* ranks_depth, int32_t* ranks_feat,
                               int32_t* interval_starts, int32_t* interval_lengths,
                               int64_t* counts, int64_t* counts_host, int32_t* tile_start,
                               int32_t* tile_istart, uint32_t* tile_occ, int32_t* tile_heavy,
                               int32_t* point_interval, void* workspace,
                               size_t workspace_bytes, void* stream_) {
  if (!coor) return VEON_E_BADARG;
  return prepare_impl(coor, nullptr, nullptr, B, N, D, H, W, lower, interval, grid_size, ranks_bev,
                      ranks_depth, ranks_feat, interval_starts, interval_lengths, counts,
                      counts_host, tile_start, tile_istart, tile_occ, tile_heavy, point_interval,
                      workspace, workspace_bytes, stream_);
}

// get_lidar_coor fused into the preparation (SURVEY 8f-3): same ranks as
// veon_lidar_coor + veon_prepare_v2, without the [B,N,D,H,W,3] coordinate tensor.
// depth / depth_eps (veon_prepare_v2_calib_sparse): points with depth weight <= depth_eps are
// dropped as well.
static int prepare_calib(const float* frustum, const float* sensor2ego,
                                     const float* cam2imgs, const float* post_rots,
                                     const float* post_trans, const float* bda, int B, int N,
                                     int D, int H, int W, const float* lower,
                                     const float* interval, const float* grid_size,
                                     int32_t* ranks_bev, int32_t* ranks_depth,
                                     int32_t* ranks_feat, int32_t* interval_starts,
                                     int32_t* interval_lengths, int64_t* counts,
                                     int64_t* counts_host, int32_t* tile_start,
                                     int32_t* tile_istart, uint32_t* tile_occ,
                                     int32_t* tile_heavy, int32_t* point_interval,
                                     void* xform_workspace, size_t xform_workspace_bytes,
                                     void* workspace, size_t workspace_bytes, void* stream_,
                                     const float* depth_w, float depth_eps) {
  if (!frustum || !sensor2ego || !cam2imgs || !post_rots || !post_trans || !bda ||
      !xform_workspace || B <= 0 || N <= 0)
    return VEON_E_BADARG;
  if (xform_workspace_bytes < sizeof(CamXform) * (size_t)B * N) return VEON_E_WORKSPACE;
  CamXform* xf = (CamXform*)xform_workspace;
  int rc = launch_cam_xforms(sensor2ego, cam2imgs, post_rots, post_trans, bda, B, N, xf,
                             (cudaStream_t)stream_);
  if (rc) return rc;
  return prepare_impl(nullptr, frustum, xf, B, N, D, H, W, lower, interval, grid_size, ranks_bev,
                      ranks_depth, ranks_feat, interval_starts, interval_lengths, counts,
                      counts_host, tile_start, tile_istart, tile_occ, tile_heavy, point_interval,
                      workspace, workspace_bytes, stream_, depth_w, depth_eps);
}

extern "C" int veon_prepare_v2_calib_sparse(
    const float* frustum, const float* sensor2ego, const float* cam2imgs, const float* post_rots,
    const float* post_trans, const float* bda, const float* depth, float depth_eps, int B, int N,
    int D, int H, int W, const float* lower, const float* interval, const float* grid_size,
    int32_t* ranks_bev, int32_t* ranks_depth, int32_t* ranks_feat, int32_t* interval_starts,
    int32_t* interval_lengths, int64_t* counts, int64_t* counts_host, int32_t* tile_start,
    int32_t* tile_istart, uint32_t* tile_occ, int32_t* tile_heavy, int32_t* point_interval,
    void* xform_workspace, size_t xform_workspace_bytes, void* workspace, size_t workspace_bytes,
    void* stream_) {
  if (!depth || !(depth_eps >= 0.f)) return VEON_E_BADARG;
  return prepare_calib(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda, B, N, D, H, W,
                       lower, interval, grid_size, ranks_bev, ranks_depth, ranks_feat,
                       interval_starts, interval_lengths, counts, counts_host, tile_start,
                       tile_istart, tile_occ, tile_heavy, point_interval, xform_workspace,
                       xform_workspace_bytes, workspace, workspace_bytes, stream_, depth, depth_eps);
}

extern "C" int veon_prepare_v2_calib(const float* frustum, const float* sensor2ego,
                                     const float* cam2imgs, const float* post_rots,
                                     const float* post_trans, const float* bda, int B, int N,
                                     int D, int H, int W, const float* lower,
                                     const float* interval, const float* grid_size,
                                     int32_t* ranks_bev, int32_t* ranks_depth,
                                     int32_t* ranks_feat, int32_t* interval_starts,
                                     int32_t* interval_lengths, int64_t* counts,
                                     int64_t* counts_host, int32_t* tile_start,
                                     int32_t* tile_istart, uint32_t* tile_occ,
                                     int32_t* tile_heavy, int32_t* point_interval,
                                     void* xform_workspace, size_t xform_workspace_bytes,
                                     void* workspace, size_t workspace_bytes, void* stream_) {
  return prepare_calib(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda, B, N, D, H, W,
                       lower, interval, grid_size, ranks_bev, ranks_depth, ranks_feat,
                       interval_starts, interval_lengths, counts, counts_host, tile_start,
                       tile_istart, tile_occ, tile_heavy, point_interval, xform_workspace,
                       xform_workspace_bytes, workspace, workspace_bytes, stream_, nullptr, 0.f);
}

extern "C" int veon_pool_plan_build(const int32_t* ranks_depth, const int32_t* ranks_feat,
                                    const int32_t* ranks_bev, const int32_t* interval_starts,
                                    const int32_t* interval_lengths, int64_t n_points,
                                    int64_t n_intervals, int B, int N, int D, int H, int W,
                                    int64_t V, int32_t* tile_start, int32_t* tile_istart,
                                    uint32_t* tile_occ, int32_t* tile_heavy,
                                    int32_t* point_interval, int32_t* flags, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int64_t P;
  int rc = check_dims(B, N, D, H, W, &P);
  if (rc) return rc;
  if (!ranks_depth || !ranks_feat || !ranks_bev || !interval_starts || !interval_lengths ||
      !tile_start || !tile_istart || !tile_occ || !point_interval || !flags || V <= 0 ||
      n_points <= 0 ||
      n_intervals <= 0)
    return VEON_E_BADARG;
  if ((int64_t)B * V > 0x7fffffffLL) return VEON_E_RANGE;
  {
    FillJobs jobs = {};
    jobs.j[0] = {reinterpret_cast<uint32_t*>(flags), 1, 0u};
    jobs.j[1] = {reinterpret_cast<uint32_t*>(point_interval), P, 0xffffffffu};
    if (tile_heavy) jobs.j[2] = {reinterpret_cast<uint32_t*>(tile_heavy), 2, 0u};
    rc = launch_fill(jobs, stream);
    if (rc) return rc;
  }
  PointDims dims{D, H * W, D * H * W};
  k_plan_points<<<(unsigned)ceil_div64(n_points, 256), 256, 0, stream>>>(
      ranks_depth, ranks_feat, ranks_bev, n_points, P, (int64_t)B * N * H * W, (int64_t)B * V,
      dims, flags);
  VEON_LAUNCH_CHECK();
  k_plan_intervals<<<(unsigned)ceil_div64(n_intervals, 256), 256, 0, stream>>>(
      ranks_depth, ranks_bev, n_points, interval_starts, interval_lengths, n_intervals, P, dims,
      point_interval, flags);
  VEON_LAUNCH_CHECK();
  const int64_t tps = ceil_div64(V, kTileVoxels), n_tiles = (int64_t)B * tps;
  k_plan_tiles<<<(unsigned)ceil_div64(n_tiles + 1, 256), 256, 0, stream>>>(
      ranks_bev, n_points, interval_starts, n_intervals, n_tiles, tps, V, tile_start,
      tile_istart, tile_occ);
  VEON_LAUNCH_CHECK();
  if (tile_heavy) return build_heavy_list(tile_start, n_tiles, n_points, tile_heavy, stream);
  return 0;
}
