// bev_pool_v2 forward as two warp-specialised roles around an L2-resident ring of compact rows.
//
// Reference behaviour: QuickCumsumCuda.forward (bev_pool.py:17-41: new_zeros +
// bev_pool_v2_kernel, bev_pool_cuda.cu:21-48) followed by `.permute(0,4,1,2,3).contiguous()`
// (bev_pool.py:91).
//
// The forward has an irregular half (gather the points of every occupied voxel: a chain of
// dependent load latencies) and a regular half (write the dense [B,C,Z,Y,X] volume, 1.3 GB at
// C2: the actual HBM cost).  When one warp does both for a tile the two halves do not overlap
// on an SM (round 1: T = max + 0.3 min, 0.63 of the copy bandwidth).  Here ONE persistent
// kernel (a CTA per SM) runs them as separate roles that meet in L2:
//
//   role A, 16 warps  A warp takes a 32-voxel tile, walks its points in rank order -- index
//                     records prefetched three stages ahead by cp.async, 12 feature rows in
//                     flight, lanes = channels, acc = fma(feat, depth, acc) starting from 0: the
//                     reference kernel's rounding sequence, so the result stays bit-identical --
//                     and stores ONE channel-contiguous row per occupied voxel into the CTA's
//                     ring.  No tile buffer, no zero fill, no transposition.
//   role E, 16 warps  Two groups of 8 warps; a group's item is 8 consecutive tiles x a
//                     64-channel chunk (an aligned 1 KB run of every channel plane).  A warp
//                     copies its tile's rows out of the ring into shared memory (16-byte
//                     cp.async, L2 only), the group meets at a named barrier, and every warp
//                     writes its 32-voxel x 64-channel block with 16-byte streaming stores, zeros
//                     where the occupancy mask says so: the group emits whole 1 KB runs in
//                     lockstep.  While one group waits for its copies the other one writes.  E
//                     reads nothing from DRAM: its only long-latency traffic is the store stream.
//
// Work is dealt in ROUNDS of 16 consecutive tiles (round r -> CTA r mod grid: every CTA samples
// the whole volume, so the point density averages out).  A round is produced by the 16 A warps
// of a CTA and consumed by the 16 E warps of the SAME CTA, through one of the CTA's own NS ring
// slots (512 rows x 64 channels; rows of the round's tiles packed by the running count of
// occupied voxels).  All flow control is two shared-memory counters per
// slot (filled by A, drained by E): no global flags, no atomics on global memory, no dependence
// between CTAs.  The ring (grid x NS slots, only the occupied prefix of a slot is ever touched)
// is a few tens of MB: its lines are rewritten while still dirty in L2 and never reach DRAM;
// DRAM sees the inputs once and the volume once.
//
// Rows are 64 channels wide, the only width at which this kernel beats k_pool_fwd (pool_fwd.cu);
// every other width takes that kernel.
//
// Tiles at or above the plan's heavy threshold are left to k_pool_fwd_heavy (pool_fwd.cu),
// which writes them straight into the volume, queued behind this grid.
#include "common.cuh"
#include "pool_fwd.cuh"

namespace veon {

constexpr int kRoundTiles = 16;         // tiles per round
constexpr int kAWarps = 16;             // role A warps per CTA: a tile each
constexpr int kEWarps = 16;             // role E warps per CTA: a tile each, two groups of 8
constexpr int CU = 64;                  // channels of a row
constexpr int kEGroup = 8;
constexpr int kStreamWarps = kAWarps + kEWarps;
// Registers are re-dealt between the warpgroups at role entry (setmaxnreg).  The pool is what
// the CTA was launched with (1024 threads x 64): what role E gives back must cover what role A
// takes -- anything less and the increase never returns.
constexpr int kLaunchRegs = 64, kARegs = 80, kERegs = 48;
static_assert(kEWarps * (kLaunchRegs - kERegs) >= kAWarps * (kARegs - kLaunchRegs),
              "setmaxnreg: role E must release what role A acquires");
template <int N>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
constexpr int kSlotRows = kRoundTiles * kTileVoxels;   // rows a ring slot can hold
constexpr int kMaxSlots = 16;           // ring slots per CTA (NS <= this)
// per-warp prefetch ring of role A.  slot = header + 32 point records of 4 ints.
// header: [0..16] tile_start of the round's 16 tiles (+ the end), [17..32] their occupancy masks
constexpr int kAHdr = 36;
constexpr int kASlotInts = kAHdr + 4 * 32;
constexpr int kADist = 1;               // prefetch distance in rounds per stage
constexpr int kASlots = 4 * kADist;
// Tiles at or above the plan's heavy threshold (96 points) are left to the CTA-per-tile kernel.
// Raising the bar for this kernel (role A claims dynamically and the ring has rounds of slack)
// was measured and loses: 128 / 256 / 384 / 768 points -> 321 / 357 / 386 / 487 us at C2.
constexpr int kStreamHeavyMin = 0;
constexpr int kEChunk = 32;             // channels per E step (two staging buffers per warp)
constexpr int kERows = 33;              // staged rows per tile: <= 32 occupied voxels + 1 of zeros

__device__ __forceinline__ void cpa4(void* smem_dst, const void* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cpa_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cpa_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cpa16_cg(uint32_t smem_dst, const void* gsrc) {   // L2 only
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}

#ifdef VEON_FWD_TRACE   // tools/fwd_trace.sh only: cycles per phase, CTA 0, every warp
__device__ unsigned long long veon_fwd_trace[32 * 8];
#define VEON_T0 long long _tt = clock64();
#define VEON_TACC(slotid)                                                             \
  {                                                                                   \
    const long long _n = clock64();                                                   \
    if (blockIdx.x == 0 && (threadIdx.x & 31) == 0)                                   \
      veon_fwd_trace[(threadIdx.x >> 5) * 8 + (slotid)] += (unsigned long long)(_n - _tt); \
    _tt = _n;                                                                         \
  }
#else
#define VEON_T0
#define VEON_TACC(slotid)
#endif

struct FwdStreamParams {
  const float *depth, *feat;
  const int32_t *ranks_depth, *ranks_feat, *ranks_bev;
  const int32_t* tile_start;
  const uint32_t* tile_occ;
  const int32_t* heavy;      // plan's heavy list ([1] = threshold) or NULL
  float* ring;               // [grid][ns][kSlotRows][CU]
  float* out;
  int64_t V;
  uint32_t n_tiles, n_rounds, tiles_per_sample;
  int C, ns_log2;            // 2^ns_log2 ring slots per CTA
};

// Per ring slot: `full`, an mbarrier on which every tile of a round arrives when its rows are in
// the slot (a generation of the slot = one phase; the E warps, which visit every round in order,
// wait on it suspended by the hardware, not spinning through the issue slots);
// and `drained`, a plain counter every E warp bumps when it has copied its rows out.  The
// way back is a COUNTER, not an mbarrier phase, on purpose: role A claims its tiles
// dynamically, so a warp may meet a slot it has not touched for several generations, and a
// parity wait can only tell the current phase from the one before it.
struct StreamShared {
  uint64_t full[kMaxSlots];
  volatile uint32_t drained[kMaxSlots];   // + 1 per E warp per use of the slot
  uint32_t next_item;   // role A: next (round, tile) of this CTA's sequence to be claimed
  // what role E needs to know about tile w of the round in slot s, published by the A warp that
  // produced it (before its arrival on `full`): .x = occupancy mask, .y = first slot row of the
  // tile | kMetaMine when the tile is this kernel's (inside the volume, not heavy)
  uint2 meta[kMaxSlots][kRoundTiles];
};
constexpr uint32_t kMetaMine = 0x80000000u;
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)),
               "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {   // release.cta
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::
               "r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {   // acquire.cta
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@!p bra W_%=;\n\t}" ::"r"(a), "r"(parity), "r"(20000u) : "memory");   // suspend <= 20 us per try
}

// Rows the round's tiles in front of tile w contribute to the slot (their occupied voxels; a
// heavy tile contributes none).  ts / occ: lane l < 17 holds tile_start of tile l, lane l < 16
// its mask.  `live_w`: tile w itself is this kernel's (not heavy).
__device__ __forceinline__ int rows_before(int32_t ts, uint32_t occ, int lane, int w,
                                           int32_t heavy_thr, bool& live_w) {
  const int32_t ts_next = __shfl_down_sync(0xffffffffu, ts, 1);
  const bool live = lane < kRoundTiles && (ts_next - ts) < heavy_thr;
  live_w = __shfl_sync(0xffffffffu, (int)live, w) != 0;
  return __reduce_add_sync(0xffffffffu, (live && lane < w) ? __popc(occ) : 0);
}

// ------------------------------------------------------------------------------------------
// role A: rows of the occupied voxels -> the CTA's ring.  A lane owns 2 consecutive channels.
// The tiles of the CTA's rounds are CLAIMED one by one from a shared counter (three stages
// ahead, when their index records start to travel), not dealt statically: a warp that draws a
// 90-point tile simply claims fewer, so a round is not held up by its slowest tile any longer
// than the ring's slack allows.  A tile's arrival on its round's `full` barrier is per tile.
// ------------------------------------------------------------------------------------------
constexpr int kHdrItem = 33;   // header word: the claimed item (round-in-CTA * 16 + tile-in-round)

__device__ __forceinline__ void role_rows(const FwdStreamParams& p, int32_t* ring_idx,
                                          StreamShared* sh, int lane) {
  __builtin_assume(__isShared(ring_idx));   // LDS/STS instead of generic accesses
  constexpr int U = 12;   // feature-row pieces in flight per lane (3 KB per warp)
  if (blockIdx.x >= p.n_rounds) return;
  const uint32_t my_rounds = (p.n_rounds - blockIdx.x + gridDim.x - 1) / gridDim.x;
  const uint32_t my_items = my_rounds * kRoundTiles;
  const int32_t heavy_thr = p.heavy ? max(__ldg(p.heavy + 1), kStreamHeavyMin) : 0x7fffffff;
  const uint32_t ns_mask = (1u << p.ns_log2) - 1u;
  float* const cta_ring = p.ring + ((size_t)blockIdx.x << p.ns_log2) * (kSlotRows * CU);
  const uint32_t row_bytes = (uint32_t)p.C * 4u;

  auto slot_of = [&](uint32_t k) { return ring_idx + (k & (kASlots - 1)) * kASlotInts; };
  // stage 1 of this warp's k-th item: claim it, start its round header
  auto issue_bounds = [&](uint32_t k) {
    int32_t* sl = slot_of(k);
    uint32_t g = 0;
    if (lane == 0) g = atomicAdd(&sh->next_item, 1u);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g < my_items) {
      const uint32_t t0 = (blockIdx.x + (g / kRoundTiles) * gridDim.x) * kRoundTiles;
      // 17 tile_start words (lanes 0..16) + 16 masks (lanes 17..31 and, for the last one, lane 16)
      if (lane <= kRoundTiles) cpa4(sl + lane, p.tile_start + min(t0 + lane, p.n_tiles));
      if (lane >= kRoundTiles) {
        const int wq = lane == kRoundTiles ? kRoundTiles - 1 : lane - kRoundTiles - 1;
        const uint32_t t = t0 + wq;
        if (t < p.n_tiles) cpa4(sl + 17 + wq, p.tile_occ + t);
        else sl[17 + wq] = 0;
      }
    } else {
      sl[lane] = 0;   // past the end: an empty item
      if (lane == 0) sl[32] = 0;
    }
    if (lane == 0) sl[kHdrItem] = (int32_t)g;
  };
  // the point range of the item's tile (none when the tile is heavy)
  auto tile_range = [&](const int32_t* sl, int32_t& s, int32_t& e) {
    const int w = sl[kHdrItem] & (kRoundTiles - 1);
    s = sl[w];
    e = sl[w + 1];
    if (e - s >= heavy_thr) e = s;
  };
  auto issue_ranks = [&](uint32_t k) {
    int32_t* sl = slot_of(k);
    int32_t* pt = sl + kAHdr + 4 * lane;
    int32_t s, e;
    tile_range(sl, s, e);
    const int32_t i = s + lane;
    if (i < e) {
      cpa4(pt + 0, p.ranks_bev + i);
      cpa4(pt + 1, p.ranks_feat + i);
      cpa4(pt + 2, p.ranks_depth + i);
    } else {
      pt[0] = -1;
    }
  };
  auto issue_depth = [&](uint32_t k) {   // depth gather + fix-up of the landed ranks
    int32_t* sl = slot_of(k);
    int32_t* pt = sl + kAHdr + 4 * lane;
    const int32_t rb = pt[0];
    if (rb >= 0) {
      cpa4(pt + 3, p.depth + pt[2]);
      const int32_t up = lane ? pt[-4] : -1;
      // byte offset of the feature row (a multiple of 256) | first point of its voxel
      pt[2] = (int32_t)(((uint32_t)pt[1] * row_bytes) | (rb != up ? 1u : 0u));
    }
  };

#pragma unroll
  for (int i = 0; i < 3 * kADist; ++i) issue_bounds(i);
  cpa_commit(); cpa_wait<0>(); __syncwarp();
#pragma unroll
  for (int i = 0; i < 2 * kADist; ++i) issue_ranks(i);
  cpa_commit(); cpa_wait<0>(); __syncwarp();
#pragma unroll
  for (int i = 0; i < kADist; ++i) issue_depth(i);
  cpa_commit(); cpa_wait<0>(); __syncwarp();

  const uint32_t lane_off = (uint32_t)lane * 8u;

  VEON_T0
  for (uint32_t k = 0;; ++k) {
    cpa_wait<kADist - 1>();
    __syncwarp();
    VEON_TACC(0)
    int32_t* sl = slot_of(k);
    const uint32_t g = (uint32_t)sl[kHdrItem];
    if (g >= my_items) break;   // claims only grow: everything this warp still holds is past the end
    const uint32_t m = g / kRoundTiles;
    const int w = (int)(g & (kRoundTiles - 1));
    int32_t s0, e0;
    tile_range(sl, s0, e0);
    bool live_w;
    const int base_row = rows_before(lane <= kRoundTiles ? sl[lane] : 0,
                                     lane < kRoundTiles ? (uint32_t)sl[17 + lane] : 0u, lane, w,
                                     heavy_thr, live_w);
    __syncwarp();               // the header has been read: its slot may be claimed again below
    issue_bounds(k + 3 * kADist);
    issue_ranks(k + 2 * kADist);
    issue_depth(k + kADist);
    cpa_commit();

    const uint32_t slot = m & ns_mask;
    const uint32_t gen = m >> p.ns_log2;
    // every earlier use of the slot has been read out by all E warps
    VEON_TACC(1)
    while (sh->drained[slot] < kEWarps * gen) __nanosleep(256);
    VEON_TACC(2)
    if (e0 > s0) {
      char* const slotb = reinterpret_cast<char*>(cta_ring + (size_t)slot * (kSlotRows * CU));
      const char* const featb = reinterpret_cast<const char*>(p.feat);
      // byte offset, inside the slot, of this lane's piece of the row being accumulated; the
      // first point always opens a voxel, so the -1 row is stepped over before any store
      uint32_t rowoff = (uint32_t)(base_row - 1) * (CU * 4) + lane_off;
      float acc[2] = {0.f, 0.f};
      for (int32_t base = s0; base < e0; base += 32) {
        const int cnt = min(32, e0 - base);
        if (base != s0) {
          // more than 32 points: the records of every 32-point piece but the prefetched
          // first one are fetched synchronously
          const int32_t i = base + lane;
          __syncwarp();
          int32_t rb = -1, rf = 0;
          float d = 0.f;
          if (i < e0) {
            rb = __ldg(p.ranks_bev + i);
            rf = __ldg(p.ranks_feat + i);
            d = __ldg(p.depth + __ldg(p.ranks_depth + i));
          }
          int32_t up = __shfl_up_sync(0xffffffffu, rb, 1);
          int32_t* pt = sl + kAHdr + 4 * lane;
          if (lane == 0) up = base == s0 ? -1 : sl[kAHdr + 4 * 31 + 0];   // last point before
          __syncwarp();
          pt[0] = rb;
          pt[2] = (int32_t)(((uint32_t)rf * row_bytes) | (rb != up ? 1u : 0u));
          pt[3] = __float_as_int(d);
          __syncwarp();
        }
        const int32_t* pts = sl + kAHdr + 2;   // record j: {row offset | first, depth} at pts[4 j]
        // Branch-free body: loads in groups of four (a group past the last point is skipped
        // as a whole, warp-uniformly), then one predicated fma chain per point; the running
        // sum is stored after EVERY point (the last store of a voxel leaves its total), which
        // costs L2 some repeated row writes and saves the flush branches.
        for (int j0 = 0; j0 < cnt; j0 += U) {
          int2 q[U];
          float2 f[U];
#pragma unroll
          for (int gq = 0; gq < U; gq += 4) {
            if (j0 + gq < cnt) {
#pragma unroll
              for (int uu = 0; uu < 4; ++uu) {
                const int u = gq + uu;
                q[u] = *reinterpret_cast<const int2*>(pts + 4 * min(j0 + u, cnt - 1));
                f[u] = __ldg(reinterpret_cast<const float2*>(featb + (((uint32_t)q[u].x & ~1u) + lane_off)));
              }
            }
          }
#pragma unroll
          for (int gq = 0; gq < U; gq += 4) {
            if (j0 + gq < cnt) {
#pragma unroll
              for (int uu = 0; uu < 4; ++uu) {
                const int u = gq + uu;
                const bool ok = j0 + u < cnt;
                const bool first = q[u].x & 1;
                const float dj = __int_as_float(q[u].y);
                rowoff += (ok && first) ? (uint32_t)(CU * 4) : 0u;
                acc[0] = ok ? fmaf(f[u].x, dj, first ? 0.f : acc[0]) : acc[0];
                acc[1] = ok ? fmaf(f[u].y, dj, first ? 0.f : acc[1]) : acc[1];
                if (ok) *reinterpret_cast<float2*>(slotb + rowoff) = make_float2(acc[0], acc[1]);
              }
            }
          }
        }
      }
    }
    // this tile's rows of the round are in the slot
    __syncwarp();
    VEON_TACC(3)
    if (lane == 0) {
      const uint32_t t = (blockIdx.x + m * gridDim.x) * kRoundTiles + w;
      sh->meta[slot][w] = make_uint2((uint32_t)sl[17 + w],
                                     (uint32_t)base_row | ((live_w && t < p.n_tiles) ? kMetaMine : 0u));
      mbar_arrive(&sh->full[slot]);   // release: the rows and the meta word are visible with it
    }
  }
  cpa_wait<0>();
}

// ------------------------------------------------------------------------------------------
// role E: ring -> dense volume.  Warp ew: tile ew of every round; group = ew / 8.
// ------------------------------------------------------------------------------------------
// staged row j of a tile: 8 chunks of 16 bytes, chunk k at position k ^ swz(j) so that the
// eight lanes of a store quad-row (eight different rows, same channel) hit different banks
__device__ __forceinline__ uint32_t e_swz(uint32_t j) { return (j ^ (j >> 2)) & 7u; }

// One E step = (round, 32-channel sub-chunk).  The steps are software-pipelined over two staging
// buffers: the copies of step i+1 (ring -> shared memory, L2 latency) are in flight while step i is
// written out, and the wait for role A's next round happens a step early.
struct ECursor {
  uint32_t m, sub;            // round of this CTA, sub-chunk
  uint32_t b, vt;             // sample and tile inside the sample of this warp's tile
  uint32_t occ;
  int base, n;
  bool mine;
};

__device__ __forceinline__ void role_expand(const FwdStreamParams& p, float* stage,
                                            StreamShared* sh, int lane, int ew) {
  constexpr int kSub = CU / kEChunk;
  constexpr uint32_t kBufBytes = kERows * kEChunk * 4;
  __builtin_assume(__isShared(stage));
  if (blockIdx.x >= p.n_rounds) return;
  const uint32_t my_rounds = (p.n_rounds - blockIdx.x + gridDim.x - 1) / gridDim.x;
  const uint32_t ns_mask = (1u << p.ns_log2) - 1u;
  const float* const cta_ring = p.ring + ((size_t)blockIdx.x << p.ns_log2) * (kSlotRows * CU);
  const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
  const int q4 = (lane & 7) * 4, r = lane >> 3;
  const int group = ew / kEGroup;
  const uint32_t t_step = gridDim.x * kRoundTiles;

  // zero rows (row 32 of both buffers; nothing is ever copied there)
  for (int i = lane; i < kEChunk; i += 32) {
    stage[32 * kEChunk + i] = 0.f;
    stage[kERows * kEChunk + 32 * kEChunk + i] = 0.f;
  }
  __syncwarp();

  auto start = [&](ECursor& c) {
    c.m = 0; c.sub = 0;
    const uint32_t t = blockIdx.x * kRoundTiles + ew;
    c.b = t / p.tiles_per_sample;
    c.vt = t - c.b * p.tiles_per_sample;
    c.occ = 0u; c.base = 0; c.n = 0; c.mine = false;
  };
  auto advance = [&](ECursor& c) {
    if (++c.sub < (uint32_t)kSub) return;
    c.sub = 0;
    ++c.m;
    c.vt += t_step;
    while (c.vt >= p.tiles_per_sample) {
      c.vt -= p.tiles_per_sample;
      ++c.b;
    }
  };
  // start the copies of the cursor's step into buffer `buf`
  auto issue = [&](ECursor& c, uint32_t buf) {
    const uint32_t slot = c.m & ns_mask;
    if (c.sub == 0) {
      // Role A has put the round's rows into the slot.  EVERY E warp waits here, also one whose
      // tile is empty: no E warp may run a slot generation ahead of the others (its tick on
      // `drained` would be taken for a slower warp's).
      mbar_wait(&sh->full[slot], (c.m >> p.ns_log2) & 1u);
      // what role A published about this warp's tile
      const uint2 mt = sh->meta[slot][ew];
      c.occ = mt.x;
      c.base = (int)(mt.y & ~kMetaMine);
      c.mine = (mt.y & kMetaMine) != 0u;
      c.n = __popc(c.occ);
    }
    if (c.mine && c.n > 0) {
      const float* src = cta_ring + (size_t)slot * (kSlotRows * CU) + (size_t)c.base * CU +
                         c.sub * kEChunk + (lane & 7) * 4;
      const uint32_t dst = stage_s + buf * kBufBytes;
      for (int j = lane >> 3; j < c.n; j += 4)
        cpa16_cg(dst + (uint32_t)j * (kEChunk * 4) + ((((uint32_t)lane & 7u) ^ e_swz(j)) << 4),
                 src + (size_t)j * CU);
    }
    cpa_commit();
  };

  const uint32_t n_steps = my_rounds * kSub;
  ECursor wc, ic;     // step being written, step whose copies are issued next
  start(wc);
  start(ic);
  static_assert(kSub >= 2, "the issue cursor must still be on the write cursor's tile one step on");
  VEON_T0
  issue(ic, 0);
  wc.occ = ic.occ; wc.base = ic.base; wc.n = ic.n; wc.mine = ic.mine;
  uint32_t rel[4] = {0u, 0u, 0u, 0u};
  for (uint32_t st = 0; st < n_steps; ++st) {
    const uint32_t buf = st & 1u;
    VEON_TACC(0)
    // this step's copies (issued a step ago) have landed; the slot is released BEFORE the wait
    // for role A's next round: an A warp may be blocked on exactly this slot while other tiles
    // of the next round are still unclaimed (tiles are claimed dynamically)
    cpa_wait<0>();
    __syncwarp();
    if (wc.sub == (uint32_t)kSub - 1 && lane == 0)   // slot needed no more
      atomicAdd(const_cast<uint32_t*>(&sh->drained[wc.m & ns_mask]), 1u);
    VEON_TACC(2)
    if (st + 1 < n_steps) {   // the next step's copies fly during the barrier and the write-out
      advance(ic);
      issue(ic, buf ^ 1u);    // (a new tile's meta stays in `ic` until the write cursor gets there)
    }
    VEON_TACC(1)
#ifndef VEON_FWD_NO_LOCKSTEP
    // the group's 8 tiles are written together: aligned 1 KB runs per channel plane
    if (group == 0) asm volatile("bar.sync 1, %0;" ::"n"(kEGroup * 32) : "memory");
    else asm volatile("bar.sync 2, %0;" ::"n"(kEGroup * 32) : "memory");
#endif
    VEON_TACC(3)
    if (wc.sub == 0) {
      // offset of channel r of the staged row of each of this lane's four voxels inside a
      // buffer, the row's swizzle folded in; the zero row for empty voxels
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int v = q4 + i;
        const bool set = (wc.occ >> v) & 1u;
        const uint32_t j = set ? (uint32_t)__popc(wc.occ & ((1u << v) - 1u)) : 32u;
        rel[i] = j * (kEChunk * 4) + (uint32_t)r * 4u;
        if (set) rel[i] ^= e_swz(j) << 4;
      }
    }
    if (wc.mine) {
      float* o = p.out + ((int64_t)wc.b * p.C + wc.sub * kEChunk + r) * p.V +
                 wc.vt * kTileVoxels + q4;
      const int64_t ostep = 4 * p.V;
      if (wc.n == 0) {
#pragma unroll 4
        for (int k = 0; k < kEChunk / 4; ++k, o += ostep)
          st_stream4(o, make_float4(0.f, 0.f, 0.f, 0.f));
      } else {
        const uint32_t bs = stage_s + buf * kBufBytes;
#pragma unroll
        for (int k0 = 0; k0 < kEChunk / 4; k0 += 4) {   // 16 loads in flight, then 4 stores
          float4 v4[4];
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint32_t x = (uint32_t)((k0 + kk) << 4);
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v4[kk].x) : "r"(bs + (rel[0] ^ x)));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v4[kk].y) : "r"(bs + (rel[1] ^ x)));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v4[kk].z) : "r"(bs + (rel[2] ^ x)));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v4[kk].w) : "r"(bs + (rel[3] ^ x)));
          }
#pragma unroll
          for (int kk = 0; kk < 4; ++kk, o += ostep) st_stream4(o, v4[kk]);
        }
      }
    }
    __syncwarp();   // this buffer is refilled by the step after next
    VEON_TACC(4)
    // move the write cursor; a new tile takes over the meta the issue cursor has read
    advance(wc);
    if (wc.sub == 0) { wc.occ = ic.occ; wc.base = ic.base; wc.n = ic.n; wc.mine = ic.mine; }
  }
}

__global__ void __launch_bounds__(kStreamWarps * 32, 1)
k_fwd_stream(const FwdStreamParams p) {
  extern __shared__ __align__(16) float fs_smem_raw[];
  __shared__ StreamShared sh;
  // the E staging addresses are formed with XORs on bits 4..7: 256-byte aligned base
  float* fs_smem = reinterpret_cast<float*>(
      (reinterpret_cast<uintptr_t>(fs_smem_raw) + 255) & ~(uintptr_t)255);
  pdl_launch_dependents();   // the heavy-tile grid may be queued behind this one
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < kMaxSlots) {
    mbar_init(&sh.full[threadIdx.x], kRoundTiles);   // one arrival per tile of the round
    sh.drained[threadIdx.x] = 0;
  }
  if (threadIdx.x == 0) sh.next_item = 0;
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  constexpr int kEStageFloats = kEWarps * 2 * kERows * kEChunk;
  if (warp < kAWarps) {
    reg_inc<kARegs>();
    role_rows(p, reinterpret_cast<int32_t*>(fs_smem + kEStageFloats) + warp * (kASlots * kASlotInts),
              &sh, lane);
  } else {
    reg_dec<kERegs>();
    const int ew = warp - kAWarps;
    role_expand(p, fs_smem + ew * 2 * kERows * kEChunk, &sh, lane, ew);
  }
}

bool fwd_stream_supported(int B, int C, int64_t V, const void* feat, const void* out,
                          int64_t n_feat_rows) {
  if (V % kTileVoxels != 0) return false;
  // 64-channel rows only: there the kernel wins (318 vs 337 us at C2); wider rows at VEON's point
  // density were faster through the general kernel (B200, round 2: 1.15-1.5 ms vs 1.10 ms for a
  // 2.6 GB volume)
  if (C != 64) return false;
  if (((uintptr_t)feat | (uintptr_t)out) & 15) return false;
  if ((int64_t)B * V > 0x7fffffffLL || n_feat_rows * (int64_t)C > 0x3fffffffLL) return false;
  return true;
}

static int launch_stream_kernel(FwdStreamParams& p, size_t ring_bytes, cudaStream_t stream) {
  const size_t smem = sizeof(float) * kEWarps * 2 * kERows * kEChunk +
                      sizeof(int32_t) * kAWarps * kASlots * kASlotInts + 256;
  static int per_sm[kMaxDevices] = {};
  const int dev = current_device();
  if (per_sm[dev] == 0) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(k_fwd_stream,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int n = 0;
    VEON_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_fwd_stream,
                                                                kStreamWarps * 32, smem));
    per_sm[dev] = n > 0 ? n : -1;
  }
  if (per_sm[dev] < 1) return VEON_E_UNSUPPORTED;
  int64_t grid = sm_count();
  if (grid > p.n_rounds) grid = p.n_rounds;
  // ring slots per CTA from what the caller gave us
  const size_t slot_bytes = sizeof(float) * kSlotRows * CU;
  const int64_t ns = (int64_t)(ring_bytes / ((size_t)grid * slot_bytes));
  if (ns < 2) return VEON_E_WORKSPACE;
  p.ns_log2 = 1;   // the largest power of two that fits, at most kMaxSlots
  while ((2 << p.ns_log2) <= ns && (2 << p.ns_log2) <= kMaxSlots) ++p.ns_log2;
  k_fwd_stream<<<(unsigned)grid, kStreamWarps * 32, smem, stream>>>(p);
  VEON_LAUNCH_CHECK();
  return 0;
}

size_t fwd_stream_workspace_bytes(int C) {
  // (SM count of the current device) x 8 slots = 148 x 1 MB; no ring where the kernel is not used
  if (C != 64) return 0;
  return (size_t)sm_count_total() * 8 * sizeof(float) * kSlotRows * CU;
}

int launch_fwd_stream(const float* depth, const float* feat, const int32_t* rd, const int32_t* rf,
                      const int32_t* rb, const int32_t* tile_start, const uint32_t* tile_occ,
                      const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                      float* out, void* workspace, size_t ws_bytes, cudaStream_t stream) {
  const int64_t tps = V / kTileVoxels, n_tiles = (int64_t)B * tps;
  if (!workspace || ((uintptr_t)workspace & 255)) return VEON_E_WORKSPACE;
  FwdStreamParams p;
  p.depth = depth; p.feat = feat; p.ranks_depth = rd; p.ranks_feat = rf; p.ranks_bev = rb;
  p.tile_start = tile_start; p.tile_occ = tile_occ; p.heavy = heavy;
  p.ring = reinterpret_cast<float*>(workspace);
  p.out = out; p.V = V; p.n_tiles = (uint32_t)n_tiles;
  p.n_rounds = (uint32_t)ceil_div64(n_tiles, kRoundTiles);
  p.tiles_per_sample = (uint32_t)tps;
  p.C = C; p.ns_log2 = 1;
  int rc = launch_stream_kernel(p, ws_bytes, stream);
  if (rc) return rc;
  if (heavy) return launch_heavy_behind(depth, feat, rd, rf, rb, tile_start, heavy, heavy_ints, B, C,
                                        V, out, kStreamHeavyMin, stream);
  return 0;
}

}  // namespace veon

#ifdef VEON_FWD_TRACE
extern "C" int veon_internal_fwd_trace(unsigned long long* host_out, int clear) {
  if (clear) {
    static unsigned long long zeros[32 * 8] = {};
    return (int)cudaMemcpyToSymbol(veon::veon_fwd_trace, zeros, sizeof(zeros));
  }
  return (int)cudaMemcpyFromSymbol(host_out, veon::veon_fwd_trace, sizeof(unsigned long long) * 32 * 8);
}
#endif
