// Open-vocabulary tail on the 5th-generation tensor cores (tcgen05 + TMEM).
//
//   logits[v, q] = sum_c feat_occ[b, c, v] * W[q, c]      san_in_veon_temporal.py:257-259
//   per-class max over prompts, first-index argmax         san_in_veon_entry_temporal.py:273-297
//   occupancy gate, free label, [B,X,Y,Z] uint8            veon_temporal.py:223-229,240
//
// GEMM view per CTA tile: M = 128 voxels, N = padded prompt count, K = C.
//   * A = feat tile, from TENSOR MEMORY (tcgen05.mma with a TMEM A operand: lanes = voxels, one
//     32-bit column per channel).  In HBM the voxel index is contiguous, so a thread that owns
//     a voxel reads a COLUMN of the tile: loader warps bring the raw [32 channels][128 voxels]
//     block into a shared-memory ring with 16-byte cp.async copies (completion on the slot's
//     mbarrier; nothing in registers, ~112 KB in flight per SM), converter threads read their
//     column (conflict-free), split it and write hi and lo with tcgen05.st.  The tensor core
//     therefore never reads A through the shared-memory pipe, which carries 128 + 128
//     wavefronts per stage instead of the 128 (LDG) + 256 (STS hi/lo) + 256 (MMA reads) of the
//     round-1 kernel that kept A in shared memory (MN-major SWIZZLE_128B_BASE32B).
//   * B = W, K-major SW128, from shared memory: k_w_image splits W once per call into a global
//     image laid out chunk by chunk exactly like a stage's [W_hi ; W_lo] block, and one lane
//     copies a chunk per stage with a 1-D bulk copy that completes on the stage's `full` barrier.
//   * D in TMEM (fp32), two accumulator buffers so the epilogue of tile i overlaps the main
//     loop of tile i+1.
//   * fp32 fidelity: 3xTF32.  a = a_hi + a_lo, w = w_hi + w_lo with *_hi exactly
//     TF32-representable; every (voxel, prompt) column accumulates a_hi*w_hi + a_hi*w_lo +
//     a_lo*w_hi.  Error ~2^-21 relative, which is what keeps the labels at >= 99.99 %
//     agreement (plain TF32 would flip ~0.3 % of near-tie voxels).
//   * The MMA warp runs its loop warp-uniformly and an elected lane issues, so descriptors and
//     tensor-memory addresses stay in uniform registers (see the note in that role).
// Warp roles (23 warps): 0-15 converters, 16 MMA issuer (+TMEM alloc), 17-20 epilogue,
// 21-22 loaders.
//
// bfloat16 features (T = bf16): a widened bfloat16 value is exactly TF32-representable, so
// a_hi = a and a_lo = 0 and the third product of every 3xTF32 sum is exactly zero.  That
// instance reads half the bytes ([KC][TM] bf16 raw tiles, twice as many in flight), writes one
// tensor-memory column per channel (no lo half) and issues a*w_hi + a*w_lo per K-step: the
// float32 instance's sums on x.float(), bit for bit.
//
// Channels-last features (CL = true, feat_occ [B,Z,Y,X,C]): a voxel's 32 channels of a stage are
// one contiguous 128-byte (bfloat16: 64-byte) segment.  The loaders copy those segments into a
// voxel-major raw tile [TM][KC] of T whose 16-byte pieces are XOR-swizzled by voxel, and a
// converter thread reads its voxel's kRows channels with 16-byte loads, conflict-free.  From the
// registers on nothing changes: the same values go to the same tensor-memory lanes and columns and
// the MMAs are the same, so a channels-last volume gives the bits of its contiguous copy.
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace veon {
namespace tc {

constexpr int KC = 32;        // channels per pipeline stage = 4 UMMA K-steps of 8 (tf32)
constexpr int TM = 128;       // voxels per tile = UMMA M
constexpr int kProdWarps = 16;  // warp % 4 = TMEM lane quarter (32 voxels), warp / 4 = channel group
constexpr int kRows = KC / 4;   // channels of a stage per producer thread
constexpr uint32_t kTmemCols = 512;
constexpr int kMmaWarp = 16;
// warps 17..20: epilogue (warp % 4 = 1,2,3,0 -> the four TMEM lane quarters)
constexpr int kLoadWarp0 = 21;  // 21, 22: loaders
constexpr int kLoadWarps = 2;
constexpr int kWarps = 23;
constexpr int kMaxStages = 6;
// per element type T of the features: raw tiles [KC][TM] of T, ~112 KB in flight per SM either way
template <typename T> constexpr int kRawOf = 7 * 4 / (int)sizeof(T);            // 7 (f32), 14 (bf16)
template <typename T> constexpr uint32_t kRawBytesOf = KC * TM * sizeof(T);     // 16 KB, 8 KB
template <typename T> constexpr int kVec = 16 / (int)sizeof(T);   // voxels per 16-byte copy
// tensor-memory columns of one operand slot: a_hi and a_lo (f32), a alone (bf16)
template <typename T> constexpr int kSlotCols = sizeof(T) == 4 ? 2 * KC : KC;
// channels-last raw tiles: one row of KC channels per voxel, kPieces 16-byte pieces (8 f32, 4 bf16)
template <typename T> constexpr int kPieces = KC * (int)sizeof(T) / 16;
// where piece j of voxel row v sits in its row: the 8 lanes of a quarter-warp phase (8 consecutive
// voxels, one piece index) land on 8 distinct 16-byte positions of a 128-byte line.  f32: one row
// per line, j ^ (v & 7); bf16: two rows per line, j ^ ((v >> 1) & 3).
template <typename T> __device__ __forceinline__ uint32_t cl_piece(int j, int v) {
  return (uint32_t)(j ^ ((v / (8 / kPieces<T>)) & (kPieces<T> - 1)));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
#ifndef VEON_TAIL_SUSPEND_NS
#define VEON_TAIL_SUSPEND_NS 0
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  do {  // try_wait suspends the thread in hardware for a bounded time, so this is not a hot spin
#if VEON_TAIL_SUSPEND_NS > 0
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"((uint32_t)VEON_TAIL_SUSPEND_NS)
        : "memory");
#else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
#endif
  } while (!done);
}
__device__ __forceinline__ bool elect_one() {   // one lane of the (converged) warp
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// completion of all previously issued MMAs of this thread -> one arrival on `bar`
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// 32 lanes x 16 consecutive columns -> 16 registers per thread (thread i <-> lane base+i)
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, "
      "%12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, version 1):
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version 1<<46 | layout type [61,64)
constexpr uint64_t kSw128 = 2;         // SWIZZLE_128B         (B operand, K-major)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes,
                                              uint32_t sbo_bytes, uint64_t layout_type) {
  return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46) | (layout_type << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=tf32, A (tensor memory)
// and B K-major, M=128, N=n
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(TM >> 4) << 24);
}

__device__ __forceinline__ float tf32_hi(float x) {  // exactly TF32-representable part
  return __uint_as_float(__float_as_uint(x) & 0xffffe000u);
}

struct Params {
  const void* feat;      // [B,C,V] of T; channels-last instances: [B,V,C]
  const float* w_image;  // k_w_image's output
  const int32_t* cls;    // [Q]
  const float* bin_occ;  // [B,2,V]
  uint8_t* labels;       // [B,X,Y,Z]
  float* logits;         // LOGITS variant: sem_occ [B,Q,V] instead of labels
  int B, C, Q, Z, Y, X, npad, stages, free_label;
  int64_t V;
};

// [W_hi ; W_lo] of every 32-channel chunk in the shared-memory layout of a stage's W block:
// row n (prompt) of the chunk = 128 B at (n/8)*1024 + (n%8)*128, its 16-byte pieces XOR-swizzled
// by n%8; the lo rows follow the npad hi rows.  Rows >= Q are zero.
__global__ void k_w_image(const float* __restrict__ w, int Q, int C, int npad, float* __restrict__ image) {
  const int n_chunks = C / KC;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_chunks * npad * 8) return;
  const int j4 = (int)(idx & 7), n = (int)((idx >> 3) % npad), ch = (int)((idx >> 3) / npad);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (n < Q) v = __ldg(reinterpret_cast<const float4*>(w + (int64_t)n * C + ch * KC) + j4);
  float4 hi, lo;
  hi.x = tf32_hi(v.x); hi.y = tf32_hi(v.y); hi.z = tf32_hi(v.z); hi.w = tf32_hi(v.w);
  lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
  uint8_t* blk = reinterpret_cast<uint8_t*>(image) + (size_t)ch * (2 * npad * KC * 4);
  const uint32_t off = (uint32_t)(n >> 3) * 1024u + (uint32_t)(n & 7) * 128u + (uint32_t)((j4 ^ (n & 7)) << 4);
  *reinterpret_cast<float4*>(blk + off) = hi;
  *reinterpret_cast<float4*>(blk + off + (uint32_t)npad * 128u) = lo;
}

#ifdef VEON_TAIL_TRACE   // tools/tail_trace.py only: cycles per phase, CTA 0, every warp
__device__ unsigned long long veon_tail_trace[32 * 8];
#define VEON_T0 long long _tt = clock64(), _ta[4] = {0, 0, 0, 0};
#define VEON_TACC(slotid)          \
  {                                \
    const long long _n = clock64(); \
    _ta[slotid] += _n - _tt;       \
    _tt = _n;                      \
  }
#define VEON_TEND                                                                   \
  if (blockIdx.x == 0 && (threadIdx.x & 31) == 0)                                   \
    for (int _i = 0; _i < 4; ++_i) veon_tail_trace[(threadIdx.x >> 5) * 8 + _i] = _ta[_i];
#else
#define VEON_T0
#define VEON_TACC(slotid)
#define VEON_TEND
#endif

// 32 lanes x 8 consecutive columns <- 8 registers per thread (thread i <-> lane base+i)
__device__ __forceinline__ void tc_st8(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
      "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
      "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
      : "memory");
}
// A from tensor memory (lanes = rows, one 32-bit column per K element), B from shared memory
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}

// a bfloat16 feature widened for the A operand.  The float32 route splits an infinite a into
// hi = a, lo = a - a = NaN, so every logit it touches is NaN; without a lo half the same
// logits would be +-inf, so an infinity is widened to a NaN instead (same NaN positions).
__device__ __forceinline__ float widen_operand(uint16_t h) {
  const uint32_t x = (uint32_t)h << 16;
  return __uint_as_float((x << 1) == 0xff000000u ? 0x7fc00000u : x);
}

// Tensor-memory map (all 512 columns): [0, 2*npad) two accumulator buffers of npad columns
// (every (voxel, prompt) sum lives in ONE column: a_hi*w_hi + a_hi*w_lo + a_lo*w_hi), then
// `stages` operand slots of kSlotCols<T> columns: a_hi (KC columns, one per channel) and a_lo,
// or for bfloat16 features a alone.
// Shared memory holds only the W ring: one [W_hi ; W_lo] block per stage.
// LOGITS: the epilogue stores the raw logits (semantic_inference_3d alone) instead of labels.
// CL: feat is channels-last [B,V,C]; only the loaders and the converters' shared-memory reads
// differ (raw tiles [TM][KC] of T, swizzled by cl_piece).
template <bool LOGITS, typename T, bool CL = false>
__global__ void __launch_bounds__(kWarps * 32, 1) k_tail_tc(const Params p) {
  constexpr int kRaw = kRawOf<T>;
  constexpr uint32_t kRawBytes = kRawBytesOf<T>;
  constexpr uint32_t kSlot = (uint32_t)kSlotCols<T>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int npad = p.npad, stages = p.stages;
  const uint32_t w_bytes = 2 * npad * KC * 4;    // [W_hi ; W_lo] chunk
  uint8_t* raw_base = smem_raw;                                  // [kRaw] raw tiles [KC][TM] of T
  uint8_t* stage_base = smem_raw + (size_t)kRaw * kRawBytes;     // [stages] W blocks
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_base + (size_t)stages * w_bytes);
  uint64_t* full = bars;                  // [stages]   converters + W copy -> MMA
  uint64_t* empty = bars + kMaxStages;    // [stages]   MMA -> converters
  uint64_t* acc_full = bars + 2 * kMaxStages;   // [2]  MMA -> epilogue
  uint64_t* acc_empty = acc_full + 2;           // [2]  epilogue -> MMA
  uint64_t* raw_full = acc_empty + 2;           // [kRaw] loader (bulk copies) -> converters
  uint64_t* raw_empty = raw_full + kRaw;        // [kRaw] converters -> loader
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + kRaw);

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(full + s, kProdWarps + 1);   // + the expect_tx arrival of the W copy
      mbar_init(empty + s, 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(acc_full + a, 1); mbar_init(acc_empty + a, 4); }
    for (int r = 0; r < kRaw; ++r) { mbar_init(raw_full + r, 32 * kLoadWarps); mbar_init(raw_empty + r, kProdWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {  // TMEM allocation is warp-wide
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t a_base = tmem_base + 2u * (uint32_t)npad;   // first operand slot

  const int64_t vtiles = (p.V + TM - 1) / TM;
  const int64_t n_tiles = (int64_t)p.B * vtiles;
  const int n_chunks = p.C / KC;
#ifdef VEON_TAIL_BLOCKED   // experiment: a contiguous run of tiles per CTA instead of a grid stride
  const int64_t per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
  const int64_t tile_begin = (int64_t)blockIdx.x * per_cta, tile_step = 1;
  const int64_t tile_end = tile_begin + per_cta < n_tiles ? tile_begin + per_cta : n_tiles;
  const int64_t my_tiles = tile_end > tile_begin ? tile_end - tile_begin : 0;
#else
  const int64_t tile_begin = blockIdx.x, tile_step = gridDim.x, tile_end = n_tiles;
  const int64_t my_tiles = (n_tiles > (int64_t)blockIdx.x)
                               ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
#endif
  const int64_t n_stages_total = my_tiles * n_chunks;

  if (warp >= kLoadWarp0) {
    // ============================ LOADERS ============================
    // 16-byte cp.async copies, a warp-instruction per 512-byte row segment (128 voxels of one
    // channel plane; for bfloat16 two rows of 256 bytes, 16 lanes each), completion reported to
    // the raw slot's barrier.  Nothing passes through registers, so the bytes in flight are
    // bounded only by the raw ring (kRaw x kRawBytes, ~112 KB per SM).
    // (One 512-byte bulk copy per row instead: 77 cycles per copy, 1.9 TB/s in all.)
    if constexpr (CL) {
      // channels-last: kPieces lanes per voxel segment (KC channels of one voxel), 32 / kPieces
      // voxels per warp-instruction, so the instruction count per stage is the channels-first one
      constexpr int kVoxPerCopy = 32 / kPieces<T>;
      constexpr int kVoxStep = kLoadWarps * kVoxPerCopy;
      constexpr int kRowBytes = KC * (int)sizeof(T);
      const int lw = warp - kLoadWarp0;
      const int vox = lw * kVoxPerCopy + lane / kPieces<T>;  // voxels vox, vox + kVoxStep, ...
      const int piece = lane % kPieces<T>;
      const T* feat = static_cast<const T*>(p.feat) + piece * kVec<T>;
      uint32_t rs = 0, rphase = 0;
      bool first_round = true;
      for (int64_t tile = tile_begin; tile < tile_end; tile += tile_step) {
        const int64_t b = tile / vtiles;
        const int64_t v0 = (tile - b * vtiles) * TM + vox;
        for (int ch = 0; ch < n_chunks; ++ch) {
          if (!first_round) mbar_wait(raw_empty + rs, rphase);
          const uint32_t dst = smem_u32(raw_base + (size_t)rs * kRawBytes);
#ifndef VEON_TAIL_X_NOLOAD
#pragma unroll
          for (int r = 0; r < TM / kVoxStep; ++r) {
            const int vl = vox + r * kVoxStep;
            const int64_t v = v0 + r * kVoxStep;
            const uint32_t nbytes = v < p.V ? 16u : 0u;   // past the end: zero-fill
            const T* src = feat + ((int64_t)b * p.V + (v < p.V ? v : 0)) * p.C + ch * KC;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(
                             dst + (uint32_t)(vl * kRowBytes) + (cl_piece<T>(piece, vl) << 4)),
                         "l"(src), "r"(nbytes)
                         : "memory");
          }
#endif
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(raw_full + rs))
                       : "memory");
          if (++rs == kRaw) {
            rs = 0;
            if (first_round) first_round = false; else rphase ^= 1;
          }
        }
      }
      asm volatile("cp.async.wait_all;" ::: "memory");
    } else {
      constexpr int kRowLanes = TM / kVec<T>;                  // lanes per channel row: 32, 16
      constexpr int kRowsPerCopy = 32 / kRowLanes;             // channel rows per warp-instruction
      constexpr int kRowStep = kLoadWarps * kRowsPerCopy;
      const int lw = warp - kLoadWarp0;
      const int row = lw * kRowsPerCopy + lane / kRowLanes;    // rows row, row + kRowStep, ...
      const int seg = lane % kRowLanes;                        // 16-byte piece of the row
      uint32_t rs = 0, rphase = 0;
      bool first_round = true;
      for (int64_t tile = tile_begin; tile < tile_end; tile += tile_step) {
        const int64_t b = tile / vtiles;
        const int64_t v = (tile - b * vtiles) * TM + kVec<T> * seg;
        const uint32_t nbytes = v < p.V ? 16u : 0u;           // V % kVec == 0; past the end: zero-fill
        const T* src = static_cast<const T*>(p.feat) + ((int64_t)b * p.C + row) * p.V + (v < p.V ? v : 0);
        for (int ch = 0; ch < n_chunks; ++ch, src += (int64_t)KC * p.V) {
          if (!first_round) mbar_wait(raw_empty + rs, rphase);
          const uint32_t dst = smem_u32(raw_base + (size_t)rs * kRawBytes) +
                               (uint32_t)(row * TM * (int)sizeof(T) + seg * 16);
#ifndef VEON_TAIL_X_NOLOAD
#pragma unroll
          for (int r = 0; r < KC / kRowStep; ++r)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(
                             dst + (uint32_t)(r * kRowStep * TM * (int)sizeof(T))),
                         "l"(src + (int64_t)r * kRowStep * p.V), "r"(nbytes)
                         : "memory");
#endif
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(raw_full + rs))
                       : "memory");
          if (++rs == kRaw) {
            rs = 0;
            if (first_round) first_round = false; else rphase ^= 1;
          }
        }
      }
      asm volatile("cp.async.wait_all;" ::: "memory");
    }
  } else if (warp < kProdWarps) {
    // ============================ CONVERTERS ============================
    // thread <-> voxel (TMEM lane 32*quarter + lane; a warp reaches only the lanes of warp % 4),
    // warp / 4 = which 8 of the stage's 32 channels.  Column reads of the raw tile are
    // conflict-free (lanes = consecutive voxels); the values go hi/lo-split (bfloat16: widened)
    // from registers straight into tensor memory, so the tensor core never reads A from shared
    // memory.
    const int quarter = warp & 3, grp = warp >> 2;
    const uint32_t lane_field = (uint32_t)(32 * quarter) << 16;
    using Raw = typename std::conditional<sizeof(T) == 4, float, uint16_t>::type;
    const Raw* raw_col = reinterpret_cast<const Raw*>(raw_base) + (kRows * grp) * TM + 32 * quarter + lane;
    // channels-last: this voxel's row of the [TM][KC] tile and the pieces holding its kRows
    // channels (two for f32, one for bf16)
    const int cl_vox = 32 * quarter + lane;
    const uint32_t cl_row = (uint32_t)(cl_vox * KC * (int)sizeof(T));
    const uint32_t cl_off0 = cl_row + (cl_piece<T>(kRows * grp * (int)sizeof(T) / 16, cl_vox) << 4);
    const uint32_t cl_off1 = cl_row + (cl_piece<T>(kRows * grp * (int)sizeof(T) / 16 + 1, cl_vox) << 4);
    uint32_t s = 0, phase = 0;     // operand slot and the parity its `empty` barrier completes next
    uint32_t rs = 0, rphase = 0;   // raw slot and the parity its `raw_full` barrier completes next
    bool first_round = true;
    int sch = 0;
    VEON_T0
    for (int64_t k = 0; k < n_stages_total; ++k) {
      mbar_wait(raw_full + rs, rphase);
      VEON_TACC(0)
      float hi[kRows], lo[kRows];
      if constexpr (CL) {
        const uint8_t* tile = raw_base + (size_t)rs * kRawBytes;
        if constexpr (sizeof(T) == 4) {
          const float4 x0 = *reinterpret_cast<const float4*>(tile + cl_off0);
          const float4 x1 = *reinterpret_cast<const float4*>(tile + cl_off1);
          const float a[kRows] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
          for (int i = 0; i < kRows; ++i) {
            hi[i] = tf32_hi(a[i]);
            lo[i] = a[i] - hi[i];
          }
        } else {
          const uint4 x = *reinterpret_cast<const uint4*>(tile + cl_off0);
          const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int i = 0; i < kRows; ++i) hi[i] = widen_operand((uint16_t)(w[i / 2] >> (16 * (i & 1))));
        }
      } else {
        const Raw* col = raw_col + (size_t)rs * (kRawBytes / sizeof(Raw));
#pragma unroll
        for (int i = 0; i < kRows; ++i) {
          if constexpr (sizeof(T) == 4) {
            const float a = col[i * TM];
            hi[i] = tf32_hi(a);
            lo[i] = a - hi[i];
          } else {
            hi[i] = widen_operand(col[i * TM]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(raw_empty + rs);   // the values are in registers
      if (++rs == kRaw) { rs = 0; rphase ^= 1; }
      VEON_TACC(2)
      if (!first_round) {
        mbar_wait(empty + s, phase);
        tc_fence_after();
      }
      VEON_TACC(1)
      if (threadIdx.x == 0) {   // this stage's [W_hi ; W_lo] block: one bulk copy, L2-resident source
        const uint32_t bar = smem_u32(full + s);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(w_bytes)
                     : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32(stage_base + (size_t)s * w_bytes)),
            "l"(reinterpret_cast<const uint8_t*>(p.w_image) + (size_t)sch * w_bytes), "r"(w_bytes), "r"(bar)
            : "memory");
      }
      if (++sch == n_chunks) sch = 0;
      const uint32_t slot = a_base + s * kSlot + lane_field + (uint32_t)(kRows * grp);
      tc_st8(slot, hi);
      if constexpr (sizeof(T) == 4) tc_st8(slot + KC, lo);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(full + s);
      VEON_TACC(3)
      if (++s == (uint32_t)stages) {
        s = 0;
        if (first_round) first_round = false; else phase ^= 1;
      }
    }
    VEON_TEND
  } else if (warp == kMmaWarp) {
    // ============================ MMA ISSUER ============================
    // The whole warp runs this loop and one elected lane issues: with warp-uniform control flow
    // the descriptors and tensor-memory addresses live in uniform registers.  (Inside an
    // `if (lane == 0)` branch every tcgen05.mma was wrapped in an ELECT / 4 x R2UR / branch
    // loop, ~75 cycles per instruction: the issuing thread, not the tensor pipe, set the pace.)
    {
      const uint32_t idesc = make_idesc(npad);
      const uint32_t w_lo_off = (uint32_t)npad * 128u;   // the lo rows follow the npad hi rows
      const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t a0 = tmem0 + 2u * (uint32_t)npad;
      const uint32_t sw0 = smem_u32(stage_base);
      const bool leader = elect_one();
      uint32_t s = 0, fphase = 0, tcount = 0;
      VEON_T0
      for (int64_t tile = tile_begin; tile < tile_end; tile += tile_step, ++tcount) {
        const uint32_t acc = tcount & 1;
        const uint32_t around = tcount >> 1;
        if (around > 0) mbar_wait(acc_empty + acc, (around - 1) & 1);
        tc_fence_after();
        VEON_TACC(0)
        const uint32_t d = tmem0 + acc * (uint32_t)npad;
        for (int ch = 0; ch < n_chunks; ++ch) {
          mbar_wait(full + s, fphase);
          tc_fence_after();
          VEON_TACC(1)
          const uint32_t sw = sw0 + s * w_bytes;
          const uint32_t a_hi = a0 + s * kSlot, a_lo = a_hi + KC;
#ifndef VEON_TAIL_X_NOMMA
#pragma unroll
          for (int k = 0; k < KC / 8; ++k) {
            const uint64_t w_hi = make_desc(sw + k * 32, 16, 1024, kSw128);
            const uint64_t w_lo = make_desc(sw + w_lo_off + k * 32, 16, 1024, kSw128);
            if (leader) {
              tc_mma_tf32_ts(d, a_hi + 8 * k, w_hi, idesc, (ch > 0 || k > 0) ? 1u : 0u);
              tc_mma_tf32_ts(d, a_hi + 8 * k, w_lo, idesc, 1u);
              // bfloat16: a_lo = 0, every product of the third MMA is zero and it is not issued
              if constexpr (sizeof(T) == 4) tc_mma_tf32_ts(d, a_lo + 8 * k, w_hi, idesc, 1u);
            }
          }
#endif
          if (leader) tc_commit(empty + s);  // operand slot + W block reusable once these MMAs have read them
          __syncwarp();
          VEON_TACC(2)
          if (++s == (uint32_t)stages) { s = 0; fphase ^= 1; }
        }
        if (leader) tc_commit(acc_full + acc);
        __syncwarp();
      }
      VEON_TEND
    }
  } else {
    // ============================ EPILOGUE ============================
    const int quarter = warp & 3;  // TMEM lanes a warp may touch: 32*(warp%4) ..
    uint32_t heads0 = 0, heads1 = 0, heads2 = 0, heads3 = 0;   // bit q: prompt q starts a class
    if constexpr (!LOGITS) {
      auto head_word = [&](int base) -> uint32_t {
        const int q = base + lane;
        const bool h = q < p.Q && (q == 0 || __ldg(p.cls + q) != __ldg(p.cls + q - 1));
        return __ballot_sync(0xffffffffu, h);
      };
      heads0 = head_word(0); heads1 = head_word(32); heads2 = head_word(64); heads3 = head_word(96);
    }
    uint32_t tcount = 0;
    VEON_T0
    for (int64_t tile = tile_begin; tile < tile_end; tile += tile_step, ++tcount) {
      VEON_TACC(1)
      const int acc = tcount & 1;
      mbar_wait(acc_full + acc, (tcount >> 1) & 1);
      tc_fence_after();
      VEON_TACC(0)
      const int64_t b = tile / vtiles;
      const int64_t v = (tile - b * vtiles) * TM + 32 * quarter + lane;
      const uint32_t taddr = tmem_base + (uint32_t)(acc * npad) + ((uint32_t)(32 * quarter) << 16);
      if constexpr (LOGITS) {
        float* dst = p.logits + (int64_t)b * p.Q * p.V + v;  // lanes = consecutive voxels
        for (int q0 = 0; q0 < npad; q0 += 16) {
          float m[16];
          tc_ld16(taddr + q0, m);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (q0 + i < p.Q && v < p.V) dst[(int64_t)(q0 + i) * p.V] = m[i];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + acc);
        continue;
      }
      // class-wise max over the prompts and first-index arg-max over the classes, branch-free:
      // `heads` marks the first prompt of every class; a group is closed when the next one
      // starts.  Padded columns (q >= Q) enter as -inf and change nothing.
      float best = -INFINITY, cur = -INFINITY;
      int best_q = 0, cur_q = 0;
      bool bad = false;
#pragma unroll 1
      for (int q0 = 0; q0 < npad; q0 += 16) {
        float m[16];
        tc_ld16(taddr + q0, m);
        const uint32_t word = (q0 & 64) ? ((q0 & 32) ? heads3 : heads2) : ((q0 & 32) ? heads1 : heads0);
        const uint32_t h16 = word >> (q0 & 16);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int q = q0 + i;
          const float logit = q < p.Q ? m[i] : -INFINITY;
          bad |= !(logit < INFINITY);
          const bool head = (h16 >> i) & 1u;
          const bool take = head && (cur > best);
          best = take ? cur : best;
          best_q = take ? cur_q : best_q;
          cur = head ? logit : fmaxf(cur, logit);
          cur_q = head ? q : cur_q;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + acc);  // accumulator drained
      if (cur > best) { best = cur; best_q = cur_q; }
      const int best_cls = __ldg(p.cls + best_q);
      if (v < p.V) {
        bad |= (best == -INFINITY);
        const float b0 = __ldg(p.bin_occ + ((int64_t)b * 2 + 0) * p.V + v);
        const float b1 = __ldg(p.bin_occ + ((int64_t)b * 2 + 1) * p.V + v);
        const float mx = fmaxf(b0, b1);
        const float e0 = expf(b0 - mx), e1 = expf(b1 - mx);
        const bool occupied = (e0 / (e0 + e1)) > 0.5f;
        const int label = (occupied && !bad) ? best_cls : p.free_label;
        const uint32_t vv = (uint32_t)v, row = vv / (uint32_t)p.X;   // V < 2^31 (checked by the launcher)
        const int xx = (int)(vv - row * (uint32_t)p.X);
        const int zz = (int)(row / (uint32_t)p.Y);
        const int yy = (int)(row - (uint32_t)zz * (uint32_t)p.Y);
        p.labels[(((int64_t)b * p.X + xx) * p.Y + yy) * p.Z + zz] = (uint8_t)label;
      }
    }
    VEON_TEND
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(kTmemCols)
                 : "memory");
  }
}

}  // namespace tc
}  // namespace veon

using namespace veon;

#ifdef VEON_TAIL_TRACE
extern "C" int veon_internal_tail_trace(unsigned long long* host_out, int clear) {
  if (clear) {
    static unsigned long long zeros[32 * 8] = {};
    return (int)cudaMemcpyToSymbol(tc::veon_tail_trace, zeros, sizeof(zeros));
  }
  return (int)cudaMemcpyFromSymbol(host_out, tc::veon_tail_trace, sizeof(unsigned long long) * 32 * 8);
}
#endif

// returns 0 when launched, VEON_E_UNSUPPORTED when the shape does not fit this path.
// logits != nullptr: write sem_occ [B,Q,V] (cls / bin_occ / labels unused).
template <bool LOGITS, typename T, bool CL>
static int launch_variant(const tc::Params& p, unsigned grid, size_t smem, cudaStream_t stream) {
  static size_t attr_smem_dev[kMaxDevices] = {};   // per device: one process may drive several GPUs
  size_t& attr_smem = attr_smem_dev[current_device()];
  if (smem > attr_smem) {
    VEON_CUDA_TRY(cudaFuncSetAttribute(tc::k_tail_tc<LOGITS, T, CL>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem = smem;
  }
  tc::k_tail_tc<LOGITS, T, CL><<<grid, tc::kWarps * 32, smem, stream>>>(p);
  VEON_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t veon_text_classifier_image_bytes(int Q, int C) {
  const int npad = ((Q + 15) / 16) * 16;
  if (Q <= 0 || C <= 0 || C % tc::KC != 0 || npad > 128) return 0;
  return (size_t)(C / tc::KC) * 2 * npad * tc::KC * 4;
}

extern "C" int veon_text_classifier_image(const float* text_w, int Q, int C, void* image,
                                          size_t image_bytes, void* stream) {
  const size_t need = veon_text_classifier_image_bytes(Q, C);
  if (!text_w || !image || ((uintptr_t)text_w & 15) || ((uintptr_t)image & 15)) return VEON_E_BADARG;
  if (need == 0) return VEON_E_UNSUPPORTED;
  if (image_bytes < need) return VEON_E_WORKSPACE;
  const int npad = ((Q + 15) / 16) * 16;
  const int64_t pieces = (int64_t)(C / tc::KC) * npad * 8;
  tc::k_w_image<<<(unsigned)((pieces + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      text_w, Q, C, npad, static_cast<float*>(image));
  VEON_LAUNCH_CHECK();
  return 0;
}

// The shapes the float32 instance takes.  The bfloat16 one also needs V % 8 == 0 (a 16-byte copy
// carries 8 voxels); both need a 16-byte aligned feat_occ.  The channels-last instances need
// neither V % 4 nor V % 8 (a copy carries channels of one voxel), but they keep V % 4 == 0: the
// channels-first call takes the FFMA kernel otherwise, whose sums differ from tcgen05's, and a
// channels-last volume must give its contiguous copy's bits.
bool veon_tail_tc_takes(int C, int Q, int64_t V, const float* text_w) {
  const int npad = ((Q + 15) / 16) * 16;
  return C % tc::KC == 0 && (V & 3) == 0 && V < (int64_t(1) << 31) && npad <= 128 &&
         ((uintptr_t)text_w & 15) == 0;
}

// CL: feat_occ is channels-last [B,Z,Y,X,C]
template <typename T, bool CL>
int veon_tail_tc_launch(const T* feat_occ, const float* text_w, const int32_t* cls,
                        const float* bin_occ, int B, int C, int Q, int Z, int Y, int X,
                        int free_label, uint8_t* labels, float* logits, const void* w_image,
                        cudaStream_t stream) {
  const int64_t V = (int64_t)Z * Y * X;
  const int npad = ((Q + 15) / 16) * 16;
  if (!veon_tail_tc_takes(C, Q, V, text_w) || (!CL && V % tc::kVec<T> != 0) || ((uintptr_t)feat_occ & 15))
    return VEON_E_UNSUPPORTED;
  const size_t w_bytes = 2 * (size_t)npad * tc::KC * 4;
  const size_t tail = 1024;  // barriers + tmem slot
  int stages = (int)((tc::kTmemCols - 2 * npad) / tc::kSlotCols<T>);   // operand slots in tensor memory
  if (stages > tc::kMaxStages) stages = tc::kMaxStages;
  const size_t raw = (size_t)tc::kRawOf<T> * tc::kRawBytesOf<T>;
  if (raw + (size_t)stages * w_bytes + tail > 227 * 1024) stages = (int)((227 * 1024 - tail - raw) / w_bytes);
  if (stages < 2) return VEON_E_UNSUPPORTED;
  const size_t smem = raw + stages * w_bytes + tail;
  tc::Params p;
  p.feat = feat_occ; p.cls = cls; p.bin_occ = bin_occ; p.labels = labels;
  p.logits = logits;
  p.B = B; p.C = C; p.Q = Q; p.Z = Z; p.Y = Y; p.X = X; p.npad = npad; p.stages = stages;
  p.free_label = free_label; p.V = V;
  const int sms = sm_count();
  const int64_t n_tiles = (int64_t)B * ((V + tc::TM - 1) / tc::TM);
  const unsigned grid = (unsigned)(n_tiles < sms ? n_tiles : sms);
  if (w_image) {
    if ((uintptr_t)w_image & 15) return VEON_E_BADARG;
    p.w_image = static_cast<const float*>(w_image);
    return logits ? launch_variant<true, T, CL>(p, grid, smem, stream)
                  : launch_variant<false, T, CL>(p, grid, smem, stream);
  }
  // no prepared image: build one for the duration of the call in a stream-ordered allocation
  float* image = nullptr;
  const size_t image_bytes = veon_text_classifier_image_bytes(Q, C);
  VEON_CUDA_TRY(cudaMallocAsync((void**)&image, image_bytes, stream));
  int rc = veon_text_classifier_image(text_w, Q, C, image, image_bytes, stream);
  p.w_image = image;
  if (rc == 0)
    rc = logits ? launch_variant<true, T, CL>(p, grid, smem, stream)
                : launch_variant<false, T, CL>(p, grid, smem, stream);
  cudaFreeAsync(image, stream);
  return rc;
}
#define VEON_TAIL_TC_INSTANCE(T, CL)                                                              \
  template int veon_tail_tc_launch<T, CL>(const T*, const float*, const int32_t*, const float*, int, \
                                          int, int, int, int, int, int, uint8_t*, float*,            \
                                          const void*, cudaStream_t);
VEON_TAIL_TC_INSTANCE(float, false)
VEON_TAIL_TC_INSTANCE(bf16, false)
VEON_TAIL_TC_INSTANCE(float, true)
VEON_TAIL_TC_INSTANCE(bf16, true)
