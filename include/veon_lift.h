/*
 * veon_lift.h -- C ABI of libveonlift.so: the B200 (sm_100a) implementation of
 * VEON's 2D->3D lifting hot path (SURVEY.md section 8).
 *
 * Plain pointers and sizes only; no torch / ATen types.  All pointers are
 * DEVICE pointers on the current CUDA device unless the parameter is marked
 * [host].  `stream` is a cudaStream_t passed as void* (NULL = legacy default
 * stream, which is what the reference launches on, bev_pool_cuda.cu:127,136).
 * Nothing here allocates, synchronises the host, or keeps state between calls;
 * the caller owns every buffer (same ownership rule as the reference,
 * bev_pool.py:27,67-68).
 *
 * Return value: 0 on success, a positive cudaError_t on a CUDA failure, or a
 * negative VEON_E_* code for argument errors.  (The reference checks nothing:
 * bev_pool.cpp has no CHECK_* macros and no cudaGetLastError.)
 *
 * Citations are relative to /root/reference.
 */
#ifndef VEON_LIFT_H_
#define VEON_LIFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VEON_ABI_VERSION 11

#define VEON_E_BADARG    (-1)  /* NULL pointer / non-positive dimension          */
#define VEON_E_WORKSPACE (-2)  /* workspace smaller than *_workspace_bytes()     */
#define VEON_E_RANGE     (-3)  /* index space does not fit the int32 rank arrays */
#define VEON_E_UNSUPPORTED (-4)

/* Feature-volume layouts.  The reference kernel writes channels-last
 * (out[rank*C + c], bev_pool_cuda.cu:46) and bev_pool.py:91 then transposes to
 * channels-first; the fast path here emits channels-first directly. */
#define VEON_LAYOUT_BZYXC 0   /* [B, Z, Y, X, C]  (reference kernel layout)     */
#define VEON_LAYOUT_BCZYX 1   /* [B, C, Z, Y, X]  (what bev_pool_v2() returns)  */

/* plan-validation flag bits written by veon_pool_plan_build() */
#define VEON_PLAN_UNSORTED       1   /* ranks_bev not non-decreasing                       */
#define VEON_PLAN_BAD_INTERVALS  2   /* intervals are not exactly the runs of ranks_bev    */
#define VEON_PLAN_NONCANONICAL   4   /* ranks_feat != pixel-of(ranks_depth)                */
#define VEON_PLAN_OUT_OF_RANGE   8   /* an index outside its tensor                        */
#define VEON_PLAN_DUPLICATE     16   /* a depth element referenced twice                   */

int veon_abi_version(void);
/* static string for any code returned by this library */
const char* veon_error_string(int code);
/* number of CUDA kernels this library has launched in this process so far */
uint64_t veon_kernel_launch_count(void);

/* ------------------------------------------------------------------------
 * (1) Literal drop-ins for the two functions bev_pool.cpp binds
 *     (bev_pool.cpp:7-14; kernels bev_pool_cuda.cu:21-48, 67-121; launchers
 *     :125-140).  Same arguments in the same order plus a stream; same
 *     semantics: channels-last `out` / `out_grad`, caller-zeroed outputs, one
 *     output row per interval, intervals taken as given (for the backward they
 *     are the by-ranks_feat intervals built at bev_pool.py:47-57).  Indexing is
 *     64-bit (the reference's 32-bit `rank * c` overflows at C4, SURVEY 7).
 * ------------------------------------------------------------------------ */
int veon_bev_pool_v2(int c, int n_intervals,
                     const float* depth, const float* feat,
                     const int32_t* ranks_depth, const int32_t* ranks_feat,
                     const int32_t* ranks_bev,
                     const int32_t* interval_starts,
                     const int32_t* interval_lengths,
                     float* out, void* stream);

int veon_bev_pool_v2_grad(int c, int n_intervals, const float* out_grad,
                          const float* depth, const float* feat,
                          const int32_t* ranks_depth, const int32_t* ranks_feat,
                          const int32_t* ranks_bev,
                          const int32_t* interval_starts,
                          const int32_t* interval_lengths,
                          float* depth_grad, float* feat_grad, void* stream);

/* Same two operations for arbitrary (unsorted / non-canonical) rank arrays but
 * with a selectable volume layout; `voxels_per_sample` = Z*Y*X is needed to
 * split a rank into (b, voxel) for VEON_LAYOUT_BCZYX.  Used by the Python
 * operator when veon_pool_plan_build() rejects the ranks.  The backward is
 * point-driven (it needs no by-ranks_feat intervals): feat_grad is accumulated
 * with float atomics (order not deterministic).  Outputs must be zeroed by the
 * caller. */
int veon_bev_pool_v2_generic(int c, int n_intervals, int layout,
                             int64_t voxels_per_sample,
                             const float* depth, const float* feat,
                             const int32_t* ranks_depth, const int32_t* ranks_feat,
                             const int32_t* ranks_bev,
                             const int32_t* interval_starts,
                             const int32_t* interval_lengths,
                             float* out, void* stream);

int veon_bev_pool_v2_grad_generic(int c, int64_t n_points, int layout,
                                  int64_t voxels_per_sample, const float* out_grad,
                                  const float* depth, const float* feat,
                                  const int32_t* ranks_depth, const int32_t* ranks_feat,
                                  const int32_t* ranks_bev,
                                  float* depth_grad, float* feat_grad, void* stream);

/* ------------------------------------------------------------------------
 * (1b) get_lidar_coor (view_transformer.py:114-152; view_transformer_raw.py:121-158):
 *      frustum [D,H,W,3] + per-camera calibration -> coor [B,N,D,H,W,3], the
 *      input of voxel_pooling_prepare_v2.  sensor2ego [B,N,4,4], cam2imgs /
 *      post_rots [B,N,3,3], post_trans [B,N,3], bda [B,3,3], all float32
 *      contiguous on the device.  Float-tolerance parity (upstream of the
 *      bit-exact boundary).
 * ------------------------------------------------------------------------ */
size_t veon_lidar_coor_workspace_bytes(int B, int N);
int veon_lidar_coor(const float* frustum, const float* sensor2ego, const float* cam2imgs,
                    const float* post_rots, const float* post_trans, const float* bda,
                    int B, int N, int D, int H, int W, float* coor,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * (2) voxel_pooling_prepare_v2 (view_transformer.py:202-260; duplicated at
 *     view_transformer_raw.py:244-302).
 *
 *  coor            [B,N,D,H,W,3] float32, contiguous
 *  lower/interval/grid_size  [host] float32[3] = grid_lower_bound,
 *                  grid_interval, grid_size (view_transformer.py:79-82; all
 *                  three are FLOAT tensors in the reference and every rank is
 *                  computed in float32, :241-244 -- reproduced bit for bit)
 *  outputs, each with capacity P = B*N*D*H*W int32:
 *      ranks_bev, ranks_depth, ranks_feat   first n_kept entries valid
 *      interval_starts, interval_lengths    first n_int  entries valid
 *  counts          device int64[2] = {n_kept, n_int}
 *  counts_host     optional PINNED HOST int64[2] (device-accessible, e.g. cudaHostAlloc):
 *                  the scan kernel stores the same two numbers there, so the host can
 *                  read them after an event on `stream` without queueing a copy behind
 *                  the caller's bulk transfers; NULL to skip
 *  Order: points sorted by ranks_bev; inside one voxel by ascending
 *  ranks_depth (the reference's argsort is unstable, so its in-voxel order is
 *  arbitrary; ours is the canonical stable one).
 *
 *  Optional by-products ("plan") consumed by the *_planar pool entry points
 *  (pass NULL to skip them all; tile_heavy may be NULL on its own):
 *      tile_start   int32[n_tiles+1]  first point of each 32-voxel tile
 *      tile_istart  int32[n_tiles+1]  first interval of each tile
 *      tile_occ     uint32[n_tiles+1] bit v set <=> voxel v of the tile is occupied
 *      point_interval int32[P]        interval index of depth element
 *                   (b,n,d,h,w) stored PIXEL-major at ((b*N+n)*H*W+hw)*D+d,
 *                   -1 where the point was dropped
 *      tile_heavy   int32[veon_pool_heavy_list_ints(P, n_tiles)]: [0] = number of
 *                   listed tiles, [1] = the point-count threshold used, [2..] = ids
 *                   (arbitrary order) of the tiles holding at least that many
 *                   points; the forward gives each of them to a whole thread
 *                   block instead of one warp
 *    with n_tiles = B * ceil(Z*Y*X / 32), see veon_pool_num_tiles().
 * ------------------------------------------------------------------------ */
size_t veon_prepare_v2_workspace_bytes(int B, int N, int D, int H, int W,
                                       const float* grid_size /*[host]*/);
int64_t veon_pool_num_tiles(int B, int64_t voxels_per_sample);
/* int32 elements a tile_heavy buffer needs for a plan over at most n_points points */
int64_t veon_pool_heavy_list_ints(int64_t n_points, int64_t n_tiles);

int veon_prepare_v2(const float* coor, int B, int N, int D, int H, int W,
                    const float* lower, const float* interval,
                    const float* grid_size,
                    int32_t* ranks_bev, int32_t* ranks_depth, int32_t* ranks_feat,
                    int32_t* interval_starts, int32_t* interval_lengths,
                    int64_t* counts, int64_t* counts_host,
                    int32_t* tile_start, int32_t* tile_istart, uint32_t* tile_occ,
                    int32_t* tile_heavy, int32_t* point_interval,
                    void* workspace, size_t workspace_bytes, void* stream);

/* The same with get_lidar_coor fused in (view_transformer.py:114-152 + :202-260): takes the
 * frustum and the calibration tensors of veon_lidar_coor instead of `coor`; the coordinate tensor
 * is never materialised.  The ranks are bit-identical to veon_lidar_coor + veon_prepare_v2.
 * xform_workspace: veon_lidar_coor_workspace_bytes(B, N) bytes. */
int veon_prepare_v2_calib(const float* frustum, const float* sensor2ego, const float* cam2imgs,
                          const float* post_rots, const float* post_trans, const float* bda,
                          int B, int N, int D, int H, int W,
                          const float* lower, const float* interval, const float* grid_size,
                          int32_t* ranks_bev, int32_t* ranks_depth, int32_t* ranks_feat,
                          int32_t* interval_starts, int32_t* interval_lengths,
                          int64_t* counts, int64_t* counts_host,
                          int32_t* tile_start, int32_t* tile_istart, uint32_t* tile_occ,
                          int32_t* tile_heavy, int32_t* point_interval,
                          void* xform_workspace, size_t xform_workspace_bytes,
                          void* workspace, size_t workspace_bytes, void* stream);

/* veon_prepare_v2_calib with an inference-time point filter (SURVEY 8f-2): a point whose depth
 * weight depth[b,n,d,h,w] is <= depth_eps is dropped like an out-of-grid point.  VEON's two-hot
 * depth (view_transformer_raw.py:406-429) leaves most bins at the e^-16 clamp, i.e. ~1e-7 of
 * the weight: with depth_eps = 1e-6 about 90 % of the points carry no signal and leave the
 * pooled volume unchanged to ~1e-6 relative.  The gradient of a dropped point is zero, so this
 * is for inference; depth_eps >= 0. */
int veon_prepare_v2_calib_sparse(const float* frustum, const float* sensor2ego,
                                 const float* cam2imgs, const float* post_rots,
                                 const float* post_trans, const float* bda,
                                 const float* depth, float depth_eps,
                                 int B, int N, int D, int H, int W,
                                 const float* lower, const float* interval, const float* grid_size,
                                 int32_t* ranks_bev, int32_t* ranks_depth, int32_t* ranks_feat,
                                 int32_t* interval_starts, int32_t* interval_lengths,
                                 int64_t* counts, int64_t* counts_host,
                                 int32_t* tile_start, int32_t* tile_istart, uint32_t* tile_occ,
                                 int32_t* tile_heavy, int32_t* point_interval,
                                 void* xform_workspace, size_t xform_workspace_bytes,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* 64-bit hash of the BITS of the five calibration tensors get_lidar_coor consumes (layouts as in
 * veon_lidar_coor), written to `out` -- device memory or pinned host memory the device can
 * write (then readable after an event on `stream`, no copy).  Key of a rank cache that
 * generalises the reference's `accelerate` mode (view_transformer.py:154-173) to any number of
 * recurring rigs. */
int veon_calib_hash(const float* sensor2ego, const float* cam2imgs, const float* post_rots,
                    const float* post_trans, const float* bda, int B, int N, uint64_t* out,
                    void* stream);

/* Build the same plan from rank arrays the caller already holds (the
 * `accelerate=True` cache, view_transformer.py:154-173, or any user input) and
 * validate them.  *flags (device int32) receives an OR of VEON_PLAN_* bits; the
 * planar entry points are only valid for flags == 0. */
int veon_pool_plan_build(const int32_t* ranks_depth, const int32_t* ranks_feat,
                         const int32_t* ranks_bev,
                         const int32_t* interval_starts,
                         const int32_t* interval_lengths,
                         int64_t n_points, int64_t n_intervals,
                         int B, int N, int D, int H, int W,
                         int64_t voxels_per_sample,
                         int32_t* tile_start, int32_t* tile_istart, uint32_t* tile_occ,
                         int32_t* tile_heavy /* sized for n_points; may be NULL */,
                         int32_t* point_interval, int32_t* flags, void* stream);

/* Batched transpose [batch][R][S] -> [batch][S][R] (float32, contiguous).  Replaces the
 * `feat.permute(0,1,3,4,2)` + `.contiguous()` copy (view_transformer.py:279, bev_pool.py:88)
 * on the way in and its inverse on feat_grad on the way out. */
int veon_transpose_batched(const float* src, int64_t batch, int R, int S, float* dst,
                           void* stream);

/* ------------------------------------------------------------------------
 * (3) Fast pooling path: bev_pool_v2() INCLUDING its transpose
 *     (bev_pool.py:86-92 = QuickCumsumCuda.forward :17-41 + permute :91).
 *     `out` is [B,C,Z,Y,X]; every element is written exactly once (zeros for
 *     empty voxels), so the caller need not zero it.  Requires a valid plan.
 *     The result is bit-identical to the reference kernel for every C.
 *     Kernel selection: rows of at most 32 channels (C % 4 == 0, tile_heavy
 *     given, B*V <= 2^24) take a lane-per-voxel kernel; aligned volumes
 *     (V % 32 == 0) with C == 64, a complete plan (tile_istart, tile_occ,
 *     tile_heavy) and a workspace take the two-role streaming kernel (compact
 *     rows through an L2-resident ring, the volume written as a pure store
 *     stream); everything else the general lane-per-channel kernel.
 *   workspace   optional scratch of veon_bev_pool_v2_fwd_workspace_bytes()
 *               bytes, 256-byte aligned (a larger or smaller buffer is legal: it
 *               sizes the ring; too small a one selects the general kernel);
 *               contents need not be preserved between calls, but one buffer
 *               must not be shared by calls that may run concurrently.  The
 *               size is 0 for every C other than 64: no kernel needs a
 *               workspace there, and NULL with workspace_bytes = 0 is correct.
 * ------------------------------------------------------------------------ */
size_t veon_bev_pool_v2_fwd_workspace_bytes(int B, int C, int64_t voxels_per_sample);
int veon_bev_pool_v2_fwd_planar(const float* depth, const float* feat,
                                const int32_t* ranks_depth,
                                const int32_t* ranks_feat,
                                const int32_t* ranks_bev,
                                const int32_t* tile_start,
                                const int32_t* tile_istart /* may be NULL */,
                                const uint32_t* tile_occ /* may be NULL */,
                                const int32_t* tile_heavy /* may be NULL */,
                                int64_t tile_heavy_ints /* its size in int32 */,
                                int B, int C, int64_t voxels_per_sample,
                                int64_t n_feat_rows /* B*N*H*W rows of feat */,
                                float* out, void* workspace, size_t workspace_bytes,
                                void* stream);

/* The same pooling into a CHANNELS-LAST volume: out is [B,Z,Y,X,C] (the reference kernel's own
 * layout, bev_pool_cuda.cu:46), every element written exactly once (zero rows for empty voxels),
 * no workspace.  The sums are the same bits as veon_bev_pool_v2_fwd_planar's, only their order in
 * memory differs: torch's channels_last_3d view of [B,C,Z,Y,X] has exactly this storage.
 * Requires a valid plan; any C >= 1, any V (ragged x-runs), B >= 1.  Kernel selection: rows of at
 * most 32 channels (C % 4 == 0, tile_heavy given, V % 32 == 0, B*V <= 2^24, 16-byte aligned feat
 * and out) take the lane-per-voxel kernel; everything else the lane-per-channel kernel, which
 * stages a tile's rows in shared memory and writes them as contiguous rows.  Tiles listed in
 * tile_heavy get a thread block each, queued behind the main grid as a programmatic dependent
 * that completes only after it: the next kernel in the stream, or the next node of a captured
 * graph, sees the whole volume.  VEON_E_RANGE when B*V, B or the 32-bit feature row offsets
 * overflow (as veon_bev_pool_v2_fwd_planar). */
int veon_bev_pool_v2_fwd_planar_cl(const float* depth, const float* feat,
                                   const int32_t* ranks_depth,
                                   const int32_t* ranks_feat,
                                   const int32_t* ranks_bev,
                                   const int32_t* tile_start,
                                   const int32_t* tile_heavy /* may be NULL */,
                                   int64_t tile_heavy_ints /* its size in int32 */,
                                   int B, int C, int64_t voxels_per_sample,
                                   int64_t n_feat_rows /* B*N*H*W rows of feat */,
                                   float* out, void* stream);

/* bfloat16 volumes.  The same pooling as veon_bev_pool_v2_fwd_planar / _cl (same arguments, same
 * checks and error codes, same kernel selection), but `out` holds bfloat16 bit patterns: every
 * sum is accumulated in float32 exactly as the float32 twin does and rounded once, when it is
 * stored, to nearest even (as `cvt.rn.bf16.f32` does, which is what torch's device-side cast to
 * bfloat16 uses).  So the result is, bit for bit, the float32 twin's volume cast to bfloat16.
 * out must be 8-byte aligned for the vector stores (an unaligned one takes scalar stores).  The
 * channels-first one never takes the streaming kernel: its workspace arguments are accepted and
 * ignored. */
int veon_bev_pool_v2_fwd_planar_bf16(const float* depth, const float* feat,
                                     const int32_t* ranks_depth,
                                     const int32_t* ranks_feat,
                                     const int32_t* ranks_bev,
                                     const int32_t* tile_start,
                                     const int32_t* tile_istart /* may be NULL */,
                                     const uint32_t* tile_occ /* may be NULL */,
                                     const int32_t* tile_heavy /* may be NULL */,
                                     int64_t tile_heavy_ints /* its size in int32 */,
                                     int B, int C, int64_t voxels_per_sample,
                                     int64_t n_feat_rows /* B*N*H*W rows of feat */,
                                     uint16_t* out /* bfloat16 [B,C,Z,Y,X] */,
                                     void* workspace, size_t workspace_bytes, void* stream);
int veon_bev_pool_v2_fwd_planar_cl_bf16(const float* depth, const float* feat,
                                        const int32_t* ranks_depth,
                                        const int32_t* ranks_feat,
                                        const int32_t* ranks_bev,
                                        const int32_t* tile_start,
                                        const int32_t* tile_heavy /* may be NULL */,
                                        int64_t tile_heavy_ints /* its size in int32 */,
                                        int B, int C, int64_t voxels_per_sample,
                                        int64_t n_feat_rows /* B*N*H*W rows of feat */,
                                        uint16_t* out /* bfloat16 [B,Z,Y,X,C] */, void* stream);

/* Depth-distribution producer in front of the path: LSSViewTransformerRaw.downsample_depth +
 * get_two_hot_depth (view_transformer_raw.py:393-429).  depths [BN, H_out*s, W_out*s] metric
 * depth (0 = no measurement), s = downsample (<= 1: none); out [BN, D, H_out, W_out]:
 * softmax over the D+1 bin centres of max(-|d - c_k| * gamma, -16) with the last bin dropped.
 * Forward only. */
int veon_two_hot_depth(const float* depths, int64_t BN, int H_out, int W_out, int downsample,
                       int D, float depth_lo, float depth_step, float gamma, float* out,
                       void* stream);

/* The neck's 2x2x2 max-downsample on its own (view_transformer_raw.py:549-553: einops
 * rearrange to a trailing (dz dh dw) axis + torch.max(dim=-1).values) and its gradient (the
 * backward of max(dim): the whole gradient to the first arg-max of each block).  in / grad_in
 * [BC,Z,Y,X], out / grad_out [BC,Z/2,Y/2,X/2], float32, contiguous; Z, Y even and X % 4 == 0,
 * else VEON_E_UNSUPPORTED. */
int veon_maxdown2_fwd(const float* in, int64_t BC, int Z, int Y, int X, float* out, void* stream);
/* Forward that also emits, per output, an 8-bit mask with ONE bit set: the arg-max input
 * (bit (dz*2+dy)*2+dx, the first maximum on ties) -- all veon_bev_pool_v2_bwd_planar_ds
 * needs. */
int veon_maxdown2_fwd_mask(const float* in, int64_t BC, int Z, int Y, int X, float* out,
                           uint8_t* mask, void* stream);
int veon_maxdown2_bwd(const float* in, const float* out, const float* grad_out,
                      int64_t BC, int Z, int Y, int X, float* grad_in, void* stream);
/* The same two operations on CHANNELS-LAST volumes: in / grad_in [B,Z,Y,X,C], out / grad_out
 * [B,Z/2,Y/2,X/2,C], float32, contiguous, any alignment.  Same reduction tree, NaN rule, -0/+0
 * result and first-arg-max gradient as veon_maxdown2_fwd / _bwd, so the values are the same
 * bits in the other layout.  Z, Y, X even, else VEON_E_UNSUPPORTED; VEON_E_RANGE when the output
 * has 2^32 voxels or more. */
int veon_maxdown2_cl_fwd(const float* in, int B, int C, int Z, int Y, int X, float* out,
                         void* stream);
int veon_maxdown2_cl_bwd(const float* in, const float* out, const float* grad_out,
                         int B, int C, int Z, int Y, int X, float* grad_in, void* stream);
/* The same operations on bfloat16 volumes (uint16_t bit patterns), with the arguments, checks and
 * error codes of the float32 twins, except that the channels-first entries need in / grad_in
 * 8-byte and out / grad_out 4-byte aligned (else VEON_E_UNSUPPORTED).  Values are widened exactly
 * where they are loaded and compared as the twins compare them, so out and grad_in are, bit for
 * bit, `rearrange + torch.max(dim=-1)` on the bfloat16 tensor and its gradient (NaN payloads
 * aside).  veon_maxdown2_fwd_mask_bf16 reads a float32 volume (16-byte aligned, as its twin) and
 * stores the float32 maximum rounded once to nearest even as bfloat16 out (4-byte aligned); the
 * mask is its twin's, taken over the float32 values. */
int veon_maxdown2_fwd_bf16(const uint16_t* in, int64_t BC, int Z, int Y, int X, uint16_t* out,
                           void* stream);
int veon_maxdown2_fwd_mask_bf16(const float* in, int64_t BC, int Z, int Y, int X, uint16_t* out,
                                uint8_t* mask, void* stream);
int veon_maxdown2_bwd_bf16(const uint16_t* in, const uint16_t* out, const uint16_t* grad_out,
                           int64_t BC, int Z, int Y, int X, uint16_t* grad_in, void* stream);
int veon_maxdown2_cl_fwd_bf16(const uint16_t* in, int B, int C, int Z, int Y, int X,
                              uint16_t* out, void* stream);
int veon_maxdown2_cl_bwd_bf16(const uint16_t* in, const uint16_t* out, const uint16_t* grad_out,
                              int B, int C, int Z, int Y, int X, uint16_t* grad_in, void* stream);

/* QuickCumsumCuda.backward (bev_pool.py:43-83) for a [B,C,Z,Y,X] out_grad.
 *   rows_ws      float scratch of at least veon_bev_pool_v2_bwd_workspace_floats() elements
 *                (one compact gradient row per interval; rows_ws_floats says how many floats it
 *                holds, VEON_E_WORKSPACE if too few)
 *   depth_grad   [B,N,D,H,W], feat_grad [B,N,H,W,C]: fully written (no need to
 *                zero).  Deterministic: no atomics, fixed summation order.
 *   Two launches: a row pass over the occupied 32-voxel tiles of out_grad and a pixel pass. */
size_t veon_bev_pool_v2_bwd_workspace_floats(int64_t n_intervals, int B, int N, int D, int H,
                                             int W, int C, int64_t voxels_per_sample);
int veon_bev_pool_v2_bwd_planar(const float* out_grad,
                                const float* depth, const float* feat,
                                const int32_t* tile_istart,
                                const uint32_t* tile_occ,
                                const int32_t* point_interval,
                                int64_t n_intervals,
                                int B, int N, int D, int H, int W, int C,
                                int64_t voxels_per_sample,
                                float* rows_ws, int64_t rows_ws_floats,
                                float* depth_grad, float* feat_grad,
                                void* stream);

/* QuickCumsumCuda.backward for a CHANNELS-LAST out_grad [B,Z,Y,X,C] in ONE launch: an occupied
 * voxel's gradient is already one contiguous row there, so the pixel pass reads it in place --
 * no row pass and no rows_ws scratch.  The row of a kept point is that of its voxel,
 * ranks_bev[interval_starts[point_interval[...]]]; only intervals named by point_interval are
 * read, so a capacity-sized interval_starts (the sync-free prepare outputs) is never read beyond
 * the device-side interval count.  depth_grad / feat_grad as in veon_bev_pool_v2_bwd_planar and
 * the same bits (same rows, same order of operations).  Requires a valid plan.  VEON_E_RANGE when
 * B*V >= 2^31; VEON_E_UNSUPPORTED when D is too large for the per-warp point lists (as the
 * channels-first pixel pass). */
int veon_bev_pool_v2_bwd_planar_cl(const float* out_grad,
                                   const float* depth, const float* feat,
                                   const int32_t* ranks_bev,
                                   const int32_t* interval_starts,
                                   const int32_t* point_interval,
                                   int B, int N, int D, int H, int W, int C,
                                   int64_t voxels_per_sample,
                                   float* depth_grad, float* feat_grad, void* stream);

/* The two backward routes above for a bfloat16 out_grad (uint16_t bit patterns; same arguments,
 * checks and error codes as the float32 twins; rows_ws is the same float32 scratch, sized by
 * veon_bev_pool_v2_bwd_workspace_floats).  Every gradient value is widened to float32 exactly
 * where it is read, and everything after that is the float32 twin's arithmetic: depth_grad /
 * feat_grad (float32) are the same bits as the twin's given the widened gradient. */
int veon_bev_pool_v2_bwd_planar_bf16(const uint16_t* out_grad /* bfloat16 [B,C,Z,Y,X] */,
                                     const float* depth, const float* feat,
                                     const int32_t* tile_istart,
                                     const uint32_t* tile_occ,
                                     const int32_t* point_interval,
                                     int64_t n_intervals,
                                     int B, int N, int D, int H, int W, int C,
                                     int64_t voxels_per_sample,
                                     float* rows_ws, int64_t rows_ws_floats,
                                     float* depth_grad, float* feat_grad,
                                     void* stream);
int veon_bev_pool_v2_bwd_planar_cl_bf16(const uint16_t* out_grad /* bfloat16 [B,Z,Y,X,C] */,
                                        const float* depth, const float* feat,
                                        const int32_t* ranks_bev,
                                        const int32_t* interval_starts,
                                        const int32_t* point_interval,
                                        int B, int N, int D, int H, int W, int C,
                                        int64_t voxels_per_sample,
                                        float* depth_grad, float* feat_grad, void* stream);

/* QuickCumsumCuda.backward for a gradient that arrives BEHIND the 2x2x2 max-downsample:
 * grad_ds [B,C,Z/2,Y/2,X/2] and the mask of veon_maxdown2_fwd_mask replace out_grad; the
 * full-resolution gradient is never formed (max(dim) gradient semantics: all to the arg-max).
 * rows_ws as in veon_bev_pool_v2_bwd_planar; even Z, Y, X. */
int veon_bev_pool_v2_bwd_planar_ds(const float* grad_ds, const uint8_t* mask,
                                   const float* depth, const float* feat,
                                   const int32_t* tile_istart, const uint32_t* tile_occ,
                                   const int32_t* point_interval, int64_t n_intervals,
                                   int B, int N, int D, int H, int W, int C, int Z, int Y, int X,
                                   float* rows_ws, float* depth_grad, float* feat_grad,
                                   void* stream);

/* bfloat16 feature rows.  The planar forwards and backwards above for feat given as bfloat16
 * [B*N*H*W, C] rows (uint16_t bit patterns), the input a network running under bfloat16 autocast
 * hands the lift.  Same arguments, checks and error codes as the twin without `_bf16feat`.
 * Every feature value is widened to float32 exactly where it is loaded, and everything after the
 * load is the twin's float32 arithmetic in the same order: each volume (float32 or bfloat16) is,
 * bit for bit, the twin's volume on the widened rows, and depth_grad (float32) is the twin's
 * depth_grad.  feat_grad is bfloat16 [B*N*H*W, C]: the twin's float32 feat_grad rounded once, to
 * nearest even.  The vectorised kernels need C % 4 == 0 and 8-byte aligned rows (else the
 * lane-per-channel kernel, which reads any alignment).  The feature-row range check is the
 * float32 one.  veon_bev_pool_v2_fwd_planar_bf16feat returns VEON_E_UNSUPPORTED where its twin
 * would take the two-role streaming kernel, which reads float32 rows only: the caller then widens
 * the rows and calls veon_bev_pool_v2_fwd_planar. */
int veon_bev_pool_v2_fwd_planar_bf16feat(const float* depth, const uint16_t* feat,
                                         const int32_t* ranks_depth, const int32_t* ranks_feat,
                                         const int32_t* ranks_bev, const int32_t* tile_start,
                                         const int32_t* tile_istart /* may be NULL */,
                                         const uint32_t* tile_occ /* may be NULL */,
                                         const int32_t* tile_heavy /* may be NULL */,
                                         int64_t tile_heavy_ints, int B, int C,
                                         int64_t voxels_per_sample, int64_t n_feat_rows,
                                         float* out, void* workspace, size_t workspace_bytes,
                                         void* stream);
int veon_bev_pool_v2_fwd_planar_bf16_bf16feat(const float* depth, const uint16_t* feat,
                                              const int32_t* ranks_depth,
                                              const int32_t* ranks_feat,
                                              const int32_t* ranks_bev,
                                              const int32_t* tile_start,
                                              const int32_t* tile_istart /* may be NULL */,
                                              const uint32_t* tile_occ /* may be NULL */,
                                              const int32_t* tile_heavy /* may be NULL */,
                                              int64_t tile_heavy_ints, int B, int C,
                                              int64_t voxels_per_sample, int64_t n_feat_rows,
                                              uint16_t* out /* bfloat16 [B,C,Z,Y,X] */,
                                              void* workspace, size_t workspace_bytes,
                                              void* stream);
int veon_bev_pool_v2_fwd_planar_cl_bf16feat(const float* depth, const uint16_t* feat,
                                            const int32_t* ranks_depth, const int32_t* ranks_feat,
                                            const int32_t* ranks_bev, const int32_t* tile_start,
                                            const int32_t* tile_heavy /* may be NULL */,
                                            int64_t tile_heavy_ints, int B, int C,
                                            int64_t voxels_per_sample, int64_t n_feat_rows,
                                            float* out /* [B,Z,Y,X,C] */, void* stream);
int veon_bev_pool_v2_fwd_planar_cl_bf16_bf16feat(const float* depth, const uint16_t* feat,
                                                 const int32_t* ranks_depth,
                                                 const int32_t* ranks_feat,
                                                 const int32_t* ranks_bev,
                                                 const int32_t* tile_start,
                                                 const int32_t* tile_heavy /* may be NULL */,
                                                 int64_t tile_heavy_ints, int B, int C,
                                                 int64_t voxels_per_sample, int64_t n_feat_rows,
                                                 uint16_t* out /* bfloat16 [B,Z,Y,X,C] */,
                                                 void* stream);
int veon_bev_pool_v2_bwd_planar_bf16feat(const float* out_grad, const float* depth,
                                         const uint16_t* feat, const int32_t* tile_istart,
                                         const uint32_t* tile_occ, const int32_t* point_interval,
                                         int64_t n_intervals, int B, int N, int D, int H, int W,
                                         int C, int64_t voxels_per_sample, float* rows_ws,
                                         int64_t rows_ws_floats, float* depth_grad,
                                         uint16_t* feat_grad, void* stream);
int veon_bev_pool_v2_bwd_planar_bf16_bf16feat(const uint16_t* out_grad, const float* depth,
                                              const uint16_t* feat, const int32_t* tile_istart,
                                              const uint32_t* tile_occ,
                                              const int32_t* point_interval, int64_t n_intervals,
                                              int B, int N, int D, int H, int W, int C,
                                              int64_t voxels_per_sample, float* rows_ws,
                                              int64_t rows_ws_floats, float* depth_grad,
                                              uint16_t* feat_grad, void* stream);
int veon_bev_pool_v2_bwd_planar_cl_bf16feat(const float* out_grad, const float* depth,
                                            const uint16_t* feat, const int32_t* ranks_bev,
                                            const int32_t* interval_starts,
                                            const int32_t* point_interval, int B, int N, int D,
                                            int H, int W, int C, int64_t voxels_per_sample,
                                            float* depth_grad, uint16_t* feat_grad, void* stream);
int veon_bev_pool_v2_bwd_planar_cl_bf16_bf16feat(const uint16_t* out_grad, const float* depth,
                                                 const uint16_t* feat, const int32_t* ranks_bev,
                                                 const int32_t* interval_starts,
                                                 const int32_t* point_interval, int B, int N,
                                                 int D, int H, int W, int C,
                                                 int64_t voxels_per_sample, float* depth_grad,
                                                 uint16_t* feat_grad, void* stream);
int veon_bev_pool_v2_bwd_planar_ds_bf16feat(const float* grad_ds, const uint8_t* mask,
                                            const float* depth, const uint16_t* feat,
                                            const int32_t* tile_istart, const uint32_t* tile_occ,
                                            const int32_t* point_interval, int64_t n_intervals,
                                            int B, int N, int D, int H, int W, int C, int Z, int Y,
                                            int X, float* rows_ws, float* depth_grad,
                                            uint16_t* feat_grad, void* stream);
/* veon_bev_pool_v2_bwd_planar_ds (and its _bf16feat form) for a bfloat16 grad_ds, the reduced
 * volume of veon_maxdown2_fwd_mask_bf16: every value is widened exactly where the row pass loads
 * it, everything after is the float32 twin's, so depth_grad / feat_grad are the twin's bits given
 * the widened gradient.  Same arguments, checks and error codes as the twins. */
int veon_bev_pool_v2_bwd_planar_ds_bf16(const uint16_t* grad_ds, const uint8_t* mask,
                                        const float* depth, const float* feat,
                                        const int32_t* tile_istart, const uint32_t* tile_occ,
                                        const int32_t* point_interval, int64_t n_intervals,
                                        int B, int N, int D, int H, int W, int C, int Z, int Y,
                                        int X, float* rows_ws, float* depth_grad,
                                        float* feat_grad, void* stream);
int veon_bev_pool_v2_bwd_planar_ds_bf16_bf16feat(const uint16_t* grad_ds, const uint8_t* mask,
                                                 const float* depth, const uint16_t* feat,
                                                 const int32_t* tile_istart,
                                                 const uint32_t* tile_occ,
                                                 const int32_t* point_interval,
                                                 int64_t n_intervals, int B, int N, int D, int H,
                                                 int W, int C, int Z, int Y, int X,
                                                 float* rows_ws, float* depth_grad,
                                                 uint16_t* feat_grad, void* stream);
/* veon_transpose_batched for 2-byte elements (bfloat16 maps and feature gradients): the same
 * tiles and checks, the bits moved unchanged. */
int veon_transpose_batched_u16(const uint16_t* src, int64_t batch, int R, int S, uint16_t* dst,
                               void* stream);

/* ------------------------------------------------------------------------
 * (4) Open-vocabulary tail: voxel-feature x text-embedding logits, per-class
 *     max over prompts, argmax, occupancy gate, uint8 labels.
 *       semantic_inference_3d   san_in_veon_temporal.py:257-259
 *       _merge_classes_prob     san_in_veon_entry_temporal.py:273-297
 *       label rule              veon_temporal.py:223-229,240
 *   feat_occ [B,C,Z,Y,X] f32; text_w [Q,C] f32; class_of_prompt [Q] int32
 *   (non-decreasing, the merged class of every prompt row incl. the trailing
 *   background row); bin_occ [B,2,Z,Y,X] f32; labels uint8 [B,X,Y,Z].
 * ------------------------------------------------------------------------ */
int veon_voxel_text_argmax(const float* feat_occ, const float* text_w,
                           const int32_t* class_of_prompt, const float* bin_occ,
                           int B, int C, int Q, int Z, int Y, int X,
                           int free_label, uint8_t* labels, const void* w_image, void* stream);

/* The text classifier is fixed per vocabulary (the reference builds it once,
 * san_in_veon_temporal.py:261-266), so its tensor-core operand form is prepared once too:
 * [W_hi ; W_lo] (the 3xTF32 split) of every 32-channel chunk in the shared-memory layout of
 * the tail kernel's B operand.  veon_text_classifier_image_bytes(Q, C) = its size (0 when the
 * tensor-core path does not take the shape: C % 32 != 0 or Q > 128);
 * veon_text_classifier_image fills `image` (>= that many bytes, 16-byte aligned,
 * VEON_E_WORKSPACE if short).  The three tail entry points take it as `w_image`; it must come
 * from the same text_w, Q and C.  w_image == NULL is allowed: the library then builds the image
 * for the duration of the call in a stream-ordered allocation (cudaMallocAsync on `stream`), the
 * one place where it allocates. */
size_t veon_text_classifier_image_bytes(int Q, int C);
int veon_text_classifier_image(const float* text_w, int Q, int C, void* image, size_t image_bytes,
                               void* stream);

/* semantic_inference_3d alone (san_in_veon_temporal.py:257-259, argument order of the
 * reference method): sem_occ[b,q,z,y,x] = sum_c text_w[q,c] * feat_occ[b,c,z,y,x], fp32
 * (3xTF32 on tcgen05 when C % 32 == 0, V % 4 == 0 and Q <= 128, else fp32 FFMA).
 *   text_w [Q,C]; feat_occ [B,C,Z,Y,X]; sem_occ [B,Q,Z,Y,X] (written, not accumulated). */
int veon_semantic_inference_3d(const float* text_w, const float* feat_occ,
                               int B, int C, int Q, int Z, int Y, int X,
                               float* sem_occ, const void* w_image, void* stream);

/* Training-time voxel x text arg-max over a point list (Proj2Dto3DLoss,
 * loss/occ_loss_utils/occ3d_nuscenes.py:472-482): logits [Q, ldn] = the Q prompt rows (no
 * background row) over N <= ldn points, as veon_semantic_inference_3d writes them for a [C, N]
 * operand; class_of_prompt [Q] non-decreasing merged class of each row
 * (_merge_classes_prob, :249-265).  prompt_idx[n] = arg-max prompt, class_idx[n] = arg-max of
 * the per-class maxima; first index on ties, like torch.max(dim).indices.  int64 outputs. */
int veon_point_text_argmax(const float* logits, const int32_t* class_of_prompt, int Q,
                           int64_t N, int64_t ldn, int64_t* prompt_idx, int64_t* class_idx,
                           void* stream);

/* ------------------------------------------------------------------------
 * (5) Tail at the decoder's resolution (SURVEY.md 8f-4).  The reference
 *     up-samples feat_occ and bin_occ to occ_size with
 *     F.interpolate(mode="trilinear", align_corners=False)
 *     (san_in_veon_temporal.py:196-207) and classifies the up-sampled volume.
 *     Interpolation and classifier are linear, so the logits are computed on
 *     the low-resolution volume and only Q + 2 channels are interpolated.
 *
 *   veon_upsample_classify: sem_occ_lr [B,Q,Zi,Yi,Xi] and bin_occ_lr
 *     [B,2,Zi,Yi,Xi] -> trilinear (align_corners=False) to [Z,Y,X], class
 *     merge, arg-max, gate -> labels uint8 [B,X,Y,Z].
 *   veon_voxel_text_argmax_lowres: feat_occ_lr [B,C,Zi,Yi,Xi] -> the same
 *     labels; `workspace` holds the low-resolution logits
 *     (veon_voxel_text_argmax_lowres_workspace_bytes, VEON_E_WORKSPACE if short).
 * ------------------------------------------------------------------------ */
int veon_upsample_classify(const float* sem_occ_lr, const float* bin_occ_lr,
                           const int32_t* class_of_prompt, int B, int Q,
                           int Zi, int Yi, int Xi, int Z, int Y, int X,
                           int free_label, uint8_t* labels, void* stream);
/* _merge_classes_prob + the label rule alone (san_in_veon_entry_temporal.py:273-297,
 * veon_temporal.py:223-229,240) on ready-made logits: sem_occ [B,Q,Z,Y,X], bin_occ [B,2,Z,Y,X]
 * -> labels uint8 [B,X,Y,Z].  The batch strides (in floats) are free, so both inputs may be
 * channel slices of one volume; everything inside a sample is contiguous. */
int veon_classify_logits(const float* sem_occ, int64_t sem_batch_stride,
                         const float* bin_occ, int64_t bin_batch_stride,
                         const int32_t* class_of_prompt, int B, int Q, int Z, int Y, int X,
                         int free_label, uint8_t* labels, void* stream);
/* Lift + classify in one pass (SURVEY.md 8f-4, BASELINE configs[2]): pooling is linear, so the
 * classifier and the gate head run on the image features first (veon_semantic_inference_3d over
 * [B*N, C, H*W]) and the per-pixel rows
 *     pix [n_pix_rows, Cp] = [gate 0, gate 1, logit 0 .. Q-1, zero padding]   (Cp = 4k <= 32, 8k in 40..64 or 12k in 72..96)
 * are pooled with the unchanged index preparation.  A lane owns a voxel and holds the sums in
 * registers (the same fma chain in rank order as veon_bev_pool_v2_fwd_planar: the same bits; rows
 * wider than 32 channels are walked in two or three passes, the class-merge state carried between
 * them), so the tile ends as 32 labels -- class merge, first-index arg-max, gate (the rule of
 * veon_classify_logits) -- and the pooled logit volume [B,Cp,Z,Y,X] is never written.
 * Tiles from 512 points up go to a CTA each, which classifies from its shared-memory tile.
 * Needs the plan's tile_start / tile_heavy tables, V % 32 == 0 and B*V <= 2^24, else
 * VEON_E_UNSUPPORTED / VEON_E_RANGE (the caller then pools the volume and calls
 * veon_classify_logits).  labels uint8 [B,X,Y,Z]. */
int veon_lift_classify_fwd(const float* depth, const float* pix,
                           const int32_t* ranks_depth, const int32_t* ranks_feat,
                           const int32_t* ranks_bev, const int32_t* tile_start,
                           const int32_t* tile_heavy, int64_t tile_heavy_ints,
                           int B, int Cp, int Q, int Z, int Y, int X, int64_t n_pix_rows,
                           const int32_t* class_of_prompt, int free_label,
                           uint8_t* labels, void* stream);
size_t veon_voxel_text_argmax_lowres_workspace_bytes(int B, int Q, int Zi, int Yi, int Xi);
int veon_voxel_text_argmax_lowres(const float* feat_occ_lr, const float* text_w,
                                  const int32_t* class_of_prompt, const float* bin_occ_lr,
                                  int B, int C, int Q, int Zi, int Yi, int Xi,
                                  int Z, int Y, int X, int free_label, uint8_t* labels,
                                  void* workspace, size_t ws_bytes, const void* w_image,
                                  void* stream);

/* The three tail entry points on a bfloat16 feature volume (feat_occ / feat_occ_lr: bfloat16
 * [B,C,Z,Y,X], as the pooling's _bf16 entries write it or a 3D decoder under autocast returns
 * it).  Every result equals the float32 twin's on the volume widened to float32: the same
 * labels byte for byte and the same logits value for value (NaN where it has NaN; only the sign
 * of an exact zero may differ).  A widened bfloat16 value is exactly TF32-representable, so the
 * tensor-core kernel reads the volume as it is (half the bytes) and drops the third product of
 * the 3xTF32 sum, which is exactly zero.  text_w, bin_occ / bin_occ_lr, w_image and every
 * output are the float32 twins'; so are the arguments, checks and error codes.  The route is
 * the one the float32 twin would take: the fp32 FFMA kernel reading bfloat16 where that one
 * takes it (C % 32 != 0, V % 4 != 0, Q > 128), else tcgen05, which here needs V % 8 == 0 and a
 * 16-byte aligned feat_occ; where it cannot have them the entry returns VEON_E_UNSUPPORTED and
 * the caller widens the volume and calls the float32 twin.  The workspace of the low-resolution
 * entry is sized by veon_voxel_text_argmax_lowres_workspace_bytes. */
int veon_voxel_text_argmax_bf16(const uint16_t* feat_occ, const float* text_w,
                                const int32_t* class_of_prompt, const float* bin_occ,
                                int B, int C, int Q, int Z, int Y, int X,
                                int free_label, uint8_t* labels, const void* w_image,
                                void* stream);
int veon_semantic_inference_3d_bf16(const float* text_w, const uint16_t* feat_occ,
                                    int B, int C, int Q, int Z, int Y, int X,
                                    float* sem_occ, const void* w_image, void* stream);
int veon_voxel_text_argmax_lowres_bf16(const uint16_t* feat_occ_lr, const float* text_w,
                                       const int32_t* class_of_prompt, const float* bin_occ_lr,
                                       int B, int C, int Q, int Zi, int Yi, int Xi,
                                       int Z, int Y, int X, int free_label, uint8_t* labels,
                                       void* workspace, size_t ws_bytes, const void* w_image,
                                       void* stream);

/* The three tail entry points, float32 and bfloat16, on a channels-last feature volume:
 * feat_occ / feat_occ_lr hold
 * [B,Z,Y,X,C] (float32, or bfloat16 for _cl_bf16), as a channels_last_3d [B,C,Z,Y,X] tensor
 * stores it, e.g. a 3D decoder running cuDNN's conv3d in that layout, or the pooling's _cl
 * entries.  Every result equals the channels-first twin's on the same volume made contiguous, bit
 * for bit: the tensor-core kernel reads each voxel's 32-channel segments into the same
 * tensor-memory lanes and columns and issues the same MMAs.  Only that kernel has a channels-last
 * loader, so these entries run exactly where the channels-first call on the contiguous volume
 * takes tcgen05 (C % 32 == 0, Q <= 128, V % 4 == 0) and feat_occ is 16-byte aligned; elsewhere
 * they return VEON_E_UNSUPPORTED and the caller makes the volume contiguous.  A bfloat16 volume
 * with V % 8 == 4 runs here although its channels-first twin widens it: the bits are the same.
 * Arguments, checks and error codes are the channels-first twins'; text_w, bin_occ /
 * bin_occ_lr, w_image and every output keep their layout. */
int veon_voxel_text_argmax_cl(const float* feat_occ, const float* text_w,
                              const int32_t* class_of_prompt, const float* bin_occ,
                              int B, int C, int Q, int Z, int Y, int X,
                              int free_label, uint8_t* labels, const void* w_image,
                              void* stream);
int veon_voxel_text_argmax_cl_bf16(const uint16_t* feat_occ, const float* text_w,
                                   const int32_t* class_of_prompt, const float* bin_occ,
                                   int B, int C, int Q, int Z, int Y, int X,
                                   int free_label, uint8_t* labels, const void* w_image,
                                   void* stream);
int veon_semantic_inference_3d_cl(const float* text_w, const float* feat_occ,
                                  int B, int C, int Q, int Z, int Y, int X,
                                  float* sem_occ, const void* w_image, void* stream);
int veon_semantic_inference_3d_cl_bf16(const float* text_w, const uint16_t* feat_occ,
                                       int B, int C, int Q, int Z, int Y, int X,
                                       float* sem_occ, const void* w_image, void* stream);
int veon_voxel_text_argmax_lowres_cl(const float* feat_occ_lr, const float* text_w,
                                     const int32_t* class_of_prompt, const float* bin_occ_lr,
                                     int B, int C, int Q, int Zi, int Yi, int Xi,
                                     int Z, int Y, int X, int free_label, uint8_t* labels,
                                     void* workspace, size_t ws_bytes, const void* w_image,
                                     void* stream);
int veon_voxel_text_argmax_lowres_cl_bf16(const uint16_t* feat_occ_lr, const float* text_w,
                                          const int32_t* class_of_prompt,
                                          const float* bin_occ_lr,
                                          int B, int C, int Q, int Zi, int Yi, int Xi,
                                          int Z, int Y, int X, int free_label, uint8_t* labels,
                                          void* workspace, size_t ws_bytes,
                                          const void* w_image, void* stream);

/* Multi-GPU callers that overlap a collective (NCCL on another stream) with the path: the
 * persistent grids here fill every SM, so the collective's CTAs wait for a kernel boundary.
 * veon_reserve_sms(n) makes every persistent grid of the library launch on (SM count - n) SMs;
 * returns the previous value; 0 (the default) uses them all.  Process-wide setting. */
int veon_reserve_sms(int n);

#ifdef __cplusplus
}
#endif
#endif  /* VEON_LIFT_H_ */
