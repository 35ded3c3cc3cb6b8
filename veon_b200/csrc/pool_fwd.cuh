// Internal interface between the forward pooling translation units.
#pragma once
#include "common.cuh"

namespace veon {

// pool_fwd_stream.cu: the two-role streaming forward (rows -> L2 ring -> dense volume)
bool fwd_stream_supported(int B, int C, int64_t V, const void* feat, const void* out,
                          int64_t n_feat_rows);
size_t fwd_stream_workspace_bytes(int C);
int launch_fwd_stream(const float* depth, const float* feat, const int32_t* rd, const int32_t* rf,
                      const int32_t* rb, const int32_t* tile_start, const uint32_t* tile_occ,
                      const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                      float* out, void* workspace, size_t ws_bytes, cudaStream_t stream);

// pool_fwd.cu: the CTA-per-heavy-tile grid, queued as a programmatic dependent of whatever was
// launched last on `stream` (it joins that grid before it completes)
int launch_heavy_behind(const float* depth, const float* feat, const int32_t* rd,
                        const int32_t* rf, const int32_t* rb, const int32_t* tile_start,
                        const int32_t* heavy, int64_t heavy_ints, int B, int C, int64_t V,
                        float* out, int min_points, cudaStream_t stream);

}  // namespace veon
