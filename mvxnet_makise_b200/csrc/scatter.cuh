// Internal interface of stage 4 (dense grid fill), shared with the fused path.
#pragma once
#include "common.cuh"

namespace mvx {
// out (B, C, G) fp32 = cell2vid[b][g] < 0 ? 0 : feat[b][vid][c]; feat frames at stride vcap*C. Needs G % 4 == 0.
int launch_grid_fill(const int *cell2vid, const float *feat, float *out, int B, long long G, int C, int vcap, cudaStream_t st);
int launch_occ_from_map(const int *cell2vid, unsigned *occ, int B, long long G, cudaStream_t st);
// plane-sequential fill: feat element (v, c) of frame f at feat[f*feat_frame_stride + v*feat_vs + c*feat_cs]
int launch_grid_fill_planes(const unsigned *occ, const int *cell2vid, const float *feat, long long feat_frame_stride, int feat_vs,
                            int feat_cs, float *out, int B, long long G, int C, cudaStream_t st);
}  // namespace mvx
