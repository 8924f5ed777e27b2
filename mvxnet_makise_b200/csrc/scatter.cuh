// Internal interface of stage 4 (dense grid fill), shared with the fused path and the backward passes.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mvx {

// ---- element types of the dense grid (MVX_DTYPE_*) --------------------------------------------------------------------
// Every element of a 16-bit grid is one fp32 feature rounded once to nearest-even (what torch's `.to(dtype)` of the fp32 grid
// gives); a 16-bit grid gradient widens to fp32 exactly.
template <typename T> __device__ __forceinline__ T grid_elem(float v);
template <> __device__ __forceinline__ float grid_elem<float>(float v) { return v; }
template <> __device__ __forceinline__ __half grid_elem<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 grid_elem<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ float grid_f32(float v) { return v; }
__device__ __forceinline__ float grid_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float grid_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

// Calls f(T{}) with the element type that `dtype` names and returns its status; MVX_EINVAL for any other value.
inline bool grid_dtype_ok(int dtype) { return dtype == MVX_DTYPE_F32 || dtype == MVX_DTYPE_F16 || dtype == MVX_DTYPE_BF16; }
#define MVX_GRID_DTYPE_MSG "grid dtype must be MVX_DTYPE_F32 (0), MVX_DTYPE_F16 (1) or MVX_DTYPE_BF16 (2)"
template <typename F>
int with_grid_dtype(int dtype, F &&f) {
    MVX_REQUIRE(grid_dtype_ok(dtype), MVX_EINVAL, MVX_GRID_DTYPE_MSG);
    switch (dtype) {
    case MVX_DTYPE_F16: return f(__half{});
    case MVX_DTYPE_BF16: return f(__nv_bfloat16{});
    default: return f(float{});
    }
}

// out (B, C, G) of element type `out_dtype` = cell2vid[b][g] < 0 ? 0 : feat[b][vid][c]; feat frames at stride vcap*C. Needs G % 4 == 0.
int launch_grid_fill(const int *cell2vid, const float *feat, void *out, int out_dtype, int B, long long G, int C, int vcap,
                     cudaStream_t st);
int launch_occ_from_map(const int *cell2vid, unsigned *occ, int B, long long G, cudaStream_t st);
// plane-sequential fill: feat element (v, c) of frame f at feat[f*feat_frame_stride + v*feat_vs + c*feat_cs]
int launch_grid_fill_planes(const unsigned *occ, const int *cell2vid, const float *feat, long long feat_frame_stride, int feat_vs,
                            int feat_cs, void *out, int out_dtype, int B, long long G, int C, cudaStream_t st);
}  // namespace mvx
