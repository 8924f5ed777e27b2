// Internal interface of the stage-1 voxelizer (shared with the fused path).
#pragma once
#include "common.cuh"

namespace mvx {

constexpr int kMaxFrames = 32;  // frames per call (offsets travel as a by-value kernel argument)

struct FrameOffsets {
    int off[kMaxFrames + 1];
};

struct VoxLayout {
    unsigned H;  // hash slots per frame (power of two >= 2*cap)
    int nblk;    // 1024-point blocks per frame
    size_t ff_begin, ff_end, zero_begin, zero_end;
    size_t hkeys, hfirst, hcount, hvid, pslot, blocksum, vox_total, seg_off, cursor, seg_pts, seg_vid;
    size_t total;
};

struct VoxParams {
    FrameOffsets fo;
    const float *points;
    int point_stride;
    const int *cell_idx;
    double lo[3], size[3];
    int shape[3];
    int have_grid;
    long long G;
    int T, cap;
    unsigned H;
    int nblk;
    unsigned long long *hkeys;
    unsigned *hfirst, *hcount;
    int *hvid, *pslot, *blocksum, *vox_total, *seg_off, *cursor, *seg_pts, *seg_vid;
    int *counts;
    mvx_voxel_out_t out;
};

// Cell of a point: fp64 subtract and TRUE division, C truncation (Preprocessing.py:67-69; SURVEY.md trap 1). Returns whether
// the cell lies inside the grid. The voxelizer keys points with it, and the pixel-tile mark of the fused path (gather.cu)
// filters with it, so the mark sees exactly the points that can become rows.
__device__ __forceinline__ bool vox_cell_index(const double (&lo)[3], const double (&size)[3], const int (&shape)[3], float x, float y,
                                               float z, int &ix, int &iy, int &iz) {
    ix = (int)(((double)x - lo[0]) / size[0]);
    iy = (int)(((double)y - lo[1]) / size[1]);
    iz = (int)(((double)z - lo[2]) / size[2]);
    return ix >= 0 && ix < shape[0] && iy >= 0 && iy < shape[1] && iz >= 0 && iz < shape[2];
}

VoxLayout vox_layout(int B, int cap);
size_t vox_workspace_bytes(int B, int cap);
int vox_run(const mvx_grid_t *grid, int B, int cap, const float *points, int point_stride, const int32_t *pt_off_host,
            const int32_t *cell_idx, int T, const mvx_voxel_out_t *out, void *workspace, size_t workspace_bytes,
            cudaStream_t st);

}  // namespace mvx
