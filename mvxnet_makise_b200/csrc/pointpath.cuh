// Workspace layout of the fused point path, shared by the forward (pointpath.cu) and the training-mode backward
// (backward.cu).
#pragma once
#include "common.cuh"

namespace mvx {

enum Region {
    R_VOXWS = 0, R_VOX_COORD, R_VOX_CNT, R_VOX_ROW0, R_ROW_POINT, R_ROW_VOX, R_CELL2VID, R_NHWC0, R_NHWC1, R_NHWC2,
    R_VOX8, R_PROJ, R_ROWA_W, R_A1, R_Y1, R_Y2, R_Y3, R_Y4, R_Y5, R_X6, R_Y6, R_X7, R_Y7, R_ROWB_W, R_ROWB_V, R_X8,
    R_VFEAT, R_STATS, R_VMAX6, R_VMAX7, R_VMAX8, R_WPACK, R_OCC, R_VFEAT_T, R_Z, R_BINCNT, R_BINSTART, R_PERM, R_ROWMAX, R_CHMAX, R_A1MAX, R_TILES, R_Y8, R_COUNT
};
static_assert(R_COUNT <= MVX_WS_REGIONS, "too many regions");

extern const char *kRegionNames[R_COUNT];

constexpr int kCin[MVX_NUM_LAYERS] = {768, 768, 128, 128, 16, 32, 32, 128};   // padded
constexpr int kCout[MVX_NUM_LAYERS] = {768, 128, 128, 16, 16, 16, 64, 128};
constexpr int kStatStride = 768 * 2;  // doubles per (layer, frame)

struct Layout {
    size_t off[R_COUNT];
    size_t total;        // inference workspace (everything but Y8)
    size_t total_train;  // + Y8, the raw output of the last FCN, which only the backward needs
    int capA, capB;
    long long G;
};

int make_layout(const mvx_pointpath_args_t *a, Layout &L);
int pointpath_forward(const mvx_pointpath_args_t *a, bool train);

// backward workspace of mvx_pointpath_backward (backward.cu): its size, and where fcn1's dpre [B][capA][768] stays after it
void backward_ws_layout(const mvx_pointpath_args_t *a, const Layout &L, size_t *total, size_t *dpre1_off);
// W (Cout, Cin) row-major from W^T (Cin, Cout)
int launch_transpose_w(const float *wt, float *w, int Cin, int Cout, cudaStream_t st);

}  // namespace mvx
