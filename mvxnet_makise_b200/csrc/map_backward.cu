// Backward of the PointFusion gather into the FPN maps (modules/imhead/Pipe.py:23-82): dLoss/d maps of the last training
// forward, from fcn1's dpre that mvx_pointpath_backward leaves in its workspace. Pixel-first, the adjoint of the pixel-first
// fcn1 of the forward (DESIGN.md §2):
//     dZ_l[p] = sum over the (row r, corner c) that sample pixel p of wgt_c(r) * dpre1[r]          (768 wide)
//     dF_l[p] = dZ_l[p] W1[:, 256 l : 256 (l+1)]                                                     (pixels x 768) (768 x 256)
// 18 GFLOP per KITTI frame, against 120 for the row-first order (dA1 = dpre1 W1, then a scatter of dA1).
//  (1) per level, a pixel CSR: the kept rows bucketed by the 2x2 corner block ("cell") they sample, cells in 4x4 blocks with
//      Morton order inside, like the forward's combine sort. Counting sort (histogram, scan, scatter), made stable in the
//      compact row index by a rank pass: every sum below runs in one fixed order (no fp32 atomics, reruns are bit-identical);
//  (2) dZ per pixel: the rows of the at most four cells that touch it, corner order 00 10 01 11, CSR order inside a cell, one
//      thread per 4 columns. A CTA owns a 4x4 pixel block in Morton order (four thread groups, one 2x2 quarter each), so the
//      dpre rows of neighbouring cells are L1 / L2 hits;
//  (3) per level dZ_l W1_l on the one-tile layer kernel in 3xTF32 (gradients have no bounded range), stored channel-major:
//      the (B, 256, H_l, W_l) layout of the caller's maps.
#include "gather.cuh"
#include "layers.cuh"
#include "pointpath.cuh"

namespace mvx {
namespace {

constexpr int kMbCols = 768;              // fcn1 outputs = columns of dpre1 and dZ
constexpr int kMbGroup = kMbCols / 4;     // dZ kernel: a group owns one pixel at a time, one float4 column group per thread
constexpr int kMbGroups = 4;              // groups per CTA, one 2x2 quarter of the 4x4 pixel block each

struct MbLevel {
    int h, w;              // map extent
    float rs_h, rs_w;      // regionSize = imsize / (h, w) in fp32 (Pipe.py:41-45)
    int nbins;             // cells over the top-left corners (i0, i1) in [-1, h-1] x [-1, w-1], 4x4 blocks of 16
    int *bin_count;        // [B][nbins]: histogram, then the scatter cursor
    int *bin_start;        // [B][nbins + 1]
    int *tmp;              // [B][capA]: rows in scatter (arrival) order
    int *row;              // [B][capA]: CSR, compact row of every entry (ascending inside a cell)
    float4 *wgt;           // [B][capA]: the entry's four corner weights
    float *dz;             // [B][h * w][768]
};

struct MbRows {
    const int *counts;     // [B][4]
    const float *vox8;     // [B][capA][8] of the training forward
    const float *proj;     // [B][capA][2]
    int capA;
    float eps;
};

inline int mb_bins(int h, int w) { return ((h + 1 + 3) / 4) * ((w + 1 + 3) / 4) * 16; }

__device__ __forceinline__ int mb_cell_key(int ys, int xs, int w) {   // ys = i0 + 1 in [0, h], xs = i1 + 1 in [0, w]
    const int wb = (w + 1 + 3) / 4;
    const int inner = ((ys & 2) << 2) | ((xs & 2) << 1) | ((ys & 1) << 1) | (xs & 1);
    return ((ys >> 2) * wb + (xs >> 2)) * 16 + inner;
}

// cell of compact row r at this level, or -1: the frame's pad row, an origin point (the forward zeroes its features,
// Pipe.py:53-59,80), or a cell with no corner inside the map
__device__ __forceinline__ int mb_cell_of(const MbLevel &L, float prow, float pcol, float eps, CellRef *cr) {
    const CellRef c = cell_of(prow, pcol, L.rs_h, L.rs_w, eps);
    if (c.i0 < -1 || c.i0 >= L.h || c.i1 < -1 || c.i1 >= L.w) return -1;
    if (cr) *cr = c;
    return mb_cell_key(c.i0 + 1, c.i1 + 1, L.w);
}
__device__ __forceinline__ int mb_row_key(const MbRows &a, const MbLevel &L, int f, int r, CellRef *cr) {
    if (r >= a.counts[f * 4 + 1]) return -1;
    const size_t ro = (size_t)f * a.capA + r;
    const float4 xyz = __ldg(reinterpret_cast<const float4 *>(a.vox8 + ro * 8));
    if (xyz.x == 0.f && xyz.y == 0.f && xyz.z == 0.f) return -1;
    const float2 pr = __ldg(reinterpret_cast<const float2 *>(a.proj) + ro);
    return mb_cell_of(L, pr.x, pr.y, a.eps, cr);
}

// the same rows read straight from a dense (R, 9) voxel tensor after featureMaping's forward (one frame, f = 0): every slot is a
// row, pad slots (x == y == z == 0) sample nothing, the projection (row, col) is in columns 7 and 8
struct MbDenseRows {
    const float *vox9;
    int capA;              // R: the row count and the stride of the CSR arrays
    float eps;
};
__device__ __forceinline__ int mb_row_key(const MbDenseRows &a, const MbLevel &L, int f, int r, CellRef *cr) {
    if (r >= a.capA) return -1;
    const float *s = a.vox9 + (size_t)r * 9;
    if (s[0] == 0.f && s[1] == 0.f && s[2] == 0.f) return -1;
    return mb_cell_of(L, s[7], s[8], a.eps, cr);
}

template <class Rows>
__device__ __forceinline__ void mb_hist(const Rows &a, const MbLevel &L) {
    const int f = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
    const int key = mb_row_key(a, L, f, r, nullptr);
    if (key >= 0) atomicAdd(L.bin_count + (size_t)f * L.nbins + key, 1);
}
__global__ void __launch_bounds__(256) mb_hist_kernel(MbRows a, MbLevel L) { mb_hist(a, L); }
__global__ void __launch_bounds__(256) mbd_hist_kernel(MbDenseRows a, MbLevel L) { mb_hist(a, L); }

__global__ void __launch_bounds__(1024) mb_scan_kernel(MbLevel L) {   // one CTA per frame, four bins per thread and round
    const int f = blockIdx.x, nb = L.nbins;
    int *cnt = L.bin_count + (size_t)f * nb, *start = L.bin_start + (size_t)f * (nb + 1);
    int carry = 0;
    for (int b0 = 0; b0 < nb; b0 += 4096) {
        const int b = b0 + threadIdx.x * 4;
        int v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = b + q < nb ? cnt[b + q] : 0;
        int total;
        int ex = carry + block_exclusive_scan(v[0] + v[1] + v[2] + v[3], &total);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (b + q < nb) {
                start[b + q] = ex;
                cnt[b + q] = 0;   // becomes the scatter cursor
            }
            ex += v[q];
        }
        carry += total;
    }
    if (threadIdx.x == 0) start[nb] = carry;
}

template <class Rows>
__device__ __forceinline__ void mb_scatter(const Rows &a, const MbLevel &L) {
    const int f = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
    const int key = mb_row_key(a, L, f, r, nullptr);
    if (key < 0) return;
    const int pos = L.bin_start[(size_t)f * (L.nbins + 1) + key] + atomicAdd(L.bin_count + (size_t)f * L.nbins + key, 1);
    L.tmp[(size_t)f * a.capA + pos] = r;
}
__global__ void __launch_bounds__(256) mb_scatter_kernel(MbRows a, MbLevel L) { mb_scatter(a, L); }
__global__ void __launch_bounds__(256) mbd_scatter_kernel(MbDenseRows a, MbLevel L) { mb_scatter(a, L); }

// the scatter's order inside a cell depends on which atomic came first: place every row at its rank among the cell's rows
template <class Rows>
__device__ __forceinline__ void mb_rank(const Rows &a, const MbLevel &L) {
    const int f = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
    CellRef c;
    const int key = mb_row_key(a, L, f, r, &c);
    if (key < 0) return;
    const int *start = L.bin_start + (size_t)f * (L.nbins + 1);
    const int s0 = start[key], s1 = start[key + 1];
    const int *seg = L.tmp + (size_t)f * a.capA;
    int rank = 0;
    for (int e = s0; e < s1; ++e) rank += seg[e] < r;
    const size_t o = (size_t)f * a.capA + s0 + rank;
    L.row[o] = r;
    L.wgt[o] = corner_weights(c, L.h, L.w);
}
__global__ void __launch_bounds__(256) mb_rank_kernel(MbRows a, MbLevel L) { mb_rank(a, L); }
__global__ void __launch_bounds__(256) mbd_rank_kernel(MbDenseRows a, MbLevel L) { mb_rank(a, L); }

__global__ void __launch_bounds__(kMbGroup * kMbGroups) mb_dz_kernel(MbRows a, MbLevel L, const float *__restrict__ dpre1) {
    const int f = blockIdx.y, grp = threadIdx.x / kMbGroup, col0 = (threadIdx.x % kMbGroup) * 4;
    const int wbp = (L.w + 3) / 4, by = blockIdx.x / wbp, bx = blockIdx.x - by * wbp;
    const int *start = L.bin_start + (size_t)f * (L.nbins + 1);
    const int *rows = L.row + (size_t)f * a.capA;
    const float4 *wgt = L.wgt + (size_t)f * a.capA;
    const float *D = dpre1 + (size_t)f * a.capA * kMbCols + col0;
    for (int i = grp * 4; i < grp * 4 + 4; ++i) {   // Morton order inside the 4x4 pixel block
        const int y = by * 4 + ((((i >> 3) & 1) << 1) | ((i >> 1) & 1)), x = bx * 4 + ((((i >> 2) & 1) << 1) | (i & 1));
        if (y >= L.h || x >= L.w) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < 4; ++c) {   // pixel (y, x) is corner c = 00, 10, 01, 11 of the cell with top-left (y - dy, x - dx)
            const int dy = c & 1, dx = c >> 1;
            const int key = mb_cell_key(y - dy + 1, x - dx + 1, L.w);
            const int e1 = start[key + 1];
#pragma unroll 4
            for (int e = start[key]; e < e1; ++e) {
                const float4 w4 = wgt[e];
                const float w = c == 0 ? w4.x : (c == 1 ? w4.y : (c == 2 ? w4.z : w4.w));
                const float4 d = __ldg(reinterpret_cast<const float4 *>(D + (size_t)rows[e] * kMbCols));
                acc.x = fmaf(w, d.x, acc.x), acc.y = fmaf(w, d.y, acc.y), acc.z = fmaf(w, d.z, acc.z), acc.w = fmaf(w, d.w, acc.w);
            }
        }
        *reinterpret_cast<float4 *>(L.dz + ((size_t)f * L.h * L.w + (size_t)y * L.w + x) * kMbCols + col0) = acc;
    }
}

// featureMaping's adjoint (dense rows, one frame): d_map[c][p] = sum over the (row r, corner) that sample pixel p of
// wgt * d_out[r][col0 + c], channel-major. A CTA owns 32 consecutive pixels x 32 channels, a warp four of the pixels with one
// channel per lane (coalesced reads of the d_out rows); the sums run in the CSR order of mb_dz_kernel, then go through a shared
// tile to the (C, H, W) map
constexpr int kFmPix = 32;
__global__ void __launch_bounds__(256) mbd_dz_kernel(MbDenseRows a, MbLevel L, const float *__restrict__ d_out, int ld, int col0, int C,
                                                     float *__restrict__ d_map) {
    __shared__ float tile[32][kFmPix + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hw = L.h * L.w, p0 = blockIdx.x * kFmPix, c0 = blockIdx.y * 32, c = c0 + lane;
    const int *start = L.bin_start, *rows = L.row;
    for (int i = 0; i < kFmPix / 8; ++i) {
        const int pl = warp * (kFmPix / 8) + i, p = p0 + pl;
        float acc = 0.f;
        if (p < hw && c < C) {
            const int y = p / L.w, x = p - y * L.w;
#pragma unroll
            for (int q = 0; q < 4; ++q) {   // pixel (y, x) is corner q = 00, 10, 01, 11 of the cell with top-left (y - dy, x - dx)
                const int dy = q & 1, dx = q >> 1;
                const int key = mb_cell_key(y - dy + 1, x - dx + 1, L.w);
                const int e1 = start[key + 1];
                for (int e = start[key]; e < e1; ++e) {
                    const float4 w4 = L.wgt[e];
                    const float w = q == 0 ? w4.x : (q == 1 ? w4.y : (q == 2 ? w4.z : w4.w));
                    acc = fmaf(w, __ldg(d_out + (size_t)rows[e] * ld + col0 + c), acc);
                }
            }
        }
        tile[lane][pl] = acc;
    }
    __syncthreads();
    for (int cc = warp; cc < 32; cc += 8)
        if (c0 + cc < C && p0 + lane < hw) d_map[(size_t)(c0 + cc) * hw + p0 + lane] = tile[cc][lane];
}

struct MbLayout {
    size_t wt1, wpack, cnt[MVX_NUM_LEVELS], start[MVX_NUM_LEVELS], tmp[MVX_NUM_LEVELS], row[MVX_NUM_LEVELS], wgt[MVX_NUM_LEVELS],
        dz[MVX_NUM_LEVELS], total;
};

void mb_layout(const mvx_pointpath_args_t *a, const Layout &L, MbLayout &M) {
    size_t o = 0;
    auto take = [&](size_t &slot, size_t bytes) {
        slot = o;
        o += (bytes + 255) / 256 * 256;
    };
    const size_t B = a->B, capA = L.capA;
    take(M.wt1, (size_t)MVX_NUM_LEVELS * kMbCols * a->map_c * 4);
    take(M.wpack, tc_wpack_bytes(kMbCols, a->map_c));
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        const size_t nb = mb_bins(a->map_h[l], a->map_w[l]);
        take(M.cnt[l], B * nb * 4);
        take(M.start[l], B * (nb + 1) * 4);
        take(M.tmp[l], B * capA * 4);
        take(M.row[l], B * capA * 4);
        take(M.wgt[l], B * capA * 16);
        take(M.dz[l], B * (size_t)a->map_h[l] * a->map_w[l] * kMbCols * 4);
    }
    M.total = o;
}

}  // namespace

int pointpath_backward_maps(const mvx_pointpath_args_t *a, const void *bws_v, size_t bws_bytes, float *const d_maps[MVX_NUM_LEVELS],
                            void *ws_v, size_t ws_bytes) {
    Layout L;
    int rc = make_layout(a, L);
    if (rc) return rc;
    MbLayout M;
    mb_layout(a, L, M);
    size_t bws_total = 0, dpre1_off = 0;
    backward_ws_layout(a, L, &bws_total, &dpre1_off);
    MVX_REQUIRE(d_maps && bws_v && ws_v && a->workspace && a->counts && a->wt[0], MVX_EINVAL, "null pointer");
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) MVX_REQUIRE(d_maps[l], MVX_EINVAL, "null map gradient");
    MVX_REQUIRE(a->workspace_bytes >= L.total_train, MVX_ESPACE, "the map backward needs the training workspace of the forward");
    MVX_REQUIRE(bws_bytes >= bws_total, MVX_ESPACE, "backward workspace too small");
    MVX_REQUIRE(ws_bytes >= M.total, MVX_ESPACE, "map backward workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    char *ws = static_cast<char *>(ws_v), *pws = static_cast<char *>(a->workspace);
    const int B = a->B, C = a->map_c;
    const float *dpre1 = reinterpret_cast<const float *>(static_cast<const char *>(bws_v) + dpre1_off);
    float *wt1 = reinterpret_cast<float *>(ws + M.wt1);
    const MbRows rows{a->counts, reinterpret_cast<const float *>(pws + L.off[R_VOX8]), reinterpret_cast<const float *>(pws + L.off[R_PROJ]),
                      L.capA, a->gather_eps};
    MbLevel lv[MVX_NUM_LEVELS];
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        MbLevel &v = lv[l];
        v.h = a->map_h[l], v.w = a->map_w[l];
        v.rs_h = a->imsize_h / (float)v.h, v.rs_w = a->imsize_w / (float)v.w;   // as the forward's MapSet
        v.nbins = mb_bins(v.h, v.w);
        v.bin_count = reinterpret_cast<int *>(ws + M.cnt[l]), v.bin_start = reinterpret_cast<int *>(ws + M.start[l]);
        v.tmp = reinterpret_cast<int *>(ws + M.tmp[l]), v.row = reinterpret_cast<int *>(ws + M.row[l]);
        v.wgt = reinterpret_cast<float4 *>(ws + M.wgt[l]), v.dz = reinterpret_cast<float *>(ws + M.dz[l]);
    }
    // (1) pixel CSR of every level
    const dim3 rgrid((unsigned)ceil_div(L.capA, 256), B);
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        MVX_CUDA_CHECK(cudaMemsetAsync(lv[l].bin_count, 0, (size_t)B * lv[l].nbins * 4, st));
        mb_hist_kernel<<<rgrid, 256, 0, st>>>(rows, lv[l]);
        MVX_LAUNCH_CHECK();
        mb_scan_kernel<<<B, 1024, 0, st>>>(lv[l]);
        MVX_LAUNCH_CHECK();
        mb_scatter_kernel<<<rgrid, 256, 0, st>>>(rows, lv[l]);
        MVX_LAUNCH_CHECK();
        mb_rank_kernel<<<rgrid, 256, 0, st>>>(rows, lv[l]);
        MVX_LAUNCH_CHECK();
    }
    // (2) dZ of every level
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        const unsigned blocks = (unsigned)(ceil_div(lv[l].h, 4) * ceil_div(lv[l].w, 4));
        mb_dz_kernel<<<dim3(blocks, B), kMbGroup * kMbGroups, 0, st>>>(rows, lv[l], dpre1);
        MVX_LAUNCH_CHECK();
    }
    // (3) dF_l = dZ_l W1_l: W1_l (768, 256) = the transposed rows 256 l .. 256 l + 255 of the stored W1^T (768, 768)
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        float *w1l = wt1 + (size_t)l * kMbCols * C;
        rc = launch_transpose_w(a->wt[0] + (size_t)l * C * kMbCols, w1l, C, kMbCols, st);
        if (rc) return rc;
        const long long px = (long long)lv[l].h * lv[l].w;
        LayerArgs la{};
        la.X = lv[l].dz, la.ldx = kMbCols, la.Cin = kMbCols, la.Wt = w1l, la.bias = nullptr, la.Cout = C;
        la.Y = d_maps[l], la.ldy = C, la.rows_mode = 0, la.rows_fixed = px, la.rowcap = (int)px, la.T = 1, la.eps = a->bn_eps;
        la.plain = 1, la.f16_ok = 0, la.y_nchw = 1;
        rc = launch_layer_tc(la, B, reinterpret_cast<float *>(ws + M.wpack), st);
        if (rc) return rc;
    }
    return MVX_OK;
}

}  // namespace mvx

extern "C" int mvx_pointpath_backward_maps_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes) {
    mvx::Layout L;
    int rc = mvx::make_layout(args, L);
    if (rc) return rc;
    if (!bytes) return MVX_EINVAL;
    mvx::MbLayout M;
    mvx::mb_layout(args, L, M);
    *bytes = M.total;
    return MVX_OK;
}

extern "C" int mvx_pointpath_backward_maps(const mvx_pointpath_args_t *args, const void *backward_ws, size_t backward_ws_bytes,
                                           float *const d_maps[MVX_NUM_LEVELS], void *ws, size_t ws_bytes) {
    return mvx::pointpath_backward_maps(args, backward_ws, backward_ws_bytes, d_maps, ws, ws_bytes);
}

namespace mvx {
namespace {

struct FmLayout {
    size_t cnt[MVX_NUM_LEVELS], start[MVX_NUM_LEVELS], tmp[MVX_NUM_LEVELS], row[MVX_NUM_LEVELS], wgt[MVX_NUM_LEVELS], total;
};

int fm_layout(long long R, const int32_t *map_h, const int32_t *map_w, FmLayout &M) {
    MVX_REQUIRE(map_h && map_w, MVX_EINVAL, "null map extents");
    MVX_REQUIRE(R >= 0 && R <= 0x7FFFFFFF, MVX_EINVAL, "feature mapping backward: R must be in [0, 2^31)");
    size_t o = 0;
    auto take = [&](size_t &slot, size_t bytes) {
        slot = o;
        o += (bytes + 255) / 256 * 256;
    };
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        MVX_REQUIRE(map_h[l] > 0 && map_w[l] > 0, MVX_EINVAL, "bad map extent");
        const size_t nb = mb_bins(map_h[l], map_w[l]);
        take(M.cnt[l], nb * 4);
        take(M.start[l], (nb + 1) * 4);
        take(M.tmp[l], (size_t)R * 4);
        take(M.row[l], (size_t)R * 4);
        take(M.wgt[l], (size_t)R * 16);
    }
    M.total = o;
    return MVX_OK;
}

}  // namespace
}  // namespace mvx

extern "C" int mvx_feature_mapping_backward_workspace_bytes(int64_t R, const int32_t *map_h, const int32_t *map_w, size_t *bytes) {
    MVX_REQUIRE(bytes, MVX_EINVAL, "null pointer");
    mvx::FmLayout M;
    const int rc = mvx::fm_layout(R, map_h, map_w, M);
    if (rc) return rc;
    *bytes = M.total;
    return MVX_OK;
}

extern "C" int mvx_feature_mapping_backward(const float *voxels, int64_t R, const float *d_out, const int32_t *map_h, const int32_t *map_w,
                                            int32_t C, float imsize_h, float imsize_w, float eps, float *const *d_maps, void *ws_v,
                                            size_t ws_bytes, void *stream) {
    mvx::FmLayout M;
    int rc = mvx::fm_layout(R, map_h, map_w, M);
    if (rc) return rc;
    MVX_REQUIRE(d_maps && ws_v && (R == 0 || (voxels && d_out)), MVX_EINVAL, "null pointer");
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) MVX_REQUIRE(d_maps[l], MVX_EINVAL, "null map gradient");
    MVX_REQUIRE(C > 0 && C % 4 == 0, MVX_EINVAL, "C must be a multiple of 4");
    MVX_REQUIRE(ws_bytes >= M.total, MVX_ESPACE, "feature mapping backward workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char *ws = static_cast<char *>(ws_v);
    const mvx::MbDenseRows rows{voxels, (int)R, eps};
    const dim3 rgrid((unsigned)mvx::ceil_div(R, 256), 1);
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        mvx::MbLevel v{};
        v.h = map_h[l], v.w = map_w[l];
        v.rs_h = imsize_h / (float)v.h, v.rs_w = imsize_w / (float)v.w;   // as mvx_feature_mapping's MapSet
        v.nbins = mvx::mb_bins(v.h, v.w);
        v.bin_count = reinterpret_cast<int *>(ws + M.cnt[l]), v.bin_start = reinterpret_cast<int *>(ws + M.start[l]);
        v.tmp = reinterpret_cast<int *>(ws + M.tmp[l]), v.row = reinterpret_cast<int *>(ws + M.row[l]);
        v.wgt = reinterpret_cast<float4 *>(ws + M.wgt[l]), v.dz = nullptr;
        MVX_CUDA_CHECK(cudaMemsetAsync(v.bin_count, 0, (size_t)v.nbins * 4, st));
        if (R > 0) {
            mvx::mbd_hist_kernel<<<rgrid, 256, 0, st>>>(rows, v);
            MVX_LAUNCH_CHECK();
        }
        mvx::mb_scan_kernel<<<1, 1024, 0, st>>>(v);
        MVX_LAUNCH_CHECK();
        if (R > 0) {
            mvx::mbd_scatter_kernel<<<rgrid, 256, 0, st>>>(rows, v);
            MVX_LAUNCH_CHECK();
            mvx::mbd_rank_kernel<<<rgrid, 256, 0, st>>>(rows, v);
            MVX_LAUNCH_CHECK();
        }
        const long long hw = (long long)v.h * v.w;
        mvx::mbd_dz_kernel<<<dim3((unsigned)mvx::ceil_div(hw, mvx::kFmPix), (unsigned)mvx::ceil_div(C, 32)), 256, 0, st>>>(
            rows, v, d_out, 3 * C, l * C, C, d_maps[l]);
        MVX_LAUNCH_CHECK();
    }
    return MVX_OK;
}
