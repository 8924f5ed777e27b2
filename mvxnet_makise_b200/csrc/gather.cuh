// Internal interface of stage 2 (projection + PointFusion gather), shared with the fused path.
#pragma once
#include "common.cuh"

namespace mvx {

struct MapSet {
    const float *nhwc[MVX_NUM_LEVELS];  // channels-last copies (per frame stride = frame_stride[l] floats)
    size_t frame_stride[MVX_NUM_LEVELS];
    int h[MVX_NUM_LEVELS], w[MVX_NUM_LEVELS];
    float rs_h[MVX_NUM_LEVELS], rs_w[MVX_NUM_LEVELS];  // regionSize = imsize / (Hf, Wf) in fp32 (Pipe.py:41-45)
    int C;
};

// The 2x2 corner block a projected point samples at one FPN level: top-left corner (i0, i1) and the fractional parts.
// Index math and (inverted) weights of Pipe.py:62-75 in the fp32 order of gather_row_warp; the forward's combine and the
// map backward's pixel CSR both take their corners from here, so the adjoint picks exactly the forward's pixels.
struct CellRef {
    int i0, i1;
    float wa, wb;
};
__device__ __forceinline__ CellRef cell_of(float prow, float pcol, float rs_h, float rs_w, float eps) {
    const float q0 = __fsub_rn(__fdiv_rn(prow, rs_h), eps);
    const float q1 = __fsub_rn(__fdiv_rn(pcol, rs_w), eps);
    CellRef c;
    c.i0 = (int)q0, c.i1 = (int)q1;   // .long(): truncation toward zero
    c.wa = __fsub_rn(q0, (float)c.i0), c.wb = __fsub_rn(q1, (float)c.i1);
    return c;
}
// weights of the corners (i0,i1), (i0+1,i1), (i0,i1+1), (i0+1,i1+1); 0 where the corner lies outside the H x W map (row H /
// column W are the zero pad of Pipe.py:47-48)
__device__ __forceinline__ float4 corner_weights(const CellRef &c, int H, int W) {
    const bool r0 = c.i0 >= 0 && c.i0 < H, r1 = c.i0 + 1 >= 0 && c.i0 + 1 < H;
    const bool c0 = c.i1 >= 0 && c.i1 < W, c1 = c.i1 + 1 >= 0 && c.i1 + 1 < W;
    const float wa_ = __fsub_rn(1.0f, c.wa), wb_ = __fsub_rn(1.0f, c.wb);
    return make_float4((r0 && c0) ? c.wa * c.wb : 0.f, (r1 && c0) ? wa_ * c.wb : 0.f, (r0 && c1) ? c.wa * wb_ : 0.f,
                       (r1 && c1) ? wa_ * wb_ : 0.f);
}
// The pixels a combine kernel LOADS for a cell: the four corners clamped to [0,H-1] x [0,W-1]. A corner with weight 0 is still
// loaded (its product is multiplied by 0), so a point projecting outside the map reads a border pixel. Both combine kernels
// and the pixel-tile mark take their corner positions from here.
struct CornerPos {
    int y0, y1, x0, x1;
};
__device__ __forceinline__ CornerPos corner_pos(const CellRef &c, int H, int W) {
    CornerPos p;
    p.y0 = min(max(c.i0, 0), H - 1), p.y1 = min(max(c.i0 + 1, 0), H - 1);
    p.x0 = min(max(c.i1, 0), W - 1), p.x1 = min(max(c.i1 + 1, 0), W - 1);
    return p;
}

// NCHW (B,C,H,W) -> NHWC (B,H,W,C)
// rowmax (optional): [B][HW] max |x| over the C channels of every pixel (float; zeroed and filled here)
// chmax (optional): [B][chmax_stride] ints (float bits, zeroed by the caller): max |x| of every channel over the frame's pixels
int launch_nchw_to_nhwc(const float *in, float *out, int B, int C, int HW, float *rowmax, int *chmax, int chmax_stride, cudaStream_t st);

// NCHW (B,C,HW) fp32 -> pre-packed fp16 hi/lo A operand of the pixel GEMM (rows R = f*HW + p), rowinv[R] = 1 / row scale.
// apack must hold round_up(B*HW, 256) * C * 4 bytes; rows beyond B*HW are never read back (their outputs are not stored).
// tile_bits (optional): the level's active row-tile bitmap (PixelTiles); rows of inactive tiles are neither packed nor scaled.
int launch_pack_maps_f16(const float *in, void *apack, float *rowinv, int B, int C, int HW, const unsigned *tile_bits, cudaStream_t st);

// ---- active pixel tiles of the pixel-first fcn1 ---------------------------------------------------------------------------
// The per-pixel GEMM computes Z_l for 256-row tiles (rows R = f*HW_l + p) of every level, but the combine reads only the corner
// pixels of the kept rows, and LiDAR points never project into the upper image. The mark kernel sets the bit of every row tile
// that some point's clamped corners (corner_pos) fall in; the list kernel compacts the bitmap into entries (level << 24 | tile):
// the active ones in ascending (level, tile) order, then the inactive tiles that may hold products of an earlier call, then the
// inactive tiles already known to be zero (each group ascending). The pixel GEMM multiplies the active tiles and writes zeros into
// the second group, so after every call an inactive tile of Z is zero. The zero state persists in the workspace (zbits, and the
// element size of Z it refers to in meta[5]); a workspace whose `tiles` region is zeroed (PointPath does that when it allocates
// one) starts with every tile unknown. Nothing the path computes reads an inactive tile, so the state only decides which zeros
// must be rewritten: the sky band no point samples is zeroed once per workspace, not once per call.
constexpr int kPixTileRows = 256;
struct PixelTiles {
    int ntiles[MVX_NUM_LEVELS];   // row tiles of level l: ceil(B * HW_l / 256)
    int tile0[MVX_NUM_LEVELS + 1];// first list index of level l in the (level, tile) order of all tiles; tile0[3] = all tiles
    int word0[MVX_NUM_LEVELS + 1];// first bitmap word of level l; word0[3] = bitmap words
    unsigned *bits;               // [word0[3]] active tiles of this call
    unsigned *zbits;              // [word0[3]] tiles of Z known to hold zeros (persists across calls)
    int *list;                    // [tile0[3]] entries: active, then inactive to zero, then inactive and already zero
    int *meta;                    // [8]: first active entry of each level (meta[0..2]), number of active entries (meta[3]), end of
                                  // the entries to zero (meta[4]), element size of Z the zero state refers to (meta[5], 0: none)
};
inline size_t pixel_tiles_bytes(const int *ntiles) {
    size_t t = 0, w = 0;
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) t += ntiles[l], w += (ntiles[l] + 31) / 32;
    return (2 * w + t + 8) * 4;
}
void pixel_tiles_init(PixelTiles &pt, int B, const int *map_h, const int *map_w, void *mem);   // fills the extents and pointers
struct TileMarkArgs {
    const float *points;
    int point_stride;
    int off[33];            // frame point offsets (host)
    // the calibration choice of rows_build_kernel (RowsParams)
    const float *calib32;
    const int *point_calib;
    const double *calib64;
    const int *calib_f64;
    double lo[3], size[3];  // the voxel grid: only in-grid points become rows
    int shape[3];
    int h[MVX_NUM_LEVELS], w[MVX_NUM_LEVELS];
    float rs_h[MVX_NUM_LEVELS], rs_w[MVX_NUM_LEVELS];
    float eps;
};
// zero the bitmap, mark (raw points) or mark everything (all = true: the dense-voxel entry), then build the list; z_esize = bytes per
// element of Z in this call (4: fp32, 2: bf16)
int launch_pixel_tiles(const TileMarkArgs &m, const PixelTiles &pt, int B, bool all, int z_esize, cudaStream_t st);

struct RowsParams {
    int B, cap, capA, T;
    const float *points;
    int point_stride;
    int off[33];
    const float *calib32;   // [B][32], or the calibration table that point_calib indexes
    const int *point_calib; // optional [sum P]: calibration set of every point (merged point sets with their own calibrations)
    const double *calib64;  // optional fp64 copy of the calibration table (same indexing as calib32)
    const int *calib_f64;   // optional flag per calibration set: 1 = project in fp64 from calib64, then round to fp32 (the
                            // reference's numpy branch with readCalib's float64 matrices, train.py:36-39); NULL / 0 = fp32
    const int *counts;      // [B][4]
    const int *vox_cnt, *vox_row0, *row_point, *row_vox;
    float *vox8;            // [B][capA][8]  x,y,z,dx,dy,dz,r,0   (pad row K_f = zeros)
    float *proj;            // [B][capA][2]  (row, col) image coordinates
    float *rowA_w;          // [B][capA]     BN multiplicity of each compact row
};
int launch_rows_build(const RowsParams &p, cudaStream_t st);

// compact gather: A1[f][r][0:3C] for r <= K_f (row K_f is the all-zero pad row)
// rowmax (optional): [B][capA] max |A1[r][:]| of every row
int launch_gather_rows(const MapSet &m, int B, int capA, const int *counts, const float *vox8, const float *proj,
                       float eps, float *A1, float *rowmax, cudaStream_t st);

// Pixel-first form of gather + fcn1. The 4-corner sample is linear in the map values, so
//   relu(A1[r] W^T + b) = relu(b + sum_l sum_corner wgt(r,l,corner) * Z_l[pixel(r,l,corner)]),   Z_l = F_l W_l^T
// with Z_l computed ONCE per pixel (B*sum(HW_l) = 45 864 pixel rows per frame instead of K = 102 000 point rows:
// 6.7x fewer FLOPs, and the (K,768) gathered matrix A1 is never materialised).
struct CombineArgs {
    const float *Z[MVX_NUM_LEVELS];         // [B][HW_l][Cout] per-pixel products of level l
    size_t frame_stride[MVX_NUM_LEVELS];    // HW_l * Cout floats
    int h[MVX_NUM_LEVELS], w[MVX_NUM_LEVELS];
    float rs_h[MVX_NUM_LEVELS], rs_w[MVX_NUM_LEVELS];
    int capA;
    const int *counts;      // [B][4]
    const float *vox8, *proj, *row_w;
    float eps;
    const float *bias;      // (768)
    float *Y1;              // [B][capA][768] raw relu output
    double *out_stats;      // [B][768][2]
    // rows sorted by their level-0 cell (4x4 cell blocks, Morton order inside a block) so that consecutive rows share
    // their corners at all three levels and a warp re-loads a corner only when the cell changes
    int *bin_count;         // [B][nbins + 1] scratch (zeroed by the launcher); bin nbins = rows without corners
    int *bin_start;         // [B][nbins + 2] scratch
    int *perm;              // [B][capA] sorted position -> compact row
    int nbins;
    // bf16 mode (mvx_set_gemm_mode(6)): Z and / or Y1 hold bf16 elements (same indexing in elements, half the bytes)
    int z_bf16, y1_bf16;
};
// scratch sizes (ints per frame) for the level-0 extents of the call
inline int combine_bins(int h0, int w0) { return ((h0 + 3) / 4) * ((w0 + 3) / 4) * 16; }
int launch_combine_sort(const CombineArgs &a, int B, cudaStream_t st);   // counting sort of the rows (needs vox8 / proj only)
int launch_combine_rows(const CombineArgs &a, int B, cudaStream_t st);   // the combine itself (needs Z and the sort)

// dense-voxel entry (dense_entry.cu): compact rows from the reference's (N,T,9) voxel tensor + (N,4) index list
int dense_rows_run(const mvx_pointpath_args_t *a, int capA, long long G, int *vox_coord, int *vox_cnt, int *vox_row0, int *row_point,
                   int *row_vox, int *cell2vid, float *vox8, float *proj, float *rowA_w, cudaStream_t st);

}  // namespace mvx
