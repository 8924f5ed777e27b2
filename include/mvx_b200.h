/*
 * mvx_b200 — C-ABI of the B200-native (sm_100a) point-side hot path of MVXNet.
 *
 * Drop-in boundary (SURVEY.md §8b): every entry point takes plain device/host pointers, extents and a
 * cudaStream_t (passed as void*), never throws, never allocates its outputs (caller-owned buffers; the
 * *_bytes / *_layout queries size them) and returns 0 or a negative MVX_E* code. There is NO CPU
 * fallback: without a CUDA device every compute entry point returns MVX_ECUDA.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference tree).
 */
#ifndef MVX_B200_H_
#define MVX_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVX_OK 0
#define MVX_EINVAL (-1)   /* bad argument (null pointer, bad extent, unsupported channel count) */
#define MVX_ECUDA (-2)    /* CUDA runtime error; mvx_last_error() has the text */
#define MVX_ESPACE (-3)   /* workspace or capacity too small */
#define MVX_ERANGE (-4)   /* a point fell outside the voxel grid / key range (device-detected) */

#define MVX_NUM_LAYERS 8  /* fcn1 conv1 fcn2 conv2 fcn3 | vfe1 vfe2 | fcn   (SURVEY.md §8a row 12) */
#define MVX_NUM_LEVELS 3  /* FPN levels '0','1','2' (modules/imhead/Pipe.py:20) */

/* config.yml:3-13,21 + modules/config/Config.py:7 (voxelsize is the python double (hi-lo)/shape) */
typedef struct {
    double range_lo[3];   /* velorange[0:3] */
    double voxel_size[3]; /* cfg.voxelsize */
    int32_t shape[3];     /* cfg.voxelshape = (nx, ny, nz); dense grid is (C, nz, nx, ny) */
    int32_t T;            /* cfg.samplenum */
} mvx_grid_t;

const char *mvx_last_error(void);
int mvx_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t mvx_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Stage 1 — voxelization.  Replaces cpp/voxelutil.cpp:325-360 (`_group`) and the grouping loop of
 * modules/data/Preprocessing.py:75-116 (`group`).  Deterministic: voxel order = first occurrence in
 * input order, kept points = first T occurrences (SURVEY.md trap 2).
 *
 * Batched over B frames whose points are concatenated; pt_off_host[B+1] are HOST offsets (in points).
 * `cap` = per-frame capacity (>= max points per frame, multiple of 128).
 * Either `cell_idx` (device int32 (P,3), the caller-computed idx of `_group`) is given, or it is NULL and
 * the cell index is computed from the grid in fp64: trunc(((double)x - lo) / size) (trap 1); then points
 * outside the grid are counted in counts[f][2] and skipped.
 * Outputs (device, per frame f at stride cap): see mvx_voxel_out_t.
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t *counts;     /* [B][4]   : N_f voxels, K_f kept rows, #invalid points, max points in one voxel */
    int32_t *vox_coord;  /* [B][cap][4] : ix, iy, iz, linear cell (iz*nx+ix)*ny+iy (or -1 without grid) */
    int32_t *vox_cnt;    /* [B][cap]    : min(#points, T) */
    int32_t *vox_row0;   /* [B][cap+1]  : first compact row of voxel v (exclusive scan of vox_cnt) */
    int32_t *row_point;  /* [B][cap]    : frame-local point index of compact row r (voxel-major, slot order) */
    int32_t *row_vox;    /* [B][cap]    : voxel of compact row r */
    int32_t *cell2vid;   /* [B][G] or NULL : dense cell -> voxel id map (-1 empty), needs a grid */
} mvx_voxel_out_t;

int mvx_voxelize_workspace_bytes(int32_t B, int32_t cap, size_t *bytes);
int mvx_voxelize(const mvx_grid_t *grid, int32_t B, int32_t cap, const float *points, int32_t point_stride,
                 const int32_t *pt_off_host, const int32_t *cell_idx, int32_t T, const mvx_voxel_out_t *out,
                 void *workspace, size_t workspace_bytes, void *stream);

/* `_group` result layout for ONE frame (voxelutil.cpp:344-359): voxel (V,T,7) fp32 zero-filled, cols 0-2 xyz,
 * col 6 = pcd[:,3]; x,y,z,cnt int64[V].  V comes from counts[0] (read it back first). */
int mvx_group_emit7(const float *points, int32_t point_stride, int32_t V, int32_t T, const int32_t *vox_coord,
                    const int32_t *vox_cnt, const int32_t *vox_row0, const int32_t *row_point, float *voxel,
                    int64_t *x, int64_t *y, int64_t *z, int64_t *cnt, void *stream);
/* numba `group` result layout (Preprocessing.py:103-115): voxel (V,T,9) [x,y,z,dx,dy,dz,r,row,col], centroid in
 * fp64 over the kept points; written as fp64 (out_f64) and/or fp32 (= torch.Tensor(voxel), train.py:125).
 * points are (P,6) rows [x,y,z,r,row,col] (train.py:32-35). uidx (V,3) fp64 optional. */
int mvx_group_emit9(const float *points, int32_t point_stride, int32_t V, int32_t T, const int32_t *vox_coord,
                    const int32_t *vox_cnt, const int32_t *vox_row0, const int32_t *row_point, double *out_f64,
                    float *out_f32, double *uidx_f64, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Before the path (SURVEY.md §8f rank 1) — `crop` (modules/data/Preprocessing.py:12-17) and `cropToSight`
 * (Preprocessing.py:26-55; callers modules/data/Load.py:59,73, cropdata.py:32-65) with an order-preserving
 * compaction, batched over B frames (pt_off_host[B+1] HOST offsets into `points`, which may start at a non-zero
 * offset). range6 = velorange (lo xyz, hi xyz) or NULL (no range filter); calib32 = device [B][32]
 * (R0@Tr | P2) or NULL (no sight filter); imsize as (w, h) like the reference. The kept points of frame f are
 * written, in input order and with all `point_stride` columns, to out_points starting at row pt_off_host[f];
 * out_counts[f] (device) = how many. Decisions are the reference's: fp32 coordinates promoted to fp64 against the
 * fp64 range, camera z > 0, 0 <= (u, v) and (double)(u, v) < imsize - 1e-3.
 * ------------------------------------------------------------------------------------------------ */
int mvx_crop_workspace_bytes(int32_t B, int64_t total_points, int64_t max_points, size_t *bytes);
int mvx_crop_points(const float *points, int32_t point_stride, int32_t B, const int32_t *pt_off_host, const double *range6,
                    const float *calib32, double imsize_w, double imsize_h, float *out_points, int32_t *out_counts,
                    void *workspace, size_t workspace_bytes, void *stream);
/* The same with float64 calibrations (calib64 = device [B][32] doubles, (R0@Tr | P2) with the 4x4 product formed in fp64):
 * what the reference's numpy branch evaluates when `calib` holds the float64 matrices `readCalib` returns
 * (modules/data/Load.py:24-41, caller Load.py:73): projection, depth test and image-bound test all in fp64. */
int mvx_crop_points_f64(const float *points, int32_t point_stride, int32_t B, const int32_t *pt_off_host, const double *range6,
                        const double *calib64, double imsize_w, double imsize_h, float *out_points, int32_t *out_counts,
                        void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Stage 2a — projection.  Replaces modules/utils/Calib.py:47-70 (`lidar2Img(pcd, calib, True)`).
 * calib32 (device, 32 floats): M = R0_rect @ Tr_velo_to_cam (row-major 4x4, host-multiplied like the
 * reference does) followed by P2.  out_uv (P,2) = (u,v) = (width, height) coordinates.
 * ------------------------------------------------------------------------------------------------ */
int mvx_lidar2img(const float *points, int32_t point_stride, int64_t P, const float *calib32, float *out_uv,
                  void *stream);
/* numpy branch with float64 calibration matrices (train.py:36-39 projects the pasted ground-truth sets through the float64
 * dicts of modules/augment/LoadGT.py:31): fp32 coordinates promoted, fp64 arithmetic, fp64 (P,2) result. */
int mvx_lidar2img_f64(const float *points, int32_t point_stride, int64_t P, const double *calib64, double *out_uv,
                      void *stream);

/* ------------------------------------------------------------------------------------------------
 * Stage 2b — PointFusion gather.  Replaces modules/imhead/Pipe.py:23-82 (`featureMaping`) for one frame.
 * maps: 3 device pointers to NCHW fp32 maps (C, Hf, Wf) of this frame (NOT padded: the +1 row/col zero pad of
 * Pipe.py:47-48 is a bounds predicate here).  nhwc_ws: scratch of mvx_maps_nhwc_bytes().
 * voxels (R,9) fp32 is updated IN PLACE like the reference (pad rows, x==y==z==0, are zeroed; Pipe.py:53-59).
 * out (R, 3*C) fp32.  Inverted "bilinear" weights and index math exactly as Pipe.py:62-75 (traps 9, 10).
 * ------------------------------------------------------------------------------------------------ */
int mvx_maps_nhwc_bytes(const int32_t *map_h, const int32_t *map_w, int32_t C, size_t *bytes);
int mvx_feature_mapping(float *voxels, int64_t R, const float *const *maps, const int32_t *map_h,
                        const int32_t *map_w, int32_t C, float imsize_h, float imsize_w, float eps, float *out,
                        void *nhwc_ws, size_t nhwc_ws_bytes, void *stream);

/* Backward of mvx_feature_mapping (Pipe.py:62-75, the 4-corner sample) with respect to the three maps of the frame.
 * voxels (R,9) as the forward left them (pad slots zeroed, projection (row, col) in columns 7-8), d_out (R, 3*C) = dLoss/d out;
 * d_maps[l]: (C, map_h[l], map_w[l]) fp32 NCHW, OVERWRITTEN. Pad slots and corners on the zero pad row / column of Pipe.py:47-48
 * contribute nothing. Deterministic: per-pixel sums in a fixed order, no floating-point atomics (two calls give bit-identical
 * results). No gradient flows to voxels / the projection (data in the reference too). ws: the _workspace_bytes() of scratch. */
int mvx_feature_mapping_backward_workspace_bytes(int64_t R, const int32_t *map_h, const int32_t *map_w, size_t *bytes);
int mvx_feature_mapping_backward(const float *voxels, int64_t R, const float *d_out, const int32_t *map_h, const int32_t *map_w,
                                 int32_t C, float imsize_h, float imsize_w, float eps, float *const *d_maps, void *ws, size_t ws_bytes,
                                 void *stream);

/* ------------------------------------------------------------------------------------------------
 * Stage 3 — one layer primitive.  Replaces modules/layers/Blocks.py:5-18 (FCN) and :31-40 (CRB2d, k=1):
 * y = BatchNorm(relu(x W^T + b)), batch statistics over all R rows, biased variance, no affine.
 * x (R,Cin) fp32 row-major (Cin multiple of 16, <= 768), wt (Cin,Cout) = W^T, bias (Cout), y (R,Cout).
 * stats_ws: mvx_layer_workspace_bytes(Cin, Cout) of scratch.  Layers with Cout % 128 == 0 run on the tensor cores
 * (tcgen05, 3xTF32 split: fp32-accurate) unless mvx_set_gemm_mode(0) selects the exact-fp32 SIMT kernel everywhere.
 * mvx_vfe_forward additionally appends the per-voxel max over each
 * group of T rows: y (R, 2*Cout) = [pointwise | max] (modules/voxelnet/Pipe.py:12-18).
 * mvx_fcn_max_forward returns only the per-voxel max (R/T, Cout) (VoxelNet.py:28-32).
 * ------------------------------------------------------------------------------------------------ */
int mvx_set_gemm_mode(int32_t mode); /* 0 = SIMT fp32 everywhere, 1 = tensor cores (default): fp16 hi/lo operands ("3xFP16") for the layers of the fused path whose inputs are BatchNorm-ed or row-scaled, 3xTF32 for the dense layer entry points below; conv1 / fcn2 / the last FCN of the fused path run in the persistent TMA-fed kernel with the A operand in tensor memory (csrc/tc3_layer.cu), 5 = like 1 with those layers in the one-tile kernel of csrc/tc_layer.cu, and the dense layer entry points also use fp16 operands (caller promises inputs of O(1) magnitude), 6 = bf16 mode: one bf16 product per K-step instead of the three-product split for the 3xFP16 layers (reduced precision; tolerance in tests/test_gpu_parity.py::test_bf16_mode_tolerance), 9 = like 1 but conv1 / fcn2 / the last FCN in the one-tile kernel of csrc/tc_layer.cu (kept for A/B timing), 10 = like 1 with the VFE inputs materialised by prep kernels as in training (inspection of X6 / X7, A/B timing), 12 = like 1 with the one-tile two-CTAs-per-SM kernel for the per-pixel GEMM of fcn1 instead of the persistent one (A/B timing). Every other value, among them the removed modes 2, 3, 4, 7 and 8, is rejected with MVX_EINVAL. */
int mvx_layer_workspace_bytes(int32_t Cin, int32_t Cout, size_t *bytes);
int mvx_fcn_forward(const float *x, int64_t R, int32_t Cin, const float *wt, const float *bias, int32_t Cout,
                    double eps, float *y, void *stats_ws, void *stream);
int mvx_vfe_forward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                    int32_t Cout, double eps, float *y, void *stats_ws, void *vmax_ws, void *stream);
int mvx_fcn_max_forward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                        int32_t Cout, double eps, float *y_max, void *stats_ws, void *vmax_ws, void *stream);

/* Training through the dense layer entries (the backward of FCN / CRB2d, Blocks.py:5-18, 31-40; VFE, voxelnet/Pipe.py:5-18; the last
 * FCN + max over T, VoxelNet.py:27-32; what autograd computes through the reference modules).
 *   mvx_*_forward_train: the arguments and outputs of the forward entries above, bit-identical, plus y_raw (R, Cout) = the raw
 *     post-ReLU output relu(x W^T + b); stats_ws then holds the layer's fp64 sums for the backward.
 *   mvx_*_backward: x, wt, y_raw, stats_ws, eps of that training forward; dy = dLoss/d output in the forward's output layout:
 *     (R, Cout) for FCN, (R, 2*Cout) = [pointwise | max tiled over T] for VFE, (R/T, Cout) for the last FCN's max. The max half goes
 *     per voxel and column to the first row (slot order) attaining the maximum of y_raw. BatchNorm backward in fp64 over all R
 *     rows. dx (R, Cin) = dLoss/d x (NULL skips that product); dW (Cout, Cin) and db (Cout) receive the parameter gradients
 *     (accumulate != 0: added to their contents; the sums use fp32 atomics). Cin is the padded width of the forward (a multiple of 16,
 *     <= 768): dW and dx have zero-input columns there. Every layer shape of the path is accepted (Cin/Cout 768/768, 768/128,
 *     128/128, 128/16, 16/16, 32/16, 32/64). ws: mvx_*_backward_workspace_bytes() of scratch. */
int mvx_fcn_forward_train(const float *x, int64_t R, int32_t Cin, const float *wt, const float *bias, int32_t Cout,
                          double eps, float *y, float *y_raw, void *stats_ws, void *stream);
int mvx_vfe_forward_train(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                          int32_t Cout, double eps, float *y, float *y_raw, void *stats_ws, void *vmax_ws, void *stream);
int mvx_fcn_max_forward_train(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                              int32_t Cout, double eps, float *y_max, float *y_raw, void *stats_ws, void *vmax_ws, void *stream);
int mvx_fcn_backward_workspace_bytes(int64_t R, int32_t Cin, int32_t Cout, size_t *bytes);
int mvx_vfe_backward_workspace_bytes(int64_t R, int32_t T, int32_t Cin, int32_t Cout, size_t *bytes);
int mvx_fcn_max_backward_workspace_bytes(int64_t R, int32_t T, int32_t Cin, int32_t Cout, size_t *bytes);
int mvx_fcn_backward(const float *x, int64_t R, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw, const void *stats_ws,
                     double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate, void *ws, size_t ws_bytes,
                     void *stream);
int mvx_vfe_backward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw,
                     const void *stats_ws, double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate, void *ws,
                     size_t ws_bytes, void *stream);
int mvx_fcn_max_backward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw,
                         const void *stats_ws, double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate,
                         void *ws, size_t ws_bytes, void *stream);

/* Element types of a dense grid (the `*_typed` scatter entries, mvx_pointpath_args_t.grid_dtype). A 16-bit grid holds every fp32
 * feature rounded once to nearest-even (what `grid_fp32.to(torch.float16 / torch.bfloat16)` gives); a 16-bit grid gradient is
 * widened to fp32 exactly. Any other value is rejected with MVX_EINVAL (mvx_last_error() names the accepted values). */
#define MVX_DTYPE_F32 0
#define MVX_DTYPE_F16 1
#define MVX_DTYPE_BF16 2

/* ------------------------------------------------------------------------------------------------
 * Stage 4 — scatter into the dense middle-layer grid.  Replaces modules/voxelnet/VoxelNet.py:16-22
 * (`reindex`): out (1,C,nz,nx,ny) fully written (zeros + features) in ONE streaming pass, fp32 or, with the typed entry,
 * out_dtype (MVX_DTYPE_*; `out` is then read as that element type).
 * idx (N,4) int64 [batch, ix, iy, iz] (train.py:119,126).  map_ws: (G + G/32 + 1) int32 of scratch, G = nz*nx*ny.
 * ------------------------------------------------------------------------------------------------ */
int mvx_scatter_dense_typed(const float *feat, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny,
                            int32_t nz, void *out, int32_t out_dtype, int32_t *map_ws, void *stream);
int mvx_scatter_dense(const float *feat, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny,
                      int32_t nz, float *out, int32_t *map_ws, void *stream);   /* = the typed entry with MVX_DTYPE_F32 */
/* Backward of `reindex` for the values (torch's index_put_ backward): d_feat (N,C)[n][c] = d_grid (1,C,nz,nx,ny)[0][c][iz][ix][iy], a
 * gather, so voxels sharing a cell each receive that cell's gradient; rows whose cell lies outside the grid receive 0.
 * d_feat is fp32; d_grid has element type `dtype` (MVX_DTYPE_*) in the typed entry, fp32 in the other. */
int mvx_scatter_dense_backward_typed(const void *d_grid, int32_t dtype, const int64_t *idx, int64_t N, int32_t C, int32_t nx,
                                     int32_t ny, int32_t nz, float *d_feat, void *stream);
int mvx_scatter_dense_backward(const float *d_grid, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny, int32_t nz,
                               float *d_feat, void *stream);

/* ------------------------------------------------------------------------------------------------
 * The fused batched path: stages 1-4 for B frames in one stream-ordered sequence with no host sync
 * (MVXNet.forward up to the CML input: MVXNet.py:21-27, modules/imhead/Head.py:14-22,
 * modules/voxelnet/VoxelNet.py:24-34, with train.py:26-49's CPU half moved onto the GPU).
 * BatchNorm statistics stay per frame (the reference is batch-1; SURVEY.md §7 hard part 6).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
    mvx_grid_t grid;
    int32_t B;                 /* frames in this call */
    int32_t cap;               /* per-frame capacity, multiple of 128, >= max points per frame */
    const float *points;       /* device, concatenated (sum P, point_stride) fp32 rows [x,y,z,r,...] */
    int32_t point_stride;      /* floats per point row (>= 4) */
    const int32_t *pt_off_host;/* HOST [B+1] point offsets */
    const float *calib32;      /* device [B][32]: (R0@Tr, P2) per frame */
    const float *maps[MVX_NUM_LEVELS]; /* device NCHW (B, C, Hf, Wf) fp32 */
    int32_t map_h[MVX_NUM_LEVELS], map_w[MVX_NUM_LEVELS];
    int32_t map_c;             /* 256 */
    float imsize_h, imsize_w;  /* cfg.imsize (370, 1224) */
    float gather_eps;          /* cfg.eps as fp32 (Pipe.py:62) */
    double bn_eps;             /* cfg.eps (Blocks.py:10) */
    const float *wt[MVX_NUM_LAYERS];   /* device W^T (Cin_pad, Cout) fp32; Cin_pad: 768,768,128,128,16,32,32,128 */
    const float *bias[MVX_NUM_LAYERS]; /* device (Cout) */
    float *grid_out;           /* device (B, 128, nz, nx, ny), fully overwritten; may be NULL (skip stage 4). Elements of type
                                  grid_dtype: with MVX_DTYPE_F16 / MVX_DTYPE_BF16 the pointer is reinterpreted as a 16-bit grid */
    int32_t *counts;           /* device [B][4]: N_f, K_f, #invalid points, max points per voxel */
    void *workspace;
    size_t workspace_bytes;
    void *stream;
    /* Optional (SURVEY.md §8f rank 4, GT-paste: train.py:29-42 projects every pasted object through ITS OWN calibration
     * before the point sets are merged and voxelized together): device [sum P] calibration index of every point; calib32
     * then holds max(index)+1 sets instead of one per frame. NULL: every point of frame f uses calib32[f]. */
    const int32_t *point_calib;
    /* Optional float64 calibrations: calib64 = device doubles, indexed like calib32; calib_f64 = device int32 flag per
     * calibration set (1: project this set in fp64 from calib64 and round the pixel coordinates to fp32 once - the reference's
     * numpy lidar2Img with readCalib's float64 matrices followed by `torch.Tensor(voxel)`, train.py:36-39,125; 0: fp32
     * arithmetic from calib32 - the torch branch, train.py:31-33). Both NULL: every set is fp32. */
    const double *calib64;
    const int32_t *calib_f64;
    /* Optional dense-voxel input - the arguments of the reference's own `MVXNet.forward(voxels, imgs, idx, calibs, imsize)`
     * (MVXNet.py:21-27; produced by pre.group + train.py:118-128): voxels_dense = device (sum N_f, T, 9) fp32
     * [x,y,z,dx,dy,dz,r,row,col], voxel_idx = device (sum N_f, 4) int64 [batch, ix, iy, iz], vox_off_host = HOST [B+1] voxel
     * offsets. When voxels_dense is set, stage 1 and the projection are skipped (points / pt_off_host / calib32 are not
     * read): slots with x == y == z == 0 are pad slots exactly as featureMaping decides (Pipe.py:53-54) and, like there, are
     * zeroed IN PLACE in the caller's tensor (Pipe.py:58-59); every other slot becomes one compact row.
     * cap must be >= max_f max(N_f, K_f) with K_f = real slots of frame f (mvx_dense_voxel_counts reports them). */
    float *voxels_dense;
    const int64_t *voxel_idx;
    const int32_t *vox_off_host;
    /* Element type of grid_out (forward, forward_train) and of d_grid (mvx_pointpath_backward): MVX_DTYPE_F32 (0, what a
     * zero-initialised struct holds), MVX_DTYPE_F16 or MVX_DTYPE_BF16; any other value is rejected with MVX_EINVAL before any
     * CUDA call. Nothing else of the path depends on it. */
    int32_t grid_dtype;
} mvx_pointpath_args_t;

/* counts[f] = (N_f, K_f = slots of frame f with (x,y,z) != 0, 0, max real slots per voxel) for a dense voxel tensor: what a
 * caller needs to size `cap` before mvx_pointpath_forward with voxels_dense. counts: device [B][4]. */
int mvx_dense_voxel_counts(const float *voxels_dense, const int32_t *vox_off_host, int32_t B, int32_t T, int32_t *counts,
                           void *stream);

/* byte offsets of named workspace regions, for tests/diagnostics (names in mvx_pointpath_layout_name) */
#define MVX_WS_REGIONS 64
int mvx_pointpath_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes);
int mvx_pointpath_layout(const mvx_pointpath_args_t *args, int64_t *offsets /* [MVX_WS_REGIONS] */);
const char *mvx_pointpath_layout_name(int32_t region);
/* The workspace carries state from one call to the next in its "tiles" region: which row tiles of the per-pixel products Z are
 * known to hold zeros. Zero that region when the workspace is new (or was used for anything else); then every row tile of Z that
 * no point samples is zero after each call. No output depends on it: only inactive tiles of Z, which nothing reads. */
int mvx_pointpath_forward(const mvx_pointpath_args_t *args);
/* How gather + fcn1 (Pipe.py:62-82 + Pipe.py:94) are evaluated inside the fused path. The 4-corner sample is linear in
 * the map values, so fcn1 commutes with it:
 *   1 (default) pixel-first: Z_l = F_l W1_l^T once per map pixel (tensor cores), then per point row
 *               relu(b + sum of 12 weighted Z rows); the (K,768) gathered matrix is never materialised (6.7x fewer FLOPs);
 *   0           row-first: gather the (K,768) matrix A1, then fcn1 over the point rows (the reference's order; the
 *               layout the training-mode backward uses).  Timing segments "gather"/"fcn1" then mean
 *               (pixel GEMMs, combine) in mode 1 and (gather, row GEMM) in mode 0.
 *   2           pixel-first like 1 but without running the map branch (channels-last copy + pixel GEMMs) on a side stream
 *               concurrently with the point branch (voxelization, row build, row sort) - for per-stage profiling.
 * Any other value is rejected with MVX_EINVAL (mvx_last_error() names the accepted values). */
int mvx_set_fusion_mode(int32_t mode);
/* Pixel-first inference only. 0: the run-structured combine kernel (default);
 * 2: the first version of the combine kernel (row-by-row walk; kept for A/B measurements). Any other value is rejected with
 * MVX_EINVAL (1, conv1 with fcn1's BatchNorm folded into per-frame weights, was removed). */
int mvx_set_fold_mode(int32_t mode);

/* ------------------------------------------------------------------------------------------------
 * Training mode (BASELINE.json configs[3]): forward that keeps every activation, then the backward of the 8 hot-path
 * layers.  What loss.backward() does through modules/imhead/Pipe.py:84-104, modules/voxelnet/Pipe.py:5-29 and
 * modules/voxelnet/VoxelNet.py:16-32 in train.py:140-166, for the parameters of SURVEY.md §8b.
 *   mvx_pointpath_forward_train: same arguments and outputs as mvx_pointpath_forward; always row-first (keeps the
 *     gathered matrix A1) and also keeps the raw output of the last FCN; args->workspace must hold `forward_bytes`.
 *   mvx_pointpath_backward: call after forward_train with the SAME args (same workspace, weights, counts).
 *     Upstream gradient: exactly one of d_vfeat (B, cap, 128: dLoss/d voxel features, reference voxel order, rows
 *     >= N_f ignored) or d_grid (B,128,nz,nx,ny: dLoss/d dense grid; reindex's backward is an index select), whose
 *     elements are of type args->grid_dtype (the d_grid pointer is reinterpreted as a 16-bit grid for F16 / BF16).
 *     grad_flat: mvx_grad_floats() = 726 880 fp32, per layer [weight (Cout,Cin) | bias (Cout)] in checkpoint order
 *     (fcn1 conv1 fcn2 conv2 fcn3 vfe1 vfe2 fcn) - the one flat bucket the NCCL all-reduce sums; gradients of all B
 *     frames are summed into it (accumulate != 0: added to its current contents).
 * ------------------------------------------------------------------------------------------------ */
int mvx_pointpath_train_workspace_bytes(const mvx_pointpath_args_t *args, size_t *forward_bytes, size_t *backward_bytes);
int mvx_pointpath_forward_train(const mvx_pointpath_args_t *args);
int64_t mvx_grad_floats(void);
int mvx_pointpath_backward(const mvx_pointpath_args_t *args, const float *d_vfeat, const float *d_grid, float *grad_flat,
                           int32_t accumulate, void *backward_ws, size_t backward_ws_bytes);

/* Gradient into the FPN maps (the adjoint of featureMaping's 4-corner gather, modules/imhead/Pipe.py:62-75), for callers
 * that train the image backbone. Call after mvx_pointpath_backward with the SAME args and backward workspace (it reads
 * fcn1's dpre that this left there, and the projections of the training forward). d_maps[l]: (B, 256, map_h[l], map_w[l])
 * fp32 contiguous, OVERWRITTEN with dLoss/d map l; corners on the zero pad row / column of Pipe.py:47-48, pad slots and
 * origin points contribute nothing. Deterministic: no floating-point atomics, two calls give bit-identical results.
 * ws: mvx_pointpath_backward_maps_workspace_bytes() of scratch. */
int mvx_pointpath_backward_maps_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes);
int mvx_pointpath_backward_maps(const mvx_pointpath_args_t *args, const void *backward_ws, size_t backward_ws_bytes,
                                float *const d_maps[MVX_NUM_LEVELS], void *ws, size_t ws_bytes);

/* ------------------------------------------------------------------------------------------------
 * After the path (SURVEY.md §8f rank 2) — sparse hand-off to the first middle-layer convolution.
 * Replaces `CML.conv1` = CRB3d(128, 64, 3, (2,1,1), (1,1,1)) (modules/voxelnet/Pipe.py:31-43; Blocks.py CRB3d:
 * relu(Conv3d) then batch-statistic BatchNorm3d) applied to the dense grid of VoxelNet.reindex, WITHOUT the dense grid:
 * call after mvx_pointpath_forward with the SAME args (the voxel features and the cell -> voxel map are read from
 * args->workspace; args->grid_out may be NULL in that forward). conv_w (64,128,3,3,3), conv_b (64) device fp32 in
 * torch's Conv3d layout; out (B, 64, (nz+1)/2, nx, ny) fp32 fully written; per-frame statistics like the batch-1
 * reference. ws: mvx_cml_conv1_workspace_bytes() of scratch.
 * ------------------------------------------------------------------------------------------------ */
int mvx_cml_conv1_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes);
int mvx_cml_conv1_sparse(const mvx_pointpath_args_t *args, const float *conv_w, const float *conv_b, double eps, float *out,
                         void *ws, size_t ws_bytes);

/* Training through the hand-off: the backward of mvx_cml_conv1_sparse, i.e. of CRB3d (voxelnet/Pipe.py:31-43, Blocks.py
 * CRB3d: relu, Conv3d(128, 64, 3, (2,1,1), (1,1,1)), BatchNorm3d with batch statistics) with respect to conv_w, conv_b and
 * the voxel features the layer read. Call after mvx_cml_conv1_sparse with the SAME args, conv_w, conv_b, eps and the same
 * untouched ws (read only here); the path workspace of that forward must still hold its voxel features.
 * d_out (B, 64, (nz+1)/2, nx, ny) fp32 = dLoss/d out. d_w (64,128,3,3,3) and d_b (64) receive the gradients summed over the
 * frames (accumulate != 0: added to their contents). d_vfeat (B, cap, 128) receives dLoss/d voxel features for rows
 * 0 .. N_f-1 of every frame (other rows untouched), the input of mvx_pointpath_backward; NULL skips that product.
 * bws: mvx_cml_conv1_backward_workspace_bytes() of scratch. */
int mvx_cml_conv1_backward_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes);
int mvx_cml_conv1_sparse_backward(const mvx_pointpath_args_t *args, const float *conv_w, const float *conv_b, double eps,
                                  const float *d_out, float *d_vfeat, float *d_w, float *d_b, int32_t accumulate,
                                  const void *ws, size_t ws_bytes, void *bws, size_t bws_bytes);

/* ------------------------------------------------------------------------------------------------
 * Label side of the same native extension (SURVEY.md §8f rank 3).
 *
 * mvx_bbox_pairwise replaces `bboxOverlap` (mode 0: IoU, cpp/voxelutil.cpp:96-116; caller modules/augment/Augment.py:54)
 * and `bboxIntersection` (mode 1: intersection area, voxelutil.cpp:118-139) on top of the polygon clipper
 * voxelutil.cpp:15-93: bboxes1 (n,4,2), bboxes2 (m,4,2) device fp32 corner quads (16-byte aligned) -> out (n,m) fp32.
 * Bit-identical to the reference's scalar fp32 arithmetic; the second quad is read corner by corner (the reference
 * indexes it by box number, voxelutil.cpp:108,129 — a slip that mixes stale corners and overruns its 5-element global).
 *
 * mvx_classify_anchors replaces `classifyAnchors` (voxelutil.cpp:141-316, bound as `_classifyAnchors`; python caller
 * modules/Calc.py:88-96): gts (G,4,2) ground-truth BEV quads, anchors (L,W,A,4,2) anchor BEV quads, nls/nws int64[G] start
 * cells. For every ground truth and anchor rotation the anchors reachable from the start cell through IoU >= 0.1
 * (column walk up then down, row walk right then left) are classified: IoU >= pos_thr -> appended to pos (+ gi = ground
 * truth index) AND neg, else IoU >= neg_thr -> appended to neg ("not negative"). pos/neg are (cap,3) int64 rows
 * (l, w, z), gi (cap) int64, all in the reference's append order. counts (device int64[4]) = {npos, nneg, ground
 * truths whose start cell is outside the anchor grid (undefined behaviour in the reference; skipped here), 0}; entries
 * beyond cap are counted but not stored (re-run with a larger cap). No host synchronisation.
 * ------------------------------------------------------------------------------------------------ */
int mvx_bbox_pairwise(const float *bboxes1, int64_t n, const float *bboxes2, int64_t m, int32_t mode, float *out, void *stream);
int mvx_classify_anchors_workspace_bytes(int64_t G, int64_t L, int64_t W, int32_t A, size_t *bytes);
int mvx_classify_anchors(const float *gts, int64_t G, const float *anchors, int64_t L, int64_t W, int32_t A, const int64_t *nls,
                         const int64_t *nws, float neg_thr, float pos_thr, int64_t *pos, int64_t *neg, int64_t *gi, int64_t cap,
                         int64_t *counts, void *workspace, size_t workspace_bytes, void *stream);

/* Optional per-kernel timing of mvx_pointpath_forward with CUDA events recorded on the launching stream
 * (bench.py's roofline leg). mvx_timing_enable(n) arms n event sets (one per forward call, n = 0 disables);
 * mvx_timing_read(call, ms) waits for that call's last event and returns MVX_NUM_SEGMENTS durations in ms, in the
 * order of mvx_timing_segment_name(). */
#define MVX_NUM_SEGMENTS 20
int mvx_timing_enable(int32_t max_calls);
int mvx_timing_read(int32_t call, float *ms /* [MVX_NUM_SEGMENTS] */);
const char *mvx_timing_segment_name(int32_t segment);

#ifdef __cplusplus
}
#endif
#endif /* MVX_B200_H_ */
