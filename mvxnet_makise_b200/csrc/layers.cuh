// Internal interface of stage 3 (the Linear -> ReLU -> batch-stat BN layer primitive and the VFE glue).
#pragma once
#include "common.cuh"

namespace mvx {

// One launch = y = relu(norm_in(X) W^T + b) for every frame of the batch, plus the weighted per-channel
// sums (sum w*y, sum w*y^2, fp64) that the consumer turns into (mean, rstd), plus an optional per-voxel max.
struct LayerArgs {
    const float *X;        // [F][rowcap][ldx] raw input rows
    int ldx, Cin;          // Cin multiple of 16 (zero-padded columns/weights)
    const float *Wt;       // (Cin, Cout) = W^T
    const float *bias;     // (Cout)
    int Cout;
    float *Y;              // [F][rowcap][ldy] raw (pre-BN) output, or NULL
    int ldy;
    const double *in_stats;  // [F][Cin][2] sums of the producer layer -> normalise X on load; NULL = X is used as is
    double *out_stats;       // [F][Cout][2]
    int *vmax;               // [F][vcap][Cout] float bits (y >= 0), or NULL
    const float *row_w;      // [F][rowcap] BN multiplicity of each row, or NULL (all 1)
    const int *row_v;        // [F][rowv_cap] voxel of each row (-1: none), or NULL (v = r / T); in rows_mode 1 the
                             // pad row (r == K_f) belongs to no voxel
    int rowv_cap;            // frame stride of row_v
    const int *counts;       // [F][4] device (N_f, K_f, ..), or NULL
    int rows_mode;           // 0: rows_fixed rows; 1: K_f + 1 rows; 2: K_f + N_f rows; 3: N_f rows (one per voxel)
    long long rows_fixed;
    int rowcap, vcap, T;
    double eps;
    int dbg;                 // work-skipping timing switches; only read in -DMVX_DEVTOOLS builds (MVX_DBG() is the constant 0 otherwise)
    int f16_ok;              // 1: the tensor-core kernel may use fp16 operands (3xFP16): inputs are BatchNorm-ed (in_stats, or
                             // stored normalised) or row_max is given; 0 keeps 3xTF32 (arbitrary input range)
    const float *row_max;    // [F][rowcap] max|x| of each input row for the fp16 row scaling, or NULL (scale 1)
    // pre-packed A (rows_mode 0, one frame): the producing kernel already wrote the fp16 hi/lo shared-memory images of every
    // (256-row tile, 32-k chunk) [hi 16 KB | lo 16 KB], tile t and chunk kc at (t * nk + kc) * 32 KB; the layer kernel then has no
    // register producers at all, the A tiles arrive by bulk copy like the weights. a_rowinv[r] = 1 / (power-of-two scale the packer
    // applied to row r).
    const void *a_pack;
    const float *a_rowinv;   // NULL: no per-row scale
    // fused concat (16-bit tensor-core producer only): input columns [Cin - x2_cols, Cin) of row r come from
    // X2[f][v(r)][0:x2_cols] (float bits, e.g. the per-voxel max of the producer layer) instead of X, with
    // v(r) = r >= K_f ? r - K_f : cat_row_vox[f][r]; both parts are normalised with the same in_stats (in_C channels)
    const int *X2;           // [F][vcap][x2_cols] or NULL
    int x2_cols;
    const int *cat_row_vox;  // [F][cat_rowv_cap] voxel of the rows below K_f
    int cat_rowv_cap;
    int in_C;                // channels of in_stats (0: Cin)
    int y_bf16;              // 1 (bf16 mode): Y holds bf16 elements (ldy in elements)
    int x_bf16;              // 1 (bf16 mode, tc3 kernel): X holds bf16 elements (ldx in elements)
    int plain;               // 1: Y = norm_in(X) W^T only (no bias, no ReLU, no statistics, no max) - the per-pixel half of fcn1
    int y_nchw;              // 1 (plain 3xTF32 one-tile kernel only): Y is channel-major [F][Cout][rowcap], e.g. (B, C, H, W)
                             // maps with rows_fixed = rowcap = H * W pixel rows per frame
};
// Work-skipping switches (no epilogue, no producers ...) exist for timing experiments only: a release build compiles them
// out (the expression is the literal 0), so no environment variable can remove work from a timed region.
#ifdef MVX_DEVTOOLS
#define MVX_DBG(a) ((a).dbg)
#else
#define MVX_DBG(a) 0
#endif
int launch_layer(const LayerArgs &a, int F, cudaStream_t st);            // exact-fp32 SIMT kernel

// Fused VFE loaders (inference): the SIMT kernel builds VFE1's / VFE2's input tile on the fly instead of reading the X6 / X7
// matrices that prep_vfe1 / prep_vfe2 materialise (one launch and one round trip through HBM less per VFE).
struct RowFuseArgs {
    const float *vox8;       // VFE1: [F][capA][8] x,y,z,dx,dy,dz,r,0
    const float *Y;          // VFE1: Y5 [F][capA][16] raw fcn3 rows; VFE2: Y6 [F][capA][16] raw VFE1 rows (row K_f = the frame's pad row)
    const double *in_stats;  // [F][16][2] sums of that producer layer
    const int *vmax;         // VFE2: [F][cap][16] per-voxel max of Y6 (float bits)
    const int *vox_cnt, *row_vox;   // VFE2: [F][cap] points kept per voxel, voxel of each kept row
    float *rowB_w;           // VFE2 out: [F][capB] BatchNorm multiplicity of the K_f + N_f rows (1 / T - cnt)
    int *rowB_v;             // VFE2 out: [F][capB] voxel of each row (-1: a pad row of a full voxel)
    int cap, capA;
};
int launch_vfe1_fused(const LayerArgs &a, const RowFuseArgs &z, int F, cudaStream_t st);   // a.X unused: input = [vox7 | norm5(Y5) | 0]
int launch_vfe2_fused(const LayerArgs &a, const RowFuseArgs &z, int F, cudaStream_t st);   // a.X unused: input = [norm6(Y6) | norm6(max6[v])]; writes rowB_w / rowB_v
bool vfe_fused_enabled();
void set_vfe_fused(int on);

// tensor-core (tcgen05, 3xTF32) implementation of the same layer; wpack = tc_wpack_bytes() of scratch
bool tc_layer_eligible(const LayerArgs &a);
size_t tc_wpack_bytes(int Cin, int Cout);
int launch_layer_tc(const LayerArgs &a, int F, float *wpack, cudaStream_t st);
// TMA-fed persistent kernel with the A operand in tensor memory (tc3_layer.cu): BatchNorm-ed 128-column layers of the fused path
bool tc3_layer_eligible(const LayerArgs &a);
int launch_layer_tc3(const LayerArgs &a, int F, float *wpack, cudaStream_t st);
// persistent pre-packed-operand GEMM for the per-pixel half of fcn1 (tc3_layer.cu)
bool pixel_gemm_persistent_eligible(const LayerArgs &a);
int launch_pixel_gemm_persistent(const LayerArgs &a, float *wpack, cudaStream_t st);
void set_pixel_persistent(int on);
bool pixel_persistent_enabled();
void set_tc3(int on);
bool tc_bf16_enabled();
void set_tc_bf16(int on);  // 1: single-pass bf16 operands where LayerArgs::f16_ok (reduced precision, tolerance stated in the tests)
// dispatch by mvx_set_gemm_mode(): 0 = SIMT everywhere, 1 = tensor cores where eligible (default)
int gemm_mode();
int launch_layer_auto(const LayerArgs &a, int F, float *wpack, cudaStream_t st);

// dW (Cout, Cin) += sum over the frames and their N_f voxel rows r of D[f][r]^T X[f][r] (backward.cu): rows of weight 1, X used
// as stored (no BatchNorm on load, |x| = O(1)); D [B][rowcap][Cout], X [B][rowcap][Cin]; dmax [B][Cout] bounds |D| per column
// (float bits) for the power-of-two scales of the tensor-core kernel; xmax [B][Cin] bounds |X| per column the same way, or NULL
// (scale 1)
int launch_dw_voxel_rows(const float *D, int Cout, const float *X, int Cin, const int *counts, int rowcap, const int *dmax, float *dW, int B,
                         cudaStream_t st, const int *xmax = nullptr);
// batch-statistic BatchNorm + ReLU backward of ONE frame of N_f = counts[0] rows of multiplicity row_w (backward.cu, T = 1): G (rowcap,
// C) holds dz on entry and dpre on exit; dbias (C) += column sums of dpre (fp32 atomics); bstats (C, 2) must be zeroed; dmax (C) as in
// launch_dw_voxel_rows (zeroed by the caller) or NULL. C: 768 or a multiple of 4 up to 512 with C / 4 dividing 256.
int launch_bn_back_voxel_rows(float *G, const float *Y, int C, const double *stats, double *bstats, float *dbias, double eps, const int *counts,
                              int rowcap, const float *row_w, int *dmax, cudaStream_t st);

// number of rows BN statistics are taken over for frame f: N_f * T (fused path) or rows_fixed (dense API)
struct NormSrc {
    const double *stats;   // [F][C][2]
    const int *counts;     // [F][4] or NULL
    long long rows_fixed;
    int T;
    double eps;
};

struct VfePrepArgs {
    int B, cap, capA, capB, T;
    const int *counts, *vox_cnt, *row_vox;
    // VFE1 input: X6[r] = [vox7 | norm5(Y5[r]) | 0-pad] (32 cols), rows 0..K_f
    const float *vox8, *Y5;
    float *X6;
    // VFE2 input: X7[r] = [norm6(Y6[r]) | norm6(vmax6[v])] (32), rows 0..K_f-1 real + one pad row per voxel
    const float *Y6;
    const int *vmax6;
    float *X7;
    float *rowB_w;
    int *rowB_v;
    // FCN input: X8[r] = [norm7(Y7[r]) | norm7(vmax7[v])] (128)
    const float *Y7;
    const int *vmax7;
    float *X8;
    // final: vfeat[v] = norm8(vmax8[v]) (128)
    const int *vmax8;
    float *vfeat;
    float *vfeat_t;        // optional channel-major copy (128, cap) per frame
    NormSrc n5, n6, n7, n8;
};
int launch_prep_vfe1(const VfePrepArgs &a, cudaStream_t st);
int launch_prep_vfe2(const VfePrepArgs &a, cudaStream_t st);
int launch_prep_fcn(const VfePrepArgs &a, cudaStream_t st);
int launch_finalize_vfeat(const VfePrepArgs &a, cudaStream_t st);

}  // namespace mvx
