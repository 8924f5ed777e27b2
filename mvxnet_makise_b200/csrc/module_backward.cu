// Backward of the per-module drop-ins (mvxnet_makise_b200/modules.py): the dense (reference-layout) form of the layer backward
// of backward.cu, for callers that swap the reference's FCN / CRB2d (modules/layers/Blocks.py:5-18, 31-40), VFE
// (modules/voxelnet/Pipe.py:5-18) and the last FCN + max over T (modules/voxelnet/VoxelNet.py:27-32) for the dense layer entries,
// and the backward of `reindex` (VoxelNet.py:16-22). The adjoint of `featureMaping`'s gather is in map_backward.cu, next to the
// pixel CSR it shares with the fused path.
//
// Rows are the R = N * T dense rows of the forward, pad rows included, each of multiplicity 1; BatchNorm statistics are over all
// R rows like the forward's. Per layer, with raw output y = relu(pre) and z = (y - mean) * rstd (fp64, from the forward's sums):
//     dz   = dy (FCN), dy[:, :C] + routed max half (VFE), routed dy (last FCN)
//     dpre = rstd * (dz - S1 / R - z * S2 / R) * [y > 0],   S1 = sum dz, S2 = sum dz z        (bn_back_*_kernel, mode 3, T = 1)
//     db = sum dpre,  dW = dpre^T x,  dx = dpre W
// The gradient of the max half goes, per voxel and column, to the FIRST row in slot order that attains the maximum of raw y
// (torch.max's argmax on the dense tensor); for VFE that half of dy is first summed over the T rows it was tiled onto.
#include "layers.cuh"
#include "pointpath.cuh"

namespace mvx {

namespace {

enum LayerKind { kFcn, kVfe, kFcnMax };

// one thread per (voxel, column): G[v T + t][c] = (VFE: dy[v T + t][c]) + (first argmax row ? dM : 0)
//   VFE: dy (R, 2C) = [pointwise | max tiled over T], dM = sum_t dy[v T + t][C + c];   last FCN: dy (R / T, C), dM = dy[v][c]
template <bool kVfeHalf>
__global__ void __launch_bounds__(256) route_max_kernel(const float *__restrict__ y_raw, const float *__restrict__ dy, float *__restrict__ G,
                                                        long long V, int T, int C) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= V * C) return;
    const long long v = e / C;
    const int c = (int)(e - v * C);
    const size_t r0 = (size_t)v * T;
    float m = -INFINITY, dM = kVfeHalf ? 0.f : dy[(size_t)v * C + c];
    int arg = 0;
#pragma unroll 4
    for (int t = 0; t < T; ++t) {
        const float y = y_raw[(r0 + t) * C + c];
        if (y > m) m = y, arg = t;   // strict: the first row attaining the maximum wins
        if (kVfeHalf) dM += dy[(r0 + t) * 2 * C + C + c];
    }
    for (int t = 0; t < T; ++t) {
        const float g = kVfeHalf ? dy[(r0 + t) * 2 * C + c] : 0.f;
        G[(r0 + t) * C + c] = g + (t == arg ? dM : 0.f);
    }
}

// the dense RowSet of backward.cu: one frame of R rows of multiplicity 1 (counts = {R, 0, 0, 0}, row_w = 1)
__global__ void __launch_bounds__(256) dense_rowset_kernel(int *counts, float *row_w, int R) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) counts[0] = R, counts[1] = 0, counts[2] = 0, counts[3] = 0;
    if (r < R) row_w[r] = 1.f;
}

// xmax[c] = max_r |x[r][c]| as float bits (zeroed by the caller): the per-column power-of-two scales of the tensor-core dW, whose
// X operand is raw caller data here (the fused path's layer inputs are BatchNorm-ed and need none)
constexpr int kColRows = 256;
__global__ void __launch_bounds__(256) col_absmax_kernel(const float *__restrict__ x, int R, int Cin, int *__restrict__ xmax) {
    const int r0 = blockIdx.x * kColRows, r1 = min(r0 + kColRows, R);
    for (int c = threadIdx.x; c < Cin; c += blockDim.x) {
        float m = 0.f;
        for (int r = r0; r < r1; ++r) m = fmaxf(m, fabsf(x[(size_t)r * Cin + c]));
        if (m > 0.f) atomicMax(xmax + c, __float_as_int(m));
    }
}

// d_feat[n][c] = d_grid[0][c][iz][ix][iy] (the adjoint of reindex's index_put_ for the values: a gather, also with duplicate cells);
// rows whose cell lies outside the grid (the forward skips them, the reference would raise) get 0
__global__ void __launch_bounds__(256) scatter_back_kernel(const float *__restrict__ d_grid, const long long *__restrict__ idx, long long N,
                                                           int C, int nx, int ny, int nz, float *__restrict__ d_feat) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N * C) return;
    const long long n = e / C;
    const int c = (int)(e - n * C);
    const long long ix = idx[n * 4 + 1], iy = idx[n * 4 + 2], iz = idx[n * 4 + 3];
    float g = 0.f;
    if (ix >= 0 && ix < nx && iy >= 0 && iy < ny && iz >= 0 && iz < nz)
        g = d_grid[(size_t)c * nx * ny * nz + ((size_t)iz * nx + ix) * ny + iy];   // grid is (nz, nx, ny) (VoxelNet.py:19-21)
    d_feat[e] = g;
}

struct MwLayout {
    size_t counts, bstats, dmax, xmax, ones, g, w, wpack, total;
};

MwLayout mw_layout(long long R, int Cin, int Cout) {
    MwLayout M;
    size_t o = 0;
    auto take = [&](size_t &slot, size_t bytes) {
        slot = o;
        o += (bytes + 255) / 256 * 256;
    };
    take(M.counts, 4 * sizeof(int));
    take(M.bstats, (size_t)Cout * 2 * sizeof(double));
    take(M.dmax, (size_t)Cout * sizeof(int));
    take(M.xmax, (size_t)Cin * sizeof(int));
    take(M.ones, (size_t)R * sizeof(float));
    take(M.g, (size_t)R * Cout * sizeof(float));
    take(M.w, (size_t)Cin * Cout * sizeof(float));
    take(M.wpack, tc_wpack_bytes(Cout, Cin));
    M.total = o;
    return M;
}

// the layer shapes dW (backward.cu launch_dw_auto) and the BatchNorm backward serve: every layer of the path
bool dense_shape_ok(int Cin, int Cout) {
    if (Cout % 128 == 0 && Cin % 128 == 0) return Cout == 768 || Cout <= 512;
    return (Cout == 64 && Cin == 32) || (Cout == 16 && (Cin % 128 == 0 || Cin == 32 || Cin == 16));
}

int check_layer_args(long long R, int T, int Cin, int Cout) {
    MVX_REQUIRE(R > 0 && R <= 0x7FFFFFFF, MVX_EINVAL, "layer backward: R must be in [1, 2^31)");
    MVX_REQUIRE(T > 0 && R % T == 0, MVX_EINVAL, "layer backward: R must be a multiple of T");
    MVX_REQUIRE(Cin > 0 && Cin % 16 == 0 && Cin <= 768, MVX_EINVAL, "layer backward: Cin must be a multiple of 16, <= 768");
    MVX_REQUIRE(Cout > 0 && dense_shape_ok(Cin, Cout), MVX_EINVAL, "layer backward: unsupported layer shape");
    return MVX_OK;
}

int layer_backward(LayerKind kind, const float *x, long long R, int T, int Cin, const float *wt, int Cout, const float *y_raw, const void *stats_ws,
                   double eps, const float *dy, float *dx, float *dW, float *db, int accumulate, void *ws_v, size_t ws_bytes, cudaStream_t st) {
    int rc = check_layer_args(R, T, Cin, Cout);
    if (rc) return rc;
    MVX_REQUIRE(x && wt && y_raw && stats_ws && dy && dW && db && ws_v, MVX_EINVAL, "layer backward: null pointer");
    const MwLayout M = mw_layout(R, Cin, Cout);
    MVX_REQUIRE(ws_bytes >= M.total, MVX_ESPACE, "layer backward workspace too small");
    char *ws = static_cast<char *>(ws_v);
    int *counts = reinterpret_cast<int *>(ws + M.counts), *dmax = reinterpret_cast<int *>(ws + M.dmax);
    int *xmax = reinterpret_cast<int *>(ws + M.xmax);
    double *bstats = reinterpret_cast<double *>(ws + M.bstats);
    float *ones = reinterpret_cast<float *>(ws + M.ones), *G = reinterpret_cast<float *>(ws + M.g);
    const int Ri = (int)R;
    if (!accumulate) {
        MVX_CUDA_CHECK(cudaMemsetAsync(dW, 0, (size_t)Cout * Cin * sizeof(float), st));
        MVX_CUDA_CHECK(cudaMemsetAsync(db, 0, (size_t)Cout * sizeof(float), st));
    }
    // bstats, dmax and xmax are consecutive regions
    MVX_CUDA_CHECK(cudaMemsetAsync(ws + M.bstats, 0, M.ones - M.bstats, st));
    dense_rowset_kernel<<<(unsigned)ceil_div(R, 256), 256, 0, st>>>(counts, ones, Ri);
    MVX_LAUNCH_CHECK();
    // dz
    if (kind != kFcn) {
        const long long V = R / T;
        const unsigned blocks = (unsigned)ceil_div(V * Cout, 256);
        if (kind == kVfe) route_max_kernel<true><<<blocks, 256, 0, st>>>(y_raw, dy, G, V, T, Cout);
        else route_max_kernel<false><<<blocks, 256, 0, st>>>(y_raw, dy, G, V, T, Cout);
        MVX_LAUNCH_CHECK();
    } else {
        MVX_CUDA_CHECK(cudaMemcpyAsync(G, dy, (size_t)R * Cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    // dpre (in place) and db
    rc = launch_bn_back_voxel_rows(G, y_raw, Cout, static_cast<const double *>(stats_ws), bstats, db, eps, counts, Ri, ones, dmax, st);
    if (rc) return rc;
    // dW = dpre^T x: the tensor-core kernel scales the raw x per column
    const bool tc_dw = gemm_mode() == 1 && Cout % 128 == 0 && Cin % 128 == 0;
    if (tc_dw) {
        col_absmax_kernel<<<(unsigned)ceil_div(R, kColRows), 256, 0, st>>>(x, Ri, Cin, xmax);
        MVX_LAUNCH_CHECK();
    }
    rc = launch_dw_voxel_rows(G, Cout, x, Cin, counts, Ri, dmax, dW, 1, st, tc_dw ? xmax : nullptr);
    if (rc) return rc;
    if (!dx) return MVX_OK;
    // dx = dpre W: a plain product (3xTF32 on the one-tile tensor-core kernel where eligible; gradients have no bounded range)
    float *w = reinterpret_cast<float *>(ws + M.w);
    rc = launch_transpose_w(wt, w, Cin, Cout, st);
    if (rc) return rc;
    LayerArgs la{};
    la.X = G, la.ldx = Cout, la.Cin = Cout, la.Wt = w, la.bias = nullptr, la.Cout = Cin;
    la.Y = dx, la.ldy = Cin, la.rows_mode = 0, la.rows_fixed = R, la.rowcap = Ri, la.T = 1, la.eps = eps;
    la.plain = 1, la.f16_ok = 0;
    return launch_layer_auto(la, 1, reinterpret_cast<float *>(ws + M.wpack), st);
}

int layer_workspace(long long R, int T, int Cin, int Cout, size_t *bytes) {
    MVX_REQUIRE(bytes, MVX_EINVAL, "null pointer");
    int rc = check_layer_args(R, T, Cin, Cout);
    if (rc) return rc;
    *bytes = mw_layout(R, Cin, Cout).total;
    return MVX_OK;
}

}  // namespace

}  // namespace mvx

extern "C" int mvx_fcn_backward_workspace_bytes(int64_t R, int32_t Cin, int32_t Cout, size_t *bytes) {
    return mvx::layer_workspace(R, 1, Cin, Cout, bytes);
}
extern "C" int mvx_vfe_backward_workspace_bytes(int64_t R, int32_t T, int32_t Cin, int32_t Cout, size_t *bytes) {
    return mvx::layer_workspace(R, T, Cin, Cout, bytes);
}
extern "C" int mvx_fcn_max_backward_workspace_bytes(int64_t R, int32_t T, int32_t Cin, int32_t Cout, size_t *bytes) {
    return mvx::layer_workspace(R, T, Cin, Cout, bytes);
}

extern "C" int mvx_fcn_backward(const float *x, int64_t R, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw, const void *stats_ws,
                                double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate, void *ws, size_t ws_bytes,
                                void *stream) {
    return mvx::layer_backward(mvx::kFcn, x, R, 1, Cin, wt, Cout, y_raw, stats_ws, eps, dy, dx, dW, db, accumulate, ws, ws_bytes,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int mvx_vfe_backward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw,
                                const void *stats_ws, double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate, void *ws,
                                size_t ws_bytes, void *stream) {
    return mvx::layer_backward(mvx::kVfe, x, R, T, Cin, wt, Cout, y_raw, stats_ws, eps, dy, dx, dW, db, accumulate, ws, ws_bytes,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int mvx_fcn_max_backward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, int32_t Cout, const float *y_raw,
                                    const void *stats_ws, double eps, const float *dy, float *dx, float *dW, float *db, int32_t accumulate,
                                    void *ws, size_t ws_bytes, void *stream) {
    return mvx::layer_backward(mvx::kFcnMax, x, R, T, Cin, wt, Cout, y_raw, stats_ws, eps, dy, dx, dW, db, accumulate, ws, ws_bytes,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int mvx_scatter_dense_backward(const float *d_grid, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny, int32_t nz,
                                          float *d_feat, void *stream) {
    MVX_REQUIRE(N >= 0 && C > 0 && nx > 0 && ny > 0 && nz > 0, MVX_EINVAL, "bad scatter backward argument");
    if (N == 0) return MVX_OK;
    MVX_REQUIRE(d_grid && idx && d_feat, MVX_EINVAL, "null d_grid / idx / d_feat");
    mvx::scatter_back_kernel<<<(unsigned)mvx::ceil_div(N * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        d_grid, reinterpret_cast<const long long *>(idx), N, C, nx, ny, nz, d_feat);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
