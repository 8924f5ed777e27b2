// §8f rank 2 — the step immediately AFTER the path: the first middle-layer convolution of VoxelNet's CML,
// CRB3d(128, 64, k=3, stride (2,1,1), pad (1,1,1)) = relu(Conv3d) then batch-statistic BatchNorm3d
// (modules/voxelnet/Pipe.py:31-43 `CML.conv1`, modules/layers/Blocks.py CRB3d), evaluated SPARSELY from the voxel features
// instead of from the dense (128,10,352,400) grid: > 98 % of that grid is zero, writing it is 93 % of the path's
// compulsory HBM bytes and the dense convolution then re-reads it (311 GFLOP per frame).
//
// Formulation: conv(grid)[o] = b + sum over the 27 taps t of W_t feat[vid(neighbour_t(o))], over the non-empty neighbours.
//   (1) P[v][t][0:64] = W_t feat[v] for every voxel and tap: ONE tensor-core GEMM (N_f x 128) x (128 x 1728, padded to
//       1792) per frame - 9.4 GFLOP instead of 311, through the plain 3xFP16 layer kernel;
//   (2) per output position: look the 27 neighbours up in the cell -> voxel map (L2-resident), sum the P rows of the
//       non-empty ones, + bias, ReLU. Positions with no non-empty neighbour ("background") equal relu(b) and are not
//       stored: active positions go to a compact (n_act, 64) buffer with a position -> index map;
//   (3) BatchNorm statistics = column sums of the active rows + n_background * relu(b) analytically (fp64);
//   (4) one streaming pass writes the dense (64, 5, nx, ny) result: normalised active rows and the normalised background
//       constant of each channel. 1.44 GB per 8 frames instead of the 5.8 GB grid.
#include "layers.cuh"
#include "pointpath.cuh"

#include <algorithm>

namespace mvx {

namespace {

constexpr int kSC_Cout = 64, kSC_Cin = 128, kSC_Taps = 27, kSC_PLd = 1792;   // 27 * 64 = 1728 columns, padded to 14 * 128

struct ScGeom {
    int nz, nx, ny, oz;          // input grid (nz, nx, ny), output depth oz = (nz + 2 - 3) / 2 + 1
    long long G, Go;             // cells of the input grid / positions of the output (oz * nx * ny)
};

// W (64,128,3,3,3) [o][c][kz][kx][ky] -> Wt (128, 1792): column t * 64 + o, t = (kz * 3 + kx) * 3 + ky; padding columns zero
__global__ void __launch_bounds__(256) sc_pack_w_kernel(const float *__restrict__ W, float *__restrict__ Wt) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= kSC_Cin * kSC_PLd) return;
    const int c = e / kSC_PLd, col = e - c * kSC_PLd;
    float v = 0.f;
    if (col < kSC_Taps * kSC_Cout) {
        const int t = col / kSC_Cout, o = col - t * kSC_Cout;
        v = W[((size_t)o * kSC_Cin + c) * kSC_Taps + t];
    }
    Wt[e] = v;
}

// pass 2: one thread per output position. Neighbour look-ups, sum of the P rows, bias + ReLU, compact store.
__global__ void __launch_bounds__(128) sc_gather_kernel(ScGeom g, const int *__restrict__ cell2vid, const float *__restrict__ P, int cap,
                                                        const float *__restrict__ bias, int *__restrict__ act_count, int *__restrict__ act_idx,
                                                        float *__restrict__ Yact, int act_cap) {
    const int f = blockIdx.y;
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.Go) return;
    const int oy = (int)(p % g.ny), ox = (int)((p / g.ny) % g.nx), oz = (int)(p / ((long long)g.ny * g.nx));
    const int *map = cell2vid + (size_t)f * g.G;
    int vids[kSC_Taps];
    int any = 0;
#pragma unroll
    for (int t = 0; t < kSC_Taps; ++t) {
        const int kz = t / 9, kx = (t / 3) % 3, ky = t % 3;
        const int iz = 2 * oz + kz - 1, ix = ox + kx - 1, iy = oy + ky - 1;
        int v = -1;
        if (iz >= 0 && iz < g.nz && ix >= 0 && ix < g.nx && iy >= 0 && iy < g.ny) v = __ldg(map + ((size_t)iz * g.nx + ix) * g.ny + iy);
        vids[t] = v;
        any |= (v >= 0);
    }
    int idx = -1;
    if (any) {   // warp-aggregated claim of a compact row
        const unsigned m = __activemask();
        const int leader = __ffs(m) - 1, lane = threadIdx.x & 31;
        int base = 0;
        if (lane == leader) base = atomicAdd(act_count + f, __popc(m));
        base = __shfl_sync(m, base, leader);
        idx = base + __popc(m & ((1u << lane) - 1));
    }
    act_idx[(size_t)f * g.Go + p] = (idx >= 0 && idx < act_cap) ? idx : -1;
    if (idx < 0 || idx >= act_cap) return;
    float acc[kSC_Cout];
#pragma unroll
    for (int o = 0; o < kSC_Cout; ++o) acc[o] = __ldg(bias + o);
    const float *Pf = P + (size_t)f * cap * kSC_PLd;
#pragma unroll 1
    for (int t = 0; t < kSC_Taps; ++t) {
        const int v = vids[t];
        if (v < 0) continue;
        const float4 *row = reinterpret_cast<const float4 *>(Pf + (size_t)v * kSC_PLd + t * kSC_Cout);
#pragma unroll
        for (int q = 0; q < kSC_Cout / 4; ++q) {
            const float4 x = __ldg(row + q);
            acc[4 * q] += x.x, acc[4 * q + 1] += x.y, acc[4 * q + 2] += x.z, acc[4 * q + 3] += x.w;
        }
    }
    float4 *out = reinterpret_cast<float4 *>(Yact + ((size_t)f * act_cap + idx) * kSC_Cout);
#pragma unroll
    for (int q = 0; q < kSC_Cout / 4; ++q)
        out[q] = make_float4(fmaxf(acc[4 * q], 0.f), fmaxf(acc[4 * q + 1], 0.f), fmaxf(acc[4 * q + 2], 0.f), fmaxf(acc[4 * q + 3], 0.f));
}

// pass 3: column sums of the active rows (fp64), 64 columns
__global__ void __launch_bounds__(256) sc_stats_kernel(const float *__restrict__ Yact, const int *__restrict__ act_count, int act_cap,
                                                       double *__restrict__ stats) {
    __shared__ double s_acc[kSC_Cout * 2];
    const int f = blockIdx.y, tid = threadIdx.x;
    const int n = min(act_count[f], act_cap);
    const int row0 = blockIdx.x * 1024;
    if (row0 >= n) return;
    if (tid < kSC_Cout * 2) s_acc[tid] = 0.0;
    __syncthreads();
    const int c = (tid & 15) * 4, rg = tid >> 4;   // 16 column groups x 16 row groups
    double s[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
    const int rend = min(row0 + 1024, n);
    for (int r = row0 + rg; r < rend; r += 16) {
        const float4 y = *reinterpret_cast<const float4 *>(Yact + ((size_t)f * act_cap + r) * kSC_Cout + c);
        s[0] += y.x, s[1] += y.y, s[2] += y.z, s[3] += y.w;
        ss[0] += (double)y.x * y.x, ss[1] += (double)y.y * y.y, ss[2] += (double)y.z * y.z, ss[3] += (double)y.w * y.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {   // lanes l and l + 16 share the columns
        s[j] += __shfl_xor_sync(0xffffffffu, s[j], 16);
        ss[j] += __shfl_xor_sync(0xffffffffu, ss[j], 16);
    }
    if ((tid & 31) < 16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_acc[(c + j) * 2], s[j]);
            atomicAdd(&s_acc[(c + j) * 2 + 1], ss[j]);
        }
    }
    __syncthreads();
    if (tid < kSC_Cout * 2) atomicAdd(stats + (size_t)f * kSC_Cout * 2 + tid, s_acc[tid]);
}

// per-channel BatchNorm moments of frame f over all Go positions: the active rows' sums plus n_background * relu(b)
struct ScMoments {
    double R, n_bg, bg, m, r;   // positions, background positions, relu(b), mean, rstd
};
__device__ __forceinline__ ScMoments sc_moments(const ScGeom &g, const int *act_count, int act_cap, const float *bias,
                                                const double *stats, double eps, int f, int c) {
    ScMoments M;
    const double n_act = (double)min(act_count[f], act_cap);
    M.R = (double)g.Go, M.n_bg = M.R - n_act;
    M.bg = fmax((double)bias[c], 0.0);
    const double *st = stats + ((size_t)f * kSC_Cout + c) * 2;
    M.m = (st[0] + M.n_bg * M.bg) / M.R;
    double var = (st[1] + M.n_bg * M.bg * M.bg) / M.R - M.m * M.m;
    var = var < 0.0 ? 0.0 : var;
    M.r = 1.0 / sqrt(var + eps);
    return M;
}

// pass 4: dense (64, Go) output: normalised active rows, normalised background constant elsewhere.
// CTA = 32 consecutive positions x 64 channels through a padded shared tile (coalesced on both sides).
__global__ void __launch_bounds__(256) sc_write_kernel(ScGeom g, const int *__restrict__ act_idx, const float *__restrict__ Yact,
                                                       const int *__restrict__ act_count, int act_cap, const float *__restrict__ bias,
                                                       const double *__restrict__ stats, double eps, float *__restrict__ out) {
    __shared__ float s_mean[kSC_Cout], s_rstd[kSC_Cout], s_bg[kSC_Cout];
    __shared__ float tile[kSC_Cout][33];
    __shared__ int s_idx[32];
    const int f = blockIdx.y, tid = threadIdx.x;
    if (tid < kSC_Cout) {
        const ScMoments M = sc_moments(g, act_count, act_cap, bias, stats, eps, f, tid);
        const double m = M.m, r = M.r, bg = M.bg;
        s_mean[tid] = (float)m, s_rstd[tid] = (float)r;
        s_bg[tid] = (float)(((double)(float)bg - m) * r);
    }
    const long long p0 = (long long)blockIdx.x * 32;
    if (tid < 32) s_idx[tid] = p0 + tid < g.Go ? act_idx[(size_t)f * g.Go + p0 + tid] : -1;
    __syncthreads();
    // gather phase: thread = (position tid / 8, 8 channels): a compact row is 256 contiguous bytes
    {
        const int pl = tid >> 3, c0 = (tid & 7) * 8, idx = s_idx[pl];
        if (idx >= 0) {
            const float4 *row = reinterpret_cast<const float4 *>(Yact + ((size_t)f * act_cap + idx) * kSC_Cout + c0);
            const float4 a = row[0], b = row[1];
            const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) tile[c0 + j][pl] = (v[j] - s_mean[c0 + j]) * s_rstd[c0 + j];
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) tile[c0 + j][pl] = s_bg[c0 + j];
        }
    }
    __syncthreads();
    // store phase: a warp writes 32 consecutive positions of one channel plane (128 contiguous bytes)
    const int lane = tid & 31, w = tid >> 5;
    if (p0 + lane < g.Go) {
#pragma unroll
        for (int c = w; c < kSC_Cout; c += 8)
            out[((size_t)f * kSC_Cout + c) * g.Go + p0 + lane] = tile[c][lane];
    }
}

// ---- backward ------------------------------------------------------------------------------------------------------
// Per-frame sums of the backward, [B][64][4] fp64: S1 = sum_all g, A1 = sum_A g, A2 = sum_A g * Yact, DA = sum_A dpre.
enum { kScS1 = 0, kScA1, kScA2, kScDA, kScSums };

// S2 = sum_all g * z = r * (sum_all g * y - m * S1), with sum_all g * y = A2 + relu(b) * (S1 - A1) (background y = relu(b))
__device__ __forceinline__ double sc_s2(const ScMoments &M, const double *s) {
    return M.r * (s[kScA2] + M.bg * (s[kScS1] - s[kScA1]) - M.m * s[kScS1]);
}

// b1: one streaming pass over dOut, tiled like sc_write_kernel (32 positions x 64 channels, coalesced along the planes).
// Column sums S1 / A1 / A2 in fp64 registers over all tiles of the CTA, one atomic per CTA and sum; the dOut values of
// the active positions go to the compact G (n_act, 64), so nothing later reads the dense tensor again.
__global__ void __launch_bounds__(256) scb_reduce_kernel(ScGeom g, const int *__restrict__ act_idx, const float *__restrict__ Yact, int act_cap,
                                                         const float *__restrict__ dout, float *__restrict__ G, double *__restrict__ sums) {
    __shared__ float tile[kSC_Cout][33];
    __shared__ int s_idx[32];
    __shared__ double s_acc[kSC_Cout * 3];
    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int pl = tid >> 3, c0 = (tid & 7) * 8;   // second phase: position pl, channels c0 .. c0 + 7 (a 32-byte piece of a row)
    if (tid < kSC_Cout * 3) s_acc[tid] = 0.0;
    __syncthreads();
    double s1[8], a1[8], a2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s1[j] = a1[j] = a2[j] = 0.0;
    const float *df = dout + (size_t)f * kSC_Cout * g.Go;
    const long long ntiles = (g.Go + 31) / 32;
    for (long long tt = blockIdx.x; tt < ntiles; tt += gridDim.x) {
        const long long p0 = tt * 32;
        const bool in = p0 + lane < g.Go;
        if (tid < 32) s_idx[tid] = in ? act_idx[(size_t)f * g.Go + p0 + tid] : -1;
#pragma unroll
        for (int c = w; c < kSC_Cout; c += 8) tile[c][lane] = in ? __ldg(df + (size_t)c * g.Go + p0 + lane) : 0.f;
        __syncthreads();
        const int idx = s_idx[pl];
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            v[j] = tile[c0 + j][pl];
            s1[j] += (double)v[j];
        }
        if (idx >= 0) {
            const size_t ro = ((size_t)f * act_cap + idx) * kSC_Cout + c0;
            const float4 ya = *reinterpret_cast<const float4 *>(Yact + ro), yb = *reinterpret_cast<const float4 *>(Yact + ro + 4);
            const float y[8] = {ya.x, ya.y, ya.z, ya.w, yb.x, yb.y, yb.z, yb.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                a1[j] += (double)v[j];
                a2[j] += (double)v[j] * (double)y[j];
            }
            *reinterpret_cast<float4 *>(G + ro) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4 *>(G + ro + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {   // lanes l, l ^ 8, l ^ 16, l ^ 24 hold the same columns
#pragma unroll
        for (int d = 8; d <= 16; d <<= 1) {
            s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], d);
            a1[j] += __shfl_xor_sync(0xffffffffu, a1[j], d);
            a2[j] += __shfl_xor_sync(0xffffffffu, a2[j], d);
        }
    }
    if (lane < 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            atomicAdd(&s_acc[(c0 + j) * 3 + 0], s1[j]);
            atomicAdd(&s_acc[(c0 + j) * 3 + 1], a1[j]);
            atomicAdd(&s_acc[(c0 + j) * 3 + 2], a2[j]);
        }
    }
    __syncthreads();
    if (tid < kSC_Cout * 3) {
        const double s = s_acc[tid];
        if (s != 0.0) atomicAdd(sums + ((size_t)f * kSC_Cout + tid / 3) * kScSums + tid % 3, s);
    }
}

// b2: dpre = r (g - S1/R - z S2/R) [Yact > 0] on the compact rows, in place in G; DA = column sums of dpre and the
// column maxima of |dpre| (the power-of-two scales of the tensor-core dW)
constexpr int kScbRows = 1024;
__global__ void __launch_bounds__(256) scb_dpre_kernel(ScGeom g, const int *__restrict__ act_count, int act_cap, const float *__restrict__ Yact,
                                                       const float *__restrict__ bias, const double *__restrict__ stats, double eps,
                                                       double *__restrict__ sums, float *__restrict__ G, int *__restrict__ dmax64) {
    __shared__ double s_acc[kSC_Cout];
    __shared__ int s_mx[kSC_Cout];
    const int f = blockIdx.y, tid = threadIdx.x;
    const int n = min(act_count[f], act_cap);
    const int row0 = blockIdx.x * kScbRows;
    if (row0 >= n) return;
    if (tid < kSC_Cout) s_acc[tid] = 0.0, s_mx[tid] = 0;
    const int c = (tid & 15) * 4, rg = tid >> 4;   // 16 column groups x 16 row groups
    double m[4], r[4], k1[4], k2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const ScMoments M = sc_moments(g, act_count, act_cap, bias, stats, eps, f, c + j);
        const double *s = sums + ((size_t)f * kSC_Cout + c + j) * kScSums;
        m[j] = M.m, r[j] = M.r, k1[j] = s[kScS1] / M.R, k2[j] = sc_s2(M, s) / M.R;
    }
    __syncthreads();
    double sb[4] = {0, 0, 0, 0};
    float mx[4] = {0.f, 0.f, 0.f, 0.f};
    const int rend = min(row0 + kScbRows, n);
    for (int rr = row0 + rg; rr < rend; rr += 16) {
        const size_t o = ((size_t)f * act_cap + rr) * kSC_Cout + c;
        const float4 gv = *reinterpret_cast<const float4 *>(G + o), yv = *reinterpret_cast<const float4 *>(Yact + o);
        const float gg[4] = {gv.x, gv.y, gv.z, gv.w}, y[4] = {yv.x, yv.y, yv.z, yv.w};
        float d[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double z = ((double)y[j] - m[j]) * r[j];
            d[j] = y[j] > 0.f ? (float)(r[j] * ((double)gg[j] - k1[j] - z * k2[j])) : 0.f;
            sb[j] += (double)d[j];
            mx[j] = fmaxf(mx[j], fabsf(d[j]));
        }
        *reinterpret_cast<float4 *>(G + o) = make_float4(d[0], d[1], d[2], d[3]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {   // lanes l and l + 16 share the columns
        sb[j] += __shfl_xor_sync(0xffffffffu, sb[j], 16);
        mx[j] = fmaxf(mx[j], __shfl_xor_sync(0xffffffffu, mx[j], 16));
    }
    if ((tid & 31) < 16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_acc[c + j], sb[j]);
            atomicMax(&s_mx[c + j], __float_as_int(mx[j]));   // |dpre| >= 0: float bits order like ints
        }
    }
    __syncthreads();
    if (tid < kSC_Cout) {
        atomicAdd(sums + ((size_t)f * kSC_Cout + tid) * kScSums + kScDA, s_acc[tid]);
        atomicMax(dmax64 + (size_t)f * kSC_Cout + tid, s_mx[tid]);
    }
}

// b3: db = sum over frames of DA + [b > 0] r ((S1 - A1) - n_bg S1/R - z_bg n_bg S2/R): the background part is analytic
__global__ void __launch_bounds__(kSC_Cout) scb_bias_kernel(ScGeom g, int B, const int *__restrict__ act_count, int act_cap,
                                                            const float *__restrict__ bias, const double *__restrict__ stats, double eps,
                                                            const double *__restrict__ sums, float *__restrict__ d_b, int accumulate) {
    const int c = threadIdx.x;
    double acc = 0.0;
    for (int f = 0; f < B; ++f) {
        const ScMoments M = sc_moments(g, act_count, act_cap, bias, stats, eps, f, c);
        const double *s = sums + ((size_t)f * kSC_Cout + c) * kScSums;
        acc += s[kScDA];
        if (bias[c] > 0.f) {
            const double z_bg = ((double)(float)M.bg - M.m) * M.r;
            acc += M.r * ((s[kScS1] - s[kScA1]) - M.n_bg * s[kScS1] / M.R - z_bg * M.n_bg * sc_s2(M, s) / M.R);
        }
    }
    d_b[c] = (accumulate ? d_b[c] : 0.f) + (float)acc;
}

// b4: D[v][t * 64 + o] = dpre[pos(v, t)][o], the mirror of P[v][t] = W_t feat[v]: voxel v reaches output position
// pos(v, t) through tap t when iz + 1 - kz is even and the position lies inside the output grid; zero otherwise and in
// the padding slot t = 27. Thread = one float4 of one (voxel, tap slot): 256-byte rows, no atomics. Block 0 of each frame
// also spreads the channel maxima of |dpre| over the 1792 columns of D (a bound of every tap's column maximum).
__global__ void __launch_bounds__(256) scb_tap_gather_kernel(ScGeom g, const int *__restrict__ counts, const int *__restrict__ vox_coord, int cap,
                                                             const int *__restrict__ act_idx, const float *__restrict__ G, int act_cap,
                                                             float *__restrict__ D, const int *__restrict__ dmax64, int *__restrict__ dmax) {
    constexpr int kSlots = kSC_PLd / kSC_Cout, kQ = kSC_Cout / 4;   // 28 tap slots of 16 float4
    const int f = blockIdx.y;
    if (blockIdx.x == 0)
        for (int col = threadIdx.x; col < kSC_PLd; col += blockDim.x)
            dmax[(size_t)f * kSC_PLd + col] = col < kSC_Taps * kSC_Cout ? dmax64[(size_t)f * kSC_Cout + (col & (kSC_Cout - 1))] : 0;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int v = (int)(e / (kSlots * kQ)), rem = (int)(e - (long long)v * (kSlots * kQ)), t = rem / kQ, q = rem - t * kQ;
    if (v >= counts[f * 4 + 0]) return;
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < kSC_Taps) {
        const int4 vc = *reinterpret_cast<const int4 *>(vox_coord + ((size_t)f * cap + v) * 4);   // ix, iy, iz, cell (-1: outside)
        const int kz = t / 9, kx = (t / 3) % 3, ky = t % 3;
        const int oz2 = vc.z + 1 - kz, ox = vc.x + 1 - kx, oy = vc.y + 1 - ky;
        if (vc.w >= 0 && oz2 >= 0 && (oz2 & 1) == 0 && (oz2 >> 1) < g.oz && ox >= 0 && ox < g.nx && oy >= 0 && oy < g.ny) {
            const int idx = act_idx[(size_t)f * g.Go + ((size_t)(oz2 >> 1) * g.nx + ox) * g.ny + oy];
            if (idx >= 0) val = __ldg(reinterpret_cast<const float4 *>(G + ((size_t)f * act_cap + idx) * kSC_Cout) + q);
        }
    }
    reinterpret_cast<float4 *>(D + ((size_t)f * cap + v) * kSC_PLd + t * kSC_Cout)[q] = val;
}

// W (64,128,3,3,3) -> Wb (1792, 128): row t * 64 + o, column c holds W[o][c][t]; padding rows zero (d_vfeat = D Wb)
__global__ void __launch_bounds__(256) scb_pack_wb_kernel(const float *__restrict__ W, float *__restrict__ Wb) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= kSC_PLd * kSC_Cin) return;
    const int k = e / kSC_Cin, c = e - k * kSC_Cin;
    float v = 0.f;
    if (k < kSC_Taps * kSC_Cout) {
        const int t = k / kSC_Cout, o = k - t * kSC_Cout;
        v = W[((size_t)o * kSC_Cin + c) * kSC_Taps + t];
    }
    Wb[e] = v;
}

// dWcat (1792, 128) -> d_w (64,128,3,3,3): d_w[o][c][t] (+)= dWcat[t * 64 + o][c]
__global__ void __launch_bounds__(256) scb_unpack_dw_kernel(const float *__restrict__ dWcat, float *__restrict__ d_w, int accumulate) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= kSC_Cout * kSC_Cin * kSC_Taps) return;
    const int o = e / (kSC_Cin * kSC_Taps), c = (e / kSC_Taps) % kSC_Cin, t = e % kSC_Taps;
    const float v = dWcat[((size_t)t * kSC_Cout + o) * kSC_Cin + c];
    d_w[e] = accumulate ? d_w[e] + v : v;
}

struct ScLayout {
    size_t wt, wpack, P, act_count, act_idx, yact, stats, total;
    ScGeom g;
};

int sc_layout(const mvx_pointpath_args_t *a, ScLayout &S) {
    MVX_REQUIRE(a && a->B >= 1 && a->B <= 32 && a->cap >= 128, MVX_EINVAL, "bad path arguments");
    S.g.nx = a->grid.shape[0], S.g.ny = a->grid.shape[1], S.g.nz = a->grid.shape[2];
    MVX_REQUIRE(S.g.nx > 0 && S.g.ny > 0 && S.g.nz > 0, MVX_EINVAL, "bad grid shape");
    S.g.oz = (S.g.nz + 2 - 3) / 2 + 1;
    S.g.G = (long long)S.g.nz * S.g.nx * S.g.ny;
    S.g.Go = (long long)S.g.oz * S.g.nx * S.g.ny;
    size_t o = 0;
    auto take = [&](size_t &slot, size_t bytes) {
        slot = o;
        o += (bytes + 255) / 256 * 256;
    };
    const size_t B = a->B;
    take(S.wt, (size_t)kSC_Cin * kSC_PLd * 4);
    take(S.wpack, tc_wpack_bytes(kSC_Cin, kSC_PLd));
    take(S.P, B * a->cap * kSC_PLd * 4);
    take(S.act_count, B * 4);
    take(S.act_idx, B * (size_t)S.g.Go * 4);
    take(S.yact, B * (size_t)S.g.Go * kSC_Cout * 4);
    take(S.stats, B * kSC_Cout * 2 * 8);
    S.total = o;
    return MVX_OK;
}

// backward scratch: D lives here rather than in the forward's (dead) P region, so the forward's workspace stays read-only
// and the backward can be repeated (accumulate)
struct ScbLayout {
    size_t wb, wpack, G, sums, dmax64, dmax, D, dwcat, total;
};

void scb_layout(const mvx_pointpath_args_t *a, const ScLayout &S, ScbLayout &Q) {
    size_t o = 0;
    auto take = [&](size_t &slot, size_t bytes) {
        slot = o;
        o += (bytes + 255) / 256 * 256;
    };
    const size_t B = a->B;
    take(Q.wb, (size_t)kSC_PLd * kSC_Cin * 4);
    take(Q.wpack, tc_wpack_bytes(kSC_PLd, kSC_Cin));
    take(Q.G, B * (size_t)S.g.Go * kSC_Cout * 4);
    take(Q.sums, B * kSC_Cout * kScSums * 8);
    take(Q.dmax64, B * kSC_Cout * 4);
    take(Q.dmax, B * kSC_PLd * 4);
    take(Q.D, B * a->cap * kSC_PLd * 4);
    take(Q.dwcat, (size_t)kSC_PLd * kSC_Cin * 4);
    Q.total = o;
}

}  // namespace
}  // namespace mvx

extern "C" int mvx_cml_conv1_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes) {
    mvx::ScLayout S;
    int rc = mvx::sc_layout(args, S);
    if (rc) return rc;
    if (!bytes) return MVX_EINVAL;
    *bytes = S.total;
    return MVX_OK;
}

extern "C" int mvx_cml_conv1_sparse(const mvx_pointpath_args_t *a, const float *conv_w, const float *conv_b, double eps, float *out,
                                    void *ws_v, size_t ws_bytes) {
    using namespace mvx;
    ScLayout S;
    int rc = sc_layout(a, S);
    if (rc) return rc;
    Layout L;
    rc = make_layout(a, L);
    if (rc) return rc;
    MVX_REQUIRE(conv_w && conv_b && out && ws_v && a->workspace && a->counts, MVX_EINVAL, "null pointer");
    MVX_REQUIRE(ws_bytes >= S.total && a->workspace_bytes >= L.total, MVX_ESPACE, "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    char *ws = static_cast<char *>(ws_v), *pws = static_cast<char *>(a->workspace);
    const int B = a->B, cap = a->cap;
    float *Wt = reinterpret_cast<float *>(ws + S.wt), *P = reinterpret_cast<float *>(ws + S.P);
    int *act_count = reinterpret_cast<int *>(ws + S.act_count), *act_idx = reinterpret_cast<int *>(ws + S.act_idx);
    float *Yact = reinterpret_cast<float *>(ws + S.yact);
    double *stats = reinterpret_cast<double *>(ws + S.stats);
    const float *vfeat = reinterpret_cast<const float *>(pws + L.off[R_VFEAT]);
    const int *cell2vid = reinterpret_cast<const int *>(pws + L.off[R_CELL2VID]);

    sc_pack_w_kernel<<<(kSC_Cin * kSC_PLd + 255) / 256, 256, 0, st>>>(conv_w, Wt);
    MVX_LAUNCH_CHECK();
    // (1) P[v] = feat[v] Wcat for the N_f voxels of every frame: plain tensor-core GEMM (the voxel features are BatchNorm-ed)
    LayerArgs la{};
    la.X = vfeat, la.ldx = kSC_Cin, la.Cin = kSC_Cin, la.Wt = Wt, la.bias = nullptr, la.Cout = kSC_PLd;
    la.Y = P, la.ldy = kSC_PLd, la.counts = a->counts, la.rows_mode = 3, la.rowcap = cap, la.vcap = cap, la.T = a->grid.T;
    la.eps = eps, la.plain = 1, la.f16_ok = 1;
    rc = launch_layer_auto(la, B, reinterpret_cast<float *>(ws + S.wpack), st);
    if (rc) return rc;
    // (2) gather per output position
    MVX_CUDA_CHECK(cudaMemsetAsync(act_count, 0, (size_t)B * 4, st));
    MVX_CUDA_CHECK(cudaMemsetAsync(stats, 0, (size_t)B * kSC_Cout * 2 * 8, st));
    const int act_cap = (int)S.g.Go;
    sc_gather_kernel<<<dim3((unsigned)ceil_div(S.g.Go, 128), B), 128, 0, st>>>(S.g, cell2vid, P, cap, conv_b, act_count, act_idx, Yact, act_cap);
    MVX_LAUNCH_CHECK();
    // (3) statistics of the active rows
    sc_stats_kernel<<<dim3((unsigned)ceil_div(S.g.Go, 1024), B), 256, 0, st>>>(Yact, act_count, act_cap, stats);
    MVX_LAUNCH_CHECK();
    // (4) dense normalised output
    sc_write_kernel<<<dim3((unsigned)ceil_div(S.g.Go, 32), B), 256, 0, st>>>(S.g, act_idx, Yact, act_count, act_cap, conv_b, stats, eps, out);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

// Backward of the hand-off: gradients of sum(out * d_out) with respect to conv_w, conv_b and the voxel features, for the
// CRB3d of voxelnet/Pipe.py:31-43 (Blocks.py CRB3d: BatchNorm3d(relu(Conv3d(x))), batch statistics, affine=False).
// Background positions see only zero inputs, so they add nothing to dW or d_vfeat, and their share of db is analytic.
//   (b1) S1 / A1 / A2 and the compact dOut rows of the active positions      (one pass over d_out, HBM-bound)
//   (b2) dpre on the compact rows, DA = their column sums                      (b3) db
//   (b4) D[v][t * 64 + o] = dpre[pos(v, t)][o]                                 (B x cap x 1792, padded like P)
//   (b5) dWcat = sum_f D^T vfeat (1792 x 128) on the tensor-core dW kernel (3xFP16, power-of-two column scales of D)
//   (b6) d_vfeat = D Wb (Wb = the 1792 x 128 tap-major weights) on the tensor-core layer kernel in 3xTF32: gradients
//        have no O(1) bound
extern "C" int mvx_cml_conv1_backward_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes) {
    mvx::ScLayout S;
    int rc = mvx::sc_layout(args, S);
    if (rc) return rc;
    if (!bytes) return MVX_EINVAL;
    mvx::ScbLayout Q;
    mvx::scb_layout(args, S, Q);
    *bytes = Q.total;
    return MVX_OK;
}

extern "C" int mvx_cml_conv1_sparse_backward(const mvx_pointpath_args_t *a, const float *conv_w, const float *conv_b, double eps,
                                             const float *d_out, float *d_vfeat, float *d_w, float *d_b, int32_t accumulate,
                                             const void *ws_v, size_t ws_bytes, void *bws_v, size_t bws_bytes) {
    using namespace mvx;
    ScLayout S;
    int rc = sc_layout(a, S);
    if (rc) return rc;
    Layout L;
    rc = make_layout(a, L);
    if (rc) return rc;
    ScbLayout Q;
    scb_layout(a, S, Q);
    MVX_REQUIRE(conv_w && conv_b && d_out && d_w && d_b && ws_v && bws_v && a->workspace && a->counts, MVX_EINVAL, "null pointer");
    MVX_REQUIRE(ws_bytes >= S.total && bws_bytes >= Q.total && a->workspace_bytes >= L.total, MVX_ESPACE, "workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    const char *ws = static_cast<const char *>(ws_v), *pws = static_cast<const char *>(a->workspace);
    char *bws = static_cast<char *>(bws_v);
    const int B = a->B, cap = a->cap, act_cap = (int)S.g.Go;
    const int *act_count = reinterpret_cast<const int *>(ws + S.act_count), *act_idx = reinterpret_cast<const int *>(ws + S.act_idx);
    const float *Yact = reinterpret_cast<const float *>(ws + S.yact);
    const double *stats = reinterpret_cast<const double *>(ws + S.stats);
    const float *vfeat = reinterpret_cast<const float *>(pws + L.off[R_VFEAT]);
    const int *vox_coord = reinterpret_cast<const int *>(pws + L.off[R_VOX_COORD]);
    float *G = reinterpret_cast<float *>(bws + Q.G), *D = reinterpret_cast<float *>(bws + Q.D);
    float *dwcat = reinterpret_cast<float *>(bws + Q.dwcat), *Wb = reinterpret_cast<float *>(bws + Q.wb);
    double *sums = reinterpret_cast<double *>(bws + Q.sums);
    int *dmax64 = reinterpret_cast<int *>(bws + Q.dmax64), *dmax = reinterpret_cast<int *>(bws + Q.dmax);

    MVX_CUDA_CHECK(cudaMemsetAsync(sums, 0, (size_t)B * kSC_Cout * kScSums * 8, st));
    MVX_CUDA_CHECK(cudaMemsetAsync(dmax64, 0, (size_t)B * kSC_Cout * 4, st));
    MVX_CUDA_CHECK(cudaMemsetAsync(dwcat, 0, (size_t)kSC_PLd * kSC_Cin * 4, st));
    // (b1) enough CTAs for eight per SM over the batch; each walks its share of the frame's 32-position tiles
    const long long tiles = ceil_div(S.g.Go, 32);
    const unsigned per_frame = (unsigned)std::max<long long>(1, std::min<long long>(tiles, ceil_div(kSMs * 8, B)));
    scb_reduce_kernel<<<dim3(per_frame, B), 256, 0, st>>>(S.g, act_idx, Yact, act_cap, d_out, G, sums);
    MVX_LAUNCH_CHECK();
    scb_dpre_kernel<<<dim3((unsigned)ceil_div(S.g.Go, kScbRows), B), 256, 0, st>>>(S.g, act_count, act_cap, Yact, conv_b, stats, eps, sums,
                                                                                   G, dmax64);
    MVX_LAUNCH_CHECK();
    scb_bias_kernel<<<1, kSC_Cout, 0, st>>>(S.g, B, act_count, act_cap, conv_b, stats, eps, sums, d_b, accumulate);
    MVX_LAUNCH_CHECK();
    scb_tap_gather_kernel<<<dim3((unsigned)ceil_div((long long)cap * kSC_PLd / 4, 256), B), 256, 0, st>>>(S.g, a->counts, vox_coord, cap,
                                                                                                          act_idx, G, act_cap, D, dmax64, dmax);
    MVX_LAUNCH_CHECK();
    // (b5) voxel rows of weight 1, vfeat is stored normalised (no BatchNorm on load)
    rc = launch_dw_voxel_rows(D, kSC_PLd, vfeat, kSC_Cin, a->counts, cap, dmax, dwcat, B, st);
    if (rc) return rc;
    scb_unpack_dw_kernel<<<(kSC_Cout * kSC_Cin * kSC_Taps + 255) / 256, 256, 0, st>>>(dwcat, d_w, accumulate);
    MVX_LAUNCH_CHECK();
    if (d_vfeat) {   // (b6) rows >= N_f of every frame are left as they are
        scb_pack_wb_kernel<<<(kSC_PLd * kSC_Cin + 255) / 256, 256, 0, st>>>(conv_w, Wb);
        MVX_LAUNCH_CHECK();
        LayerArgs la{};
        la.X = D, la.ldx = kSC_PLd, la.Cin = kSC_PLd, la.Wt = Wb, la.bias = nullptr, la.Cout = kSC_Cin;
        la.Y = d_vfeat, la.ldy = kSC_Cin, la.counts = a->counts, la.rows_mode = 3, la.rowcap = cap, la.vcap = cap, la.T = a->grid.T;
        la.eps = eps, la.plain = 1, la.f16_ok = 0;
        rc = launch_layer_auto(la, B, reinterpret_cast<float *>(bws + Q.wpack), st);
        if (rc) return rc;
    }
    return MVX_OK;
}
