// Stage 3 — the layer primitive of the path: relu(Linear) followed by batch-statistic BatchNorm
// (modules/layers/Blocks.py:5-18 FCN, :31-40 CRB2d with k=1), the VFE max/concat glue
// (modules/voxelnet/Pipe.py:12-18) and the final FCN + max (modules/voxelnet/VoxelNet.py:27-32).
//
// BatchNorm needs the statistics of ALL rows of a frame before any row can be normalised, so a layer is
// one launch that writes the raw post-ReLU activations and accumulates weighted per-channel sums in fp64;
// the NEXT consumer applies (y - mean) * rstd while loading.  max over T commutes with the (monotone)
// normalisation, so per-voxel maxima are taken on raw values with an integer atomicMax (y >= 0).
//
// This file holds the exact-fp32 SIMT implementation (FFMA, 128 x BN tiles). It is the parity baseline
// for the tensor-core kernels and serves the small layers, which are bandwidth- not FLOP-bound.
#include "layers.cuh"

namespace mvx {

namespace {

constexpr int kBM = 128, kBK = 16;
constexpr int kTilesPerCta = 4;   // row tiles per CTA of the SIMT layer kernel
constexpr int kAS = kBM + 4;  // padded A^T tile row (floats), keeps 16-byte alignment

__device__ __forceinline__ void norm_coef(const double *stats, double R, double eps, float &mean, float &rstd) {
    const double m = stats[0] / R;
    double var = stats[1] / R - m * m;  // biased variance (BatchNorm2d batch statistics)
    var = var < 0.0 ? 0.0 : var;
    mean = (float)m;
    rstd = (float)(1.0 / sqrt(var + eps));
}

__device__ __forceinline__ double stat_rows(const NormSrc &n, int f) {
    return n.counts ? (double)n.counts[f * 4 + 0] * (double)n.T : (double)n.rows_fixed;
}

// LD: 0 = the A tile comes from a.X (normalised with a.in_stats when given); 1 / 2 = VFE1 / VFE2 with the input rows built on the
// fly from z (what prep_vfe1_kernel / prep_vfe2_kernel below materialise as X6 / X7): Cin = 32
template <int BN, int LD = 0>
__global__ void __launch_bounds__(256, BN == 64 ? 3 : (BN == 16 ? 4 : 0)) fcn_layer_kernel(LayerArgs a, RowFuseArgs z) {
    // thread tile: RT rows x TN columns. The 16-column layers use 4 x 2 (8 x 1 needs two broadcast LDS.128 of A per 8 FFMA and is
    // bound by the shared-memory pipe: 928 wavefront cycles per tile and k chunk against 256 FFMA issue cycles)
    constexpr int TN = BN == 16 ? 2 : BN / 16;
    constexpr int RT = BN == 16 ? 4 : 8;        // rows per thread
    constexpr int TX = BN / TN;                 // threads across the columns (8 or 16); 256 / TX row groups x RT rows = 128 rows
    static_assert((256 / TX) * RT == kBM, "thread tile does not cover the CTA tile");
    // BN <= 64 (the narrow layers this kernel serves by default): the A / B tiles are double-buffered and the next k chunk travels
    // in registers while the current one is multiplied - one block barrier per chunk and no exposed global-load latency (the
    // single-buffered loop paid two barriers and one round trip per 16-k chunk). BN = 128 keeps one buffer (48 KB static limit).
    constexpr int NBUF = BN <= 64 ? 2 : 1;
    constexpr int kTileFloats = kBK * kAS + kBK * BN;
    __shared__ __align__(16) float smem[NBUF * kTileFloats];
    __shared__ float s_mean[768], s_rstd[768];
    __shared__ double s_red[2 * 8 * BN];   // [sum | sum of squares][8 warps][BN], accumulated over the tiles of this CTA
    // BatchNorm multiplicity and voxel id of the tile's rows: fetched (LD 0 / 1) or built (LD 2) at the head of the tile, so that the
    // epilogue does not start with a round trip to global memory. Two copies by tile parity: the head of tile t + 1 may run while a
    // slow warp still reads tile t's copy; tile t + 2 writes it again only behind the barriers of tile t + 1's k loop.
    __shared__ float s_roww2[2][kBM];
    __shared__ int s_rowv2[2][kBM];

    const int f = blockIdx.z, n0 = blockIdx.y * BN, tid = threadIdx.x;
    const int tx = tid % TX, ty = tid / TX;
    long long n_rows = a.rows_fixed;
    double Rstat = (double)a.rows_fixed;
    int K = 0;
    if (a.counts) {
        const int N = a.counts[f * 4 + 0];
        K = a.counts[f * 4 + 1];
        n_rows = a.rows_mode == 1 ? K + 1 : (a.rows_mode == 2 ? K + N : (a.rows_mode == 3 ? N : a.rows_fixed));
        Rstat = (double)N * (double)a.T;
    }
    // A CTA walks kTilesPerCta consecutive 128-row tiles and keeps its BatchNorm partial sums in shared memory across
    // them: the fp64 atomics of all CTAs of a frame land on 2 x Cout addresses (one or two 128-byte lines for the 16-channel
    // layers), where they serialise at about 6 ns each - with one tile per CTA that chain, not the math, bounded fcn3 / vfe1
    if ((long long)blockIdx.x * kTilesPerCta * kBM >= n_rows) return;
    for (int i = tid; i < 2 * 8 * BN; i += 256) s_red[i] = 0.0;

    if (LD != 0) {
        if (tid < 16) norm_coef(z.in_stats + ((size_t)f * 16 + tid) * 2, Rstat, a.eps, s_mean[tid], s_rstd[tid]);
    } else if (a.in_stats) {
        for (int c = tid; c < a.Cin; c += 256)
            norm_coef(a.in_stats + ((size_t)f * a.Cin + c) * 2, Rstat, a.eps, s_mean[c], s_rstd[c]);
    }
    __syncthreads();

    for (int tile = 0; tile < kTilesPerCta; ++tile) {
    float *s_roww = s_roww2[tile & 1];
    int *s_rowv = s_rowv2[tile & 1];
    const long long row0 = ((long long)blockIdx.x * kTilesPerCta + tile) * kBM;
    if (row0 >= n_rows) break;
    float acc[RT][TN];
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    const float *Xf = a.X + ((size_t)f * a.rowcap + row0) * a.ldx;
    if (tid < kBM) {   // visible to the epilogue through the barriers of the k loop (LD 2 fills the valid rows in its loader)
        const long long r = row0 + tid;
        const bool valid = r < n_rows;
        float wq = 0.f;
        int vq = -1;
        if (LD != 2 && valid) {
            wq = a.row_w ? a.row_w[(size_t)f * a.rowcap + r] : 1.f;
            if (a.vmax && wq != 0.f) {
                if (a.row_v) vq = (a.rows_mode == 1 && r >= K) ? -1 : a.row_v[(size_t)f * a.rowv_cap + r];
                else vq = (int)(r / a.T);
            }
        }
        if (LD != 2 || !valid) s_roww[tid] = wq, s_rowv[tid] = vq;
    }
    // one 16-byte piece of the A tile (row r = idx / 4, columns k0 + 4 (idx % 4) ..) as the layer reads it: normalised / built on the fly
    auto load_a = [&](int k0, int j) -> float4 {
        const int idx = tid + j * 256, r = idx >> 2, c4 = idx & 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (LD == 1) {
            // [x y z dx dy dz r | norm5(Y5) | 0 x 9]: the concat of MVXNet.py:26 (columns 23..31 are zero padding)
            if (row0 + r < n_rows) {
                const size_t ro = (size_t)f * z.capA + row0 + r;
                float e[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int k = k0 + c4 * 4 + q;
                    e[q] = k < 7 ? __ldg(z.vox8 + ro * 8 + k) : (k < 23 ? (__ldg(z.Y + ro * 16 + (k - 7)) - s_mean[k - 7]) * s_rstd[k - 7] : 0.f);
                }
                v = make_float4(e[0], e[1], e[2], e[3]);
            }
        } else if (LD == 2) {
            // rows [0, K): the kept points, voxel-major; rows [K, K + N): one pad row per voxel standing for its T - cnt empty slots
            // (value = the frame's pad row after VFE1's FCN, multiplicity T - cnt): [norm6(y) | norm6(max over the voxel)]
            const long long rr = row0 + r;
            if (rr < n_rows) {
                const bool pad = rr >= K;
                const int vv = pad ? (int)(rr - K) : __ldg(z.row_vox + (size_t)f * z.cap + rr);
                const int cnt = __ldg(z.vox_cnt + (size_t)f * z.cap + vv);
                const int c = (k0 + c4 * 4) & 15;
                const float4 yp = __ldg(reinterpret_cast<const float4 *>(z.Y + ((size_t)f * z.capA + K) * 16 + c));
                if (k0 + c4 * 4 < 16) {
                    v = pad ? yp : __ldg(reinterpret_cast<const float4 *>(z.Y + ((size_t)f * z.capA + rr) * 16 + c));
                } else {
                    const int4 mi = __ldg(reinterpret_cast<const int4 *>(z.vmax + ((size_t)f * z.cap + vv) * 16 + c));
                    v = make_float4(__int_as_float(mi.x), __int_as_float(mi.y), __int_as_float(mi.z), __int_as_float(mi.w));
                    if (cnt < a.T) v = make_float4(fmaxf(v.x, yp.x), fmaxf(v.y, yp.y), fmaxf(v.z, yp.z), fmaxf(v.w, yp.w));   // pad slots join the max over T
                }
                v.x = (v.x - s_mean[c + 0]) * s_rstd[c + 0];
                v.y = (v.y - s_mean[c + 1]) * s_rstd[c + 1];
                v.z = (v.z - s_mean[c + 2]) * s_rstd[c + 2];
                v.w = (v.w - s_mean[c + 3]) * s_rstd[c + 3];
                if (k0 == 0 && c4 == 0 && blockIdx.y == 0) {   // once per row: what the epilogue below and the last FCN read
                    const int wpad = a.T - cnt;
                    const float wq = pad ? (float)wpad : 1.f;
                    const int vq = (pad && wpad == 0) ? -1 : vv;
                    z.rowB_w[(size_t)f * a.rowcap + rr] = wq;
                    z.rowB_v[(size_t)f * a.rowcap + rr] = vq;
                    s_roww[r] = wq;
                    s_rowv[r] = wq != 0.f ? vq : -1;
                }
            }
        } else if (row0 + r < n_rows) {
            v = *reinterpret_cast<const float4 *>(Xf + (size_t)r * a.ldx + k0 + c4 * 4);
            if (a.in_stats) {
                const int k = k0 + c4 * 4;
                v.x = (v.x - s_mean[k + 0]) * s_rstd[k + 0];
                v.y = (v.y - s_mean[k + 1]) * s_rstd[k + 1];
                v.z = (v.z - s_mean[k + 2]) * s_rstd[k + 2];
                v.w = (v.w - s_mean[k + 3]) * s_rstd[k + 3];
            }
        }
        return v;
    };
    constexpr int NBP = (BN * 4 + 255) / 256;       // 16-byte pieces of the B tile (16 k x BN) per thread
    auto load_b = [&](int k0, int q) -> float4 {
        const int idx = tid + q * 256;
        if (idx >= BN * 4) return make_float4(0.f, 0.f, 0.f, 0.f);
        const int k = idx / (BN / 4), n4 = idx % (BN / 4);
        return __ldg(reinterpret_cast<const float4 *>(a.Wt + (size_t)(k0 + k) * a.Cout + n0 + n4 * 4));
    };
    auto store_tiles = [&](float *As, float *Bs, const float4 (&va)[2], const float4 (&vb)[NBP]) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {  // A tile: 128 rows x 16 k, stored transposed
            const int idx = tid + j * 256, r = idx >> 2, c4 = idx & 3;
            As[(c4 * 4 + 0) * kAS + r] = va[j].x;
            As[(c4 * 4 + 1) * kAS + r] = va[j].y;
            As[(c4 * 4 + 2) * kAS + r] = va[j].z;
            As[(c4 * 4 + 3) * kAS + r] = va[j].w;
        }
#pragma unroll
        for (int q = 0; q < NBP; ++q) {
            const int idx = tid + q * 256;
            if (idx < BN * 4) *reinterpret_cast<float4 *>(Bs + (idx / (BN / 4)) * BN + (idx % (BN / 4)) * 4) = vb[q];
        }
    };
    float4 va[2], vb[NBP];
#pragma unroll
    for (int j = 0; j < 2; ++j) va[j] = load_a(0, j);
#pragma unroll
    for (int q = 0; q < NBP; ++q) vb[q] = load_b(0, q);
    int buf = 0;
    for (int k0 = 0; k0 < a.Cin; k0 += kBK) {
        float *As = smem + buf * kTileFloats, *Bs = As + kBK * kAS;
        store_tiles(As, Bs, va, vb);
        __syncthreads();
        if (k0 + kBK < a.Cin) {   // the next chunk: in flight while this one is multiplied
#pragma unroll
            for (int j = 0; j < 2; ++j) va[j] = load_a(k0 + kBK, j);
#pragma unroll
            for (int q = 0; q < NBP; ++q) vb[q] = load_b(k0 + kBK, q);
        }
        #pragma unroll
        for (int k = 0; k < kBK; ++k) {
            float av[RT], bv[TN];
            *reinterpret_cast<float4 *>(av) = *reinterpret_cast<const float4 *>(As + k * kAS + ty * RT);
            if constexpr (RT == 8) *reinterpret_cast<float4 *>(av + 4) = *reinterpret_cast<const float4 *>(As + k * kAS + ty * RT + 4);
            if constexpr (TN == 8) {
                *reinterpret_cast<float4 *>(bv) = *reinterpret_cast<const float4 *>(Bs + k * BN + tx * 4);
                *reinterpret_cast<float4 *>(bv + 4) = *reinterpret_cast<const float4 *>(Bs + k * BN + 64 + tx * 4);
            } else if constexpr (TN == 4) {
                *reinterpret_cast<float4 *>(bv) = *reinterpret_cast<const float4 *>(Bs + k * BN + tx * 4);
            } else {
                *reinterpret_cast<float2 *>(bv) = *reinterpret_cast<const float2 *>(Bs + k * BN + tx * 2);
            }
#pragma unroll
            for (int i = 0; i < RT; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (NBUF == 1) __syncthreads();   // single buffer: everybody is done reading before the next chunk is stored
        else buf ^= 1;                     // double buffer: the barrier of the next chunk orders its stores behind these reads (two chunks back)
    }
    if (NBUF == 2) __syncthreads();        // the next tile of this CTA stores into a buffer that may still be read

    // ---- epilogue: bias, ReLU, raw store, weighted fp64 statistics, per-voxel max ------------------------
    float w[RT];
    int vox[RT];
#pragma unroll
    for (int i = 0; i < RT; ++i) {
        w[i] = s_roww[ty * RT + i];
        vox[i] = a.vmax ? s_rowv[ty * RT + i] : -1;
    }
    double *red = s_red;
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
        const int col = TN == 8 ? (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4)) : (TN == 4 ? tx * 4 + j : tx * 2 + j);
        const float b = a.plain ? 0.f : __ldg(a.bias + n0 + col);
        const float floor_v = a.plain ? -INFINITY : 0.f;
        double s = 0.0, ss = 0.0;
        int cv = -1;
        float cm = 0.f;
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const float y = fmaxf(acc[i][j] + b, floor_v);
            acc[i][j] = y;
            if (w[i] != 0.f) {
                const double yd = (double)y, wd = (double)w[i];
                s += wd * yd;
                ss += wd * yd * yd;
            }
            if (a.vmax) {
                const int v = vox[i];
                if (v != cv) {
                    if (cv >= 0) atomicMax(a.vmax + ((size_t)f * a.vcap + cv) * a.Cout + n0 + col, __float_as_int(cm));
                    cv = v;
                    cm = y;
                } else {
                    cm = fmaxf(cm, y);
                }
            }
        }
        if (a.vmax && cv >= 0) atomicMax(a.vmax + ((size_t)f * a.vcap + cv) * a.Cout + n0 + col, __float_as_int(cm));
        s += __shfl_xor_sync(0xffffffffu, s, 16);   // lanes that hold the same columns (lane % TX)
        ss += __shfl_xor_sync(0xffffffffu, ss, 16);
        if constexpr (TX == 8) {
            s += __shfl_xor_sync(0xffffffffu, s, 8);
            ss += __shfl_xor_sync(0xffffffffu, ss, 8);
        }
        if (lane < TX) {   // every (warp, column) entry has one owner thread
            red[(0 * 8 + warp) * BN + col] += s;
            red[(1 * 8 + warp) * BN + col] += ss;
        }
    }
    if (a.Y) {
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const long long r = row0 + ty * RT + i;
            if (r >= n_rows) continue;
            float *yr = a.Y + ((size_t)f * a.rowcap + r) * a.ldy + n0;
            if constexpr (TN == 8) {
                *reinterpret_cast<float4 *>(yr + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                *reinterpret_cast<float4 *>(yr + 64 + tx * 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
            } else if constexpr (TN == 4) {
                *reinterpret_cast<float4 *>(yr + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            } else {
                *reinterpret_cast<float2 *>(yr + tx * 2) = make_float2(acc[i][0], acc[i][1]);
            }
        }
    }
    }   // tiles of this CTA
    __syncthreads();
    if (tid < BN && !a.plain) {
        double s = 0.0, ss = 0.0;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) {
            s += s_red[(0 * 8 + wv) * BN + tid];
            ss += s_red[(1 * 8 + wv) * BN + tid];
        }
        double *o = a.out_stats + ((size_t)f * a.Cout + n0 + tid) * 2;
        atomicAdd(o, s);
        atomicAdd(o + 1, ss);
    }
}

// ---- dense-API helpers ---------------------------------------------------------------------------------
// y[r][0:C] = norm(y[r][0:C]) in place; optionally y[r][C:2C] = norm(vmax[r / T]) (VFE concat)
__global__ void __launch_bounds__(256) normalize_rows_kernel(float *__restrict__ y, long long R, int C, int ldy, NormSrc n,
                                                             const int *__restrict__ vmax, int T) {
    __shared__ float s_mean[768], s_rstd[768];
    const double Rs = stat_rows(n, 0);
    for (int c = threadIdx.x; c < C; c += blockDim.x) norm_coef(n.stats + (size_t)c * 2, Rs, n.eps, s_mean[c], s_rstd[c]);
    __syncthreads();
    const int c4n = C / 4;
    const long long total = R * c4n;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / c4n;
        const int c = (int)(e - r * c4n) * 4;
        float4 *p = reinterpret_cast<float4 *>(y + (size_t)r * ldy + c);
        float4 v = *p;
        v.x = (v.x - s_mean[c]) * s_rstd[c];
        v.y = (v.y - s_mean[c + 1]) * s_rstd[c + 1];
        v.z = (v.z - s_mean[c + 2]) * s_rstd[c + 2];
        v.w = (v.w - s_mean[c + 3]) * s_rstd[c + 3];
        *p = v;
        if (vmax) {
            const int4 m = *reinterpret_cast<const int4 *>(vmax + (size_t)(r / T) * C + c);
            float4 q;
            q.x = (__int_as_float(m.x) - s_mean[c]) * s_rstd[c];
            q.y = (__int_as_float(m.y) - s_mean[c + 1]) * s_rstd[c + 1];
            q.z = (__int_as_float(m.z) - s_mean[c + 2]) * s_rstd[c + 2];
            q.w = (__int_as_float(m.w) - s_mean[c + 3]) * s_rstd[c + 3];
            *reinterpret_cast<float4 *>(y + (size_t)r * ldy + C + c) = q;
        }
    }
}

// out[v][0:C] = norm(vmax[v][0:C])   (frames at stride vcap for both)
__global__ void __launch_bounds__(256) normalize_vmax_kernel(const int *__restrict__ vmax, float *__restrict__ out, int C,
                                                             int vcap, long long nvox_fixed, NormSrc n) {
    __shared__ float s_mean[768], s_rstd[768];
    const int f = blockIdx.y;
    const double Rs = stat_rows(n, f);
    for (int c = threadIdx.x; c < C; c += blockDim.x)
        norm_coef(n.stats + ((size_t)f * C + c) * 2, Rs, n.eps, s_mean[c], s_rstd[c]);
    __syncthreads();
    const long long nv = n.counts ? n.counts[f * 4 + 0] : nvox_fixed;
    const int c4n = C / 4;
    const long long total = nv * c4n;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long v = e / c4n;
        const int c = (int)(e - v * c4n) * 4;
        const int4 m = *reinterpret_cast<const int4 *>(vmax + ((size_t)f * vcap + v) * C + c);
        float4 q;
        q.x = (__int_as_float(m.x) - s_mean[c]) * s_rstd[c];
        q.y = (__int_as_float(m.y) - s_mean[c + 1]) * s_rstd[c + 1];
        q.z = (__int_as_float(m.z) - s_mean[c + 2]) * s_rstd[c + 2];
        q.w = (__int_as_float(m.w) - s_mean[c + 3]) * s_rstd[c + 3];
        *reinterpret_cast<float4 *>(out + ((size_t)f * vcap + v) * C + c) = q;
    }
}

// fused-path finalize: vfeat[v][0:128] = norm8(vmax8[v]) (voxel-major, the (N,128) result) and, through a padded
// shared-memory tile, the channel-major copy vfeat_t[c][v] that the plane-sequential grid fill reads.
__global__ void __launch_bounds__(256) finalize_vfeat_kernel(const int *__restrict__ vmax, float *__restrict__ out,
                                                             float *__restrict__ out_t, int vcap, NormSrc n) {
    constexpr int C = 128;
    __shared__ float s_mean[C], s_rstd[C];
    __shared__ float tile[C][33];
    const int f = blockIdx.y;
    const int N = n.counts[f * 4 + 0];
    const int v0 = blockIdx.x * 32;
    if (v0 >= N) return;
    if (threadIdx.x < C) norm_coef(n.stats + ((size_t)f * C + threadIdx.x) * 2, stat_rows(n, f), n.eps, s_mean[threadIdx.x], s_rstd[threadIdx.x]);
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 4; ++it) {  // 32 voxels x 32 float4 per voxel
        const int e = it * 256 + threadIdx.x, vl = e >> 5, c = (e & 31) * 4;
        if (v0 + vl < N) {
            const int4 m = *reinterpret_cast<const int4 *>(vmax + ((size_t)f * vcap + v0 + vl) * C + c);
            float4 q;
            q.x = (__int_as_float(m.x) - s_mean[c]) * s_rstd[c];
            q.y = (__int_as_float(m.y) - s_mean[c + 1]) * s_rstd[c + 1];
            q.z = (__int_as_float(m.z) - s_mean[c + 2]) * s_rstd[c + 2];
            q.w = (__int_as_float(m.w) - s_mean[c + 3]) * s_rstd[c + 3];
            *reinterpret_cast<float4 *>(out + ((size_t)f * vcap + v0 + vl) * C + c) = q;
            tile[c][vl] = q.x, tile[c + 1][vl] = q.y, tile[c + 2][vl] = q.z, tile[c + 3][vl] = q.w;
        }
    }
    if (!out_t) return;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int c = w; c < C; c += 8)
        if (v0 + lane < N) out_t[((size_t)f * C + c) * vcap + v0 + lane] = tile[c][lane];
}

// ---- fused-path glue ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) prep_vfe1_kernel(VfePrepArgs a) {
    __shared__ float s_mean[16], s_rstd[16];
    const int f = blockIdx.y;
    if (threadIdx.x < 16)
        norm_coef(a.n5.stats + ((size_t)f * 16 + threadIdx.x) * 2, stat_rows(a.n5, f), a.n5.eps, s_mean[threadIdx.x],
                  s_rstd[threadIdx.x]);
    __syncthreads();
    const int K = a.counts[f * 4 + 1];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > K) return;
    const size_t ro = (size_t)f * a.capA + r;
    const float4 v0 = *reinterpret_cast<const float4 *>(a.vox8 + ro * 8);
    const float4 v1 = *reinterpret_cast<const float4 *>(a.vox8 + ro * 8 + 4);
    float y[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<float4 *>(y + q * 4) = *reinterpret_cast<const float4 *>(a.Y5 + ro * 16 + q * 4);
#pragma unroll
    for (int c = 0; c < 16; ++c) y[c] = (y[c] - s_mean[c]) * s_rstd[c];
    // [x y z dx dy dz r | im16 | 0 x 9]  (MVXNet.py:26; Cin 23 zero-padded to 32)
    float4 *o = reinterpret_cast<float4 *>(a.X6 + ro * 32);
    o[0] = v0;
    o[1] = make_float4(v1.x, v1.y, v1.z, y[0]);
    o[2] = make_float4(y[1], y[2], y[3], y[4]);
    o[3] = make_float4(y[5], y[6], y[7], y[8]);
    o[4] = make_float4(y[9], y[10], y[11], y[12]);
    o[5] = make_float4(y[13], y[14], y[15], 0.f);
    o[6] = make_float4(0.f, 0.f, 0.f, 0.f);
    o[7] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void __launch_bounds__(256) prep_vfe2_kernel(VfePrepArgs a) {
    __shared__ float s_mean[16], s_rstd[16];
    const int f = blockIdx.y;
    if (threadIdx.x < 16)
        norm_coef(a.n6.stats + ((size_t)f * 16 + threadIdx.x) * 2, stat_rows(a.n6, f), a.n6.eps, s_mean[threadIdx.x],
                  s_rstd[threadIdx.x]);
    __syncthreads();
    const int N = a.counts[f * 4 + 0], K = a.counts[f * 4 + 1];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= K + N) return;
    const bool pad = r >= K;
    const int v = pad ? r - K : a.row_vox[(size_t)f * a.cap + r];
    const int cnt = a.vox_cnt[(size_t)f * a.cap + v];
    const float *ypad = a.Y6 + ((size_t)f * a.capA + K) * 16;            // the frame's pad row after VFE1's FCN
    const float *ysrc = pad ? ypad : a.Y6 + ((size_t)f * a.capA + r) * 16;
    const int *vm = a.vmax6 + ((size_t)f * a.cap + v) * 16;
    float o[32], ys[16], yp[16], mv[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {   // 16-byte loads: the rows are 64 bytes
        *reinterpret_cast<float4 *>(ys + q * 4) = __ldg(reinterpret_cast<const float4 *>(ysrc) + q);
        *reinterpret_cast<float4 *>(yp + q * 4) = __ldg(reinterpret_cast<const float4 *>(ypad) + q);
        *reinterpret_cast<int4 *>(mv + q * 4) = __ldg(reinterpret_cast<const int4 *>(vm) + q);
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        float m = mv[c];
        if (cnt < a.T) m = fmaxf(m, yp[c]);  // pad slots take part in the max over T (SURVEY.md trap 6)
        o[c] = (ys[c] - s_mean[c]) * s_rstd[c];
        o[16 + c] = (m - s_mean[c]) * s_rstd[c];
    }
    float4 *dst = reinterpret_cast<float4 *>(a.X7 + ((size_t)f * a.capB + r) * 32);
#pragma unroll
    for (int q = 0; q < 8; ++q) dst[q] = make_float4(o[q * 4], o[q * 4 + 1], o[q * 4 + 2], o[q * 4 + 3]);
    const int wpad = a.T - cnt;
    a.rowB_w[(size_t)f * a.capB + r] = pad ? (float)wpad : 1.f;
    a.rowB_v[(size_t)f * a.capB + r] = (pad && wpad == 0) ? -1 : v;
}

__global__ void __launch_bounds__(256) prep_fcn_kernel(VfePrepArgs a) {
    __shared__ float s_mean[64], s_rstd[64];
    const int f = blockIdx.y;
    if (threadIdx.x < 64)
        norm_coef(a.n7.stats + ((size_t)f * 64 + threadIdx.x) * 2, stat_rows(a.n7, f), a.n7.eps, s_mean[threadIdx.x],
                  s_rstd[threadIdx.x]);
    __syncthreads();
    const int N = a.counts[f * 4 + 0], K = a.counts[f * 4 + 1];
    const int r = blockIdx.x * 32 + (threadIdx.x >> 3), part = threadIdx.x & 7;  // 8 threads per row, 16 floats each
    if (r >= K + N) return;
    const int v = r >= K ? r - K : a.row_vox[(size_t)f * a.cap + r];
    const size_t ro = (size_t)f * a.capB + r;
    float *dst = a.X8 + ro * 128 + part * 16;
    if (part < 4) {
        const float *src = a.Y7 + ro * 64 + part * 16;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float4 t = *reinterpret_cast<const float4 *>(src + q * 4);
            const int c = part * 16 + q * 4;
            t.x = (t.x - s_mean[c]) * s_rstd[c];
            t.y = (t.y - s_mean[c + 1]) * s_rstd[c + 1];
            t.z = (t.z - s_mean[c + 2]) * s_rstd[c + 2];
            t.w = (t.w - s_mean[c + 3]) * s_rstd[c + 3];
            *reinterpret_cast<float4 *>(dst + q * 4) = t;
        }
    } else {
        const int *src = a.vmax7 + ((size_t)f * a.cap + v) * 64 + (part - 4) * 16;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int4 m = *reinterpret_cast<const int4 *>(src + q * 4);
            const int c = (part - 4) * 16 + q * 4;
            float4 t;
            t.x = (__int_as_float(m.x) - s_mean[c]) * s_rstd[c];
            t.y = (__int_as_float(m.y) - s_mean[c + 1]) * s_rstd[c + 1];
            t.z = (__int_as_float(m.z) - s_mean[c + 2]) * s_rstd[c + 2];
            t.w = (__int_as_float(m.w) - s_mean[c + 3]) * s_rstd[c + 3];
            *reinterpret_cast<float4 *>(dst + q * 4) = t;
        }
    }
}

}  // namespace

int launch_layer(const LayerArgs &a, int F, cudaStream_t st) {
    MVX_REQUIRE(a.Cin % 16 == 0 && a.Cin <= 768 && a.ldx % 4 == 0, MVX_EINVAL, "layer: Cin must be a multiple of 16, <= 768");
    MVX_REQUIRE(a.Cout % 16 == 0 && (a.Y == nullptr || a.ldy % 4 == 0), MVX_EINVAL, "layer: Cout must be a multiple of 16");
    const long long max_rows = a.counts ? a.rowcap : a.rows_fixed;
    if (max_rows <= 0) return MVX_OK;
    const unsigned tiles = (unsigned)ceil_div(ceil_div(max_rows, kBM), kTilesPerCta);
    if (a.Cout % 128 == 0) {
        fcn_layer_kernel<128><<<dim3(tiles, a.Cout / 128, F), 256, 0, st>>>(a, RowFuseArgs{});
    } else if (a.Cout % 64 == 0) {
        fcn_layer_kernel<64><<<dim3(tiles, a.Cout / 64, F), 256, 0, st>>>(a, RowFuseArgs{});
    } else {
        fcn_layer_kernel<16><<<dim3(tiles, a.Cout / 16, F), 256, 0, st>>>(a, RowFuseArgs{});
    }
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_vfe1_fused(const LayerArgs &a, const RowFuseArgs &z, int F, cudaStream_t st) {
    MVX_REQUIRE(a.Cin == 32 && a.Cout == 16 && a.rows_mode == 1 && a.counts && z.vox8 && z.Y && z.in_stats, MVX_EINVAL, "vfe1 fused: bad arguments");
    const unsigned tiles = (unsigned)ceil_div(ceil_div((long long)a.rowcap, kBM), kTilesPerCta);
    fcn_layer_kernel<16, 1><<<dim3(tiles, 1, F), 256, 0, st>>>(a, z);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
int launch_vfe2_fused(const LayerArgs &a, const RowFuseArgs &z, int F, cudaStream_t st) {
    MVX_REQUIRE(a.Cin == 32 && a.Cout == 64 && a.rows_mode == 2 && a.counts && z.Y && z.vmax && z.vox_cnt && z.row_vox && z.rowB_w && z.rowB_v && z.in_stats,
                MVX_EINVAL, "vfe2 fused: bad arguments");
    const unsigned tiles = (unsigned)ceil_div(ceil_div((long long)a.rowcap, kBM), kTilesPerCta);
    fcn_layer_kernel<64, 2><<<dim3(tiles, 1, F), 256, 0, st>>>(a, z);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_layer_auto(const LayerArgs &a, int F, float *wpack, cudaStream_t st) {
    if (!simt_only() && wpack) {
        if (tc_layer_eligible(a)) return launch_layer_tc(a, F, wpack, st);
    }
    return launch_layer(a, F, st);
}

int launch_prep_vfe1(const VfePrepArgs &a, cudaStream_t st) {
    prep_vfe1_kernel<<<dim3((a.cap + 1 + 255) / 256, a.B), 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
int launch_prep_vfe2(const VfePrepArgs &a, cudaStream_t st) {
    prep_vfe2_kernel<<<dim3((a.capB + 255) / 256, a.B), 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
int launch_prep_fcn(const VfePrepArgs &a, cudaStream_t st) {
    prep_fcn_kernel<<<dim3((a.capB + 31) / 32, a.B), 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
int launch_finalize_vfeat(const VfePrepArgs &a, cudaStream_t st) {
    finalize_vfeat_kernel<<<dim3((a.cap + 31) / 32, a.B), 256, 0, st>>>(a.vmax8, a.vfeat, a.vfeat_t, a.cap, a.n8);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

// ---- dense module API ------------------------------------------------------------------------------------
static size_t dense_stats_bytes(int Cout) { return ((size_t)Cout * 2 * sizeof(double) + 255) / 256 * 256; }

static int dense_layer(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias, int32_t Cout,
                       double eps, float *y, int ldy, void *ws, int *vmax, cudaStream_t st) {
    MVX_REQUIRE(x && wt && bias && ws && R > 0, MVX_EINVAL, "null pointer / empty input");
    double *stats = static_cast<double *>(ws);
    float *wpack = reinterpret_cast<float *>(static_cast<char *>(ws) + dense_stats_bytes(Cout));
    MVX_CUDA_CHECK(cudaMemsetAsync(stats, 0, (size_t)Cout * 2 * sizeof(double), st));
    if (vmax) MVX_CUDA_CHECK(cudaMemsetAsync(vmax, 0, (size_t)(R / T) * Cout * sizeof(int), st));
    LayerArgs a{};
    a.X = x, a.ldx = Cin, a.Cin = Cin, a.Wt = wt, a.bias = bias, a.Cout = Cout, a.Y = y, a.ldy = ldy;
    a.out_stats = stats, a.vmax = vmax, a.rows_mode = 0, a.rows_fixed = R, a.rowcap = 0, a.vcap = 0, a.T = T > 0 ? T : 1;
    a.eps = eps;
    a.f16_ok = dense_f16();   // arbitrary caller data: 3xTF32 unless mode 5 promises O(1) inputs
    return launch_layer_auto(a, 1, wpack, st);
}

}  // namespace mvx

extern "C" int mvx_layer_workspace_bytes(int32_t Cin, int32_t Cout, size_t *bytes) {
    if (!bytes || Cin <= 0 || Cout <= 0) return MVX_EINVAL;
    *bytes = mvx::dense_stats_bytes(Cout) + mvx::tc_wpack_bytes(Cin, Cout);
    return MVX_OK;
}

extern "C" int mvx_fcn_forward(const float *x, int64_t R, int32_t Cin, const float *wt, const float *bias, int32_t Cout,
                               double eps, float *y, void *stats_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y, MVX_EINVAL, "null output");
    int rc = mvx::dense_layer(x, R, 1, Cin, wt, bias, Cout, eps, y, Cout, stats_ws, nullptr, st);
    if (rc) return rc;
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_rows_kernel<<<mvx::kSMs * 8, 256, 0, st>>>(y, R, Cout, Cout, n, nullptr, 1);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_vfe_forward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                               int32_t Cout, double eps, float *y, void *stats_ws, void *vmax_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y && vmax_ws && T > 0 && R % T == 0, MVX_EINVAL, "bad vfe argument");
    int rc = mvx::dense_layer(x, R, T, Cin, wt, bias, Cout, eps, y, 2 * Cout, stats_ws, static_cast<int *>(vmax_ws), st);
    if (rc) return rc;
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_rows_kernel<<<mvx::kSMs * 8, 256, 0, st>>>(y, R, Cout, 2 * Cout, n, static_cast<const int *>(vmax_ws), T);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_fcn_max_forward(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                                   int32_t Cout, double eps, float *y_max, void *stats_ws, void *vmax_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y_max && vmax_ws && T > 0 && R % T == 0, MVX_EINVAL, "bad fcn_max argument");
    int rc = mvx::dense_layer(x, R, T, Cin, wt, bias, Cout, eps, nullptr, 0, stats_ws, static_cast<int *>(vmax_ws), st);
    if (rc) return rc;
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_vmax_kernel<<<dim3(mvx::kSMs * 2, 1), 256, 0, st>>>(static_cast<const int *>(vmax_ws), y_max, Cout, 0,
                                                                      R / T, n);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

// ---- training forward of the dense module API: the same launches plus the raw post-ReLU output y_raw (R, Cout) that the
// backward (module_backward.cu) needs; stats_ws keeps the fp64 sums of the layer for it. The outputs are bit-identical to the
// forward-only entries above: the same layer kernel, the same normalisation, and one extra copy (the last FCN: one extra store).
extern "C" int mvx_fcn_forward_train(const float *x, int64_t R, int32_t Cin, const float *wt, const float *bias, int32_t Cout,
                                     double eps, float *y, float *y_raw, void *stats_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y && y_raw, MVX_EINVAL, "null output");
    int rc = mvx::dense_layer(x, R, 1, Cin, wt, bias, Cout, eps, y, Cout, stats_ws, nullptr, st);
    if (rc) return rc;
    MVX_CUDA_CHECK(cudaMemcpyAsync(y_raw, y, (size_t)R * Cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_rows_kernel<<<mvx::kSMs * 8, 256, 0, st>>>(y, R, Cout, Cout, n, nullptr, 1);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_vfe_forward_train(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                                     int32_t Cout, double eps, float *y, float *y_raw, void *stats_ws, void *vmax_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y && y_raw && vmax_ws && T > 0 && R % T == 0, MVX_EINVAL, "bad vfe argument");
    int rc = mvx::dense_layer(x, R, T, Cin, wt, bias, Cout, eps, y, 2 * Cout, stats_ws, static_cast<int *>(vmax_ws), st);
    if (rc) return rc;
    MVX_CUDA_CHECK(cudaMemcpy2DAsync(y_raw, (size_t)Cout * sizeof(float), y, (size_t)2 * Cout * sizeof(float), (size_t)Cout * sizeof(float),
                                     (size_t)R, cudaMemcpyDeviceToDevice, st));
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_rows_kernel<<<mvx::kSMs * 8, 256, 0, st>>>(y, R, Cout, 2 * Cout, n, static_cast<const int *>(vmax_ws), T);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_fcn_max_forward_train(const float *x, int64_t R, int32_t T, int32_t Cin, const float *wt, const float *bias,
                                         int32_t Cout, double eps, float *y_max, float *y_raw, void *stats_ws, void *vmax_ws, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MVX_REQUIRE(y_max && y_raw && vmax_ws && T > 0 && R % T == 0, MVX_EINVAL, "bad fcn_max argument");
    int rc = mvx::dense_layer(x, R, T, Cin, wt, bias, Cout, eps, y_raw, Cout, stats_ws, static_cast<int *>(vmax_ws), st);
    if (rc) return rc;
    mvx::NormSrc n{static_cast<const double *>(stats_ws), nullptr, R, 1, eps};
    mvx::normalize_vmax_kernel<<<dim3(mvx::kSMs * 2, 1), 256, 0, st>>>(static_cast<const int *>(vmax_ws), y_max, Cout, 0,
                                                                      R / T, n);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
