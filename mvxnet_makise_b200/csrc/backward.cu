// Training-mode backward of the fusion / VFE layer stack (BASELINE.json configs[3]): the gradients of the 8 hot-path
// layers (modules/imhead/Pipe.py:84-104, modules/voxelnet/Pipe.py:5-29, modules/voxelnet/VoxelNet.py:27-32) with
// respect to their weights and biases, written into ONE flat fp32 bucket laid out like the checkpoint
// (SURVEY.md §8b: [weight (Cout,Cin) | bias (Cout)] per layer), which is what the NCCL all-reduce sums across ranks.
//
// Same compact formulation as the forward (pointpath.cu): K kept point rows plus weighted pad rows. What autograd does
// on the dense (N*T)-row tensors becomes, per layer with raw output y = relu(pre), z = (y - mean) * rstd:
//     S1 = sum_r dz,  S2 = sum_r dz * z              (dz of a weighted row is already the sum over its copies)
//     dpre = rstd * (dz - w * S1/R - w * z * S2/R) * [y > 0]        (batch-statistic BatchNorm + ReLU backward)
//     dW = dpre^T x,  db = sum_r dpre,  dx = dpre W
// and the per-voxel max routes its gradient to the FIRST row (slot order) that attains the maximum, or to the voxel's
// pad slot when that is strictly larger (torch.max's argmax on the dense tensor: real slots come before pad slots).
// tools/compact_backward_proto.py validates these formulas against autograd through the dense oracle chain.
#include "layers.cuh"
#include "pointpath.cuh"
#include "tc_common.cuh"

#include <algorithm>

namespace mvx {

namespace {

constexpr int kCinTrue[MVX_NUM_LAYERS] = {768, 768, 128, 128, 16, 23, 32, 128};

struct RowSet {            // which rows of a frame a kernel walks
    const int *counts;     // [B][4]
    int mode;              // 1: K_f + 1 rows (frame pad row last), 2: K_f + N_f rows (one pad row per voxel), 3: N_f rows (one per voxel)
    int rowcap;            // frame stride in rows
    const float *row_w;    // [B][rowcap] BatchNorm multiplicity
    int T;
};
__device__ __forceinline__ int rows_of(const RowSet &rs, int f) {
    const int N = rs.counts[f * 4 + 0], K = rs.counts[f * 4 + 1];
    return rs.mode == 1 ? K + 1 : (rs.mode == 3 ? N : K + N);
}

struct BnArgs {
    float *G;              // [B][rowcap][C]: dz in, dpre out (in place)
    const float *Y;        // [B][rowcap][C] raw layer output
    int C;
    const double *stats;   // [B][C][2] forward sums (sum w y, sum w y^2)
    double *bstats;        // [B][C][2] backward sums S1, S2
    float *dbias;          // (C) slice of the flat gradient bucket
    double eps;
    RowSet rs;
    int *dmax;             // [B][C] max |dpre| per column as float bits (zeroed by the caller), or NULL: the power-of-two
                           // column scales of the tensor-core dW; the frame pad row of mode 1 (huge multiplicity) is excluded
};

constexpr int kBnRows = 512;  // rows per CTA

// ---- S1 = sum dz, S2 = sum dz * z ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_back_reduce_kernel(BnArgs a) {
    __shared__ double s_acc[768 * 2];
    const int f = blockIdx.y, C = a.C, tpr = C / 4, tid = threadIdx.x;
    const int n_rows = rows_of(a.rs, f);
    const int row0 = blockIdx.x * kBnRows;
    if (row0 >= n_rows) return;
    for (int i = tid; i < C * 2; i += blockDim.x) s_acc[i] = 0.0;
    __syncthreads();
    const int cg = tid % tpr, rg = tid / tpr, rpp = blockDim.x / tpr;
    const int c = cg * 4;
    const double R = (double)a.rs.counts[f * 4 + 0] * (double)a.rs.T;
    // fp64 throughout: with 86 % identical pad rows a channel can be driven by a few rows at z ~ sqrt(R); then
    // dz - z * mean(dz z) cancels to O(1/R) and fp32 rounding of z is amplified by ~R (measured: the fp32 reference's own
    // autograd is 1e-2 .. 6e-2 away from its fp64 evaluation, tests/test_gpu_backward.py)
    double mean[4], rstd[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double *st = a.stats + ((size_t)f * C + c + j) * 2;
        const double m = st[0] / R;
        double var = st[1] / R - m * m;
        var = var < 0.0 ? 0.0 : var;
        mean[j] = m, rstd[j] = 1.0 / sqrt(var + a.eps);
    }
    double s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    const int rend = min(row0 + kBnRows, n_rows);
#pragma unroll 4
    for (int r = row0 + rg; r < rend; r += rpp) {   // unrolled: four rows of loads in flight per thread
        const size_t o = ((size_t)f * a.rs.rowcap + r) * C + c;
        const float4 g = *reinterpret_cast<const float4 *>(a.G + o);
        const float4 y = *reinterpret_cast<const float4 *>(a.Y + o);
        const float gv[4] = {g.x, g.y, g.z, g.w}, yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double z = ((double)yv[j] - mean[j]) * rstd[j];
            s1[j] += (double)gv[j];
            s2[j] += (double)gv[j] * z;
        }
    }
    // narrow layers put 32 / tpr lanes of a warp on the same columns: combine them with shuffles first (64 threads
    // CAS-looping on one shared fp64 address cost 0.8 ms per 16-column layer)
    for (int d = 16; d >= tpr; d >>= 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], d);
            s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], d);
        }
    }
    if (tpr >= 32 || (tid & 31) < tpr) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_acc[(c + j) * 2], s1[j]);
            atomicAdd(&s_acc[(c + j) * 2 + 1], s2[j]);
        }
    }
    __syncthreads();
    for (int i = tid; i < C * 2; i += blockDim.x) atomicAdd(a.bstats + (size_t)f * C * 2 + i, s_acc[i]);
}

// ---- dpre = rstd (dz - w S1/R - w z S2/R) [y > 0], in place; db += column sums -------------------------------
__global__ void __launch_bounds__(256) bn_back_apply_kernel(BnArgs a) {
    __shared__ double s_acc[768];
    const int f = blockIdx.y, C = a.C, tpr = C / 4, tid = threadIdx.x;
    const int n_rows = rows_of(a.rs, f);
    const int row0 = blockIdx.x * kBnRows;
    if (row0 >= n_rows) return;
    for (int i = tid; i < C; i += blockDim.x) s_acc[i] = 0.0;
    __syncthreads();
    const int cg = tid % tpr, rg = tid / tpr, rpp = blockDim.x / tpr;
    const int c = cg * 4;
    const double R = (double)a.rs.counts[f * 4 + 0] * (double)a.rs.T;
    double mean[4], rstd[4], m1[4], m2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double *st = a.stats + ((size_t)f * C + c + j) * 2;
        const double m = st[0] / R;
        double var = st[1] / R - m * m;
        var = var < 0.0 ? 0.0 : var;
        mean[j] = m, rstd[j] = 1.0 / sqrt(var + a.eps);
        const double *bs = a.bstats + ((size_t)f * C + c + j) * 2;
        m1[j] = bs[0] / R, m2[j] = bs[1] / R;
    }
    double sb[4] = {0, 0, 0, 0};
    float mx[4] = {0.f, 0.f, 0.f, 0.f};
    const int pad_row = a.rs.mode == 1 ? a.rs.counts[f * 4 + 1] : -1;
    const int rend = min(row0 + kBnRows, n_rows);
#pragma unroll 4
    for (int r = row0 + rg; r < rend; r += rpp) {
        const size_t ro = (size_t)f * a.rs.rowcap + r;
        const float w = a.rs.row_w[ro];
        float4 *gp = reinterpret_cast<float4 *>(a.G + ro * C + c);
        const float4 g = *gp;
        const float4 y = *reinterpret_cast<const float4 *>(a.Y + ro * C + c);
        const float gv[4] = {g.x, g.y, g.z, g.w}, yv[4] = {y.x, y.y, y.z, y.w};
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double z = ((double)yv[j] - mean[j]) * rstd[j];
            const double wd = (double)w;
            const float d = (float)(rstd[j] * ((double)gv[j] - wd * m1[j] - wd * z * m2[j]));
            o[j] = yv[j] > 0.f ? d : 0.f;
            sb[j] += (double)o[j];
            if (r != pad_row) mx[j] = fmaxf(mx[j], fabsf(o[j]));
        }
        *gp = make_float4(o[0], o[1], o[2], o[3]);
    }
    for (int d = 16; d >= tpr; d >>= 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            sb[j] += __shfl_xor_sync(0xffffffffu, sb[j], d);
            mx[j] = fmaxf(mx[j], __shfl_xor_sync(0xffffffffu, mx[j], d));
        }
    }
    if (tpr >= 32 || (tid & 31) < tpr) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_acc[c + j], sb[j]);
            if (a.dmax && mx[j] > 0.f) atomicMax(a.dmax + (size_t)f * C + c + j, __float_as_int(mx[j]));
        }
    }
    __syncthreads();
    for (int i = tid; i < C; i += blockDim.x) atomicAdd(a.dbias + i, (float)s_acc[i]);
}

// ---- dW += dpre^T xhat over the rows of every frame (SIMT fp32, split over row chunks, atomics into the bucket) ----
struct DwArgs {
    const float *D;        // [B][rowcap][Cout] dpre
    const float *X;        // [B][rowcap][ldx] layer input (raw producer output if in_stats, else as is)
    int ldx, Cin, CinTrue, Cout;
    const double *in_stats;  // [B][Cin][2] or NULL
    double eps;
    float *dW;             // (Cout, CinTrue) slice of the flat gradient bucket
    int chunk_rows;
    RowSet rs;
    const int *dmax;       // tensor-core path: [B][Cout] max |dpre| per column (float bits)
    const int *xmax;       // tensor-core path: [B][Cin] max |x| per column (float bits) or NULL (BatchNorm-ed input: scale 1)
};

template <int TN, int TK>
__global__ void __launch_bounds__(256) dw_gemm_kernel(DwArgs a) {
    constexpr int MN = TN / 16, MK = TK / 16;
    __shared__ __align__(16) float sD[16][TN];
    __shared__ __align__(16) float sX[16][TK];
    __shared__ float s_mean[TK], s_rstd[TK];
    const int f = blockIdx.z, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int tiles_k = a.Cin / TK;
    const int n0 = (blockIdx.x / tiles_k) * TN, k0 = (blockIdx.x % tiles_k) * TK;
    const int n_rows = rows_of(a.rs, f);
    const int row0 = blockIdx.y * a.chunk_rows;
    if (row0 >= n_rows) return;
    const int rend = min(row0 + a.chunk_rows, n_rows);
    if (a.in_stats) {
        const double R = (double)a.rs.counts[f * 4 + 0] * (double)a.rs.T;
        for (int k = tid; k < TK; k += 256) {
            const double *st = a.in_stats + ((size_t)f * a.Cin + k0 + k) * 2;
            const double m = st[0] / R;
            double var = st[1] / R - m * m;
            var = var < 0.0 ? 0.0 : var;
            s_mean[k] = (float)m, s_rstd[k] = (float)(1.0 / sqrt(var + a.eps));
        }
    }
    float acc[MN][MK];
#pragma unroll
    for (int i = 0; i < MN; ++i)
#pragma unroll
        for (int j = 0; j < MK; ++j) acc[i][j] = 0.f;
    const float *Df = a.D + (size_t)f * a.rs.rowcap * a.Cout + n0;
    const float *Xf = a.X + (size_t)f * a.rs.rowcap * a.ldx + k0;
    __syncthreads();
    for (int r0 = row0; r0 < rend; r0 += 16) {
        for (int e = tid; e < 16 * TN / 4; e += 256) {
            const int i = e / (TN / 4), c4 = (e % (TN / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + i < rend) v = *reinterpret_cast<const float4 *>(Df + (size_t)(r0 + i) * a.Cout + c4);
            *reinterpret_cast<float4 *>(&sD[i][c4]) = v;
        }
        for (int e = tid; e < 16 * TK / 4; e += 256) {
            const int i = e / (TK / 4), c4 = (e % (TK / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + i < rend) {
                v = *reinterpret_cast<const float4 *>(Xf + (size_t)(r0 + i) * a.ldx + c4);
                if (a.in_stats) {
                    v.x = (v.x - s_mean[c4]) * s_rstd[c4];
                    v.y = (v.y - s_mean[c4 + 1]) * s_rstd[c4 + 1];
                    v.z = (v.z - s_mean[c4 + 2]) * s_rstd[c4 + 2];
                    v.w = (v.w - s_mean[c4 + 3]) * s_rstd[c4 + 3];
                }
            }
            *reinterpret_cast<float4 *>(&sX[i][c4]) = v;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            float av[MN], bv[MK];
            if constexpr (MN == 8) {
                *reinterpret_cast<float4 *>(av) = *reinterpret_cast<const float4 *>(&sD[i][ty * 4]);
                *reinterpret_cast<float4 *>(av + 4) = *reinterpret_cast<const float4 *>(&sD[i][64 + ty * 4]);
            } else if constexpr (MN == 4) {
                *reinterpret_cast<float4 *>(av) = *reinterpret_cast<const float4 *>(&sD[i][ty * 4]);
            } else {
                av[0] = sD[i][ty];
            }
            if constexpr (MK == 8) {
                *reinterpret_cast<float4 *>(bv) = *reinterpret_cast<const float4 *>(&sX[i][tx * 4]);
                *reinterpret_cast<float4 *>(bv + 4) = *reinterpret_cast<const float4 *>(&sX[i][64 + tx * 4]);
            } else if constexpr (MK == 2) {
                *reinterpret_cast<float2 *>(bv) = *reinterpret_cast<const float2 *>(&sX[i][tx * 2]);
            } else {
                bv[0] = sX[i][tx];
            }
#pragma unroll
            for (int p = 0; p < MN; ++p)
#pragma unroll
                for (int q = 0; q < MK; ++q) acc[p][q] = fmaf(av[p], bv[q], acc[p][q]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int p = 0; p < MN; ++p) {
        const int n = n0 + (MN == 8 ? (p < 4 ? ty * 4 + p : 64 + ty * 4 + (p - 4)) : (MN == 4 ? ty * 4 + p : ty));
#pragma unroll
        for (int q = 0; q < MK; ++q) {
            const int k = k0 + (MK == 8 ? (q < 4 ? tx * 4 + q : 64 + tx * 4 + (q - 4)) : (MK == 2 ? tx * 2 + q : tx));
            if (k < a.CinTrue && acc[p][q] != 0.f) atomicAdd(a.dW + (size_t)n * a.CinTrue + k, acc[p][q]);
        }
    }
}

template <int TN, int TK>
int launch_dw(const DwArgs &a_in, int B, cudaStream_t st) {
    DwArgs a = a_in;
    const int tiles = (a.Cout / TN) * (a.Cin / TK);
    const int chunks = (int)std::max<long long>(1, std::min<long long>(ceil_div(a.rs.rowcap, 256), ceil_div(kSMs * 6, (long long)tiles * B)));
    a.chunk_rows = (int)round_up(ceil_div(a.rs.rowcap, chunks), 16);
    dw_gemm_kernel<TN, TK><<<dim3(tiles, (unsigned)ceil_div(a.rs.rowcap, a.chunk_rows), B), 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

// ---- dW on the tensor cores -----------------------------------------------------------------------------------------
// dW[n][k] += sum_r D[r][n] * X[r][k]: both operands are row-major with the REDUCTION index r as the slow dimension, i.e.
// "MN-major" for tcgen05. They are staged in the no-swizzle MN-major canonical layout (8 (r) x 16-byte core matrices,
// 128 contiguous bytes each): a producer lane loads 8 consecutive columns of one row (two float4), applies BatchNorm of
// the producer layer (X), scales by a per-COLUMN power of two (the sum runs over rows, so only column scales factor
// out), splits into fp16 hi/lo and writes one 16-byte core-matrix row; a warp writes 4 whole core matrices (512
// contiguous bytes) per store. One CTA owns a (MH*128) x TK tile of dW for one row chunk of one frame: MH M=128
// accumulators of TK fp32 columns in TMEM, 32 rows per pipeline stage, three products per K=16 step (3xFP16), and the
// epilogue adds acc / (scale_n * scale_k) into the flat bucket with fp32 atomics. The frame pad row of the fusion stack
// (multiplicity ~N*T) is orders of magnitude larger than ordinary rows and would eat the fp16 dynamic range of its
// columns: it is left out here and added as an exact fp32 rank-1 update by dw_pad_row_kernel.
constexpr int kDwStages = 3;
constexpr int kDwRows = 32;                 // rows (K extent) per stage = two K=16 MMA steps
constexpr int kDwProducers = 256;
constexpr int kDwThreads = kDwProducers + 32;

template <int MH, int TK>
struct DwSmem {
    static constexpr int kMT = MH * 128;
    static constexpr int kAPart = kMT * kDwRows * 2;      // bytes of the hi (or lo) image of the D tile
    static constexpr int kBPart = TK * kDwRows * 2;
    static constexpr int kStage = 2 * kAPart + 2 * kBPart;
    static constexpr int kTiles = kDwStages * kStage;
    static constexpr int kMean = kTiles;                   // [TK]
    static constexpr int kRstd = kMean + TK * 4;
    static constexpr int kDScale = kRstd + TK * 4;         // [kMT] forward scales of the D columns
    static constexpr int kXScale = kDScale + kMT * 4;      // [TK]
    static constexpr int kBars = kXScale + TK * 4;         // full[3], empty[3], accum
    static constexpr int kTmemPtr = kBars + 8 * 8;
    static constexpr int kTotal = kTmemPtr + 16 + 1024;
};

template <int MH, int TK>
__global__ void __launch_bounds__(kDwThreads, 1) dw_tc_kernel(DwArgs a) {
    using S = DwSmem<MH, TK>;
    constexpr int MT = S::kMT;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    float *s_mean = reinterpret_cast<float *>(smem + S::kMean), *s_rstd = reinterpret_cast<float *>(smem + S::kRstd);
    float *s_dscale = reinterpret_cast<float *>(smem + S::kDScale), *s_xscale = reinterpret_cast<float *>(smem + S::kXScale);
    const uint32_t bars = sbase + S::kBars;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (kDwStages + s); };
    const uint32_t accum_bar = bars + 8u * (2 * kDwStages);
    volatile uint32_t *tmem_ptr = reinterpret_cast<volatile uint32_t *>(smem + S::kTmemPtr);

    const int f = blockIdx.z, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_k = a.Cin / TK;
    const int n0 = (blockIdx.x / tiles_k) * MT, k0 = (blockIdx.x % tiles_k) * TK;
    const int n_rows = rows_of(a.rs, f);
    const int row0 = blockIdx.y * a.chunk_rows;
    if (row0 >= n_rows) return;
    const int rend = min(row0 + a.chunk_rows, n_rows);
    const int pad_row = a.rs.mode == 1 ? a.rs.counts[f * 4 + 1] : -1;   // handled by dw_pad_row_kernel
    const int nst = (rend - row0 + kDwRows - 1) / kDwRows;

    for (int k = tid; k < TK; k += kDwThreads) {
        float m = 0.f, r = 1.f;
        if (a.in_stats) {
            const double R = (double)a.rs.counts[f * 4 + 0] * (double)a.rs.T;
            const double *st = a.in_stats + ((size_t)f * a.Cin + k0 + k) * 2;
            const double mu = st[0] / R;
            double var = st[1] / R - mu * mu;
            var = var < 0.0 ? 0.0 : var;
            m = (float)mu, r = (float)(1.0 / sqrt(var + a.eps));
        }
        s_mean[k] = m, s_rstd[k] = r;
        s_xscale[k] = a.xmax ? pow2_scale(__int_as_float(a.xmax[(size_t)f * a.Cin + k0 + k])) : 1.f;
    }
    for (int n = tid; n < MT; n += kDwThreads) s_dscale[n] = pow2_scale(__int_as_float(a.dmax[(size_t)f * a.Cout + n0 + n]));
    if (tid == 0) {
        for (int s = 0; s < kDwStages; ++s) {
            mbar_init(full_bar(s), kDwProducers);
            mbar_init(empty_bar(s), 1);
        }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + S::kTmemPtr), "r"(MH * TK) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp < 8) {
        // ================= producers: granule = 8 rows x 32 columns of D or X; lane = (row lane&7, 8-column block lane>>3) ====
        constexpr int GD = 4 * (MT / 32), GX = 4 * (TK / 32), G = GD + GX, GPW = G / 8;   // granules per stage / per warp
        static_assert(G % 8 == 0, "granules must divide over the 8 producer warps");
        const int lr = lane & 7, lb = lane >> 3;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        // granule q of this warp: operand (D or X), 8-row group j, 32-column group cg
        auto geom = [&](int q, bool &isx, int &cgs, int &j, int &cg) {
            const int g = warp + 8 * q;
            isx = g >= GD;
            const int gg = isx ? g - GD : g;
            cgs = isx ? TK / 32 : MT / 32;
            j = gg / cgs, cg = gg - j * cgs;
        };
        auto load_stage = [&](float4 (&v)[GPW][2], int t) {   // all loads of a stage first (memory-level parallelism)
            const int r0 = row0 + t * kDwRows;
#pragma unroll
            for (int q = 0; q < GPW; ++q) {
                bool isx;
                int cgs, j, cg;
                geom(q, isx, cgs, j, cg);
                const int r = r0 + 8 * j + lr, col = cg * 32 + lb * 8;
                const bool ok = r < rend && r != pad_row;
                const float *src = isx ? a.X + ((size_t)f * a.rs.rowcap + r) * a.ldx + k0 + col
                                       : a.D + ((size_t)f * a.rs.rowcap + r) * a.Cout + n0 + col;
                v[q][0] = ok ? __ldg(reinterpret_cast<const float4 *>(src)) : z4;
                v[q][1] = ok ? __ldg(reinterpret_cast<const float4 *>(src) + 1) : z4;
            }
        };
        auto store_stage = [&](float4 (&v)[GPW][2], int t) {
            const int r0 = row0 + t * kDwRows;
            const int s = t % kDwStages;
            const uint32_t ph = (t / kDwStages) & 1;
            if (lane == 0) mbar_wait(empty_bar(s), ph ^ 1);
            __syncwarp();
            uint8_t *stage = smem + (size_t)s * S::kStage;
#pragma unroll
            for (int q = 0; q < GPW; ++q) {
                bool isx;
                int cgs, j, cg;
                geom(q, isx, cgs, j, cg);
                const int col = cg * 32 + lb * 8;
                const int r = r0 + 8 * j + lr;
                const bool ok = r < rend && r != pad_row;
                float x[8] = {v[q][0].x, v[q][0].y, v[q][0].z, v[q][0].w, v[q][1].x, v[q][1].y, v[q][1].z, v[q][1].w};
                const float *sc = (isx ? s_xscale : s_dscale) + col;
                if (isx && ok) {                    // BatchNorm of the producer layer (absent rows stay zero)
#pragma unroll
                    for (int e = 0; e < 8; ++e) x[e] = (x[e] - s_mean[col + e]) * s_rstd[col + e];
                }
                uint4 hi, lo;
                split_f16_pair(x[0] * sc[0], x[1] * sc[1], hi.x, lo.x);
                split_f16_pair(x[2] * sc[2], x[3] * sc[3], hi.y, lo.y);
                split_f16_pair(x[4] * sc[4], x[5] * sc[5], hi.z, lo.z);
                split_f16_pair(x[6] * sc[6], x[7] * sc[7], hi.w, lo.w);
                const uint32_t part = isx ? 2 * S::kAPart : 0, psz = isx ? S::kBPart : S::kAPart;
                const uint32_t off = part + (uint32_t)((j * cgs * 4 + cg * 4 + lb) * 128 + lr * 16);
                *reinterpret_cast<uint4 *>(stage + off) = hi;
                *reinterpret_cast<uint4 *>(stage + off + psz) = lo;
            }
            fence_async_smem();
            mbar_arrive(full_bar(s));
        };
        // the raw rows of the next stage are already in flight in registers while this stage is converted and stored
        float4 va[GPW][2], vb[GPW][2];
        load_stage(va, 0);
        for (int t = 0; t < nst; t += 2) {
            if (t + 1 < nst) load_stage(vb, t + 1);
            store_stage(va, t);
            if (t + 1 < nst) {
                if (t + 2 < nst) load_stage(va, t + 2);
                store_stage(vb, t + 1);
            }
        }
    } else if (lane == 0) {
        // ================= MMA issuer: D fp32, A/B fp16, both MN-major, M = 128, N = TK =============================
        constexpr uint32_t idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(TK >> 3) << 17) | ((128u >> 4) << 24);
        constexpr uint32_t lboA = (MT / 8) * 128, lboB = (TK / 8) * 128;
        for (int t = 0; t < nst; ++t) {
            const int s = t % kDwStages;
            const uint32_t ph = (t / kDwStages) & 1;
            mbar_wait(full_bar(s), ph);
            tc_fence_after();
            const uint32_t sA = sbase + s * S::kStage, sB = sA + 2 * S::kAPart;
#pragma unroll
            for (int h = 0; h < MH; ++h) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {   // K = 16 rows = two groups of 8
                    const uint64_t a_hi = make_desc_mn(sA + h * 16 * 128 + ks * 2 * lboA, lboA, 128);
                    const uint64_t a_lo = make_desc_mn(sA + S::kAPart + h * 16 * 128 + ks * 2 * lboA, lboA, 128);
                    const uint64_t b_hi = make_desc_mn(sB + ks * 2 * lboB, lboB, 128);
                    const uint64_t b_lo = make_desc_mn(sB + S::kBPart + ks * 2 * lboB, lboB, 128);
                    const uint32_t d = tmem_base + h * TK;
                    mma_f16(d, a_lo, b_hi, idesc, (t | ks) != 0);
                    mma_f16(d, a_hi, b_lo, idesc, 1);
                    mma_f16(d, a_hi, b_hi, idesc, 1);
                }
            }
            mma_commit(empty_bar(s));
        }
        mma_commit(accum_bar);
    }

    // ================= epilogue: TMEM -> unscale -> fp32 atomics into the flat bucket ===================================
    __syncwarp();
    if (warp < 4 * MH) {
        mbar_wait(accum_bar, 0);
        tc_fence_after();
        const int h = warp >> 2, q = warp & 3;
        const int n = h * 128 + q * 32 + lane;           // accumulator row = output channel
        const float dinv = 1.f / s_dscale[n];
        float *orow = a.dW + (size_t)(n0 + n) * a.CinTrue + k0;
#pragma unroll 1
        for (int cb = 0; cb < TK / 32; ++cb) {
            float v[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + h * TK + cb * 32, v);
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const int k = cb * 32 + e;
                const float g = v[e] * dinv / s_xscale[k];
                if (k0 + k < a.CinTrue && g != 0.f) atomicAdd(orow + k, g);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(MH * TK) : "memory");
}

// the frame pad row of a mode-1 layer, exact fp32: dW[n][k] += D[K][n] * xhat[K][k]
__global__ void __launch_bounds__(256) dw_pad_row_kernel(DwArgs a) {
    const int f = blockIdx.y, n = blockIdx.x, K = a.rs.counts[f * 4 + 1];
    const float d = a.D[((size_t)f * a.rs.rowcap + K) * a.Cout + n];
    if (d == 0.f) return;
    const double R = (double)a.rs.counts[f * 4 + 0] * (double)a.rs.T;
    for (int k = threadIdx.x; k < a.CinTrue; k += blockDim.x) {
        float x = a.X[((size_t)f * a.rs.rowcap + K) * a.ldx + k];
        if (a.in_stats) {
            const double *st = a.in_stats + ((size_t)f * a.Cin + k) * 2;
            const double mu = st[0] / R;
            double var = st[1] / R - mu * mu;
            var = var < 0.0 ? 0.0 : var;
            x = (x - (float)mu) * (float)(1.0 / sqrt(var + a.eps));
        }
        const float g = d * x;
        if (g != 0.f) atomicAdd(a.dW + (size_t)n * a.CinTrue + k, g);
    }
}

template <int MH, int TK>
int launch_dw_tc(const DwArgs &a_in, int B, cudaStream_t st) {
    using S = DwSmem<MH, TK>;
    static bool attr_set = false;
    if (!attr_set) {
        MVX_CUDA_CHECK(cudaFuncSetAttribute(dw_tc_kernel<MH, TK>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
        attr_set = true;
    }
    DwArgs a = a_in;
    const int tiles = (a.Cout / (MH * 128)) * (a.Cin / TK);
    const long long per = (long long)tiles * B;
    const int chunks = (int)std::max<long long>(1, std::min<long long>(ceil_div(a.rs.rowcap, 2048), (kSMs + per / 2) / per));
    a.chunk_rows = (int)round_up(ceil_div(a.rs.rowcap, chunks), kDwRows);
    dw_tc_kernel<MH, TK><<<dim3(tiles, (unsigned)ceil_div(a.rs.rowcap, a.chunk_rows), B), kDwThreads, S::kTotal, st>>>(a);
    MVX_LAUNCH_CHECK();
    if (a.rs.mode == 1) {
        dw_pad_row_kernel<<<dim3(a.Cout, B), 256, 0, st>>>(a);
        MVX_LAUNCH_CHECK();
    }
    return MVX_OK;
}

static int g_dw_tc = 1;   // 1: tensor-core dW where eligible, 0: SIMT everywhere (mvx_set_gemm_mode(0) also selects SIMT)

int launch_dw_auto(const DwArgs &a, int B, cudaStream_t st) {
    if (g_dw_tc && gemm_mode() == 1 && a.dmax && a.Cout % 128 == 0 && a.Cin % 128 == 0) {
        if (a.Cout % 256 == 0 && a.Cin % 256 == 0) return launch_dw_tc<2, 256>(a, B, st);
        if (a.Cin % 256 == 0) return launch_dw_tc<1, 256>(a, B, st);
        return launch_dw_tc<1, 128>(a, B, st);
    }
    if (a.Cout % 128 == 0 && a.Cin % 128 == 0) return launch_dw<128, 128>(a, B, st);
    if (a.Cout == 64 && a.Cin == 32) return launch_dw<64, 32>(a, B, st);
    if (a.Cout == 16 && a.Cin % 128 == 0) return launch_dw<16, 128>(a, B, st);
    if (a.Cout == 16 && a.Cin == 32) return launch_dw<16, 32>(a, B, st);
    if (a.Cout == 16 && a.Cin == 16) return launch_dw<16, 16>(a, B, st);
    set_error("dw_gemm: unsupported layer shape %d x %d", a.Cout, a.Cin);
    return MVX_EINVAL;
}

}  // namespace

int launch_dw_voxel_rows(const float *D, int Cout, const float *X, int Cin, const int *counts, int rowcap, const int *dmax, float *dW, int B,
                         cudaStream_t st, const int *xmax) {
    const DwArgs dw{D, X, Cin, Cin, Cin, Cout, nullptr, 0.0, dW, 0, RowSet{counts, 3, rowcap, nullptr, 1}, dmax, xmax};
    return launch_dw_auto(dw, B, st);
}

int launch_bn_back_voxel_rows(float *G, const float *Y, int C, const double *stats, double *bstats, float *dbias, double eps, const int *counts,
                              int rowcap, const float *row_w, int *dmax, cudaStream_t st) {
    MVX_REQUIRE(C == 768 || (C % 4 == 0 && C <= 512 && 256 % (C / 4) == 0), MVX_EINVAL,
                "BatchNorm backward: C must be 768 or a multiple of 4 whose quarter divides 256");
    const BnArgs bn{G, Y, C, stats, bstats, dbias, eps, RowSet{counts, 3, rowcap, row_w, 1}, dmax};
    const int threads = C == 768 ? 192 : 256;
    const dim3 grid((unsigned)ceil_div(rowcap, kBnRows), 1);
    bn_back_reduce_kernel<<<grid, threads, 0, st>>>(bn);
    MVX_LAUNCH_CHECK();
    bn_back_apply_kernel<<<grid, threads, 0, st>>>(bn);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

namespace {

// ---- W (Cout, CinPad) row-major from the stored W^T (CinPad, Cout) -------------------------------------------
__global__ void __launch_bounds__(256) transpose_w_kernel(const float *__restrict__ wt, float *__restrict__ w, int Cin, int Cout) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= Cin * Cout) return;
    const int n = e / Cin, k = e - n * Cin;
    w[e] = wt[(size_t)k * Cout + n];
}

// ---- per-voxel max backward (+ the concat split of the VFE layers) --------------------------------------------
// One thread per (voxel, channel). Y: raw outputs of the layer whose max is taken; real rows of voxel v are
// row0[v] .. row0[v]+cnt[v]-1, its pad slot is row K_f + v (kSharedPad: the frame's single pad row K_f).
// dXn: gradient w.r.t. the NEXT layer's input [pointwise C | per-voxel max C] in (K_f + N_f)-row indexing, or, for the
// last layer (kFinal), dOut[v][c] = dLoss/d vfeat.  G: dz of this layer.
struct MaxBackArgs {
    const int *counts, *vox_cnt, *vox_row0;
    int cap, T;
    const float *Y;
    int y_rowcap;
    const float *dXn;      // [B][capB][2C]   (kFinal: NULL)
    int capB;
    const float *dOut;     // [B][cap][C]     (kFinal only)
    float *G;              // [B][g_rowcap][C]
    int g_rowcap;
};

template <int C, bool kSharedPad, bool kFinal>
__global__ void __launch_bounds__(256) max_back_kernel(MaxBackArgs a) {
    constexpr int VPB = 256 / C;   // voxels per CTA
    __shared__ float s_pad[256];
    const int f = blockIdx.y, tid = threadIdx.x, c = tid % C;
    const int N = a.counts[f * 4 + 0], K = a.counts[f * 4 + 1];
    const int v = blockIdx.x * VPB + tid / C;
    float pad_grad = 0.f;
    if (v < N) {
        const int row0 = a.vox_row0[(size_t)f * (a.cap + 1) + v], cnt = a.vox_cnt[(size_t)f * a.cap + v];
        const float *Yf = a.Y + (size_t)f * a.y_rowcap * C + c;
        const float *Xf = kFinal ? nullptr : a.dXn + (size_t)f * a.capB * (2 * C) + c;
        float *Gf = a.G + (size_t)f * a.g_rowcap * C + c;
        float mreal = -INFINITY, dM = kFinal ? a.dOut[((size_t)f * a.cap + v) * C + c] : 0.f;
        int arg = -1;
        for (int i = 0; i < cnt; ++i) {
            const int r = row0 + i;
            const float y = Yf[(size_t)r * C];
            if (y > mreal) mreal = y, arg = r;   // strict: the first row attaining the maximum wins
            if (!kFinal) dM += Xf[(size_t)r * (2 * C) + C];
        }
        const int rp = K + v;                    // pad slot of this voxel in (K + N)-row indexing
        if (!kFinal) dM += Xf[(size_t)rp * (2 * C) + C];
        const float ypad = Yf[(size_t)(kSharedPad ? K : rp) * C];
        const bool pad_wins = cnt < a.T && ypad > mreal;
        for (int i = 0; i < cnt; ++i) {
            const int r = row0 + i;
            const float g = kFinal ? 0.f : Xf[(size_t)r * (2 * C)];
            Gf[(size_t)r * C] = g + ((!pad_wins && r == arg) ? dM : 0.f);
        }
        const float gp = (kFinal ? 0.f : Xf[(size_t)rp * (2 * C)]) + (pad_wins ? dM : 0.f);
        if (kSharedPad) pad_grad = gp; else Gf[(size_t)rp * C] = gp;
    }
    if (kSharedPad) {   // every voxel's pad slot is the frame's single pad row: block-reduce, then one atomic per channel
        s_pad[tid] = pad_grad;
        __syncthreads();
        if (tid < C) {
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < VPB; ++q) s += s_pad[q * C + tid];
            if (s != 0.f) atomicAdd(a.G + ((size_t)f * a.g_rowcap + K) * C + tid, s);
        }
    }
}

// zero the frame pad row K_f of a (B, rowcap, C) gradient buffer before the shared-pad accumulation
__global__ void zero_pad_row_kernel(float *G, const int *counts, int rowcap, int C) {
    const int f = blockIdx.x, K = counts[f * 4 + 1];
    for (int c = threadIdx.x; c < C; c += blockDim.x) G[((size_t)f * rowcap + K) * C + c] = 0.f;
}

// G5[r][0:16] = dX6[r][7:23]  (the image-feature columns of VFE1's input, MVXNet.py:26)
__global__ void __launch_bounds__(256) slice_im16_kernel(const float *__restrict__ dX6, float *__restrict__ G5, const int *counts, int capA) {
    const int f = blockIdx.y, K = counts[f * 4 + 1];
    const int e = blockIdx.x * blockDim.x + threadIdx.x, r = e >> 4, c = e & 15;
    if (r > K) return;
    G5[((size_t)f * capA + r) * 16 + c] = dX6[((size_t)f * capA + r) * 32 + 7 + c];
}

// d vfeat[f][v][c] = d grid[f][c][cell(v)]   (backward of VoxelNet.reindex, VoxelNet.py:16-22: an index select)
__global__ void __launch_bounds__(256) grid_grad_gather_kernel(const float *__restrict__ dgrid, const int *__restrict__ vox_coord,
                                                               const int *counts, int cap, long long G, float *__restrict__ dv) {
    const int f = blockIdx.y, N = counts[f * 4 + 0];
    const int e = blockIdx.x * blockDim.x + threadIdx.x, v = e >> 7, c = e & 127;
    if (v >= N) return;
    const int cell = vox_coord[((size_t)f * cap + v) * 4 + 3];
    dv[((size_t)f * cap + v) * 128 + c] = dgrid[((size_t)f * 128 + c) * G + cell];
}

enum BRegion { BR_G1 = 0, BR_G2, BR_G3, BR_G4, BR_G5, BR_DX6, BR_G6, BR_DX7, BR_G7, BR_DX8, BR_G8, BR_BSTATS, BR_WT, BR_DVFEAT, BR_DMAX, BR_COUNT };

struct BLayout {
    size_t off[BR_COUNT];
    size_t wt_off[MVX_NUM_LAYERS];   // floats inside BR_WT
    size_t total;
};

void make_blayout(const mvx_pointpath_args_t *a, const Layout &L, BLayout &BL) {
    const size_t B = a->B, capA = L.capA, capB = L.capB, cap = a->cap;
    size_t o = 0;
    auto take = [&](BRegion r, size_t bytes) {
        BL.off[r] = o;
        o += (bytes + 255) / 256 * 256;
    };
    take(BR_G1, B * capA * 768 * 4);
    take(BR_G2, B * capA * 128 * 4);
    take(BR_G3, B * capA * 128 * 4);
    take(BR_G4, B * capA * 16 * 4);
    take(BR_G5, B * capA * 16 * 4);
    take(BR_DX6, B * capA * 32 * 4);
    take(BR_G6, B * capA * 16 * 4);
    take(BR_DX7, B * capB * 32 * 4);
    take(BR_G7, B * capB * 64 * 4);
    take(BR_DX8, B * capB * 128 * 4);
    take(BR_G8, B * capB * 128 * 4);
    take(BR_BSTATS, (size_t)MVX_NUM_LAYERS * B * kStatStride * 8);
    size_t w = 0;
    for (int l = 0; l < MVX_NUM_LAYERS; ++l) {
        BL.wt_off[l] = w;
        w += (size_t)kCin[l] * kCout[l];
    }
    take(BR_WT, w * 4);
    take(BR_DVFEAT, B * cap * 128 * 4);
    take(BR_DMAX, (size_t)MVX_NUM_LAYERS * B * 768 * 4);
    BL.total = o;
}

}  // namespace

void backward_ws_layout(const mvx_pointpath_args_t *a, const Layout &L, size_t *total, size_t *dpre1_off) {
    BLayout BL;
    make_blayout(a, L, BL);
    *total = BL.total;
    *dpre1_off = BL.off[BR_G1];
}

int launch_transpose_w(const float *wt, float *w, int Cin, int Cout, cudaStream_t st) {
    const int n = Cin * Cout;
    transpose_w_kernel<<<(n + 255) / 256, 256, 0, st>>>(wt, w, Cin, Cout);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

size_t grad_floats() {
    size_t n = 0;
    for (int l = 0; l < MVX_NUM_LAYERS; ++l) n += (size_t)kCout[l] * kCinTrue[l] + kCout[l];
    return n;
}

int pointpath_backward(const mvx_pointpath_args_t *a, const float *d_vfeat, const float *d_grid, float *grad_flat, int accumulate,
                       void *bws_v, size_t bws_bytes) {
    Layout L;
    int rc = make_layout(a, L);
    if (rc) return rc;
    BLayout BL;
    make_blayout(a, L, BL);
    MVX_REQUIRE(a->workspace && a->workspace_bytes >= L.total_train, MVX_ESPACE, "backward needs the training workspace of the forward");
    MVX_REQUIRE(bws_v && bws_bytes >= BL.total, MVX_ESPACE, "backward workspace too small");
    MVX_REQUIRE((d_vfeat != nullptr) != (d_grid != nullptr), MVX_EINVAL, "give exactly one of d_vfeat / d_grid");
    MVX_REQUIRE(grad_flat && a->counts, MVX_EINVAL, "null pointer");
    for (int l = 0; l < MVX_NUM_LAYERS; ++l) MVX_REQUIRE(a->wt[l], MVX_EINVAL, "null layer weights");
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    char *ws = static_cast<char *>(a->workspace), *bws = static_cast<char *>(bws_v);
    const int B = a->B, cap = a->cap, T = a->grid.T;
    auto F32 = [&](Region r) { return reinterpret_cast<float *>(ws + L.off[r]); };
    auto I32 = [&](Region r) { return reinterpret_cast<int *>(ws + L.off[r]); };
    auto BF = [&](BRegion r) { return reinterpret_cast<float *>(bws + BL.off[r]); };
    double *stats = reinterpret_cast<double *>(ws + L.off[R_STATS]);
    double *bstats = reinterpret_cast<double *>(bws + BL.off[BR_BSTATS]);
    auto stat_of = [&](int l) { return stats + (size_t)l * B * kStatStride; };
    auto bstat_of = [&](int l) { return bstats + (size_t)l * B * kStatStride; };

    // flat bucket offsets: [weight (Cout, CinTrue) | bias (Cout)] per layer, checkpoint order
    size_t w_off[MVX_NUM_LAYERS], b_off[MVX_NUM_LAYERS], o = 0;
    for (int l = 0; l < MVX_NUM_LAYERS; ++l) {
        w_off[l] = o, o += (size_t)kCout[l] * kCinTrue[l];
        b_off[l] = o, o += kCout[l];
    }
    if (!accumulate) MVX_CUDA_CHECK(cudaMemsetAsync(grad_flat, 0, o * sizeof(float), st));
    MVX_CUDA_CHECK(cudaMemsetAsync(bstats, 0, (size_t)MVX_NUM_LAYERS * B * kStatStride * 8, st));
    int *dmax = reinterpret_cast<int *>(bws + BL.off[BR_DMAX]);
    MVX_CUDA_CHECK(cudaMemsetAsync(dmax, 0, (size_t)MVX_NUM_LAYERS * B * 768 * 4, st));
    auto dmax_of = [&](int l) { return dmax + (size_t)l * B * 768; };   // [B][Cout_l] inside
    float *wT = BF(BR_WT);
    for (int l = 1; l < MVX_NUM_LAYERS; ++l) {   // fcn1 needs no dx here: the map gradient is pixel-first (map_backward.cu)
        const int n = kCin[l] * kCout[l];
        transpose_w_kernel<<<(n + 255) / 256, 256, 0, st>>>(a->wt[l], wT + BL.wt_off[l], kCin[l], kCout[l]);
        MVX_LAUNCH_CHECK();
    }
    if (d_grid) {
        grid_grad_gather_kernel<<<dim3((unsigned)ceil_div((long long)cap * 128, 256), B), 256, 0, st>>>(d_grid, I32(R_VOX_COORD), a->counts, cap,
                                                                                                         L.G, BF(BR_DVFEAT));
        MVX_LAUNCH_CHECK();
        d_vfeat = BF(BR_DVFEAT);
    }
    const RowSet rsA{a->counts, 1, L.capA, F32(R_ROWA_W), T}, rsB{a->counts, 2, L.capB, F32(R_ROWB_W), T};

    // one layer: S1/S2, dpre (in place) + db, dW, and (optionally) dx = dpre W into dX
    auto layer_back = [&](int l, float *G, const float *Y, const RowSet &rs, const float *X, int ldx, const double *in_stats,
                          float *dX) -> int {
        const int C = kCout[l];
        BnArgs bn{G, Y, C, stat_of(l), bstat_of(l), grad_flat + b_off[l], a->bn_eps, rs, dmax_of(l)};
        const int threads = C == 768 ? 192 : 256;
        const dim3 grid((unsigned)ceil_div(rs.rowcap, kBnRows), B);
        bn_back_reduce_kernel<<<grid, threads, 0, st>>>(bn);
        MVX_LAUNCH_CHECK();
        bn_back_apply_kernel<<<grid, threads, 0, st>>>(bn);
        MVX_LAUNCH_CHECK();
        // column maxima for the fp16 scaling of the tensor-core dW: dpre from bn_back_apply; X is BatchNorm-ed (scale 1)
        // except fcn1's gathered features, bounded per column by the channel maxima of the FPN maps (convex combination)
        DwArgs dw{G, X, ldx, kCin[l], kCinTrue[l], C, in_stats, a->bn_eps, grad_flat + w_off[l], 0, rs, dmax_of(l),
                  l == 0 ? I32(R_CHMAX) : nullptr};
        int r = launch_dw_auto(dw, B, st);
        if (r) return r;
        if (dX) {
            LayerArgs la{};
            la.X = G, la.ldx = C, la.Cin = C, la.Wt = wT + BL.wt_off[l], la.bias = nullptr, la.Cout = kCin[l];
            la.Y = dX, la.ldy = kCin[l], la.counts = a->counts, la.rows_mode = rs.mode, la.rowcap = rs.rowcap, la.vcap = cap;
            la.T = T, la.eps = a->bn_eps, la.plain = 1;
            r = launch_layer_auto(la, B, F32(R_WPACK), st);
            if (r) return r;
        }
        return MVX_OK;
    };

    MaxBackArgs mb{};
    mb.counts = a->counts, mb.vox_cnt = I32(R_VOX_CNT), mb.vox_row0 = I32(R_VOX_ROW0), mb.cap = cap, mb.T = T, mb.capB = L.capB;
    // ---- FCN (128 -> 128) + max over T ------------------------------------------------------------------------------
    mb.Y = F32(R_Y8), mb.y_rowcap = L.capB, mb.dXn = nullptr, mb.dOut = d_vfeat, mb.G = BF(BR_G8), mb.g_rowcap = L.capB;
    max_back_kernel<128, false, true><<<dim3((unsigned)ceil_div(cap, 2), B), 256, 0, st>>>(mb);
    MVX_LAUNCH_CHECK();
    rc = layer_back(7, BF(BR_G8), F32(R_Y8), rsB, F32(R_X8), 128, nullptr, BF(BR_DX8));
    if (rc) return rc;
    // ---- VFE2 (32 -> 64): X8 = [z7 | max z7] ------------------------------------------------------------------------
    mb.Y = F32(R_Y7), mb.y_rowcap = L.capB, mb.dXn = BF(BR_DX8), mb.dOut = nullptr, mb.G = BF(BR_G7), mb.g_rowcap = L.capB;
    max_back_kernel<64, false, false><<<dim3((unsigned)ceil_div(cap, 4), B), 256, 0, st>>>(mb);
    MVX_LAUNCH_CHECK();
    rc = layer_back(6, BF(BR_G7), F32(R_Y7), rsB, F32(R_X7), 32, nullptr, BF(BR_DX7));
    if (rc) return rc;
    // ---- VFE1 (23 -> 16): X7 = [z6 | max z6], every pad slot is the frame's pad row ---------------------------------
    zero_pad_row_kernel<<<B, 32, 0, st>>>(BF(BR_G6), a->counts, L.capA, 16);
    MVX_LAUNCH_CHECK();
    mb.Y = F32(R_Y6), mb.y_rowcap = L.capA, mb.dXn = BF(BR_DX7), mb.G = BF(BR_G6), mb.g_rowcap = L.capA;
    max_back_kernel<16, true, false><<<dim3((unsigned)ceil_div(cap, 16), B), 256, 0, st>>>(mb);
    MVX_LAUNCH_CHECK();
    rc = layer_back(5, BF(BR_G6), F32(R_Y6), rsA, F32(R_X6), 32, nullptr, BF(BR_DX6));
    if (rc) return rc;
    slice_im16_kernel<<<dim3((unsigned)ceil_div((long long)L.capA * 16, 256), B), 256, 0, st>>>(BF(BR_DX6), BF(BR_G5), a->counts, L.capA);
    MVX_LAUNCH_CHECK();
    // ---- fusion stack, last to first: fcn3 conv2 fcn2 conv1 fcn1 ----------------------------------------------------
    rc = layer_back(4, BF(BR_G5), F32(R_Y5), rsA, F32(R_Y4), 16, stat_of(3), BF(BR_G4));
    if (rc) return rc;
    rc = layer_back(3, BF(BR_G4), F32(R_Y4), rsA, F32(R_Y3), 128, stat_of(2), BF(BR_G3));
    if (rc) return rc;
    rc = layer_back(2, BF(BR_G3), F32(R_Y3), rsA, F32(R_Y2), 128, stat_of(1), BF(BR_G2));
    if (rc) return rc;
    rc = layer_back(1, BF(BR_G2), F32(R_Y2), rsA, F32(R_Y1), 768, stat_of(0), BF(BR_G1));
    if (rc) return rc;
    rc = layer_back(0, BF(BR_G1), F32(R_Y1), rsA, F32(R_A1), 768, nullptr, nullptr);
    return rc;
}

}  // namespace mvx

extern "C" int mvx_pointpath_train_workspace_bytes(const mvx_pointpath_args_t *args, size_t *forward_bytes, size_t *backward_bytes) {
    mvx::Layout L;
    int rc = mvx::make_layout(args, L);
    if (rc) return rc;
    if (!forward_bytes || !backward_bytes) return MVX_EINVAL;
    mvx::BLayout BL;
    mvx::make_blayout(args, L, BL);
    *forward_bytes = L.total_train;
    *backward_bytes = BL.total;
    return MVX_OK;
}

extern "C" int mvx_pointpath_forward_train(const mvx_pointpath_args_t *args) { return mvx::pointpath_forward(args, true); }

extern "C" int64_t mvx_grad_floats(void) { return (int64_t)mvx::grad_floats(); }

extern "C" int mvx_pointpath_backward(const mvx_pointpath_args_t *args, const float *d_vfeat, const float *d_grid, float *grad_flat,
                                      int32_t accumulate, void *backward_ws, size_t backward_ws_bytes) {
    return mvx::pointpath_backward(args, d_vfeat, d_grid, grad_flat, accumulate, backward_ws, backward_ws_bytes);
}
