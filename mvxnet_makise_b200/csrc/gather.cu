// Stage 2 — calibrated projection (modules/utils/Calib.py:47-70) and the PointFusion gather
// (modules/imhead/Pipe.py:23-82).  The FPN maps are re-laid out channels-last once per call so that every
// corner read is a contiguous, coalesced run of channels (NCHW would cost one 32-byte sector per channel).
#include "gather.cuh"

#include <cuda_bf16.h>
#include "project.cuh"

#include <climits>
#include <cuda_fp16.h>

namespace mvx {

namespace {

// ---- NCHW -> NHWC ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float *__restrict__ in, float *__restrict__ out, int C,
                                                           int HW, int *__restrict__ rowmax, int *__restrict__ chmax, int chmax_stride) {
    __shared__ float tile[32][33];
    const size_t fb = (size_t)blockIdx.z * C * HW;
    const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + ty + k * 8, p = p0 + tx;
        tile[ty + k * 8][tx] = (c < C && p < HW) ? __ldg(in + fb + (size_t)c * HW + p) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int p = p0 + ty + k * 8, c = c0 + tx;
        if (c < C && p < HW) out[fb + (size_t)p * C + c] = tile[tx][ty + k * 8];
    }
    if (rowmax && threadIdx.x < 32 && p0 + tx < HW) {   // max |x| of each pixel row (as float bits), for the fp16 row scaling of the pixel GEMM
        float m = 0.f;
#pragma unroll
        for (int c = 0; c < 32; ++c) m = fmaxf(m, fabsf(tile[c][tx]));
        atomicMax(rowmax + (size_t)blockIdx.z * HW + p0 + tx, __float_as_int(m));
    }
    if (chmax && threadIdx.x >= 32 && threadIdx.x < 64 && c0 + tx < C) {   // max |x| of each channel over the frame (training:
        float m = 0.f;                                                      // column bound of the gathered matrix for the dW scaling)
        for (int p = 0; p < 32; ++p) m = fmaxf(m, fabsf(tile[tx][p]));     // pixels beyond HW were loaded as 0
        atomicMax(chmax + (size_t)blockIdx.z * chmax_stride + c0 + tx, __float_as_int(m));
    }
}

__global__ void __launch_bounds__(256) lidar2img_f64_kernel(const float *__restrict__ pts, int stride, long long P,
                                                            const double *__restrict__ calib64, double *__restrict__ out_uv) {
    __shared__ double c64[32];
    if (threadIdx.x < 32) c64[threadIdx.x] = calib64[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float *q = pts + (size_t)i * stride;
    double u, v, cz;
    project_point_z_f64(c64, q[0], q[1], q[2], u, v, cz);
    reinterpret_cast<double2 *>(out_uv)[i] = make_double2(u, v);
}

__global__ void __launch_bounds__(256) lidar2img_kernel(const float *__restrict__ pts, int stride, long long P,
                                                        const float *__restrict__ calib32, float *__restrict__ out_uv) {
    __shared__ float c32[32];
    if (threadIdx.x < 32) c32[threadIdx.x] = calib32[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float *q = pts + (size_t)i * stride;
    float u, v;
    project_point(c32, q[0], q[1], q[2], u, v);
    reinterpret_cast<float2 *>(out_uv)[i] = make_float2(u, v);
}

// ---- NCHW fp32 maps -> pre-packed fp16 hi/lo A operand of the pixel GEMM -------------------------------------------------
// Row R = f * HW + p of the GEMM is pixel p of frame f. Per (256-row tile, 32-channel chunk) the output holds the exact
// shared-memory image of the tensor-core kernel: [hi: 256 rows x 64 B, SWIZZLE_64B | lo: same], so the GEMM fetches a
// stage of A with ONE bulk copy and has no register producers. A CTA owns 32 pixels x all C = 256 channels, finds each
// pixel's max |x| (power-of-two scale into [0.5,1)), splits and stores; rowinv[R] = 1 / scale.
__device__ __forceinline__ uint32_t pk_half2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
__device__ __forceinline__ void pk_split(float x0, float x1, uint32_t &hi, uint32_t &lo) {
    hi = pk_half2(x0, x1);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2 *>(&hi));
    lo = pk_half2(x0 - hf.x, x1 - hf.y);
}
#ifndef MVX_PACK_UNROLL
#define MVX_PACK_UNROLL 16
#endif
constexpr int kPackUnroll = MVX_PACK_UNROLL;   // channel rows in flight per thread (A/B on the serialised stage: 4: 0.147-0.167 ms, 8: 0.181, 16: 0.133-0.147, 32: 0.167)
__global__ void __launch_bounds__(256) pack_maps_f16_kernel(const float *__restrict__ in, int C, int HW, uint8_t *__restrict__ apack,
                                                            float *__restrict__ rowinv) {
    __shared__ float tile[256][33];
    __shared__ float s_max[8][32];
    __shared__ float s_scale[32];
    const int f = blockIdx.y, p0 = blockIdx.x * 32, tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const float *src = in + (size_t)f * C * HW;
    float mx = 0.f;
#pragma unroll kPackUnroll
    for (int k = 0; k < 32; ++k) {
        const int c = ty + 8 * k;
        const float v = (p0 + tx < HW) ? __ldg(src + (size_t)c * HW + p0 + tx) : 0.f;
        tile[c][tx] = v;
        mx = fmaxf(mx, fabsf(v));
    }
    s_max[ty][tx] = mx;
    __syncthreads();
    if (tid < 32) {
        float m = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) m = fmaxf(m, s_max[q][tid]);
        float sc = 1.f;
        if (m > 0.f && isfinite(m)) {
            int e;
            frexpf(m, &e);
            e = max(-100, min(100, e));
            sc = exp2f((float)-e);
        }
        s_scale[tid] = sc;
        if (p0 + tid < HW) rowinv[(size_t)f * HW + p0 + tid] = 1.f / sc;
    }
    __syncthreads();
    const int nkc = C / 32;
    for (int q = tid; q < nkc * 128; q += 256) {   // one 16-byte piece (8 channels of one pixel) of hi and of lo per iteration
        const int kc = q >> 7, rem = q & 127, r = rem >> 2, c16 = rem & 3;
        if (p0 + r >= HW) continue;
        const float sc = s_scale[r];
        const int ch = kc * 32 + c16 * 8;
        uint4 hi, lo;
        pk_split(tile[ch][r] * sc, tile[ch + 1][r] * sc, hi.x, lo.x);
        pk_split(tile[ch + 2][r] * sc, tile[ch + 3][r] * sc, hi.y, lo.y);
        pk_split(tile[ch + 4][r] * sc, tile[ch + 5][r] * sc, hi.z, lo.z);
        pk_split(tile[ch + 6][r] * sc, tile[ch + 7][r] * sc, hi.w, lo.w);
        const size_t R = (size_t)f * HW + p0 + r;
        const size_t t = R >> 8;
        const uint32_t rr = (uint32_t)(R & 255);
        uint8_t *dst = apack + (t * nkc + kc) * 32768 + rr * 64u + ((c16 ^ ((rr >> 1) & 3u)) << 4);
        *reinterpret_cast<uint4 *>(dst) = hi;
        *reinterpret_cast<uint4 *>(dst + 16384) = lo;
    }
}

// ---- the 4-corner weighted gather of one row, one warp, all levels ------------------------------------
// Index math and the (inverted) weights are those of Pipe.py:62-75, evaluated in the same fp32 order with no
// FMA contraction, so the result is bit-identical to the reference's eager ops for the same `proj`.
// returns this lane's max |value| over the row (for the fp16 row scaling of a tensor-core consumer)
template <bool kStreaming>
__device__ __forceinline__ float gather_row_warp(const MapSet &m, int f, float prow, float pcol, float eps, int lane,
                                                 float *__restrict__ out_row) {
    float amax = 0.f;
#pragma unroll
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        const float q0 = __fsub_rn(__fdiv_rn(prow, m.rs_h[l]), eps);
        const float q1 = __fsub_rn(__fdiv_rn(pcol, m.rs_w[l]), eps);
        const int i0 = (int)q0, i1 = (int)q1;  // .long(): truncation toward zero
        const float a = __fsub_rn(q0, (float)i0), b = __fsub_rn(q1, (float)i1);
        const float a_ = __fsub_rn(1.0f, a), b_ = __fsub_rn(1.0f, b);
        const int H = m.h[l], W = m.w[l], C = m.C;
        const float *base = m.nhwc[l] + (size_t)f * m.frame_stride[l];
        // corner validity: row H / column W are the zero pad of Pipe.py:47-48
        const bool r0 = i0 >= 0 && i0 < H, r1 = i0 + 1 >= 0 && i0 + 1 < H;
        const bool c0 = i1 >= 0 && i1 < W, c1 = i1 + 1 >= 0 && i1 + 1 < W;
        const float4 *p00 = reinterpret_cast<const float4 *>(base + ((size_t)i0 * W + i1) * C);
        const float4 *p10 = reinterpret_cast<const float4 *>(base + ((size_t)(i0 + 1) * W + i1) * C);
        const float4 *p01 = reinterpret_cast<const float4 *>(base + ((size_t)i0 * W + i1 + 1) * C);
        const float4 *p11 = reinterpret_cast<const float4 *>(base + ((size_t)(i0 + 1) * W + i1 + 1) * C);
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c4 = lane; c4 < C / 4; c4 += 32) {
            const float4 f00 = (r0 && c0) ? __ldg(p00 + c4) : z4;
            const float4 f10 = (r1 && c0) ? __ldg(p10 + c4) : z4;
            const float4 f01 = (r0 && c1) ? __ldg(p01 + c4) : z4;
            const float4 f11 = (r1 && c1) ? __ldg(p11 + c4) : z4;
            float4 g;
#define MVX_CORNERS(e)                                                     \
    g.e = __fmul_rn(__fmul_rn(f00.e, a), b);                               \
    g.e = __fadd_rn(g.e, __fmul_rn(__fmul_rn(f10.e, a_), b));              \
    g.e = __fadd_rn(g.e, __fmul_rn(__fmul_rn(f01.e, a), b_));              \
    g.e = __fadd_rn(g.e, __fmul_rn(__fmul_rn(f11.e, a_), b_));
            MVX_CORNERS(x) MVX_CORNERS(y) MVX_CORNERS(z) MVX_CORNERS(w)
#undef MVX_CORNERS
            float4 *dst = reinterpret_cast<float4 *>(out_row + (size_t)l * C) + c4;
            if (kStreaming) st_cs_f4(dst, g); else *dst = g;
            amax = fmaxf(fmaxf(amax, fmaxf(fabsf(g.x), fabsf(g.y))), fmaxf(fabsf(g.z), fabsf(g.w)));
        }
    }
    return amax;
}

template <bool kStreaming>
__device__ __forceinline__ void zero_row_warp(int C3, int lane, float *__restrict__ out_row) {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c4 = lane; c4 < C3 / 4; c4 += 32) {
        float4 *dst = reinterpret_cast<float4 *>(out_row) + c4;
        if (kStreaming) st_cs_f4(dst, z4); else *dst = z4;
    }
}

// ---- featureMaping drop-in: dense (R,9) voxel rows in/out, (R,3C) out ----------------------------------
__global__ void __launch_bounds__(256) feature_mapping_kernel(float *__restrict__ voxels, long long R, MapSet m, float eps,
                                                              float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= R) return;
    float *vrow = voxels + (size_t)r * 9;
    const float mine = lane < 9 ? vrow[lane] : 0.f;
    const float x = __shfl_sync(0xffffffffu, mine, 0), y = __shfl_sync(0xffffffffu, mine, 1),
                z = __shfl_sync(0xffffffffu, mine, 2);
    const float prow = __shfl_sync(0xffffffffu, mine, 7), pcol = __shfl_sync(0xffffffffu, mine, 8);
    float *orow = out + (size_t)r * 3 * m.C;
    if (x == 0.f && y == 0.f && z == 0.f) {  // Pipe.py:53-59,80: pad slot -> zero the voxel row and its features
        if (lane < 9) vrow[lane] = 0.f;
        zero_row_warp<true>(3 * m.C, lane, orow);
    } else {
        gather_row_warp<true>(m, 0, prow, pcol, eps, lane, orow);
    }
}

// ---- fused path: per compact row, voxel features + projection -------------------------------------------
__global__ void __launch_bounds__(256) rows_build_kernel(RowsParams p) {
    __shared__ float c32[32];
    const int f = blockIdx.y;
    if (!p.point_calib && threadIdx.x < 32) c32[threadIdx.x] = p.calib32[f * 32 + threadIdx.x];
    __syncthreads();
    const int N = p.counts[f * 4 + 0], K = p.counts[f * 4 + 1];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > K) return;
    const size_t ro = (size_t)f * p.capA + r;
    float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
    float2 pr = make_float2(0.f, 0.f);
    float w;
    if (r == K) {
        w = (float)((long long)N * p.T - K);  // the pad slots of this frame, all identical rows (SURVEY.md §7 hard part 4)
    } else {
        w = 1.f;
        const float *pts = p.points + (size_t)p.off[f] * p.point_stride;
        const int v = p.row_vox[(size_t)f * p.cap + r];
        const int r0 = p.vox_row0[(size_t)f * (p.cap + 1) + v], n = p.vox_cnt[(size_t)f * p.cap + v];
        double sx = 0, sy = 0, sz = 0;  // fp64 centroid over the kept points in slot order (Preprocessing.py:112-113)
        for (int k = 0; k < n; ++k) {
            const float *q = pts + (size_t)p.row_point[(size_t)f * p.cap + r0 + k] * p.point_stride;
            sx += (double)q[0], sy += (double)q[1], sz += (double)q[2];
        }
        const int pi = p.row_point[(size_t)f * p.cap + r];
        const float *q = pts + (size_t)pi * p.point_stride;
        const float x = q[0], y = q[1], z = q[2], refl = q[3];
        if (!(x == 0.f && y == 0.f && z == 0.f)) {  // a real point at the exact origin is treated as a pad slot (Pipe.py:53-59)
            lo = make_float4(x, y, z, (float)((double)x - sx / (double)n));
            hi = make_float4((float)((double)y - sy / (double)n), (float)((double)z - sz / (double)n), refl, 0.f);
            float u, vv;
            // merged point sets (GT-paste, train.py:36-41): every point is projected through the calibration it came with
            const int cs = p.point_calib ? p.point_calib[p.off[f] + pi] : f;
            if (p.calib_f64 && p.calib_f64[cs]) {   // float64 calibration: fp64 projection, rounded once (torch.Tensor(voxel), train.py:125)
                double ud, vd, czd;
                project_point_z_f64(p.calib64 + (size_t)cs * 32, x, y, z, ud, vd, czd);
                u = (float)ud, vv = (float)vd;
            } else {
                project_point(p.point_calib ? p.calib32 + (size_t)cs * 32 : c32, x, y, z, u, vv);
            }
            pr = make_float2(vv, u);  // (row, col) = lidar2Img(...)[:, [1, 0]]  (train.py:33)
        }
    }
    float4 *dst = reinterpret_cast<float4 *>(p.vox8 + ro * 8);
    dst[0] = lo;
    dst[1] = hi;
    reinterpret_cast<float2 *>(p.proj)[ro] = pr;
    p.rowA_w[ro] = w;
}

__global__ void __launch_bounds__(256) gather_rows_kernel(MapSet m, int capA, const int *__restrict__ counts,
                                                          const float *__restrict__ vox8, const float *__restrict__ proj,
                                                          float eps, float *__restrict__ A1, float *__restrict__ rowmax) {
    const int f = blockIdx.y, lane = threadIdx.x & 31;
    const int K = counts[f * 4 + 1];
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r > K) return;
    const size_t ro = (size_t)f * capA + r;
    const float4 xyz = *reinterpret_cast<const float4 *>(vox8 + ro * 8);
    float *orow = A1 + ro * 3 * m.C;
    if (xyz.x == 0.f && xyz.y == 0.f && xyz.z == 0.f) {
        zero_row_warp<false>(3 * m.C, lane, orow);
        if (rowmax && lane == 0) rowmax[ro] = 0.f;
    } else {
        const float2 pr = reinterpret_cast<const float2 *>(proj)[ro];
        float amax = gather_row_warp<false>(m, f, pr.x, pr.y, eps, lane, orow);
        if (rowmax) {
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, d));
            if (lane == 0) rowmax[ro] = amax;
        }
    }
}


// ---- pixel-first fcn1: per compact row, bias + 12 weighted rows of Z, ReLU, raw store, BatchNorm sums ------------
// Rows are first sorted by the level-0 cell they sample (counting sort: histogram, scan, scatter), cells ordered in
// 4x4 blocks with Morton order inside a block, so consecutive sorted rows share their level-0 cell and, almost always,
// their level-1/level-2 cells. The combine kernel walks sorted rows; a warp keeps the 4 corner vectors of each level in
// registers and re-loads them only when that level's cell changes (about every 5th / 17th / 60th row at KITTI
// density), which cuts the corner traffic ~10x against a row-by-row gather. Output rows are written back to their
// compact position (one contiguous 3 KB row per CTA step).
constexpr int kCombCout = 768;
constexpr int kCombWarps = 6;        // one warp per 128 output columns (one float4 per lane)
constexpr int kCombRows = 256;       // sorted rows per CTA

__device__ __forceinline__ int combine_key(const CombineArgs &a, int f, int r, int K) {
    const size_t ro = (size_t)f * a.capA + r;
    const float4 xyz = __ldg(reinterpret_cast<const float4 *>(a.vox8 + ro * 8));
    if (r >= K || (xyz.x == 0.f && xyz.y == 0.f && xyz.z == 0.f)) return a.nbins;  // pad row / origin point: no corners
    const float2 pr = __ldg(reinterpret_cast<const float2 *>(a.proj) + ro);
    const CellRef c = cell_of(pr.x, pr.y, a.rs_h[0], a.rs_w[0], a.eps);
    const int y = min(max(c.i0, 0), a.h[0] - 1), x = min(max(c.i1, 0), a.w[0] - 1);
    const int wb = (a.w[0] + 3) / 4;
    const int inner = ((y & 2) << 2) | ((x & 2) << 1) | ((y & 1) << 1) | (x & 1);  // Morton order inside the 4x4 block
    return ((y >> 2) * wb + (x >> 2)) * 16 + inner;
}

__global__ void __launch_bounds__(256) combine_hist_kernel(CombineArgs a) {
    const int f = blockIdx.y, K = a.counts[f * 4 + 1];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > K) return;
    atomicAdd(a.bin_count + (size_t)f * (a.nbins + 1) + combine_key(a, f, r, K), 1);
}

__global__ void __launch_bounds__(1024) combine_scan_kernel(CombineArgs a) {  // one CTA per frame, four bins per thread and round
    const int f = blockIdx.x, nb = a.nbins + 1;
    int *cnt = a.bin_count + (size_t)f * nb, *start = a.bin_start + (size_t)f * (nb + 1);
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
                cnt[b + q] = 0;  // becomes the scatter cursor
            }
            ex += v[q];
        }
        carry += total;
    }
    if (threadIdx.x == 0) start[nb] = carry;
}

__global__ void __launch_bounds__(256) combine_scatter_kernel(CombineArgs a) {
    const int f = blockIdx.y, K = a.counts[f * 4 + 1];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > K) return;
    const int nb = a.nbins + 1;
    const int key = combine_key(a, f, r, K);
    const int pos = a.bin_start[(size_t)f * (nb + 1) + key] + atomicAdd(a.bin_count + (size_t)f * nb + key, 1);
    a.perm[(size_t)f * a.capA + pos] = r;
}

// per-row, per-level sampling record, computed once per row by one thread (the six column warps only read it)
struct CombRec {
    int cell;        // x0 | y0 << 12 | dx << 24 | dy << 25 : clamped corner coordinates; also the cache tag
    float w[4];      // w00, w10, w01, w11 (0 where the corner lies on the zero pad row/column of Pipe.py:47-48)
};

#ifndef MVX_COMB_MINB
#define MVX_COMB_MINB 3
#endif
__device__ __forceinline__ float4 bf16x4_to_f4(uint2 v) {   // exact: bf16 is the top half of an fp32
    return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xFFFF0000u), __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xFFFF0000u));
}
__device__ __forceinline__ uint2 f4_to_bf16x4(float4 v) {
    uint2 r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.x) : "f"(v.y), "f"(v.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.y) : "f"(v.w), "f"(v.z));
    return r;
}

// ZB / YB: Z is read / Y1 is written as bf16 (the reduced-precision mode; the arithmetic in between stays fp32)
template <bool ZB = false, bool YB = false>
__global__ void __launch_bounds__(kCombWarps * 32, MVX_COMB_MINB) combine_rows_kernel(CombineArgs a) {
    __shared__ int s_row[kCombRows];                     // compact row; ~row for rows without corners
    __shared__ float s_w[kCombRows];                     // BatchNorm multiplicity
    __shared__ float4 s_recw[kCombRows][MVX_NUM_LEVELS];   // corner weights: one 16-byte broadcast load per row and level
    __shared__ int s_cell[kCombRows][MVX_NUM_LEVELS];      // packed corner coordinates (the cache tag)
    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.counts[f * 4 + 1];
    const int p0 = blockIdx.x * kCombRows;
    if (p0 > K) return;
    const int pend = min(p0 + kCombRows, K + 1);
    // stage this CTA's rows: sorted position -> row, weights and corner coordinates of the three levels. One parallel
    // round of gathers and ONE evaluation of the index math per row, instead of one per column warp.
    for (int i = tid; i < pend - p0; i += kCombWarps * 32) {
        const int r = a.perm[(size_t)f * a.capA + p0 + i];
        const size_t ro = (size_t)f * a.capA + r;
        const float4 xyz = __ldg(reinterpret_cast<const float4 *>(a.vox8 + ro * 8));
        const bool none = r >= K || (xyz.x == 0.f && xyz.y == 0.f && xyz.z == 0.f);  // pad row / origin point: A1 row is zero
        s_row[i] = none ? ~r : r;
        s_w[i] = __ldg(a.row_w + ro);
        const float2 pr = __ldg(reinterpret_cast<const float2 *>(a.proj) + ro);
#pragma unroll
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
            const CellRef c = cell_of(pr.x, pr.y, a.rs_h[l], a.rs_w[l], a.eps);
            const int H = a.h[l], W = a.w[l];
            const float4 cw = corner_weights(c, H, W);
            CombRec rec;
            rec.w[0] = cw.x, rec.w[1] = cw.y, rec.w[2] = cw.z, rec.w[3] = cw.w;
            const int y0 = min(max(c.i0, 0), H - 1), y1 = min(max(c.i0 + 1, 0), H - 1);
            const int x0 = min(max(c.i1, 0), W - 1), x1 = min(max(c.i1 + 1, 0), W - 1);
            rec.cell = x0 | (y0 << 12) | ((x1 - x0) << 24) | ((y1 - y0) << 25);
            s_recw[i][l] = make_float4(rec.w[0], rec.w[1], rec.w[2], rec.w[3]);
            s_cell[i][l] = rec.cell;
        }
    }
    __syncthreads();
    const int col0 = warp * 128 + lane * 4;
    const float4 bias = __ldg(reinterpret_cast<const float4 *>(a.bias + col0));
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 ps = z4, pss = z4;                  // fp32 column sums over runs of 16 rows
    double ds[4] = {0, 0, 0, 0}, dss[4] = {0, 0, 0, 0};   // this lane owns its 4 columns within the CTA: fp64 in registers
    float4 v00[MVX_NUM_LEVELS], v10[MVX_NUM_LEVELS], v01[MVX_NUM_LEVELS], v11[MVX_NUM_LEVELS];
    int tag[MVX_NUM_LEVELS];
#pragma unroll
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) tag[l] = -1, v00[l] = v10[l] = v01[l] = v11[l] = z4;
    auto fold = [&]() {
        ds[0] += (double)ps.x, ds[1] += (double)ps.y, ds[2] += (double)ps.z, ds[3] += (double)ps.w;
        dss[0] += (double)pss.x, dss[1] += (double)pss.y, dss[2] += (double)pss.z, dss[3] += (double)pss.w;
        ps = z4, pss = z4;
    };
    for (int p = p0; p < pend; ++p) {
        const int i = p - p0;
        const int rr = s_row[i];
        const int r = rr < 0 ? ~rr : rr;
        float4 acc = bias;
        if (rr >= 0) {
#pragma unroll
            for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
                const float4 rw = s_recw[i][l];
                const int cell = s_cell[i][l];
                if (cell != tag[l]) {  // warp-uniform: this level's cell changed, fetch its 4 corner vectors
                    tag[l] = cell;
                    const int W = a.w[l];
                    const int x0 = cell & 0xFFF, y0 = (cell >> 12) & 0xFFF, dx = (cell >> 24) & 1, dy = (cell >> 25) & 1;
                    const size_t e00 = (size_t)f * a.frame_stride[l] + ((size_t)y0 * W + x0) * kCombCout + col0;   // element index
                    if constexpr (ZB) {
                        const __nv_bfloat16 *b00 = reinterpret_cast<const __nv_bfloat16 *>(a.Z[l]) + e00;
                        v00[l] = bf16x4_to_f4(__ldg(reinterpret_cast<const uint2 *>(b00)));
                        v10[l] = bf16x4_to_f4(__ldg(reinterpret_cast<const uint2 *>(b00 + (size_t)dy * W * kCombCout)));
                        v01[l] = bf16x4_to_f4(__ldg(reinterpret_cast<const uint2 *>(b00 + (size_t)dx * kCombCout)));
                        v11[l] = bf16x4_to_f4(__ldg(reinterpret_cast<const uint2 *>(b00 + ((size_t)dy * W + dx) * kCombCout)));
                    } else {
                    const float *b00 = a.Z[l] + e00;
                    v00[l] = __ldg(reinterpret_cast<const float4 *>(b00));
                    v10[l] = __ldg(reinterpret_cast<const float4 *>(b00 + (size_t)dy * W * kCombCout));
                    v01[l] = __ldg(reinterpret_cast<const float4 *>(b00 + (size_t)dx * kCombCout));
                    v11[l] = __ldg(reinterpret_cast<const float4 *>(b00 + ((size_t)dy * W + dx) * kCombCout));
                    }
                }
#define MVX_COMB(e) acc.e = fmaf(v11[l].e, rw.w, fmaf(v01[l].e, rw.z, fmaf(v10[l].e, rw.y, fmaf(v00[l].e, rw.x, acc.e))));
                MVX_COMB(x) MVX_COMB(y) MVX_COMB(z) MVX_COMB(w)
#undef MVX_COMB
            }
        }
        float4 y;
        y.x = fmaxf(acc.x, 0.f), y.y = fmaxf(acc.y, 0.f), y.z = fmaxf(acc.z, 0.f), y.w = fmaxf(acc.w, 0.f);
        if constexpr (YB) {
            // the statistics below are those of the values conv1 will actually read: the bf16-rounded ones
            const uint2 yb = f4_to_bf16x4(y);
            *reinterpret_cast<uint2 *>(reinterpret_cast<__nv_bfloat16 *>(a.Y1) + ((size_t)f * a.capA + r) * kCombCout + col0) = yb;
            y = bf16x4_to_f4(yb);
        } else {
            *reinterpret_cast<float4 *>(a.Y1 + ((size_t)f * a.capA + r) * kCombCout + col0) = y;
        }
        const float w = s_w[i];
        if (w == 1.f) {
            ps.x += y.x, ps.y += y.y, ps.z += y.z, ps.w += y.w;
            pss.x = fmaf(y.x, y.x, pss.x), pss.y = fmaf(y.y, y.y, pss.y);
            pss.z = fmaf(y.z, y.z, pss.z), pss.w = fmaf(y.w, y.w, pss.w);
        } else if (w != 0.f) {   // the weighted pad row: exact fp64 side path
            const double wd = (double)w;
            ds[0] += wd * y.x, ds[1] += wd * y.y, ds[2] += wd * y.z, ds[3] += wd * y.w;
            dss[0] += wd * y.x * y.x, dss[1] += wd * y.y * y.y, dss[2] += wd * y.z * y.z, dss[3] += wd * y.w * y.w;
        }
        if ((i & 15) == 15) fold();
    }
    fold();
    double *o = a.out_stats + ((size_t)f * kCombCout + col0) * 2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        atomicAdd(o + 2 * j, ds[j]);
        atomicAdd(o + 2 * j + 1, dss[j]);
    }
}


// ---- combine, second version: run-structured main loop + asynchronous corner ring ------------------------------------------
// What bounded the first version (ncu, r5e): not the issue rate and not the bytes - removing all stores or all corner loads, or
// cutting the instructions per row by a third, left it at 0.95 ms. Every warp walked its rows through a serial chain of
// shared-load -> test -> branch steps (8 branches per row) and stalled for a full DRAM round trip at each cell change, with only
// 18 warps per SM to cover for it: ~900 cycles per row and warp. This version
//  (1) cuts the sorted rows into RUNS in the staging phase (a run = up to 16 consecutive ordinary rows that sample the same cells
//      at all three levels): the per-row loop body is branch-free (3 broadcast LDS.128 + 48 FFMA + ReLU + store + sums) and the
//      compiler overlaps consecutive rows; cell changes, rows without corners and weighted rows are handled at run heads only;
//  (2) lists the cell changes of the CTA in order ("events") and lets every warp fetch the corner vectors of the next NS events
//      ahead of time with cp.async (LDGSTS: global -> shared without registers) into a private ring; a cell change then costs a
//      wait on an already landed group plus four LDS.128.
// Arithmetic and its order are those of the first version: Y1 is bit-identical.
#ifndef MVX_COMB_NS
#define MVX_COMB_NS 4
#endif
constexpr int kCombNS = MVX_COMB_NS;                                  // ring slots (events in flight) per warp
template <bool ZB>
struct CombSmem {
    static constexpr int kSlotBytes = 4 * 32 * (ZB ? 8 : 16);       // four corners x 32 lanes x this lane's 4 columns
    static constexpr int kRow = 0;                                  // int[256]
    static constexpr int kW = kRow + kCombRows * 4;                 // float[256]
    static constexpr int kRecw = kW + kCombRows * 4;                // float4[256][3]
    static constexpr int kCell = kRecw + kCombRows * MVX_NUM_LEVELS * 16;   // int[256][3]
    static constexpr int kRun = kCell + kCombRows * MVX_NUM_LEVELS * 4;     // uint8[256]
    static constexpr int kEv = kRun + kCombRows;                    // uint16[768]
    static constexpr int kRing = kEv + kCombRows * MVX_NUM_LEVELS * 2;      // [warps][NS][slot]
    static constexpr int kTotal = kRing + kCombWarps * kCombNS * kSlotBytes;
};
__device__ __forceinline__ void cp_async_wait_allow(int allow) {   // wait until at most `allow` of this thread's groups are pending
    if (allow >= 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
    else if (allow == 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
    else if (allow == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
}

template <bool ZB, bool YB>
__global__ void __launch_bounds__(kCombWarps * 32, MVX_COMB_MINB) combine_runs_kernel(CombineArgs a) {
    using S = CombSmem<ZB>;
    constexpr int kRowMask = 0xFFFFFF, kChg0 = 1 << 24, kChgAny = 7 << 24, kNone = 1 << 27, kWgt = 1 << 28;
    extern __shared__ __align__(16) unsigned char comb_smem[];
    int *s_row = reinterpret_cast<int *>(comb_smem + S::kRow);
    float *s_w = reinterpret_cast<float *>(comb_smem + S::kW);
    float4(*s_recw)[MVX_NUM_LEVELS] = reinterpret_cast<float4(*)[MVX_NUM_LEVELS]>(comb_smem + S::kRecw);
    int(*s_cell)[MVX_NUM_LEVELS] = reinterpret_cast<int(*)[MVX_NUM_LEVELS]>(comb_smem + S::kCell);
    unsigned char *s_run = comb_smem + S::kRun;
    unsigned short *s_ev = reinterpret_cast<unsigned short *>(comb_smem + S::kEv);
    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.counts[f * 4 + 1];
    const int p0 = blockIdx.x * kCombRows;
    if (p0 > K) return;
    const int n_rows = min(p0 + kCombRows, K + 1) - p0;
    // ---- staging 1: sorted position -> row, weight, corner weights and coordinates of the three levels (once per row) -------
    for (int i = tid; i < n_rows; i += kCombWarps * 32) {
        const int r = a.perm[(size_t)f * a.capA + p0 + i];
        const size_t ro = (size_t)f * a.capA + r;
        const float4 xyz = __ldg(reinterpret_cast<const float4 *>(a.vox8 + ro * 8));
        const bool none = r >= K || (xyz.x == 0.f && xyz.y == 0.f && xyz.z == 0.f);  // pad row / origin point: A1 row is zero
        const float wgt = __ldg(a.row_w + ro);
        s_row[i] = r | (none ? kNone : 0) | (wgt != 1.f ? kWgt : 0);
        s_w[i] = wgt;
        const float2 pr = __ldg(reinterpret_cast<const float2 *>(a.proj) + ro);
#pragma unroll
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
            const CellRef c = cell_of(pr.x, pr.y, a.rs_h[l], a.rs_w[l], a.eps);
            const int H = a.h[l], W = a.w[l];
            const int y0 = min(max(c.i0, 0), H - 1), y1 = min(max(c.i0 + 1, 0), H - 1);
            const int x0 = min(max(c.i1, 0), W - 1), x1 = min(max(c.i1 + 1, 0), W - 1);
            s_recw[i][l] = corner_weights(c, H, W);
            s_cell[i][l] = none ? -1 : (x0 | (y0 << 12) | ((x1 - x0) << 24) | ((y1 - y0) << 25));
        }
    }
    __syncthreads();
    // ---- staging 2: change flags against the previous row of the CTA (the row behind one without corners reloads everything) --
    for (int i = tid; i < n_rows; i += kCombWarps * 32) {
        int flags = 0;
        if (s_cell[i][0] != -1) {
#pragma unroll
            for (int l = 0; l < MVX_NUM_LEVELS; ++l)
                if (i == 0 || s_cell[i][l] != s_cell[i - 1][l]) flags |= kChg0 << l;
        }
        s_row[i] |= flags;
    }
    __syncthreads();
    // ---- staging 3: run lengths (valid at EVERY row: the walk below may land anywhere) and the ordered event list -----------
    for (int i = tid; i < n_rows; i += kCombWarps * 32) {
        int n = 1;
        if (!(s_row[i] & (kNone | kWgt)))
            while (n < 16 && i + n < n_rows && !(s_row[i + n] & (kChgAny | kNone | kWgt))) ++n;
        s_run[i] = (unsigned char)n;
    }
    int n_ev;
    {
        const int i0 = 2 * tid, i1 = 2 * tid + 1;     // threads 0..127 own two consecutive rows each
        const int f0 = i0 < n_rows ? (s_row[i0] & kChgAny) >> 24 : 0, f1 = i1 < n_rows ? (s_row[i1] & kChgAny) >> 24 : 0;
        int k = block_exclusive_scan(__popc(f0) + __popc(f1), &n_ev);
#pragma unroll
        for (int l = 0; l < MVX_NUM_LEVELS; ++l)
            if (f0 & (1 << l)) s_ev[k++] = (unsigned short)(i0 | (l << 8));
#pragma unroll
        for (int l = 0; l < MVX_NUM_LEVELS; ++l)
            if (f1 & (1 << l)) s_ev[k++] = (unsigned short)(i1 | (l << 8));
    }
    __syncthreads();

    const int col0 = warp * 128 + lane * 4;
    const float4 bias = __ldg(reinterpret_cast<const float4 *>(a.bias + col0));
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 ps = z4, pss = z4;                  // fp32 column sums over at most 16 rows
    double ds[4] = {0, 0, 0, 0}, dss[4] = {0, 0, 0, 0};   // this lane owns its 4 columns within the CTA: fp64 in registers
    float4 v00[MVX_NUM_LEVELS], v10[MVX_NUM_LEVELS], v01[MVX_NUM_LEVELS], v11[MVX_NUM_LEVELS];
#pragma unroll
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) v00[l] = v10[l] = v01[l] = v11[l] = z4;
    auto fold = [&]() {
        ds[0] += (double)ps.x, ds[1] += (double)ps.y, ds[2] += (double)ps.z, ds[3] += (double)ps.w;
        dss[0] += (double)pss.x, dss[1] += (double)pss.y, dss[2] += (double)pss.z, dss[3] += (double)pss.w;
        ps = z4, pss = z4;
    };
    // this warp's ring: slot (k % NS) of event k; inside a slot corner c of lane `lane` sits at c * 32 * EB + lane * EB
    constexpr int EB = ZB ? 8 : 16;
    unsigned char *ring = comb_smem + S::kRing + warp * (kCombNS * S::kSlotBytes) + lane * EB;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    auto issue = [&](int k) {   // start the copy of event k's four corner vectors (this lane's 4 columns of each)
        const int ev = s_ev[k];
        const int i = ev & 0xFF, l = ev >> 8;
        const int cell = s_cell[i][l];
        const int W = a.w[l];
        const int x0 = cell & 0xFFF, y0 = (cell >> 12) & 0xFFF, dx = (cell >> 24) & 1, dy = (cell >> 25) & 1;
        const size_t e00 = (size_t)f * a.frame_stride[l] + ((size_t)y0 * W + x0) * kCombCout + col0;   // element index
        const char *b00 = reinterpret_cast<const char *>(a.Z[l]) + e00 * (ZB ? 2 : 4);
        const size_t sx = (size_t)dx * kCombCout * (ZB ? 2 : 4), sy = (size_t)dy * W * kCombCout * (ZB ? 2 : 4);
        const uint32_t dst = ring_s + (uint32_t)(k % kCombNS) * S::kSlotBytes;
        if constexpr (ZB) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(b00) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 32 * EB), "l"(b00 + sy) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 64 * EB), "l"(b00 + sx) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 96 * EB), "l"(b00 + sy + sx) : "memory");
        } else {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(b00) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 32 * EB), "l"(b00 + sy) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 64 * EB), "l"(b00 + sx) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 96 * EB), "l"(b00 + sy + sx) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    int issued = 0, consumed = 0;
    for (; issued < min(kCombNS, n_ev); ++issued) issue(issued);
    float *const y_f32 = a.Y1 + (size_t)f * a.capA * kCombCout + col0;     // this lane's 4 columns of row 0 of the frame
    __nv_bfloat16 *const y_b16 = reinterpret_cast<__nv_bfloat16 *>(a.Y1) + (size_t)f * a.capA * kCombCout + col0;
    auto row_value = [&](int ii, bool corners) -> float4 {
        float4 acc = bias;
        if (corners) {
#pragma unroll
            for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
                const float4 rw = s_recw[ii][l];
#define MVX_COMB(e) acc.e = fmaf(v11[l].e, rw.w, fmaf(v01[l].e, rw.z, fmaf(v10[l].e, rw.y, fmaf(v00[l].e, rw.x, acc.e))));
                MVX_COMB(x) MVX_COMB(y) MVX_COMB(z) MVX_COMB(w)
#undef MVX_COMB
            }
        }
        float4 y;
        y.x = fmaxf(acc.x, 0.f), y.y = fmaxf(acc.y, 0.f), y.z = fmaxf(acc.z, 0.f), y.w = fmaxf(acc.w, 0.f);
        return y;
    };
    auto store_row = [&](unsigned r, float4 &y) {
        if constexpr (YB) {   // the statistics are those of the values conv1 will actually read: the bf16-rounded ones
            const uint2 yb = f4_to_bf16x4(y);
            *reinterpret_cast<uint2 *>(y_b16 + (size_t)r * kCombCout) = yb;
            y = bf16x4_to_f4(yb);
        } else {
            *reinterpret_cast<float4 *>(y_f32 + (size_t)r * kCombCout) = y;
        }
    };
    int i = 0, since = 0;
    while (i < n_rows) {
        const int rw_ = s_row[i];
        if (rw_ & kChgAny) {
#pragma unroll
            for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
                if (rw_ & (kChg0 << l)) {   // warp-uniform: level l samples another cell from this row on
                    cp_async_wait_allow(issued - consumed - 1);
                    const unsigned char *slot = ring + (consumed % kCombNS) * S::kSlotBytes;
                    if constexpr (ZB) {
                        v00[l] = bf16x4_to_f4(*reinterpret_cast<const uint2 *>(slot));
                        v10[l] = bf16x4_to_f4(*reinterpret_cast<const uint2 *>(slot + 32 * EB));
                        v01[l] = bf16x4_to_f4(*reinterpret_cast<const uint2 *>(slot + 64 * EB));
                        v11[l] = bf16x4_to_f4(*reinterpret_cast<const uint2 *>(slot + 96 * EB));
                    } else {
                        v00[l] = *reinterpret_cast<const float4 *>(slot);
                        v10[l] = *reinterpret_cast<const float4 *>(slot + 32 * EB);
                        v01[l] = *reinterpret_cast<const float4 *>(slot + 64 * EB);
                        v11[l] = *reinterpret_cast<const float4 *>(slot + 96 * EB);
                    }
                    ++consumed;
                    if (issued < n_ev) {   // the slot just read is free again: this lane wrote and read only its own bytes of it
                        issue(issued);
                        ++issued;
                    }
                }
            }
        }
        if (rw_ & (kNone | kWgt)) {   // a row without corners and / or with a BatchNorm multiplicity != 1 (the pad row): on its own
            float4 y = row_value(i, !(rw_ & kNone));
            store_row((unsigned)(rw_ & kRowMask), y);
            if (rw_ & kWgt) {   // exact fp64 side path
                const double wd = (double)s_w[i];
                ds[0] += wd * y.x, ds[1] += wd * y.y, ds[2] += wd * y.z, ds[3] += wd * y.w;
                dss[0] += wd * y.x * y.x, dss[1] += wd * y.y * y.y, dss[2] += wd * y.z * y.z, dss[3] += wd * y.w * y.w;
            } else {
                if (since == 16) fold(), since = 0;
                ++since;
                ps.x += y.x, ps.y += y.y, ps.z += y.z, ps.w += y.w;
                pss.x = fmaf(y.x, y.x, pss.x), pss.y = fmaf(y.y, y.y, pss.y), pss.z = fmaf(y.z, y.z, pss.z), pss.w = fmaf(y.w, y.w, pss.w);
            }
            ++i;
            continue;
        }
        const int n = s_run[i];
        if (since + n > 16) fold(), since = 0;
        since += n;
#pragma unroll 2
        for (int j = 0; j < n; ++j) {   // the run: ordinary rows on the cached corner vectors, no decisions
            float4 y = row_value(i + j, true);
            store_row((unsigned)(s_row[i + j] & kRowMask), y);
            ps.x += y.x, ps.y += y.y, ps.z += y.z, ps.w += y.w;
            pss.x = fmaf(y.x, y.x, pss.x), pss.y = fmaf(y.y, y.y, pss.y), pss.z = fmaf(y.z, y.z, pss.z), pss.w = fmaf(y.w, y.w, pss.w);
        }
        i += n;
    }
    fold();
    double *o = a.out_stats + ((size_t)f * kCombCout + col0) * 2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        atomicAdd(o + 2 * j, ds[j]);
        atomicAdd(o + 2 * j + 1, dss[j]);
    }
}

}  // namespace

int launch_combine_sort(const CombineArgs &a, int B, cudaStream_t st) {
    MVX_REQUIRE(a.bin_count && a.bin_start && a.perm && a.nbins == combine_bins(a.h[0], a.w[0]), MVX_EINVAL, "combine: bad sort scratch");
    MVX_CUDA_CHECK(cudaMemsetAsync(a.bin_count, 0, (size_t)B * (a.nbins + 1) * sizeof(int), st));
    const dim3 rows_grid((a.capA + 255) / 256, B);
    combine_hist_kernel<<<rows_grid, 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    combine_scan_kernel<<<B, 1024, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    combine_scatter_kernel<<<rows_grid, 256, 0, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

static int g_comb_v1 = 0;     // 1: the first combine kernel (row-by-row walk) instead of the run-structured one - kept for A/B runs
void set_combine_v1(int on) { g_comb_v1 = on; }

template <bool ZB, bool YB>
static int launch_combine_runs_t(const CombineArgs &a, dim3 grid, cudaStream_t st) {
    using S = CombSmem<ZB>;
    static bool attr_set = false;
    if (!attr_set) {
        MVX_CUDA_CHECK(cudaFuncSetAttribute(combine_runs_kernel<ZB, YB>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
        attr_set = true;
    }
    combine_runs_kernel<ZB, YB><<<grid, kCombWarps * 32, S::kTotal, st>>>(a);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_combine_rows(const CombineArgs &a, int B, cudaStream_t st) {
    dim3 grid((a.capA + kCombRows - 1) / kCombRows, B);
    MVX_REQUIRE(a.capA <= 0xFFFFFF, MVX_EINVAL, "combine: more than 2^24 rows per frame");
    if (a.z_bf16 || a.y1_bf16) {
        MVX_REQUIRE(a.z_bf16 && a.y1_bf16, MVX_EINVAL, "combine: the bf16 mode stores both Z and Y1 as bf16");
        if (!g_comb_v1) return launch_combine_runs_t<true, true>(a, grid, st);
        combine_rows_kernel<true, true><<<grid, kCombWarps * 32, 0, st>>>(a);
    } else {
        if (!g_comb_v1) return launch_combine_runs_t<false, false>(a, grid, st);
        combine_rows_kernel<><<<grid, kCombWarps * 32, 0, st>>>(a);
    }
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_pack_maps_f16(const float *in, void *apack, float *rowinv, int B, int C, int HW, cudaStream_t st) {
    MVX_REQUIRE(C == 256, MVX_EINVAL, "pack_maps: C must be 256");
    pack_maps_f16_kernel<<<dim3((HW + 31) / 32, B), 256, 0, st>>>(in, C, HW, static_cast<uint8_t *>(apack), rowinv);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_nchw_to_nhwc(const float *in, float *out, int B, int C, int HW, float *rowmax, int *chmax, int chmax_stride, cudaStream_t st) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    if (rowmax) MVX_CUDA_CHECK(cudaMemsetAsync(rowmax, 0, (size_t)B * HW * sizeof(float), st));
    nchw_to_nhwc_kernel<<<grid, 256, 0, st>>>(in, out, C, HW, reinterpret_cast<int *>(rowmax), chmax, chmax_stride);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_rows_build(const RowsParams &p, cudaStream_t st) {
    dim3 grid((p.cap + 1 + 255) / 256, p.B);
    rows_build_kernel<<<grid, 256, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_gather_rows(const MapSet &m, int B, int capA, const int *counts, const float *vox8, const float *proj, float eps,
                       float *A1, float *rowmax, cudaStream_t st) {
    dim3 grid((capA + 7) / 8, B);
    gather_rows_kernel<<<grid, 256, 0, st>>>(m, capA, counts, vox8, proj, eps, A1, rowmax);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

}  // namespace mvx

// ---- C ABI ---------------------------------------------------------------------------------------------
extern "C" int mvx_lidar2img(const float *points, int32_t point_stride, int64_t P, const float *calib32, float *out_uv,
                             void *stream) {
    if (P == 0) return MVX_OK;
    MVX_REQUIRE(points && calib32 && out_uv && P > 0 && point_stride >= 3, MVX_EINVAL, "bad lidar2img argument");
    mvx::lidar2img_kernel<<<(unsigned)((P + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(points, point_stride, P,
                                                                                                     calib32, out_uv);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_lidar2img_f64(const float *points, int32_t point_stride, int64_t P, const double *calib64, double *out_uv,
                                 void *stream) {
    if (P == 0) return MVX_OK;
    MVX_REQUIRE(points && calib64 && out_uv && P > 0 && point_stride >= 3, MVX_EINVAL, "bad lidar2img argument");
    mvx::lidar2img_f64_kernel<<<(unsigned)((P + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(points, point_stride, P,
                                                                                                         calib64, out_uv);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_maps_nhwc_bytes(const int32_t *map_h, const int32_t *map_w, int32_t C, size_t *bytes) {
    if (!map_h || !map_w || !bytes || C <= 0) return MVX_EINVAL;
    size_t n = 0;
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) n += (size_t)map_h[l] * map_w[l] * C * sizeof(float);
    *bytes = n;
    return MVX_OK;
}

extern "C" int mvx_feature_mapping(float *voxels, int64_t R, const float *const *maps, const int32_t *map_h,
                                   const int32_t *map_w, int32_t C, float imsize_h, float imsize_w, float eps, float *out,
                                   void *nhwc_ws, size_t nhwc_ws_bytes, void *stream) {
    MVX_REQUIRE(voxels && maps && map_h && map_w && out && nhwc_ws, MVX_EINVAL, "null pointer");
    MVX_REQUIRE(C > 0 && C % 4 == 0, MVX_EINVAL, "C must be a multiple of 4");
    size_t need = 0;
    mvx_maps_nhwc_bytes(map_h, map_w, C, &need);
    MVX_REQUIRE(nhwc_ws_bytes >= need, MVX_ESPACE, "nhwc workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    mvx::MapSet m{};
    m.C = C;
    float *ws = static_cast<float *>(nhwc_ws);
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        MVX_REQUIRE(maps[l] && map_h[l] > 0 && map_w[l] > 0, MVX_EINVAL, "bad map");
        m.h[l] = map_h[l], m.w[l] = map_w[l];
        m.rs_h[l] = imsize_h / (float)map_h[l];
        m.rs_w[l] = imsize_w / (float)map_w[l];
        m.nhwc[l] = ws;
        m.frame_stride[l] = 0;
        int rc = mvx::launch_nchw_to_nhwc(maps[l], ws, 1, C, map_h[l] * map_w[l], nullptr, nullptr, 0, st);
        if (rc) return rc;
        ws += (size_t)map_h[l] * map_w[l] * C;
    }
    if (R == 0) return MVX_OK;
    mvx::feature_mapping_kernel<<<(unsigned)((R + 7) / 8), 256, 0, st>>>(voxels, R, m, eps, out);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
