// Stage 4 — dense middle-layer grid (modules/voxelnet/VoxelNet.py:16-22 `reindex`).
// The reference zero-fills 721 MB and then scatters N*128 isolated 4-byte values (stride G between channels).
// Here the grid is produced in ONE streaming pass: every CTA owns a run of cells, reads the dense
// cell -> voxel map (int32, L2 resident) and writes each channel plane with coalesced 16-byte evict-first
// stores: value = map < 0 ? 0 : feat[vid][c].  HBM traffic = the grid once + the map.
#include "scatter.cuh"

namespace mvx {

namespace {

constexpr int kCellsPerBlock = 1024;  // 256 threads x 4 consecutive cells

// one streaming store of 4 consecutive grid elements, each rounded once from fp32
__device__ __forceinline__ void st_cs_cells(float *p, const float (&q)[4]) {
    st_cs_f4(reinterpret_cast<float4 *>(p), make_float4(q[0], q[1], q[2], q[3]));
}
__device__ __forceinline__ unsigned short elem_bits(__half v) { return __half_as_ushort(v); }
__device__ __forceinline__ unsigned short elem_bits(__nv_bfloat16 v) { return __bfloat16_as_ushort(v); }
template <typename T>
__device__ __forceinline__ unsigned pack2(float a, float b) {
    return (unsigned)elem_bits(grid_elem<T>(a)) | (unsigned)elem_bits(grid_elem<T>(b)) << 16;
}
template <typename T>
__device__ __forceinline__ void st_cs_cells(T *p, const float (&q)[4]) {
    st_cs_u2(reinterpret_cast<uint2 *>(p), make_uint2(pack2<T>(q[0], q[1]), pack2<T>(q[2], q[3])));
}

template <typename T>
__global__ void __launch_bounds__(256) grid_fill_kernel(const int *__restrict__ cell2vid, const float *__restrict__ feat,
                                                        T *__restrict__ out, long long G, int C, int vcap, int cgroups) {
    const int f = blockIdx.z;
    const int cg = blockIdx.y;                      // channel group
    const int cper = C / cgroups;
    const long long cell = (long long)blockIdx.x * kCellsPerBlock + threadIdx.x * 4;
    if (cell >= G) return;
    const int *map = cell2vid + (size_t)f * G;
    const float *ff = feat + (size_t)f * vcap * C;
    T *o = out + ((size_t)f * C + (size_t)cg * cper) * G + cell;
    if (cell + 3 < G) {
        const int4 v = *reinterpret_cast<const int4 *>(map + cell);
        if ((v.x & v.y & v.z & v.w) < 0) {          // all four empty (-1): the common case, pure zero fill
            const float z4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
            for (int c = 0; c < cper; ++c) st_cs_cells(o + (size_t)c * G, z4);
        } else {
            const float *p0 = v.x >= 0 ? ff + (size_t)v.x * C + cg * cper : nullptr;
            const float *p1 = v.y >= 0 ? ff + (size_t)v.y * C + cg * cper : nullptr;
            const float *p2 = v.z >= 0 ? ff + (size_t)v.z * C + cg * cper : nullptr;
            const float *p3 = v.w >= 0 ? ff + (size_t)v.w * C + cg * cper : nullptr;
            for (int c = 0; c < cper; ++c) {
                float q[4];
                q[0] = p0 ? p0[c] : 0.f;
                q[1] = p1 ? p1[c] : 0.f;
                q[2] = p2 ? p2[c] : 0.f;
                q[3] = p3 ? p3[c] : 0.f;
                st_cs_cells(o + (size_t)c * G, q);
            }
        }
    } else {  // ragged tail (G not a multiple of 4)
        for (long long g = cell; g < G; ++g) {
            const int v = map[g];
            for (int c = 0; c < cper; ++c)
                out[((size_t)f * C + (size_t)cg * cper + c) * G + g] = grid_elem<T>(v >= 0 ? ff[(size_t)v * C + cg * cper + c] : 0.f);
        }
    }
}

// ---- plane-sequential variant (every grid whose cell count is a multiple of 32) ----------------------------
// HBM only reaches its write peak (7.5 TB/s measured for a plain fill) when the CTAs of a wave write one long
// contiguous region. So the launch order walks ONE channel plane at a time: blockIdx.x = run of kRunCells cells,
// blockIdx.y = channel, blockIdx.z = frame. Per run a CTA reads 1 KB of occupancy bits (not the 32 KB int map);
// only set bits (1.5 % of the cells) fetch a voxel id and its feature value. Every thread stores 16 bytes at a time:
// 4 fp32 cells, or 8 cells of a 16-bit grid (one occupancy byte); a run is 32 KB of grid in every element type.
constexpr int kRunBytes = 32768;
template <typename T> __host__ __device__ constexpr int run_cells() { return kRunBytes / (int)sizeof(T); }

// the store of grid_fill_planes_kernel. fp32: q holds the 4 cells. 16-bit: the kernel gathered nothing (lo == 0 below); all 8
// cells are gathered here in one block - both int4 halves of the map first, then every feature load - so an occupied store
// waits for one map and one feature latency, as in the fp32 kernel. (Issuing the loads of several stores before the first of
// them measured slower: the gathers become unconditional selects, and the registers cut the CTAs per SM.)
__device__ __forceinline__ void store_cells(float *o, float4 q, unsigned, const float *, const int *, int) {
    st_cs_f4(reinterpret_cast<float4 *>(o), q);
}
template <typename T>
__device__ __forceinline__ void store_cells(T *o, float4, unsigned nib, const float *ff, const int *map, int feat_vs) {
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (nib) {
        const int4 m0 = __ldg(reinterpret_cast<const int4 *>(map)), m1 = __ldg(reinterpret_cast<const int4 *>(map) + 1);
        const int id[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (nib & (1u << j)) v[j] = __ldg(ff + (size_t)id[j] * feat_vs);
    }
    st_cs_u4(reinterpret_cast<uint4 *>(o), make_uint4(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3]), pack2<T>(v[4], v[5]), pack2<T>(v[6], v[7])));
}

template <typename T>
__global__ void __launch_bounds__(256) grid_fill_planes_kernel(const unsigned *__restrict__ occ, const int *__restrict__ cell2vid,
                                                               const float *__restrict__ feat, long long feat_frame_stride,
                                                               int feat_vs, int feat_cs, T *__restrict__ out, long long G,
                                                               int C) {
    constexpr int V = 16 / sizeof(T);               // cells per thread and store
    constexpr int kStep = 256 * V;
    constexpr int kRunCells = run_cells<T>();
    const int f = blockIdx.z, c = blockIdx.y, tid = threadIdx.x;
    const long long cell0 = (long long)blockIdx.x * kRunCells;
    const unsigned *bits = occ + (size_t)f * (G / 32) + cell0 / 32;
    const int *map = cell2vid + (size_t)f * G + cell0;
    const float *ff = feat + (size_t)f * feat_frame_stride + (size_t)c * feat_cs;
    T *o = out + ((size_t)f * C + c) * G + cell0;
    const int nrun = (int)min((long long)kRunCells, G - cell0);
#pragma unroll
    for (int i = 0; i < kRunCells / kStep; ++i) {
        const int cell = i * kStep + tid * V;
        if (cell >= nrun) break;
        const unsigned nib = (__ldg(bits + (cell >> 5)) >> (cell & 31)) & ((1u << V) - 1u);
        const unsigned lo = V == 4 ? nib : 0u;      // a 16-bit grid gathers its 8 cells in store_cells
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lo) {
            if (lo & 1u) q.x = __ldg(ff + (size_t)__ldg(map + cell) * feat_vs);
            if (lo & 2u) q.y = __ldg(ff + (size_t)__ldg(map + cell + 1) * feat_vs);
            if (lo & 4u) q.z = __ldg(ff + (size_t)__ldg(map + cell + 2) * feat_vs);
            if (lo & 8u) q.w = __ldg(ff + (size_t)__ldg(map + cell + 3) * feat_vs);
        }
        store_cells(o + cell, q, nib, ff, map + cell, feat_vs);
    }
}

__global__ void __launch_bounds__(256) occ_from_map_kernel(const int *__restrict__ cell2vid, unsigned *__restrict__ occ, long long G) {
    const int f = blockIdx.y;
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per 32 cells
    if (w >= G / 32) return;
    const int4 *m = reinterpret_cast<const int4 *>(cell2vid + (size_t)f * G + w * 32);
    unsigned bits = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int4 v = __ldg(m + q);
        bits |= ((v.x >= 0 ? 1u : 0u) | (v.y >= 0 ? 2u : 0u) | (v.z >= 0 ? 4u : 0u) | (v.w >= 0 ? 8u : 0u)) << (q * 4);
    }
    occ[(size_t)f * (G / 32) + w] = bits;
}

__global__ void __launch_bounds__(256) map_from_idx_kernel(const long long *__restrict__ idx, long long N, int nx, int ny,
                                                           int nz, int *__restrict__ map) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    // idx row = [batch, ix, iy, iz] (train.py:119); grid is (nz, nx, ny) (VoxelNet.py:19-21)
    const long long ix = idx[n * 4 + 1], iy = idx[n * 4 + 2], iz = idx[n * 4 + 3];
    if (ix < 0 || ix >= nx || iy < 0 || iy >= ny || iz < 0 || iz >= nz) return;
    map[(iz * nx + ix) * ny + iy] = (int)n;
}

}  // namespace

int launch_occ_from_map(const int *cell2vid, unsigned *occ, int B, long long G, cudaStream_t st) {
    dim3 grid((unsigned)ceil_div(G / 32, 256), B);
    occ_from_map_kernel<<<grid, 256, 0, st>>>(cell2vid, occ, G);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_grid_fill_planes(const unsigned *occ, const int *cell2vid, const float *feat, long long feat_frame_stride, int feat_vs,
                            int feat_cs, void *out, int out_dtype, int B, long long G, int C, cudaStream_t st) {
    MVX_REQUIRE(G % 32 == 0, MVX_EINVAL, "plane-sequential grid fill needs a cell count divisible by 32");
    return with_grid_dtype(out_dtype, [&](auto t) {
        using T = decltype(t);
        dim3 grid((unsigned)ceil_div(G, run_cells<T>()), C, B);
        grid_fill_planes_kernel<T><<<grid, 256, 0, st>>>(occ, cell2vid, feat, feat_frame_stride, feat_vs, feat_cs, static_cast<T *>(out), G, C);
        MVX_LAUNCH_CHECK();
        return MVX_OK;
    });
}

int launch_grid_fill(const int *cell2vid, const float *feat, void *out, int out_dtype, int B, long long G, int C, int vcap,
                     cudaStream_t st) {
    const int cgroups = (C % 4 == 0) ? 4 : 1;
    dim3 grid((unsigned)ceil_div(G, kCellsPerBlock), cgroups, B);
    return with_grid_dtype(out_dtype, [&](auto t) {
        using T = decltype(t);
        grid_fill_kernel<T><<<grid, 256, 0, st>>>(cell2vid, feat, static_cast<T *>(out), G, C, vcap, cgroups);
        MVX_LAUNCH_CHECK();
        return MVX_OK;
    });
}

}  // namespace mvx

extern "C" int mvx_scatter_dense_typed(const float *feat, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny,
                                       int32_t nz, void *out, int32_t out_dtype, int32_t *map_ws, void *stream) {
    MVX_REQUIRE(mvx::grid_dtype_ok(out_dtype), MVX_EINVAL, MVX_GRID_DTYPE_MSG);
    MVX_REQUIRE(out && map_ws && nx > 0 && ny > 0 && nz > 0 && C > 0, MVX_EINVAL, "bad scatter argument");
    MVX_REQUIRE(N == 0 || (feat && idx), MVX_EINVAL, "null feat/idx");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long G = (long long)nx * ny * nz;
    MVX_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (G % 4 == 0), MVX_EINVAL,
                "grid must be 16-byte aligned with a cell count divisible by 4");
    MVX_CUDA_CHECK(cudaMemsetAsync(map_ws, 0xFF, (size_t)G * sizeof(int), st));
    if (N > 0) {
        mvx::map_from_idx_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(reinterpret_cast<const long long *>(idx), N, nx,
                                                                               ny, nz, map_ws);
        MVX_LAUNCH_CHECK();
    }
    if (G % 32 == 0) {  // map_ws holds G map entries followed by G/32 occupancy words
        unsigned *occ = reinterpret_cast<unsigned *>(map_ws + G);
        int rc = mvx::launch_occ_from_map(map_ws, occ, 1, G, st);
        if (rc) return rc;
        return mvx::launch_grid_fill_planes(occ, map_ws, feat, 0, C, 1, out, out_dtype, 1, G, C, st);
    }
    return mvx::launch_grid_fill(map_ws, feat, out, out_dtype, 1, G, C, (int)N, st);
}

extern "C" int mvx_scatter_dense(const float *feat, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny,
                                 int32_t nz, float *out, int32_t *map_ws, void *stream) {
    return mvx_scatter_dense_typed(feat, idx, N, C, nx, ny, nz, out, MVX_DTYPE_F32, map_ws, stream);
}
