// Stage 4 — dense middle-layer grid (modules/voxelnet/VoxelNet.py:16-22 `reindex`).
// The reference zero-fills 721 MB and then scatters N*128 isolated 4-byte values (stride G between channels).
// Here the grid is produced in ONE streaming pass: every CTA owns a run of cells, reads the dense
// cell -> voxel map (int32, L2 resident) and writes each channel plane with coalesced 16-byte evict-first
// stores: value = map < 0 ? 0 : feat[vid][c].  HBM traffic = the grid once + the map.
#include "scatter.cuh"

namespace mvx {

namespace {

constexpr int kCellsPerBlock = 1024;  // 256 threads x 4 consecutive cells

__global__ void __launch_bounds__(256) grid_fill_kernel(const int *__restrict__ cell2vid, const float *__restrict__ feat,
                                                        float *__restrict__ out, long long G, int C, int vcap, int cgroups) {
    const int f = blockIdx.z;
    const int cg = blockIdx.y;                      // channel group
    const int cper = C / cgroups;
    const long long cell = (long long)blockIdx.x * kCellsPerBlock + threadIdx.x * 4;
    if (cell >= G) return;
    const int *map = cell2vid + (size_t)f * G;
    const float *ff = feat + (size_t)f * vcap * C;
    float *o = out + ((size_t)f * C + (size_t)cg * cper) * G + cell;
    if (cell + 3 < G) {
        const int4 v = *reinterpret_cast<const int4 *>(map + cell);
        if ((v.x & v.y & v.z & v.w) < 0) {          // all four empty (-1): the common case, pure zero fill
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
            for (int c = 0; c < cper; ++c) st_cs_f4(reinterpret_cast<float4 *>(o + (size_t)c * G), z4);
        } else {
            const float *p0 = v.x >= 0 ? ff + (size_t)v.x * C + cg * cper : nullptr;
            const float *p1 = v.y >= 0 ? ff + (size_t)v.y * C + cg * cper : nullptr;
            const float *p2 = v.z >= 0 ? ff + (size_t)v.z * C + cg * cper : nullptr;
            const float *p3 = v.w >= 0 ? ff + (size_t)v.w * C + cg * cper : nullptr;
            for (int c = 0; c < cper; ++c) {
                float4 q;
                q.x = p0 ? p0[c] : 0.f;
                q.y = p1 ? p1[c] : 0.f;
                q.z = p2 ? p2[c] : 0.f;
                q.w = p3 ? p3[c] : 0.f;
                st_cs_f4(reinterpret_cast<float4 *>(o + (size_t)c * G), q);
            }
        }
    } else {  // ragged tail (G not a multiple of 4)
        for (long long g = cell; g < G; ++g) {
            const int v = map[g];
            for (int c = 0; c < cper; ++c) out[((size_t)f * C + (size_t)cg * cper + c) * G + g] = v >= 0 ? ff[(size_t)v * C + cg * cper + c] : 0.f;
        }
    }
}

// ---- plane-sequential variant (every grid whose cell count is a multiple of 32) ----------------------------
// HBM only reaches its write peak (7.5 TB/s measured for a plain fill) when the CTAs of a wave write one long
// contiguous region. So the launch order walks ONE channel plane at a time: blockIdx.x = 32 KB run of cells,
// blockIdx.y = channel, blockIdx.z = frame. Per run a CTA reads 1 KB of occupancy bits (not the 32 KB int map);
// only set bits (1.5 % of the cells) fetch a voxel id and its feature value.
constexpr int kRunCells = 8192;

__global__ void __launch_bounds__(256) grid_fill_planes_kernel(const unsigned *__restrict__ occ, const int *__restrict__ cell2vid,
                                                               const float *__restrict__ feat, long long feat_frame_stride,
                                                               int feat_vs, int feat_cs, float *__restrict__ out, long long G,
                                                               int C) {
    const int f = blockIdx.z, c = blockIdx.y, tid = threadIdx.x;
    const long long cell0 = (long long)blockIdx.x * kRunCells;
    const unsigned *bits = occ + (size_t)f * (G / 32) + cell0 / 32;
    const int *map = cell2vid + (size_t)f * G + cell0;
    const float *ff = feat + (size_t)f * feat_frame_stride + (size_t)c * feat_cs;
    float *o = out + ((size_t)f * C + c) * G + cell0;
    const int nrun = (int)min((long long)kRunCells, G - cell0);
#pragma unroll
    for (int i = 0; i < kRunCells / 1024; ++i) {
        const int cell = i * 1024 + tid * 4;
        if (cell >= nrun) break;
        const unsigned nib = (__ldg(bits + (cell >> 5)) >> (cell & 31)) & 0xFu;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (nib) {
            if (nib & 1u) q.x = __ldg(ff + (size_t)__ldg(map + cell) * feat_vs);
            if (nib & 2u) q.y = __ldg(ff + (size_t)__ldg(map + cell + 1) * feat_vs);
            if (nib & 4u) q.z = __ldg(ff + (size_t)__ldg(map + cell + 2) * feat_vs);
            if (nib & 8u) q.w = __ldg(ff + (size_t)__ldg(map + cell + 3) * feat_vs);
        }
        st_cs_f4(reinterpret_cast<float4 *>(o + cell), q);
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
                            int feat_cs, float *out, int B, long long G, int C, cudaStream_t st) {
    MVX_REQUIRE(G % 32 == 0, MVX_EINVAL, "plane-sequential grid fill needs a cell count divisible by 32");
    dim3 grid((unsigned)ceil_div(G, kRunCells), C, B);
    grid_fill_planes_kernel<<<grid, 256, 0, st>>>(occ, cell2vid, feat, feat_frame_stride, feat_vs, feat_cs, out, G, C);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int launch_grid_fill(const int *cell2vid, const float *feat, float *out, int B, long long G, int C, int vcap, cudaStream_t st) {
    const int cgroups = (C % 4 == 0) ? 4 : 1;
    dim3 grid((unsigned)ceil_div(G, kCellsPerBlock), cgroups, B);
    grid_fill_kernel<<<grid, 256, 0, st>>>(cell2vid, feat, out, G, C, vcap, cgroups);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

}  // namespace mvx

extern "C" int mvx_scatter_dense(const float *feat, const int64_t *idx, int64_t N, int32_t C, int32_t nx, int32_t ny,
                                 int32_t nz, float *out, int32_t *map_ws, void *stream) {
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
        return mvx::launch_grid_fill_planes(occ, map_ws, feat, 0, C, 1, out, 1, G, C, st);
    }
    return mvx::launch_grid_fill(map_ws, feat, out, 1, G, C, (int)N, st);
}
