// Stage 1 — deterministic GPU voxelization (replaces cpp/voxelutil.cpp:325-360 `_group` and the grouping loop
// of modules/data/Preprocessing.py:94-104).
//
// The reference is a sequential pass ("voxel list in first-occurrence order, first T points kept"). Atomic
// claims are order-free, so the parallel version canonicalises:
//   K1  insert   : point -> open-addressing hash slot (atomicCAS on a packed 63-bit key, warp-aggregated with
//                  __match_any_sync), atomicMin(first point index), atomicAdd(point count) per slot
//   K2  order    : flag = "I am my slot's first point"; exclusive scan over the point index  => voxel id in
//                  first-occurrence order (3-phase scan, no spin-waits)
//   K3  rank     : per-voxel segments (CSR) filled in arbitrary order, then rank-by-counting inside each
//                  segment => slot = #points of the same voxel with a smaller input index; keep slot < T
// Everything is batched over B frames (blockIdx.y = frame) and needs no host synchronisation.
#include "common.cuh"
#include "voxelize.cuh"

namespace mvx {

namespace {

constexpr unsigned long long kEmptyKey = 0xFFFFFFFFFFFFFFFFull;
constexpr int kKeyBias = 1 << 20;

__device__ __forceinline__ unsigned long long pack_key(int ix, int iy, int iz) {
    return ((unsigned long long)(unsigned)(ix + kKeyBias) << 42) | ((unsigned long long)(unsigned)(iy + kKeyBias) << 21) |
           (unsigned long long)(unsigned)(iz + kKeyBias);
}
__device__ __forceinline__ void unpack_key(unsigned long long k, int &ix, int &iy, int &iz) {
    ix = (int)((k >> 42) & 0x1FFFFF) - kKeyBias;
    iy = (int)((k >> 21) & 0x1FFFFF) - kKeyBias;
    iz = (int)(k & 0x1FFFFF) - kKeyBias;
}
__device__ __forceinline__ unsigned hash_key(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return (unsigned)k;
}

// ---- K1 -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vox_insert_kernel(VoxParams p) {
    const int f = blockIdx.y;
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x * blockDim.x >= P) return;  // whole block idle (uniform)
    const size_t gp = (size_t)p.fo.off[f] + i;
    unsigned long long key = kEmptyKey;
    bool in_frame = i < P, bad = false;
    if (in_frame) {
        int ix, iy, iz;
        if (p.cell_idx) {
            ix = p.cell_idx[gp * 3 + 0];
            iy = p.cell_idx[gp * 3 + 1];
            iz = p.cell_idx[gp * 3 + 2];
            bad = ix < -kKeyBias || ix >= kKeyBias || iy < -kKeyBias || iy >= kKeyBias || iz < -kKeyBias || iz >= kKeyBias;
        } else {
            float x, y, z;
            if (p.point_stride == 4) {  // coalesced 16-byte point loads
                const float4 q = __ldg(reinterpret_cast<const float4 *>(p.points) + gp);
                x = q.x, y = q.y, z = q.z;
            } else {
                const float *q = p.points + gp * p.point_stride;
                x = q[0], y = q[1], z = q[2];
            }
            bad = !vox_cell_index(p.lo, p.size, p.shape, x, y, z, ix, iy, iz);
        }
        if (!bad) key = pack_key(ix, iy, iz);
    }
    // warp-aggregated claim: lanes holding the same key elect their lowest lane (= lowest point index)
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int leader = __ffs(peers) - 1;
    const int lane = threadIdx.x & 31;
    int slot = -1;
    if (key != kEmptyKey && lane == leader) {
        unsigned long long *keys = p.hkeys + (size_t)f * p.H;
        unsigned h = hash_key(key) & (p.H - 1);
        while (true) {
            const unsigned long long prev = atomicCAS(&keys[h], kEmptyKey, key);
            if (prev == kEmptyKey || prev == key) break;
            h = (h + 1) & (p.H - 1);
        }
        slot = (int)h;
        atomicMin(p.hfirst + (size_t)f * p.H + h, (unsigned)i);
        atomicAdd(p.hcount + (size_t)f * p.H + h, (unsigned)__popc(peers));
    }
    slot = __shfl_sync(0xffffffffu, slot, leader);
    if (in_frame) {
        p.pslot[(size_t)f * p.cap + i] = bad ? -1 : slot;
        if (bad) atomicAdd(&p.counts[f * 4 + 2], 1);
    }
}

// ---- K2a: per-1024-point block, number of first-occurrence points ----------------------------------
__device__ __forceinline__ bool is_first(const VoxParams &p, int f, int i, int P, int &slot) {
    slot = -1;
    if (i >= P) return false;
    slot = p.pslot[(size_t)f * p.cap + i];
    return slot >= 0 && p.hfirst[(size_t)f * p.H + slot] == (unsigned)i;
}

__global__ void __launch_bounds__(1024) vox_flag_count_kernel(VoxParams p) {
    const int f = blockIdx.y;
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    if (blockIdx.x * 1024 >= P) return;
    int slot;
    const bool first = is_first(p, f, blockIdx.x * 1024 + threadIdx.x, P, slot);
    const int n = __syncthreads_count(first);
    if (threadIdx.x == 0) p.blocksum[f * p.nblk + blockIdx.x] = n;
}

// ---- K2b: exclusive scan of the block sums, one CTA per frame --------------------------------------
__global__ void __launch_bounds__(1024) vox_scan_blocks_kernel(VoxParams p) {
    const int f = blockIdx.x;
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    const int nb = (P + 1023) / 1024;
    int carry = 0;
    for (int base = 0; base < nb; base += 1024) {
        const int b = base + threadIdx.x;
        const int v = b < nb ? p.blocksum[f * p.nblk + b] : 0;
        int total;
        const int ex = block_exclusive_scan(v, &total);
        if (b < nb) p.blocksum[f * p.nblk + b] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) p.counts[f * 4 + 0] = carry;  // N_f
}

// ---- K2c: voxel ids in first-occurrence order ------------------------------------------------------
__global__ void __launch_bounds__(1024) vox_assign_vid_kernel(VoxParams p) {
    const int f = blockIdx.y;
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    if (blockIdx.x * 1024 >= P) return;
    int slot;
    const bool first = is_first(p, f, blockIdx.x * 1024 + threadIdx.x, P, slot);
    int total;
    const int ex = block_exclusive_scan(first ? 1 : 0, &total);
    if (!first) return;
    const int vid = p.blocksum[f * p.nblk + blockIdx.x] + ex;
    p.hvid[(size_t)f * p.H + slot] = vid;
    int ix, iy, iz;
    unpack_key(p.hkeys[(size_t)f * p.H + slot], ix, iy, iz);
    int cell = -1;
    if (p.have_grid && ix >= 0 && ix < p.shape[0] && iy >= 0 && iy < p.shape[1] && iz >= 0 && iz < p.shape[2])
        cell = (iz * p.shape[0] + ix) * p.shape[1] + iy;  // dense grid is (nz, nx, ny) (VoxelNet.py:19-21)
    reinterpret_cast<int4 *>(p.out.vox_coord)[(size_t)f * p.cap + vid] = make_int4(ix, iy, iz, cell);
    p.vox_total[(size_t)f * p.cap + vid] = (int)p.hcount[(size_t)f * p.H + slot];
    if (p.out.cell2vid && cell >= 0) p.out.cell2vid[(size_t)f * p.G + cell] = vid;
}

// ---- K3a: per-voxel offsets (segment start, first compact row), one CTA per frame -------------------
__global__ void __launch_bounds__(1024) vox_scan_voxels_kernel(VoxParams p) {
    // One CTA per frame walks the N_f voxels; a thread takes FOUR consecutive voxels per round and the two running sums (all points /
    // kept points) scan together as one 64-bit value: 6 rounds of one block scan for ~21 000 voxels instead of 21 rounds of two (this
    // kernel was the longest of stage 1: 33 us on eight SMs).
    const int f = blockIdx.x;
    const int N = p.counts[f * 4 + 0];
    unsigned long long carry = 0ull;   // (segment offset << 32) | compact row
    int maxtot = 0;
    for (int base = 0; base < N; base += 4096) {
        const int v0 = base + threadIdx.x * 4;
        int tot[4], kept[4];
        unsigned long long mine = 0ull;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            tot[q] = v0 + q < N ? p.vox_total[(size_t)f * p.cap + v0 + q] : 0;
            kept[q] = min(tot[q], p.T);
            mine += ((unsigned long long)(unsigned)tot[q] << 32) | (unsigned)kept[q];
            maxtot = max(maxtot, tot[q]);
        }
        unsigned long long total;
        unsigned long long ex = carry + block_exclusive_scan_u64(mine, &total);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (v0 + q < N) {
                p.seg_off[(size_t)f * (p.cap + 1) + v0 + q] = (int)(ex >> 32);
                p.out.vox_row0[(size_t)f * (p.cap + 1) + v0 + q] = (int)(ex & 0xFFFFFFFFull);
                p.out.vox_cnt[(size_t)f * p.cap + v0 + q] = kept[q];
            }
            ex += ((unsigned long long)(unsigned)tot[q] << 32) | (unsigned)kept[q];
        }
        carry += total;
    }
    maxtot = __reduce_max_sync(0xffffffffu, maxtot);
    if ((threadIdx.x & 31) == 0 && maxtot > 0) atomicMax(&p.counts[f * 4 + 3], maxtot);
    if (threadIdx.x == 0) {
        p.seg_off[(size_t)f * (p.cap + 1) + N] = (int)(carry >> 32);
        p.out.vox_row0[(size_t)f * (p.cap + 1) + N] = (int)(carry & 0xFFFFFFFFull);
        p.counts[f * 4 + 1] = (int)(carry & 0xFFFFFFFFull);  // K_f
    }
}

// ---- K3b: fill the per-voxel segments (arbitrary order inside a segment) ----------------------------
__global__ void __launch_bounds__(256) vox_fill_segments_kernel(VoxParams p) {
    const int f = blockIdx.y;
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int slot = p.pslot[(size_t)f * p.cap + i];
    if (slot < 0) return;
    const int v = p.hvid[(size_t)f * p.H + slot];
    const int pos = atomicAdd(&p.cursor[(size_t)f * p.cap + v], 1);
    const int q = p.seg_off[(size_t)f * (p.cap + 1) + v] + pos;
    p.seg_pts[(size_t)f * p.cap + q] = i;
    p.seg_vid[(size_t)f * p.cap + q] = v;
}

// A voxel with more points than this is ranked by vox_rank_big_kernel (selection of the T smallest point indices by a CTA)
// instead of the per-point counting loop below, whose cost is quadratic in the points of a voxel: a parked sensor facing a
// wall (or an adversarial input) can put a whole sweep into one voxel - 120 000^2 compares would stall the frame for seconds.
constexpr int kRankDirect = 256;
constexpr int kBigCtas = 32;    // CTAs per frame that look for crowded voxels

// ---- K3c: canonical slot = rank of the point index inside its voxel; keep the first T ---------------
__global__ void __launch_bounds__(256) vox_rank_emit_kernel(VoxParams p) {
    const int f = blockIdx.y;
    const int N = p.counts[f * 4 + 0];
    const int nvalid = p.seg_off[(size_t)f * (p.cap + 1) + N];
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nvalid) return;
    const int *seg = p.seg_pts + (size_t)f * p.cap;
    const int i = seg[q];
    const int v = p.seg_vid[(size_t)f * p.cap + q];
    const int start = p.seg_off[(size_t)f * (p.cap + 1) + v];
    const int n = p.vox_total[(size_t)f * p.cap + v];
    if (n > kRankDirect) return;   // crowded voxel: vox_rank_big_kernel
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += seg[start + j] < i ? 1 : 0;
    if (rank < p.T) {
        const int row = p.out.vox_row0[(size_t)f * (p.cap + 1) + v] + rank;
        p.out.row_point[(size_t)f * p.cap + row] = i;
        p.out.row_vox[(size_t)f * p.cap + row] = v;
    }
}

// ---- K3d: crowded voxels (more than kRankDirect points): the T smallest point indices by bisection on the index value.
// CTA c of a frame takes the crowded voxels v with v % kBigCtas == c; per voxel ~17 counting passes over its segment
// (n loads each, 1024 threads) find the T-th smallest index, one more pass collects the T kept points, ranked among
// themselves. Linear in the points of the voxel; ordinary frames have no such voxel and the CTAs exit after one scan of
// the per-voxel totals.
__global__ void __launch_bounds__(1024) vox_rank_big_kernel(VoxParams p) {
    __shared__ int s_cnt, s_nbig;
    __shared__ int s_keep[1024];
    __shared__ int s_big[64];        // crowded voxels found in the current scan window
    const int f = blockIdx.y, tid = threadIdx.x;
    if (p.counts[f * 4 + 3] <= kRankDirect) return;   // no crowded voxel in this frame (max points per voxel, from K3a)
    const int N = p.counts[f * 4 + 0];
    const int P = p.fo.off[f + 1] - p.fo.off[f];
    const int *seg_all = p.seg_pts + (size_t)f * p.cap;
    const int T = p.T;   // <= 1024 (checked by vox_run)
    // CTA c scans the voxel windows c, c + kBigCtas, ... of 1024 voxels each, one voxel per thread
    for (int base = blockIdx.x * 1024; base < N; base += kBigCtas * 1024) {
        if (tid == 0) s_nbig = 0;
        __syncthreads();
        const int vv = base + tid;
        bool mine = vv < N && p.vox_total[(size_t)f * p.cap + vv] > kRankDirect;
        while (true) {   // at most 64 crowded voxels per round (a window holds at most cap / 256 = a few hundred)
            if (mine) {
                const int k = atomicAdd(&s_nbig, 1);
                if (k < 64) s_big[k] = vv, mine = false;
            }
            __syncthreads();
            const int nbig = min(s_nbig, 64);
            for (int b = 0; b < nbig; ++b) {
                const int v = s_big[b];
                const int n = p.vox_total[(size_t)f * p.cap + v];
                const int *seg = seg_all + p.seg_off[(size_t)f * (p.cap + 1) + v];
                // smallest x with #{idx <= x} >= T  (indices are distinct, so exactly min(n, T) of them are <= x)
                int lo = 0, hi = P - 1;
                while (lo < hi) {
                    const int mid = lo + ((hi - lo) >> 1);
                    if (tid == 0) s_cnt = 0;
                    __syncthreads();
                    int c = 0;
                    for (int j = tid; j < n; j += 1024) c += seg[j] <= mid ? 1 : 0;
                    c = __reduce_add_sync(0xffffffffu, c);
                    if ((tid & 31) == 0 && c) atomicAdd(&s_cnt, c);
                    __syncthreads();
                    const int total = s_cnt;
                    __syncthreads();
                    if (total >= T) hi = mid; else lo = mid + 1;
                }
                if (tid == 0) s_cnt = 0;
                __syncthreads();
                for (int j = tid; j < n; j += 1024) {
                    const int i = seg[j];
                    if (i <= lo) s_keep[atomicAdd(&s_cnt, 1)] = i;
                }
                __syncthreads();
                const int kept = s_cnt;   // min(n, T)
                if (tid < kept) {
                    const int i = s_keep[tid];
                    int rank = 0;
                    for (int j = 0; j < kept; ++j) rank += s_keep[j] < i ? 1 : 0;
                    const int row = p.out.vox_row0[(size_t)f * (p.cap + 1) + v] + rank;
                    p.out.row_point[(size_t)f * p.cap + row] = i;
                    p.out.row_vox[(size_t)f * p.cap + row] = v;
                }
                __syncthreads();
            }
            const int found = s_nbig;
            __syncthreads();
            if (found <= 64) break;
            if (tid == 0) s_nbig = 0;   // more than 64 in this window: another round for the ones that did not get a slot
            __syncthreads();
        }
    }
}

// ---- reference-layout emitters ----------------------------------------------------------------------
__global__ void __launch_bounds__(256)
group_emit7_kernel(const float *__restrict__ pts, int stride, int V, int T, const int *__restrict__ vox_coord,
                   const int *__restrict__ vox_cnt, const int *__restrict__ vox_row0, const int *__restrict__ row_point,
                   float *__restrict__ voxel, int64_t *x, int64_t *y, int64_t *z, int64_t *cnt) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)V * T * 7;
    if (e < V) {
        x[e] = vox_coord[e * 4 + 0];
        y[e] = vox_coord[e * 4 + 1];
        z[e] = vox_coord[e * 4 + 2];
        cnt[e] = vox_cnt[e];
    }
    if (e >= total) return;
    const int v = (int)(e / (T * 7));
    const int rem = (int)(e - (long long)v * T * 7);
    const int j = rem / 7, c = rem - j * 7;
    float val = 0.f;
    if (j < vox_cnt[v] && (c < 3 || c == 6)) {
        const int i = row_point[vox_row0[v] + j];
        val = pts[(size_t)i * stride + (c == 6 ? 3 : c)];
    }
    voxel[e] = val;
}

__global__ void __launch_bounds__(256)
group_emit9_kernel(const float *__restrict__ pts, int stride, int V, int T, const int *__restrict__ vox_coord,
                   const int *__restrict__ vox_cnt, const int *__restrict__ vox_row0, const int *__restrict__ row_point,
                   double *out64, float *out32, double *uidx) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (voxel, slot)
    if (e >= (long long)V * T) return;
    const int v = (int)(e / T), j = (int)(e - (long long)v * T);
    const int n = vox_cnt[v], r0 = vox_row0[v];
    if (uidx && j == 0) {
        uidx[v * 3 + 0] = vox_coord[v * 4 + 0];
        uidx[v * 3 + 1] = vox_coord[v * 4 + 1];
        uidx[v * 3 + 2] = vox_coord[v * 4 + 2];
    }
    // centroid over the kept points, fp64, slot order (Preprocessing.py:112-113; pad slots add +0)
    double sx = 0, sy = 0, sz = 0;
    for (int k = 0; k < n; ++k) {
        const float *q = pts + (size_t)row_point[r0 + k] * stride;
        sx += (double)q[0], sy += (double)q[1], sz += (double)q[2];
    }
    const double cx = sx / (double)n, cy = sy / (double)n, cz = sz / (double)n;
    double o[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (j < n) {
        const float *q = pts + (size_t)row_point[r0 + j] * stride;
        o[0] = q[0], o[1] = q[1], o[2] = q[2], o[6] = q[3];
        if (stride >= 6) o[7] = q[4], o[8] = q[5];
    }
    o[3] = o[0] - cx, o[4] = o[1] - cy, o[5] = o[2] - cz;  // ALL T slots, pads hold -centroid (Preprocessing.py:115)
#pragma unroll
    for (int c = 0; c < 9; ++c) {
        if (out64) out64[e * 9 + c] = o[c];
        if (out32) out32[e * 9 + c] = (float)o[c];
    }
}

}  // namespace

// ----------------------------------------------------------------------------------------------------
size_t vox_workspace_bytes(int B, int cap) {
    VoxLayout L = vox_layout(B, cap);
    return L.total;
}

VoxLayout vox_layout(int B, int cap) {
    VoxLayout L;
    unsigned H = 1024;
    while (H < 2u * (unsigned)cap) H <<= 1;
    L.H = H;
    L.nblk = (cap + 1023) / 1024;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t r = o;
        o += (bytes + 255) / 256 * 256;
        return r;
    };
    // 0xFF-initialised region
    L.ff_begin = o;
    L.hkeys = take((size_t)B * H * 8);
    L.hfirst = take((size_t)B * H * 4);
    L.ff_end = o;
    // zero-initialised region
    L.zero_begin = o;
    L.hcount = take((size_t)B * H * 4);
    L.cursor = take((size_t)B * cap * 4);
    L.zero_end = o;
    L.hvid = take((size_t)B * H * 4);
    L.pslot = take((size_t)B * cap * 4);
    L.blocksum = take((size_t)B * L.nblk * 4);
    L.vox_total = take((size_t)B * cap * 4);
    L.seg_off = take((size_t)B * (cap + 1) * 4);
    L.seg_pts = take((size_t)B * cap * 4);
    L.seg_vid = take((size_t)B * cap * 4);
    L.total = o;
    return L;
}

int vox_run(const mvx_grid_t *grid, int B, int cap, const float *points, int point_stride, const int32_t *pt_off_host,
            const int32_t *cell_idx, int T, const mvx_voxel_out_t *out, void *workspace, size_t workspace_bytes,
            cudaStream_t st) {
    MVX_REQUIRE(B >= 1 && B <= kMaxFrames, MVX_EINVAL, "B must be in [1,32]");
    MVX_REQUIRE(cap >= 128 && cap % 128 == 0, MVX_EINVAL, "cap must be a positive multiple of 128");
    MVX_REQUIRE(points || cell_idx, MVX_EINVAL, "points or cell_idx required");
    MVX_REQUIRE(grid || cell_idx, MVX_EINVAL, "a grid is required when cell_idx is NULL");
    MVX_REQUIRE(out && out->counts && out->vox_coord && out->vox_cnt && out->vox_row0 && out->row_point && out->row_vox,
                MVX_EINVAL, "null output pointer");
    MVX_REQUIRE(!out->cell2vid || grid, MVX_EINVAL, "cell2vid needs a grid");
    MVX_REQUIRE(T >= 1 && T <= 1024, MVX_EINVAL, "T must be in [1, 1024]");
    VoxLayout L = vox_layout(B, cap);
    MVX_REQUIRE(workspace && workspace_bytes >= L.total, MVX_ESPACE, "voxelize workspace too small");

    VoxParams p{};
    int maxP = 0;
    for (int f = 0; f <= B; ++f) p.fo.off[f] = pt_off_host[f];
    for (int f = 0; f < B; ++f) {
        const int P = pt_off_host[f + 1] - pt_off_host[f];
        MVX_REQUIRE(P >= 0 && P <= cap, MVX_ESPACE, "frame has more points than cap");
        maxP = P > maxP ? P : maxP;
    }
    char *ws = static_cast<char *>(workspace);
    p.points = points, p.point_stride = point_stride, p.cell_idx = cell_idx;
    p.have_grid = grid != nullptr;
    p.G = 0;
    if (grid) {
        for (int d = 0; d < 3; ++d) p.lo[d] = grid->range_lo[d], p.size[d] = grid->voxel_size[d], p.shape[d] = grid->shape[d];
        p.G = (long long)grid->shape[0] * grid->shape[1] * grid->shape[2];
        MVX_REQUIRE(grid->shape[0] < kKeyBias && grid->shape[1] < kKeyBias && grid->shape[2] < kKeyBias, MVX_EINVAL,
                    "grid too large");
    }
    p.T = T, p.cap = cap, p.H = L.H, p.nblk = L.nblk;
    p.hkeys = reinterpret_cast<unsigned long long *>(ws + L.hkeys);
    p.hfirst = reinterpret_cast<unsigned *>(ws + L.hfirst);
    p.hcount = reinterpret_cast<unsigned *>(ws + L.hcount);
    p.hvid = reinterpret_cast<int *>(ws + L.hvid);
    p.pslot = reinterpret_cast<int *>(ws + L.pslot);
    p.blocksum = reinterpret_cast<int *>(ws + L.blocksum);
    p.vox_total = reinterpret_cast<int *>(ws + L.vox_total);
    p.seg_off = reinterpret_cast<int *>(ws + L.seg_off);
    p.cursor = reinterpret_cast<int *>(ws + L.cursor);
    p.seg_pts = reinterpret_cast<int *>(ws + L.seg_pts);
    p.seg_vid = reinterpret_cast<int *>(ws + L.seg_vid);
    p.counts = out->counts;
    p.out = *out;

    MVX_CUDA_CHECK(cudaMemsetAsync(ws + L.ff_begin, 0xFF, L.ff_end - L.ff_begin, st));
    MVX_CUDA_CHECK(cudaMemsetAsync(ws + L.zero_begin, 0, L.zero_end - L.zero_begin, st));
    MVX_CUDA_CHECK(cudaMemsetAsync(out->counts, 0, (size_t)B * 4 * sizeof(int), st));
    if (out->cell2vid) MVX_CUDA_CHECK(cudaMemsetAsync(out->cell2vid, 0xFF, (size_t)B * p.G * sizeof(int), st));
    if (maxP == 0) {  // empty batch: N = K = 0 everywhere, row0[0] = 0
        MVX_CUDA_CHECK(cudaMemsetAsync(out->vox_row0, 0, (size_t)B * (cap + 1) * sizeof(int), st));
        return MVX_OK;
    }
    const dim3 g256((maxP + 255) / 256, B), g1024((maxP + 1023) / 1024, B);
    vox_insert_kernel<<<g256, 256, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_flag_count_kernel<<<g1024, 1024, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_scan_blocks_kernel<<<B, 1024, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_assign_vid_kernel<<<g1024, 1024, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_scan_voxels_kernel<<<B, 1024, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_fill_segments_kernel<<<g256, 256, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    vox_rank_emit_kernel<<<g256, 256, 0, st>>>(p);
    MVX_LAUNCH_CHECK();
    if (maxP > kRankDirect) {   // a voxel can only be crowded if the frame has that many points
        vox_rank_big_kernel<<<dim3(kBigCtas, B), 1024, 0, st>>>(p);
        MVX_LAUNCH_CHECK();
    }
    return MVX_OK;
}

}  // namespace mvx

// ---- C ABI -------------------------------------------------------------------------------------------
extern "C" int mvx_voxelize_workspace_bytes(int32_t B, int32_t cap, size_t *bytes) {
    if (!bytes || B < 1 || cap < 128) return MVX_EINVAL;
    *bytes = mvx::vox_workspace_bytes(B, cap);
    return MVX_OK;
}

extern "C" int mvx_voxelize(const mvx_grid_t *grid, int32_t B, int32_t cap, const float *points, int32_t point_stride,
                            const int32_t *pt_off_host, const int32_t *cell_idx, int32_t T, const mvx_voxel_out_t *out,
                            void *workspace, size_t workspace_bytes, void *stream) {
    if (!pt_off_host) return MVX_EINVAL;
    return mvx::vox_run(grid, B, cap, points, point_stride, pt_off_host, cell_idx, T, out, workspace, workspace_bytes,
                        static_cast<cudaStream_t>(stream));
}

extern "C" int mvx_group_emit7(const float *points, int32_t point_stride, int32_t V, int32_t T, const int32_t *vox_coord,
                               const int32_t *vox_cnt, const int32_t *vox_row0, const int32_t *row_point, float *voxel,
                               int64_t *x, int64_t *y, int64_t *z, int64_t *cnt, void *stream) {
    if (V == 0) return MVX_OK;
    MVX_REQUIRE(points && voxel && x && y && z && cnt && V > 0 && T > 0, MVX_EINVAL, "bad emit7 argument");
    const long long total = (long long)V * T * 7;
    mvx::group_emit7_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        points, point_stride, V, T, vox_coord, vox_cnt, vox_row0, row_point, voxel, x, y, z, cnt);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

extern "C" int mvx_group_emit9(const float *points, int32_t point_stride, int32_t V, int32_t T, const int32_t *vox_coord,
                               const int32_t *vox_cnt, const int32_t *vox_row0, const int32_t *row_point, double *out_f64,
                               float *out_f32, double *uidx_f64, void *stream) {
    if (V == 0) return MVX_OK;
    MVX_REQUIRE(points && (out_f64 || out_f32) && V > 0 && T > 0, MVX_EINVAL, "bad emit9 argument");
    const long long total = (long long)V * T;
    mvx::group_emit9_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        points, point_stride, V, T, vox_coord, vox_cnt, vox_row0, row_point, out_f64, out_f32, uidx_f64);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}
