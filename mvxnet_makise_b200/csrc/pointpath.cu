// The fused batched point path: voxelize -> project + gather -> fusion/VFE layer stack -> dense grid, for B
// frames per call, stream-ordered, no host synchronisation (MVXNet.py:21-27 up to the CML input, with
// train.py:26-49's CPU half moved onto the GPU).
//
// Compact formulation (SURVEY.md §7 hard part 4): the reference pushes all R = N*T rows (86 % of them
// identical pad rows) through every layer. Here only the K kept points are rows; pad slots are one weighted
// row per frame (fusion stack, VFE1) or one per voxel (VFE2, FCN) whose multiplicity enters the BatchNorm
// sums and whose value joins the per-voxel max, so statistics and outputs equal the dense computation.
#include "gather.cuh"
#include "layers.cuh"
#include "scatter.cuh"
#include "voxelize.cuh"
#include "pointpath.cuh"

#include <vector>

namespace mvx {

const char *kRegionNames[R_COUNT] = {
    "vox_ws", "vox_coord", "vox_cnt", "vox_row0", "row_point", "row_vox", "cell2vid", "nhwc0", "nhwc1", "nhwc2",
    "vox8", "proj", "rowA_w", "A1", "Y1", "Y2", "Y3", "Y4", "Y5", "X6", "Y6", "X7", "Y7", "rowB_w", "rowB_v", "X8",
    "vfeat", "stats", "vmax6", "vmax7", "vmax8", "wpack", "occ", "vfeat_t", "Z", "bin_count", "bin_start", "perm", "rowmax", "chmax", "A1max", "tiles", "Y8"};

int make_layout(const mvx_pointpath_args_t *a, Layout &L) {
    MVX_REQUIRE(a, MVX_EINVAL, "null args");
    MVX_REQUIRE(a->B >= 1 && a->B <= kMaxFrames, MVX_EINVAL, "B must be in [1,32]");
    MVX_REQUIRE(a->cap >= 128 && a->cap % 128 == 0, MVX_EINVAL, "cap must be a positive multiple of 128");
    MVX_REQUIRE(a->map_c == 256, MVX_EINVAL, "map_c must be 256 (3 x 256 = the 768 inputs of fcn1)");
    MVX_REQUIRE(grid_dtype_ok(a->grid_dtype), MVX_EINVAL, MVX_GRID_DTYPE_MSG);   // element type of grid_out / d_grid
    const size_t B = a->B, cap = a->cap;
    L.capA = a->cap + 128;
    L.capB = 2 * a->cap;
    L.G = (long long)a->grid.shape[0] * a->grid.shape[1] * a->grid.shape[2];
    MVX_REQUIRE(L.G > 0 && L.G % 4 == 0, MVX_EINVAL, "grid cell count must be a positive multiple of 4");
    size_t o = 0;
    auto take = [&](Region r, size_t bytes) {
        L.off[r] = o;
        o += (bytes + 255) / 256 * 256;
    };
    take(R_VOXWS, vox_workspace_bytes(a->B, a->cap));
    take(R_VOX_COORD, B * cap * 16);
    take(R_VOX_CNT, B * cap * 4);
    take(R_VOX_ROW0, B * (cap + 1) * 4);
    take(R_ROW_POINT, B * cap * 4);
    take(R_ROW_VOX, B * cap * 4);
    take(R_CELL2VID, B * (size_t)L.G * 4);
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
        MVX_REQUIRE(a->map_h[l] > 0 && a->map_w[l] > 0, MVX_EINVAL, "bad FPN map extent");
        take((Region)(R_NHWC0 + l), (size_t)round_up((int64_t)B * a->map_h[l] * a->map_w[l], 256) * a->map_c * 4);   // NHWC fp32, or the packed fp16 hi/lo image
    }
    const size_t capA = L.capA, capB = L.capB;
    take(R_VOX8, B * capA * 8 * 4);
    take(R_PROJ, B * capA * 2 * 4);
    take(R_ROWA_W, B * capA * 4);
    take(R_A1, B * capA * 768 * 4);
    take(R_Y1, B * capA * 768 * 4);
    take(R_Y2, B * capA * 128 * 4);
    take(R_Y3, B * capA * 128 * 4);
    take(R_Y4, B * capA * 16 * 4);
    take(R_Y5, B * capA * 16 * 4);
    take(R_X6, B * capA * 32 * 4);
    take(R_Y6, B * capA * 16 * 4);
    take(R_X7, B * capB * 32 * 4);
    take(R_Y7, B * capB * 64 * 4);
    take(R_ROWB_W, B * capB * 4);
    take(R_ROWB_V, B * capB * 4);
    take(R_X8, B * capB * 128 * 4);
    take(R_VFEAT, B * cap * 128 * 4);
    take(R_STATS, (size_t)MVX_NUM_LAYERS * B * kStatStride * 8);
    take(R_VMAX6, B * cap * 16 * 4);
    take(R_VMAX7, B * cap * 64 * 4);
    take(R_VMAX8, B * cap * 128 * 4);
    take(R_WPACK, tc_wpack_bytes(768, 768));
    take(R_OCC, B * (size_t)(L.G / 32 + 1) * 4);
    take(R_VFEAT_T, B * cap * 128 * 4);
    {   // per-pixel fcn1 products of the three FPN levels, (B, HW_l, 768) each
        size_t px = 0;
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) px += (size_t)a->map_h[l] * a->map_w[l];
        take(R_Z, B * px * 768 * 4);
        const size_t nb = combine_bins(a->map_h[0], a->map_w[0]);
        take(R_BINCNT, B * (nb + 1) * 4);
        take(R_BINSTART, B * (nb + 2) * 4);
        take(R_PERM, B * capA * 4);
        take(R_ROWMAX, B * px * 4);
        take(R_CHMAX, B * 768 * 4);
        take(R_A1MAX, B * capA * 4);
        int ntiles[MVX_NUM_LEVELS];
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) ntiles[l] = (int)ceil_div((long long)B * a->map_h[l] * a->map_w[l], kPixTileRows);
        take(R_TILES, pixel_tiles_bytes(ntiles));   // active pixel tiles of the pixel GEMM: bitmap, list, counts
    }
    L.total = o;
    take(R_Y8, B * capB * 128 * 4);   // last region: only present in a training workspace
    L.total_train = o;
    return MVX_OK;
}

// ---- optional CUDA-event timing of the stages (bench.py roofline leg) -------------------------------------
enum Segment {
    S_VOXELIZE = 0, S_NHWC, S_ROWS, S_GATHER, S_CLEAR, S_FCN1, S_CONV1, S_FCN2, S_CONV2, S_FCN3, S_PREP1, S_VFE1,
    S_PREP2, S_VFE2, S_PREP3, S_FCN, S_VFEAT, S_GRID, S_COUNT
};
static_assert(S_COUNT <= MVX_NUM_SEGMENTS, "too many segments");
const char *kSegmentNames[S_COUNT] = {"voxelize", "maps_nhwc", "rows_build", "gather", "clear", "fcn1", "conv1", "fcn2",
                                      "conv2", "fcn3", "prep_vfe1", "vfe1", "prep_vfe2", "vfe2", "prep_fcn", "fcn",
                                      "finalize_vfeat", "grid_fill"};
struct Timing {
    std::vector<cudaEvent_t> ev;      // [calls][S_COUNT][2]: begin / end of every segment, recorded on the stream it runs on
    std::vector<unsigned> recorded;   // [calls] bit i: segment i was timed in this call
    int max_calls = 0, next = 0;
};
static Timing g_timing;

struct Stamp {
    cudaEvent_t *ev = nullptr;
    unsigned *rec = nullptr;
    cudaStream_t st;
    mutable int cur = -1;
    explicit Stamp(cudaStream_t s) : st(s) {
        if (g_timing.max_calls > 0 && g_timing.next < g_timing.max_calls) {
            rec = &g_timing.recorded[g_timing.next];
            *rec = 0;
            ev = &g_timing.ev[(size_t)g_timing.next++ * (S_COUNT * 2)];
        }
    }
    void begin(int i, cudaStream_t s) const {
        if (ev) cudaEventRecord(ev[2 * i], s), *rec |= 1u << i;
    }
    void end(int i, cudaStream_t s) const {
        if (ev) cudaEventRecord(ev[2 * i + 1], s);
    }
    // main-stream segments are back to back: mark(i) closes the running one and opens segment i (S_COUNT: just close)
    void mark(int i) const {
        if (!ev) return;
        if (cur >= 0) end(cur, st);
        cur = -1;
        if (i < S_COUNT) begin(i, st), cur = i;
    }
};

// the map branch (channels-last copy + per-pixel GEMM) does not depend on the point branch (voxelization, row build, row
// sort): it runs on a side stream, forked from and joined back into the caller's stream with events
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    int device = -1;
};
static int side_stream(SideStream **out) {
    static SideStream per_device[kMaxDevices];
    int dev = 0;
    MVX_CUDA_CHECK(cudaGetDevice(&dev));
    MVX_REQUIRE(dev >= 0 && dev < kMaxDevices, MVX_EINVAL, "device ordinal out of range");
    SideStream &s = per_device[dev];
    if (!s.stream) {
        MVX_CUDA_CHECK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        MVX_CUDA_CHECK(cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming));
        MVX_CUDA_CHECK(cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming));
        s.device = dev;
    }
    *out = &s;
    return MVX_OK;
}

// zero vmax rows [0, N_f) of each frame (bounded by the device-side voxel count, not by cap)
__global__ void __launch_bounds__(256) zero_vmax_kernel(const int *__restrict__ counts, int cap, int *__restrict__ v6,
                                                        int *__restrict__ v7, int *__restrict__ v8) {
    const int f = blockIdx.y;
    const long long N = counts[f * 4 + 0];
    const int4 z = make_int4(0, 0, 0, 0);
    int4 *p6 = reinterpret_cast<int4 *>(v6 + (size_t)f * cap * 16);
    int4 *p7 = reinterpret_cast<int4 *>(v7 + (size_t)f * cap * 64);
    int4 *p8 = reinterpret_cast<int4 *>(v8 + (size_t)f * cap * 128);
    const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long e = t0; e < N * 4; e += stride) p6[e] = z;
    for (long long e = t0; e < N * 16; e += stride) p7[e] = z;
    for (long long e = t0; e < N * 32; e += stride) p8[e] = z;
}

int pointpath_forward(const mvx_pointpath_args_t *a, bool train) {
    Layout L;
    int rc = make_layout(a, L);
    if (rc) return rc;
    MVX_REQUIRE(a->workspace && a->workspace_bytes >= (train ? L.total_train : L.total), MVX_ESPACE, "pointpath workspace too small");
    const bool dense_in = a->voxels_dense != nullptr || a->vox_off_host != nullptr;   // the reference's (voxels, idx) arguments instead of raw points
    MVX_REQUIRE(a->counts, MVX_EINVAL, "null counts pointer");
    if (!dense_in) {
        MVX_REQUIRE(a->pt_off_host && a->calib32, MVX_EINVAL, "null input pointer");
        MVX_REQUIRE(a->points || a->pt_off_host[a->B] == a->pt_off_host[0], MVX_EINVAL, "null points pointer");   // an all-empty batch may pass NULL
        MVX_REQUIRE(a->point_stride >= 4, MVX_EINVAL, "point_stride must be >= 4");
    }
    for (int l = 0; l < MVX_NUM_LEVELS; ++l) MVX_REQUIRE(a->maps[l], MVX_EINVAL, "null FPN map");
    for (int l = 0; l < MVX_NUM_LAYERS; ++l) MVX_REQUIRE(a->wt[l] && a->bias[l], MVX_EINVAL, "null layer weights");
    cudaStream_t st = static_cast<cudaStream_t>(a->stream);
    char *ws = static_cast<char *>(a->workspace);
    const int B = a->B, cap = a->cap, T = a->grid.T;
    auto F32 = [&](Region r) { return reinterpret_cast<float *>(ws + L.off[r]); };
    auto I32 = [&](Region r) { return reinterpret_cast<int *>(ws + L.off[r]); };

    const Stamp stamp(st);
    if (train) MVX_CUDA_CHECK(cudaMemsetAsync(I32(R_CHMAX), 0, (size_t)B * 768 * 4, st));
    // training keeps the gathered matrix A1 (dW1 = dpre1^T A1), so it always runs row-first
    const bool pixel_first = mvx::pixel_first(train);
    double *stats = reinterpret_cast<double *>(ws + L.off[R_STATS]);
    auto stat_of = [&](int layer) { return stats + (size_t)layer * B * kStatStride; };
    // NOTE: stats are stored [F][Cout][2] with the layer's own Cout as the frame stride

    // ---- map branch (independent of the points): channels-last copy, then in pixel-first mode Z_l = F_l W1_l^T ----------
    // forked onto a side stream so that the latency-bound point branch below (voxelization, row build, row sort) hides
    // under it; joined before the first kernel that needs both
    cudaStream_t ms = st;
    SideStream *side = nullptr;
    if (pixel_first && map_on_side_stream()) {
        rc = side_stream(&side);
        if (rc) return rc;
        ms = side->stream;
        MVX_CUDA_CHECK(cudaEventRecord(side->fork, st));
        MVX_CUDA_CHECK(cudaStreamWaitEvent(ms, side->fork, 0));
    }
    // bf16 mode (mvx_set_gemm_mode(6)): the two largest intermediates - the per-pixel products Z and the raw fcn1 rows Y1 - are
    // stored as bf16 (half the bytes written and read back); every sum in between stays fp32
    const bool bf16_mem = pixel_first && bf16_mode();
    auto z_at = [&](size_t elem_off) -> float * {   // element offset into Z, whatever its element size
        return bf16_mem ? reinterpret_cast<float *>(reinterpret_cast<uint16_t *>(ws + L.off[R_Z]) + elem_off) : F32(R_Z) + elem_off;
    };
    PixelTiles pt{};
    pixel_tiles_init(pt, B, a->map_h, a->map_w, ws + L.off[R_TILES]);
    auto map_branch = [&](MapSet &m) -> int {
        stamp.begin(S_NHWC, ms);
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
            m.h[l] = a->map_h[l], m.w[l] = a->map_w[l];
            m.rs_h[l] = a->imsize_h / (float)a->map_h[l];
            m.rs_w[l] = a->imsize_w / (float)a->map_w[l];
            m.nhwc[l] = F32((Region)(R_NHWC0 + l));
            m.frame_stride[l] = (size_t)a->map_h[l] * a->map_w[l] * a->map_c;
        }
        if (pixel_first) {   // which 256-row tiles of Z the combine can read: from the raw points and the calibration only
            TileMarkArgs tm{};
            if (!dense_in) {
                tm.points = a->points, tm.point_stride = a->point_stride;
                for (int f = 0; f <= B; ++f) tm.off[f] = a->pt_off_host[f];
                tm.calib32 = a->calib32, tm.point_calib = a->point_calib;
                tm.calib64 = a->calib64, tm.calib_f64 = a->calib64 ? a->calib_f64 : nullptr;   // as RowsParams below
                for (int d = 0; d < 3; ++d) tm.lo[d] = a->grid.range_lo[d], tm.size[d] = a->grid.voxel_size[d], tm.shape[d] = a->grid.shape[d];
                for (int l = 0; l < MVX_NUM_LEVELS; ++l) tm.h[l] = m.h[l], tm.w[l] = m.w[l], tm.rs_h[l] = m.rs_h[l], tm.rs_w[l] = m.rs_w[l];
                tm.eps = a->gather_eps;
            }
            int r = launch_pixel_tiles(tm, pt, B, dense_in, bf16_mem ? 2 : 4, ms);   // dense-voxel entry: no raw points, every tile is active
            if (r) return r;
        }
        size_t rowmax_off = 0;
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
            const int HW = a->map_h[l] * a->map_w[l];
            // pixel-first: the maps are written directly as the pre-packed 3xFP16 A operand of the pixel GEMM (no NHWC copy), in the
            // bf16 mode too (the persistent kernel is bound by its loads and stores, not by the MMAs; only Z is written as bf16)
            const int r = pixel_first ? launch_pack_maps_f16(a->maps[l], ws + L.off[R_NHWC0 + l], F32(R_ROWMAX) + rowmax_off, B, a->map_c, HW,
                                                             dense_in ? nullptr : pt.bits + pt.word0[l], ms)
                                      : launch_nchw_to_nhwc(a->maps[l], F32((Region)(R_NHWC0 + l)), B, a->map_c, HW, F32(R_ROWMAX) + rowmax_off,
                                                            train ? I32(R_CHMAX) + l * a->map_c : nullptr, MVX_NUM_LEVELS * a->map_c, ms);
            if (r) return r;
            rowmax_off += (size_t)B * HW;
        }
        stamp.end(S_NHWC, ms);
        if (!pixel_first) return MVX_OK;
        // Z_l = F_l W1[:, 256 l : 256 (l+1)]^T for the active pixel tiles of every level, zeros elsewhere (plain GEMM: no bias /
        // ReLU / statistics)
        stamp.begin(S_GATHER, ms);
        PixelGemmArgs pg{};
        size_t zoff = 0;
        for (int l = 0; l < MVX_NUM_LEVELS; ++l) {
            const long long px = (long long)B * a->map_h[l] * a->map_w[l];
            pg.a_pack[l] = ws + L.off[R_NHWC0 + l], pg.a_rowinv[l] = F32(R_ROWMAX) + zoff / 768;
            pg.Z[l] = z_at(zoff), pg.R[l] = px;
            zoff += (size_t)px * 768;
        }
        pg.Wt = a->wt[0], pg.Cin = a->map_c, pg.Cout = 768, pg.z_bf16 = bf16_mem;
        pg.list = pt.list, pg.meta = pt.meta, pg.n_entries = pt.tile0[MVX_NUM_LEVELS];
        int r = pixel_gemm_persistent() ? launch_pixel_gemm_levels(pg, F32(R_WPACK), ms) : launch_pixel_gemm_one_tile(pg, F32(R_WPACK), ms);
        if (r) return r;
        stamp.end(S_GATHER, ms);
        return MVX_OK;
    };
    MapSet m{};
    m.C = a->map_c;
    rc = map_branch(m);
    if (rc) return rc;
    if (side) MVX_CUDA_CHECK(cudaEventRecord(side->join, ms));

    // ---- point branch: stage 1 (voxelization), compact rows, clears, row sort -----------------------------------------------
    stamp.mark(S_VOXELIZE);
    mvx_voxel_out_t vo{};
    vo.counts = a->counts;
    vo.vox_coord = I32(R_VOX_COORD), vo.vox_cnt = I32(R_VOX_CNT), vo.vox_row0 = I32(R_VOX_ROW0);
    vo.row_point = I32(R_ROW_POINT), vo.row_vox = I32(R_ROW_VOX), vo.cell2vid = I32(R_CELL2VID);
    if (dense_in) {   // stage 1 and the projection were done by the caller (pre.group on the host): compact the dense tensor
        rc = dense_rows_run(a, L.capA, L.G, vo.vox_coord, vo.vox_cnt, vo.vox_row0, vo.row_point, vo.row_vox, vo.cell2vid, F32(R_VOX8),
                            F32(R_PROJ), F32(R_ROWA_W), st);
        if (rc) return rc;
    } else {
    rc = vox_run(&a->grid, B, cap, a->points, a->point_stride, a->pt_off_host, nullptr, T, &vo, ws + L.off[R_VOXWS],
                 vox_workspace_bytes(B, cap), st);
    if (rc) return rc;
    stamp.mark(S_ROWS);
    RowsParams rp{};
    rp.B = B, rp.cap = cap, rp.capA = L.capA, rp.T = T;
    rp.points = a->points, rp.point_stride = a->point_stride;
    for (int f = 0; f <= B; ++f) rp.off[f] = a->pt_off_host[f];
    rp.calib32 = a->calib32, rp.point_calib = a->point_calib, rp.counts = a->counts;
    rp.calib64 = a->calib64, rp.calib_f64 = a->calib64 ? a->calib_f64 : nullptr;
    rp.vox_cnt = vo.vox_cnt, rp.vox_row0 = vo.vox_row0, rp.row_point = vo.row_point, rp.row_vox = vo.row_vox;
    rp.vox8 = F32(R_VOX8), rp.proj = F32(R_PROJ), rp.rowA_w = F32(R_ROWA_W);
    rc = launch_rows_build(rp, st);
    if (rc) return rc;
    }

    stamp.mark(S_CLEAR);
    MVX_CUDA_CHECK(cudaMemsetAsync(stats, 0, (size_t)MVX_NUM_LAYERS * B * kStatStride * 8, st));
    zero_vmax_kernel<<<dim3(kSMs, B), 256, 0, st>>>(a->counts, cap, I32(R_VMAX6), I32(R_VMAX7), I32(R_VMAX8));
    MVX_LAUNCH_CHECK();
    CombineArgs ca{};
    if (pixel_first) {
        size_t zoff = 0;
        for (int lv = 0; lv < MVX_NUM_LEVELS; ++lv) {
            ca.Z[lv] = z_at(zoff);
            ca.frame_stride[lv] = (size_t)a->map_h[lv] * a->map_w[lv] * 768;
            ca.h[lv] = m.h[lv], ca.w[lv] = m.w[lv], ca.rs_h[lv] = m.rs_h[lv], ca.rs_w[lv] = m.rs_w[lv];
            zoff += (size_t)B * a->map_h[lv] * a->map_w[lv] * 768;
        }
        ca.capA = L.capA, ca.counts = a->counts, ca.vox8 = F32(R_VOX8), ca.proj = F32(R_PROJ), ca.row_w = F32(R_ROWA_W);
        ca.eps = a->gather_eps, ca.bias = a->bias[0], ca.Y1 = F32(R_Y1), ca.out_stats = stat_of(0);
        ca.bin_count = I32(R_BINCNT), ca.bin_start = I32(R_BINSTART), ca.perm = I32(R_PERM);
        ca.nbins = combine_bins(a->map_h[0], a->map_w[0]);
        ca.z_bf16 = ca.y1_bf16 = bf16_mem;
        rc = launch_combine_sort(ca, B, st);      // needs only the projections: still part of the point branch
        if (rc) return rc;
    }
    stamp.mark(S_COUNT);   // close the running segment before the join wait (it must not absorb the map branch's time)
    if (side) MVX_CUDA_CHECK(cudaStreamWaitEvent(st, side->join, 0));   // ---- join: both branches done ----

    // ---- stage 2b / 3 -------------------------------------------------------------------------------------------------------
    if (!pixel_first) {
        stamp.mark(S_GATHER);
        rc = launch_gather_rows(m, B, L.capA, a->counts, F32(R_VOX8), F32(R_PROJ), a->gather_eps, F32(R_A1), F32(R_A1MAX), st);
        if (rc) return rc;
    }
    const float *xin[5] = {F32(R_A1), F32(R_Y1), F32(R_Y2), F32(R_Y3), F32(R_Y4)};
    float *yout[5] = {F32(R_Y1), F32(R_Y2), F32(R_Y3), F32(R_Y4), F32(R_Y5)};
    for (int l = 0; l < 5; ++l) {  // fusion stack: fcn1 conv1 fcn2 conv2 fcn3 (Pipe.py:94-104)
        stamp.mark(S_FCN1 + l);
        if (l == 0 && pixel_first) {
            rc = launch_combine_rows(ca, B, st);
            if (rc) return rc;
            continue;
        }
        LayerArgs la{};
        la.X = xin[l], la.ldx = kCin[l], la.Cin = kCin[l], la.Wt = a->wt[l], la.bias = a->bias[l], la.Cout = kCout[l];
        la.Y = yout[l], la.ldy = kCout[l];
        la.in_stats = l == 0 ? nullptr : stat_of(l - 1);
        la.out_stats = stat_of(l);
        la.row_w = F32(R_ROWA_W), la.counts = a->counts, la.rows_mode = 1, la.rowcap = L.capA, la.vcap = cap, la.T = T;
        la.eps = a->bn_eps;
        la.f16_ok = 1;       // BatchNorm-ed inputs; fcn1 row-first reads raw gathered features: per-row power-of-two scaling
        if (l == 0) la.row_max = F32(R_A1MAX);
        if (l == 1) la.x_bf16 = bf16_mem;   // conv1 reads the bf16 Y1 of the combine kernel
        rc = launch_layer_auto(la, B, F32(R_WPACK), st);
        if (rc) return rc;
    }
    VfePrepArgs vp{};
    vp.B = B, vp.cap = cap, vp.capA = L.capA, vp.capB = L.capB, vp.T = T;
    vp.counts = a->counts, vp.vox_cnt = vo.vox_cnt, vp.row_vox = vo.row_vox;
    vp.vox8 = F32(R_VOX8), vp.Y5 = F32(R_Y5), vp.X6 = F32(R_X6);
    vp.Y6 = F32(R_Y6), vp.vmax6 = I32(R_VMAX6), vp.X7 = F32(R_X7), vp.rowB_w = F32(R_ROWB_W), vp.rowB_v = I32(R_ROWB_V);
    vp.Y7 = F32(R_Y7), vp.vmax7 = I32(R_VMAX7), vp.X8 = F32(R_X8);
    vp.vmax8 = I32(R_VMAX8), vp.vfeat = F32(R_VFEAT);
    vp.vfeat_t = (L.G % 32 == 0 && a->grid_out) ? F32(R_VFEAT_T) : nullptr;
    vp.n5 = NormSrc{stat_of(4), a->counts, 0, T, a->bn_eps};
    vp.n6 = NormSrc{stat_of(5), a->counts, 0, T, a->bn_eps};
    vp.n7 = NormSrc{stat_of(6), a->counts, 0, T, a->bn_eps};
    vp.n8 = NormSrc{stat_of(7), a->counts, 0, T, a->bn_eps};

    // inference: VFE1 / VFE2 build their input rows on the fly (fused loaders of the SIMT kernel) instead of reading the X6 / X7 matrices that
    // prep_vfe1 / prep_vfe2 materialise; training keeps X6 / X7 (dW = dpre^T X)
    const bool fuse_vfe = !train && vfe_fused();
    stamp.mark(S_PREP1);
    if (!fuse_vfe) {
        rc = launch_prep_vfe1(vp, st);
        if (rc) return rc;
    }
    {  // VFE1's FCN (23 -> 16) + per-voxel max (voxelnet/Pipe.py:12-18)
        stamp.mark(S_VFE1);
        LayerArgs la{};
        la.X = F32(R_X6), la.ldx = 32, la.Cin = 32, la.Wt = a->wt[5], la.bias = a->bias[5], la.Cout = 16;
        la.Y = F32(R_Y6), la.ldy = 16, la.out_stats = stat_of(5), la.vmax = I32(R_VMAX6);
        la.row_w = F32(R_ROWA_W), la.row_v = vo.row_vox, la.rowv_cap = cap, la.counts = a->counts, la.rows_mode = 1;
        la.rowcap = L.capA, la.vcap = cap, la.T = T, la.eps = a->bn_eps;
        if (fuse_vfe) {
            RowFuseArgs z{};
            z.vox8 = F32(R_VOX8), z.Y = F32(R_Y5), z.in_stats = stat_of(4), z.cap = cap, z.capA = L.capA;
            rc = launch_vfe1_fused(la, z, B, st);
        } else {
            rc = launch_layer_auto(la, B, F32(R_WPACK), st);
        }
        if (rc) return rc;
    }
    stamp.mark(S_PREP2);
    if (!fuse_vfe) {
        rc = launch_prep_vfe2(vp, st);
        if (rc) return rc;
    }
    {  // VFE2's FCN (32 -> 64) + per-voxel max; rows = K_f kept points + one weighted pad row per voxel
        stamp.mark(S_VFE2);
        LayerArgs la{};
        la.X = F32(R_X7), la.ldx = 32, la.Cin = 32, la.Wt = a->wt[6], la.bias = a->bias[6], la.Cout = 64;
        la.Y = F32(R_Y7), la.ldy = 64, la.out_stats = stat_of(6), la.vmax = I32(R_VMAX7);
        la.row_w = F32(R_ROWB_W), la.row_v = I32(R_ROWB_V), la.rowv_cap = L.capB, la.counts = a->counts, la.rows_mode = 2;
        la.rowcap = L.capB, la.vcap = cap, la.T = T, la.eps = a->bn_eps;
        if (fuse_vfe) {
            RowFuseArgs z{};
            z.Y = F32(R_Y6), z.in_stats = stat_of(5), z.vmax = I32(R_VMAX6), z.vox_cnt = vo.vox_cnt, z.row_vox = vo.row_vox;
            z.rowB_w = F32(R_ROWB_W), z.rowB_v = I32(R_ROWB_V), z.cap = cap, z.capA = L.capA;
            rc = launch_vfe2_fused(la, z, B, st);
        } else {
            rc = launch_layer_auto(la, B, F32(R_WPACK), st);
        }
        if (rc) return rc;
    }
    stamp.mark(S_PREP3);
    // inference: the concat [norm7(Y7) | norm7(max7)] that prep_fcn materialises as X8 is built by the FCN's own
    // A-producer instead (16-bit tensor-core kernel); training keeps X8 (dW8 = dpre8^T X8)
    const bool fuse_cat = !train && !simt_only();
    if (!fuse_cat) {
        rc = launch_prep_fcn(vp, st);
        if (rc) return rc;
    }
    {  // FCN(128,128) + max over T (VoxelNet.py:27-32): only the per-voxel max and the statistics are kept
        stamp.mark(S_FCN);
        LayerArgs la{};
        la.X = F32(R_X8), la.ldx = 128, la.Cin = 128, la.Wt = a->wt[7], la.bias = a->bias[7], la.Cout = 128;
        if (fuse_cat) {
            la.X = F32(R_Y7), la.ldx = 64, la.in_stats = stat_of(6), la.in_C = 64;
            la.X2 = I32(R_VMAX7), la.x2_cols = 64, la.cat_row_vox = vo.row_vox, la.cat_rowv_cap = cap;
        }
        la.Y = train ? F32(R_Y8) : nullptr, la.ldy = train ? 128 : 0, la.out_stats = stat_of(7), la.vmax = I32(R_VMAX8);
        la.row_w = F32(R_ROWB_W), la.row_v = I32(R_ROWB_V), la.rowv_cap = L.capB, la.counts = a->counts, la.rows_mode = 2;
        la.rowcap = L.capB, la.vcap = cap, la.T = T, la.eps = a->bn_eps;
        la.f16_ok = 1;       // X8 is stored BatchNorm-ed
        rc = launch_layer_auto(la, B, F32(R_WPACK), st);
        if (rc) return rc;
    }
    stamp.mark(S_VFEAT);
    rc = launch_finalize_vfeat(vp, st);   // vfeat[v] = BN8(max_T) : the (N,128) voxel features in reference voxel order
    if (rc) return rc;

    stamp.mark(S_GRID);
    // ---- stage 4 ----------------------------------------------------------------------------------------
    if (a->grid_out) {
        MVX_REQUIRE((reinterpret_cast<uintptr_t>(a->grid_out) & 15) == 0, MVX_EINVAL, "grid_out must be 16-byte aligned");
        if (vp.vfeat_t) {
            unsigned *occ = reinterpret_cast<unsigned *>(ws + L.off[R_OCC]);
            rc = launch_occ_from_map(vo.cell2vid, occ, B, L.G, st);
            if (rc) return rc;
            rc = launch_grid_fill_planes(occ, vo.cell2vid, F32(R_VFEAT_T), (long long)cap * 128, 1, cap, a->grid_out, a->grid_dtype, B, L.G, 128,
                                         st);
        } else {
            rc = launch_grid_fill(vo.cell2vid, F32(R_VFEAT), a->grid_out, a->grid_dtype, B, L.G, 128, cap, st);
        }
        if (rc) return rc;
    }
    stamp.mark(S_COUNT);
    return MVX_OK;
}

}  // namespace mvx

extern "C" int mvx_timing_enable(int32_t max_calls) {
    auto &t = mvx::g_timing;
    for (cudaEvent_t e : t.ev) cudaEventDestroy(e);
    t.ev.clear();
    t.recorded.clear();
    t.max_calls = 0, t.next = 0;
    if (max_calls <= 0) return MVX_OK;
    t.ev.resize((size_t)max_calls * mvx::S_COUNT * 2);
    t.recorded.assign(max_calls, 0u);
    for (auto &e : t.ev) MVX_CUDA_CHECK(cudaEventCreate(&e));
    t.max_calls = max_calls;
    return MVX_OK;
}

extern "C" int mvx_timing_read(int32_t call, float *ms) {
    auto &t = mvx::g_timing;
    MVX_REQUIRE(ms && call >= 0 && call < t.next, MVX_EINVAL, "no timing recorded for this call");
    cudaEvent_t *ev = &t.ev[(size_t)call * mvx::S_COUNT * 2];
    for (int i = 0; i < MVX_NUM_SEGMENTS; ++i) ms[i] = 0.f;
    for (int i = 0; i < mvx::S_COUNT; ++i) {
        if (!(t.recorded[call] >> i & 1u)) continue;
        MVX_CUDA_CHECK(cudaEventSynchronize(ev[2 * i + 1]));
        MVX_CUDA_CHECK(cudaEventElapsedTime(&ms[i], ev[2 * i], ev[2 * i + 1]));
    }
    return MVX_OK;
}

extern "C" const char *mvx_timing_segment_name(int32_t segment) {
    if (segment < 0 || segment >= mvx::S_COUNT) return nullptr;
    if (mvx::pixel_first(false)) {  // the timing leg times inference; pixel-first fcn1: the two segments change meaning
        if (segment == mvx::S_GATHER) return "pixel_gemm";
        if (segment == mvx::S_FCN1) return "fcn1_combine";
    }
    return mvx::kSegmentNames[segment];
}

extern "C" int mvx_pointpath_workspace_bytes(const mvx_pointpath_args_t *args, size_t *bytes) {
    mvx::Layout L;
    int rc = mvx::make_layout(args, L);
    if (rc) return rc;
    if (!bytes) return MVX_EINVAL;
    *bytes = L.total;
    return MVX_OK;
}

extern "C" int mvx_pointpath_layout(const mvx_pointpath_args_t *args, int64_t *offsets) {
    mvx::Layout L;
    int rc = mvx::make_layout(args, L);
    if (rc) return rc;
    if (!offsets) return MVX_EINVAL;
    for (int r = 0; r < MVX_WS_REGIONS; ++r) offsets[r] = r < mvx::R_COUNT ? (int64_t)L.off[r] : -1;
    return MVX_OK;
}

extern "C" const char *mvx_pointpath_layout_name(int32_t region) {
    return (region >= 0 && region < mvx::R_COUNT) ? mvx::kRegionNames[region] : nullptr;
}

extern "C" int mvx_pointpath_forward(const mvx_pointpath_args_t *args) { return mvx::pointpath_forward(args, false); }
