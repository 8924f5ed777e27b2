// Stage 3 on the tensor cores, third generation of the layer kernel: persistent, warp-specialised, the raw fp32 activations
// staged by the TMA engine (cp.async.bulk.tensor, SASS UTMALDG) and the A operand fed to tcgen05.mma from TENSOR MEMORY.
//
// Why: the one-tile kernel (tc_layer.cu) runs its three phases one after the other - register producers (global loads, two
// chunks in flight, 96 registers), MMAs, epilogue - and both persistent attempts that kept the register producers ran out of
// registers before they could overlap them (DESIGN.md §5). Here nobody holds global-memory latency in registers:
//   warp 0      producer: one elected thread issues the 2-D tensor copies of the raw fp32 A tiles (128 rows x 32 k, 16 KB,
//               SWIZZLE_128B) into a 4-deep shared-memory ring, and the bulk copies of the pre-packed fp16 hi/lo weights
//               (resident for K = 128 layers, a 3-deep ring otherwise)
//   warp 1      MMA issuer (+ TMEM allocation): per 16-k step D += A_lo B_hi + A_hi B_lo + A_hi B_hi (3xFP16, fp32 accumulate),
//               A from tensor memory, B from shared memory
//   warps 2-9   converters, two groups of four that take alternate stages: one thread per tile row: ld.shared of the raw row
//               piece (29-cycle latency instead of a DRAM round trip; the group's next piece is fetched before the current one
//               is converted), BatchNorm of the producer layer, fp16 hi/lo split, tcgen05.st into the A stage in TMEM
//   warps 10-17 epilogue, two groups of four that split the column blocks of a tile: tcgen05.ld of a finished accumulator
//               (the other one is being filled: TMEM double buffering), scale / bias / ReLU, 128 x 32 staging blocks in shared
//               memory -> tensor store (UTMASTG) of the raw output rows, column statistics and per-voxel maxima from the
//               staged block; the BatchNorm sums stay in the CTA across its tiles and reach global memory as ONE fp64 atomic
//               pair per column, CTA and frame
// A from TMEM halves what the MMAs read from shared memory (only B), which is what leaves shared-memory bandwidth for the
// raw-tile traffic: per 32-k stage 48 KB (B, 6 MMAs x 2 halves... see DESIGN.md) instead of 96 KB.
// TMEM: 2 x 128 accumulator columns + 4 A stages x (16 hi + 16 lo) columns = 384 of 512.
#include "layers.cuh"
#include "tc_common.cuh"

#include <cuda.h>

namespace mvx {

namespace {

constexpr int T3_TM = 128;           // rows per tile (UMMA M)
constexpr int T3_BN = 128;           // output columns (UMMA N)
constexpr int T3_KB = 32;            // k per pipeline stage
constexpr int T3_RAW_RES = 6, T3_RAW_STR = 7;   // raw A ring depth (weights resident / streamed): the ring has to hold DRAM latency x the
                                                // SM's share of the bandwidth (~1.5 us x 44 GB/s = 66 KB) on top of the stage being converted
constexpr int T3_AST = 4;            // A stages in TMEM
constexpr int T3_BRING = 3;          // streamed-weights ring depth
// Converter and epilogue warps come in groups of four (one warp per TMEM lane quarter). Weights resident (K = 128: fcn2, last FCN,
// epilogue-bound): 2 converter groups + 2 epilogue groups. Weights streamed (conv1, K = 768, converter-bound: 24 chunks per tile
// and an epilogue that idles most of the time): 3 converter groups + 1 epilogue group - the same 19 warps and 96 registers.
constexpr int T3_W_PROD = 0, T3_W_MMA = 1, T3_W_CONV = 2;
__host__ __device__ constexpr int t3_threads(int ncg, int neg) { return (3 + 4 * ncg + 4 * neg) * 32; }
constexpr int T3_RAW_BYTES = T3_TM * T3_KB * 4;      // 16 KB
constexpr int T3_B_STAGE = 2 * T3_BN * 64;           // 16 KB: [hi | lo] images of one 32-k chunk
constexpr int T3_STG_BYTES = T3_TM * 32 * 4;         // 16 KB: one 128 x 32 fp32 output block
constexpr uint32_t T3_TMEM_COLS = 512;
constexpr uint32_t T3_ACC_COL = 0, T3_A_COL = 256;   // accumulators at columns [0,256), A stages at [256,384)

template <bool RESIDENT>
struct T3Smem {
    static constexpr int T3_RAW = RESIDENT ? T3_RAW_RES : T3_RAW_STR;
    static constexpr int kRaw = 0;
    static constexpr int kB = kRaw + T3_RAW * T3_RAW_BYTES;
    static constexpr int kBBytes = RESIDENT ? 4 * T3_B_STAGE : T3_BRING * T3_B_STAGE;   // resident: K = 128 -> 4 chunks
    static constexpr int kStg = kB + kBBytes;                       // [2 epilogue groups] one staging block each
    static constexpr int kMean = kStg + 2 * T3_STG_BYTES;
    static constexpr int kRstd = kMean + 768 * 4;
    static constexpr int kBias = kRstd + 768 * 4;
    static constexpr int kColInv = kBias + T3_BN * 4;
    static constexpr int kRowW = kColInv + T3_BN * 4;               // [2 epilogue groups][2 accumulator buffers][128] BN multiplicity of the tile rows
    static constexpr int kRowV = kRowW + 4 * T3_TM * 4;             // [2][2][128] voxel of the tile rows
    static constexpr int kStat = kRowV + 4 * T3_TM * 4;             // [128 columns][2] fp64 running sums of this CTA for the current frame
    static constexpr int kPart = kStat + T3_BN * 2 * 8;             // [2 groups][4 row groups][32 columns][2] fp64 partials of one block
    static constexpr int kBars = kPart + 2 * 4 * 32 * 2 * 8;
    static constexpr int kNumBars = 2 * T3_RAW + 2 * T3_AST + 2 * T3_BRING + 4 + 1;
    static constexpr int kTmemPtr = kBars + 8 * kNumBars;
    static constexpr int kTotal = kTmemPtr + 16 + 1024;
};
static_assert(T3Smem<true>::kTotal <= 232448 && T3Smem<false>::kTotal <= 232448, "tc3: shared memory");

// ---- PTX not in tc_common.cuh --------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *tmap, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *tmap, int c0, int c1, uint32_t src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(tmap), "r"(c0), "r"(c1), "r"(src)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap *tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
                 "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

struct T3Args {
    LayerArgs a;
    const void *wpack;     // [fp16 hi|lo chunk images: Cin*Cout*4 bytes][inverse column scales: Cout floats]
    int F, row_tiles;
    int store;             // 1: a.Y is written (through tmY)
};

// CAT: the trailing a.x2_cols input columns of a row come from a.X2[f][v(row)] (fused concat of the last FCN). The rows of a
// tile belong to a CONTIGUOUS range of at most 128 voxels (rows are voxel-major and every voxel owns at least one row; the
// pad rows behind them are one per voxel, in voxel order), so that half is a plain 2-D tile of X2 as well: rows
// [v_first, v_first + 128), fetched by the same tensor copies into the same ring; a converter thread reads row v(r) - v_first.
// Only the one tile per frame that straddles the real-row / pad-row boundary needs two ranges: its pad rows read global memory.
// PREC: 0 = fp32-accurate 3xFP16 from fp32 rows; 1 = bf16 mode (ONE bf16 product per k-step, reduced precision) from fp32 rows;
//       2 = bf16 mode from bf16 rows (conv1 reading the bf16 Y1 of the combine kernel: half the bytes per stage)
template <bool RESIDENT, bool CAT, int PREC, int NCG = RESIDENT ? 2 : 3, int NEG = RESIDENT ? 2 : 1>
__global__ void __launch_bounds__(t3_threads(NCG, NEG), 1) tc3_layer_kernel(const __grid_constant__ T3Args g, const __grid_constant__ CUtensorMap tmX,
                                                                  const __grid_constant__ CUtensorMap tmY,
                                                                  const __grid_constant__ CUtensorMap tmX2) {
    using S = T3Smem<RESIDENT>;
    constexpr int T3_RAW = S::T3_RAW;
    constexpr bool BF = PREC != 0, RAWBF = PREC == 2;
    constexpr int T3_CONV_WARPS = 4 * NCG, T3_EPI_WARPS = 4 * NEG, T3_THREADS = t3_threads(NCG, NEG);
    constexpr int T3_W_EPI = T3_W_CONV + T3_CONV_WARPS, T3_W_BPROD = T3_W_EPI + T3_EPI_WARPS;
    constexpr int CBG = (T3_BN / 32) / NEG;          // 32-column blocks per epilogue group
    static_assert(NEG == 1 || NEG == 2, "epilogue groups");
    constexpr int RAW_TX = RAWBF ? T3_RAW_BYTES / 2 : T3_RAW_BYTES;     // bytes one raw stage receives
    constexpr int B_TX = BF ? T3_B_STAGE / 2 : T3_B_STAGE;              // bf16 weights: the hi image only
    static_assert(!(CAT && RAWBF), "the concat layer reads fp32 rows");
    const LayerArgs &a = g.a;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    float *s_mean = reinterpret_cast<float *>(smem + S::kMean);
    float *s_rstd = reinterpret_cast<float *>(smem + S::kRstd);
    float *s_bias = reinterpret_cast<float *>(smem + S::kBias);
    float *s_colinv = reinterpret_cast<float *>(smem + S::kColInv);
    float *s_roww = reinterpret_cast<float *>(smem + S::kRowW);
    int *s_rowv = reinterpret_cast<int *>(smem + S::kRowV);
    double *s_stat = reinterpret_cast<double *>(smem + S::kStat);
    const uint32_t bars = sbase + S::kBars;
    auto raw_full = [&](int s) { return bars + 8u * s; };
    auto raw_empty = [&](int s) { return bars + 8u * (T3_RAW + s); };
    auto a_full = [&](int s) { return bars + 8u * (2 * T3_RAW + s); };
    auto a_empty = [&](int s) { return bars + 8u * (2 * T3_RAW + T3_AST + s); };
    auto b_full = [&](int s) { return bars + 8u * (2 * T3_RAW + 2 * T3_AST + s); };
    auto b_empty = [&](int s) { return bars + 8u * (2 * T3_RAW + 2 * T3_AST + T3_BRING + s); };
    auto acc_full = [&](int b) { return bars + 8u * (2 * T3_RAW + 2 * T3_AST + 2 * T3_BRING + b); };
    auto acc_empty = [&](int b) { return bars + 8u * (2 * T3_RAW + 2 * T3_AST + 2 * T3_BRING + 2 + b); };
    const uint32_t b_ready = bars + 8u * (2 * T3_RAW + 2 * T3_AST + 2 * T3_BRING + 4);
    volatile uint32_t *tmem_ptr = reinterpret_cast<volatile uint32_t *>(smem + S::kTmemPtr);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nk = a.Cin / T3_KB;                                 // a multiple of NCG (checked by the launcher): chunk kc of every tile goes to converter group kc % NCG
    const int nk_x = CAT ? (a.Cin - a.x2_cols) / T3_KB : nk;     // chunks that come from X; the others from X2
    const int total = g.F * g.row_tiles;

    // tile decode shared by every role: identical decisions => identical ring bookkeeping
    auto decode = [&](int t, int &f, long long &row0, long long &n_rows, int &Kf) -> bool {
        if (t >= total) return false;
        f = t / g.row_tiles;
        const int rt = t - f * g.row_tiles;
        const int N = a.counts[f * 4 + 0];
        Kf = a.counts[f * 4 + 1];
        n_rows = a.rows_mode == 1 ? Kf + 1 : (long long)Kf + N;
        row0 = (long long)rt * T3_TM;
        return row0 < n_rows;
    };
    // first voxel of the X2 tile that serves the rows [row0, row0 + 128) of frame f
    auto x2_first = [&](int f, long long row0, int Kf) -> int {
        return row0 >= Kf ? (int)(row0 - Kf) : a.cat_row_vox[(size_t)f * a.cat_rowv_cap + row0];
    };

    if (tid == 0) {
        for (int s = 0; s < T3_RAW; ++s) mbar_init(raw_full(s), 1), mbar_init(raw_empty(s), 4);
        for (int s = 0; s < T3_AST; ++s) mbar_init(a_full(s), 4), mbar_init(a_empty(s), 1);
        for (int s = 0; s < T3_BRING; ++s) mbar_init(b_full(s), 1), mbar_init(b_empty(s), 1);
        for (int b = 0; b < 2; ++b) mbar_init(acc_full(b), 1), mbar_init(acc_empty(b), T3_EPI_WARPS);
        mbar_init(b_ready, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int c = tid; c < T3_BN; c += T3_THREADS) {
        s_bias[c] = a.bias[c];
        s_colinv[c] = reinterpret_cast<const float *>(static_cast<const uint8_t *>(g.wpack) + (size_t)a.Cin * a.Cout * 4)[c];
    }
    if (warp == T3_W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + S::kTmemPtr), "r"(T3_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == T3_W_PROD) {
        // ================= producer: raw A tiles by tensor copy, weights by bulk copy ===================================
        if (lane == 0) {
            prefetch_tmap(&tmX);
            if (CAT) prefetch_tmap(&tmX2);
            int gc = 0;   // ring position
            for (int t = blockIdx.x; t < total; t += gridDim.x) {
                int f, Kf;
                long long row0, n_rows;
                if (!decode(t, f, row0, n_rows, Kf)) continue;
                int vfirst = 0;
                if (CAT) vfirst = x2_first(f, row0, Kf);   // its latency hides behind the ring's run-ahead (one tile deep)
                for (int kc = 0; kc < nk; ++kc, ++gc) {
                    const int s = gc % T3_RAW;
                    mbar_wait(raw_empty(s), ((gc / T3_RAW) & 1) ^ 1);
                    mbar_arrive_expect_tx(raw_full(s), RAW_TX);
                    if (!CAT || kc < nk_x)
                        tma_load_2d(sbase + S::kRaw + s * T3_RAW_BYTES, &tmX, kc * T3_KB, (int)((long long)f * a.rowcap + row0), raw_full(s));
                    else
                        tma_load_2d(sbase + S::kRaw + s * T3_RAW_BYTES, &tmX2, (kc - nk_x) * T3_KB, (int)((long long)f * a.vcap + vfirst), raw_full(s));
                }
            }
        }
    } else if (warp == T3_W_BPROD) {
        // ================= weights: resident (one load) or streamed through their own ring by their own thread, so that a wait
        // for a free weight stage never holds back the raw-tile copies ===================================================
        if (lane == 0) {
            const uint8_t *wsrc = static_cast<const uint8_t *>(g.wpack);
            if (RESIDENT) {
                mbar_arrive_expect_tx(b_ready, nk * B_TX);
                for (int kc = 0; kc < nk; ++kc) bulk_g2s(sbase + S::kB + kc * T3_B_STAGE, wsrc + (size_t)kc * T3_B_STAGE, B_TX, b_ready);
            } else {
                int gb = 0;
                for (int t = blockIdx.x; t < total; t += gridDim.x) {
                    int f, Kf;
                    long long row0, n_rows;
                    if (!decode(t, f, row0, n_rows, Kf)) continue;
                    for (int kc = 0; kc < nk; ++kc, ++gb) {
                        const int sb = gb % T3_BRING;
                        mbar_wait(b_empty(sb), ((gb / T3_BRING) & 1) ^ 1);
                        mbar_arrive_expect_tx(b_full(sb), B_TX);
                        bulk_g2s(sbase + S::kB + sb * T3_B_STAGE, wsrc + (size_t)kc * T3_B_STAGE, B_TX, b_full(sb));
                    }
                }
            }
        }
    } else if (warp == T3_W_MMA) {
        // ================= MMA issuer ==================================================================================
        if (lane == 0) {
            constexpr uint32_t fmt = BF ? 1u : 0u;   // kind::f16 operand format: 0 = fp16, 1 = bf16
            constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(T3_BN >> 3) << 17) | ((128u >> 4) << 24);   // fp32 accumulate
            if (RESIDENT) mbar_wait(b_ready, 0);
            int ga = 0, gb = 0, it = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x) {
                int f, Kf;
                long long row0, n_rows;
                if (!decode(t, f, row0, n_rows, Kf)) continue;
                const int ab = it & 1;
                mbar_wait(acc_empty(ab), ((it >> 1) & 1) ^ 1);   // the epilogue drained this accumulator two tiles ago
                tc_fence_after();
                const uint32_t d = tmem_base + T3_ACC_COL + ab * T3_BN;
                for (int kc = 0; kc < nk; ++kc, ++ga) {
                    const int sa = ga % T3_AST;
                    int sb = kc;
                    if (!RESIDENT) {
                        sb = gb % T3_BRING;
                        mbar_wait(b_full(sb), (gb / T3_BRING) & 1);
                    }
                    mbar_wait(a_full(sa), (ga / T3_AST) & 1);
                    tc_fence_after();
                    const uint32_t sB = sbase + S::kB + sb * T3_B_STAGE;
                    const uint32_t tA = tmem_base + T3_A_COL + sa * 32;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {   // two 16-k steps per stage
                        const uint64_t b_hi = make_desc(sB + ks * 32), b_lo = make_desc(sB + T3_BN * 64 + ks * 32);
                        const uint32_t a_hi = tA + ks * 8, a_lo = tA + 16 + ks * 8;
                        if constexpr (BF) {
                            mma_f16_ts(d, a_hi, b_hi, idesc, (kc | ks) != 0);
                        } else {
                            mma_f16_ts(d, a_lo, b_hi, idesc, (kc | ks) != 0);
                            mma_f16_ts(d, a_hi, b_lo, idesc, 1);
                            mma_f16_ts(d, a_hi, b_hi, idesc, 1);
                        }
                    }
                    mma_commit(a_empty(sa));
                    if (!RESIDENT) {
                        mma_commit(b_empty(sb));
                        ++gb;
                    }
                }
                mma_commit(acc_full(ab));
                ++it;
            }
        }
    } else if (warp < T3_W_EPI) {
        // ================= converters: two groups of four warps; group cg converts the chunks with (chunk counter & 1) == cg,
        // a thread one whole row piece (32 k). The raw piece of the group's NEXT chunk is read into registers before the
        // current one is converted (its shared-memory latency and the stage hand-back overlap the arithmetic).
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
        const int cg = (warp - T3_W_CONV) >> 2;       // converter group
        const int r = q * 32 + lane;                  // row inside the tile
        const int ct = tid - T3_W_CONV * 32;          // 0 .. 255
        int n_chunks = 0;                             // chunks this CTA will see in total (ring positions run 0 .. n_chunks-1)
        for (int t = blockIdx.x; t < total; t += gridDim.x) {
            int f, Kf;
            long long row0, n_rows;
            if (decode(t, f, row0, n_rows, Kf)) n_chunks += nk;
        }
        float4 xn[8];                                 // the group's next raw row piece
        auto fetch = [&](int gcn, int srow) {         // read row `srow` of ring position gcn, hand the stage back
            const int s = gcn % T3_RAW;
            mbar_wait(raw_full(s), (gcn / T3_RAW) & 1);
            if constexpr (RAWBF) {   // bf16 rows: 64 bytes, SWIZZLE_64B: chunk j of row i at position j ^ ((i >> 1) & 3)
                const uint8_t *rowp = smem + S::kRaw + s * T3_RAW_BYTES + srow * 64;
#pragma unroll
                for (int j = 0; j < 4; ++j) xn[j] = *reinterpret_cast<const float4 *>(rowp + ((j ^ ((srow >> 1) & 3)) << 4));
            } else {
            const uint8_t *rowp = smem + S::kRaw + s * T3_RAW_BYTES + srow * 128;   // SWIZZLE_128B: chunk j of row i at position j ^ (i & 7)
#pragma unroll
            for (int j = 0; j < 8; ++j) xn[j] = *reinterpret_cast<const float4 *>(rowp + ((j ^ (srow & 7)) << 4));
            }
            // The stage goes back to the TMA engine, which writes through the ASYNC proxy: a plain arrive after the ld.shared is not
            // enough (the loads are only issued, and the arrive travels a different path; with L2-resident inputs the refill came
            // back before a few lanes had read their rows: sporadic wrong rows, found with tools/tc3_race.py). The proxy fence
            // orders this thread's generic-proxy reads before the async-proxy writes that follow the arrive.
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(raw_empty(s));
        };
        int gc = 0, cur_f = -1;
        bool primed = false;
        for (int t = blockIdx.x; t < total; t += gridDim.x) {
            int f, Kf;
            long long row0, n_rows;
            if (!decode(t, f, row0, n_rows, Kf)) continue;
            if (f != cur_f) {   // BatchNorm coefficients of the producer layer for this frame
                named_bar_sync(1, T3_CONV_WARPS * 32);
                const double Rstat = (double)a.counts[f * 4 + 0] * (double)a.T;
                const int inC = a.in_C > 0 ? a.in_C : a.Cin;
                for (int c = ct; c < a.Cin; c += T3_CONV_WARPS * 32) {
                    const double *st = a.in_stats + ((size_t)f * inC + c % inC) * 2;
                    const double m = st[0] / Rstat;
                    double var = st[1] / Rstat - m * m;
                    var = var < 0.0 ? 0.0 : var;
                    s_mean[c] = (float)m;
                    s_rstd[c] = (float)(1.0 / sqrt(var + a.eps));
                }
                named_bar_sync(1, T3_CONV_WARPS * 32);
                cur_f = f;
            }
            const long long rr = row0 + r;
            const bool valid = rr < n_rows;
            int vrel = 0;               // CAT: row of the X2 tile that serves this row
            bool x2_global = false;     // CAT: pad row of the straddling tile -> its voxel lies outside the tile's X2 range
            int vrow = 0;
            if (CAT) {
                const int vfirst = x2_first(f, row0, Kf);
                vrow = valid ? (rr >= Kf ? (int)(rr - Kf) : a.cat_row_vox[(size_t)f * a.cat_rowv_cap + rr]) : vfirst;
                x2_global = valid && rr >= Kf && row0 < Kf;
                vrel = x2_global ? 0 : vrow - vfirst;
            }
            if (!primed) {              // very first chunk of this group
                fetch(cg, r);
                primed = true;
            }
            for (int kc = cg; kc < nk; kc += NCG) {
                const int gcur = gc + kc;
                float4 x[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) x[j] = xn[j];
                if (CAT && kc >= nk_x && x2_global) {   // rare: one tile per frame
                    const float4 *src = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(a.X2) + ((size_t)f * a.vcap + vrow) * a.x2_cols +
                                                                         (kc - nk_x) * T3_KB);
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = __ldg(src + j);
                }
                // the group's next chunk: same tile (kc + NCG) or its first one of the next tile (always an X chunk: row r)
                if (gcur + NCG < n_chunks) fetch(gcur + NCG, (CAT && kc + NCG < nk && kc + NCG >= nk_x) ? vrel : r);
                const int k0 = kc * T3_KB;
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 m4 = *reinterpret_cast<const float4 *>(s_mean + k0 + j * 4);
                    const float4 r4 = *reinterpret_cast<const float4 *>(s_rstd + k0 + j * 4);
                    float4 xv;
                    if constexpr (RAWBF) {   // elements 4j .. 4j+3 of the row piece: two 32-bit words of x[j / 2]
                        const uint32_t w0 = __float_as_uint(j & 1 ? x[j >> 1].z : x[j >> 1].x), w1 = __float_as_uint(j & 1 ? x[j >> 1].w : x[j >> 1].y);
                        xv = make_float4(__uint_as_float(w0 << 16), __uint_as_float(w0 & 0xFFFF0000u), __uint_as_float(w1 << 16), __uint_as_float(w1 & 0xFFFF0000u));
                    } else {
                        xv = x[j];
                    }
                    float z0 = (xv.x - m4.x) * r4.x, z1 = (xv.y - m4.y) * r4.y, z2 = (xv.z - m4.z) * r4.z, z3 = (xv.w - m4.w) * r4.w;
                    if (!valid) z0 = z1 = z2 = z3 = 0.f;
                    if constexpr (BF) {
                        hi[2 * j] = pack_bf16x2(z0, z1), hi[2 * j + 1] = pack_bf16x2(z2, z3);
                    } else {
                        split_f16_pair(z0, z1, hi[2 * j], lo[2 * j]);
                        split_f16_pair(z2, z3, hi[2 * j + 1], lo[2 * j + 1]);
                    }
                }
                const int sa = gcur % T3_AST;
                mbar_wait(a_empty(sa), ((gcur / T3_AST) & 1) ^ 1);   // the MMAs that read this A stage have completed
                tc_fence_after();
                const uint32_t tA = tmem_base + ((uint32_t)(q * 32) << 16) + T3_A_COL + sa * 32;
                tmem_st16(tA, hi);
                if constexpr (!BF) tmem_st16(tA + 16, lo);
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full(sa));
            }
            gc += nk;
        }
    } else {
        // ================= epilogue: two groups of four warps (TMEM lane quarter q = warp % 4); group eg takes the column
        // blocks 2 eg and 2 eg + 1 of every tile, with its own staging blocks, partials and named barrier ==================
        const int q = warp & 3, eg = (warp - T3_W_EPI) >> 2;
        const int et = (tid - T3_W_EPI * 32) & 127;         // thread inside the group
        const int ecol = lane;                              // statistics / maxima: lane = column of a 32-column block ...
        const int erow = q * 32 + lane;                     // ... over the warp's OWN 32 rows (its TMEM lane quarter); metadata: lane = row
        const int bar_id = 2 + eg;
        // Every warp is self-contained inside the tile loop: it stages, stores (its own 32-row tensor store) and walks only the 32 rows
        // it drained from tensor memory, and keeps its BatchNorm sums in registers until the frame changes - no named barrier between
        // the four warps of a group per block (there were three; with K = 128 the epilogue bounds the kernel and its warps spent their
        // time waiting for each other).
        constexpr int SG = 2 * T3_BN / NEG;                  // this group's columns x {sum, sum of squares}
        uint8_t *stg = smem + S::kStg + eg * T3_STG_BYTES;
        if (et == 0 && g.store) prefetch_tmap(&tmY);
        for (int i = et; i < SG; i += 128) s_stat[eg * SG + i] = 0.0;
        named_bar_sync(bar_id, 128);
        int it = 0, cur_f = -1;
        double acc_sy[CBG], acc_syy[CBG];                  // this lane's column of every block of the group, this warp's rows
#pragma unroll
        for (int c = 0; c < CBG; ++c) acc_sy[c] = acc_syy[c] = 0.0;
        auto flush_stats = [&](int f) {   // warps -> CTA (shared fp64 atomics), then one fp64 atomic pair per column, CTA and frame
#pragma unroll
            for (int c = 0; c < CBG; ++c) {
                atomicAdd(&s_stat[((eg * CBG + c) * 32 + lane) * 2], acc_sy[c]);
                atomicAdd(&s_stat[((eg * CBG + c) * 32 + lane) * 2 + 1], acc_syy[c]);
                acc_sy[c] = acc_syy[c] = 0.0;
            }
            named_bar_sync(bar_id, 128);
            for (int i = eg * SG + et; i < (eg + 1) * SG; i += 128) {
                const double v = s_stat[i];
                if (v != 0.0) atomicAdd(a.out_stats + (size_t)f * a.Cout * 2 + i, v);
                s_stat[i] = 0.0;
            }
            named_bar_sync(bar_id, 128);
        };
        // The walk over the tiles carries the row metadata of the NEXT tile in registers: the two global loads per row (multiplicity,
        // voxel id) used to sit at the head of every tile, a full memory round trip that nothing covered (14 % of the epilogue's
        // stall samples; with K = 128 the epilogue, not the four-stage main loop, bounds the kernel).
        auto next_valid = [&](int tn, int &f, long long &row0, long long &n_rows, int &Kf) -> int {
            while (tn < total && !decode(tn, f, row0, n_rows, Kf)) tn += gridDim.x;
            return tn;
        };
        auto load_meta = [&](int f, long long row0, long long n_rows, int Kf, float &w, int &v) {
            const long long rr = row0 + erow;
            const bool has_v = a.vmax && rr < n_rows && !(a.rows_mode == 1 && rr >= Kf);
            // both loads are issued back to back (the voxel id does not wait for the multiplicity to arrive)
            const int vl = has_v ? a.row_v[(size_t)f * a.rowv_cap + rr] : -1;
            w = rr < n_rows ? (a.row_w ? a.row_w[(size_t)f * a.rowcap + rr] : 1.f) : 0.f;
            v = w != 0.f ? vl : -1;
        };
        int f = 0, Kf = 0;
        long long row0 = 0, n_rows = 0;
        int t = next_valid(blockIdx.x, f, row0, n_rows, Kf);
        float pw = 0.f;
        int pv = -1;
        if (t < total) load_meta(f, row0, n_rows, Kf, pw, pv);
        while (t < total) {
            if (f != cur_f) {
                if (cur_f >= 0) flush_stats(cur_f);
                cur_f = f;
            }
            const int ab = it & 1;
            // row metadata of this tile: every group keeps its own copy (no cross-group synchronisation)
            float *roww = s_roww + (eg * 2 + ab) * T3_TM;
            int *rowv = s_rowv + (eg * 2 + ab) * T3_TM;
            const float w_own = pw;
            const int v_own = pv;
            int fn = 0, Kfn = 0;
            long long row0n = 0, n_rowsn = 0;
            const int tn = next_valid(t + gridDim.x, fn, row0n, n_rowsn, Kfn);
            if (tn < total) load_meta(fn, row0n, n_rowsn, Kfn, pw, pv);     // in flight during this tile
            roww[erow] = w_own;
            rowv[erow] = v_own;
            // This warp's lanes hold the rows q * 32 + lane - exactly the rows its threads walk below. Run structure of the voxel
            // ids as bit masks (a row starts / ends a run of equal ids), rows of multiplicity 1, and whether any row is weighted
            // (neither 0 nor 1: the pad rows; the fp64 side path is skipped by whole warps on ordinary tiles): the walk tests
            // register bits instead of chasing shared-memory loads with compares and branches row by row.
            const int v_prev = __shfl_up_sync(0xffffffffu, v_own, 1), v_next = __shfl_down_sync(0xffffffffu, v_own, 1);
            const unsigned startmask = __ballot_sync(0xffffffffu, lane == 0 || v_own != v_prev);
            const unsigned endmask = __ballot_sync(0xffffffffu, v_own >= 0 && (lane == 31 || v_own != v_next));
            const unsigned onesmask = __ballot_sync(0xffffffffu, w_own == 1.f);
            const bool heavy = __any_sync(0xffffffffu, w_own != 1.f && w_own != 0.f);
            __syncwarp();                                    // roww / rowv of this warp's rows are read by its own lanes only
            mbar_wait(acc_full(ab), (it >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int cbl = 0; cbl < CBG; ++cbl) {
                const int cb = eg * CBG + cbl;
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + T3_ACC_COL + ab * T3_BN + cb * 32, v);
                if (cbl == CBG - 1) {   // the accumulator is in registers: the MMA warp may start the tile after next
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty(ab));
                }
                if (g.store && lane == 0) tma_store_wait_read<0>();   // this warp's previous tensor store is done reading its staging rows
                __syncwarp();                                         // ... and all its lanes are done with the column walk of that block
                const int rloc = q * 32 + lane;
                uint8_t *rowp = stg + rloc * 128;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = cb * 32 + j * 4;
                    const float4 ci = *reinterpret_cast<const float4 *>(s_colinv + c), bi = *reinterpret_cast<const float4 *>(s_bias + c);
                    float4 o;
                    o.x = fmaxf(v[j * 4 + 0] * ci.x + bi.x, 0.f);
                    o.y = fmaxf(v[j * 4 + 1] * ci.y + bi.y, 0.f);
                    o.z = fmaxf(v[j * 4 + 2] * ci.z + bi.z, 0.f);
                    o.w = fmaxf(v[j * 4 + 3] * ci.w + bi.w, 0.f);
                    *reinterpret_cast<float4 *>(rowp + ((j ^ (rloc & 7)) << 4)) = o;   // SWIZZLE_128B like the store's tensor map
                }
                fence_async_smem();
                __syncwarp();
                if (g.store && lane == 0) {   // this warp's 32 rows x 32 columns (the tensor map's box)
                    tma_store_2d(&tmY, cb * 32, (int)((long long)f * a.rowcap + row0 + q * 32), smem_u32(stg + q * 4096));
                    tma_store_commit();
                }
                // column walk over this thread's 32 rows: sums of the ordinary rows in fp32 over 16 rows, fp64 beyond; weighted
                // rows take an exact fp64 side path; per-voxel running maximum with one atomicMax per run
                {
                    double sy = 0.0, syy = 0.0;
                    int *vm = a.vmax ? a.vmax + (size_t)f * a.vcap * a.Cout + cb * 32 + ecol : nullptr;
                    float cm = 0.f;                       // running maximum of the current run (y >= 0 after the ReLU: 0 is neutral)
                    const float *rw_ = roww + q * 32;
                    const int *rv_ = rowv + q * 32;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        float yv[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int rw = q * 32 + h * 16 + j;
                            yv[j] = *reinterpret_cast<const float *>(stg + rw * 128 + (((ecol >> 2) ^ (rw & 7)) << 4) + (ecol & 3) * 4);
                        }
                        float ps = 0.f, pss = 0.f;
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float my = (onesmask >> (h * 16 + j)) & 1u ? yv[j] : 0.f;
                            ps += my;
                            pss = fmaf(my, yv[j], pss);
                        }
                        sy += (double)ps;
                        syy += (double)pss;
                        if (heavy) {
                            for (int j = 0; j < 16; ++j) {
                                const float w = rw_[h * 16 + j];
                                if (w != 1.f && w != 0.f) {
                                    const double wy = (double)w * (double)yv[j];
                                    sy += wy;
                                    syy = fma(wy, (double)yv[j], syy);
                                }
                            }
                        }
                        if (vm) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const int b = h * 16 + j;
                                cm = fmaxf((startmask >> b) & 1u ? 0.f : cm, yv[j]);
                                if ((endmask >> b) & 1u) atomicMax(vm + (size_t)rv_[b] * a.Cout, __float_as_int(cm));   // one atomic per run
                            }
                        }
                    }
                    acc_sy[cbl] += sy;
                    acc_syy[cbl] += syy;
                }
            }
            ++it;
            t = tn, f = fn, row0 = row0n, n_rows = n_rowsn, Kf = Kfn;
        }
        if (cur_f >= 0) flush_stats(cur_f);
        if (g.store && lane == 0) tma_store_wait_all();
    }
    __syncwarp();   // single-lane role warps: lanes 1-31 wait here for their looping lane 0
    tc_fence_before();
    __syncthreads();
    if (warp == T3_W_MMA) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(T3_TMEM_COLS) : "memory");
    }
}

// =====================================================================================================================
// Persistent per-pixel GEMM of the pixel-first fcn1 (Z_l = F_l W1_l^T, plain: no bias / ReLU / statistics): both operands arrive
// pre-packed (fp16 hi / lo shared-memory images: the FPN maps by pack_maps_f16_kernel, the weights by pack_weights_f16_kernel), so
// there are no converters at all - a bulk-copy thread, an MMA thread and eight epilogue warps:
//   warp 0      producer: per 32-k chunk one cp.async.bulk of the A tile (256 rows: [hi 16 KB | lo 16 KB]) and one of the weight
//               chunk of the tile's 128-column block ([hi 8 KB | lo 8 KB]) into a 3-deep ring that keeps streaming ACROSS tiles
//   warp 1      MMA issuer (+ TMEM allocation): per 16-k step and 128-row half D += A_lo B_hi + A_hi B_lo + A_hi B_hi, both
//               operands from shared memory; two accumulator buffers of 2 x 128 TMEM columns (all 512)
//   warps 2-9   epilogue, two groups of four (group = 128-row half, warp = TMEM lane quarter): tcgen05.ld of the finished buffer
//               while the MMAs fill the other one, exact power-of-two rescale (row x column), 128 x 32 staging block, tensor store
// The one-tile kernel it replaces (tc_layer_kernel<128, F16, -, TWO, APK>, two CTAs per SM) restarts its 2-stage ring for every
// tile: ncu attributes 42 % of its samples to the epilogue warps idling through an ~6 us main loop that exposes one L2 round trip
// per pair of chunks, then ~10 us of epilogue per CTA for 3.7 us of MMAs (profiles/r5v_pixel_gemm_stall_lines.txt).
// Tile order: t = row tile x 6 + column block, striped over the CTAs, so the six tiles that share an A tile run at the same time
// on neighbouring CTAs (one DRAM read of A, five L2 hits).
// =====================================================================================================================
#ifndef MVX_PG_STAGES
#define MVX_PG_STAGES 3
#endif
// 3 x 48 KB. A fourth stage makes the kernel itself faster (0.535 -> 0.484 ms next to the point branch) but the STEP slower (4.43 -> 4.46 ms,
// three A/B pairs): at 228 KB the CTA leaves no shared memory for the point-branch kernels that share the SMs with it during the front
constexpr int PG_TM = 256, PG_BN = 128, PG_KB = 32, PG_STAGES = MVX_PG_STAGES;
constexpr int PG_A_HALF = PG_TM * 64, PG_B_HALF = PG_BN * 64;        // 16 KB, 8 KB: one fp16 image of a chunk
constexpr int PG_STAGE = 2 * PG_A_HALF + 2 * PG_B_HALF;             // 48 KB
constexpr int PG_EPI_WARPS = 8, PG_THREADS = (2 + PG_EPI_WARPS) * 32;
struct PgSmem {
    static constexpr int kRing = 0;
    static constexpr int kStg = kRing + PG_STAGES * PG_STAGE;        // [2 groups] 128 x 32 fp32 staging block
    static constexpr int kBars = kStg + 2 * T3_STG_BYTES;            // full[], empty[], acc_full[2], acc_empty[2] (the column scales are read from global memory: L1 hits, and the fourth stage needs their 3 KB)
    static constexpr int kTmemPtr = kBars + 8 * (2 * PG_STAGES + 4);
    static constexpr int kTotal = kTmemPtr + 16 + 1024;
};
static_assert(PgSmem::kTotal <= 232448, "pixel GEMM: shared memory");

struct PgArgs {
    const uint8_t *a_pack;     // [row tiles][nk][hi 16 KB | lo 16 KB]
    const float *a_rowinv;     // [R] inverse power-of-two row scales (or NULL)
    const uint8_t *wpack;      // [column blocks][nk][hi 8 KB | lo 8 KB], then Cout inverse column scales
    long long R;               // rows (pixels of all frames of the level)
    int Cin, Cout, row_tiles;
};

// ZB: Z is written as bf16 (the bf16 mode stores its two largest intermediates, Z and Y1, as bf16; the products stay 3xFP16)
template <bool ZB>
__global__ void __launch_bounds__(PG_THREADS, 1) pixel_gemm_persistent_kernel(const __grid_constant__ PgArgs g, const __grid_constant__ CUtensorMap tmZ) {
    using S = PgSmem;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    const float *colinv = reinterpret_cast<const float *>(g.wpack + (size_t)g.Cin * g.Cout * 4);
    const uint32_t bars = sbase + S::kBars;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (PG_STAGES + s); };
    auto acc_full = [&](int b) { return bars + 8u * (2 * PG_STAGES + b); };
    auto acc_empty = [&](int b) { return bars + 8u * (2 * PG_STAGES + 2 + b); };
    volatile uint32_t *tmem_ptr = reinterpret_cast<volatile uint32_t *>(smem + S::kTmemPtr);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nk = g.Cin / PG_KB, ncb = g.Cout / PG_BN;
    const int total = g.row_tiles * ncb;

    if (tid == 0) {
        for (int s = 0; s < PG_STAGES; ++s) mbar_init(full_bar(s), 1), mbar_init(empty_bar(s), 1);
        for (int b = 0; b < 2; ++b) mbar_init(acc_full(b), 1), mbar_init(acc_empty(b), PG_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + S::kTmemPtr), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ================= producer =====================================================================================
        if (lane == 0) {
            int gc = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x) {
                const int rt = t / ncb, cb = t - rt * ncb;
                const uint8_t *asrc = g.a_pack + (size_t)rt * nk * (2 * PG_A_HALF);
                const uint8_t *bsrc = g.wpack + (size_t)cb * nk * (2 * PG_B_HALF);
                for (int kc = 0; kc < nk; ++kc, ++gc) {
                    const int s = gc % PG_STAGES;
                    mbar_wait(empty_bar(s), ((gc / PG_STAGES) & 1) ^ 1);
                    mbar_arrive_expect_tx(full_bar(s), PG_STAGE);
                    bulk_g2s(sbase + S::kRing + s * PG_STAGE, asrc + (size_t)kc * (2 * PG_A_HALF), 2 * PG_A_HALF, full_bar(s));
                    bulk_g2s(sbase + S::kRing + s * PG_STAGE + 2 * PG_A_HALF, bsrc + (size_t)kc * (2 * PG_B_HALF), 2 * PG_B_HALF, full_bar(s));
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer ===================================================================================
        if (lane == 0) {
            constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(PG_BN >> 3) << 17) | ((128u >> 4) << 24);   // fp16 x fp16 -> fp32, N = 128, M = 128
            int gc = 0, it = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
                const int ab = it & 1;
                mbar_wait(acc_empty(ab), ((it >> 1) & 1) ^ 1);   // the epilogue drained this buffer two tiles ago
                tc_fence_after();
                for (int kc = 0; kc < nk; ++kc, ++gc) {
                    const int s = gc % PG_STAGES;
                    mbar_wait(full_bar(s), (gc / PG_STAGES) & 1);
                    tc_fence_after();
                    const uint32_t sA = sbase + S::kRing + s * PG_STAGE, sB = sA + 2 * PG_A_HALF;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint32_t d = tmem_base + ab * (2 * PG_BN) + h * PG_BN;
                        const uint32_t aoff = h * (128 * 64);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            const uint64_t a_hi = make_desc(sA + aoff + ks * 32), a_lo = make_desc(sA + PG_A_HALF + aoff + ks * 32);
                            const uint64_t b_hi = make_desc(sB + ks * 32), b_lo = make_desc(sB + PG_B_HALF + ks * 32);
                            mma_f16(d, a_lo, b_hi, idesc, (kc | ks) != 0);
                            mma_f16(d, a_hi, b_lo, idesc, 1);
                            mma_f16(d, a_hi, b_hi, idesc, 1);
                        }
                    }
                    mma_commit(empty_bar(s));
                }
                mma_commit(acc_full(ab));
            }
        }
    } else {
        // ================= epilogue: group = 128-row half of the tile, warp = TMEM lane quarter ==========================
        const int q = warp & 3, eg = (warp - 2) >> 2;
        const int et = (tid - 64) & 127;
        uint8_t *stg = smem + S::kStg + eg * T3_STG_BYTES;
        if (et == 0) prefetch_tmap(&tmZ);
        int it = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
            const int rt = t / ncb, cb = t - rt * ncb;
            const int ab = it & 1;
            const long long row0 = (long long)rt * PG_TM + eg * 128;
            const int rloc = q * 32 + lane;
            const float rinv = (g.a_rowinv && row0 + rloc < g.R) ? __ldg(g.a_rowinv + row0 + rloc) : 1.f;   // in flight during the wait below
            mbar_wait(acc_full(ab), (it >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int c32 = 0; c32 < 4; ++c32) {
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + ab * (2 * PG_BN) + eg * PG_BN + c32 * 32, v);
                if (c32 == 3) {   // the accumulator half is in registers: the MMA warp may reuse the buffer once every warp has said so
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty(ab));
                }
                if (lane == 0) tma_store_wait_read<0>();   // this warp's previous tensor store is done reading its 32 staging rows
                __syncwarp();                              // (every warp stages and stores its own rows: no barrier between the warps)
                const float4 *ci = reinterpret_cast<const float4 *>(colinv + cb * PG_BN + c32 * 32);
                if constexpr (ZB) {   // 64-byte rows, SWIZZLE_64B: 16-byte piece j of row i at position j ^ ((i >> 1) & 3)
                    uint8_t *rowp = stg + rloc * 64;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 ca = __ldg(ci + 2 * j), cb4 = __ldg(ci + 2 * j + 1);
                        uint4 o;
                        o.x = pack_bf16x2(v[j * 8 + 0] * (rinv * ca.x), v[j * 8 + 1] * (rinv * ca.y));
                        o.y = pack_bf16x2(v[j * 8 + 2] * (rinv * ca.z), v[j * 8 + 3] * (rinv * ca.w));
                        o.z = pack_bf16x2(v[j * 8 + 4] * (rinv * cb4.x), v[j * 8 + 5] * (rinv * cb4.y));
                        o.w = pack_bf16x2(v[j * 8 + 6] * (rinv * cb4.z), v[j * 8 + 7] * (rinv * cb4.w));
                        *reinterpret_cast<uint4 *>(rowp + ((j ^ ((rloc >> 1) & 3)) << 4)) = o;
                    }
                } else {
                uint8_t *rowp = stg + rloc * 128;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 c4 = __ldg(ci + j);
                    float4 o;
                    o.x = v[j * 4 + 0] * (rinv * c4.x), o.y = v[j * 4 + 1] * (rinv * c4.y);
                    o.z = v[j * 4 + 2] * (rinv * c4.z), o.w = v[j * 4 + 3] * (rinv * c4.w);
                    *reinterpret_cast<float4 *>(rowp + ((j ^ (rloc & 7)) << 4)) = o;   // SWIZZLE_128B like the store's tensor map
                }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {   // 32 rows x 32 columns: rows beyond R are clipped by the tensor map
                    tma_store_2d(&tmZ, cb * PG_BN + c32 * 32, (int)(row0 + q * 32), smem_u32(stg + q * (ZB ? 2048 : 4096)));
                    tma_store_commit();
                }
            }
        }
        if (lane == 0) tma_store_wait_all();
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// 2-D tensor (rows, cols) of fp32 (or bf16) elements with row pitch ld elements; box = 128 rows x 32 columns: 128-byte rows with
// SWIZZLE_128B (fp32), 64-byte rows with SWIZZLE_64B (bf16)
static int make_tmap(CUtensorMap *m, const void *base, long long rows, int cols, int ld, bool bf16 = false, int box_rows = T3_TM) {
    EncodeTiledFn fn = encode_fn();
    MVX_REQUIRE(fn, MVX_ECUDA, "cuTensorMapEncodeTiled entry point not available");
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * (bf16 ? 2 : 4)};
    const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MVX_REQUIRE(r == CUDA_SUCCESS, MVX_ECUDA, "cuTensorMapEncodeTiled failed");
    return MVX_OK;
}

template <bool RESIDENT, bool CAT, int PREC>
int launch_tc3_t(const T3Args &g, const CUtensorMap &tmX, const CUtensorMap &tmY, const CUtensorMap &tmX2, int grid, cudaStream_t st) {
    using S = T3Smem<RESIDENT>;
    static bool attr_set = false;
    if (!attr_set) {
        MVX_CUDA_CHECK(cudaFuncSetAttribute(tc3_layer_kernel<RESIDENT, CAT, PREC>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
        attr_set = true;
    }
    tc3_layer_kernel<RESIDENT, CAT, PREC><<<grid, t3_threads(RESIDENT ? 2 : 3, RESIDENT ? 2 : 1), S::kTotal, st>>>(g, tmX, tmY, tmX2);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

}  // namespace

bool tc3_layer_eligible(const LayerArgs &a) {
    if (!(a.f16_ok && a.in_stats && a.counts && !a.row_max && !a.plain && !a.a_pack)) return false;
    if (a.Cout != T3_BN || a.Cin % (2 * T3_KB) != 0 || (a.Cin != 128 && a.Cin % (3 * T3_KB) != 0) || a.Cin > 768 || (a.rows_mode != 1 && a.rows_mode != 2)) return false;
    if (a.rowcap % T3_TM != 0 || a.ldx % 4 != 0 || (a.Y && a.ldy % 4 != 0)) return false;
    if (a.vmax && !a.row_v) return false;
    if (a.y_bf16 || (a.x_bf16 && a.X2)) return false;
    if (a.X2) return a.x2_cols == 64 && a.Cin == 128 && a.in_C == 64 && a.cat_row_vox && a.ldx == 64;   // the fused concat of the last FCN
    return a.ldx == a.Cin && a.in_C == 0;
}

// defined in tc_layer.cu: packs W^T into the fp16 hi/lo (or bf16) chunk images + inverse column scales for 128-column tiles
int pack_weights_f16_128(const float *Wt, int Cin, int Cout, void *wpack, cudaStream_t st, bool bf16);

int launch_layer_tc3(const LayerArgs &a, int F, float *wpack, cudaStream_t st) {
    MVX_REQUIRE(tc3_layer_eligible(a) && wpack, MVX_EINVAL, "layer not eligible for the TMA-fed tensor-core kernel");
    const bool bf = tc_bf16_enabled();
    MVX_REQUIRE(bf || !a.x_bf16, MVX_EINVAL, "bf16 rows need the bf16 mode");
    int rc = pack_weights_f16_128(a.Wt, a.Cin, a.Cout, wpack, st, bf);
    if (rc) return rc;
    T3Args g{};
    g.a = a, g.wpack = wpack, g.F = F, g.row_tiles = a.rowcap / T3_TM, g.store = a.Y != nullptr;
    CUtensorMap tmX, tmY, tmX2;
    const int xcols = a.X2 ? a.Cin - a.x2_cols : a.Cin;
    rc = make_tmap(&tmX, a.X, (long long)F * a.rowcap, xcols, a.ldx, a.x_bf16 != 0);
    if (rc) return rc;
    if (a.Y) {
        rc = make_tmap(&tmY, a.Y, (long long)F * a.rowcap, a.Cout, a.ldy, false, 32);   // one box per epilogue warp
        if (rc) return rc;
    } else {
        tmY = tmX;
    }
    if (a.X2) {   // per-voxel half of the fused concat: (F * vcap, x2_cols) float bits
        rc = make_tmap(&tmX2, reinterpret_cast<const float *>(a.X2), (long long)F * a.vcap, a.x2_cols, a.x2_cols);
        if (rc) return rc;
    } else {
        tmX2 = tmX;
    }
    const long long slots = (long long)F * g.row_tiles;
    const int grid = (int)(slots < kSMs ? slots : kSMs);
    const bool resident = a.Cin == 128;
    if (bf) {
        if (a.X2) return launch_tc3_t<true, true, 1>(g, tmX, tmY, tmX2, grid, st);
        if (a.x_bf16) return resident ? launch_tc3_t<true, false, 2>(g, tmX, tmY, tmX2, grid, st) : launch_tc3_t<false, false, 2>(g, tmX, tmY, tmX2, grid, st);
        return resident ? launch_tc3_t<true, false, 1>(g, tmX, tmY, tmX2, grid, st) : launch_tc3_t<false, false, 1>(g, tmX, tmY, tmX2, grid, st);
    }
    if (a.X2) return launch_tc3_t<true, true, 0>(g, tmX, tmY, tmX2, grid, st);
    if (resident) return launch_tc3_t<true, false, 0>(g, tmX, tmY, tmX2, grid, st);
    return launch_tc3_t<false, false, 0>(g, tmX, tmY, tmX2, grid, st);
}

// defined in tc_layer.cu
static int g_pixel_persistent = 1;   // 0: the one-tile two-CTAs-per-SM kernel of tc_layer.cu for the pixel GEMM (mvx_set_gemm_mode(12), A/B timing)
void set_pixel_persistent(int on) { g_pixel_persistent = on; }
bool pixel_persistent_enabled() { return g_pixel_persistent != 0; }

bool pixel_gemm_persistent_eligible(const LayerArgs &a) {
    return g_pixel_persistent && a.plain && a.a_pack && a.Y && !a.counts && a.rows_fixed > 0 && a.Cin % PG_KB == 0 && a.Cout % PG_BN == 0 &&
           a.Cout <= 768 && a.ldy % 8 == 0;
}

int launch_pixel_gemm_persistent(const LayerArgs &a, float *wpack, cudaStream_t st) {
    MVX_REQUIRE(pixel_gemm_persistent_eligible(a) && wpack, MVX_EINVAL, "layer not eligible for the persistent pixel GEMM");
    int rc = pack_weights_f16_128(a.Wt, a.Cin, a.Cout, wpack, st, false);
    if (rc) return rc;
    PgArgs g{};
    g.a_pack = static_cast<const uint8_t *>(a.a_pack), g.a_rowinv = a.a_rowinv, g.wpack = reinterpret_cast<const uint8_t *>(wpack);
    g.R = a.rows_fixed, g.Cin = a.Cin, g.Cout = a.Cout, g.row_tiles = (int)ceil_div(a.rows_fixed, (long long)PG_TM);
    CUtensorMap tmZ;
    rc = make_tmap(&tmZ, a.Y, a.rows_fixed, a.Cout, a.ldy, a.y_bf16 != 0, 32);   // one 32-row box per epilogue warp
    if (rc) return rc;
    static bool attr_set = false;
    if (!attr_set) {
        MVX_CUDA_CHECK(cudaFuncSetAttribute(pixel_gemm_persistent_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PgSmem::kTotal));
        MVX_CUDA_CHECK(cudaFuncSetAttribute(pixel_gemm_persistent_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PgSmem::kTotal));
        attr_set = true;
    }
    const long long tiles = (long long)g.row_tiles * (a.Cout / PG_BN);
    const int grid = (int)(tiles < kSMs ? tiles : kSMs);
    if (a.y_bf16) pixel_gemm_persistent_kernel<true><<<grid, PG_THREADS, PgSmem::kTotal, st>>>(g, tmZ);
    else pixel_gemm_persistent_kernel<false><<<grid, PG_THREADS, PgSmem::kTotal, st>>>(g, tmZ);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

}  // namespace mvx
