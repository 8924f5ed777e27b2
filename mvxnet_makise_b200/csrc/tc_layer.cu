// Stage 3 on the 5th-generation tensor cores: y = relu(norm_in(X) W^T + b) + weighted BatchNorm sums, for the
// GEMM-shaped layers (fcn1 768->768, conv1 768->128, fcn2 128->128), hand-written tcgen05 / TMEM / bulk-copy PTX.
//
// fp32-accurate on TF32 hardware ("3xTF32"): every fp32 operand is split hi = top 19 bits, lo = x - hi (exact), and
// D += A_lo*B_hi + A_hi*B_lo + A_hi*B_hi with fp32 accumulation in TMEM; the dropped A_lo*B_lo term and the
// truncation of the lo parts are ~2^-22 relative (measured parity: see tests/test_gpu_parity.py).
//
// One CTA = 256 rows x BN columns (two M=128 accumulators in TMEM, 2*BN columns), K in chunks of 16 fp32
// (64-byte rows, SWIZZLE_64B K-major canonical layout), 3-stage mbarrier pipeline:
//   warps 0-7 : A producers. Coalesced 16-byte loads of the raw activations, BatchNorm of the producer layer
//               applied in registers ((x - mean) * rstd), hi/lo split, swizzled st.shared, fence.proxy.async,
//               mbarrier arrive. After the main loop the same warps run the epilogue.
//   warp 8    : B producer. One cp.async.bulk (TMA engine, SASS UBLKCP) per stage: the weights were pre-split
//               and pre-swizzled into the exact shared-memory image by pack_weights_kernel (32 KB per stage).
//   warp 9    : TMEM allocation, then the single-thread tcgen05.mma issuer; tcgen05.commit frees the stage.
// Epilogue: tcgen05.ld (32 lanes x 32 columns per warp) -> +bias, ReLU -> padded smem tile -> (a) coalesced
// row-major stores of the raw activations, (b) per-column weighted sums in fp64 -> one atomicAdd per column.
// A 256-row tile amortises the weight stream: per 16-k chunk a CTA pulls 16 KB of A and 32 KB of B for
// 1536 tensor cycles (31 B/cycle/SM), which the 148-SM L2 can sustain; a 128-row tile could not (53 B/cycle/SM).
#include "layers.cuh"
#include "tc_common.cuh"


#include <cstdlib>

namespace mvx {

namespace {

constexpr int kTM = 256;        // rows per CTA
constexpr int kStages = 3;
constexpr int kEpiCols = 128;   // columns per epilogue pass
constexpr int kEpiLd = kEpiCols + 4;

template <int BN, int STAGES = kStages, bool HALF_EPI = false>
struct Smem {
    static constexpr int kAHalf = kTM * kBK * 4;      // 16 KB: A_hi (then A_lo)
    static constexpr int kBHalf = BN * kBK * 4;       // B_hi (then B_lo)
    static constexpr int kStage = 2 * kAHalf + 2 * kBHalf;
    static constexpr int kTiles = STAGES * kStage;
    static constexpr int kEpi = (HALF_EPI ? 1 : 2) * 128 * kEpiLd * 4;  // 128-row halves of one 128-column pass (one at a time if HALF_EPI)
    static constexpr int kMain = kTiles > kEpi ? kTiles : kEpi;
    // after the tiles: mean[768], rstd[768], bias[BN], row_w[256], barriers, tmem pointer
    static constexpr int kMean = kMain;
    static constexpr int kRstd = kMean + 768 * 4;
    static constexpr int kBias = kRstd + 768 * 4;
    static constexpr int kRowW = kBias + BN * 4;
    static constexpr int kRowV = kRowW + kTM * 4;      // voxel id of each row (per-voxel max), -1 = none
    static constexpr int kRowInv = kRowV + kTM * 4;    // fp16 variant: inverse row scales
    static constexpr int kColInv = kRowInv + kTM * 4;  // fp16 variant: inverse column scales
    static constexpr int kBars = kColInv + BN * 4;     // full[3], empty[3], accum
    static constexpr int kTmemPtr = kBars + 8 * 8;
    static constexpr int kTotal = kTmemPtr + 16 + 1024;  // + slack for the 1024-byte alignment of the base
};

// ---- weight packing: W^T (Cin, Cout) fp32 -> per (column tile, k chunk) the shared-memory image [hi | lo] ----
template <int BN>
__global__ void __launch_bounds__(256) pack_weights_kernel(const float *__restrict__ Wt, int Cin, int Cout, float *__restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= Cin * Cout) return;
    const int k = e / Cout, n = e - k * Cout;
    const int ct = n / BN, nl = n - ct * BN, kc = k / kBK, kl = k - kc * kBK;
    float hi, lo;
    split_tf32(Wt[e], hi, lo);
    const size_t blob = ((size_t)ct * (Cin / kBK) + kc) * (2 * BN * kBK);  // floats
    const uint32_t off = sw64_offset(nl, kl >> 2) / 4 + (kl & 3);
    out[blob + off] = hi;
    out[blob + BN * kBK + off] = lo;
}

// ---- fp16 operand variant ("3xFP16") ---------------------------------------------------------------------------
// Same three-product split, but hi/lo are IEEE fp16 (11 significant bits, like TF32) fed to kind::f16 MMAs, which run
// at twice the TF32 rate and read half the shared-memory bytes per MAC. fp16 has a 5-bit exponent, so operands are
// first scaled by an exact power of two: every weight column (output channel) by 2^-e with max|w| in [0.5,1), activation
// rows by a per-row power of two when the caller supplies row maxima (raw FPN features) and by 1 for BatchNorm-ed
// inputs (|z| <= sqrt(R) << 65504). The epilogue multiplies the accumulator by the inverse scales (exact). With hi =
// rn16(x) and lo = rn16(x - hi) the representation error is max(2^-23 |x|, 2^-25) per element (lo may be subnormal),
// i.e. fp32-level relative to the row scale; products of two fp16 values are exact in the fp32 accumulator.
// W^T (Cin, Cout) -> per (column tile, 32-k chunk) the shared-memory image [hi | lo] in fp16, columns pre-scaled;
// colinv[n] = 1 / scale_n. One CTA per output column.
template <int BN, bool BF1>
// blockIdx.y = K block: W^T rows [y Cin, (y+1) Cin) packed at out + y * level_bytes (the pixel GEMM's three FPN levels in one launch)
__global__ void __launch_bounds__(256) pack_weights_f16_kernel(const float *__restrict__ Wt, int Cin, int Cout, uint8_t *__restrict__ out,
                                                               float *__restrict__ colinv, size_t level_bytes = 0) {
    __shared__ float s_max[256];
    const int n = blockIdx.x, tid = threadIdx.x;
    Wt += (size_t)blockIdx.y * Cin * Cout;
    out += blockIdx.y * level_bytes;
    colinv = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(colinv) + blockIdx.y * level_bytes);
    float mx = 0.f;
    for (int k = tid; k < Cin; k += 256) mx = fmaxf(mx, fabsf(Wt[(size_t)k * Cout + n]));
    s_max[tid] = mx;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s) s_max[tid] = fmaxf(s_max[tid], s_max[tid + s]);
        __syncthreads();
    }
    const float sc = BF1 ? 1.f : pow2_scale(s_max[0]);
    if (tid == 0) colinv[n] = 1.f / sc;
    const int ct = n / BN, nl = n - ct * BN;
    for (int k = tid; k < Cin; k += 256) {
        const int kc = k >> 5, kl = k & 31;
        const float v = Wt[(size_t)k * Cout + n] * sc;
        const size_t blob = ((size_t)ct * (Cin / 32) + kc) * (2 * BN * 64);  // bytes
        const uint32_t off = sw64_offset(nl, kl >> 3) + (kl & 7) * 2;
        if constexpr (BF1) {
            *reinterpret_cast<__nv_bfloat16 *>(out + blob + off) = __float2bfloat16_rn(v);
        } else {
            const __half h = __float2half_rn(v);
            const __half l = __float2half_rn(v - __half2float(h));
            *reinterpret_cast<__half *>(out + blob + off) = h;
            *reinterpret_cast<__half *>(out + blob + BN * 64 + off) = l;
        }
    }
}

// BF1: single-pass bf16 operands (no lo parts, one MMA per K-step, no scaling: bf16 has the fp32 exponent range) - the
// reduced-precision mode whose tolerance is stated separately (tests/test_gpu_parity.py::test_bf16_mode_tolerance).
// TWO: two CTAs per SM (BN = 128, 16-bit operands): 2 pipeline stages, the epilogue staged one 128-row half at a time (96 KB of
// shared memory, 256 TMEM columns, <= 102 registers), so one CTA's epilogue overlaps the other's main loop.
// producer warps: the 16-bit producers are instruction-latency bound with 8 warps (ncu: ~1.8 warp instructions per cycle
// and SM, conv1 at 2.7k cycles per stage against 0.8k of MMA), so the one-CTA-per-SM variant runs 16 of them (2 rows of
// a stage per thread instead of 4)
__host__ __device__ constexpr int tc_producer_warps(bool f16, bool two) { return (f16 && !two) ? 16 : 8; }

// APK: the A operand arrives pre-packed (LayerArgs::a_pack): no register producers, one bulk copy of 32 KB per stage.
template <int BN, bool F16, bool BF1 = false, bool TWO = false, bool APK = false>
__global__ void __launch_bounds__(tc_producer_warps(F16, TWO) * 32 + 64, TWO ? 2 : 1) tc_layer_kernel(LayerArgs a, const float *__restrict__ wpack) {
    static_assert(!APK || (F16 && !BF1), "pre-packed A is a 3xFP16 variant");
    constexpr int PW = tc_producer_warps(F16, TWO), PT = PW * 32, NT = PT + 64;   // producer warps / threads, CTA threads
    static_assert(!BF1 || F16, "the bf16 variant shares the 16-bit operand path");
    static_assert(!TWO || (F16 && BN == 128), "the two-CTA variant is the 16-bit, 128-column kernel");
    constexpr int STAGES = TWO ? 2 : kStages;
    using S = Smem<BN, STAGES, TWO>;
    constexpr int KB = F16 ? 32 : kBK;   // k per pipeline stage: one 64-byte swizzle row of fp16 / tf32
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // keep the pointer in the shared address space (pointer arithmetic only, no integer round trip): STS/LDS, not ST.E/LD.E
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    float *s_mean = reinterpret_cast<float *>(smem + S::kMean);
    float *s_rstd = reinterpret_cast<float *>(smem + S::kRstd);
    float *s_bias = reinterpret_cast<float *>(smem + S::kBias);
    float *s_roww = reinterpret_cast<float *>(smem + S::kRowW);
    int *s_rowv = reinterpret_cast<int *>(smem + S::kRowV);
    const uint32_t bars = sbase + S::kBars;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
    const uint32_t accum_bar = bars + 8u * (2 * STAGES);
    volatile uint32_t *tmem_ptr = reinterpret_cast<volatile uint32_t *>(smem + S::kTmemPtr);

    const int f = blockIdx.z, ctile = blockIdx.x, n0 = ctile * BN, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    long long n_rows = a.rows_fixed;
    double Rstat = (double)a.rows_fixed;
    int Kf = 0;
    if (a.counts) {
        const int N = a.counts[f * 4 + 0];
        Kf = a.counts[f * 4 + 1];
        n_rows = a.rows_mode == 1 ? Kf + 1 : (a.rows_mode == 2 ? Kf + N : (a.rows_mode == 3 ? N : a.rows_fixed));
        Rstat = (double)N * (double)a.T;
    }
    long long row_tile = blockIdx.y;
    if constexpr (APK) {
        if (a.tile_list) {   // pixel GEMM: blockIdx.y walks the level's active row tiles (gather.cuh PixelTiles)
            const int e = a.tile_bounds[0] + (int)blockIdx.y;
            if (e >= a.tile_bounds[1]) return;
            row_tile = a.tile_list[e] & 0xFFFFFF;
        }
    }
    const long long row0 = row_tile * kTM;  // column tiles of one row tile are launch-adjacent: A hits L2
    if (row0 >= n_rows) return;  // uniform for the CTA, before any barrier / TMEM allocation
    const int nk = a.Cin / KB;
    float *s_rowinv = reinterpret_cast<float *>(smem + S::kRowInv);   // F16: 1 / (power-of-two scale of each row)
    float *s_colinv = reinterpret_cast<float *>(smem + S::kColInv);   // F16: 1 / (power-of-two scale of each output column)

    // ---- one-time setup ------------------------------------------------------------------------------------
    if (a.in_stats) {
        const int inC = a.in_C > 0 ? a.in_C : a.Cin;   // fused concat: both parts share the producer layer's statistics
        for (int c = tid; c < a.Cin; c += NT) {
            const double *st = a.in_stats + ((size_t)f * inC + c % inC) * 2;
            const double m = st[0] / Rstat;
            double var = st[1] / Rstat - m * m;
            var = var < 0.0 ? 0.0 : var;
            s_mean[c] = (float)m;
            s_rstd[c] = (float)(1.0 / sqrt(var + a.eps));
        }
    }
    for (int c = tid; c < BN; c += NT) s_bias[c] = a.plain ? 0.f : a.bias[n0 + c];
    if constexpr (F16) {
        // [blob: Cin*Cout*4 bytes | colinv: Cout floats]
        const float *colinv = reinterpret_cast<const float *>(reinterpret_cast<const uint8_t *>(wpack) + (size_t)a.Cin * a.Cout * 4);
        for (int c = tid; c < BN; c += NT) s_colinv[c] = colinv[n0 + c];
        for (int r = tid; r < kTM; r += NT) {
            const long long rr = row0 + r;
            if constexpr (APK) s_rowinv[r] = (a.a_rowinv && rr < n_rows) ? a.a_rowinv[(size_t)f * a.rowcap + rr] : 1.f;
            else s_rowinv[r] = (!BF1 && a.row_max && rr < n_rows) ? 1.f / pow2_scale(a.row_max[(size_t)f * a.rowcap + rr]) : 1.f;
        }
    }
    for (int r = tid; r < kTM; r += NT) {
        const long long rr = row0 + r;
        const float w = rr < n_rows ? (a.row_w ? a.row_w[(size_t)f * a.rowcap + rr] : 1.f) : 0.f;
        s_roww[r] = w;
        int v = -1;
        if (a.vmax && w != 0.f) {
            if (a.row_v) v = (a.rows_mode == 1 && rr >= Kf) ? -1 : a.row_v[(size_t)f * a.rowv_cap + rr];
            else v = (int)(rr / a.T);
        }
        s_rowv[r] = v;
    }
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), APK ? 1 : PT + 1);   // APK: only the bulk-copy thread's expect_tx arrive
            mbar_init(empty_bar(s), 1);
        }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == PW + 1) {  // TMEM: 2*BN fp32 accumulator columns (power of two >= 32)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + S::kTmemPtr), "r"(2 * BN)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const bool mma_only = (MVX_DBG(a) & 8) != 0;
    if (mma_only && warp != PW + 1) {
    } else if (warp < PW && APK) {
        // pre-packed A: nothing to produce (these warps run the epilogue)
    } else if (warp < PW && F16) {
        // ================= A producers, fp16 operands: a thread owns 8 k (one 16-byte chunk of fp16) of 4 rows ======
        constexpr int RS = PT / 4, RPT = kTM / RS;   // row stride between a thread's rows, rows per thread (4 or 2)
        const int c = tid & 3, rsub = tid >> 2;
        const float *Xf = a.X + ((size_t)f * a.rowcap + row0) * a.ldx + c * 8;
        bool valid[RPT];
        float rs[RPT];
        const float *x2row[RPT];   // fused concat: this row's source for the trailing x2_cols input columns
        const int split = a.X2 ? a.Cin - a.x2_cols : a.Cin;
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const long long rr = row0 + rsub + RS * i;
            valid[i] = rr < n_rows;
            rs[i] = 1.f / s_rowinv[rsub + RS * i];   // power of two: exact
            x2row[i] = nullptr;
            if (a.X2 && valid[i]) {
                const int v = rr >= Kf ? (int)(rr - Kf) : a.cat_row_vox[(size_t)f * a.cat_rowv_cap + rr];
                x2row[i] = reinterpret_cast<const float *>(a.X2) + ((size_t)f * a.vcap + v) * a.x2_cols + c * 8;
            }
        }
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        constexpr int PF = TWO ? 1 : 2;   // chunks of raw activations in flight in registers
        auto load_chunk = [&](float4 (&buf)[2 * RPT], int kc) {
            const bool second = kc * KB >= split;
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                const float4 *p = second ? reinterpret_cast<const float4 *>(x2row[i] + (kc * KB - split))
                                         : reinterpret_cast<const float4 *>(Xf + (size_t)(rsub + RS * i) * a.ldx + kc * KB);
                buf[2 * i] = valid[i] ? __ldg(p) : z4;
                buf[2 * i + 1] = valid[i] ? __ldg(p + 1) : z4;
            }
        };
        auto produce = [&](float4 (&buf)[2 * RPT], int kc) {
            float4 cur[2 * RPT];
#pragma unroll
            for (int i = 0; i < 2 * RPT; ++i) cur[i] = buf[i];
            if (a.in_stats) {
                const int k = kc * KB + c * 8;
                const float4 m0 = *reinterpret_cast<const float4 *>(s_mean + k), m1 = *reinterpret_cast<const float4 *>(s_mean + k + 4);
                const float4 r0 = *reinterpret_cast<const float4 *>(s_rstd + k), r1 = *reinterpret_cast<const float4 *>(s_rstd + k + 4);
#pragma unroll
                for (int i = 0; i < RPT; ++i) {
                    if (valid[i]) {
                        cur[2 * i].x = (cur[2 * i].x - m0.x) * r0.x, cur[2 * i].y = (cur[2 * i].y - m0.y) * r0.y;
                        cur[2 * i].z = (cur[2 * i].z - m0.z) * r0.z, cur[2 * i].w = (cur[2 * i].w - m0.w) * r0.w;
                        cur[2 * i + 1].x = (cur[2 * i + 1].x - m1.x) * r1.x, cur[2 * i + 1].y = (cur[2 * i + 1].y - m1.y) * r1.y;
                        cur[2 * i + 1].z = (cur[2 * i + 1].z - m1.z) * r1.z, cur[2 * i + 1].w = (cur[2 * i + 1].w - m1.w) * r1.w;
                    }
                }
            }
            if (kc + PF < nk) load_chunk(buf, kc + PF);
            const int s = kc % STAGES;
            const uint32_t ph = (kc / STAGES) & 1;
            if (lane == 0) mbar_wait(empty_bar(s), ph ^ 1);
            __syncwarp();
            uint8_t *stage = smem + (size_t)s * S::kStage;
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                const uint32_t off = sw64_offset(rsub + RS * i, c);
                if constexpr (BF1) {
                    uint4 hi;
                    hi.x = pack_bf16x2(cur[2 * i].x, cur[2 * i].y), hi.y = pack_bf16x2(cur[2 * i].z, cur[2 * i].w);
                    hi.z = pack_bf16x2(cur[2 * i + 1].x, cur[2 * i + 1].y), hi.w = pack_bf16x2(cur[2 * i + 1].z, cur[2 * i + 1].w);
                    *reinterpret_cast<uint4 *>(stage + off) = hi;
                } else {
                    const float sc = rs[i];
                    uint4 hi, lo;
                    split_f16_pair(cur[2 * i].x * sc, cur[2 * i].y * sc, hi.x, lo.x);
                    split_f16_pair(cur[2 * i].z * sc, cur[2 * i].w * sc, hi.y, lo.y);
                    split_f16_pair(cur[2 * i + 1].x * sc, cur[2 * i + 1].y * sc, hi.z, lo.z);
                    split_f16_pair(cur[2 * i + 1].z * sc, cur[2 * i + 1].w * sc, hi.w, lo.w);
                    *reinterpret_cast<uint4 *>(stage + off) = hi;
                    *reinterpret_cast<uint4 *>(stage + S::kAHalf + off) = lo;
                }
            }
            fence_async_smem();
            mbar_arrive(full_bar(s));
        };
        if constexpr (TWO) {   // one chunk in flight per thread (register budget of two CTAs per SM; 16 producer warps per SM)
            float4 buf0[2 * RPT];
            load_chunk(buf0, 0);
            for (int kc = 0; kc < nk; ++kc) produce(buf0, kc);
        } else {
            float4 buf0[2 * RPT], buf1[2 * RPT];
            load_chunk(buf0, 0);
            if (nk > 1) load_chunk(buf1, 1);
            for (int kc = 0; kc < nk; kc += 2) {
                produce(buf0, kc);
                if (kc + 1 < nk) produce(buf1, kc + 1);
            }
        }
    } else if (warp < PW) {
        // ================= A producers ===========================================================================
        const int c = tid & 3, rsub = tid >> 2;  // 16-byte chunk of the 64-byte k-chunk row; rows rsub + 64*i
        const float *Xf = a.X + ((size_t)f * a.rowcap + row0) * a.ldx + c * 4;
        bool valid[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) valid[i] = row0 + rsub + 64 * i < n_rows;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        auto load_chunk = [&](float4 (&buf)[4], int kc) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                buf[i] = (valid[i] && !(MVX_DBG(a) & 4)) ? __ldg(reinterpret_cast<const float4 *>(Xf + (size_t)(rsub + 64 * i) * a.ldx + kc * kBK)) : z4;
        };
        // two chunks of raw activations are always in flight in registers (DRAM/L2 latency >> one chunk of MMA time)
        auto produce = [&](float4 (&buf)[4], int kc) {
            float4 cur[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) cur[i] = buf[i];
            if (a.in_stats) {
                const int k = kc * kBK + c * 4;
                const float m0 = s_mean[k], m1 = s_mean[k + 1], m2 = s_mean[k + 2], m3 = s_mean[k + 3];
                const float r0 = s_rstd[k], r1 = s_rstd[k + 1], r2 = s_rstd[k + 2], r3 = s_rstd[k + 3];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (valid[i]) {
                        cur[i].x = (cur[i].x - m0) * r0;
                        cur[i].y = (cur[i].y - m1) * r1;
                        cur[i].z = (cur[i].z - m2) * r2;
                        cur[i].w = (cur[i].w - m3) * r3;
                    }
                }
            }
            if (kc + 2 < nk) load_chunk(buf, kc + 2);
            const int s = kc % STAGES;
            const uint32_t ph = (kc / STAGES) & 1;
            if (lane == 0) mbar_wait(empty_bar(s), ph ^ 1);  // one poller per warp
            __syncwarp();
            uint8_t *stage = smem + (size_t)s * S::kStage;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float4 hi, lo;
                split_tf32(cur[i].x, hi.x, lo.x);
                split_tf32(cur[i].y, hi.y, lo.y);
                split_tf32(cur[i].z, hi.z, lo.z);
                split_tf32(cur[i].w, hi.w, lo.w);
                const uint32_t off = sw64_offset(rsub + 64 * i, c);
                *reinterpret_cast<float4 *>(stage + off) = hi;
                *reinterpret_cast<float4 *>(stage + S::kAHalf + off) = lo;
            }
            if (!(MVX_DBG(a) & 1)) fence_async_smem();  // make the generic-proxy writes visible to the tensor core (async proxy)
            mbar_arrive(full_bar(s));
        };
        float4 buf0[4], buf1[4];
        load_chunk(buf0, 0);
        if (nk > 1) load_chunk(buf1, 1);
        for (int kc = 0; kc < nk; kc += 2) {
            produce(buf0, kc);
            if (kc + 1 < nk) produce(buf1, kc + 1);
        }
    } else if (warp == PW) {
        // ================= B producer: one bulk copy per stage ===================================================
        if (lane == 0) {
            const float *src = wpack + (size_t)ctile * nk * (2 * BN * kBK);
            for (int kc = 0; kc < nk; ++kc) {
                const int s = kc % STAGES;
                const uint32_t ph = (kc / STAGES) & 1;
                mbar_wait(empty_bar(s), ph ^ 1);
                if constexpr (APK) {
                    mbar_arrive_expect_tx(full_bar(s), 2 * S::kAHalf + 2 * S::kBHalf);
                    const uint8_t *asrc = static_cast<const uint8_t *>(a.a_pack) + ((size_t)row_tile * nk + kc) * (2 * S::kAHalf);
                    bulk_g2s(sbase + s * S::kStage, asrc, 2 * S::kAHalf, full_bar(s));
                } else {
                    mbar_arrive_expect_tx(full_bar(s), 2 * S::kBHalf);
                }
                bulk_g2s(sbase + s * S::kStage + 2 * S::kAHalf, src + (size_t)kc * (2 * BN * kBK), 2 * S::kBHalf, full_bar(s));
            }
        }
    } else {
        // ================= MMA issuer (one thread) ================================================================
        if (lane == 0) {
            // D fp32, A/B TF32 (format 2) or F16 (format 0), K-major both, N = BN, M = 128
            constexpr uint32_t fmt = BF1 ? 1u : (F16 ? 0u : 2u);   // kind::f16: 0 = fp16, 1 = bf16; kind::tf32: 2 = tf32
            constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | ((128u >> 4) << 24);
            for (int kc = 0; kc < nk; ++kc) {
                const int s = kc % STAGES;
                const uint32_t ph = (kc / STAGES) & 1;
                if (!mma_only) mbar_wait(full_bar(s), ph);
                tc_fence_after();
                const uint32_t sA = sbase + s * S::kStage, sB = sA + 2 * S::kAHalf;
#pragma unroll
                for (int h = 0; h < 2; ++h) {          // the two 128-row halves -> two accumulators
                    const uint32_t d = tmem_base + h * BN;
                    const uint32_t aoff = h * (128 * 64);
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {   // two MMA K-steps (8 tf32 / 16 fp16 = 32 bytes) per stage row: +32 bytes inside the swizzle atom
                        const uint64_t a_hi = make_desc(sA + aoff + ks * 32), a_lo = make_desc(sA + S::kAHalf + aoff + ks * 32);
                        const uint64_t b_hi = make_desc(sB + ks * 32), b_lo = make_desc(sB + S::kBHalf + ks * 32);
                        if constexpr (BF1) {
                            mma_f16(d, a_hi, b_hi, idesc, (kc | ks) != 0);
                        } else if constexpr (F16) {
                            mma_f16(d, a_lo, b_hi, idesc, (kc | ks) != 0);
                            mma_f16(d, a_hi, b_lo, idesc, 1);
                            mma_f16(d, a_hi, b_hi, idesc, 1);
                        } else {
                            mma_tf32(d, a_lo, b_hi, idesc, (kc | ks) != 0);
                            mma_tf32(d, a_hi, b_lo, idesc, 1);
                            mma_tf32(d, a_hi, b_hi, idesc, 1);
                        }
                    }
                }
                mma_commit(empty_bar(s));  // frees the stage when the MMAs above have read it
            }
            mma_commit(accum_bar);         // accumulators complete
        }
    }

    // ================= epilogue (warps 0-7; warps 8-9 only join the barriers) =====================================
    __syncwarp();
    if (warp < 8) {
        mbar_wait(accum_bar, 0);
        tc_fence_after();
    }
    __syncthreads();  // every stage buffer is idle now: reuse the tile memory for the output staging
    float *ytile = reinterpret_cast<float *>(smem);  // [2 halves (TWO: 1)][128 rows][kEpiLd]
    const int q = warp & 3;                          // TMEM lane quarter of this warp
    const float floor_v = a.plain ? -INFINITY : 0.f;  // plain mode: no ReLU (bias is zero)
    constexpr int HP = TWO ? 2 : 1;                  // half passes: TWO stages one 128-row accumulator at a time
    constexpr int TR = TWO ? 128 : kTM;              // rows in the staging tile
    for (int pass = 0; pass < ((MVX_DBG(a) & 2) ? 0 : BN / kEpiCols); ++pass) {
#pragma unroll 1
        for (int hp = 0; hp < HP; ++hp) {
            if (warp < 8) {
                // TWO: all 8 warps drain accumulator `hp`, warps w and w+4 share a lane quarter and split the 128 columns;
                // otherwise warps 0-3 drain accumulator 0 and warps 4-7 accumulator 1
                const int half = TWO ? hp : (warp >> 2);
                const int cpart = TWO ? (warp >> 2) * 64 : 0, ncb = TWO ? 2 : kEpiCols / 32;
                const int rloc = half * 128 + q * 32 + lane;          // row inside the 256-row CTA tile
                float *yrow = ytile + (size_t)(TWO ? q * 32 + lane : rloc) * kEpiLd + cpart;
                const float rinv = F16 ? s_rowinv[rloc] : 1.f;
#pragma unroll 1
                for (int cb = 0; cb < ncb; ++cb) {
                    float v[32];
                    const int col = pass * kEpiCols + cpart + cb * 32;
                    tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + half * BN + col, v);
                    if constexpr (F16) {   // undo the power-of-two operand scales (exact)
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] *= rinv * s_colinv[col + j];
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 o;
                        o.x = fmaxf(v[j] + s_bias[col + j], floor_v);
                        o.y = fmaxf(v[j + 1] + s_bias[col + j + 1], floor_v);
                        o.z = fmaxf(v[j + 2] + s_bias[col + j + 2], floor_v);
                        o.w = fmaxf(v[j + 3] + s_bias[col + j + 3], floor_v);
                        *reinterpret_cast<float4 *>(yrow + cb * 32 + j) = o;
                    }
                }
            }
            __syncthreads();
            if (tid < 256) {
                const int rbase = TWO ? hp * 128 : 0;    // first CTA-tile row of the staging tile
                // coalesced raw stores first (one warp per row, 32 lanes x 16 bytes = 128 columns): they drain while the sums run
                if (a.Y && a.y_nchw) {   // channel-major: a warp stores one column, its lanes consecutive rows (128-byte runs)
                    const long long nr = min((long long)TR, n_rows - row0 - rbase);
                    for (int c = warp; c < kEpiCols; c += 8) {
                        float *ycol = a.Y + ((size_t)f * a.Cout + n0 + pass * kEpiCols + c) * a.rowcap + row0 + rbase;
                        for (int r = lane; r < nr; r += 32) ycol[r] = ytile[(size_t)r * kEpiLd + c];
                    }
                } else if (a.Y) {
                    for (int r = warp; r < TR; r += 8) {
                        if (row0 + rbase + r >= n_rows) break;
                        const float4 o = *reinterpret_cast<const float4 *>(ytile + (size_t)r * kEpiLd + lane * 4);
                        const size_t e = ((size_t)f * a.rowcap + row0 + rbase + r) * a.ldy + n0 + pass * kEpiCols + lane * 4;   // element index
                        if (a.y_bf16) {
                            uint2 ob;
                            ob.x = pack_bf16x2(o.x, o.y), ob.y = pack_bf16x2(o.z, o.w);
                            *reinterpret_cast<uint2 *>(reinterpret_cast<__nv_bfloat16 *>(a.Y) + e) = ob;
                        } else
                        *reinterpret_cast<float4 *>(a.Y + e) = o;
                    }
                }
            }
            // weighted column sums and per-voxel max: thread = (column, row group), ALL warps of the CTA take part (the
            // producer / MMA warps are idle by now), so the one-CTA 16-bit variant walks 4 groups of 64 rows instead of 2 of
            // 128. Each group of 16 rows is loaded once into registers (16 independent LDS in flight) and serves both the
            // sums and the max. Ordinary rows (multiplicity 1) are summed in fp32 over the 16 rows and the runs in fp64; the
            // weighted pad rows take an exact fp64 side path. Rows of a voxel are consecutive: running max in registers,
            // one atomicMax per run.
            constexpr int NG = (!TWO && NT >= 512) ? 4 : 2;   // row groups
            constexpr int RG = TR / NG;                       // rows per group
            double *s_part = reinterpret_cast<double *>(smem + S::kMean);
            double stat_sy = 0.0, stat_syy = 0.0;
            if (tid < NG * 128 && !a.plain) {
                const int rbase = TWO ? hp * 128 : 0;
                const int col = tid & 127, rg = tid >> 7;
                double sy = 0.0, syy = 0.0;
                int *vm = a.vmax ? a.vmax + (size_t)f * a.vcap * a.Cout + n0 + pass * kEpiCols + col : nullptr;
                int cv = -1;
                float cm = 0.f;
                for (int r0 = rg * RG; r0 < rg * RG + RG; r0 += 16) {
                    float yv[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) yv[j] = ytile[(size_t)(r0 + j) * kEpiLd + col];
                    float ps = 0.f, pss = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float w = s_roww[rbase + r0 + j];
                        const float y = yv[j];
                        const float my = w == 1.f ? y : 0.f;
                        ps += my;
                        pss = fmaf(my, y, pss);
                        if (w != 1.f && w != 0.f) {
                            const double wy = (double)w * (double)y;
                            sy += wy;
                            syy = fma(wy, (double)y, syy);
                        }
                    }
                    sy += (double)ps;
                    syy += (double)pss;
                    if (vm) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int v = s_rowv[rbase + r0 + j];
                            if (v != cv) {
                                if (cv >= 0) atomicMax(vm + (size_t)cv * a.Cout, __float_as_int(cm));
                                cv = v;
                                cm = yv[j];
                            } else {
                                cm = fmaxf(cm, yv[j]);
                            }
                        }
                    }
                }
                if (vm && cv >= 0) atomicMax(vm + (size_t)cv * a.Cout, __float_as_int(cm));
                // the fp64 atomics of all CTAs of a frame meet on 2 x Cout addresses: combine the row groups of this CTA first
                // (partials of groups 1.. go through the idle mean/rstd area: 3 x 128 x 2 doubles = its 6 KB)
                if (rg > 0) {
                    s_part[((rg - 1) * 128 + col) * 2] = sy;
                    s_part[((rg - 1) * 128 + col) * 2 + 1] = syy;
                }
                stat_sy = sy, stat_syy = syy;
            }
            __syncthreads();
            if (tid < 128 && !a.plain) {
#pragma unroll
                for (int g = 1; g < NG; ++g) {
                    stat_sy += s_part[((g - 1) * 128 + tid) * 2];
                    stat_syy += s_part[((g - 1) * 128 + tid) * 2 + 1];
                }
                double *o = a.out_stats + ((size_t)f * a.Cout + n0 + pass * kEpiCols + tid) * 2;
                atomicAdd(o, stat_sy);
                atomicAdd(o + 1, stat_syy);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == PW + 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * BN) : "memory");
    }
}

template <int BN, bool F16, bool BF1 = false, bool TWO = false, bool APK = false>
int launch_tc(const LayerArgs &a, int F, float *wpack, cudaStream_t st) {
    using S = Smem<BN, TWO ? 2 : kStages, TWO>;
    const int rc = set_smem_attributes<tc_layer_kernel<BN, F16, BF1, TWO, APK>>(S::kTotal, TWO ? 100 : -1);
    if (rc) return rc;
    const int total = a.Cin * a.Cout;
    if (F16) {   // [fp16 hi|lo images: Cin*Cout*4 bytes][inverse column scales: Cout floats]
        uint8_t *blob = reinterpret_cast<uint8_t *>(wpack);
        pack_weights_f16_kernel<BN, BF1><<<a.Cout, 256, 0, st>>>(a.Wt, a.Cin, a.Cout, blob, reinterpret_cast<float *>(blob + (size_t)total * 4));
    } else {
        pack_weights_kernel<BN><<<(total + 255) / 256, 256, 0, st>>>(a.Wt, a.Cin, a.Cout, wpack);
    }
    MVX_LAUNCH_CHECK();
    const long long max_rows = a.counts ? a.rowcap : a.rows_fixed;
    dim3 grid(a.Cout / BN, (unsigned)ceil_div(max_rows, kTM), F);
    tc_layer_kernel<BN, F16, BF1, TWO, APK><<<grid, tc_producer_warps(F16, TWO) * 32 + 64, S::kTotal, st>>>(a, wpack);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}


}  // namespace

int pack_weights_f16_128(const float *Wt, int Cin, int Cout, void *wpack, cudaStream_t st, bool bf16) {
    uint8_t *blob = static_cast<uint8_t *>(wpack);
    if (bf16) pack_weights_f16_kernel<128, true><<<Cout, 256, 0, st>>>(Wt, Cin, Cout, blob, reinterpret_cast<float *>(blob + (size_t)Cin * Cout * 4));
    else
    pack_weights_f16_kernel<128, false><<<Cout, 256, 0, st>>>(Wt, Cin, Cout, blob, reinterpret_cast<float *>(blob + (size_t)Cin * Cout * 4));
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

int pack_weights_f16_128_levels(const float *Wt, int Cin, int Cout, int levels, void *wpack, size_t level_bytes, cudaStream_t st) {
    uint8_t *blob = static_cast<uint8_t *>(wpack);
    pack_weights_f16_kernel<128, false><<<dim3(Cout, levels), 256, 0, st>>>(Wt, Cin, Cout, blob, reinterpret_cast<float *>(blob + (size_t)Cin * Cout * 4),
                                                                              level_bytes);
    MVX_LAUNCH_CHECK();
    return MVX_OK;
}

bool tc_layer_eligible(const LayerArgs &a) {
    // the 768 bound sizes the shared BatchNorm tables of the input: a plain product without them may be deeper
    return a.Cin % kBK == 0 && (a.Cin <= 768 || (a.plain && !a.in_stats)) && a.Cout % 128 == 0 && a.ldx % 4 == 0 &&
           (a.Y == nullptr || a.ldy % 4 == 0);
}

size_t tc_wpack_bytes(int Cin, int Cout) { return (size_t)2 * Cin * Cout * sizeof(float); }

int launch_layer_tc(const LayerArgs &a_in, int F, float *wpack, cudaStream_t st) {
    LayerArgs a = a_in;
#ifdef MVX_DEVTOOLS
    if (const char *e = getenv("MVX_DBG")) a.dbg = atoi(e);
#endif
    MVX_REQUIRE(tc_layer_eligible(a) && wpack, MVX_EINVAL, "layer not eligible for the tensor-core kernel");
    const long long max_rows = a.counts ? a.rowcap : a.rows_fixed;
    if (max_rows <= 0) return MVX_OK;
    if (a.y_nchw) {
        MVX_REQUIRE(a.plain && !a.f16_ok && !a.y_bf16 && !a.a_pack && !a.counts && a.rows_fixed == a.rowcap && a.Y, MVX_EINVAL,
                    "channel-major output: plain 3xTF32 product over rows_fixed == rowcap rows per frame");
        return a.Cout % 256 == 0 ? launch_tc<256, false>(a, F, wpack, st) : launch_tc<128, false>(a, F, wpack, st);
    }
    MVX_REQUIRE(!a.X2 || (a.f16_ok && a.Cin % 32 == 0 && a.x2_cols % 32 == 0 && a.counts), MVX_EINVAL,
                "fused concat input needs the 16-bit tensor-core producer");
    if (bf16_mode() && tc3_layer_eligible(a)) return launch_layer_tc3(a, F, wpack, st);   // bf16 mode of the TMA-fed kernel
    if (a.f16_ok && bf16_mode() && a.Cin % 32 == 0) {   // reduced precision: one bf16 product per K-step
        if (a.Cout % 256 == 0) return launch_tc<256, true, true>(a, F, wpack, st);
        return launch_tc<128, true, true>(a, F, wpack, st);
    }
    if (a.a_pack) {   // A pre-packed by the producing kernel: pure bulk-copy + MMA pipeline
        MVX_REQUIRE(a.Cin % 32 == 0 && !a.in_stats && !a.X2 && a.rows_mode == 0 && F == 1, MVX_EINVAL,
                    "pre-packed A: unsupported layer configuration");
        // no register producers here, so the two-CTAs-per-SM form (128-column tiles, 2 stages, half-at-a-time epilogue) costs
        // no duplicated operand conversion: one CTA's epilogue overlaps the other's bulk copies and MMAs (0.552 ms for the pixel
        // GEMM against 0.593 ms with one 256-column CTA per SM)
        return launch_tc<128, true, false, true, true>(a, F, wpack, st);
    }
    // conv1 / fcn2 / last FCN on the TMA-fed, A-from-TMEM persistent kernel (conv1 0.79 -> 0.68 ms, fcn2 0.32 -> 0.21, FCN 0.47 -> 0.39
    // against the one-tile kernel, which gemm modes 5 and 9 keep)
    if (tc3_enabled() && tc3_layer_eligible(a)) return launch_layer_tc3(a, F, wpack, st);
    if (a.f16_ok && a.Cin % 32 == 0) {   // 3xFP16: half the tensor cycles and operand bytes of 3xTF32
        if (a.Cout % 256 == 0) return launch_tc<256, true>(a, F, wpack, st);
        return launch_tc<128, true>(a, F, wpack, st);
    }
    if (a.Cout % 256 == 0) return launch_tc<256, false>(a, F, wpack, st);
    return launch_tc<128, false>(a, F, wpack, st);
}

}  // namespace mvx
