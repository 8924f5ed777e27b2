// Shared helpers for the mvx_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mvx_b200.h"

namespace mvx {

void set_error(const char *fmt, ...);
void count_launch(int n = 1);

#define MVX_CUDA_CHECK(expr)                                                                         \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            mvx::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));    \
            return MVX_ECUDA;                                                                        \
        }                                                                                            \
    } while (0)

#define MVX_LAUNCH_CHECK()                                                                           \
    do {                                                                                             \
        mvx::count_launch();                                                                         \
        cudaError_t _e = cudaGetLastError();                                                         \
        if (_e != cudaSuccess) {                                                                     \
            mvx::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MVX_ECUDA;                                                                        \
        }                                                                                            \
    } while (0)

#define MVX_REQUIRE(cond, code, msg)                                                                 \
    do {                                                                                             \
        if (!(cond)) {                                                                               \
            mvx::set_error("%s:%d: %s", __FILE__, __LINE__, msg);                                    \
            return code;                                                                             \
        }                                                                                            \
    } while (0)

// Kernel selection by the mode switches of the C ABI (defined in runtime.cu, where the modes are described)
bool simt_only();               // gemm mode 0: the exact-fp32 SIMT kernels everywhere
bool dense_f16();               // gemm mode 5: the dense layer API uses fp16 operands
bool tc3_enabled();             // gemm mode 1, 6, 10 or 12: conv1 / fcn2 / last FCN on the TMA-fed kernel (tc3_layer.cu)
bool bf16_mode();               // gemm mode 6
bool pixel_gemm_persistent();   // gemm mode other than 12: the persistent pixel GEMM
bool vfe_fused();               // gemm mode other than 10: inference builds the VFE inputs in the layer's loader
bool combine_v1();              // fold mode 2: the first (row-by-row) combine kernel
bool pixel_first(bool train);   // a forward runs fcn1 pixel-first: not training, fusion mode other than 0, gemm mode other than 0
bool map_on_side_stream();      // fusion mode other than 2: the map branch of a pixel-first forward runs on a side stream

constexpr int kSMs = 148;  // B200
constexpr int kMaxDevices = 64;

// Raises kernel K's dynamic shared-memory limit to `bytes` (and sets its shared-memory carveout when carveout >= 0) on the current
// device, once per device: function attributes belong to a device's context, so every device a process launches K on needs its own
// call.
template <auto K>
int set_smem_attributes(int bytes, int carveout = -1) {
    static bool done[kMaxDevices] = {};
    int dev = 0;
    MVX_CUDA_CHECK(cudaGetDevice(&dev));
    MVX_REQUIRE(dev >= 0 && dev < kMaxDevices, MVX_EINVAL, "device ordinal out of range");
    if (done[dev]) return MVX_OK;
    MVX_CUDA_CHECK(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (carveout >= 0) MVX_CUDA_CHECK(cudaFuncSetAttribute(K, cudaFuncAttributePreferredSharedMemoryCarveout, carveout));
    done[dev] = true;
    return MVX_OK;
}

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// streaming (evict-first) 16-byte store: the dense grid is written once and not re-read by this path
__device__ __forceinline__ void st_cs_f4(float4 *p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// the same for 16 and 8 bytes of packed 16-bit elements
__device__ __forceinline__ void st_cs_u4(uint4 *p, uint4 v) {
    asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_cs_u2(uint2 *p, uint2 v) {
    asm volatile("st.global.cs.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ float4 ld_nc_f4(const float4 *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

// block-wide exclusive scan of one int per thread (blockDim.x <= 1024, multiple of 32). Returns the
// exclusive prefix; *total receives the block sum (valid in all threads).
__device__ __forceinline__ int block_exclusive_scan(int v, int *total) {
    __shared__ int warp_sums[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    __syncthreads();  // protect warp_sums reuse across calls
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int w = lane < nw ? warp_sums[lane] : 0;
        int winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += t;
        }
        warp_sums[lane] = winc;  // inclusive over warps
    }
    __syncthreads();
    const int base = wid == 0 ? 0 : warp_sums[wid - 1];
    *total = warp_sums[nw - 1];
    return base + inc - v;
}

// the same for one 64-bit value per thread (two packed 32-bit counters scan in one pass: they do not carry into each other
// as long as each total stays below 2^32)
__device__ __forceinline__ unsigned long long block_exclusive_scan_u64(unsigned long long v, unsigned long long *total) {
    __shared__ unsigned long long warp_sums64[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    __syncthreads();  // protect warp_sums64 reuse across calls
    if (lane == 31) warp_sums64[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned long long winc = lane < nw ? warp_sums64[lane] : 0ull;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += t;
        }
        warp_sums64[lane] = winc;  // inclusive over warps
    }
    __syncthreads();
    const unsigned long long base = wid == 0 ? 0ull : warp_sums64[wid - 1];
    *total = warp_sums64[nw - 1];
    return base + inc - v;
}

}  // namespace mvx
