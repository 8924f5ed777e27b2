// Error text, launch counter, kernel-selection modes and version of the mvx_b200 C-ABI library.
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace mvx {
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// The accepted numbers of mvx_set_gemm_mode / mvx_set_fusion_mode / mvx_set_fold_mode, process-wide.
static struct {
    int gemm = 1, fusion = 1, fold = 0;
} g_modes;

// gemm mode:
// 0 = the exact-fp32 SIMT kernel everywhere
// 1 = tensor cores where eligible (default): 3xFP16 for the fused path's BatchNorm-ed layers, 3xTF32 for the dense layer API;
//     conv1 / fcn2 / last FCN through the TMA-fed A-from-TMEM persistent kernel (tc3_layer.cu)
// 5 = like 1 with tc_layer.cu's one-tile kernel for those layers, and the dense layer API (mvx_fcn_forward ...) also uses fp16
//     operands: the caller promises inputs of O(1) magnitude (tests)
// 6 = bf16 mode: single-pass bf16 operands for the same layers mode 1 runs in 3xFP16
// 9 = like 1 with the one-tile kernel of tc_layer.cu for conv1 / fcn2 / last FCN
// 10 = like 1 with prep_vfe1 / prep_vfe2 materialising the VFE inputs also in inference (the earlier default, kept for A/B timing and
//      for inspecting X6 / X7)
// 12 = like 1 with the one-tile two-CTAs-per-SM kernel (tc_layer.cu) for the pixel GEMM instead of the persistent one (A/B timing)
// 2, 3, 4, 7, 8 and 11 selected variants that have been removed (DESIGN.md §5) and are rejected; the modes above keep their numbers.
bool simt_only() { return g_modes.gemm == 0; }
bool dense_f16() { return g_modes.gemm == 5; }
bool tc3_enabled() { return g_modes.gemm == 1 || g_modes.gemm == 6 || g_modes.gemm == 10 || g_modes.gemm == 12; }
bool bf16_mode() { return g_modes.gemm == 6; }
bool pixel_gemm_persistent() { return g_modes.gemm != 12; }
bool vfe_fused() { return g_modes.gemm != 10; }

// fold mode: 0 = the run-structured combine kernel (default), 2 = the first combine kernel (row-by-row walk), kept for A/B runs;
// 1 (conv1 with fcn1's BatchNorm folded into per-frame weights) was removed: measured slower
bool combine_v1() { return g_modes.fold == 2; }

// fusion mode: 1 (default) = pixel-first fcn1 - one tensor-core GEMM per FPN level over the map pixels, then a 12-corner combine per
// point row (gather.cuh CombineArgs); 0 = materialise the gathered (K,768) matrix A1 and run fcn1 over the point rows (the layout the
// training-mode backward needs: dW1 = dpre1^T A1); 2 = pixel-first without the side stream for the map branch (serial, for per-stage
// profiling). Pixel-first needs the tensor-core pixel GEMM, so gemm mode 0 runs row-first.
bool pixel_first(bool train) { return !train && g_modes.fusion != 0 && g_modes.gemm != 0; }
bool map_on_side_stream() { return g_modes.fusion != 2; }
}  // namespace mvx

extern "C" const char *mvx_last_error(void) { return mvx::g_err; }
extern "C" int mvx_version(void) { return 100; }
extern "C" int64_t mvx_launch_count(void) { return mvx::g_launches.load(std::memory_order_relaxed); }

extern "C" int mvx_set_gemm_mode(int32_t mode) {
    constexpr unsigned kModes = 1u << 0 | 1u << 1 | 1u << 5 | 1u << 6 | 1u << 9 | 1u << 10 | 1u << 12;
    MVX_REQUIRE(mode >= 0 && mode <= 12 && (kModes >> mode & 1u), MVX_EINVAL, "gemm mode must be 0, 1, 5, 6, 9, 10 or 12");
    mvx::g_modes.gemm = mode;
    return MVX_OK;
}

extern "C" int mvx_set_fusion_mode(int32_t mode) {
    MVX_REQUIRE(mode >= 0 && mode <= 2, MVX_EINVAL, "fusion mode must be 0, 1 or 2");
    mvx::g_modes.fusion = mode;
    return MVX_OK;
}

extern "C" int mvx_set_fold_mode(int32_t mode) {
    MVX_REQUIRE(mode == 0 || mode == 2, MVX_EINVAL, "fold mode must be 0 or 2");
    mvx::g_modes.fold = mode;
    return MVX_OK;
}
