// pm_launch.h -- host-callable launchers of the PatchMatch kernels, one set per compiled window
// variant (each variant is its own translation unit so the build parallelises).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pm_core.cuh"

namespace tsar {

struct CheckerArgs {
    const float4 *plane_in[2];  // [colour] full-size arrays, colour = (x+y)&1
    const float *cost_in[2];
    float4 *plane_out;          // own colour
    float *cost_out;
    float *ratio;
    int *beview;
    const uint32_t *rng;
    int colour;
};

enum { PM_MODE_SP = 1, PM_MODE_PR = 2, PM_MODE_FUSED = 3 };

struct PmVariant {
    const char *name;
    // quad != 0 (only where has_quad; init: with u8, checker: with u8 and PmConst::k_pinhole): quad-cooperative
    // sampling (pm_core.cuh, view_cost_quad); otherwise cudaErrorInvalidValue.  Bit-identical results.
    bool has_quad;
    // u8 != 0: sample the 8-bit copies of the source views (PmConst::tex8); bit-identical results
    cudaError_t (*init)(int u8, int quad, const PmConst &, const float *ref, const uint32_t *rng, int rng_len,
                        float4 *plane, float *cost, cudaStream_t);
    cudaError_t (*checker)(int u8, int quad, int mode, const PmConst &, const float *ref, const CheckerArgs &,
                           cudaStream_t);
    cudaError_t (*eval)(int u8, int wrapper_rounding, const PmConst &, const float *ref, int n, const int2 *xy, const float4 *planes, float *cost,
                        int *beview, float *ratio, cudaStream_t);
    cudaError_t (*cost_of_state)(int u8, const PmConst &, const float *ref, const float4 *plane, float *cost, cudaStream_t);
};

extern const PmVariant pm_variant_w11;      // 11x11 window (hRad 5, 36 samples), n_best <= 2 / COMB_BEST_N
extern const PmVariant pm_variant_w19;      // 19x19 window (hRad 9, 100 samples), n_best <= 2 / COMB_BEST_N
extern const PmVariant pm_variant_generic;  // any window, any combination (run-time loops)

cudaError_t pm_launch_rng_table(uint32_t *table, int pitch, int H, int len, unsigned long long seed, cudaStream_t);
// n_tables (<= kRngBatchMax) tables in one launch, table t at tables + t * stride, seeded seeds[t]
constexpr int kRngBatchMax = 64;
cudaError_t pm_launch_rng_tables(uint32_t *tables, size_t stride, int n_tables, const unsigned long long *seeds, int pitch, int H,
                                 int len, cudaStream_t);
// candidate statistics of the checkerboard launch that would run on this state (debug instrumentation, pm_misc.cu)
constexpr int kCandStatHist = 13;    // out[13 .. 21]: pixels by number of distinct, not-own candidates (0..8)
constexpr int kCandStatWords = 22;   // out[0..12]: pixels, candidates behind the border guards, in depth range (= executed
                                     // evaluations / V), duplicates of the own plane, duplicates of an earlier candidate,
                                     // distinct; warp rounds today, with per-lane compaction, with perfect packing; warps;
                                     // the same three without the own-plane rule (distinct2 sum, max, packed)
cudaError_t pm_launch_cand_stats(const PmConst &c, const CheckerArgs &a, unsigned long long *out, cudaStream_t s);
cudaError_t pm_launch_merge_colour(int W, int H, int colour, const float4 *psrc, const float *csrc, float4 *pdst,
                                   float *cdst, cudaStream_t);

}  // namespace tsar
