// 11x11 window (scripts: --blocksize=11): 36 samples.  64-thread CTAs, >= 8 CTAs/SM (128 registers, 18.4 KB of
// shared memory for the per-thread weight table), the whole window unrolled in the branch-free sampling loop
// (36 texture fetches in flight per thread).  Chosen by measurement on B200 (profiles/r01_variants_C2.json, checker
// kernel ms at C2): this shape 19.43; 128 threads x 4 CTAs 19.51 (sampling loop unrolled 3: 19.85, 2: 20.84); 256 x 2
// 20.02; 9 CTAs of 64 threads (112 regs, 48 B spilled; round 2) 27.4; >= 5 CTAs/SM of 128 threads (96 regs) 20.1-20.6; >= 6 (80 regs) 21.3; >= 3 (168 regs) 22.1;
// the 19x19 variant's tile layout (half the shared memory per thread, -DPM_TILE=1; round 2) 19.89;
// warps covering 16 x 2 or 8 x 4 row pairs (PM_WARP_COLS) 19.56 / 19.58; texture quads of 2 columns x 4 rows instead
// of 4 x 2: 20.18; one image row per warp (quad = 7 x 1 pixels): 19.67.  All shapes give bit-identical output
// (the quad / row mappings were experiments of the commit that recorded them and are not kept in the kernel).
#define PM_FAST_UNROLL(n1) (n1)
#define PM_VARIANT pm_variant_w11
#define PM_LABEL "w11"
#define PM_NT 64
#ifndef PM_MINB
#define PM_MINB 8
#endif
#define PM_N1 6
#define PM_GEN false
#define PM_QUAD 1   // quad-cooperative sampling kernels (pm_core.cuh, view_cost_quad)
#include "pm_inst.inc"
