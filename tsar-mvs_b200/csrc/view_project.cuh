// view_project.cuh -- the float32 projection rule shared by fusion.cu (DESIGN.md 4.6) and mesh.cu (4.8).
//
// One explicit-rounding operation per step, in the written order, so the C restatements (oracle/fusion_cpu.c,
// oracle/mesh_cpu.c, compiled with -ffp-contract=off) perform the same operations.
#pragma once
#include <cuda_runtime.h>

#include "pm_math.cuh"

namespace tsar {

__device__ __forceinline__ float dot3s(float a0, float b0, float a1, float b1, float a2, float b2) {
    return fadd(fadd(fmul(a0, b0), fmul(a1, b1)), fmul(a2, b2));
}

// A depth is used when it is finite and > 0 (NaN, 0, negatives and +inf are not).
__device__ __forceinline__ bool valid_depth(float d) { return d > 0.0f && d <= 3.402823466e38f; }

// c = R X + t, z = c.z, continuous pixel = (K c) / z.  Cam has row-major float K[9], R[9], t[3].
template <class Cam>
__device__ __forceinline__ void project(const Cam &c, float3 X, float &px, float &py, float &z) {
    const float cx = fadd(dot3s(c.R[0], X.x, c.R[1], X.y, c.R[2], X.z), c.t[0]);
    const float cy = fadd(dot3s(c.R[3], X.x, c.R[4], X.y, c.R[5], X.z), c.t[1]);
    const float cz = fadd(dot3s(c.R[6], X.x, c.R[7], X.y, c.R[8], X.z), c.t[2]);
    z = cz;
    px = fdiv(dot3s(c.K[0], cx, c.K[1], cy, c.K[2], cz), cz);
    py = fdiv(dot3s(c.K[3], cx, c.K[4], cy, c.K[5], cz), cz);
}

}  // namespace tsar
