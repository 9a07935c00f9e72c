// pm_kernels.cuh -- __global__ kernels of the PatchMatch path (random init, checkerboard propagation,
// plane refinement, explicit-plane evaluation, XORWOW row tables).  Instantiated per window variant by pm_inst_*.cu.
#pragma once
#include <type_traits>

#include "pm_core.cuh"
#include "pm_launch.h"
#include "pm_neighbours.cuh"

// Kernels are templates; two translation units that instantiate the same template arguments with different macro
// settings (PM_FAST_UNROLL, PM_WARP_COLS) would otherwise share one symbol and silently run the same code.  Each
// variant TU therefore places its kernels in its own namespace.
#ifndef PM_KERNEL_NS
#define PM_KERNEL_NS pm_default
#endif
#ifndef PM_WARP_COLS
#define PM_WARP_COLS 32   // columns of the CTA tile covered by one warp: 32 (1 row pair), 16 (2 row pairs) or 8 (4)
#endif

namespace tsar {
namespace PM_KERNEL_NS {

// shared memory carve-up common to the window kernels
template <int NT>
struct WinSmem {
    float2 *wt;  // [ns][NT]
    float *sp;   // [ns]
    __device__ __forceinline__ WinSmem(unsigned char *base, int ns) {
        wt = reinterpret_cast<float2 *>(base);
        sp = reinterpret_cast<float *>(base + (size_t)ns * NT * sizeof(float2));
    }
};

// quad sampling scratch (QuadScratch) of the thread's warp, behind the window table (quad_smem_offset)
template <int NT, int N1>
__device__ __forceinline__ QuadScratch<N1 ? N1 : 2> quad_scratch(unsigned char *base, int tid) {
    using QS = QuadScratch<N1 ? N1 : 2>;
    unsigned char *w = base + quad_smem_offset(NT, N1 * N1) + (size_t)(tid >> 5) * QS::bytes_per_warp();
    QS q;
    q.h = reinterpret_cast<float4 *>(w);
    q.n = reinterpret_cast<uint16_t *>(w + 32 * kQuadHWords * sizeof(float4));
    q.lane = tid & 31;
    return q;
}

template <int N1>
__device__ __forceinline__ void fill_spatial_table(const PmConst &c, float *sp, int tid, int nthreads) {
    const int n1y = N1 ? N1 : c.n1y;
    const int hrad = N1 ? N1 - 1 : c.hrad, vrad = N1 ? N1 - 1 : c.vrad;
    const int ns = N1 ? N1 * N1 : c.ns;
    for (int k = tid; k < ns; k += nthreads) {
        const int ii = k / n1y, jj = k - ii * n1y;
        sp[k] = spatial_term(-hrad + 2 * ii, -vrad + 2 * jj);
    }
}

// ---------------------------------------------------------------------------------------------
// (1) random plane initialisation -- gipuma_init_cu2 (gipuma.cu:679-729)
// ---------------------------------------------------------------------------------------------
template <int NT, int MINB, int N1, bool GEN, bool U8, bool QUAD>
__global__ void __launch_bounds__(NT, MINB) pm_init_kernel(const __grid_constant__ PmConst c, const float *__restrict__ ref,
                                                     const uint32_t *__restrict__ rng, int rng_len,
                                                     float4 *__restrict__ plane, float *__restrict__ cost) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WinSmem<NT> sm(smem_raw, N1 ? N1 * N1 : c.ns);
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    fill_spatial_table<N1>(c, sm.sp, tid, NT);
    __syncthreads();
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    const bool inside = x < c.W && y < c.H;
    if (QUAD ? __all_sync(0xffffffffu, !inside) : !inside) return;
    // quad sampling: a lane outside the image stays as a helper that fetches for its quad-mates; it works on the
    // nearest pixel (every read in bounds) and stores nothing
    if (QUAD) { x = min(x, c.W - 1); y = min(y, c.H - 1); }
    const QuadScratch<N1 ? N1 : 2> qs = quad_scratch<NT, N1>(smem_raw, tid);
    const WPair<NT> wt{sm.wt + tid};
    const RefStats rs = window_weights<NT, N1>(c, ref, x, y, sm.sp, wt);

    const uint32_t *row = rng + (size_t)y * c.rng_pitch + x;
    const int avail = rng_len - x;  // draws available to this pixel
    float vx, vy, vz;
    view_vector(c, x, y, vx, vy, vz);
    // disparity uniform in [min_disparity, max_disparity] (gipuma.cu:709)
    const float disp = ffma(uniform01(row[0]), fsub(c.max_disp, c.min_disp), c.min_disp);
    // Marsaglia point on the sphere (gipuma.cu:118-132)
    float mx, my, sum;
    int n = 1;
    do {
        mx = ffma(uniform01(row[min(n, avail - 1)]), 2.0f, -1.0f);
        my = ffma(uniform01(row[min(n + 1, avail - 1)]), 2.0f, -1.0f);
        n += 2;
        sum = ffma(mx, mx, fmul(my, my));
    } while (sum >= 1.0f && n + 1 < avail);
    const float sq = __fsqrt_rn(fsub(1.0f, sum));
    float nx = fmul(fadd(mx, mx), sq), ny = fmul(fadd(my, my), sq), nz = fsub(1.0f, fadd(sum, sum));
    if (dot3(nx, vx, ny, vy, nz, vz) > 0.0f) { nx = -nx; ny = -ny; nz = -nz; }  // vecOnHemisphere_cu :106-112
    const float depth = fdiv(fmul(c.f_cam0, c.baseline), disp);                  // :712
    float4 pl = make_float4(nx, ny, nz, 0.f);
    pl.w = plane_d(c, nx, ny, nz, x, y, depth);                                  // :715
    const MvResult r = multiview_cost<NT, N1, GEN, false, U8, false, QUAD>(c, x, y, pl, wt, rs, inside, &qs);
    if (QUAD && !inside) return;
    const size_t p = (size_t)y * c.W + x;
    plane[p] = pl;
    cost[p] = r.cost;
}

// ---------------------------------------------------------------------------------------------
// (2) red/black checkerboard propagation + plane refinement
//     gipuma_{black,red}_spatialProp_cu / _planeRefine_cu (gipuma.cu:847-1138)
// One thread per pixel of the launch's colour; block = 32 columns x (NT/32) row pairs, lane parity
// selects the row of the pair exactly as the reference's wrappers do (gipuma.cu:1099-1103).
// State is double buffered per colour: neighbours are read from `*_in` (pre-launch snapshot of both
// colours), the thread's own result goes to `*_out` (which may alias `*_in` when DO_SP is false).
// ---------------------------------------------------------------------------------------------

template <int NT, int MINB, int N1, bool GEN, bool U8, bool DO_SP, bool DO_PR, bool TILE, bool PIN, bool QUAD>
__global__ void __launch_bounds__(NT, MINB) pm_checker_kernel(const __grid_constant__ PmConst c,
                                                        const float *__restrict__ ref, const CheckerArgs a) {
    static_assert(!TILE || N1 > 0, "the tile layout needs a compile-time window");
    static_assert(!QUAD || (!TILE && PM_WARP_COLS == 32), "quad sampling: pair table, quads of 4 adjacent columns");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WinSmem<NT> sm(smem_raw, N1 ? N1 * N1 : c.ns);   // (TILE: the table holds floats, see checker_smem_bytes)
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int W = c.W, H = c.H;
    float *tile = nullptr;
    if (TILE) {
        // reference-image tile of the CTA: 32 + 2*hrad columns x 2*(NT/32) + 2*vrad rows, clamp addressing applied
        // while loading (same coordinate clamp as the window loop of window_weights)
        constexpr int HR = N1 - 1, TW = 32 + 2 * HR, TH = 2 * (NT / 32) + 2 * HR;
        float *wtab = reinterpret_cast<float *>(smem_raw);
        sm.sp = wtab + N1 * N1 * NT;
        tile = sm.sp + N1 * N1;
        const int x0 = (int)blockIdx.x * 32 - HR, y0 = (int)blockIdx.y * (NT / 32) * 2 - HR;
        for (int idx = tid; idx < kTilePitch * TH; idx += NT) {
            const int tx = idx % kTilePitch, ty = idx / kTilePitch;
            if (tx < TW) tile[idx] = __ldg(ref + (size_t)min(max(y0 + ty, 0), H - 1) * W + min(max(x0 + tx, 0), W - 1));
        }
    }
    fill_spatial_table<N1>(c, sm.sp, tid, NT);
    __syncthreads();
    // block = 32 columns x (NT/32) row pairs; lane parity selects the row of the pair exactly as the reference's
    // wrappers do (gipuma.cu:1099-1103).  (More compact warp footprints, PM_WARP_COLS = 16 or 8, measure the same to 0.3 %: texture wavefronts are per quad.)
    constexpr int WC = PM_WARP_COLS, WPR = 32 / WC;   // warps side by side in the 32-column tile
    int x = blockIdx.x * 32 + ((int)threadIdx.y % WPR) * WC + ((int)threadIdx.x % WC);
    const int rowpair = ((int)threadIdx.y / WPR) * (32 / WC) + ((int)threadIdx.x / WC);
    int y = (blockIdx.y * (NT / 32) + rowpair) * 2 + ((x + a.colour) & 1);
    const bool inside = x < W && y < H && y < c.y_limit;
    if (QUAD ? __all_sync(0xffffffffu, !inside) : !inside) return;
    // quad sampling: a lane outside the image or past y_limit stays as a helper that fetches for its quad-mates; it
    // works on the nearest pixel of the image (every read in bounds), evaluates nothing and stores nothing
    if (QUAD) { x = min(x, W - 1); y = min(y, H - 1); }
    const QuadScratch<N1 ? N1 : 2> qs = quad_scratch<NT, N1>(smem_raw, tid);
    const int own = a.colour;
    const int pidx = y * W + x;

    using WS = typename std::conditional<TILE, WTile<NT>, WPair<NT>>::type;
    WS wt;
    if constexpr (TILE) {
        wt.w = reinterpret_cast<float *>(smem_raw) + tid;
        wt.rt = tile + (y - (int)blockIdx.y * (NT / 32) * 2) * kTilePitch + (x - (int)blockIdx.x * 32);
    } else {
        wt.p = sm.wt + tid;
    }
    const RefStats rs = window_weights<NT, N1>(c, ref, x, y, sm.sp, wt);

    // (no dynamic indexing into the by-value argument struct: that would force a local-memory copy)
    const float *cS = own ? a.cost_in[1] : a.cost_in[0];
    const float *cO = own ? a.cost_in[0] : a.cost_in[1];
    const float4 *pS = own ? a.plane_in[1] : a.plane_in[0];
    const float4 *pO = own ? a.plane_in[0] : a.plane_in[1];
    float cost_now = cS[pidx];
    float4 norm_now = pS[pidx];
    float ratio_now = 0.f;
    int beview_now = 0;
    bool meta_dirty = false;

    // refinement state (planeRefinement_cu + getRndDispAndUnitVector_cu, gipuma.cu:582-676)
    float vx = 0.f, vy = 0.f, vz = 0.f, depth_now = 0.f, deltaN = 1.0f, deltaZ = fmul(c.max_disp, 0.5f);
    const uint32_t *row = a.rng + (size_t)y * c.rng_pitch + x;
    const float fb = fmul(c.baseline, c.f_params);
    int draw = 0;

    // ONE hypothesis loop with ONE call site of the cost function: steps 0..7 are the eight propagation
    // candidates (gipuma.cu:888-1042, in the reference's order), steps >= 8 the refinement rounds.  Keeping a
    // single copy of the (large, unrolled) cost code is what keeps the kernel inside the instruction cache.
#pragma unroll 1
    for (int step = DO_SP ? 0 : 8;; step++) {
        float4 cand;
        if (QUAD) cand = norm_now;   // a lane that evaluates nothing still publishes a homography to its quad
        float cand_depth = 0.f;
        bool eval = false;
        if (step < 8) {
            // -- pick the neighbour whose plane is tried at this pixel (pm_neighbours.cuh)
            bool bown;
            const int best = pick_neighbour(step, x, y, W, H, pidx, cO, cS, bown);
            if (best >= 0) {
                // spatialPropagation_cu (gipuma.cu:525-566).  The cost has no side effect, so it is skipped when
                // the depth-range test would reject the plane anyway.
                cand = bown ? pS[best] : pO[best];
                const float dep = plane_depth(c, cand, x, y);
                eval = (dep >= c.depthMin && dep <= c.depthMax);
            }
        } else {
            if (!DO_PR) break;
            if (step == 8) {
                view_vector(c, x, y, vx, vy, vz);
                depth_now = plane_depth(c, norm_now, x, y);  // gipuma.cu:1073
            }
            if (!(deltaZ >= 0.01f)) break;                   // for (deltaZ = max/2; deltaZ >= 0.01; deltaZ /= 10)
            const float u0 = uniform01(row[draw]), u1 = uniform01(row[draw + 1]), u2 = uniform01(row[draw + 2]),
                        u3 = uniform01(row[draw + 3]);
            draw += 4;
            const float disp = fdiv(fb, depth_now);                          // :596
            const float lo = fminf(fadd(c.min_disp, disp), deltaZ);          // = -minDelta, :601
            const float hi = fminf(fsub(c.max_disp, disp), deltaZ);          // = maxDelta,  :602
            float nd = fadd(ffma(u0, fadd(lo, hi), -lo), disp);              // disp + between(minDelta, maxDelta)
            nd = fminf(c.max_disp, fmaxf(c.min_disp, nd));                   // :608
            cand_depth = fdiv(fb, nd);                                       // :610
            const float two = fadd(deltaN, deltaN);
            float nx = fadd(norm_now.x, ffma(two, u1, -deltaN));             // :613-615
            float ny = fadd(norm_now.y, ffma(two, u2, -deltaN));
            float nz = fadd(norm_now.z, ffma(two, u3, -deltaN));
            const float rn = rsqrtf(dot3(nx, nx, ny, ny, nz, nz));           // normalize_cu
            nx = fmul(nx, rn); ny = fmul(ny, rn); nz = fmul(nz, rn);
            if (dot3(vx, nx, vy, ny, vz, nz) > 0.0f) { nx = -nx; ny = -ny; nz = -nz; }
            cand = make_float4(nx, ny, nz, plane_d(c, nx, ny, nz, x, y, cand_depth));   // :654
            eval = true;                                                     // no depth-range test (:665)
            deltaZ = fdiv(deltaZ, 10.0f);
            deltaN = fmul(deltaN, 0.25f);
        }
        if (QUAD) eval = eval && inside;
        if (QUAD ? __any_sync(0xffffffffu, eval) : eval) {
            const MvResult r = multiview_cost<NT, N1, GEN, false, U8, PIN, QUAD>(c, x, y, cand, wt, rs, eval, &qs);
            if (eval && r.cost < cost_now) {
                cost_now = r.cost; norm_now = cand; ratio_now = r.ratio; beview_now = r.beview; meta_dirty = true;
                depth_now = cand_depth;  // only read by the refinement rounds
            }
        }
    }

    if (QUAD && !inside) return;
    a.cost_out[pidx] = cost_now;
    a.plane_out[pidx] = norm_now;
    if (meta_dirty) { a.ratio[pidx] = ratio_now; a.beview[pidx] = beview_now; }
}

// ---------------------------------------------------------------------------------------------
// (3) multi-view matching cost for explicit (pixel, plane) pairs -- the unit the bench counts
// ---------------------------------------------------------------------------------------------
template <int NT, int MINB, int N1, bool GEN, bool PXF, bool U8>
__global__ void __launch_bounds__(NT, MINB) pm_eval_kernel(const __grid_constant__ PmConst c, const float *__restrict__ ref,
                                                     int n, const int2 *__restrict__ xy,
                                                     const float4 *__restrict__ planes, float *__restrict__ cost,
                                                     int *__restrict__ beview, float *__restrict__ ratio) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WinSmem<NT> sm(smem_raw, N1 ? N1 * N1 : c.ns);
    const int tid = threadIdx.x;
    fill_spatial_table<N1>(c, sm.sp, tid, NT);
    __syncthreads();
    const int i = blockIdx.x * NT + tid;
    if (i >= n) return;
    const int2 p = xy[i];
    const WPair<NT> wt{sm.wt + tid};
    const RefStats rs = window_weights<NT, N1>(c, ref, p.x, p.y, sm.sp, wt);
    const MvResult r = multiview_cost<NT, N1, GEN, PXF, U8>(c, p.x, p.y, planes[i], wt, rs);
    cost[i] = r.cost;
    beview[i] = r.beview;
    ratio[i] = r.ratio;
}

// cost of the planes currently stored (used by tsar_load_planes when no cost is supplied)
template <int NT, int MINB, int N1, bool GEN, bool U8>
__global__ void __launch_bounds__(NT, MINB) pm_cost_of_state_kernel(const __grid_constant__ PmConst c,
                                                              const float *__restrict__ ref,
                                                              const float4 *__restrict__ plane,
                                                              float *__restrict__ cost) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WinSmem<NT> sm(smem_raw, N1 ? N1 * N1 : c.ns);
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    fill_spatial_table<N1>(c, sm.sp, tid, NT);
    __syncthreads();
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= c.W || y >= c.H) return;
    const WPair<NT> wt{sm.wt + tid};
    const RefStats rs = window_weights<NT, N1>(c, ref, x, y, sm.sp, wt);
    const size_t p = (size_t)y * c.W + x;
    cost[p] = multiview_cost<NT, N1, GEN, false, U8>(c, x, y, plane[p], wt, rs).cost;
}

}  // namespace PM_KERNEL_NS
using namespace PM_KERNEL_NS;
}  // namespace tsar
