// ransac_kernels.cuh -- per-region plane fitting for textureless regions ("per-segment plane fitting",
// north-star item 4; SURVEY section 8 row f1).  Reference: the CPU loop in main.cpp:1520-1730
// (calcLinePara main.cpp:147-164): for every region flagged textureless, back-project its reliable pixels,
// run 10 000 RANSAC triples with an adaptive inlier threshold, then 1000 x 4 local perturbation rounds;
// about 7e8 double residuals per region on one CPU core in the reference.
//
// Here: device-side stable compaction of the region's reliable pixels (raster order, as the reference collects
// them), back-projection, then ONE persistent cooperative kernel (ransac_fit_kernel) fits all textureless regions of the
// view: hypotheses are counted in batches by the whole grid (count phase: a CTA keeps a 256-point slice of one region in
// registers as doubles and runs through the <= 1000 planes of the batch from shared memory; per-warp ballots, shared
// then global atomics), and between two grid.sync() one CTA per region applies the loop-carried rules (select phase:
// best-so-far, adaptive threshold, commit of the first accepted perturbation and the cursor behind it).  The loop ends on
// the device; the host waits once, for the result.  Scratch lives in the context (grow-only).  All arithmetic is IEEE
// double without contraction, in the reference's evaluation order, so the result is bit-identical to the reference's own
// loop (main.cpp:1520-1730 compiled by oracle/build_ref.sh) given the same random numbers.  The reference
// draws them from rand()/system_clock (not reproducible); the caller supplies the stream instead (the values
// rand() would have returned, 46 000 per region) or a seed for a device-generated stream (ransac_rand_kernel).
// Kept quirks: the A coefficient of calcLinePara uses (y3-y1) twice (main.cpp:159); ties (>=) replace the best.
// Deviation: when a region has more than 50 000 reliable pixels the reference keeps a random subset of 49 999
// (std::shuffle with a clock seed); we keep an evenly strided subset.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "glue_kernels.cuh"

namespace tsar {

constexpr int kRansacKeepAll = 50000;      // main.cpp:1541: lists of up to 50 000 points are used whole ...
constexpr int kRansacCut = 49999;          // main.cpp:1547-1549: ... longer ones are cut to 49 999
constexpr int kRansacIters = 10000;        // main.cpp:1603
constexpr int kRefineRounds = 1000;        // main.cpp:1662
constexpr int kRansacRandPerRegion = 3 * kRansacIters + 4 * 4 * kRefineRounds;

// ---- stable compaction of one region's reliable pixels ------------------------------------------------------
__global__ void ransac_flag_kernel(const float *__restrict__ scale, const float *__restrict__ canny, int n, int region,
                                   int *__restrict__ block_counts) {
    __shared__ int warp_sums[32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = (i < n && scale[i] == 1.0f && (int)canny[i] == region) ? 1 : 0;
    const unsigned b = __ballot_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += warp_sums[w];
        block_counts[blockIdx.x] = s;
    }
}

__global__ void ransac_scan_blocks_kernel(int *block_counts, int nblocks, int *total) {  // single thread block
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nblocks; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int v = i < nblocks ? block_counts[i] : 0;
        // inclusive scan inside the block (Hillis-Steele through shared memory)
        __shared__ int buf[1024];
        buf[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < (int)blockDim.x; o <<= 1) {
            const int t = threadIdx.x >= o ? buf[threadIdx.x - o] : 0;
            __syncthreads();
            buf[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nblocks) block_counts[i] = carry + buf[threadIdx.x] - v;  // exclusive
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry += buf[threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void ransac_scatter_kernel(const float *__restrict__ scale, const float *__restrict__ canny, int n, int region,
                                      const int *__restrict__ block_offsets, int *__restrict__ list) {
    __shared__ int warp_off[32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = (i < n && scale[i] == 1.0f && (int)canny[i] == region) ? 1 : 0;
    const unsigned b = __ballot_sync(0xffffffffu, f);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_off[warp] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) { const int t = warp_off[w]; warp_off[w] = s; s += t; }
    }
    __syncthreads();
    if (f) list[block_offsets[blockIdx.x] + warp_off[warp] + __popc(b & ((1u << lane) - 1))] = i;
}

struct RansacJob {
    const float3 *pts;   // region's points
    int n;               // number of points (0: region skipped, plane left unchanged); written by ransac_points_kernel
    float size;          // cannylines->size[region]
    const uint32_t *rnd; // kRansacRandPerRegion values, in the order the reference calls rand()
    float4 *out;         // cannylines->norm4[region]
};

// back-projection of the (sub-sampled) list: main.cpp:1574-1598, float arithmetic, no contraction.  The list length stays
// on the device (*total): the kernel is launched for the largest possible list and records the number of points used in
// the region's job, so the host never waits for a count.
__global__ void ransac_points_kernel(const __grid_constant__ GlueConst g, const float *__restrict__ depth,
                                     const int *__restrict__ list, const int *__restrict__ total, float3 *__restrict__ pts,
                                     RansacJob *__restrict__ job) {
    const int n_all = *total;
    const int n_used = n_all <= kRansacKeepAll ? n_all : kRansacCut;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) job->n = n_used;
    if (k >= n_used) return;
    const int src = (n_all == n_used) ? k : (int)(((long long)k * n_all) / n_used);
    const int p = list[src];
    const float disp = fdiv(fmul(g.f_params, g.baseline), depth[p]);
    const int px = p % g.W, py = p / g.W;
    const float x = fsub(fmul(disp, (float)px), g.Pc[0]), y = fsub(fmul(disp, (float)py), g.Pc[1]), z = fsub(disp, g.Pc[2]);
    float3 o;
    o.x = fadd(fadd(fmul(g.Minv[0], x), fmul(g.Minv[1], y)), fmul(g.Minv[2], z));
    o.y = fadd(fadd(fmul(g.Minv[3], x), fmul(g.Minv[4], y)), fmul(g.Minv[5], z));
    o.z = fadd(fadd(fmul(g.Minv[6], x), fmul(g.Minv[7], y)), fmul(g.Minv[8], z));
    pts[k] = o;
}

// The values rand() would return, generated on the device from a seed (tsar_fit_region_planes_seeded): a counter-based
// stream, value i of region r = top 31 bits of splitmix64(seed ^ (r << 32) ^ i) -- non-negative ints like rand()'s.
__host__ __device__ __forceinline__ uint32_t ransac_rand_value(unsigned long long seed, int region, int index) {
    unsigned long long z = seed ^ ((unsigned long long)(uint32_t)region << 32) ^ (unsigned long long)(uint32_t)index;
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 33);
}
__global__ void ransac_rand_kernel(uint32_t *__restrict__ rnd, const int *__restrict__ regions, int n_targets, int per_region,
                                   unsigned long long seed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
    if (i < per_region && t < n_targets) rnd[(size_t)t * per_region + i] = ransac_rand_value(seed, regions[t], i);
}

// ---- the fit: one CTA per region -----------------------------------------------------------------------------
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }

// number of points with |x*a + y*b + z*c + d| < thr   (block-wide, returned to every thread)
__device__ __forceinline__ int ransac_count(const float3 *__restrict__ pts, int n, double a, double b, double c, double d,
                                            double thr, int *smem_counts) {
    int cnt = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float3 p = pts[i];
        const double r = fabs(dadd(dadd(dadd(dmul((double)p.x, a), dmul((double)p.y, b)), dmul((double)p.z, c)), d));
        cnt += (r < thr) ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) smem_counts[threadIdx.x >> 5] = cnt;
    __syncthreads();
    int tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) tot += smem_counts[w];
    return tot;
}

// Running state of one region's fit (the reference's loop-carried variables, main.cpp:1600-1710)
struct RansacState {
    double a, b, c, d, maximum;
    float depth_abs;
    int cursor;          // refinement phase: index (0..3999) of the next perturbation to try
};

constexpr int kRansacBatch = 1000;   // hypotheses evaluated per launch (the threshold only changes every 1000)
constexpr int kRefineTotal = 4 * kRefineRounds;

// plane of RANSAC hypothesis k (calcLinePara main.cpp:147-164 incl. its A coefficient as written, then the
// normalisation of main.cpp:1621-1626)
__device__ __forceinline__ void ransac_triple_plane(const RansacJob &job, int k, double &ta, double &tb, double &tc, double &td) {
    const uint32_t n = (uint32_t)job.n;
    const float3 P1 = job.pts[job.rnd[3 * k] % n], P2 = job.pts[job.rnd[3 * k + 1] % n], P3 = job.pts[job.rnd[3 * k + 2] % n];
    const double x1 = P1.x, y1 = P1.y, z1 = P1.z, x2 = P2.x, y2 = P2.y, z2 = P2.z, x3 = P3.x, y3 = P3.y, z3 = P3.z;
    ta = dadd(dmul(dadd(y3, -y1), dadd(z3, -z1)), -dmul(dadd(z2, -z1), dadd(y3, -y1)));
    tb = dadd(dmul(dadd(x3, -x1), dadd(z2, -z1)), -dmul(dadd(x2, -x1), dadd(z3, -z1)));
    tc = dadd(dmul(dadd(x2, -x1), dadd(y3, -y1)), -dmul(dadd(x3, -x1), dadd(y2, -y1)));
    td = -dadd(dadd(dmul(ta, x1), dmul(tb, y1)), dmul(tc, z1));
    const double sq = __dsqrt_rn(dadd(dadd(dmul(ta, ta), dmul(tb, tb)), dmul(tc, tc)));
    ta = __ddiv_rn(ta, sq); tb = __ddiv_rn(tb, sq); tc = __ddiv_rn(tc, sq); td = __ddiv_rn(td, sq);
}

// plane of refinement trial q (0..3999) around the current best (main.cpp:1668-1700): round q/4, scale j =
// 2000, 200, 20, 2 for q%4 = 0..3, four rand() values each
__device__ __forceinline__ void ransac_perturbed_plane(const RansacJob &job, const RansacState &st, int q, double &ra, double &rb,
                                                       double &rc, double &rd) {
    const uint32_t *rr = job.rnd + 3 * kRansacIters + 4 * q;
    const int m = q & 3;
    const int j = m == 0 ? 2000 : (m == 1 ? 200 : (m == 2 ? 20 : 2));
    const int med = j / 2;
    const double da = (double)((int)(rr[0] % (uint32_t)j) - med) / 10000.0, db = (double)((int)(rr[1] % (uint32_t)j) - med) / 10000.0;
    const double dc = (double)((int)(rr[2] % (uint32_t)j) - med) / 10000.0, dd = (double)((int)(rr[3] % (uint32_t)j) - med) / 1000.0;
    ra = dadd(st.a, da); rb = dadd(st.b, db); rc = dadd(st.c, dc); rd = dadd(st.d, dd);
    const double sq = __dsqrt_rn(dadd(dadd(dmul(ra, ra), dmul(rb, rb)), dmul(rc, rc)));
    ra = __ddiv_rn(ra, sq); rb = __ddiv_rn(rb, sq); rc = __ddiv_rn(rc, sq); rd = __ddiv_rn(rd, sq);
}

// ---- the whole fit of all regions in ONE persistent cooperative kernel ---------------------------------------------------
// The reference's loop carries only the best-so-far plane, its inlier count and the adaptive threshold (which changes after
// hypotheses 0, 1000, 2000, ...), so hypotheses are COUNTED in batches by the whole grid -- a CTA keeps 256 points of one
// region in registers (as doubles) and runs through the batch, whose plane parameters it computes into shared memory
// (60 flops per hypothesis versus 8 per point x hypothesis) -- and between two batches one CTA per region applies the
// reference's sequential rules.  The perturbation trials all depend on the current best: they are counted speculatively,
// kRefineSpec at a time, and the FIRST accepted one is committed, the cursor moves behind it.  Phases are separated by
// grid-wide barriers; the loop ends on the device when every region's cursor has passed its last trial, so the host
// launches once and reads the planes back once.
struct RansacFitArgs {
    RansacJob *jobs;          // n_jobs entries (n filled in on the device by ransac_points_kernel)
    RansacState *states;
    int *counts;              // n_jobs x kRansacBatch, zero on entry and on exit
    int n_jobs;
};
constexpr int kRefineSpec = 256;      // perturbation trials counted per speculative round
constexpr int kRansacSlice = 256;     // points per counting task = threads per CTA

struct RansacSmem {
    double pa[kRansacBatch], pb[kRansacBatch], pc[kRansacBatch], pd[kRansacBatch];
    int cnt[kRansacBatch];
    int warp_counts[32];
    RansacState st;
};

// counting phase: tasks = (region, slice of 256 points), strided over the grid
__device__ __forceinline__ void ransac_count_phase(const RansacFitArgs &a, RansacSmem &sm, int refine, int first, int count) {
    int planes_of = -1;   // region whose batch planes are in shared memory
    int base = 0;
    for (int t = 0; t < a.n_jobs; t++) {
        const RansacJob job = a.jobs[t];
        const int slices = (job.n + kRansacSlice - 1) / kRansacSlice;
        // first task index of this region that belongs to this CTA
        int task = (int)blockIdx.x - (base % (int)gridDim.x);
        if (task < 0) task += gridDim.x;
        base += slices;
        if (job.n <= 0) continue;
        const RansacState st = a.states[t];
        int f = first, c = count;
        if (refine) {
            f = st.cursor;
            c = min(count, kRefineTotal - f);
            if (c <= 0) continue;
        }
        for (int slice = task; slice < slices; slice += gridDim.x) {
            if (planes_of != t) {
                __syncthreads();
                for (int h = threadIdx.x; h < c; h += blockDim.x) {
                    double pa, pb, pc, pd;
                    if (refine) ransac_perturbed_plane(job, st, f + h, pa, pb, pc, pd);
                    else ransac_triple_plane(job, f + h, pa, pb, pc, pd);
                    sm.pa[h] = pa; sm.pb[h] = pb; sm.pc[h] = pc; sm.pd[h] = pd;
                }
                planes_of = t;
            }
            for (int h = threadIdx.x; h < c; h += blockDim.x) sm.cnt[h] = 0;
            __syncthreads();
            const int i = slice * kRansacSlice + threadIdx.x;
            const bool valid = i < job.n;
            const float3 p = job.pts[valid ? i : 0];
            const double x = p.x, y = p.y, z = p.z, thr = (double)st.depth_abs;
            const int lane = threadIdx.x & 31;
            for (int h = 0; h < c; h++) {
                const double r = fabs(dadd(dadd(dadd(dmul(x, sm.pa[h]), dmul(y, sm.pb[h])), dmul(z, sm.pc[h])), sm.pd[h]));
                const unsigned bal = __ballot_sync(0xffffffffu, valid && r < thr);
                if (lane == 0 && bal) atomicAdd(&sm.cnt[h], __popc(bal));
            }
            __syncthreads();
            int *out = a.counts + (size_t)t * kRansacBatch;
            for (int h = threadIdx.x; h < c; h += blockDim.x)
                if (sm.cnt[h]) atomicAdd(&out[h], sm.cnt[h]);
        }
    }
}

// sequential phase, one CTA per region: walks the batch's counts in hypothesis order with the reference's acceptance rule
// (>= replaces the best), applies the adaptive inlier threshold after hypotheses 0, 1000, 2000, ... (main.cpp:1645-1663),
// or -- refinement -- commits the FIRST accepted perturbation and moves the cursor behind it (later trials of the round were
// perturbations of the old best and are counted again from the new one).
__device__ __forceinline__ void ransac_select_phase(const RansacFitArgs &a, RansacSmem &sm, int refine, int first, int count) {
    for (int t = blockIdx.x; t < a.n_jobs; t += gridDim.x) {
        const RansacJob job = a.jobs[t];
        const int n = job.n;
        int *cnt = a.counts + (size_t)t * kRansacBatch;
        __syncthreads();
        if (n <= 0) {
            if (threadIdx.x == 0) a.states[t].cursor = kRefineTotal;
            continue;
        }
        if (threadIdx.x == 0) {
            RansacState st = a.states[t];
            if (!refine) {
                int best = -1;
                for (int h = 0; h < count; h++)
                    if ((double)cnt[h] >= st.maximum) { st.maximum = (double)cnt[h]; best = h; }
                if (best >= 0) ransac_triple_plane(job, first + best, st.a, st.b, st.c, st.d);
            } else {
                const int base = st.cursor, m = min(count, kRefineTotal - base);
                int hit = -1;
                for (int h = 0; h < m; h++)
                    if ((double)cnt[h] >= st.maximum) { hit = h; break; }
                if (hit >= 0) {
                    double pa, pb, pc, pd;
                    ransac_perturbed_plane(job, st, base + hit, pa, pb, pc, pd);
                    st.a = pa; st.b = pb; st.c = pc; st.d = pd; st.maximum = (double)cnt[hit];
                    st.cursor = base + hit + 1;
                } else {
                    st.cursor = base + max(m, 0);
                }
            }
            sm.st = st;
        }
        __syncthreads();
        // the adaptive threshold step follows hypothesis k whenever k % 1000 == 0; batches end exactly there
        if (!refine && ((first + count - 1) % 1000) == 0) {
            const double rat = sm.st.maximum / (double)n;
            if (rat < 0.3 && (double)sm.st.depth_abs < 0.003) {
                __syncthreads();
                if (threadIdx.x == 0) sm.st.depth_abs = (float)((double)sm.st.depth_abs + 0.0001);
            } else {
                const double m2 = (double)ransac_count(job.pts, n, sm.st.a, sm.st.b, sm.st.c, sm.st.d, dadd((double)sm.st.depth_abs, 0.0001), sm.warp_counts);
                __syncthreads();
                if (threadIdx.x == 0 && m2 > dadd(sm.st.maximum, dmul((double)n, 0.02))) {
                    sm.st.depth_abs = (float)((double)sm.st.depth_abs + 0.0001);
                    sm.st.maximum = m2;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            a.states[t] = sm.st;
            *job.out = make_float4((float)sm.st.a, (float)sm.st.b, (float)sm.st.c, (float)sm.st.d);
        }
        for (int h = threadIdx.x; h < kRansacBatch; h += blockDim.x) cnt[h] = 0;
    }
}

__global__ void __launch_bounds__(kRansacSlice) ransac_fit_kernel(const RansacFitArgs a) {
    __shared__ RansacSmem sm;
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < a.n_jobs; t += gridDim.x * blockDim.x) {
        RansacState s;
        s.a = 0; s.b = 0; s.c = 1; s.d = -1; s.maximum = 0;
        s.depth_abs = (float)(0.0003 * (double)sqrtf(a.jobs[t].size / 20.0f));  // main.cpp:1552-1553
        s.cursor = a.jobs[t].n > 0 ? 0 : kRefineTotal;
        a.states[t] = s;
    }
    grid.sync();
    // RANSAC hypotheses: the inlier threshold is constant between hypotheses 1000 j + 1 and 1000 (j + 1)
    for (int first = 0; first < kRansacIters;) {
        const int count = first == 0 ? 1 : min(kRansacBatch, kRansacIters - first);
        ransac_count_phase(a, sm, 0, first, count);
        grid.sync();
        ransac_select_phase(a, sm, 0, first, count);
        grid.sync();
        first += count;
    }
    // local refinement, until every region has tried its 4000 perturbations
    for (;;) {
        bool done = true;
        for (int t = 0; t < a.n_jobs; t++) done = done && (a.states[t].cursor >= kRefineTotal);
        if (done) break;
        ransac_count_phase(a, sm, 1, 0, kRefineSpec);
        grid.sync();
        ransac_select_phase(a, sm, 1, 0, kRefineSpec);
        grid.sync();
    }
}

}  // namespace tsar
