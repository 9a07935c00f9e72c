// cloud_eval.cu -- nearest-neighbour cloud-to-cloud evaluation: accuracy, completeness and F-score of a reconstruction
// against a ground-truth cloud (DESIGN.md section 4.7).
//
// Per cloud, one index that also serves as the query order:
//   1. eval_bbox_kernel      bounding box and count of the finite points (ordered-int atomics);
//   2. eval_key_kernel       63-bit Morton key on that box (21 bits per axis); a non-finite point gets bit 63, so the sort
//                            puts the n_finite finite points first and the non-finite ones after them;
//   3. radix sort (key, input index), then eval_gather_kernel writes the points in key order as float4;
//   4. eval_leaf_kernel      leaves of <= 32 consecutive finite points, AABB each; eval_merge_kernel, one launch per level,
//                            builds the implicit balanced tree: node j of level l has children 2j and 2j + 1 of level l - 1.
// The keys only buy locality: every box comes from the real coordinates of the points below it, so which points share a
// leaf changes the work, never the result.
// Query (eval_query_kernel): one thread per query point, in the key order of the query cloud so that a warp's lanes walk
// similar paths; a stack traversal, nearest child first, prunes a box whose lower bound is strictly greater than
// min(best d^2, cut2); the distance is scattered back to input order and the per-threshold counts are reduced on the
// device.  d^2 and the box bound use the same explicit-rounding operation sequence as the rule, so the result is the
// brute-force minimum bit for bit (oracle/eval_cpu.c, oc_eval).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include <memory>
#include <string>

#include "../../include/tsar_b200.h"
#include "dev_mem.h"
#include "pm_math.cuh"

using namespace tsar;

namespace {

constexpr int kThreads = 256;
constexpr int kQueryThreads = 128;
constexpr int kLeafSize = 32;
constexpr int kLevelShift = 26;                        // stack entry = level << 26 | node index
constexpr int kMaxLevels = 28;                         // 2^31 points -> 2^26 leaves -> 27 levels
constexpr int kStack = 32;                             // a traversal holds at most one entry per level plus one
constexpr long long kMaxPoints = (1LL << 31) - 1;      // sort indices are int
constexpr unsigned long long kNonFinite = 1ULL << 63;

struct TreeArgs {
    const float4 *pts;        // finite points of the index cloud, key order
    const float4 *lo, *hi;    // node boxes, level after level (level 0 = leaves)
    long long n_finite;
    int n_levels;
    long long off[kMaxLevels];
    int len[kMaxLevels];
};

struct QueryArgs {
    const float4 *q;          // every point of the query cloud in key order (non-finite ones last)
    const int *q_idx;         // their input indices
    long long n;
    float cut2, tau_max;
    int k;
    float tau[TSAR_EVAL_MAX_THRESHOLDS];
};

__device__ __forceinline__ bool finite3(float x, float y, float z) {
    return fabsf(x) <= 3.402823466e38f && fabsf(y) <= 3.402823466e38f && fabsf(z) <= 3.402823466e38f;
}

// Order-preserving map of a non-NaN float to an unsigned int, so that atomicMin / atomicMax on it order the floats.
__device__ __forceinline__ unsigned f2o(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float o2f(unsigned o) {
    const unsigned u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, sizeof f);
    return f;
#endif
}

// misc[0..2] = f2o(min x, y, z), misc[3..5] = f2o(max x, y, z) of the finite points; *n_finite counts them.
__global__ void __launch_bounds__(kThreads) eval_bbox_kernel(const float *__restrict__ xyz, long long n,
                                                             unsigned *__restrict__ box, unsigned long long *__restrict__ n_finite) {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    unsigned count = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        if (!finite3(x, y, z)) continue;
        ++count;
        lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
        hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
    for (int o = 16; o > 0; o >>= 1) {
        count += __shfl_xor_sync(0xffffffffu, count, o);
        for (int a = 0; a < 3; ++a) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    if ((threadIdx.x & 31) == 0 && count) {
        atomicAdd(n_finite, (unsigned long long)count);
        for (int a = 0; a < 3; ++a) {
            atomicMin(&box[a], f2o(lo[a]));
            atomicMax(&box[3 + a], f2o(hi[a]));
        }
    }
}

__device__ __forceinline__ unsigned long long spread3(unsigned v) {   // 21 bits -> every third bit of 63
    unsigned long long x = v & 0x1fffffULL;
    x = (x | x << 32) & 0x1f00000000ffffULL;
    x = (x | x << 16) & 0x1f0000ff0000ffULL;
    x = (x | x << 8) & 0x100f00f00f00f00fULL;
    x = (x | x << 4) & 0x10c30c30c30c30c3ULL;
    x = (x | x << 2) & 0x1249249249249249ULL;
    return x;
}

__device__ __forceinline__ unsigned quantise(float v, float lo, float scale) {
    const float c = fmaxf(fminf((v - lo) * scale, 2097151.0f), 0.0f);   // NaN (inf * 0) -> 0; only locality depends on it
    return (unsigned)c;
}

__global__ void __launch_bounds__(kThreads) eval_key_kernel(const float *__restrict__ xyz, long long n,
                                                            const unsigned *__restrict__ box,
                                                            unsigned long long *__restrict__ key, int *__restrict__ idx) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
    unsigned long long k = kNonFinite;
    if (finite3(x, y, z)) {
        float lo[3], scale[3];
        for (int a = 0; a < 3; ++a) {
            lo[a] = o2f(box[a]);
            const float ext = o2f(box[3 + a]) - lo[a];
            scale[a] = ext > 0.0f && ext <= 3.402823466e38f ? 2097152.0f / ext : 0.0f;
        }
        k = spread3(quantise(x, lo[0], scale[0])) | spread3(quantise(y, lo[1], scale[1])) << 1 |
            spread3(quantise(z, lo[2], scale[2])) << 2;
    }
    key[i] = k;
    idx[i] = (int)i;
}

__global__ void __launch_bounds__(kThreads) eval_gather_kernel(const float *__restrict__ xyz, long long n,
                                                               const int *__restrict__ idx, float4 *__restrict__ pts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long j = idx[i];
    pts[i] = make_float4(xyz[3 * j], xyz[3 * j + 1], xyz[3 * j + 2], 0.0f);
}

__global__ void __launch_bounds__(kThreads) eval_leaf_kernel(const float4 *__restrict__ pts, long long n_finite, int n_leaves,
                                                             float4 *__restrict__ lo, float4 *__restrict__ hi) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_leaves) return;
    const long long b = (long long)j * kLeafSize, e = min(b + kLeafSize, n_finite);
    float4 l = pts[b], h = l;
    for (long long i = b + 1; i < e; ++i) {
        const float4 p = pts[i];
        l.x = fminf(l.x, p.x); l.y = fminf(l.y, p.y); l.z = fminf(l.z, p.z);
        h.x = fmaxf(h.x, p.x); h.y = fmaxf(h.y, p.y); h.z = fmaxf(h.z, p.z);
    }
    lo[j] = l;
    hi[j] = h;
}

__global__ void __launch_bounds__(kThreads) eval_merge_kernel(const float4 *__restrict__ c_lo, const float4 *__restrict__ c_hi,
                                                              int n_children, int n_nodes, float4 *__restrict__ lo,
                                                              float4 *__restrict__ hi) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_nodes) return;
    float4 l = c_lo[2 * j], h = c_hi[2 * j];
    if (2 * j + 1 < n_children) {
        const float4 l1 = c_lo[2 * j + 1], h1 = c_hi[2 * j + 1];
        l.x = fminf(l.x, l1.x); l.y = fminf(l.y, l1.y); l.z = fminf(l.z, l1.z);
        h.x = fmaxf(h.x, h1.x); h.y = fmaxf(h.y, h1.y); h.z = fmaxf(h.z, h1.z);
    }
    lo[j] = l;
    hi[j] = h;
}

// d^2(q, p) of the rule: d = p - q, (dx dx + dy dy) + dz dz, one rounding per operation.
__device__ __forceinline__ float dist2(float4 p, float qx, float qy, float qz) {
    const float dx = fsub(p.x, qx), dy = fsub(p.y, qy), dz = fsub(p.z, qz);
    return fadd(fadd(fmul(dx, dx), fmul(dy, dy)), fmul(dz, dz));
}

// Lower bound of d^2(q, p) over the points p of a box [lo, hi], with the per-axis gap g = max(lo - q, 0, q - hi).
// Why it never exceeds the d^2 of a point p inside the box (so pruning on it is exact): on each axis lo <= p <= hi, and
// round-to-nearest is monotone, so fl(lo - q) <= fl(p - q) and fl(q - hi) <= fl(q - p) = -fl(p - q); hence
// 0 <= g <= |fl(p - q)| = |dx|.  Then fl(g g) <= fl(dx dx) (monotone again, both operands non-negative), and the two
// additions, done in the same order as in dist2, keep the inequality: bound <= d^2, with no exception for overflow
// (inf compares as the largest value).
__device__ __forceinline__ float box_bound(float4 lo, float4 hi, float qx, float qy, float qz) {
    const float gx = fmaxf(fmaxf(fsub(lo.x, qx), 0.0f), fsub(qx, hi.x));
    const float gy = fmaxf(fmaxf(fsub(lo.y, qy), 0.0f), fsub(qy, hi.y));
    const float gz = fmaxf(fmaxf(fsub(lo.z, qz), 0.0f), fsub(qz, hi.z));
    return fadd(fadd(fmul(gx, gx), fmul(gy, gy)), fmul(gz, gz));
}

__global__ void __launch_bounds__(kQueryThreads) eval_query_kernel(TreeArgs t, QueryArgs a, float *__restrict__ dist,
                                                                   unsigned long long *__restrict__ within,
                                                                   unsigned long long *__restrict__ visits_total,
                                                                   unsigned *__restrict__ visits_max) {
    __shared__ int s_node[kStack][kQueryThreads];
    __shared__ float s_bound[kStack][kQueryThreads];
    __shared__ unsigned s_within[TSAR_EVAL_MAX_THRESHOLDS];
    const int tid = threadIdx.x;
    for (int i = tid; i < a.k; i += blockDim.x) s_within[i] = 0;
    __syncthreads();
    const long long qi = (long long)blockIdx.x * blockDim.x + tid;
    float d = INFINITY;
    unsigned visits = 0;
    const bool active = qi < a.n;
    if (active) {
        const float4 q = a.q[qi];
        if (finite3(q.x, q.y, q.z) && t.n_finite > 0) {
            float best2 = INFINITY;
            int sp = 0;
            const int root = (t.n_levels - 1) << kLevelShift;
            s_node[0][tid] = root;
            s_bound[0][tid] = box_bound(t.lo[t.off[t.n_levels - 1]], t.hi[t.off[t.n_levels - 1]], q.x, q.y, q.z);
            sp = 1;
            while (sp > 0) {
                --sp;
                const int node = s_node[sp][tid];
                if (s_bound[sp][tid] > fminf(best2, a.cut2)) continue;
                const int level = node >> kLevelShift, j = node & ((1 << kLevelShift) - 1);
                if (level == 0) {
                    ++visits;
                    const long long b = (long long)j * kLeafSize, e = min(b + kLeafSize, t.n_finite);
                    for (long long i = b; i < e; ++i) {
                        const float d2 = dist2(t.pts[i], q.x, q.y, q.z);
                        best2 = d2 < best2 ? d2 : best2;
                    }
                    continue;
                }
                const long long base = t.off[level - 1];
                const int c0 = 2 * j, c1 = 2 * j + 1;
                const float b0 = box_bound(t.lo[base + c0], t.hi[base + c0], q.x, q.y, q.z);
                const float b1 = c1 < t.len[level - 1] ? box_bound(t.lo[base + c1], t.hi[base + c1], q.x, q.y, q.z) : INFINITY;
                const bool first0 = b0 <= b1;
                const int near = ((level - 1) << kLevelShift) | (first0 ? c0 : c1);
                const int far = ((level - 1) << kLevelShift) | (first0 ? c1 : c0);
                const float bn = first0 ? b0 : b1, bf = first0 ? b1 : b0;
                const float lim = fminf(best2, a.cut2);
                if (bf <= lim) {                       // the farther child waits below the nearer one
                    s_node[sp][tid] = far;
                    s_bound[sp][tid] = bf;
                    ++sp;
                }
                if (bn <= lim) {
                    s_node[sp][tid] = near;
                    s_bound[sp][tid] = bn;
                    ++sp;
                }
            }
            const float s = __fsqrt_rn(best2);
            d = s <= a.tau_max ? s : INFINITY;
        }
        dist[a.q_idx[qi]] = d;
    }
    const int lane = tid & 31;
    for (int i = 0; i < a.k; ++i) {
        const unsigned b = __ballot_sync(0xffffffffu, active && d <= a.tau[i]);
        if (lane == 0 && b) atomicAdd(&s_within[i], (unsigned)__popc(b));
    }
    unsigned vs = visits, vm = visits;
    for (int o = 16; o > 0; o >>= 1) {
        vs += __shfl_xor_sync(0xffffffffu, vs, o);
        vm = max(vm, __shfl_xor_sync(0xffffffffu, vm, o));
    }
    if (lane == 0 && vs) {
        atomicAdd(visits_total, (unsigned long long)vs);
        atomicMax(visits_max, vm);
    }
    __syncthreads();
    for (int i = tid; i < a.k; i += blockDim.x)
        if (s_within[i]) atomicAdd(&within[i], (unsigned long long)s_within[i]);
}

// Device buffers of one cloud; they only grow.
struct CloudBuf {
    DeviceBuf<float> xyz;
    DeviceBuf<unsigned long long> key[2];
    DeviceBuf<int> idx[2];
    DeviceBuf<float4> pts, lo, hi;
    DeviceBuf<float> dist;
    // of the current run
    long long n = 0, n_finite = 0;
    int n_levels = 0;
    long long off[kMaxLevels] = {};
    int len[kMaxLevels] = {};
};

// Device counters of one run: per cloud the box (6) and n_finite; per direction the counts and the visit counters.
struct Misc {
    unsigned box[2][6];
    unsigned long long n_finite[2];
    unsigned long long within[2][TSAR_EVAL_MAX_THRESHOLDS];
    unsigned long long visits_total[2];
    unsigned visits_max[2];
};

}  // namespace

struct tsar_eval : HandleCore {
    CloudBuf c[2];                  // 0 = reconstruction, 1 = ground truth
    DeviceBuf<unsigned char> sort_tmp;
    DeviceBuf<Misc> d_misc;
    PinnedBuf<Misc> h_misc;
    long long visits_total[2] = {0, 0};
    int visits_max[2] = {0, 0};
};

static unsigned blocks(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// Capacity for n points: 12 (input) + 2 x 8 (keys) + 2 x 4 (indices) + 16 (sorted points) + 4 (distances) = 56 B each.
static int cloud_reserve(tsar_eval *e, CloudBuf &c, long long n) {
    const size_t N = (size_t)n;
    TSAR_CK(e, c.xyz.reserve(3 * N));
    TSAR_CK(e, c.key[0].reserve(N));
    TSAR_CK(e, c.key[1].reserve(N));
    TSAR_CK(e, c.idx[0].reserve(N));
    TSAR_CK(e, c.idx[1].reserve(N));
    TSAR_CK(e, c.pts.reserve(N));
    TSAR_CK(e, c.dist.reserve(N));
    return TSAR_OK;
}

// Tree shape over n_finite points: level 0 = ceil(n_finite / 32) leaves, each level above halves (rounding up) to 1.
static void tree_shape(CloudBuf &c) {
    c.n_levels = 0;
    if (c.n_finite == 0) return;
    long long len = (c.n_finite + kLeafSize - 1) / kLeafSize, off = 0;
    for (;;) {
        c.off[c.n_levels] = off;
        c.len[c.n_levels] = (int)len;
        ++c.n_levels;
        off += len;
        if (len == 1) break;
        len = (len + 1) / 2;
    }
}

static long long tree_nodes(const CloudBuf &c) { return c.n_levels ? c.off[c.n_levels - 1] + 1 : 0; }

// The largest float c2 whose correctly rounded square root is <= tau_max.  A point with d^2 > c2 is farther than tau_max,
// so boxes whose bound exceeds c2 are pruned exactly.  fl(tau_max^2) alone is not enough: a d^2 just above it can still
// have sqrt_rn(d^2) == tau_max.
static float cut_square(float tau_max) {
    float c2 = tau_max * tau_max;
    while (c2 > 0.0f && !(sqrtf(c2) <= tau_max)) c2 = nextafterf(c2, 0.0f);
    for (;;) {
        const float up = nextafterf(c2, INFINITY);
        if (!(sqrtf(up) <= tau_max)) break;
        c2 = up;
    }
    return c2;
}

extern "C" {

int tsar_eval_create(int device, void *stream, tsar_eval **out) {
    if (!out) return TSAR_ERR_ARG;
    *out = nullptr;
    std::unique_ptr<tsar_eval> e(new tsar_eval);
    if (int rc = e->open(device, stream)) return rc;
    TSAR_CK(e, e->d_misc.reserve(1));
    TSAR_CK(e, e->h_misc.reserve(1));
    *out = e.release();
    return TSAR_OK;
}

int tsar_eval_destroy(tsar_eval *e) {
    if (!e) return TSAR_OK;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    delete e;
    return TSAR_OK;
}

const char *tsar_eval_last_error(const tsar_eval *e) { return e ? e->err.c_str() : "null eval handle"; }

int tsar_eval_run(tsar_eval *e, const float *recon, long long n_recon, const float *gt, long long n_gt,
                  const float *thresholds, int n_thresholds, float tau_max, long long *within_recon,
                  long long *within_gt, float *dist_recon, float *dist_gt) {
    if (!e) return TSAR_ERR_ARG;
    if (n_recon < 0 || n_gt < 0 || n_recon > kMaxPoints || n_gt > kMaxPoints)
        TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: point counts must lie in 0 .. 2^31 - 1");
    if ((n_recon && !recon) || (n_gt && !gt)) TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: null cloud");
    if (n_thresholds < 1 || n_thresholds > TSAR_EVAL_MAX_THRESHOLDS)
        TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: 1..64 thresholds");
    if (!thresholds || !within_recon || !within_gt) TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: null thresholds or counts");
    if (!(tau_max > 0.0f) || !(tau_max <= 3.402823466e38f))
        TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: tau_max must be finite and > 0");
    QueryArgs qa{};
    qa.k = n_thresholds;
    qa.tau_max = tau_max;
    qa.cut2 = cut_square(tau_max);
    for (int i = 0; i < n_thresholds; ++i) {
        const float t = thresholds[i];
        if (!(t > 0.0f) || !(t <= 3.402823466e38f)) TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: thresholds must be finite and > 0");
        if (t > tau_max) TSAR_FAIL(e, TSAR_ERR_ARG, "tsar_eval_run: a threshold exceeds tau_max");
        qa.tau[i] = t;
    }
    TSAR_CK(e, cudaSetDevice(e->device));
    const float *host[2] = {recon, gt};
    const long long n[2] = {n_recon, n_gt};
    size_t tmp_need = 0;
    for (int c = 0; c < 2; ++c) {
        int rc = cloud_reserve(e, e->c[c], n[c]);
        if (rc != TSAR_OK) return rc;
        size_t bytes = 0;
        if (n[c]) {
            TSAR_CK(e, cub::DeviceRadixSort::SortPairs(nullptr, bytes, e->c[c].key[0].get(), e->c[c].key[1].get(), e->c[c].idx[0].get(),
                                                e->c[c].idx[1].get(), (int)n[c], 0, 64, e->stream));
        }
        tmp_need = std::max(tmp_need, bytes);
    }
    TSAR_CK(e, e->sort_tmp.reserve(tmp_need));
    Misc init{};
    for (int c = 0; c < 2; ++c)
        for (int a = 0; a < 3; ++a) {
            init.box[c][a] = 0xffffffffu;
            init.box[c][3 + a] = 0u;
        }
    *e->h_misc.get() = init;
    TSAR_CK(e, cudaMemcpyAsync(e->d_misc.get(), e->h_misc.get(), sizeof(Misc), cudaMemcpyHostToDevice, e->stream));
    for (int c = 0; c < 2; ++c) {
        CloudBuf &b = e->c[c];
        b.n = n[c];
        if (!n[c]) continue;
        TSAR_CK(e, cudaMemcpyAsync(b.xyz.get(), host[c], 3 * (size_t)n[c] * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        eval_bbox_kernel<<<std::min(blocks(n[c], kThreads), 148u * 8u), kThreads, 0, e->stream>>>(
            b.xyz.get(), n[c], e->d_misc.get()->box[c], &e->d_misc.get()->n_finite[c]);
        eval_key_kernel<<<blocks(n[c], kThreads), kThreads, 0, e->stream>>>(b.xyz.get(), n[c], e->d_misc.get()->box[c], b.key[0].get(), b.idx[0].get());
        TSAR_CK(e, cudaGetLastError());
        size_t bytes = e->sort_tmp.capacity();
        TSAR_CK(e, cub::DeviceRadixSort::SortPairs(e->sort_tmp.get(), bytes, b.key[0].get(), b.key[1].get(), b.idx[0].get(), b.idx[1].get(), (int)n[c], 0, 64,
                                            e->stream));
        eval_gather_kernel<<<blocks(n[c], kThreads), kThreads, 0, e->stream>>>(b.xyz.get(), n[c], b.idx[1].get(), b.pts.get());
        TSAR_CK(e, cudaGetLastError());
    }
    TSAR_CK(e, cudaMemcpyAsync(e->h_misc.get(), e->d_misc.get(), sizeof(Misc), cudaMemcpyDeviceToHost, e->stream));
    TSAR_CK(e, cudaStreamSynchronize(e->stream));
    for (int c = 0; c < 2; ++c) {
        CloudBuf &b = e->c[c];
        b.n_finite = (long long)e->h_misc.get()->n_finite[c];
        tree_shape(b);
        const long long nodes = tree_nodes(b);
        TSAR_CK(e, b.lo.reserve((size_t)nodes));
        TSAR_CK(e, b.hi.reserve((size_t)nodes));
        if (!b.n_levels) continue;
        eval_leaf_kernel<<<blocks(b.len[0], kThreads), kThreads, 0, e->stream>>>(b.pts.get(), b.n_finite, b.len[0], b.lo.get(), b.hi.get());
        for (int l = 1; l < b.n_levels; ++l)
            eval_merge_kernel<<<blocks(b.len[l], kThreads), kThreads, 0, e->stream>>>(
                b.lo.get() + b.off[l - 1], b.hi.get() + b.off[l - 1], b.len[l - 1], b.len[l], b.lo.get() + b.off[l], b.hi.get() + b.off[l]);
        TSAR_CK(e, cudaGetLastError());
    }
    // direction 0: reconstruction points against the ground-truth index; direction 1: the reverse
    for (int dir = 0; dir < 2; ++dir) {
        const CloudBuf &q = e->c[dir], &ix = e->c[1 - dir];
        if (!q.n) continue;
        TreeArgs ta{};
        ta.pts = ix.pts.get();
        ta.lo = ix.lo.get();
        ta.hi = ix.hi.get();
        ta.n_finite = ix.n_finite;
        ta.n_levels = ix.n_levels;
        for (int l = 0; l < ix.n_levels; ++l) {
            ta.off[l] = ix.off[l];
            ta.len[l] = ix.len[l];
        }
        qa.q = q.pts.get();
        qa.q_idx = q.idx[1].get();
        qa.n = q.n;
        eval_query_kernel<<<blocks(q.n, kQueryThreads), kQueryThreads, 0, e->stream>>>(
            ta, qa, q.dist.get(), e->d_misc.get()->within[dir], &e->d_misc.get()->visits_total[dir], &e->d_misc.get()->visits_max[dir]);
        TSAR_CK(e, cudaGetLastError());
    }
    TSAR_CK(e, cudaMemcpyAsync(e->h_misc.get(), e->d_misc.get(), sizeof(Misc), cudaMemcpyDeviceToHost, e->stream));
    float *dist_out[2] = {dist_recon, dist_gt};
    for (int c = 0; c < 2; ++c)
        if (dist_out[c] && n[c])
            TSAR_CK(e, cudaMemcpyAsync(dist_out[c], e->c[c].dist.get(), (size_t)n[c] * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    TSAR_CK(e, cudaStreamSynchronize(e->stream));
    for (int i = 0; i < n_thresholds; ++i) {
        within_recon[i] = (long long)e->h_misc.get()->within[0][i];
        within_gt[i] = (long long)e->h_misc.get()->within[1][i];
    }
    for (int d = 0; d < 2; ++d) {
        e->visits_total[d] = (long long)e->h_misc.get()->visits_total[d];
        e->visits_max[d] = (int)e->h_misc.get()->visits_max[d];
    }
    return TSAR_OK;
}

int tsar_eval_dbg_visits(const tsar_eval *e, long long *total, int *max_per_query) {
    if (!e) return TSAR_ERR_ARG;
    for (int d = 0; d < 2; ++d) {
        if (total) total[d] = e->visits_total[d];
        if (max_per_query) max_per_query[d] = e->visits_max[d];
    }
    return TSAR_OK;
}

}  // extern "C"
