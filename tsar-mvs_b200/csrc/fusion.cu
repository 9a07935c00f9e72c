// fusion.cu -- multi-view depth-map fusion into one coloured point cloud (DESIGN.md section 4.6).
//
// Views are fused in order: view v reads the source-pixel masks that views < v set.  Inside one view every stage is
// parallel and the result is bit-identical to the raster-order loop of the rule (oracle/fusion_cpu.c, oc_fuse):
//   1. fusion_candidates_kernel  one thread per pixel: back-project, project into every neighbour, gather the
//                                neighbour's depth + normal (one float4), run the three checks against the masks as they
//                                stand at the start of the view; store q or -1 per (neighbour j, pixel p).
//   2. resolution rounds         owner(j, q) = the smallest non-dropped pixel holding (j, q) (atomicMin); a pixel whose
//                                candidates are all owned by itself or by a FUSED pixel is decided: FUSED when it owns at
//                                least min_consistent of them, else DROPPED.  The smallest undecided pixel is always
//                                decidable, so the loop ends; decisions read the state of the previous round only.
//   3. emit                      FUSED pixels set the masks of the sources they own, compute their point and are
//                                compacted in raster order (block counts, one-block scan, ballot prefix in the block).
// Every rounding step is spelled with an explicit-rounding intrinsic so that the C restatement, compiled with
// -ffp-contract=off, performs the same operations in the same order.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <string>
#include <vector>

#include "../../include/tsar_b200.h"
#include "dev_mem.h"
#include "pm_math.cuh"
#include "view_project.cuh"

using namespace tsar;

namespace {

struct FusionCam {
    float K[9], Kinv[9], R[9], t[3];
};
constexpr int kCamFloats = 30;

enum : unsigned char { kUndecided = 0, kFused = 1, kDropped = 2 };
constexpr int kThreads = 256;

struct ViewArgs {
    int v, n_src, W, H, min_consistent;
    float max_reproj, max_rel, cos_normal;
    int src[TSAR_FUSION_MAX_NEIGHBOURS];
};

// X = R^T (d * Kinv (x, y, 1) - t)
__device__ __forceinline__ float3 backproject(const FusionCam &c, float x, float y, float d) {
    const float rx = fadd(fadd(fmul(c.Kinv[0], x), fmul(c.Kinv[1], y)), c.Kinv[2]);
    const float ry = fadd(fadd(fmul(c.Kinv[3], x), fmul(c.Kinv[4], y)), c.Kinv[5]);
    const float rz = fadd(fadd(fmul(c.Kinv[6], x), fmul(c.Kinv[7], y)), c.Kinv[8]);
    const float cx = fsub(fmul(d, rx), c.t[0]);
    const float cy = fsub(fmul(d, ry), c.t[1]);
    const float cz = fsub(fmul(d, rz), c.t[2]);
    return make_float3(dot3s(c.R[0], cx, c.R[3], cy, c.R[6], cz), dot3s(c.R[1], cx, c.R[4], cy, c.R[7], cz),
                       dot3s(c.R[2], cx, c.R[5], cy, c.R[8], cz));
}

__device__ __forceinline__ float norm3(float x, float y, float z) { return __fsqrt_rn(dot3s(x, x, y, y, z, z)); }

// Cameras of the view (slot 0) and of its neighbours (slots 1..n_src) into shared memory.
__device__ __forceinline__ void load_cams(FusionCam *sc, const ViewArgs &a, const FusionCam *__restrict__ cams) {
    for (int i = threadIdx.x; i < (a.n_src + 1) * kCamFloats; i += blockDim.x) {
        const int k = i / kCamFloats, f = i - k * kCamFloats;
        const int view = k == 0 ? a.v : a.src[k - 1];
        reinterpret_cast<float *>(&sc[k])[f] = reinterpret_cast<const float *>(&cams[view])[f];
    }
    __syncthreads();
}

__global__ void fusion_pack_kernel(const float *__restrict__ depth, const float *__restrict__ normals,
                                   const unsigned char *__restrict__ bgr, size_t P, float4 *__restrict__ dn,
                                   uchar4 *__restrict__ col) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    dn[p] = make_float4(normals[3 * p], normals[3 * p + 1], normals[3 * p + 2], depth[p]);
    col[p] = make_uchar4(bgr[3 * p], bgr[3 * p + 1], bgr[3 * p + 2], 0);
}

__global__ void __launch_bounds__(kThreads) fusion_candidates_kernel(ViewArgs a, const FusionCam *__restrict__ cams,
                                                                     const float4 *__restrict__ dn,
                                                                     const unsigned char *__restrict__ mask,
                                                                     int *__restrict__ cand, unsigned char *__restrict__ state) {
    __shared__ FusionCam sc[TSAR_FUSION_MAX_NEIGHBOURS + 1];
    load_cams(sc, a, cams);
    const int P = a.W * a.H;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const size_t vo = (size_t)a.v * P;
    unsigned char st = kDropped;
    const float4 g0 = dn[vo + p];
    if (!mask[vo + p] && valid_depth(g0.w)) {
        const float x = (float)(p % a.W), y = (float)(p / a.W), d = g0.w;
        const float3 X = backproject(sc[0], x, y, d);
        const float thr_v = fmul(a.cos_normal, norm3(g0.x, g0.y, g0.z));
        const float max_dz = fmul(a.max_rel, d);
        int count = 0;
        for (int j = 0; j < a.n_src; ++j) {
            const FusionCam &cu = sc[1 + j];
            int q = -1;
            float px, py, z;
            project(cu, X, px, py, z);
            const float qx = floorf(fadd(px, 0.5f)), qy = floorf(fadd(py, 0.5f));
            if (z > 0.0f && qx >= 0.0f && qx < (float)a.W && qy >= 0.0f && qy < (float)a.H) {
                const int qi = (int)qy * a.W + (int)qx;
                const size_t uo = (size_t)a.src[j] * P;
                if (!mask[uo + qi]) {
                    const float4 g = dn[uo + qi];
                    if (valid_depth(g.w)) {
                        const float3 Y = backproject(cu, qx, qy, g.w);
                        float rx, ry, rz;
                        project(sc[0], Y, rx, ry, rz);
                        const float dx = fsub(rx, x), dy = fsub(ry, y);
                        const bool ok = __fsqrt_rn(fadd(fmul(dx, dx), fmul(dy, dy))) < a.max_reproj &&
                                        fabsf(fsub(rz, d)) < max_dz &&
                                        dot3s(g0.x, g.x, g0.y, g.y, g0.z, g.z) >= fmul(thr_v, norm3(g.x, g.y, g.z));
                        if (ok) q = qi;
                    }
                }
            }
            cand[(size_t)j * P + p] = q;
            count += q >= 0;
        }
        if (count >= a.min_consistent) st = kUndecided;
    }
    state[p] = st;
}

__global__ void __launch_bounds__(kThreads) fusion_claim_kernel(int n_src, int P, const int *__restrict__ cand,
                                                                const unsigned char *__restrict__ state, int *__restrict__ owner) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P || state[p] == kDropped) return;
    for (int j = 0; j < n_src; ++j) {
        const int q = cand[(size_t)j * P + p];
        if (q >= 0) atomicMin(&owner[(size_t)j * P + q], p);
    }
}

__global__ void __launch_bounds__(kThreads) fusion_decide_kernel(int n_src, int P, int min_consistent,
                                                                 const int *__restrict__ cand, const int *__restrict__ owner,
                                                                 const unsigned char *__restrict__ cur,
                                                                 unsigned char *__restrict__ nxt, int *__restrict__ undecided) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const unsigned char s = cur[p];
    if (s != kUndecided) {
        nxt[p] = s;
        return;
    }
    int own = 0;
    for (int j = 0; j < n_src; ++j) {
        const int q = cand[(size_t)j * P + p];
        if (q < 0) continue;
        const int o = owner[(size_t)j * P + q];
        if (o == p) {
            ++own;
        } else if (cur[o] != kFused) {  // o < p is still undecided: wait for it
            nxt[p] = kUndecided;
            atomicAdd(undecided, 1);
            return;
        }
    }
    nxt[p] = own >= min_consistent ? kFused : kDropped;
}

__global__ void __launch_bounds__(kThreads) fusion_count_kernel(int P, const unsigned char *__restrict__ state,
                                                                int *__restrict__ block_count) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = __syncthreads_count(p < P && state[p] == kFused);
    if (threadIdx.x == 0) block_count[blockIdx.x] = n;
}

// Exclusive scan of the block counts in one CTA of 1024 threads; total = number of points of the view.
__global__ void __launch_bounds__(1024) fusion_scan_kernel(const int *__restrict__ block_count, int nb,
                                                           int *__restrict__ block_off, int *__restrict__ total) {
    __shared__ int s[1024];
    int carry = 0;
    for (int base = 0; base < nb; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < nb ? block_count[i] : 0;
        s[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            const int t = threadIdx.x >= o ? s[threadIdx.x - o] : 0;
            __syncthreads();
            s[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nb) block_off[i] = carry + s[threadIdx.x] - v;
        carry += s[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(kThreads) fusion_emit_kernel(ViewArgs a, const FusionCam *__restrict__ cams,
                                                               const float4 *__restrict__ dn, const uchar4 *__restrict__ col,
                                                               unsigned char *__restrict__ mask, const int *__restrict__ cand,
                                                               const int *__restrict__ owner,
                                                               const unsigned char *__restrict__ state,
                                                               const int *__restrict__ block_off, float *__restrict__ out_xyz,
                                                               float *__restrict__ out_nrm, unsigned char *__restrict__ out_rgb) {
    __shared__ FusionCam sc[TSAR_FUSION_MAX_NEIGHBOURS + 1];
    __shared__ int warp_total[kThreads / 32];
    load_cams(sc, a, cams);
    const int P = a.W * a.H;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool fused = p < P && state[p] == kFused;
    const unsigned ballot = __ballot_sync(0xffffffffu, fused);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_total[warp] = __popc(ballot);
    __syncthreads();
    if (!fused) return;
    int idx = block_off[blockIdx.x] + __popc(ballot & ((1u << lane) - 1u));
    for (int w = 0; w < warp; ++w) idx += warp_total[w];

    const size_t vo = (size_t)a.v * P;
    const float4 g0 = dn[vo + p];
    const float3 X = backproject(sc[0], (float)(p % a.W), (float)(p / a.W), g0.w);
    float sx = X.x, sy = X.y, sz = X.z, nx = g0.x, ny = g0.y, nz = g0.z;
    const uchar4 c0 = col[vo + p];
    int cb = c0.x, cg = c0.y, cr = c0.z, k = 1;
    for (int j = 0; j < a.n_src; ++j) {
        const int q = cand[(size_t)j * P + p];
        if (q < 0 || owner[(size_t)j * P + q] != p) continue;
        const size_t uo = (size_t)a.src[j] * P;
        mask[uo + q] = 1;
        const float4 g = dn[uo + q];
        const float3 Y = backproject(sc[1 + j], (float)(q % a.W), (float)(q / a.W), g.w);
        sx = fadd(sx, Y.x); sy = fadd(sy, Y.y); sz = fadd(sz, Y.z);
        nx = fadd(nx, g.x); ny = fadd(ny, g.y); nz = fadd(nz, g.z);
        const uchar4 c = col[uo + q];
        cb += c.x; cg += c.y; cr += c.z;
        ++k;
    }
    const float fk = (float)k;
    out_xyz[3 * (size_t)idx] = fdiv(sx, fk);
    out_xyz[3 * (size_t)idx + 1] = fdiv(sy, fk);
    out_xyz[3 * (size_t)idx + 2] = fdiv(sz, fk);
    const float len = norm3(nx, ny, nz);
    const bool usable = len > 0.0f && len <= 3.402823466e38f;  // a zero or overflowing sum has no direction: (0, 0, 0)
    out_nrm[3 * (size_t)idx] = usable ? fdiv(nx, len) : 0.0f;
    out_nrm[3 * (size_t)idx + 1] = usable ? fdiv(ny, len) : 0.0f;
    out_nrm[3 * (size_t)idx + 2] = usable ? fdiv(nz, len) : 0.0f;
    out_rgb[3 * (size_t)idx] = (unsigned char)((2 * cr + k) / (2 * k));  // mean rounded half up
    out_rgb[3 * (size_t)idx + 1] = (unsigned char)((2 * cg + k) / (2 * k));
    out_rgb[3 * (size_t)idx + 2] = (unsigned char)((2 * cb + k) / (2 * k));
}

}  // namespace

struct tsar_fusion : HandleCore {
    int n_views = 0, W = 0, H = 0;
    size_t P = 0;
    std::vector<FusionCam> cams;
    std::vector<std::vector<int>> neighbours;  // empty = view not set
    // resident inputs: 21 B per pixel and view
    DeviceBuf<FusionCam> d_cams;
    DeviceBuf<float4> d_dn;
    DeviceBuf<uchar4> d_col;
    DeviceBuf<unsigned char> d_mask;
    // scratch for one view
    DeviceBuf<int> d_cand, d_owner;
    DeviceBuf<unsigned char> d_state[2];
    DeviceBuf<int> d_block, d_counters;  // block counts + offsets; counters = {undecided, total}
    DeviceBuf<float> d_xyz, d_nrm;
    DeviceBuf<unsigned char> d_rgb;
    // pinned landing buffers of one view, and the points of the last run
    PinnedBuf<float> h_xyz, h_nrm;
    PinnedBuf<unsigned char> h_rgb;
    PinnedBuf<int> h_counters;
    std::vector<float> xyz, nrm;
    std::vector<unsigned char> rgb;
    long long n_points = 0;
    int rounds_max = 0;
    long long rounds_total = 0;
};

// K^-1 by the adjugate in double, rounded once to float (oc_fuse computes it the same way).
static bool invert3(const float *K, float *out) {
    double m[9], a[9];
    for (int i = 0; i < 9; ++i) m[i] = K[i];
    a[0] = m[4] * m[8] - m[5] * m[7]; a[1] = m[2] * m[7] - m[1] * m[8]; a[2] = m[1] * m[5] - m[2] * m[4];
    a[3] = m[5] * m[6] - m[3] * m[8]; a[4] = m[0] * m[8] - m[2] * m[6]; a[5] = m[2] * m[3] - m[0] * m[5];
    a[6] = m[3] * m[7] - m[4] * m[6]; a[7] = m[1] * m[6] - m[0] * m[7]; a[8] = m[0] * m[4] - m[1] * m[3];
    const double det = m[0] * a[0] + m[1] * a[3] + m[2] * a[6];
    if (!(det != 0.0) || !isfinite(det)) return false;
    for (int i = 0; i < 9; ++i) out[i] = (float)(a[i] / det);
    return true;
}

extern "C" {

int tsar_fusion_create(int device, void *stream, int n_views, int W, int H, tsar_fusion **out) {
    if (!out) return TSAR_ERR_ARG;
    *out = nullptr;
    // pixel indices are int: the last block's p must not overflow, and no index may reach the owner sentinel 0x7f7f7f7f
    if (n_views < 1 || W < 1 || H < 1 || (long long)W * H > 0x7f7f7f7fLL - kThreads) return TSAR_ERR_ARG;
    std::unique_ptr<tsar_fusion> f(new tsar_fusion);
    if (int rc = f->open(device, stream)) return rc;
    f->n_views = n_views;
    f->W = W;
    f->H = H;
    f->P = (size_t)W * H;
    f->cams.resize(n_views);
    f->neighbours.resize(n_views);
    const size_t P = f->P, N = (size_t)n_views, nb = (P + kThreads - 1) / kThreads;
    TSAR_CK(f, f->d_cams.reserve(N));
    TSAR_CK(f, f->d_dn.reserve(N * P));
    TSAR_CK(f, f->d_col.reserve(N * P));
    TSAR_CK(f, f->d_mask.reserve(N * P));
    TSAR_CK(f, f->d_state[0].reserve(P));
    TSAR_CK(f, f->d_state[1].reserve(P));
    TSAR_CK(f, f->d_block.reserve(2 * nb));
    TSAR_CK(f, f->d_counters.reserve(2));
    TSAR_CK(f, f->d_xyz.reserve(3 * P));
    TSAR_CK(f, f->d_nrm.reserve(3 * P));
    TSAR_CK(f, f->d_rgb.reserve(3 * P));
    TSAR_CK(f, f->h_xyz.reserve(3 * P));
    TSAR_CK(f, f->h_nrm.reserve(3 * P));
    TSAR_CK(f, f->h_rgb.reserve(3 * P));
    TSAR_CK(f, f->h_counters.reserve(2));
    *out = f.release();
    return TSAR_OK;
}

int tsar_fusion_destroy(tsar_fusion *f) {
    if (!f) return TSAR_OK;
    cudaSetDevice(f->device);
    cudaStreamSynchronize(f->stream);
    delete f;
    return TSAR_OK;
}

const char *tsar_fusion_last_error(const tsar_fusion *f) { return f ? f->err.c_str() : "null fusion handle"; }

int tsar_fusion_set_view(tsar_fusion *f, int view, const tsar_view_camera *cam, const float *depth, const float *normals,
                         const unsigned char *bgr, const int *neighbours, int n_neighbours) {
    if (!f) return TSAR_ERR_ARG;
    if (view < 0 || view >= f->n_views) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: view index out of range");
    if (!cam || !depth || !normals || !bgr || !neighbours) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: null pointer");
    if (n_neighbours < 1 || n_neighbours > TSAR_FUSION_MAX_NEIGHBOURS)
        TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: a view needs 1..32 neighbours");
    std::vector<int> nb(neighbours, neighbours + n_neighbours);
    for (int j = 0; j < n_neighbours; ++j) {
        if (nb[j] < 0 || nb[j] >= f->n_views) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: neighbour index out of range");
        if (nb[j] == view) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: a view cannot be its own neighbour");
        for (int i = 0; i < j; ++i)
            if (nb[i] == nb[j]) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: repeated neighbour");
    }
    FusionCam c;
    memcpy(c.K, cam->K, sizeof c.K);
    memcpy(c.R, cam->R, sizeof c.R);
    memcpy(c.t, cam->t, sizeof c.t);
    if (!invert3(c.K, c.Kinv)) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_set_view: K is singular");
    TSAR_CK(f, cudaSetDevice(f->device));
    const size_t P = f->P, vo = (size_t)view * P;
    // the host arrays land in the per-view output buffers (16 + 3 of their 27 bytes per pixel), then are packed
    float *st_depth = f->d_xyz.get(), *st_normals = f->d_nrm.get();
    TSAR_CK(f, cudaMemcpyAsync(st_depth, depth, P * sizeof(float), cudaMemcpyHostToDevice, f->stream));
    TSAR_CK(f, cudaMemcpyAsync(st_normals, normals, 3 * P * sizeof(float), cudaMemcpyHostToDevice, f->stream));
    TSAR_CK(f, cudaMemcpyAsync(f->d_rgb.get(), bgr, 3 * P, cudaMemcpyHostToDevice, f->stream));
    fusion_pack_kernel<<<(unsigned)((P + kThreads - 1) / kThreads), kThreads, 0, f->stream>>>(
        st_depth, st_normals, f->d_rgb.get(), P, f->d_dn.get() + vo, f->d_col.get() + vo);
    TSAR_CK(f, cudaGetLastError());
    TSAR_CK(f, cudaMemcpyAsync(f->d_cams.get() + view, &c, sizeof c, cudaMemcpyHostToDevice, f->stream));
    TSAR_CK(f, cudaStreamSynchronize(f->stream));
    f->cams[view] = c;
    f->neighbours[view] = nb;
    return TSAR_OK;
}

int tsar_fusion_run(tsar_fusion *f, const tsar_fusion_params *prm, long long *n_points) {
    if (!f) return TSAR_ERR_ARG;
    if (!prm) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_run: null parameters");
    if (!(prm->max_reproj_px > 0.0f) || !(prm->max_rel_depth > 0.0f) || !(prm->max_normal_deg >= 0.0f) ||
        !(prm->max_normal_deg <= 180.0f) || prm->min_consistent < 1)
        TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_run: parameters out of range (max_reproj_px > 0, max_rel_depth > 0, "
                            "0 <= max_normal_deg <= 180, min_consistent >= 1)");
    int max_src = 0;
    for (int v = 0; v < f->n_views; ++v) {
        if (f->neighbours[v].empty()) {
            char buf[128];
            snprintf(buf, sizeof buf, "tsar_fusion_run: view %d was not set", v);
            TSAR_FAIL(f, TSAR_ERR_ARG, buf);
        }
        max_src = std::max(max_src, (int)f->neighbours[v].size());
    }
    TSAR_CK(f, cudaSetDevice(f->device));
    const size_t P = f->P;
    TSAR_CK(f, f->d_cand.reserve((size_t)max_src * P));
    TSAR_CK(f, f->d_owner.reserve((size_t)max_src * P));
    const double kPi = 3.14159265358979323846;
    ViewArgs a{};
    a.W = f->W;
    a.H = f->H;
    a.min_consistent = prm->min_consistent;
    a.max_reproj = prm->max_reproj_px;
    a.max_rel = prm->max_rel_depth;
    a.cos_normal = (float)cos((double)prm->max_normal_deg * (kPi / 180.0));
    const unsigned nb = (unsigned)((P + kThreads - 1) / kThreads);
    int *d_block_count = f->d_block.get(), *d_block_off = f->d_block.get() + nb;
    TSAR_CK(f, cudaMemsetAsync(f->d_mask.get(), 0, (size_t)f->n_views * P, f->stream));
    f->xyz.clear(); f->nrm.clear(); f->rgb.clear();
    f->n_points = 0;
    f->rounds_max = 0;
    f->rounds_total = 0;
    for (int v = 0; v < f->n_views; ++v) {
        const std::vector<int> &S = f->neighbours[v];
        a.v = v;
        a.n_src = (int)S.size();
        for (int j = 0; j < a.n_src; ++j) a.src[j] = S[j];
        fusion_candidates_kernel<<<nb, kThreads, 0, f->stream>>>(a, f->d_cams.get(), f->d_dn.get(), f->d_mask.get(), f->d_cand.get(), f->d_state[0].get());
        TSAR_CK(f, cudaGetLastError());
        int cur = 0, rounds = 0;
        for (;;) {
            TSAR_CK(f, cudaMemsetAsync(f->d_owner.get(), 0x7f,   // 0x7f7f7f7f: no owner (larger than any pixel index)
                                 (size_t)a.n_src * P * sizeof(int), f->stream));
            TSAR_CK(f, cudaMemsetAsync(f->d_counters.get(), 0, sizeof(int), f->stream));
            fusion_claim_kernel<<<nb, kThreads, 0, f->stream>>>(a.n_src, (int)P, f->d_cand.get(), f->d_state[cur].get(), f->d_owner.get());
            fusion_decide_kernel<<<nb, kThreads, 0, f->stream>>>(a.n_src, (int)P, a.min_consistent, f->d_cand.get(), f->d_owner.get(),
                                                                 f->d_state[cur].get(), f->d_state[cur ^ 1].get(), f->d_counters.get());
            TSAR_CK(f, cudaGetLastError());
            TSAR_CK(f, cudaMemcpyAsync(f->h_counters.get(), f->d_counters.get(), sizeof(int), cudaMemcpyDeviceToHost, f->stream));
            TSAR_CK(f, cudaStreamSynchronize(f->stream));
            cur ^= 1;
            ++rounds;
            if (f->h_counters.get()[0] == 0) break;
        }
        f->rounds_max = std::max(f->rounds_max, rounds);
        f->rounds_total += rounds;
        fusion_count_kernel<<<nb, kThreads, 0, f->stream>>>((int)P, f->d_state[cur].get(), d_block_count);
        fusion_scan_kernel<<<1, 1024, 0, f->stream>>>(d_block_count, (int)nb, d_block_off, f->d_counters.get() + 1);
        fusion_emit_kernel<<<nb, kThreads, 0, f->stream>>>(a, f->d_cams.get(), f->d_dn.get(), f->d_col.get(), f->d_mask.get(), f->d_cand.get(), f->d_owner.get(),
                                                           f->d_state[cur].get(), d_block_off, f->d_xyz.get(), f->d_nrm.get(), f->d_rgb.get());
        TSAR_CK(f, cudaGetLastError());
        TSAR_CK(f, cudaMemcpyAsync(f->h_counters.get() + 1, f->d_counters.get() + 1, sizeof(int), cudaMemcpyDeviceToHost, f->stream));
        TSAR_CK(f, cudaStreamSynchronize(f->stream));
        const size_t n = (size_t)f->h_counters.get()[1];
        if (n) {
            TSAR_CK(f, cudaMemcpyAsync(f->h_xyz.get(), f->d_xyz.get(), 3 * n * sizeof(float), cudaMemcpyDeviceToHost, f->stream));
            TSAR_CK(f, cudaMemcpyAsync(f->h_nrm.get(), f->d_nrm.get(), 3 * n * sizeof(float), cudaMemcpyDeviceToHost, f->stream));
            TSAR_CK(f, cudaMemcpyAsync(f->h_rgb.get(), f->d_rgb.get(), 3 * n, cudaMemcpyDeviceToHost, f->stream));
            TSAR_CK(f, cudaStreamSynchronize(f->stream));
            f->xyz.insert(f->xyz.end(), f->h_xyz.get(), f->h_xyz.get() + 3 * n);
            f->nrm.insert(f->nrm.end(), f->h_nrm.get(), f->h_nrm.get() + 3 * n);
            f->rgb.insert(f->rgb.end(), f->h_rgb.get(), f->h_rgb.get() + 3 * n);
            f->n_points += (long long)n;
        }
    }
    if (n_points) *n_points = f->n_points;
    return TSAR_OK;
}

int tsar_fusion_points(tsar_fusion *f, float *xyz, float *normals, unsigned char *rgb, long long capacity) {
    if (!f) return TSAR_ERR_ARG;
    if (capacity < f->n_points) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_points: capacity is smaller than the number of points");
    const size_t n = (size_t)f->n_points;
    if (n && (!xyz || !normals || !rgb)) TSAR_FAIL(f, TSAR_ERR_ARG, "tsar_fusion_points: null pointer");
    if (n) {
        memcpy(xyz, f->xyz.data(), 3 * n * sizeof(float));
        memcpy(normals, f->nrm.data(), 3 * n * sizeof(float));
        memcpy(rgb, f->rgb.data(), 3 * n);
    }
    return TSAR_OK;
}

int tsar_fusion_dbg_rounds(const tsar_fusion *f, int *max_rounds, long long *total_rounds) {
    if (!f) return TSAR_ERR_ARG;
    if (max_rounds) *max_rounds = f->rounds_max;
    if (total_rounds) *total_rounds = f->rounds_total;
    return TSAR_OK;
}

}  // extern "C"
