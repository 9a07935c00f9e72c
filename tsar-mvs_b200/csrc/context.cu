// context.cu -- host side of the C ABI declared in include/tsar_b200.h.
//
// One tsar_ctx owns the device-resident state of one reference view: images (textures for the
// hardware-filtered source samples + a linear copy of the reference image for the hoisted window
// terms), cameras, and the LineState arrays of the reference (linestate.h:10-221) as plain device
// SoA buffers -- no managed memory, no device-wide syncs, everything on one stream.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/tsar_b200.h"
#include "debug_kernels.cuh"
#include "glue_kernels.cuh"
#include "pm_launch.h"
#include "ransac_kernels.cuh"
#include "slic_kernels.cuh"
#include "wmf_kernels.cuh"

using namespace tsar;

struct RansacScratch {
    int *block_counts = nullptr, *list = nullptr, *totals = nullptr, *hyp_counts = nullptr, *regions = nullptr;
    float3 *pts = nullptr;
    uint32_t *rnd = nullptr;
    RansacJob *jobs = nullptr;
    float4 *out = nullptr;
    RansacState *states = nullptr;
    size_t px_cap = 0;
    int nt_cap = 0, grid = 0;
};

// Checkerboard launches after the planes were set that use quad-cooperative sampling (the rest use the per-lane
// loop).  Chosen by measurement, DESIGN.md 4.4.
constexpr int kQuadLaunches = 2;

struct tsar_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int W = 0, H = 0, n_images = 0, V = 0;
    bool have_views = false, have_params = false, have_planes = false;
    std::vector<tsar_camera> cams;
    float cam_f = 0.f;
    std::vector<int> subset;
    tsar_params params{};
    // images
    std::vector<cudaArray_t> arrays;
    std::vector<cudaTextureObject_t> tex;
    std::vector<cudaArray_t> arrays8;          // 8-bit copies of the views (sampling fast path)
    std::vector<cudaTextureObject_t> tex8;
    unsigned char *stage8 = nullptr;           // staging buffer for the float -> u8 conversion
    int region_cap = 0;                        // allocated entries of region_text / region_plane
    float *stage32 = nullptr;                  // linear landing buffer for host images (tsar_set_views, on_device = 0)
    size_t stage32_n = 0;
    int *d_flag = nullptr;
    int use_u8 = 0;                            // every image is 8-bit valued: sample the 8-bit textures
    bool allow_u8 = true;                      // env TSAR_B200_NO_U8=1 switches the fast path off
    bool u8_verified = false, u8_ok = false;   // one-time self-check of the 8-bit sampling identity (tsar_set_views)
    int arr_w = 0, arr_h = 0;
    float *ref_img = nullptr;
    cudaTextureObject_t *d_tex = nullptr;
    CamDev *d_cams = nullptr;
    // per-pixel state (capacity n_alloc pixels)
    size_t n_alloc = 0;
    float4 *plane[2] = {nullptr, nullptr};
    float *cost[2] = {nullptr, nullptr};
    int cur[2] = {0, 0};  // buffer holding the live values of colour 0 (black) / 1 (red)
    float *depth = nullptr, *fakedepth = nullptr, *scale = nullptr, *canny = nullptr, *ratio = nullptr,
          *lrdiff = nullptr, *confid = nullptr;
    int *beview = nullptr;
    float *region_text = nullptr;
    float4 *region_plane = nullptr;
    int n_regions = 0;
    uint32_t *rng = nullptr;
    size_t rng_alloc = 0;
    uint32_t *rng_batch = nullptr;             // tables of all refinement launches of one tsar_iterate call
    size_t rng_batch_alloc = 0;
    int rng_pitch = 0, rng_len = 0;
    // scratch for tsar_eval_planes
    void *scratch = nullptr;
    size_t scratch_bytes = 0;
    PmConst pm{};
    PmConst pm_init{};  // init uses box/2 instead of (box-1)/2 (gipuma.cu:693-694, SURVEY Q7)
    GlueConst glue{};
    const PmVariant *variant = &pm_variant_generic;       // kernels compiled for this window / combination
    const PmVariant *variant_init = &pm_variant_generic;
    long long launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool fused = true;
    // quad-cooperative sampling (pm_core.cuh, view_cost_quad) for the initialisation and the first quad_launches
    // checkerboard launches after the planes were set; -1 (env TSAR_B200_NO_QUAD_SAMPLING=1): never
    int quad_launches = kQuadLaunches;
    int checker_since_planes = 0;
    int eval_wrapper_rounding = 0;  // test-only, see tsar_dbg_eval_rounding
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;  // around every checkerboard kernel
    SlicState slic;
    RansacScratch ransac;
};

#define CK(call)                                                                                    \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) {                                                                    \
            char buf_[512];                                                                         \
            snprintf(buf_, sizeof(buf_), "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            ctx->err = buf_;                                                                        \
            return TSAR_ERR_CUDA;                                                                   \
        }                                                                                           \
    } while (0)

#define FAIL(code, msg)      \
    do {                     \
        ctx->err = (msg);    \
        return (code);       \
    } while (0)

static const char *kVersion = "tsar_b200 0.1 (sm_100a)";

// ------------------------------------------------------------------------------------------------
// 8-bit copies of the views
// ------------------------------------------------------------------------------------------------
// flag |= 1 if any value is not an integer in [0, 255]; writes the 8-bit copy on the way
__global__ void to_u8_kernel(const float *__restrict__ img, unsigned char *__restrict__ out, size_t n, int *flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = img[i];
    const float r = rintf(v);
    const bool ok = (v == r) && (v >= 0.0f) && (v <= 255.0f);
    out[i] = ok ? (unsigned char)r : 0;
    if (!ok) *flag = 1;
}

// Self-check of the 8-bit sampling identity: 4096 pseudo-random coordinates (an eighth of them pushed onto the image
// border, where clamp addressing acts) sampled through the fp32 texture and through the 8-bit copy; the 8-bit result,
// snapped as view_cost snaps it (N = rint(v * 255 * 256), value N / 256), must equal the fp32 sample bit for bit.
__global__ void u8_selfcheck_kernel(cudaTextureObject_t tex32, cudaTextureObject_t tex8, int W, int H, int *mismatches) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned h = i * 2654435761u + 12345u;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    const unsigned g = h * 3266489917u + 1u;
    float x = (float)(h % (unsigned)(W * 64)) / 64.0f, y = (float)((g >> 4) % (unsigned)(H * 64)) / 64.0f;
    if ((i & 7u) == 0u) { x = (i & 8u) ? -1.37f : (float)W + 0.61f; }
    if ((i & 7u) == 1u) { y = (i & 8u) ? -0.73f : (float)H + 1.29f; }
    const float a = tex2D<float>(tex32, x, y);
    const float v = tex2D<float>(tex8, x, y);
    const float n = __fsub_rn(__fmaf_rn(v, 65280.0f, 12582912.0f), 12582912.0f);
    if (__float_as_uint(__fmul_rn(n, 0.00390625f)) != __float_as_uint(a)) atomicAdd(mismatches, 1);
}

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
static size_t win_smem_bytes(int nt, int ns) { return (size_t)ns * nt * sizeof(float2) + (size_t)ns * sizeof(float); }

static const PmVariant *pick_variant(const tsar_params &p, bool init) {
    const int hs = p.box_hsize, vs = p.box_vsize;
    const int hr = init ? hs / 2 : (hs - 1) / 2, vr = init ? vs / 2 : (vs - 1) / 2;
    const bool fast_comb = (p.cost_comb == 1 && p.n_best <= 2);
    if (fast_comb && hr == vr && hr == 5) return &pm_variant_w11;
    if (fast_comb && hr == vr && hr == 9) return &pm_variant_w19;
    return &pm_variant_generic;
}

static void fill_window(PmConst &c, int hs, int vs, bool init) {
    c.hrad = init ? hs / 2 : (hs - 1) / 2;
    c.vrad = init ? vs / 2 : (vs - 1) / 2;
    c.n1x = c.hrad + 1;  // i = -hrad, -hrad+2, ..., <= hrad   (gipuma.cu:259)
    c.n1y = c.vrad + 1;
    c.ns = c.n1x * c.n1y;
}

static int rebuild_constants(tsar_ctx *ctx) {
    if (!ctx->have_views || !ctx->have_params) return TSAR_OK;
    PmConst &c = ctx->pm;
    memset(&c, 0, sizeof(c));
    const tsar_camera &r = ctx->cams[0];
    c.W = ctx->W; c.H = ctx->H; c.V = ctx->V;
    fill_window(c, ctx->params.box_hsize, ctx->params.box_vsize, false);
    c.n_best = ctx->params.n_best;
    c.cost_comb = ctx->params.cost_comb;
    c.y_limit = std::min(ctx->H, 32 * (((ctx->H / 2) + 15) / 16));
    c.rng_pitch = ctx->rng_pitch;
    for (int i = 0; i < 9; i++) { c.Kinv[i] = r.K_inv[i]; c.Minv[i] = r.M_inv[i]; }
    for (int i = 0; i < 3; i++) { c.Pc[i] = r.P_col34[i]; c.C[i] = r.C4[i]; }
    c.fx = r.fx; c.alpha = r.alpha; c.cx = r.K[2]; c.cy = r.K[5];
    c.f_params = ctx->cam_f; c.f_cam0 = r.f; c.baseline = r.baseline;
    c.depthMin = r.depthMin; c.depthMax = r.depthMax;
    c.min_disp = ctx->params.min_disparity; c.max_disp = ctx->params.max_disparity;
    for (int i = 0; i < ctx->V; i++) {
        const int id = ctx->subset[i];
        const tsar_camera &s = ctx->cams[id];
        c.tex[i] = ctx->tex[id];
        c.tex8[i] = ctx->use_u8 ? ctx->tex8[id] : 0;
        c.view_id[i] = id;
        for (int k = 0; k < 9; k++) { c.view[i].R[k] = s.R[k]; c.view[i].K[k] = s.K[k]; }
        for (int k = 0; k < 3; k++) c.view[i].t[k] = s.t4[k];
    }
    // zero-skew pinhole intrinsics everywhere? (lets the homography skip the products with exact zeros)
    auto pinhole = [](const float *K) { return K[1] == 0.f && K[3] == 0.f && K[6] == 0.f && K[7] == 0.f && K[8] == 1.f; };
    c.k_pinhole = pinhole(r.K_inv) ? 1 : 0;
    for (int i = 0; i < ctx->V && c.k_pinhole; i++) c.k_pinhole = pinhole(c.view[i].K) ? 1 : 0;
    const char *nk = getenv("TSAR_B200_NO_PINHOLE_FASTPATH");
    if (nk && nk[0] == '1') c.k_pinhole = 0;
    ctx->pm_init = c;
    fill_window(ctx->pm_init, ctx->params.box_hsize, ctx->params.box_vsize, true);
    ctx->variant = pick_variant(ctx->params, false);
    ctx->variant_init = pick_variant(ctx->params, true);
    if (win_smem_bytes(128, std::max(c.ns, ctx->pm_init.ns)) > 220 * 1024)
        FAIL(TSAR_ERR_ARG, "window too large for the shared-memory weight table");
    GlueConst &g = ctx->glue;
    memset(&g, 0, sizeof(g));
    g.W = ctx->W; g.H = ctx->H; g.hrad = c.hrad; g.vrad = c.vrad;
    for (int i = 0; i < 9; i++) {
        g.Kinv[i] = r.K_inv[i]; g.Minv[i] = r.M_inv[i]; g.Rorig[i] = r.R_orig[i]; g.Rorig_inv[i] = r.R_orig_inv[i];
    }
    for (int i = 0; i < 3; i++) { g.Pc[i] = r.P_col34[i]; g.C[i] = r.C4[i]; }
    g.fx = r.fx; g.alpha = r.alpha; g.cx = r.K[2]; g.cy = r.K[5];
    g.f_params = ctx->cam_f; g.baseline = r.baseline;
    g.min_disp = c.min_disp; g.max_disp = c.max_disp; g.depthMin = c.depthMin; g.depthMax = c.depthMax;
    return TSAR_OK;
}

static void free_state(tsar_ctx *ctx) {
    for (int b = 0; b < 2; b++) { cudaFree(ctx->plane[b]); cudaFree(ctx->cost[b]); ctx->plane[b] = nullptr; ctx->cost[b] = nullptr; }
    cudaFree(ctx->depth); cudaFree(ctx->fakedepth); cudaFree(ctx->scale); cudaFree(ctx->canny);
    cudaFree(ctx->ratio); cudaFree(ctx->lrdiff); cudaFree(ctx->confid); cudaFree(ctx->beview);
    ctx->depth = ctx->fakedepth = ctx->scale = ctx->canny = ctx->ratio = ctx->lrdiff = ctx->confid = nullptr;
    ctx->beview = nullptr;
    cudaFree(ctx->ref_img); ctx->ref_img = nullptr;
    ctx->n_alloc = 0;
}

static void free_images(tsar_ctx *ctx) {
    for (auto t : ctx->tex) cudaDestroyTextureObject(t);
    for (auto a : ctx->arrays) cudaFreeArray(a);
    for (auto t : ctx->tex8) cudaDestroyTextureObject(t);
    for (auto a : ctx->arrays8) cudaFreeArray(a);
    ctx->tex8.clear();
    ctx->arrays8.clear();
    cudaFree(ctx->stage8); ctx->stage8 = nullptr;
    ctx->tex.clear();
    ctx->arrays.clear();
    ctx->arr_w = ctx->arr_h = 0;
}

static int ensure_state(tsar_ctx *ctx, size_t n) {
    if (n <= ctx->n_alloc) return TSAR_OK;
    free_state(ctx);
    for (int b = 0; b < 2; b++) {
        CK(cudaMalloc(&ctx->plane[b], n * sizeof(float4)));
        CK(cudaMalloc(&ctx->cost[b], n * sizeof(float)));
    }
    CK(cudaMalloc(&ctx->depth, n * 4)); CK(cudaMalloc(&ctx->fakedepth, n * 4)); CK(cudaMalloc(&ctx->scale, n * 4));
    CK(cudaMalloc(&ctx->canny, n * 4)); CK(cudaMalloc(&ctx->ratio, n * 4)); CK(cudaMalloc(&ctx->lrdiff, n * 4));
    CK(cudaMalloc(&ctx->confid, n * 4)); CK(cudaMalloc(&ctx->beview, n * 4));
    CK(cudaMalloc(&ctx->ref_img, n * 4));
    ctx->n_alloc = n;
    return TSAR_OK;
}

// LineState::resize memsets every array to 0 (linestate.h:73-109).  caller_inputs: also clear the arrays the
// caller fills between the entry points (canny labels, reliable flags); a new view clears them, a re-run of
// the PatchMatch path on the same view keeps them.
static int zero_state(tsar_ctx *ctx, bool caller_inputs) {
    const size_t n = (size_t)ctx->W * ctx->H;
    cudaStream_t s = ctx->stream;
    for (int b = 0; b < 2; b++) { CK(cudaMemsetAsync(ctx->plane[b], 0, n * 16, s)); CK(cudaMemsetAsync(ctx->cost[b], 0, n * 4, s)); }
    CK(cudaMemsetAsync(ctx->depth, 0, n * 4, s)); CK(cudaMemsetAsync(ctx->fakedepth, 0, n * 4, s));
    if (caller_inputs) { CK(cudaMemsetAsync(ctx->scale, 0, n * 4, s)); CK(cudaMemsetAsync(ctx->canny, 0, n * 4, s)); }
    CK(cudaMemsetAsync(ctx->ratio, 0, n * 4, s)); CK(cudaMemsetAsync(ctx->lrdiff, 0, n * 4, s));
    CK(cudaMemsetAsync(ctx->confid, 0, n * 4, s)); CK(cudaMemsetAsync(ctx->beview, 0, n * 4, s));
    ctx->cur[0] = ctx->cur[1] = 0;
    return TSAR_OK;
}

static int ensure_scratch(tsar_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->scratch_bytes) return TSAR_OK;
    cudaFree(ctx->scratch);
    ctx->scratch = nullptr;
    ctx->scratch_bytes = 0;
    CK(cudaMalloc(&ctx->scratch, bytes));
    ctx->scratch_bytes = bytes;
    return TSAR_OK;
}

static int need_ready(tsar_ctx *ctx) {
    if (!ctx) return TSAR_ERR_ARG;
    if (!ctx->have_views) FAIL(TSAR_ERR_STATE, "tsar_set_views has not been called");
    if (!ctx->have_params) FAIL(TSAR_ERR_STATE, "tsar_set_params has not been called");
    CK(cudaSetDevice(ctx->device));
    return TSAR_OK;
}

// both colours back into buffer 0
static int consolidate(tsar_ctx *ctx) {
    for (int col = 0; col < 2; col++)
        if (ctx->cur[col] != 0) {
            CK(pm_launch_merge_colour(ctx->W, ctx->H, col, ctx->plane[1], ctx->cost[1], ctx->plane[0], ctx->cost[0],
                                      ctx->stream));
            ctx->launches++;
            ctx->cur[col] = 0;
        }
    return TSAR_OK;
}

static int make_rng_table(tsar_ctx *ctx, uint64_t seed) {
    CK(pm_launch_rng_table(ctx->rng, ctx->rng_pitch, ctx->H, ctx->rng_len, seed, ctx->stream));
    ctx->launches++;
    return TSAR_OK;
}

static int launch_checker(tsar_ctx *ctx, int mode, int colour, const uint32_t *rng_table = nullptr) {
    CheckerArgs a;
    for (int col = 0; col < 2; col++) { a.plane_in[col] = ctx->plane[ctx->cur[col]]; a.cost_in[col] = ctx->cost[ctx->cur[col]]; }
    const bool sp = (mode & PM_MODE_SP) != 0;
    const int out = sp ? (ctx->cur[colour] ^ 1) : ctx->cur[colour];
    a.plane_out = ctx->plane[out];
    a.cost_out = ctx->cost[out];
    a.ratio = ctx->ratio;
    a.beview = ctx->beview;
    a.rng = rng_table ? rng_table : ctx->rng;
    a.colour = colour;
    cudaEvent_t p0 = nullptr, p1 = nullptr;
    if (ctx->profiling) {
        CK(cudaEventCreate(&p0)); CK(cudaEventCreate(&p1));
        CK(cudaEventRecord(p0, ctx->stream));
    }
    const int quad = ctx->checker_since_planes < ctx->quad_launches && ctx->variant->has_quad && ctx->use_u8 && ctx->pm.k_pinhole;
    CK(ctx->variant->checker(ctx->use_u8, quad, mode, ctx->pm, ctx->ref_img, a, ctx->stream));
    ctx->checker_since_planes++;
    if (ctx->profiling) {
        CK(cudaEventRecord(p1, ctx->stream));
        ctx->prof_events.emplace_back(p0, p1);
    }
    ctx->launches++;
    ctx->cur[colour] = out;
    return TSAR_OK;
}

// rows beyond the reference's checkerboard grid are never touched by a half-step: make sure the
// alternate buffer carries them too (they keep their initial values forever)
static int seed_alt_buffers(tsar_ctx *ctx) {
    const size_t n = (size_t)ctx->W * ctx->H;
    if (ctx->pm.y_limit < ctx->H) {
        CK(cudaMemcpyAsync(ctx->plane[1], ctx->plane[0], n * 16, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->cost[1], ctx->cost[0], n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return TSAR_OK;
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char *tsar_version(void) { return kVersion; }

int tsar_create(int device, void *stream, tsar_ctx **out) {
    if (!out) return TSAR_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        fprintf(stderr, "[tsar_b200] no usable CUDA device (requested %d of %d); this library has no CPU path\n", device, ndev);
        return TSAR_ERR_NODEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
        fprintf(stderr, "[tsar_b200] device %d is sm_%d%d; this build contains sm_100a code only\n", device, prop.major, prop.minor);
        return TSAR_ERR_NODEVICE;
    }
    tsar_ctx *ctx = new tsar_ctx;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return TSAR_ERR_CUDA; }
    if (stream) ctx->stream = (cudaStream_t)stream;
    else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return TSAR_ERR_CUDA; }
        ctx->own_stream = true;
    }
    cudaEventCreate(&ctx->ev0);
    cudaEventCreate(&ctx->ev1);
    const char *uf = getenv("TSAR_B200_UNFUSED");
    ctx->fused = !(uf && uf[0] == '1');
    const char *n8 = getenv("TSAR_B200_NO_U8");
    ctx->allow_u8 = !(n8 && n8[0] == '1');
    const char *nq = getenv("TSAR_B200_NO_QUAD_SAMPLING");
    if (nq && nq[0] == '1') ctx->quad_launches = -1;
    *out = ctx;
    return TSAR_OK;
}

int tsar_destroy(tsar_ctx *ctx) {
    if (!ctx) return TSAR_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    free_state(ctx);
    free_images(ctx);
    for (auto &pr : ctx->prof_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    cudaFree(ctx->d_tex); cudaFree(ctx->d_cams); cudaFree(ctx->rng); cudaFree(ctx->rng_batch); cudaFree(ctx->scratch);
    cudaFree(ctx->region_text); cudaFree(ctx->region_plane); cudaFree(ctx->d_flag); cudaFree(ctx->stage32);
    slic_free(ctx->slic);
    { RansacScratch &r = ctx->ransac; cudaFree(r.block_counts); cudaFree(r.list); cudaFree(r.totals); cudaFree(r.hyp_counts); cudaFree(r.regions);
      cudaFree(r.pts); cudaFree(r.rnd); cudaFree(r.jobs); cudaFree(r.out); cudaFree(r.states); }
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return TSAR_OK;
}

const char *tsar_last_error(const tsar_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tsar_sync(tsar_ctx *ctx) {
    if (!ctx) return TSAR_ERR_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_set_views(tsar_ctx *ctx, int W, int H, int n_images, const float *const *images, int on_device,
                   const tsar_camera *cams, float cam_f, const int *subset, int V) {
    if (!ctx) return TSAR_ERR_ARG;
    if (W <= 0 || H <= 0 || n_images < 1 || n_images > 512 || !images || !cams) FAIL(TSAR_ERR_ARG, "bad view arguments");
    if (V < 1 || V > TSAR_MAX_VIEWS || !subset) FAIL(TSAR_ERR_ARG, "number of selected views must be in [1, 32] (pmCostMultiview_cu costVector[32])");
    for (int i = 0; i < V; i++)
        if (subset[i] < 0 || subset[i] >= n_images) FAIL(TSAR_ERR_ARG, "view subset index out of range");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)W * H;
    int rc = ensure_state(ctx, n);
    if (rc) return rc;
    // textures: same descriptor as addImageToTextureFloatGray (main.cpp:1190-1228): float, linear
    // filter, unnormalised coordinates, address mode "wrap" (which the hardware treats as clamp for
    // unnormalised coordinates, SURVEY Q9) -- identical descriptor => identical sampling
    if (ctx->arr_w != W || ctx->arr_h != H || (int)ctx->arrays.size() != n_images) {
        free_images(ctx);
        cudaChannelFormatDesc cd = cudaCreateChannelDesc(32, 0, 0, 0, cudaChannelFormatKindFloat);
        for (int i = 0; i < n_images; i++) {
            cudaArray_t a;
            CK(cudaMallocArray(&a, &cd, W, H));
            ctx->arrays.push_back(a);
            cudaResourceDesc rd;
            memset(&rd, 0, sizeof(rd));
            rd.resType = cudaResourceTypeArray;
            rd.res.array.array = a;
            cudaTextureDesc td;
            memset(&td, 0, sizeof(td));
            td.addressMode[0] = cudaAddressModeWrap;
            td.addressMode[1] = cudaAddressModeWrap;
            td.filterMode = cudaFilterModeLinear;
            td.readMode = cudaReadModeElementType;
            td.normalizedCoords = 0;
            cudaTextureObject_t t;
            CK(cudaCreateTextureObject(&t, &rd, &td, NULL));
            ctx->tex.push_back(t);
        }
        ctx->arr_w = W; ctx->arr_h = H;
        cudaFree(ctx->d_tex); cudaFree(ctx->d_cams);
        ctx->d_tex = nullptr; ctx->d_cams = nullptr;
        CK(cudaMalloc(&ctx->d_tex, n_images * sizeof(cudaTextureObject_t)));
        CK(cudaMalloc(&ctx->d_cams, n_images * sizeof(CamDev)));
        CK(cudaMemcpyAsync(ctx->d_tex, ctx->tex.data(), n_images * sizeof(cudaTextureObject_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    // 8-bit copies: the reference's inputs are 8-bit grey images converted to float (main.cpp:1423), for which an
    // 8-bit texture gives bit-identical bilinear samples at a quarter of the texel traffic (pm_core.cuh, view_cost)
    ctx->use_u8 = 0;
    if (ctx->allow_u8 && (int)ctx->arrays8.size() != n_images) {
        for (auto t : ctx->tex8) cudaDestroyTextureObject(t);
        for (auto a : ctx->arrays8) cudaFreeArray(a);
        ctx->tex8.clear(); ctx->arrays8.clear();
        cudaFree(ctx->stage8); ctx->stage8 = nullptr;
        cudaChannelFormatDesc c8 = cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned);
        for (int i = 0; i < n_images; i++) {
            cudaArray_t a;
            CK(cudaMallocArray(&a, &c8, W, H));
            ctx->arrays8.push_back(a);
            cudaResourceDesc rd;
            memset(&rd, 0, sizeof(rd));
            rd.resType = cudaResourceTypeArray;
            rd.res.array.array = a;
            cudaTextureDesc td;
            memset(&td, 0, sizeof(td));
            td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
            td.filterMode = cudaFilterModeLinear;
            td.readMode = cudaReadModeNormalizedFloat;
            td.normalizedCoords = 0;
            cudaTextureObject_t t;
            CK(cudaCreateTextureObject(&t, &rd, &td, NULL));
            ctx->tex8.push_back(t);
        }
        CK(cudaMalloc(&ctx->stage8, n));
    }
    if (!ctx->d_flag) CK(cudaMalloc(&ctx->d_flag, 2 * sizeof(int)));
    // host images cross the bus once, into a persistent linear staging buffer (no per-call cudaMalloc/cudaFree: those
    // synchronise the whole device and would serialise contexts that pipeline views on other streams)
    if (!on_device && ctx->stage32_n < n) {
        cudaFree(ctx->stage32); ctx->stage32 = nullptr; ctx->stage32_n = 0;
        CK(cudaMalloc(&ctx->stage32, n * 4));
        ctx->stage32_n = n;
    }
    CK(cudaMemsetAsync(ctx->d_flag, 0, 2 * sizeof(int), ctx->stream));
    for (int i = 0; i < n_images; i++) {
        const float *src = images[i];
        if (!on_device) {
            float *dst = (i == 0) ? ctx->ref_img : ctx->stage32;   // view 0 is also kept linear (hoisted window terms)
            CK(cudaMemcpyAsync(dst, images[i], n * 4, cudaMemcpyHostToDevice, ctx->stream));
            src = dst;
        } else if (i == 0) {
            CK(cudaMemcpyAsync(ctx->ref_img, images[0], n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        CK(cudaMemcpy2DToArrayAsync(ctx->arrays[i], 0, 0, src, (size_t)W * 4, (size_t)W * 4, H, cudaMemcpyDeviceToDevice, ctx->stream));
        if (ctx->allow_u8) {
            to_u8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(src, ctx->stage8, n, ctx->d_flag);
            CK(cudaMemcpy2DToArrayAsync(ctx->arrays8[i], 0, 0, ctx->stage8, (size_t)W, (size_t)W, H, cudaMemcpyDeviceToDevice, ctx->stream));
            ctx->launches++;
        }
    }
    ctx->W = W; ctx->H = H; ctx->n_images = n_images; ctx->V = V;
    ctx->cams.assign(cams, cams + n_images);
    ctx->cam_f = cam_f;
    ctx->subset.assign(subset, subset + V);
    std::vector<CamDev> cd(n_images);
    for (int i = 0; i < n_images; i++) {
        for (int k = 0; k < 9; k++) { cd[i].R[k] = cams[i].R[k]; cd[i].K[k] = cams[i].K[k]; }
        for (int k = 0; k < 3; k++) cd[i].t[k] = cams[i].t4[k];
    }
    CK(cudaMemcpyAsync(ctx->d_cams, cd.data(), n_images * sizeof(CamDev), cudaMemcpyHostToDevice, ctx->stream));
    // The 8-bit fast path rests on how the texture unit quantises its bilinear weights (pm_core.cuh, view_cost): checked
    // once per context on this device and driver, on the reference image incl. its borders, against the fp32 texture.
    int *flags = ctx->d_flag;   // [0] some image is not 8-bit valued, [1] mismatches of the self-check
    const bool check = ctx->allow_u8 && !ctx->u8_verified;
    if (check) {
        u8_selfcheck_kernel<<<16, 256, 0, ctx->stream>>>(ctx->tex[0], ctx->tex8[0], W, H, flags + 1);
        ctx->launches++;
    }
    int host_flags[2] = {1, 0};
    if (ctx->allow_u8) CK(cudaMemcpyAsync(host_flags, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // one wait per call: the flags are needed now, and cd / the caller's buffers may go away
    if (ctx->allow_u8) {
        if (check && host_flags[0] == 0) {     // (only meaningful when the image really is 8-bit valued)
            ctx->u8_verified = true;
            ctx->u8_ok = host_flags[1] == 0;
            if (!ctx->u8_ok) fprintf(stderr, "[tsar_b200] 8-bit texture self-check failed on this device/driver (%d of 4096 samples differ): sampling fp32 textures\n", host_flags[1]);
        }
        ctx->use_u8 = (host_flags[0] == 0) && ctx->u8_verified && ctx->u8_ok;
    }
    // XORWOW row table: W draws of offset + head-room for the Marsaglia rejection loop / 4 draws per refine round
    ctx->rng_len = W + 192;
    ctx->rng_pitch = (ctx->rng_len + 31) & ~31;
    const size_t need = (size_t)ctx->rng_pitch * H;
    if (need > ctx->rng_alloc) {
        cudaFree(ctx->rng);
        ctx->rng = nullptr;
        CK(cudaMalloc(&ctx->rng, need * sizeof(uint32_t)));
        ctx->rng_alloc = need;
    }
    ctx->have_views = true;
    ctx->have_planes = false;
    rc = zero_state(ctx, true);
    if (rc) return rc;
    return rebuild_constants(ctx);
}

int tsar_set_params(tsar_ctx *ctx, const tsar_params *p) {
    if (!ctx || !p) return TSAR_ERR_ARG;
    if (p->box_hsize < 1 || p->box_vsize < 1 || p->n_best < 1) FAIL(TSAR_ERR_ARG, "bad window / n_best");
    // color_processing: the reference then uploads BGRA float4 textures, but every kernel still samples them with
    // tex2D<float> (gipuma.cu:247, 262, 265, 341, 356, 359), which returns the first component: the arithmetic is
    // the grey path on channel x (blue).  Callers pass that channel as the view image; nothing else changes.
    ctx->params = *p;
    ctx->have_params = true;
    return rebuild_constants(ctx);
}

int tsar_init_planes(tsar_ctx *ctx, uint64_t seed) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = zero_state(ctx, false))) return rc;
    if ((rc = make_rng_table(ctx, seed))) return rc;
    const int quad = ctx->quad_launches >= 0 && ctx->variant_init->has_quad && ctx->use_u8;
    CK(ctx->variant_init->init(ctx->use_u8, quad, ctx->pm_init, ctx->ref_img, ctx->rng, ctx->rng_len, ctx->plane[0], ctx->cost[0], ctx->stream));
    ctx->launches++;
    ctx->checker_since_planes = 0;
    ctx->cur[0] = ctx->cur[1] = 0;
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_load_planes(tsar_ctx *ctx, const float *norm4, const float *cost) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!norm4) FAIL(TSAR_ERR_ARG, "norm4 is null");
    const size_t n = (size_t)ctx->W * ctx->H;
    CK(cudaMemcpyAsync(ctx->plane[0], norm4, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    if (cost) CK(cudaMemcpyAsync(ctx->cost[0], cost, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    else {
        CK(ctx->variant->cost_of_state(ctx->use_u8, ctx->pm, ctx->ref_img, ctx->plane[0], ctx->cost[0], ctx->stream));
        ctx->launches++;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->checker_since_planes = 0;
    ctx->cur[0] = ctx->cur[1] = 0;
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_launch(tsar_ctx *ctx, int kind, uint64_t seed) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->have_planes) FAIL(TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
    switch (kind) {
        case TSAR_BLACK_SPATIAL: return launch_checker(ctx, PM_MODE_SP, 0);
        case TSAR_RED_SPATIAL: return launch_checker(ctx, PM_MODE_SP, 1);
        case TSAR_BLACK_REFINE:
            if ((rc = make_rng_table(ctx, seed))) return rc;
            return launch_checker(ctx, PM_MODE_PR, 0);
        case TSAR_RED_REFINE:
            if ((rc = make_rng_table(ctx, seed))) return rc;
            return launch_checker(ctx, PM_MODE_PR, 1);
    }
    FAIL(TSAR_ERR_ARG, "unknown launch kind");
}

int tsar_iterate(tsar_ctx *ctx, int iters, uint64_t seed0, const uint64_t *refine_seeds) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->have_planes) FAIL(TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
    // XORWOW row tables of ALL refinement launches of this loop in one launch (a single table occupies 5 % of the
    // GPU): 2*iters tables of H x pitch words, when that fits a 4 GB budget and the batch limit
    const size_t table_words = (size_t)ctx->rng_pitch * ctx->H;
    const int n_tables = 2 * iters;
    const bool batch = iters > 0 && n_tables <= kRngBatchMax && table_words * n_tables * 4 <= ((size_t)4 << 30);
    if (batch) {
        if (table_words * n_tables > ctx->rng_batch_alloc) {
            cudaFree(ctx->rng_batch); ctx->rng_batch = nullptr; ctx->rng_batch_alloc = 0;
            CK(cudaMalloc(&ctx->rng_batch, table_words * n_tables * 4));
            ctx->rng_batch_alloc = table_words * n_tables;
        }
        unsigned long long seeds[kRngBatchMax];
        for (int t = 0; t < n_tables; t++) seeds[t] = refine_seeds ? refine_seeds[t] : seed0 + 1 + (uint64_t)t;
        CK(pm_launch_rng_tables(ctx->rng_batch, table_words, n_tables, seeds, ctx->rng_pitch, ctx->H, ctx->rng_len, ctx->stream));
        ctx->launches++;
    }
    for (int it = 0; it < iters; it++) {
        for (int col = 0; col < 2; col++) {
            const uint64_t seed = refine_seeds ? refine_seeds[2 * it + col] : seed0 + 1 + 2 * (uint64_t)it + col;
            const uint32_t *table = batch ? ctx->rng_batch + table_words * (2 * it + col) : nullptr;
            if (ctx->fused) {
                // spatial propagation and refinement of one colour in ONE kernel: the refinement of a
                // pixel depends only on that pixel's own state after propagation
                if (!batch && (rc = make_rng_table(ctx, seed))) return rc;
                if ((rc = launch_checker(ctx, PM_MODE_FUSED, col, table))) return rc;
            } else {
                if ((rc = launch_checker(ctx, PM_MODE_SP, col))) return rc;
                if (!batch && (rc = make_rng_table(ctx, seed))) return rc;
                if ((rc = launch_checker(ctx, PM_MODE_PR, col, table))) return rc;
            }
        }
    }
    return TSAR_OK;
}

int tsar_eval_planes(tsar_ctx *ctx, int n, const int *xy, const float *planes, float *cost, int *beview, float *ratio) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (n <= 0 || !xy || !planes || !cost) FAIL(TSAR_ERR_ARG, "bad eval arguments");
    const size_t bytes = (size_t)n * (8 + 16 + 4 + 4 + 4);
    if ((rc = ensure_scratch(ctx, bytes))) return rc;
    unsigned char *base = (unsigned char *)ctx->scratch;
    float4 *dpl = (float4 *)base;
    int2 *dxy = (int2 *)(base + (size_t)n * 16);
    float *dc = (float *)(base + (size_t)n * 24);
    int *db = (int *)(base + (size_t)n * 28);
    float *dr = (float *)(base + (size_t)n * 32);
    CK(cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dpl, planes, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx->variant->eval(ctx->use_u8, ctx->eval_wrapper_rounding, ctx->pm, ctx->ref_img, n, dxy, dpl, dc, db, dr, ctx->stream));
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(cost, dc, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (beview) CK(cudaMemcpyAsync(beview, db, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (ratio) CK(cudaMemcpyAsync(ratio, dr, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

#define PX_GRID dim3 b(32, 8), g((ctx->W + 31) / 32, (ctx->H + 7) / 8)

int tsar_lrdiff(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    lrdiff_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->d_cams, ctx->d_tex, ctx->n_images, ctx->plane[0], ctx->cost[0],
                                            ctx->beview, ctx->lrdiff);
    ctx->launches++;
    CK(cudaGetLastError());
    return TSAR_OK;
}

int tsar_getview(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    getview_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0], ctx->cost[0], ctx->lrdiff, ctx->confid, ctx->depth);
    ctx->launches++;
    CK(cudaGetLastError());
    return TSAR_OK;
}

int tsar_get_disp(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    get_disp_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0], ctx->depth);
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_compute_disp(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    compute_disp_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0], ctx->cost[0]);
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->have_planes = false;   // buffer 0 now holds the OUTPUT layout (world normal, depth in w), not (n, d) planes
    return TSAR_OK;
}

int tsar_update_scale(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->region_text) FAIL(TSAR_ERR_STATE, "tsar_set_regions has not been called");
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    update_scale_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0], ctx->cost[0], ctx->scale, ctx->depth, ctx->canny,
                                                  ctx->region_text, ctx->region_plane, ctx->n_regions);
    ctx->launches++;
    CK(cudaGetLastError());
    return seed_alt_buffers(ctx);   // rows outside the checkerboard grid live in both buffers
}

int tsar_update_scale_2(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->region_text) FAIL(TSAR_ERR_STATE, "tsar_set_regions has not been called");
    PX_GRID;
    update_scale_2_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->fakedepth, ctx->canny, ctx->region_text,
                                                    ctx->region_plane, ctx->n_regions);
    ctx->launches++;
    CK(cudaGetLastError());
    return TSAR_OK;
}

int tsar_wmf(tsar_ctx *ctx, int iter) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (iter < 0 || iter > 3) FAIL(TSAR_ERR_ARG, "WMF level must be 0..3 (gipuma.cu:1809)");
    if ((rc = consolidate(ctx))) return rc;
    const size_t npx = (size_t)ctx->W * ctx->H;
    if ((rc = ensure_scratch(ctx, npx * 4))) return rc;
    const char *pt = getenv("TSAR_B200_WMF_PER_THREAD");
    rc = wmf_launch(ctx->glue, ctx->ref_img, ctx->plane[0], ctx->depth, ctx->scale, (float *)ctx->scratch, iter, pt && pt[0] == '1',
                    ctx->stream);
    ctx->launches++;
    CK(cudaGetLastError());
    return rc;
}

int tsar_wmf_final(tsar_ctx *ctx, int iter) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (iter < 0 || iter > 5) FAIL(TSAR_ERR_ARG, "WMF_Final level must be 0..5 (gipuma.cu:1844)");
    if (!ctx->region_text) FAIL(TSAR_ERR_STATE, "tsar_set_regions has not been called");
    if ((rc = consolidate(ctx))) return rc;
    const size_t npx = (size_t)ctx->W * ctx->H;
    if ((rc = ensure_scratch(ctx, npx * 24))) return rc;
    float4 *ps = (float4 *)ctx->scratch;
    float *ds = (float *)((unsigned char *)ctx->scratch + npx * 16), *ss = ds + npx;
    rc = wmf_final_launch(ctx->glue, ctx->ref_img, ctx->plane[0], ctx->depth, ctx->scale, ps, ds, ss, ctx->canny,
                          ctx->region_text, ctx->n_regions, iter, ctx->stream);
    ctx->launches++;
    CK(cudaGetLastError());
    if (rc) return rc;
    return seed_alt_buffers(ctx);
}

int tsar_set_regions(tsar_ctx *ctx, int n_regions, const float *text, const float *norm4) {
    if (!ctx || n_regions < 1 || !text || !norm4) return TSAR_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (n_regions > ctx->region_cap) {  // grow only: cudaFree/cudaMalloc synchronise the device
        cudaFree(ctx->region_text); cudaFree(ctx->region_plane);
        ctx->region_text = nullptr; ctx->region_plane = nullptr; ctx->region_cap = 0;
        CK(cudaMalloc(&ctx->region_text, (size_t)n_regions * 4));
        CK(cudaMalloc(&ctx->region_plane, (size_t)n_regions * 16));
        ctx->region_cap = n_regions;
    }
    CK(cudaMemcpyAsync(ctx->region_text, text, (size_t)n_regions * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->region_plane, norm4, (size_t)n_regions * 16, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_regions = n_regions;
    return TSAR_OK;
}

int tsar_set_labels_quarter(tsar_ctx *ctx, const int *labels, int wq, int hq) {
    if (!ctx || !labels) return TSAR_ERR_ARG;
    if (!ctx->have_views) FAIL(TSAR_ERR_STATE, "tsar_set_views has not been called");
    if (wq < 1 || hq < 1 || 4 * (wq + 1) < ctx->W || 4 * (hq + 1) < ctx->H || 4 * wq > ctx->W + 3 || 4 * hq > ctx->H + 3)
        FAIL(TSAR_ERR_ARG, "label map is not the quarter-resolution grid of the views");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_scratch(ctx, (size_t)wq * hq * 4);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->scratch, labels, (size_t)wq * hq * 4, cudaMemcpyHostToDevice, ctx->stream));
    dim3 b(32, 8), g((ctx->W + 31) / 32, (ctx->H + 7) / 8);
    labels_quarter_kernel<<<g, b, 0, ctx->stream>>>((const int *)ctx->scratch, wq, hq, ctx->W, ctx->H, ctx->canny);
    CK(cudaGetLastError());
    ctx->launches++;
    CK(cudaStreamSynchronize(ctx->stream));  // the caller's buffer may go away
    return TSAR_OK;
}

// Persistent device scratch of the region fit (grow-only: cudaMalloc / cudaFree synchronise the whole device and would
// stall the other pipelined context).
static int ensure_ransac(tsar_ctx *ctx, size_t n_px, int nt) {
    RansacScratch &r = ctx->ransac;
    const size_t nb = (n_px + 1023) / 1024;
    if (n_px > r.px_cap) {
        cudaFree(r.block_counts); cudaFree(r.list);
        r.block_counts = nullptr; r.list = nullptr; r.px_cap = 0;
        CK(cudaMalloc(&r.block_counts, nb * sizeof(int)));
        CK(cudaMalloc(&r.list, n_px * sizeof(int)));
        r.px_cap = n_px;
    }
    if (nt > r.nt_cap) {
        cudaFree(r.totals); cudaFree(r.pts); cudaFree(r.rnd); cudaFree(r.jobs); cudaFree(r.out); cudaFree(r.states);
        cudaFree(r.hyp_counts); cudaFree(r.regions);
        r.totals = nullptr; r.pts = nullptr; r.rnd = nullptr; r.jobs = nullptr; r.out = nullptr; r.states = nullptr;
        r.hyp_counts = nullptr; r.regions = nullptr; r.nt_cap = 0;
        const int cap = std::max(nt, 4);
        CK(cudaMalloc(&r.totals, (size_t)cap * sizeof(int)));
        CK(cudaMalloc(&r.pts, (size_t)cap * kRansacKeepAll * sizeof(float3)));
        CK(cudaMalloc(&r.rnd, (size_t)cap * kRansacRandPerRegion * sizeof(uint32_t)));
        CK(cudaMalloc(&r.jobs, (size_t)cap * sizeof(RansacJob)));
        CK(cudaMalloc(&r.out, (size_t)cap * sizeof(float4)));
        CK(cudaMalloc(&r.states, (size_t)cap * sizeof(RansacState)));
        CK(cudaMalloc(&r.hyp_counts, (size_t)cap * kRansacBatch * sizeof(int)));
        CK(cudaMalloc(&r.regions, (size_t)cap * sizeof(int)));
        CK(cudaMemsetAsync(r.hyp_counts, 0, (size_t)cap * kRansacBatch * sizeof(int), ctx->stream));  // the kernel leaves it zeroed
        r.nt_cap = cap;
    }
    if (r.grid == 0) {
        int sms = 148, per_sm = 0;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ransac_fit_kernel, kRansacSlice, 0));
        if (per_sm < 1) FAIL(TSAR_ERR_CUDA, "region-fit kernel does not fit on an SM");
        r.grid = sms * std::min(per_sm, 2);   // all CTAs must be co-resident (grid-wide barriers)
    }
    return TSAR_OK;
}

// rnd != nullptr: region-major host array, kRansacRandPerRegion values for EVERY region; else the device stream of `seed`
static int fit_region_planes(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                             const uint32_t *rnd, unsigned long long seed, float *region_norm4) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (n_regions < 1 || !region_text || !region_size || !region_norm4) FAIL(TSAR_ERR_ARG, "bad region arguments");
    std::vector<int> targets;
    for (int r = 0; r < n_regions; r++)
        if (region_text[r] == -1.0f) targets.push_back(r);
    if (targets.empty()) return TSAR_OK;
    const size_t n = (size_t)ctx->W * ctx->H;
    if (n > 0x7fffffffull) FAIL(TSAR_ERR_ARG, "image too large for 32-bit pixel indices");
    const int nb = (int)((n + 1023) / 1024), nt = (int)targets.size();
    if ((rc = ensure_ransac(ctx, n, nt))) return rc;
    RansacScratch &S = ctx->ransac;
    cudaStream_t st = ctx->stream;
    std::vector<RansacJob> jobs(nt);
    std::vector<float4> out(nt);
    for (int t = 0; t < nt; t++) {
        const int r = targets[t];
        jobs[t].pts = S.pts + (size_t)t * kRansacKeepAll;
        jobs[t].n = 0;
        jobs[t].size = region_size[r];
        jobs[t].rnd = S.rnd + (size_t)t * kRansacRandPerRegion;
        jobs[t].out = S.out + t;
        out[t] = make_float4(region_norm4[4 * r], region_norm4[4 * r + 1], region_norm4[4 * r + 2], region_norm4[4 * r + 3]);
    }
    // (pageable host sources: cudaMemcpyAsync returns once they are staged, so the vectors may go out of scope)
    CK(cudaMemcpyAsync(S.jobs, jobs.data(), (size_t)nt * sizeof(RansacJob), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(S.out, out.data(), (size_t)nt * sizeof(float4), cudaMemcpyHostToDevice, st));
    if (rnd) {
        for (int t = 0; t < nt; t++)
            CK(cudaMemcpyAsync(S.rnd + (size_t)t * kRansacRandPerRegion, rnd + (size_t)targets[t] * kRansacRandPerRegion,
                               (size_t)kRansacRandPerRegion * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    } else {
        CK(cudaMemcpyAsync(S.regions, targets.data(), (size_t)nt * sizeof(int), cudaMemcpyHostToDevice, st));
        ransac_rand_kernel<<<dim3((kRansacRandPerRegion + 255) / 256, nt), 256, 0, st>>>(S.rnd, S.regions, nt, kRansacRandPerRegion, seed);
        ctx->launches++;
    }
    // stable compaction of every target region's reliable pixels (raster order, as the reference collects them) and their
    // back-projection; list lengths stay on the device
    for (int t = 0; t < nt; t++) {
        const int r = targets[t];
        ransac_flag_kernel<<<nb, 1024, 0, st>>>(ctx->scale, ctx->canny, (int)n, r, S.block_counts);
        ransac_scan_blocks_kernel<<<1, 1024, 0, st>>>(S.block_counts, nb, S.totals + t);
        ransac_scatter_kernel<<<nb, 1024, 0, st>>>(ctx->scale, ctx->canny, (int)n, r, S.block_counts, S.list);
        ransac_points_kernel<<<(kRansacKeepAll + 255) / 256, 256, 0, st>>>(ctx->glue, ctx->depth, S.list, S.totals + t,
                                                                         S.pts + (size_t)t * kRansacKeepAll, S.jobs + t);
        ctx->launches += 4;
    }
    CK(cudaGetLastError());
    // the whole fit: one cooperative launch, loop termination on the device
    RansacFitArgs fa;
    fa.jobs = S.jobs; fa.states = S.states; fa.counts = S.hyp_counts; fa.n_jobs = nt;
    void *kargs[] = {&fa};
    CK(cudaLaunchCooperativeKernel((const void *)ransac_fit_kernel, dim3(S.grid), dim3(kRansacSlice), kargs, 0, st));
    ctx->launches++;
    CK(cudaMemcpyAsync(out.data(), S.out, (size_t)nt * sizeof(float4), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));   // the only host wait: the result
    for (int t = 0; t < nt; t++) {
        float *o = region_norm4 + 4 * targets[t];
        o[0] = out[t].x; o[1] = out[t].y; o[2] = out[t].z; o[3] = out[t].w;
    }
    return TSAR_OK;
}

int tsar_fit_region_planes(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                           const uint32_t *rnd, float *region_norm4) {
    if (!ctx) return TSAR_ERR_ARG;
    if (!rnd) FAIL(TSAR_ERR_ARG, "rnd is null (use tsar_fit_region_planes_seeded for a device-generated stream)");
    return fit_region_planes(ctx, n_regions, region_text, region_size, rnd, 0ull, region_norm4);
}

int tsar_fit_region_planes_seeded(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                                  uint64_t seed, float *region_norm4) {
    if (!ctx) return TSAR_ERR_ARG;
    return fit_region_planes(ctx, n_regions, region_text, region_size, nullptr, (unsigned long long)seed, region_norm4);
}

uint32_t tsar_ransac_rand_value(uint64_t seed, int region, int index) { return ransac_rand_value((unsigned long long)seed, region, index); }

int tsar_scale_from_confidence(tsar_ctx *ctx, float threshold) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    const size_t n = (size_t)ctx->W * ctx->H;
    scale_from_confidence_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->confid, threshold, ctx->scale, n);
    ctx->launches++;
    CK(cudaGetLastError());
    return TSAR_OK;
}

int tsar_scale_from_weak_png(tsar_ctx *ctx, const unsigned char *bgr) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!bgr) FAIL(TSAR_ERR_ARG, "weak.png pixels are null");
    const size_t n = (size_t)ctx->W * ctx->H;
    if ((rc = ensure_scratch(ctx, n * 3))) return rc;
    CK(cudaMemcpyAsync(ctx->scratch, bgr, n * 3, cudaMemcpyHostToDevice, ctx->stream));
    scale_from_weak_png_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((const uchar3 *)ctx->scratch, ctx->scale, n);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));  // the caller's buffer may go away
    return TSAR_OK;
}

int tsar_download_outputs(tsar_ctx *ctx, float *depth_out, float *normals_out, float *confid_out) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    const size_t n = (size_t)ctx->W * ctx->H;
    if (depth_out || normals_out) {
        if ((rc = ensure_scratch(ctx, n * 16))) return rc;
        float *d = (float *)ctx->scratch, *nr = d + n;
        split_outputs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->plane[0], d, nr, n);
        ctx->launches++;
        CK(cudaGetLastError());
        if (depth_out) CK(cudaMemcpyAsync(depth_out, d, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (normals_out) CK(cudaMemcpyAsync(normals_out, nr, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (confid_out) CK(cudaMemcpyAsync(confid_out, ctx->confid, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_ransac_rand_per_region(void) { return kRansacRandPerRegion; }

static void *field_ptr(tsar_ctx *ctx, int field, size_t *elt, size_t *count) {
    *count = (size_t)ctx->W * ctx->H;
    *elt = 4;
    switch (field) {
        case TSAR_F_NORM4: *elt = 16; return ctx->plane[0];
        case TSAR_F_COST: return ctx->cost[0];
        case TSAR_F_DEPTH: return ctx->depth;
        case TSAR_F_FAKEDEPTH: return ctx->fakedepth;
        case TSAR_F_SCALE: return ctx->scale;
        case TSAR_F_CANNY: return ctx->canny;
        case TSAR_F_RATIO: return ctx->ratio;
        case TSAR_F_BEVIEW: return ctx->beview;
        case TSAR_F_LRDIFF: return ctx->lrdiff;
        case TSAR_F_CONFID: return ctx->confid;
        case TSAR_F_REGION_TEXT: *count = ctx->n_regions; return ctx->region_text;
        case TSAR_F_REGION_NORM4: *count = ctx->n_regions; *elt = 16; return ctx->region_plane;
    }
    return nullptr;
}

int tsar_upload(tsar_ctx *ctx, int field, const void *src, size_t bytes) {
    if (!ctx || !src) return TSAR_ERR_ARG;
    if (!ctx->have_views) FAIL(TSAR_ERR_STATE, "tsar_set_views has not been called");
    CK(cudaSetDevice(ctx->device));
    if (field == TSAR_F_NORM4 || field == TSAR_F_COST) {
        int rc = consolidate(ctx);
        if (rc) return rc;
    }
    size_t elt, count;
    void *p = field_ptr(ctx, field, &elt, &count);
    if (!p || bytes != elt * count) FAIL(TSAR_ERR_ARG, "field/size mismatch");
    CK(cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (field == TSAR_F_NORM4) {
        ctx->have_planes = true;
        return seed_alt_buffers(ctx);
    }
    if (field == TSAR_F_COST) return seed_alt_buffers(ctx);
    return TSAR_OK;
}

int tsar_download(tsar_ctx *ctx, int field, void *dst, size_t bytes) {
    if (!ctx || !dst) return TSAR_ERR_ARG;
    if (!ctx->have_views) FAIL(TSAR_ERR_STATE, "tsar_set_views has not been called");
    CK(cudaSetDevice(ctx->device));
    if (field == TSAR_F_NORM4 || field == TSAR_F_COST) {
        int rc = consolidate(ctx);
        if (rc) return rc;
    }
    size_t elt, count;
    void *p = field_ptr(ctx, field, &elt, &count);
    if (!p || bytes != elt * count) FAIL(TSAR_ERR_ARG, "field/size mismatch");
    CK(cudaMemcpyAsync(dst, p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_device_ptr(tsar_ctx *ctx, int field, void **dev_ptr) {
    if (!ctx || !dev_ptr) return TSAR_ERR_ARG;
    if (!ctx->have_views) FAIL(TSAR_ERR_STATE, "tsar_set_views has not been called");
    CK(cudaSetDevice(ctx->device));
    if (field == TSAR_F_NORM4 || field == TSAR_F_COST) {
        int rc = consolidate(ctx);
        if (rc) return rc;
    }
    size_t elt, count;
    *dev_ptr = field_ptr(ctx, field, &elt, &count);
    return *dev_ptr ? TSAR_OK : TSAR_ERR_ARG;
}

int tsar_depthmap(tsar_ctx *ctx, uint64_t seed0, float *ms_out) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if ((rc = tsar_init_planes(ctx, seed0))) return rc;
    if ((rc = tsar_iterate(ctx, ctx->params.iterations, seed0, nullptr))) return rc;
    if ((rc = tsar_lrdiff(ctx))) return rc;
    if ((rc = tsar_getview(ctx))) return rc;
    if ((rc = tsar_compute_disp(ctx))) return rc;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (ms_out) {
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    }
    return TSAR_OK;
}

int tsar_depthmap_host(tsar_ctx *ctx, int W, int H, int n_images, const float *const *images, const tsar_camera *cams,
                       float cam_f, const int *subset, int V, const tsar_params *p, uint64_t seed0, float *norm4_out,
                       float *confid_out) {
    int rc;
    if ((rc = tsar_set_views(ctx, W, H, n_images, images, 0, cams, cam_f, subset, V))) return rc;
    if ((rc = tsar_set_params(ctx, p))) return rc;
    if ((rc = tsar_depthmap(ctx, seed0, nullptr))) return rc;
    const size_t n = (size_t)W * H;
    if (norm4_out) CK(cudaMemcpyAsync(norm4_out, ctx->plane[0], n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (confid_out) CK(cudaMemcpyAsync(confid_out, ctx->confid, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_slic(tsar_ctx *ctx, const unsigned char *bgrx, const tsar_slic_settings *s, int *labels_out) {
    if (!ctx || !bgrx || !s || !labels_out) return TSAR_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    int nl = 0;
    const char *msg = slic_run(ctx->slic, bgrx, *s, labels_out, ctx->stream, &nl);
    ctx->launches += nl;
    if (msg) FAIL(TSAR_ERR_CUDA, msg);
    return TSAR_OK;
}

// debug: the superpixel records of the last tsar_slic call (8 words each: centre x, y, colour x, y, z, w, id, no_pixels,
// the layout of gSLICr::objects::spixel_info), for stage-by-stage comparison with the reference engine
int tsar_dbg_slic_centres(tsar_ctx *ctx, float *out, int max_records, int *n_records) {
    if (!ctx || !n_records) return TSAR_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->slic.last_nsp;
    *n_records = n;
    const int m = n < max_records ? n : max_records;
    if (out && m > 0) {
        std::vector<SpixelInfo> host(m);   // the device record is 48 bytes (float4 alignment); the reference's is 32
        CK(cudaMemcpyAsync(host.data(), ctx->slic.d_sp, (size_t)m * sizeof(SpixelInfo), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < m; i++) {
            float *o = out + 8 * (size_t)i;
            o[0] = host[i].cx; o[1] = host[i].cy;
            o[2] = host[i].color.x; o[3] = host[i].color.y; o[4] = host[i].color.z; o[5] = host[i].color.w;
            memcpy(o + 6, &host[i].id, 4); memcpy(o + 7, &host[i].no_pixels, 4);
        }
    }
    return TSAR_OK;
}

// debug: the CIELAB image of the last tsar_slic call (4 floats per pixel)
int tsar_dbg_slic_lab(tsar_ctx *ctx, float *out, size_t n_pixels) {
    if (!ctx || !out) return TSAR_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (n_pixels > (size_t)ctx->slic.cap_px || !ctx->slic.d_lab) FAIL(TSAR_ERR_ARG, "no Lab image of that size (run tsar_slic first)");
    CK(cudaMemcpyAsync(out, ctx->slic.d_lab, n_pixels * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_launch_count(tsar_ctx *ctx, long long *count, int reset) {
    if (!ctx || !count) return TSAR_ERR_ARG;
    *count = ctx->launches;
    if (reset) ctx->launches = 0;
    return TSAR_OK;
}

int tsar_eval_count(tsar_ctx *ctx, int iters, long long *n_evals) {
    if (!ctx || !n_evals) return TSAR_ERR_ARG;
    if (!ctx->have_views || !ctx->have_params) FAIL(TSAR_ERR_STATE, "views/params not set");
    const int W = ctx->W, H = ctx->H, yl = ctx->pm.y_limit;
    int R = 0;
    for (float dz = ctx->params.max_disparity * 0.5f; dz >= 0.01f; dz = dz / 10.0f) R++;
    long long sx = 0, sy = 0;  // direction tests passing their border guards (gipuma.cu:889-1022)
    for (int x = 0; x < W; x++) sx += (x > 2) + (x < W - 3) + (x > 0) + (x < W - 1);
    for (int y = 0; y < yl; y++) sy += (y > 2) + (y < H - 3) + (y > 0) + (y < H - 1);
    const long long prop = (long long)yl * sx + (long long)W * sy;
    const long long refine = (long long)W * yl * R;
    *n_evals = (long long)ctx->V * ((long long)W * H + (long long)iters * (prop + refine));
    return TSAR_OK;
}

// ---- instrumentation (see include/tsar_b200.h) ------------------------------------------------
int tsar_dbg_tex_sample(tsar_ctx *ctx, int image, int n, const float *xy, float *out) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (image < 0 || image >= ctx->n_images || n <= 0 || !xy || !out) FAIL(TSAR_ERR_ARG, "bad sample arguments");
    if ((rc = ensure_scratch(ctx, (size_t)n * 12))) return rc;
    float2 *dxy = (float2 *)ctx->scratch;
    float *dout = (float *)((unsigned char *)ctx->scratch + (size_t)n * 8);
    CK(cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    dbg_tex_sample_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->tex[image], n, dxy, dout);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_profile(tsar_ctx *ctx, int enable) {
    if (!ctx) return TSAR_ERR_ARG;
    ctx->profiling = enable != 0;
    return TSAR_OK;
}

int tsar_profile_read(tsar_ctx *ctx, float *checker_ms_total, int *n_launches) {
    if (!ctx || !checker_ms_total || !n_launches) return TSAR_ERR_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    float tot = 0.f;
    for (auto &pr : ctx->prof_events) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, pr.first, pr.second));
        tot += ms;
        cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
    }
    *checker_ms_total = tot;
    *n_launches = (int)ctx->prof_events.size();
    ctx->prof_events.clear();
    return TSAR_OK;
}

int tsar_profile_read_launches(tsar_ctx *ctx, float *ms, int cap, int *n_launches) {
    if (!ctx || !n_launches || cap < 0 || (cap > 0 && !ms)) return TSAR_ERR_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    int n = 0;
    for (auto &pr : ctx->prof_events) {
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, pr.first, pr.second));
        if (n < cap) ms[n] = t;
        n++;
        cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
    }
    *n_launches = n;
    ctx->prof_events.clear();
    return TSAR_OK;
}

int tsar_dbg_candidate_stats(tsar_ctx *ctx, int colour, unsigned long long *out) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!out || colour < 0 || colour > 1) FAIL(TSAR_ERR_ARG, "bad candidate-statistics arguments");
    if (!ctx->have_planes) FAIL(TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
    if ((rc = ensure_scratch(ctx, kCandStatWords * sizeof(unsigned long long)))) return rc;
    CheckerArgs a{};
    for (int col = 0; col < 2; col++) { a.plane_in[col] = ctx->plane[ctx->cur[col]]; a.cost_in[col] = ctx->cost[ctx->cur[col]]; }
    a.colour = colour;
    CK(cudaMemsetAsync(ctx->scratch, 0, kCandStatWords * sizeof(unsigned long long), ctx->stream));
    CK(pm_launch_cand_stats(ctx->pm, a, (unsigned long long *)ctx->scratch, ctx->stream));
    ctx->launches++;
    CK(cudaMemcpyAsync(out, ctx->scratch, kCandStatWords * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_dbg_eval_rounding(tsar_ctx *ctx, int wrapper_rounding) {
    if (!ctx) return TSAR_ERR_ARG;
    ctx->eval_wrapper_rounding = wrapper_rounding ? 1 : 0;
    return TSAR_OK;
}

int tsar_dbg_quad_sampling(tsar_ctx *ctx, int checker_launches) {
    if (!ctx) return TSAR_ERR_ARG;
    ctx->quad_launches = checker_launches < 0 ? -1 : checker_launches;
    return TSAR_OK;
}

// Experiment: the same image as 8-bit (normalised-float read), 16-bit unorm and fp16 textures; samples at the given
// coordinates and bilinear-fetch throughput per format.  out = 4 arrays of n floats (f32, u8, u16, f16 texels),
// rate4 = Gsamples/s per format with a warp-local access pattern.
int tsar_dbg_tex_formats(tsar_ctx *ctx, int image, int n, const float *xy, float *out, float *rate4) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    const int W = ctx->W, H = ctx->H;
    std::vector<float> host((size_t)W * H);
    CK(cudaMemcpy2DFromArray(host.data(), (size_t)W * 4, ctx->arrays[image], 0, 0, (size_t)W * 4, H, cudaMemcpyDeviceToHost));
    std::vector<unsigned char> h8((size_t)W * H);
    std::vector<unsigned short> h16((size_t)W * H), hf16((size_t)W * H);
    for (size_t i = 0; i < host.size(); i++) {
        h8[i] = (unsigned char)host[i];
        h16[i] = (unsigned short)(host[i] * 257.0f);
        hf16[i] = __half_as_ushort(__float2half(host[i]));
    }
    cudaTextureObject_t tex[4];
    cudaArray_t arr[3];
    tex[0] = ctx->tex[image];
    cudaChannelFormatDesc cds[3] = {cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned),
                                    cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindUnsigned),
                                    cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindFloat)};
    const void *srcs[3] = {h8.data(), h16.data(), hf16.data()};
    const size_t esz[3] = {1, 2, 2};
    for (int k = 0; k < 3; k++) {
        CK(cudaMallocArray(&arr[k], &cds[k], W, H));
        CK(cudaMemcpy2DToArray(arr[k], 0, 0, srcs[k], W * esz[k], W * esz[k], H, cudaMemcpyHostToDevice));
        cudaResourceDesc rd; memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeArray; rd.res.array.array = arr[k];
        cudaTextureDesc td; memset(&td, 0, sizeof(td));
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModeLinear;
        td.readMode = (k < 2) ? cudaReadModeNormalizedFloat : cudaReadModeElementType;
        td.normalizedCoords = 0;
        CK(cudaCreateTextureObject(&tex[k + 1], &rd, &td, NULL));
    }
    if ((rc = ensure_scratch(ctx, (size_t)n * 12))) return rc;
    float2 *dxy = (float2 *)ctx->scratch;
    float *dout = (float *)((unsigned char *)ctx->scratch + (size_t)n * 8);
    CK(cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    for (int k = 0; k < 4; k++) {
        dbg_tex_sample_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(tex[k], n, dxy, dout);
        CK(cudaMemcpyAsync(out + (size_t)k * n, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        float best = 0.f;
        for (int rep = 0; rep < 3; rep++) {
            float ms;
            CK(cudaEventRecord(ctx->ev0, ctx->stream));
            dbg_tex_kernel<<<sms * 8, 256, 0, ctx->stream>>>(tex[k], dout, 256, W, H);
            CK(cudaEventRecord(ctx->ev1, ctx->stream));
            CK(cudaEventSynchronize(ctx->ev1));
            CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
            best = std::max(best, (float)((double)sms * 8 * 256 * 256 * 4 / (ms * 1e-3) / 1e9));
        }
        rate4[k] = best;
    }
    for (int k = 0; k < 3; k++) { cudaDestroyTextureObject(tex[k + 1]); cudaFreeArray(arr[k]); }
    return TSAR_OK;
}

int tsar_dbg_peaks(tsar_ctx *ctx, float *out3) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!out3) return TSAR_ERR_ARG;
    if ((rc = ensure_scratch(ctx, 64))) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    const int blocks = sms * 8, threads = 256, iters = 4096;
    float best[3] = {0, 0, 0};
    for (int rep = 0; rep < 4; rep++) {
        float ms;
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_ffma_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)ctx->scratch, iters, 1.0000001f, 1e-9f);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[0] = std::max(best[0], (float)((double)blocks * threads * iters * 8 * 8 * 2 / (ms * 1e-3) / 1e12));
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_mufu_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)ctx->scratch, iters / 4);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[1] = std::max(best[1], (float)((double)blocks * threads * (iters / 4) * 8 * 8 / (ms * 1e-3) / 1e9));
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_tex_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->tex[0], (float *)ctx->scratch, iters / 16, ctx->W, ctx->H);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[2] = std::max(best[2], (float)((double)blocks * threads * (iters / 16) * 4 / (ms * 1e-3) / 1e9));
    }
    out3[0] = best[0];  // TFLOP/s FP32 FFMA
    out3[1] = best[1];  // G MUFU ops / s
    out3[2] = best[2];  // G bilinear fp32 texture samples / s
    return TSAR_OK;
}

}  // extern "C"
