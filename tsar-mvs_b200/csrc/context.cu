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
#include <memory>
#include <string>
#include <vector>

#include "../../include/tsar_b200.h"
#include "debug_kernels.cuh"
#include "dev_mem.h"
#include "glue_kernels.cuh"
#include "pm_launch.h"
#include "ransac_kernels.cuh"
#include "slic_kernels.cuh"
#include "wmf_kernels.cuh"

using namespace tsar;

struct RansacScratch {
    DeviceBuf<int> block_counts, list, totals, hyp_counts, regions;
    DeviceBuf<float3> pts;
    DeviceBuf<uint32_t> rnd;
    DeviceBuf<RansacJob> jobs;
    DeviceBuf<float4> out;
    DeviceBuf<RansacState> states;
    int grid = 0;
};

// Checkerboard launches after the planes were set that use quad-cooperative sampling (the rest use the per-lane
// loop).  Chosen by measurement, DESIGN.md 4.4.
constexpr int kQuadLaunches = 2;

struct tsar_ctx : HandleCore {
    int W = 0, H = 0, n_images = 0, V = 0;
    bool have_views = false, have_params = false, have_planes = false;
    std::vector<tsar_camera> cams;
    float cam_f = 0.f;
    std::vector<int> subset;
    tsar_params params{};
    // images
    std::vector<Texture2D> tex;
    std::vector<Texture2D> tex8;               // 8-bit copies of the views (sampling fast path)
    DeviceBuf<unsigned char> stage8;           // staging buffer for the float -> u8 conversion
    DeviceBuf<float> stage32;                  // linear landing buffer for host images (tsar_set_views, on_device = 0)
    DeviceBuf<int> d_flag;
    int use_u8 = 0;                            // every image is 8-bit valued: sample the 8-bit textures
    bool allow_u8 = true;                      // env TSAR_B200_NO_U8=1 switches the fast path off
    bool u8_verified = false, u8_ok = false;   // one-time self-check of the 8-bit sampling identity (tsar_set_views)
    int arr_w = 0, arr_h = 0;
    DeviceBuf<float> ref_img;
    DeviceBuf<cudaTextureObject_t> d_tex;
    DeviceBuf<CamDev> d_cams;
    // per-pixel state
    DeviceBuf<float4> plane[2];
    DeviceBuf<float> cost[2];
    int cur[2] = {0, 0};  // buffer holding the live values of colour 0 (black) / 1 (red)
    DeviceBuf<float> depth, fakedepth, scale, canny, ratio, lrdiff, confid;
    DeviceBuf<int> beview;
    DeviceBuf<float> region_text;
    DeviceBuf<float4> region_plane;
    int n_regions = 0;
    DeviceBuf<uint32_t> rng;
    DeviceBuf<uint32_t> rng_batch;             // tables of all refinement launches of one tsar_iterate call
    int rng_pitch = 0, rng_len = 0;
    // one scratch buffer, carved up differently by the entry points that need one
    DeviceBuf<unsigned char> scratch;
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
        c.tex[i] = ctx->tex[id].tex();
        c.tex8[i] = ctx->use_u8 ? ctx->tex8[id].tex() : 0;
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
        TSAR_FAIL(ctx, TSAR_ERR_ARG, "window too large for the shared-memory weight table");
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

// The per-pixel state grows all together, and only when W * H does.
static int ensure_state(tsar_ctx *ctx, size_t n) {
    for (int b = 0; b < 2; b++) {
        TSAR_CK(ctx, ctx->plane[b].reserve(n));
        TSAR_CK(ctx, ctx->cost[b].reserve(n));
    }
    for (DeviceBuf<float> *p : {&ctx->depth, &ctx->fakedepth, &ctx->scale, &ctx->canny, &ctx->ratio, &ctx->lrdiff,
                                &ctx->confid, &ctx->ref_img})
        TSAR_CK(ctx, p->reserve(n));
    TSAR_CK(ctx, ctx->beview.reserve(n));
    return TSAR_OK;
}

// LineState::resize memsets every array to 0 (linestate.h:73-109).  caller_inputs: also clear the arrays the
// caller fills between the entry points (canny labels, reliable flags); a new view clears them, a re-run of
// the PatchMatch path on the same view keeps them.
static int zero_state(tsar_ctx *ctx, bool caller_inputs) {
    const size_t n = (size_t)ctx->W * ctx->H;
    cudaStream_t s = ctx->stream;
    for (int b = 0; b < 2; b++) { TSAR_CK(ctx, cudaMemsetAsync(ctx->plane[b].get(), 0, n * 16, s)); TSAR_CK(ctx, cudaMemsetAsync(ctx->cost[b].get(), 0, n * 4, s)); }
    TSAR_CK(ctx, cudaMemsetAsync(ctx->depth.get(), 0, n * 4, s)); TSAR_CK(ctx, cudaMemsetAsync(ctx->fakedepth.get(), 0, n * 4, s));
    if (caller_inputs) { TSAR_CK(ctx, cudaMemsetAsync(ctx->scale.get(), 0, n * 4, s)); TSAR_CK(ctx, cudaMemsetAsync(ctx->canny.get(), 0, n * 4, s)); }
    TSAR_CK(ctx, cudaMemsetAsync(ctx->ratio.get(), 0, n * 4, s)); TSAR_CK(ctx, cudaMemsetAsync(ctx->lrdiff.get(), 0, n * 4, s));
    TSAR_CK(ctx, cudaMemsetAsync(ctx->confid.get(), 0, n * 4, s)); TSAR_CK(ctx, cudaMemsetAsync(ctx->beview.get(), 0, n * 4, s));
    ctx->cur[0] = ctx->cur[1] = 0;
    return TSAR_OK;
}

static int need_ready(tsar_ctx *ctx) {
    if (!ctx) return TSAR_ERR_ARG;
    if (!ctx->have_views) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_views has not been called");
    if (!ctx->have_params) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_params has not been called");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    return TSAR_OK;
}

// both colours back into buffer 0
static int consolidate(tsar_ctx *ctx) {
    for (int col = 0; col < 2; col++)
        if (ctx->cur[col] != 0) {
            TSAR_CK(ctx, pm_launch_merge_colour(ctx->W, ctx->H, col, ctx->plane[1].get(), ctx->cost[1].get(), ctx->plane[0].get(), ctx->cost[0].get(),
                                      ctx->stream));
            ctx->launches++;
            ctx->cur[col] = 0;
        }
    return TSAR_OK;
}

static int make_rng_table(tsar_ctx *ctx, uint64_t seed) {
    TSAR_CK(ctx, pm_launch_rng_table(ctx->rng.get(), ctx->rng_pitch, ctx->H, ctx->rng_len, seed, ctx->stream));
    ctx->launches++;
    return TSAR_OK;
}

static int launch_checker(tsar_ctx *ctx, int mode, int colour, const uint32_t *rng_table = nullptr) {
    CheckerArgs a;
    for (int col = 0; col < 2; col++) { a.plane_in[col] = ctx->plane[ctx->cur[col]].get(); a.cost_in[col] = ctx->cost[ctx->cur[col]].get(); }
    const bool sp = (mode & PM_MODE_SP) != 0;
    const int out = sp ? (ctx->cur[colour] ^ 1) : ctx->cur[colour];
    a.plane_out = ctx->plane[out].get();
    a.cost_out = ctx->cost[out].get();
    a.ratio = ctx->ratio.get();
    a.beview = ctx->beview.get();
    a.rng = rng_table ? rng_table : ctx->rng.get();
    a.colour = colour;
    cudaEvent_t p0 = nullptr, p1 = nullptr;
    if (ctx->profiling) {
        TSAR_CK(ctx, cudaEventCreate(&p0)); TSAR_CK(ctx, cudaEventCreate(&p1));
        TSAR_CK(ctx, cudaEventRecord(p0, ctx->stream));
    }
    const int quad = ctx->checker_since_planes < ctx->quad_launches && ctx->variant->has_quad && ctx->use_u8 && ctx->pm.k_pinhole;
    TSAR_CK(ctx, ctx->variant->checker(ctx->use_u8, quad, mode, ctx->pm, ctx->ref_img.get(), a, ctx->stream));
    ctx->checker_since_planes++;
    if (ctx->profiling) {
        TSAR_CK(ctx, cudaEventRecord(p1, ctx->stream));
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
        TSAR_CK(ctx, cudaMemcpyAsync(ctx->plane[1].get(), ctx->plane[0].get(), n * 16, cudaMemcpyDeviceToDevice, ctx->stream));
        TSAR_CK(ctx, cudaMemcpyAsync(ctx->cost[1].get(), ctx->cost[0].get(), n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
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
    std::unique_ptr<tsar_ctx> ctx(new tsar_ctx);
    if (int rc = ctx->open(device, stream)) return rc;
    cudaEventCreate(&ctx->ev0);
    cudaEventCreate(&ctx->ev1);
    const char *uf = getenv("TSAR_B200_UNFUSED");
    ctx->fused = !(uf && uf[0] == '1');
    const char *n8 = getenv("TSAR_B200_NO_U8");
    ctx->allow_u8 = !(n8 && n8[0] == '1');
    const char *nq = getenv("TSAR_B200_NO_QUAD_SAMPLING");
    if (nq && nq[0] == '1') ctx->quad_launches = -1;
    *out = ctx.release();
    return TSAR_OK;
}

int tsar_destroy(tsar_ctx *ctx) {
    if (!ctx) return TSAR_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &pr : ctx->prof_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    delete ctx;
    return TSAR_OK;
}

const char *tsar_last_error(const tsar_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tsar_sync(tsar_ctx *ctx) {
    if (!ctx) return TSAR_ERR_ARG;
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_set_views(tsar_ctx *ctx, int W, int H, int n_images, const float *const *images, int on_device,
                   const tsar_camera *cams, float cam_f, const int *subset, int V) {
    if (!ctx) return TSAR_ERR_ARG;
    if (W <= 0 || H <= 0 || n_images < 1 || n_images > 512 || !images || !cams) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad view arguments");
    if (V < 1 || V > TSAR_MAX_VIEWS || !subset) TSAR_FAIL(ctx, TSAR_ERR_ARG, "number of selected views must be in [1, 32] (pmCostMultiview_cu costVector[32])");
    for (int i = 0; i < V; i++)
        if (subset[i] < 0 || subset[i] >= n_images) TSAR_FAIL(ctx, TSAR_ERR_ARG, "view subset index out of range");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)W * H;
    int rc = ensure_state(ctx, n);
    if (rc) return rc;
    // textures: same descriptor as addImageToTextureFloatGray (main.cpp:1190-1228): float, linear
    // filter, unnormalised coordinates, address mode "wrap" (which the hardware treats as clamp for
    // unnormalised coordinates, SURVEY Q9) -- identical descriptor => identical sampling
    if (ctx->arr_w != W || ctx->arr_h != H || (int)ctx->tex.size() != n_images) {
        ctx->tex.clear();
        ctx->tex8.clear();
        ctx->arr_w = ctx->arr_h = 0;
        const cudaChannelFormatDesc cd = cudaCreateChannelDesc(32, 0, 0, 0, cudaChannelFormatKindFloat);
        std::vector<cudaTextureObject_t> handles;
        for (int i = 0; i < n_images; i++) {
            ctx->tex.emplace_back();
            TSAR_CK(ctx, ctx->tex.back().create(W, H, cd, cudaAddressModeWrap, cudaReadModeElementType));
            handles.push_back(ctx->tex.back().tex());
        }
        TSAR_CK(ctx, ctx->d_tex.reserve(n_images));
        TSAR_CK(ctx, ctx->d_cams.reserve(n_images));
        TSAR_CK(ctx, cudaMemcpyAsync(ctx->d_tex.get(), handles.data(), n_images * sizeof(cudaTextureObject_t), cudaMemcpyHostToDevice, ctx->stream));
        ctx->arr_w = W; ctx->arr_h = H;
    }
    // 8-bit copies: the reference's inputs are 8-bit grey images converted to float (main.cpp:1423), for which an
    // 8-bit texture gives bit-identical bilinear samples at a quarter of the texel traffic (pm_core.cuh, view_cost)
    ctx->use_u8 = 0;
    if (ctx->allow_u8 && (int)ctx->tex8.size() != n_images) {
        ctx->tex8.clear();
        const cudaChannelFormatDesc c8 = cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned);
        for (int i = 0; i < n_images; i++) {
            ctx->tex8.emplace_back();
            TSAR_CK(ctx, ctx->tex8.back().create(W, H, c8, cudaAddressModeClamp, cudaReadModeNormalizedFloat));
        }
    }
    if (ctx->allow_u8) TSAR_CK(ctx, ctx->stage8.reserve(n));
    TSAR_CK(ctx, ctx->d_flag.reserve(2));
    // host images cross the bus once, into a persistent linear staging buffer (no allocation per call: allocating and
    // freeing synchronise the whole device and would serialise contexts that pipeline views on other streams)
    if (!on_device) TSAR_CK(ctx, ctx->stage32.reserve(n));
    TSAR_CK(ctx, cudaMemsetAsync(ctx->d_flag.get(), 0, 2 * sizeof(int), ctx->stream));
    for (int i = 0; i < n_images; i++) {
        const float *src = images[i];
        if (!on_device) {
            float *dst = (i == 0) ? ctx->ref_img.get() : ctx->stage32.get();   // view 0 is also kept linear (hoisted window terms)
            TSAR_CK(ctx, cudaMemcpyAsync(dst, images[i], n * 4, cudaMemcpyHostToDevice, ctx->stream));
            src = dst;
        } else if (i == 0) {
            TSAR_CK(ctx, cudaMemcpyAsync(ctx->ref_img.get(), images[0], n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        TSAR_CK(ctx, cudaMemcpy2DToArrayAsync(ctx->tex[i].array(), 0, 0, src, (size_t)W * 4, (size_t)W * 4, H, cudaMemcpyDeviceToDevice, ctx->stream));
        if (ctx->allow_u8) {
            to_u8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(src, ctx->stage8.get(), n, ctx->d_flag.get());
            TSAR_CK(ctx, cudaMemcpy2DToArrayAsync(ctx->tex8[i].array(), 0, 0, ctx->stage8.get(), (size_t)W, (size_t)W, H, cudaMemcpyDeviceToDevice, ctx->stream));
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
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->d_cams.get(), cd.data(), n_images * sizeof(CamDev), cudaMemcpyHostToDevice, ctx->stream));
    // The 8-bit fast path rests on how the texture unit quantises its bilinear weights (pm_core.cuh, view_cost): checked
    // once per context on this device and driver, on the reference image incl. its borders, against the fp32 texture.
    int *flags = ctx->d_flag.get();   // [0] some image is not 8-bit valued, [1] mismatches of the self-check
    const bool check = ctx->allow_u8 && !ctx->u8_verified;
    if (check) {
        u8_selfcheck_kernel<<<16, 256, 0, ctx->stream>>>(ctx->tex[0].tex(), ctx->tex8[0].tex(), W, H, flags + 1);
        ctx->launches++;
    }
    int host_flags[2] = {1, 0};
    if (ctx->allow_u8) TSAR_CK(ctx, cudaMemcpyAsync(host_flags, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));  // one wait per call: the flags are needed now, and cd / the caller's buffers may go away
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
    TSAR_CK(ctx, ctx->rng.reserve(need));
    ctx->have_views = true;
    ctx->have_planes = false;
    rc = zero_state(ctx, true);
    if (rc) return rc;
    return rebuild_constants(ctx);
}

int tsar_set_params(tsar_ctx *ctx, const tsar_params *p) {
    if (!ctx || !p) return TSAR_ERR_ARG;
    if (p->box_hsize < 1 || p->box_vsize < 1 || p->n_best < 1) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad window / n_best");
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
    TSAR_CK(ctx, ctx->variant_init->init(ctx->use_u8, quad, ctx->pm_init, ctx->ref_img.get(), ctx->rng.get(), ctx->rng_len, ctx->plane[0].get(), ctx->cost[0].get(), ctx->stream));
    ctx->launches++;
    ctx->checker_since_planes = 0;
    ctx->cur[0] = ctx->cur[1] = 0;
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_load_planes(tsar_ctx *ctx, const float *norm4, const float *cost) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!norm4) TSAR_FAIL(ctx, TSAR_ERR_ARG, "norm4 is null");
    const size_t n = (size_t)ctx->W * ctx->H;
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->plane[0].get(), norm4, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    if (cost) TSAR_CK(ctx, cudaMemcpyAsync(ctx->cost[0].get(), cost, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    else {
        TSAR_CK(ctx, ctx->variant->cost_of_state(ctx->use_u8, ctx->pm, ctx->ref_img.get(), ctx->plane[0].get(), ctx->cost[0].get(), ctx->stream));
        ctx->launches++;
    }
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->checker_since_planes = 0;
    ctx->cur[0] = ctx->cur[1] = 0;
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_launch(tsar_ctx *ctx, int kind, uint64_t seed) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->have_planes) TSAR_FAIL(ctx, TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
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
    TSAR_FAIL(ctx, TSAR_ERR_ARG, "unknown launch kind");
}

int tsar_iterate(tsar_ctx *ctx, int iters, uint64_t seed0, const uint64_t *refine_seeds) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->have_planes) TSAR_FAIL(ctx, TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
    // XORWOW row tables of ALL refinement launches of this loop in one launch (a single table occupies 5 % of the
    // GPU): 2*iters tables of H x pitch words, when that fits a 4 GB budget and the batch limit
    const size_t table_words = (size_t)ctx->rng_pitch * ctx->H;
    const int n_tables = 2 * iters;
    const bool batch = iters > 0 && n_tables <= kRngBatchMax && table_words * n_tables * 4 <= ((size_t)4 << 30);
    if (batch) {
        TSAR_CK(ctx, ctx->rng_batch.reserve(table_words * n_tables));
        unsigned long long seeds[kRngBatchMax];
        for (int t = 0; t < n_tables; t++) seeds[t] = refine_seeds ? refine_seeds[t] : seed0 + 1 + (uint64_t)t;
        TSAR_CK(ctx, pm_launch_rng_tables(ctx->rng_batch.get(), table_words, n_tables, seeds, ctx->rng_pitch, ctx->H, ctx->rng_len, ctx->stream));
        ctx->launches++;
    }
    for (int it = 0; it < iters; it++) {
        for (int col = 0; col < 2; col++) {
            const uint64_t seed = refine_seeds ? refine_seeds[2 * it + col] : seed0 + 1 + 2 * (uint64_t)it + col;
            const uint32_t *table = batch ? ctx->rng_batch.get() + table_words * (2 * it + col) : nullptr;
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
    if (n <= 0 || !xy || !planes || !cost) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad eval arguments");
    const size_t bytes = (size_t)n * (8 + 16 + 4 + 4 + 4);
    TSAR_CK(ctx, ctx->scratch.reserve(bytes));
    unsigned char *base = (unsigned char *)ctx->scratch.get();
    float4 *dpl = (float4 *)base;
    int2 *dxy = (int2 *)(base + (size_t)n * 16);
    float *dc = (float *)(base + (size_t)n * 24);
    int *db = (int *)(base + (size_t)n * 28);
    float *dr = (float *)(base + (size_t)n * 32);
    TSAR_CK(ctx, cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    TSAR_CK(ctx, cudaMemcpyAsync(dpl, planes, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    TSAR_CK(ctx, ctx->variant->eval(ctx->use_u8, ctx->eval_wrapper_rounding, ctx->pm, ctx->ref_img.get(), n, dxy, dpl, dc, db, dr, ctx->stream));
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    TSAR_CK(ctx, cudaMemcpyAsync(cost, dc, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (beview) TSAR_CK(ctx, cudaMemcpyAsync(beview, db, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (ratio) TSAR_CK(ctx, cudaMemcpyAsync(ratio, dr, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

#define PX_GRID dim3 b(32, 8), g((ctx->W + 31) / 32, (ctx->H + 7) / 8)

int tsar_lrdiff(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    lrdiff_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->d_cams.get(), ctx->d_tex.get(), ctx->n_images, ctx->plane[0].get(), ctx->cost[0].get(),
                                            ctx->beview.get(), ctx->lrdiff.get());
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return TSAR_OK;
}

int tsar_getview(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    getview_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0].get(), ctx->cost[0].get(), ctx->lrdiff.get(), ctx->confid.get(), ctx->depth.get());
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return TSAR_OK;
}

int tsar_get_disp(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    get_disp_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0].get(), ctx->depth.get());
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    ctx->have_planes = true;
    return seed_alt_buffers(ctx);
}

int tsar_compute_disp(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    compute_disp_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0].get(), ctx->cost[0].get());
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    ctx->have_planes = false;   // buffer 0 now holds the OUTPUT layout (world normal, depth in w), not (n, d) planes
    return TSAR_OK;
}

int tsar_update_scale(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->region_text.get()) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_regions has not been called");
    if ((rc = consolidate(ctx))) return rc;
    PX_GRID;
    update_scale_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->plane[0].get(), ctx->cost[0].get(), ctx->scale.get(), ctx->depth.get(), ctx->canny.get(),
                                                  ctx->region_text.get(), ctx->region_plane.get(), ctx->n_regions);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return seed_alt_buffers(ctx);   // rows outside the checkerboard grid live in both buffers
}

int tsar_update_scale_2(tsar_ctx *ctx) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!ctx->region_text.get()) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_regions has not been called");
    PX_GRID;
    update_scale_2_kernel<<<g, b, 0, ctx->stream>>>(ctx->glue, ctx->fakedepth.get(), ctx->canny.get(), ctx->region_text.get(),
                                                    ctx->region_plane.get(), ctx->n_regions);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return TSAR_OK;
}

int tsar_wmf(tsar_ctx *ctx, int iter) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (iter < 0 || iter > 3) TSAR_FAIL(ctx, TSAR_ERR_ARG, "WMF level must be 0..3 (gipuma.cu:1809)");
    if ((rc = consolidate(ctx))) return rc;
    const size_t npx = (size_t)ctx->W * ctx->H;
    TSAR_CK(ctx, ctx->scratch.reserve(npx * 4));
    const char *pt = getenv("TSAR_B200_WMF_PER_THREAD");
    rc = wmf_launch(ctx->glue, ctx->ref_img.get(), ctx->plane[0].get(), ctx->depth.get(), ctx->scale.get(), (float *)ctx->scratch.get(), iter, pt && pt[0] == '1',
                    ctx->stream);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return rc;
}

int tsar_wmf_final(tsar_ctx *ctx, int iter) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (iter < 0 || iter > 5) TSAR_FAIL(ctx, TSAR_ERR_ARG, "WMF_Final level must be 0..5 (gipuma.cu:1844)");
    if (!ctx->region_text.get()) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_regions has not been called");
    if ((rc = consolidate(ctx))) return rc;
    const size_t npx = (size_t)ctx->W * ctx->H;
    TSAR_CK(ctx, ctx->scratch.reserve(npx * 24));
    float4 *ps = (float4 *)ctx->scratch.get();
    float *ds = (float *)((unsigned char *)ctx->scratch.get() + npx * 16), *ss = ds + npx;
    rc = wmf_final_launch(ctx->glue, ctx->ref_img.get(), ctx->plane[0].get(), ctx->depth.get(), ctx->scale.get(), ps, ds, ss, ctx->canny.get(),
                          ctx->region_text.get(), ctx->n_regions, iter, ctx->stream);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    if (rc) return rc;
    return seed_alt_buffers(ctx);
}

int tsar_set_regions(tsar_ctx *ctx, int n_regions, const float *text, const float *norm4) {
    if (!ctx || n_regions < 1 || !text || !norm4) return TSAR_ERR_ARG;
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    TSAR_CK(ctx, ctx->region_text.reserve(n_regions));
    TSAR_CK(ctx, ctx->region_plane.reserve(n_regions));
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->region_text.get(), text, (size_t)n_regions * 4, cudaMemcpyHostToDevice, ctx->stream));
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->region_plane.get(), norm4, (size_t)n_regions * 16, cudaMemcpyHostToDevice, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->n_regions = n_regions;
    return TSAR_OK;
}

int tsar_set_labels_quarter(tsar_ctx *ctx, const int *labels, int wq, int hq) {
    if (!ctx || !labels) return TSAR_ERR_ARG;
    if (!ctx->have_views) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_views has not been called");
    if (wq < 1 || hq < 1 || 4 * (wq + 1) < ctx->W || 4 * (hq + 1) < ctx->H || 4 * wq > ctx->W + 3 || 4 * hq > ctx->H + 3)
        TSAR_FAIL(ctx, TSAR_ERR_ARG, "label map is not the quarter-resolution grid of the views");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    TSAR_CK(ctx, ctx->scratch.reserve((size_t)wq * hq * 4));
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->scratch.get(), labels, (size_t)wq * hq * 4, cudaMemcpyHostToDevice, ctx->stream));
    dim3 b(32, 8), g((ctx->W + 31) / 32, (ctx->H + 7) / 8);
    labels_quarter_kernel<<<g, b, 0, ctx->stream>>>((const int *)ctx->scratch.get(), wq, hq, ctx->W, ctx->H, ctx->canny.get());
    TSAR_CK(ctx, cudaGetLastError());
    ctx->launches++;
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));  // the caller's buffer may go away
    return TSAR_OK;
}

// Persistent device scratch of the region fit (grow-only: allocating and freeing synchronise the whole device and would
// stall the other pipelined context).
static int ensure_ransac(tsar_ctx *ctx, size_t n_px, int nt) {
    RansacScratch &r = ctx->ransac;
    TSAR_CK(ctx, r.block_counts.reserve((n_px + 1023) / 1024));
    TSAR_CK(ctx, r.list.reserve(n_px));
    const size_t cap = std::max(nt, 4);
    if (cap * kRansacBatch > r.hyp_counts.capacity()) {
        TSAR_CK(ctx, r.hyp_counts.reserve(cap * kRansacBatch));
        TSAR_CK(ctx, cudaMemsetAsync(r.hyp_counts.get(), 0, cap * kRansacBatch * sizeof(int), ctx->stream));  // the kernel leaves it zeroed
    }
    TSAR_CK(ctx, r.totals.reserve(cap));
    TSAR_CK(ctx, r.pts.reserve(cap * kRansacKeepAll));
    TSAR_CK(ctx, r.rnd.reserve(cap * kRansacRandPerRegion));
    TSAR_CK(ctx, r.jobs.reserve(cap));
    TSAR_CK(ctx, r.out.reserve(cap));
    TSAR_CK(ctx, r.states.reserve(cap));
    TSAR_CK(ctx, r.regions.reserve(cap));
    if (r.grid == 0) {
        int sms = 148, per_sm = 0;
        TSAR_CK(ctx, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
        TSAR_CK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ransac_fit_kernel, kRansacSlice, 0));
        if (per_sm < 1) TSAR_FAIL(ctx, TSAR_ERR_CUDA, "region-fit kernel does not fit on an SM");
        r.grid = sms * std::min(per_sm, 2);   // all CTAs must be co-resident (grid-wide barriers)
    }
    return TSAR_OK;
}

// rnd != nullptr: region-major host array, kRansacRandPerRegion values for EVERY region; else the device stream of `seed`
static int fit_region_planes(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                             const uint32_t *rnd, unsigned long long seed, float *region_norm4) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (n_regions < 1 || !region_text || !region_size || !region_norm4) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad region arguments");
    std::vector<int> targets;
    for (int r = 0; r < n_regions; r++)
        if (region_text[r] == -1.0f) targets.push_back(r);
    if (targets.empty()) return TSAR_OK;
    const size_t n = (size_t)ctx->W * ctx->H;
    if (n > 0x7fffffffull) TSAR_FAIL(ctx, TSAR_ERR_ARG, "image too large for 32-bit pixel indices");
    const int nb = (int)((n + 1023) / 1024), nt = (int)targets.size();
    if ((rc = ensure_ransac(ctx, n, nt))) return rc;
    RansacScratch &S = ctx->ransac;
    cudaStream_t st = ctx->stream;
    std::vector<RansacJob> jobs(nt);
    std::vector<float4> out(nt);
    for (int t = 0; t < nt; t++) {
        const int r = targets[t];
        jobs[t].pts = S.pts.get() + (size_t)t * kRansacKeepAll;
        jobs[t].n = 0;
        jobs[t].size = region_size[r];
        jobs[t].rnd = S.rnd.get() + (size_t)t * kRansacRandPerRegion;
        jobs[t].out = S.out.get() + t;
        out[t] = make_float4(region_norm4[4 * r], region_norm4[4 * r + 1], region_norm4[4 * r + 2], region_norm4[4 * r + 3]);
    }
    // (pageable host sources: cudaMemcpyAsync returns once they are staged, so the vectors may go out of scope)
    TSAR_CK(ctx, cudaMemcpyAsync(S.jobs.get(), jobs.data(), (size_t)nt * sizeof(RansacJob), cudaMemcpyHostToDevice, st));
    TSAR_CK(ctx, cudaMemcpyAsync(S.out.get(), out.data(), (size_t)nt * sizeof(float4), cudaMemcpyHostToDevice, st));
    if (rnd) {
        for (int t = 0; t < nt; t++)
            TSAR_CK(ctx, cudaMemcpyAsync(S.rnd.get() + (size_t)t * kRansacRandPerRegion, rnd + (size_t)targets[t] * kRansacRandPerRegion,
                               (size_t)kRansacRandPerRegion * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    } else {
        TSAR_CK(ctx, cudaMemcpyAsync(S.regions.get(), targets.data(), (size_t)nt * sizeof(int), cudaMemcpyHostToDevice, st));
        ransac_rand_kernel<<<dim3((kRansacRandPerRegion + 255) / 256, nt), 256, 0, st>>>(S.rnd.get(), S.regions.get(), nt, kRansacRandPerRegion, seed);
        ctx->launches++;
    }
    // stable compaction of every target region's reliable pixels (raster order, as the reference collects them) and their
    // back-projection; list lengths stay on the device
    for (int t = 0; t < nt; t++) {
        const int r = targets[t];
        ransac_flag_kernel<<<nb, 1024, 0, st>>>(ctx->scale.get(), ctx->canny.get(), (int)n, r, S.block_counts.get());
        ransac_scan_blocks_kernel<<<1, 1024, 0, st>>>(S.block_counts.get(), nb, S.totals.get() + t);
        ransac_scatter_kernel<<<nb, 1024, 0, st>>>(ctx->scale.get(), ctx->canny.get(), (int)n, r, S.block_counts.get(), S.list.get());
        ransac_points_kernel<<<(kRansacKeepAll + 255) / 256, 256, 0, st>>>(ctx->glue, ctx->depth.get(), S.list.get(), S.totals.get() + t,
                                                                         S.pts.get() + (size_t)t * kRansacKeepAll, S.jobs.get() + t);
        ctx->launches += 4;
    }
    TSAR_CK(ctx, cudaGetLastError());
    // the whole fit: one cooperative launch, loop termination on the device
    RansacFitArgs fa;
    fa.jobs = S.jobs.get(); fa.states = S.states.get(); fa.counts = S.hyp_counts.get(); fa.n_jobs = nt;
    void *kargs[] = {&fa};
    TSAR_CK(ctx, cudaLaunchCooperativeKernel((const void *)ransac_fit_kernel, dim3(S.grid), dim3(kRansacSlice), kargs, 0, st));
    ctx->launches++;
    TSAR_CK(ctx, cudaMemcpyAsync(out.data(), S.out.get(), (size_t)nt * sizeof(float4), cudaMemcpyDeviceToHost, st));
    TSAR_CK(ctx, cudaStreamSynchronize(st));   // the only host wait: the result
    for (int t = 0; t < nt; t++) {
        float *o = region_norm4 + 4 * targets[t];
        o[0] = out[t].x; o[1] = out[t].y; o[2] = out[t].z; o[3] = out[t].w;
    }
    return TSAR_OK;
}

int tsar_fit_region_planes(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                           const uint32_t *rnd, float *region_norm4) {
    if (!ctx) return TSAR_ERR_ARG;
    if (!rnd) TSAR_FAIL(ctx, TSAR_ERR_ARG, "rnd is null (use tsar_fit_region_planes_seeded for a device-generated stream)");
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
    scale_from_confidence_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->confid.get(), threshold, ctx->scale.get(), n);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    return TSAR_OK;
}

int tsar_scale_from_weak_png(tsar_ctx *ctx, const unsigned char *bgr) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!bgr) TSAR_FAIL(ctx, TSAR_ERR_ARG, "weak.png pixels are null");
    const size_t n = (size_t)ctx->W * ctx->H;
    TSAR_CK(ctx, ctx->scratch.reserve(n * 3));
    TSAR_CK(ctx, cudaMemcpyAsync(ctx->scratch.get(), bgr, n * 3, cudaMemcpyHostToDevice, ctx->stream));
    scale_from_weak_png_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((const uchar3 *)ctx->scratch.get(), ctx->scale.get(), n);
    ctx->launches++;
    TSAR_CK(ctx, cudaGetLastError());
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));  // the caller's buffer may go away
    return TSAR_OK;
}

int tsar_download_outputs(tsar_ctx *ctx, float *depth_out, float *normals_out, float *confid_out) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if ((rc = consolidate(ctx))) return rc;
    const size_t n = (size_t)ctx->W * ctx->H;
    if (depth_out || normals_out) {
        TSAR_CK(ctx, ctx->scratch.reserve(n * 16));
        float *d = (float *)ctx->scratch.get(), *nr = d + n;
        split_outputs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->plane[0].get(), d, nr, n);
        ctx->launches++;
        TSAR_CK(ctx, cudaGetLastError());
        if (depth_out) TSAR_CK(ctx, cudaMemcpyAsync(depth_out, d, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (normals_out) TSAR_CK(ctx, cudaMemcpyAsync(normals_out, nr, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (confid_out) TSAR_CK(ctx, cudaMemcpyAsync(confid_out, ctx->confid.get(), n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_ransac_rand_per_region(void) { return kRansacRandPerRegion; }

static void *field_ptr(tsar_ctx *ctx, int field, size_t *elt, size_t *count) {
    *count = (size_t)ctx->W * ctx->H;
    *elt = 4;
    switch (field) {
        case TSAR_F_NORM4: *elt = 16; return ctx->plane[0].get();
        case TSAR_F_COST: return ctx->cost[0].get();
        case TSAR_F_DEPTH: return ctx->depth.get();
        case TSAR_F_FAKEDEPTH: return ctx->fakedepth.get();
        case TSAR_F_SCALE: return ctx->scale.get();
        case TSAR_F_CANNY: return ctx->canny.get();
        case TSAR_F_RATIO: return ctx->ratio.get();
        case TSAR_F_BEVIEW: return ctx->beview.get();
        case TSAR_F_LRDIFF: return ctx->lrdiff.get();
        case TSAR_F_CONFID: return ctx->confid.get();
        case TSAR_F_REGION_TEXT: *count = ctx->n_regions; return ctx->region_text.get();
        case TSAR_F_REGION_NORM4: *count = ctx->n_regions; *elt = 16; return ctx->region_plane.get();
    }
    return nullptr;
}

int tsar_upload(tsar_ctx *ctx, int field, const void *src, size_t bytes) {
    if (!ctx || !src) return TSAR_ERR_ARG;
    if (!ctx->have_views) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_views has not been called");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    if (field == TSAR_F_NORM4 || field == TSAR_F_COST) {
        int rc = consolidate(ctx);
        if (rc) return rc;
    }
    size_t elt, count;
    void *p = field_ptr(ctx, field, &elt, &count);
    if (!p || bytes != elt * count) TSAR_FAIL(ctx, TSAR_ERR_ARG, "field/size mismatch");
    TSAR_CK(ctx, cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (field == TSAR_F_NORM4) {
        ctx->have_planes = true;
        return seed_alt_buffers(ctx);
    }
    if (field == TSAR_F_COST) return seed_alt_buffers(ctx);
    return TSAR_OK;
}

int tsar_download(tsar_ctx *ctx, int field, void *dst, size_t bytes) {
    if (!ctx || !dst) return TSAR_ERR_ARG;
    if (!ctx->have_views) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_views has not been called");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    if (field == TSAR_F_NORM4 || field == TSAR_F_COST) {
        int rc = consolidate(ctx);
        if (rc) return rc;
    }
    size_t elt, count;
    void *p = field_ptr(ctx, field, &elt, &count);
    if (!p || bytes != elt * count) TSAR_FAIL(ctx, TSAR_ERR_ARG, "field/size mismatch");
    TSAR_CK(ctx, cudaMemcpyAsync(dst, p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_device_ptr(tsar_ctx *ctx, int field, void **dev_ptr) {
    if (!ctx || !dev_ptr) return TSAR_ERR_ARG;
    if (!ctx->have_views) TSAR_FAIL(ctx, TSAR_ERR_STATE, "tsar_set_views has not been called");
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
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
    TSAR_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if ((rc = tsar_init_planes(ctx, seed0))) return rc;
    if ((rc = tsar_iterate(ctx, ctx->params.iterations, seed0, nullptr))) return rc;
    if ((rc = tsar_lrdiff(ctx))) return rc;
    if ((rc = tsar_getview(ctx))) return rc;
    if ((rc = tsar_compute_disp(ctx))) return rc;
    TSAR_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (ms_out) {
        TSAR_CK(ctx, cudaEventSynchronize(ctx->ev1));
        TSAR_CK(ctx, cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
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
    if (norm4_out) TSAR_CK(ctx, cudaMemcpyAsync(norm4_out, ctx->plane[0].get(), n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (confid_out) TSAR_CK(ctx, cudaMemcpyAsync(confid_out, ctx->confid.get(), n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_slic(tsar_ctx *ctx, const unsigned char *bgrx, const tsar_slic_settings *s, int *labels_out) {
    if (!ctx || !bgrx || !s || !labels_out) return TSAR_ERR_ARG;
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    int nl = 0;
    const int rc = slic_run(*ctx, ctx->slic, bgrx, *s, labels_out, ctx->stream, &nl);
    ctx->launches += nl;
    return rc;
}

// debug: the superpixel records of the last tsar_slic call (8 words each: centre x, y, colour x, y, z, w, id, no_pixels,
// the layout of gSLICr::objects::spixel_info), for stage-by-stage comparison with the reference engine
int tsar_dbg_slic_centres(tsar_ctx *ctx, float *out, int max_records, int *n_records) {
    if (!ctx || !n_records) return TSAR_ERR_ARG;
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    const int n = ctx->slic.last_nsp;
    *n_records = n;
    const int m = n < max_records ? n : max_records;
    if (out && m > 0) {
        std::vector<SpixelInfo> host(m);   // the device record is 48 bytes (float4 alignment); the reference's is 32
        TSAR_CK(ctx, cudaMemcpyAsync(host.data(), ctx->slic.d_sp.get(), (size_t)m * sizeof(SpixelInfo), cudaMemcpyDeviceToHost, ctx->stream));
        TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
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
    TSAR_CK(ctx, cudaSetDevice(ctx->device));
    if (n_pixels > ctx->slic.d_lab.capacity() || !ctx->slic.d_lab.get()) TSAR_FAIL(ctx, TSAR_ERR_ARG, "no Lab image of that size (run tsar_slic first)");
    TSAR_CK(ctx, cudaMemcpyAsync(out, ctx->slic.d_lab.get(), n_pixels * 16, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
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
    if (!ctx->have_views || !ctx->have_params) TSAR_FAIL(ctx, TSAR_ERR_STATE, "views/params not set");
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
    if (image < 0 || image >= ctx->n_images || n <= 0 || !xy || !out) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad sample arguments");
    TSAR_CK(ctx, ctx->scratch.reserve((size_t)n * 12));
    float2 *dxy = (float2 *)ctx->scratch.get();
    float *dout = (float *)((unsigned char *)ctx->scratch.get() + (size_t)n * 8);
    TSAR_CK(ctx, cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    dbg_tex_sample_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->tex[image].tex(), n, dxy, dout);
    TSAR_CK(ctx, cudaGetLastError());
    TSAR_CK(ctx, cudaMemcpyAsync(out, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return TSAR_OK;
}

int tsar_profile(tsar_ctx *ctx, int enable) {
    if (!ctx) return TSAR_ERR_ARG;
    ctx->profiling = enable != 0;
    return TSAR_OK;
}

int tsar_profile_read(tsar_ctx *ctx, float *checker_ms_total, int *n_launches) {
    if (!ctx || !checker_ms_total || !n_launches) return TSAR_ERR_ARG;
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    float tot = 0.f;
    for (auto &pr : ctx->prof_events) {
        float ms = 0.f;
        TSAR_CK(ctx, cudaEventElapsedTime(&ms, pr.first, pr.second));
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
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
    int n = 0;
    for (auto &pr : ctx->prof_events) {
        float t = 0.f;
        TSAR_CK(ctx, cudaEventElapsedTime(&t, pr.first, pr.second));
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
    if (!out || colour < 0 || colour > 1) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad candidate-statistics arguments");
    if (!ctx->have_planes) TSAR_FAIL(ctx, TSAR_ERR_STATE, "no planes: call tsar_init_planes or tsar_load_planes first");
    TSAR_CK(ctx, ctx->scratch.reserve(kCandStatWords * sizeof(unsigned long long)));
    CheckerArgs a{};
    for (int col = 0; col < 2; col++) { a.plane_in[col] = ctx->plane[ctx->cur[col]].get(); a.cost_in[col] = ctx->cost[ctx->cur[col]].get(); }
    a.colour = colour;
    TSAR_CK(ctx, cudaMemsetAsync(ctx->scratch.get(), 0, kCandStatWords * sizeof(unsigned long long), ctx->stream));
    TSAR_CK(ctx, pm_launch_cand_stats(ctx->pm, a, (unsigned long long *)ctx->scratch.get(), ctx->stream));
    ctx->launches++;
    TSAR_CK(ctx, cudaMemcpyAsync(out, ctx->scratch.get(), kCandStatWords * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
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
    if (image < 0 || image >= ctx->n_images || n <= 0 || !xy || !out || !rate4) TSAR_FAIL(ctx, TSAR_ERR_ARG, "bad sample arguments");
    const int W = ctx->W, H = ctx->H;
    std::vector<float> host((size_t)W * H);
    TSAR_CK(ctx, cudaMemcpy2DFromArray(host.data(), (size_t)W * 4, ctx->tex[image].array(), 0, 0, (size_t)W * 4, H, cudaMemcpyDeviceToHost));
    std::vector<unsigned char> h8((size_t)W * H);
    std::vector<unsigned short> h16((size_t)W * H), hf16((size_t)W * H);
    for (size_t i = 0; i < host.size(); i++) {
        h8[i] = (unsigned char)host[i];
        h16[i] = (unsigned short)(host[i] * 257.0f);
        hf16[i] = __half_as_ushort(__float2half(host[i]));
    }
    Texture2D formats[3];   // freed on every return
    cudaChannelFormatDesc cds[3] = {cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned),
                                    cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindUnsigned),
                                    cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindFloat)};
    const void *srcs[3] = {h8.data(), h16.data(), hf16.data()};
    const size_t esz[3] = {1, 2, 2};
    for (int k = 0; k < 3; k++) {
        const cudaTextureReadMode read = (k < 2) ? cudaReadModeNormalizedFloat : cudaReadModeElementType;
        TSAR_CK(ctx, formats[k].create(W, H, cds[k], cudaAddressModeClamp, read));
        TSAR_CK(ctx, cudaMemcpy2DToArray(formats[k].array(), 0, 0, srcs[k], W * esz[k], W * esz[k], H, cudaMemcpyHostToDevice));
    }
    const cudaTextureObject_t tex[4] = {ctx->tex[image].tex(), formats[0].tex(), formats[1].tex(), formats[2].tex()};
    TSAR_CK(ctx, ctx->scratch.reserve((size_t)n * 12));
    float2 *dxy = (float2 *)ctx->scratch.get();
    float *dout = (float *)((unsigned char *)ctx->scratch.get() + (size_t)n * 8);
    TSAR_CK(ctx, cudaMemcpyAsync(dxy, xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    for (int k = 0; k < 4; k++) {
        dbg_tex_sample_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(tex[k], n, dxy, dout);
        TSAR_CK(ctx, cudaMemcpyAsync(out + (size_t)k * n, dout, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        TSAR_CK(ctx, cudaStreamSynchronize(ctx->stream));
        float best = 0.f;
        for (int rep = 0; rep < 3; rep++) {
            float ms;
            TSAR_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
            dbg_tex_kernel<<<sms * 8, 256, 0, ctx->stream>>>(tex[k], dout, 256, W, H);
            TSAR_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
            TSAR_CK(ctx, cudaEventSynchronize(ctx->ev1));
            TSAR_CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
            best = std::max(best, (float)((double)sms * 8 * 256 * 256 * 4 / (ms * 1e-3) / 1e9));
        }
        rate4[k] = best;
    }
    return TSAR_OK;
}

int tsar_dbg_peaks(tsar_ctx *ctx, float *out3) {
    int rc = need_ready(ctx);
    if (rc) return rc;
    if (!out3) return TSAR_ERR_ARG;
    TSAR_CK(ctx, ctx->scratch.reserve(64));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    const int blocks = sms * 8, threads = 256, iters = 4096;
    float best[3] = {0, 0, 0};
    for (int rep = 0; rep < 4; rep++) {
        float ms;
        TSAR_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_ffma_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)ctx->scratch.get(), iters, 1.0000001f, 1e-9f);
        TSAR_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        TSAR_CK(ctx, cudaEventSynchronize(ctx->ev1));
        TSAR_CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[0] = std::max(best[0], (float)((double)blocks * threads * iters * 8 * 8 * 2 / (ms * 1e-3) / 1e12));
        TSAR_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_mufu_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)ctx->scratch.get(), iters / 4);
        TSAR_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        TSAR_CK(ctx, cudaEventSynchronize(ctx->ev1));
        TSAR_CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[1] = std::max(best[1], (float)((double)blocks * threads * (iters / 4) * 8 * 8 / (ms * 1e-3) / 1e9));
        TSAR_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        dbg_tex_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->tex[0].tex(), (float *)ctx->scratch.get(), iters / 16, ctx->W, ctx->H);
        TSAR_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        TSAR_CK(ctx, cudaEventSynchronize(ctx->ev1));
        TSAR_CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best[2] = std::max(best[2], (float)((double)blocks * threads * (iters / 16) * 4 / (ms * 1e-3) / 1e9));
    }
    out3[0] = best[0];  // TFLOP/s FP32 FFMA
    out3[1] = best[1];  // G MUFU ops / s
    out3[2] = best[2];  // G bilinear fp32 texture samples / s
    return TSAR_OK;
}

}  // extern "C"
