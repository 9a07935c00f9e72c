/*
 * tsar_b200.h -- C ABI of the B200-native TSAR-MVS depthmap path.
 *
 * This is the drop-in boundary for the per-reference-view depthmap hot path of TSAR-MVS
 * (reference: gipuma.cu + gSLICr_Lib).  Every entry point names the reference interface it
 * replaces (file:line relative to the reference checkout).  Plain pointers and sizes only:
 * no C++ types, no torch types, no managed memory.  All functions return TSAR_OK (0) or a
 * negative tsar_status; they never call exit() (the reference's checkCudaErrors does,
 * helper_cuda.h:891-905).  tsar_last_error() gives the text for the last failure on a context.
 *
 * Threading: one context = one reference view in flight on one device/stream.  Contexts are
 * independent; use one per GPU (or several per GPU on different streams) to shard reference
 * views (reference: one process per view, scripts/pipes.sh:30-49).
 *
 * The C++ shims with the reference's own signatures (firstcuda/sliccuda/fakecuda/fillcuda,
 * gipuma.h:2-5) live in tsar_gipuma_abi.h and are implemented on top of this file.
 */
#ifndef TSAR_B200_H
#define TSAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSAR_MAX_VIEWS 32 /* pmCostMultiview_cu costVector[32], gipuma.cu:467-468 (Q8) */

typedef enum tsar_status {
    TSAR_OK = 0,
    TSAR_ERR_ARG = -1,     /* bad argument (null, size, V outside [1,32], ...) */
    TSAR_ERR_STATE = -2,   /* call order (e.g. iterate before set_views)        */
    TSAR_ERR_CUDA = -3,    /* a CUDA runtime call failed                        */
    TSAR_ERR_NOMEM = -4,   /* a device or pinned allocation failed              */
    TSAR_ERR_NODEVICE = -5 /* no CUDA device / not an sm_100 part: there is no CPU fallback */
} tsar_status;

/* Value fields of Camera_cu (camera.h:7-65) for one view, already moved into the frame of the
 * reference camera as getCameraParameters(transformP=true) does (cameraGeometryUtils.h:174-364).
 * All 3x3 matrices row-major. */
typedef struct tsar_camera {
    float K[9];          /* camera.h:26  own intrinsics                                   */
    float K_inv[9];      /* camera.h:27                                                   */
    float R[9];          /* camera.h:12  R' = R_i * R_0^T                                 */
    float R_orig[9];     /* camera.h:13  world->camera rotation before the move           */
    float R_orig_inv[9]; /* camera.h:14                                                   */
    float M_inv[9];      /* camera.h:11  inverse of P[:, :3], P = K_0 [R'|t']             */
    float t4[3];         /* camera.h:15  t'                                               */
    float P_col34[3];    /* camera.h:9   P[:,3]                                           */
    float C4[3];         /* camera.h:16  centre of P                                      */
    float fx, fy, f, alpha, baseline; /* camera.h:17-21 (fx=fy'=K_0 values, alpha=fx/fy)  */
    float depthMin, depthMax;         /* camera.h:23-28                                   */
} tsar_camera;

/* Hot fields of AlgorithmParameters (algorithmparameters.h:19-89). */
typedef struct tsar_params {
    int box_hsize;        /* :57 window width  (scripts: --blocksize=11)  */
    int box_vsize;        /* :58 window height                            */
    int iterations;       /* :64 red/black iterations (8)                 */
    int n_best;           /* :74                                          */
    int cost_comb;        /* :75 0 = COMB_ALL, 1 = COMB_BEST_N            */
    float min_disparity;  /* :56 = f*baseline/depthMax (main.cpp:1393)    */
    float max_disparity;  /* :55 = f*baseline/depthMin (main.cpp:1396)    */
    int color_processing; /* :65 accepted; the kernels sample float4 textures with tex2D<float> = channel x, so pass channel x (blue) of each view as its image */
} tsar_params;

/* gSLICr settings (gSLICr_settings.h:10-21); TSAR's call site: main.cpp:608-615. */
typedef struct tsar_slic_settings {
    int img_w, img_h;
    int spixel_size;             /* 20 */
    int no_iters;                /* 5  */
    float coh_weight;            /* 5  */
    int do_enforce_connectivity; /* 0  */
    int correct_reduction;       /* 0 = bit-parity with the reference build's partial warp-tail
                                    reduction (SURVEY Q10); 1 = mathematically complete sums */
} tsar_slic_settings;

/* Per-pixel / per-region arrays of LineState (linestate.h:10-221) that cross the boundary. */
typedef enum tsar_field {
    TSAR_F_NORM4 = 0,        /* float4 lines->norm4  plane (n, d), n.X + d = 0      :12  */
    TSAR_F_COST = 1,         /* float  lines->c                                      :13  */
    TSAR_F_DEPTH = 2,        /* float  lines->depth (holds a disparity, sic)         :14  */
    TSAR_F_FAKEDEPTH = 3,    /* float  lines->fakedepth                              :15  */
    TSAR_F_SCALE = 4,        /* float  lines->scale   reliable flag                  :33  */
    TSAR_F_CANNY = 5,        /* float  lines->canny   region label stored as float   :17  */
    TSAR_F_RATIO = 6,        /* float  lines->ratio                                  :40  */
    TSAR_F_BEVIEW = 7,       /* int    lines->beview                                 :41  */
    TSAR_F_LRDIFF = 8,       /* float  lines->lrdiff                                 :42  */
    TSAR_F_CONFID = 9,       /* float  lines->confid                                 :43  */
    TSAR_F_REGION_TEXT = 10, /* float  cannylines->text  (-1 = textureless region)   :36  */
    TSAR_F_REGION_NORM4 = 11 /* float4 cannylines->norm4 per-region plane            :12  */
} tsar_field;

/* Launch kinds for tsar_launch (single checkerboard half-steps, gipuma.cu:1746-1752). */
enum { TSAR_BLACK_SPATIAL = 0, TSAR_BLACK_REFINE = 1, TSAR_RED_SPATIAL = 2, TSAR_RED_REFINE = 3 };

typedef struct tsar_ctx tsar_ctx;

/* ---- context ------------------------------------------------------------------------------ */
/* Replaces selectCudaDevice + new GlobalState (main.cpp:1230-1266, 1876; globalstate.h:25-54).
 * `stream` is a cudaStream_t passed as void* (NULL = a private non-blocking stream). */
int tsar_create(int device, void *stream, tsar_ctx **out);
int tsar_destroy(tsar_ctx *ctx);
const char *tsar_last_error(const tsar_ctx *ctx);
int tsar_sync(tsar_ctx *ctx);

/* ---- inputs ------------------------------------------------------------------------------- */
/* Replaces addImageToTextureFloatGray + the camera/view-selection fill of runGipuma
 * (main.cpp:1190-1228, 1316-1385).  images[i] points to W*H float32 grey values (0..255,
 * main.cpp:1423), image 0 is the reference view; cams[i] likewise.  subset[0..V) are indices of
 * the selected source views (CameraParameters_cu::viewSelectionSubset, cameraparameters.h:17).
 * images_on_device != 0 means the pointers are device pointers (no H2D copy). */
int tsar_set_views(tsar_ctx *ctx, int W, int H, int n_images, const float *const *images,
                   int images_on_device, const tsar_camera *cams, float cam_f, const int *subset, int V);
/* Replaces gs->params = &algParams (main.cpp:1408). */
int tsar_set_params(tsar_ctx *ctx, const tsar_params *p);

/* ---- the PatchMatch path (north-star items 1-3) ---------------------------------------------- */
/* gipuma_init_cu2 (gipuma.cu:679-729) with curand_init(seed, y, x): same XORWOW streams as the
 * reference when it is given `seed` in place of clock64(). */
int tsar_init_planes(tsar_ctx *ctx, uint64_t seed);
/* Alternative to tsar_init_planes: take the reference's initial planes (host pointers;
 * norm4 = W*H float4, cost = W*H float or NULL to evaluate the cost of the loaded planes). */
int tsar_load_planes(tsar_ctx *ctx, const float *norm4, const float *cost);
/* One checkerboard half-step (gipuma_{black,red}_{spatialProp,planeRefine}_cu, gipuma.cu:1097-1138);
 * `seed` is used by the refine kinds only. */
int tsar_launch(tsar_ctx *ctx, int kind, uint64_t seed);
/* The loop of gipuma_first (gipuma.cu:1744-1754): iters x (black SP, black PR, red SP, red PR).
 * refine_seeds = 2*iters seeds (black, red per iteration) or NULL for seed0+1+2*it+colour. */
int tsar_iterate(tsar_ctx *ctx, int iters, uint64_t seed0, const uint64_t *refine_seeds);
/* pmCostMultiview_cu (gipuma.cu:456-518) for n explicit (pixel, plane) pairs; host pointers:
 * xy = n int2, planes = n float4, outputs n each (beview/ratio may be NULL). */
int tsar_eval_planes(tsar_ctx *ctx, int n, const int *xy, const float *planes, float *cost, int *beview,
                     float *ratio);

/* ---- confidence, TSAR glue and depth completion (north-star item 4) --------------------------- */
int tsar_lrdiff(tsar_ctx *ctx);          /* gipuma_getlrdiff      gipuma.cu:1161-1186            */
int tsar_getview(tsar_ctx *ctx);         /* gipuma_getview        gipuma.cu:1189-1213 (sliccuda) */
int tsar_get_disp(tsar_ctx *ctx);        /* gipuma_get_disp       gipuma.cu:732-755  (firstcuda) */
int tsar_update_scale_2(tsar_ctx *ctx);  /* gipuma_update_scale_2 gipuma.cu:1262-1292 (fakecuda) */
int tsar_update_scale(tsar_ctx *ctx);    /* gipuma_update_scale   gipuma.cu:1216-1259 (fillcuda) */
int tsar_compute_disp(tsar_ctx *ctx);    /* gipuma_compute_disp   gipuma.cu:810-844  (fillcuda)  */
int tsar_wmf(tsar_ctx *ctx, int iter);        /* gipuma_WMF       gipuma.cu:1500-1698 */
int tsar_wmf_final(tsar_ctx *ctx, int iter);  /* gipuma_WMF_Final gipuma.cu:1295-1497 */
/* Region table for the two update_scale kernels (cannylines->text / ->norm4, main.cpp:570-593,
 * 1722-1729).  Host pointers, n_regions entries. */
int tsar_set_regions(tsar_ctx *ctx, int n_regions, const float *text, const float *norm4);

/* Per-region plane fitting for textureless regions (the CPU RANSAC of main.cpp:1520-1730, calcLinePara
 * main.cpp:147-164): for every region r with region_text[r] == -1, the reliable pixels (scale == 1) carrying label r
 * in lines->canny are back-projected with lines->depth (a disparity) and a plane is fitted by 10 000 RANSAC triples
 * with the reference's adaptive inlier threshold (seeded by region_size[r] = cannylines->size[r]) followed by
 * 1000 x 4 local perturbation rounds.  rnd supplies the values the reference takes from rand():
 * tsar_ransac_rand_per_region() (= 46 000) non-negative integers per region, region-major.  region_norm4
 * (n_regions float4, host) is read for the initial value and receives (a, b, c, d) of the fitted regions;
 * pass it to tsar_set_regions afterwards.  Uses the context's scale / canny / depth arrays. */
int tsar_fit_region_planes(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                           const uint32_t *rnd, float *region_norm4);
int tsar_ransac_rand_per_region(void);
/* Same fit with the rand() stream generated on the device from `seed` (no 46 000-value host array per region): value i of
 * region r is tsar_ransac_rand_value(seed, r, i), a counter-based stream of non-negative 31-bit integers.  The reference
 * never seeds rand(), so any stream is as faithful as another; this one is reproducible. */
int tsar_fit_region_planes_seeded(tsar_ctx *ctx, int n_regions, const float *region_text, const float *region_size,
                                  uint64_t seed, float *region_norm4);
uint32_t tsar_ransac_rand_value(uint64_t seed, int region, int index);

/* lines->scale (the "reliable pixel" flags the RANSAC fit and WMF read).  The shipped flow fills it on the host from APD's
 * weak.png: 1 where the pixel is white, green or red (main.cpp:1499-1514) -- tsar_scale_from_weak_png does that on the
 * device from the decoded W*H BGR bytes (host pointer).  When PatchMatch runs inside the library there is no weak.png;
 * tsar_scale_from_confidence sets scale = (confid > threshold) from gipuma_getview's confidence instead. */
int tsar_scale_from_weak_png(tsar_ctx *ctx, const unsigned char *bgr);
int tsar_scale_from_confidence(tsar_ctx *ctx, float threshold);

/* ---- weak-texture region detector: texture() in main.cpp:365-596 (SURVEY section 8 row f3) --------------------
 * Host functions (sequential raster scans whose results depend on the scan order; the reference runs them on the
 * quarter-resolution grey image, <= 0.4 Mpx at C2).  The OpenCV stages in between -- pyrDown x2 before, HoughLinesP +
 * line() per weak label between the two labellings -- stay with the caller, who has OpenCV (the reference's main.cpp,
 * or tsar-mvs_b200/texture.py).  All buffers are host memory, row-major w x h. */
/* roberts() main.cpp:214-240 + cv::threshold(.., thr, 255, THRESH_BINARY) main.cpp:383; thr = Robthr = 4 */
int tsar_weak_edges(const unsigned char *gray, int w, int h, int thr, unsigned char *edges);
/* Connect() main.cpp:242-362: labels (0 = edge), per-label pixel counts (cap entries available), label count */
int tsar_weak_connect(const unsigned char *edges, int w, int h, int *labels, int *label_count, int cap, int *n_labels);
/* boundary image of one label, the input of HoughLinesP (main.cpp:392-421) */
int tsar_weak_boundary(const int *labels, int w, int h, int label, unsigned char *gray);
/* border closing before the second labelling (main.cpp:441-454), in place */
int tsar_weak_close_border(unsigned char *edges, int w, int h);
/* region statistics + weak decision (main.cpp:478-536, 570-593): cannylines->text / cenxi / cenyi / size;
 * min_pixels = weaktextnum = 5000, size_ratio = (int)sizerat = 2 */
int tsar_weak_regions(const int *labels, int w, int h, const int *label_count, int n_labels, int min_pixels,
                      int size_ratio, float *text, int *cenxi, int *cenyi, float *size);
/* lines->canny[] from the quarter-resolution label map (main.cpp:558-568), expanded on the device: 1/16 of the
 * host-to-device bytes of uploading the full-resolution float map. */
int tsar_set_labels_quarter(tsar_ctx *ctx, const int *labels, int wq, int hq);

/* ---- state transfer --------------------------------------------------------------------------- */
int tsar_upload(tsar_ctx *ctx, int field, const void *host_src, size_t bytes);
int tsar_download(tsar_ctx *ctx, int field, void *host_dst, size_t bytes);
/* The payloads of the reference's output files after gipuma_compute_disp (main.cpp:1785-1861): depth (W*H floats,
 * TSAR_disp.dmb), normals (W*H*3 floats, TSAR_normals.dmb) and the confidence map (W*H floats; computed but never
 * written by the reference).  The output layout is split on the device; host pointers (pinned memory makes the copies
 * asynchronous to other streams); any of them may be NULL. */
int tsar_download_outputs(tsar_ctx *ctx, float *depth_out, float *normals_out, float *confid_out);
/* Device pointer of a field (for zero-copy consumers on the same GPU).  For TSAR_F_NORM4 and
 * TSAR_F_COST the per-colour double buffers are first merged into the returned array (on the context's stream); the
 * pointer is valid until the next call that launches propagation or refinement (tsar_launch, tsar_iterate,
 * tsar_depthmap), after which the live values of one colour sit in the other buffer again. */
int tsar_device_ptr(tsar_ctx *ctx, int field, void **dev_ptr);

/* ---- whole north-star sequence ------------------------------------------------------------------ */
/* init -> iters x (bSP,bPR,rSP,rPR) -> getlrdiff -> getview -> compute_disp, everything resident.
 * ms_out (optional) receives the CUDA-event time of the sequence on the context's stream. */
int tsar_depthmap(tsar_ctx *ctx, uint64_t seed0, float *ms_out);
/* Host-buffer entry (the e2e path): uploads the views, runs tsar_depthmap, downloads the output
 * layout of gipuma_compute_disp (norm4_out: xyz = world normal, w = depth; W*H float4) and the
 * confidence map (W*H float).  Either output may be NULL. */
int tsar_depthmap_host(tsar_ctx *ctx, int W, int H, int n_images, const float *const *images,
                       const tsar_camera *cams, float cam_f, const int *subset, int V,
                       const tsar_params *p, uint64_t seed0, float *norm4_out, float *confid_out);

/* ---- gSLICr (north-star item 4) ------------------------------------------------------------------- */
/* core_engine::Process_Frame + Get_Seg_Res (gSLICr_core_engine.h:11-33; sequence
 * gSLICr_seg_engine.cpp:30-46).  bgrx = img_w*img_h uchar4 with the bytes of the reference's UChar4Image: its colour
 * conversion reads byte 0 as blue, byte 1 as green, byte 2 as red (gSLICr_seg_engine_shared.h:21-23).  Note that the
 * reference's load_image (main.cpp:190-201) stores OpenCV's B into `.b` = byte 2 and R into `.r` = byte 0, so TSAR runs
 * the conversion with red and blue exchanged; callers that want the reference's labels fill the bytes as load_image
 * does (R, G, B, x).  The C++ class itself is exported as well (include/tsar_gslicr_abi.h).
 * labels_out = img_w*img_h int32.  Host pointers. */
int tsar_slic(tsar_ctx *ctx, const unsigned char *bgrx, const tsar_slic_settings *s, int *labels_out);

/* ---- instrumentation --------------------------------------------------------------------------------- */
/* Kernels launched by this context since creation (or since the last reset). */
int tsar_launch_count(tsar_ctx *ctx, long long *count, int reset);
/* pmCost evaluations (plane x source view x window) executed, from the closed form of
 * BASELINE.md section 3 evaluated with the exact border guards. */
int tsar_eval_count(tsar_ctx *ctx, int iters, long long *n_evals);
/* CUDA-event timing of the dominant kernel (the fused checkerboard propagation+refinement kernel) on the
 * stream it is launched on: enable, run, then read the summed duration and the number of launches. */
int tsar_profile(tsar_ctx *ctx, int enable);
int tsar_profile_read(tsar_ctx *ctx, float *checker_ms_total, int *n_launches);
/* The same events one by one: ms[i] = CUDA-event time of the i-th checkerboard launch since profiling was enabled (the
 * first cap of them); *n_launches = how many there were.  Consumes the events as tsar_profile_read does. */
int tsar_profile_read_launches(tsar_ctx *ctx, float *ms, int cap, int *n_launches);
const char *tsar_version(void);
/* tex2D<float> of image `image` at n unnormalised coordinates (xy = n float2, host): used to
 * calibrate software models of the texture unit's bilinear filter (SURVEY Q9). */
int tsar_dbg_tex_sample(tsar_ctx *ctx, int image, int n, const float *xy, float *out);
/* Issue-rate microbenchmarks on this GPU: out3 = {FP32 FFMA TFLOP/s, MUFU Gop/s, bilinear fp32
 * texture Gsamples/s}; the measured denominators of the PatchMatch roofline (DESIGN.md). */
int tsar_dbg_peaks(tsar_ctx *ctx, float *out3);
/* Experiment: samples + bilinear fetch rate of the same image stored as f32 / u8-unorm / u16-unorm / f16 texels
 * (out = 4*n floats, rate4 = Gsamples/s per format). */
int tsar_dbg_tex_formats(tsar_ctx *ctx, int image, int n, const float *xy, float *out, float *rate4);
/* Device-side counter of the propagation candidates of the checkerboard launch of `colour` that would run on the
 * current state (BASELINE.md section 3): out = 22 counters -- pixels of the colour, candidates behind their border guards
 * (the closed form of tsar_eval_count), candidates inside the depth range (= cost evaluations the reference executes,
 * per source view), bitwise duplicates of the pixel's own plane, duplicates of an earlier candidate of the same pixel,
 * distinct candidates; warp-wide evaluation rounds as written / with per-lane lists of distinct candidates / perfectly
 * packed; warps; the same three figures without the own-plane rule; then pixels by number of distinct candidates 0..8. */
/* Debug: superpixel records of the last tsar_slic call, 8 words each in the layout of gSLICr::objects::spixel_info
 * (gSLICr_spixel_info.h:10-16: centre x, y; colour x, y, z, w; int id; int no_pixels). */
int tsar_dbg_slic_centres(tsar_ctx *ctx, float *out, int max_records, int *n_records);
/* Debug: the CIELAB image (4 floats per pixel) tsar_slic computed from its last input (rgb2CIELab, gSLICr_seg_engine_shared.h:30-59). */
int tsar_dbg_slic_lab(tsar_ctx *ctx, float *out, size_t n_pixels);
int tsar_dbg_candidate_stats(tsar_ctx *ctx, int colour, unsigned long long *out22);
/* Test-only: tsar_eval_planes normally rounds H*(x,y,1) as the reference's real kernels do
 * (fma(m0,x, m1*y) + m2).  The oracle's stand-alone wrapper kernel around pmCostMultiview_cu is compiled
 * by nvcc with the loop-hoisted form (fma(m1,y, m0*x) + m2); wrapper_rounding=1 selects that form so the
 * unit-level test can require bit equality against the wrapper.  Production kernels are unaffected. */
int tsar_dbg_eval_rounding(tsar_ctx *ctx, int wrapper_rounding);

/* Quad-cooperative sampling (DESIGN.md 4.2): the four lanes of a texture quad fetch samples of one window at a time.
 * checker_launches < 0: off everywhere (as env TSAR_B200_NO_QUAD_SAMPLING=1); >= 0: used by tsar_init_planes and by
 * the first checker_launches checkerboard launches after tsar_init_planes / tsar_load_planes.  Applies to the 11x11
 * window with 8-bit textures (and, for the checkerboard, pinhole cameras).  Results are bit-identical either way. */
int tsar_dbg_quad_sampling(tsar_ctx *ctx, int checker_launches);

/* ---- multi-view fusion (DESIGN.md section 4.6) ------------------------------------------------------------------------
 * Fuses the per-view depth maps of a dataset (TSAR_disp.dmb / TSAR_normals.dmb + the colour images) into one coloured
 * point cloud by a multi-view consistency check.  The stage of the reference pipeline after TSAR is Fusion.exe, a closed
 * binary; this rule follows the published ACMM/ACMMP RunFusion family with the differences listed in DESIGN.md 4.6.
 * A handle of its own, since fusion spans many views and a tsar_ctx holds one.  All views have the same W x H.
 * Views are fused in index order (view v skips source pixels that views < v already used); inside a view the work is
 * parallel and the result identical to the sequential rule.  Device memory: 21 B per pixel and view (depth + normal
 * float4, BGR + pad, mask) plus scratch for one view (8 B per pixel and neighbour, 29 B per pixel); the points leave the
 * device view by view. */
#define TSAR_FUSION_MAX_NEIGHBOURS 32

typedef struct tsar_view_camera { float K[9], R[9], t[3]; } tsar_view_camera;   /* world -> camera, row-major */
typedef struct tsar_fusion_params {
    float max_reproj_px;   /* 2.0   round-trip reprojection error, pixels (strict <)                  */
    float max_rel_depth;   /* 0.01  |z' - D| < max_rel_depth * D (strict)                              */
    float max_normal_deg;  /* 10    n_v.n_u >= cos(max_normal_deg) |n_v| |n_u| (cosine taken in double) */
    int min_consistent;    /* 2     consistent source pixels a point needs                             */
} tsar_fusion_params;
typedef struct tsar_fusion tsar_fusion;

/* `stream` as in tsar_create.  TSAR_ERR_ARG unless n_views >= 1 and 1 <= W*H <= 0x7f7f7f7f - 256; TSAR_ERR_NODEVICE
 * without an sm_100 device, TSAR_ERR_NOMEM when the views do not fit. */
int tsar_fusion_create(int device, void *stream, int n_views, int W, int H, tsar_fusion **out);
/* Host pointers: depth = W*H floats (camera z, 0 = no depth; a pixel is used when its depth is finite and > 0),
 * normals = W*H*3 floats (world frame), bgr = W*H*3 bytes.  neighbours = 1..32 distinct view indices, not `view`. */
int tsar_fusion_set_view(tsar_fusion *f, int view, const tsar_view_camera *cam, const float *depth,
                         const float *normals, const unsigned char *bgr, const int *neighbours, int n_neighbours);
/* Fuses every view (all must be set; masks are reset first, so it may be called again with other parameters).
 * n_points (may be NULL) receives the number of points, ordered by view, then by raster order of the reference pixel. */
int tsar_fusion_run(tsar_fusion *f, const tsar_fusion_params *p, long long *n_points);
/* The points of the last run: xyz and normals 3 floats, rgb 3 bytes each; TSAR_ERR_ARG when capacity < n_points. */
int tsar_fusion_points(tsar_fusion *f, float *xyz, float *normals, unsigned char *rgb, long long capacity);
int tsar_fusion_destroy(tsar_fusion *f);
const char *tsar_fusion_last_error(const tsar_fusion *f);
/* Resolution rounds of the last run: the most any view needed and the sum over the views (data-dependent). */
int tsar_fusion_dbg_rounds(const tsar_fusion *f, int *max_rounds, long long *total_rounds);

/* ---- cloud-to-cloud evaluation (DESIGN.md section 4.7) ---------------------------------------------------------------
 * Scores a reconstruction R (n points) against a ground truth G (m points), float32 xyz in one frame and unit.
 * dist(q, P) = sqrt_rn(min over the finite p of P of (dx dx + dy dy) + dz dz, d = p - q, float32, one rounding per
 * operation) when that root is <= tau_max, else +inf; +inf for a non-finite q or a P without finite points.
 * within_R[i] = #{r in R : dist(r, G) <= thresholds[i]}, within_G[i] = #{g in G : dist(g, R) <= thresholds[i]}.
 * Accuracy = within_R / n, completeness = within_G / m (tsar-mvs_b200/cloud_eval.py).  This is not the ETH3D or
 * Tanks and Temples evaluator.  A handle of its own; its device scratch only grows, so a second run with clouds no
 * larger than before allocates nothing.  Device memory: 56 B per point of each cloud plus about 2 B per point of tree
 * and the radix-sort scratch. */
#define TSAR_EVAL_MAX_THRESHOLDS 64

typedef struct tsar_eval tsar_eval;

/* `stream` as in tsar_create.  TSAR_ERR_NODEVICE without an sm_100 device. */
int tsar_eval_create(int device, void *stream, tsar_eval **out);
/* Host pointers: recon = n_recon * 3 floats, gt = n_gt * 3 floats (either count may be 0; at most 2^31 - 1 each),
 * thresholds = 1..64 finite values > 0, none above tau_max (finite, > 0).  within_recon / within_gt receive
 * n_thresholds counts each.  dist_recon (n_recon floats) / dist_gt (n_gt floats) receive the per-point distances in
 * input order; NULL = not wanted.  TSAR_ERR_ARG on bad sizes, pointers or thresholds, TSAR_ERR_NOMEM when the clouds
 * do not fit. */
int tsar_eval_run(tsar_eval *e, const float *recon, long long n_recon, const float *gt, long long n_gt,
                  const float *thresholds, int n_thresholds, float tau_max, long long *within_recon,
                  long long *within_gt, float *dist_recon, float *dist_gt);
int tsar_eval_destroy(tsar_eval *e);
const char *tsar_eval_last_error(const tsar_eval *e);
/* Tree leaves visited in the last run, per direction (0 = R against G, 1 = G against R): total over the queries and
 * the most one query visited. */
int tsar_eval_dbg_visits(const tsar_eval *e, long long total[2], int max_per_query[2]);

#ifdef __cplusplus
}
#endif
#endif /* TSAR_B200_H */
