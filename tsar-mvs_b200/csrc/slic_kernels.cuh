// slic_kernels.cuh -- gSLICr superpixel segmentation (north-star item 4), re-designed for sm_100a.
//
// Reference: gSLICr_Lib/engines/gSLICr_seg_engine_GPU.cu + gSLICr_seg_engine_shared.h, sequence
// gSLICr_seg_engine.cpp:30-46.  Labels must be bit-exact against the reference build, which pins three
// things that look like bugs but define the output (SURVEY Q10, Q11):
//   * the cluster update's warp-synchronous reduction tail has no volatile/__syncwarp; nvcc 12.9 loads
//     slots id, id+32, +16, +8, +4, +2, +1 up front and stores once, so block thread 0 ends with
//       ((((((S0+S32)+S16)+S8)+S4)+S2)+S1),   S_k = (o[k]+o[k+128]) + (o[k+64]+o[k+192])
//     i.e. only 28 of the 256 threads' pixels reach each sub-block partial (SASS of the reference build
//     read with tools/sass_trace.py; re-check when the toolkit changes);
//   * the 15 sub-blocks tile 48x80 of the 60x60 search window (no_blocks_per_line = 60/16 = 3);
//   * map size = floor(w/size) x floor(h/size).
// The reference spends 950 x 15 CTAs of 256 threads + a finalise kernel per iteration on this; since only
// 28 fixed slots per sub-block matter, one thread per superpixel does update + finalise here.
// `correct_reduction` switches to the mathematically complete sums (NOT the parity mode).
#pragma once
#include <cuda_runtime.h>

#include "../../include/tsar_b200.h"
#include "dev_mem.h"
#include "pm_math.cuh"

namespace tsar {

struct SpixelInfo {  // the fields of gSLICr::objects::spixel_info (gSLICr_spixel_info.h:10-16); 48 bytes here (float4 alignment)
    float cx, cy;
    float4 color;
    int id;
    int no_pixels;
};

struct SlicState {
    int last_nsp = 0;       // superpixels of the last run (debug read-back)
    DeviceBuf<uchar4> d_in;
    DeviceBuf<float4> d_lab;
    DeviceBuf<int> d_idx, d_tmp;
    DeviceBuf<SpixelInfo> d_sp;
};

// rgb2CIELab (gSLICr_seg_engine_shared.h:30-59); fusion pattern of the reference build: first product
// rounded, the next two fused on top, divisions by the white point IEEE, L = fma(116, fy, -16)
__global__ void slic_cvt_lab_kernel(const uchar4 *__restrict__ in, float4 *__restrict__ out, int w, int h) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const uchar4 p = in[y * w + x];
    const float b = fmul((float)p.x, 0.0039216f), g = fmul((float)p.y, 0.0039216f), r = fmul((float)p.z, 0.0039216f);
    const float X = ffma(b, 0.180423f, ffma(g, 0.357580f, fmul(r, 0.412453f)));
    const float Y = ffma(b, 0.072169f, ffma(g, 0.715160f, fmul(r, 0.212671f)));
    const float Z = ffma(b, 0.950227f, ffma(g, 0.119193f, fmul(r, 0.019334f)));
    const float xr = fdiv(X, 0.950456f), yr = Y, zr = fdiv(Z, 1.088754f);
    const float eps = 0.008856f, kappa = 903.3f;
    const float fx = (xr > eps) ? powf(xr, 1.0f / 3.0f) : fdiv(ffma(kappa, xr, 16.0f), 116.0f);
    const float fy = (yr > eps) ? powf(yr, 1.0f / 3.0f) : fdiv(ffma(kappa, yr, 16.0f), 116.0f);
    const float fz = (zr > eps) ? powf(zr, 1.0f / 3.0f) : fdiv(ffma(kappa, zr, 16.0f), 116.0f);
    out[y * w + x] = make_float4(ffma(116.0f, fy, -16.0f), fmul(500.0f, fsub(fx, fy)), fmul(200.0f, fsub(fy, fz)), 0.0f);
}

// init_cluster_centers_shared (shared.h:73-90)
__global__ void slic_init_centers_kernel(const float4 *__restrict__ lab, SpixelInfo *__restrict__ sp, int mw, int mh,
                                         int w, int h, int size) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= mw || y >= mh) return;
    int ix = x * size + size / 2, iy = y * size + size / 2;
    ix = ix >= w ? (x * size + w) / 2 : ix;
    iy = iy >= h ? (y * size + h) / 2 : iy;
    SpixelInfo s;
    s.id = y * mw + x;
    s.cx = (float)ix; s.cy = (float)iy;
    s.color = lab[iy * w + ix];
    s.no_pixels = 0;
    sp[s.id] = s;
}

// find_center_association_shared + compute_slic_distance (shared.h:92-134): argmin over the 3x3 neighbouring
// centres, strict <, first wins.  The <= 9 candidate centres are read straight from global memory (32-byte records,
// a few hundred of them: they live in L1/L2; the kernel takes 14 us at C2).
__global__ void slic_assign_kernel(const float4 *__restrict__ lab, const SpixelInfo *__restrict__ sp, int *__restrict__ idx,
                                   int mw, int mh, int w, int h, int size, float weight, float norm_xy) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const float4 pix = lab[y * w + x];
    const int cx = x / size, cy = y / size;
    int minidx = -1;
    float dist = 999999.9999f;
    for (int i = -1; i <= 1; i++)
        for (int j = -1; j <= 1; j++) {
            const int xx = cx + j, yy = cy + i;
            if (xx >= 0 && yy >= 0 && xx < mw && yy < mh) {
                const SpixelInfo c = sp[yy * mw + xx];
                const float d0 = fsub(pix.x, c.color.x), d1 = fsub(pix.y, c.color.y), d2 = fsub(pix.z, c.color.z);
                // contraction as compiled in all nine unrolled candidates of the reference build (SASS of
                // Find_Center_Association_device): the MIDDLE square is rounded first and the others fused on top, like every
                // 3-term sum of products there; of two squares the second is rounded first.  A last-ulp matter that decides
                // exact ties only (piecewise-constant images) -- found by tools/gpu_slic_sweep.py in round 2.
                const float dcolor = __fsqrt_rn(ffma(d2, d2, ffma(d0, d0, fmul(d1, d1))));
                const float ex = fsub((float)x, c.cx), ey = fsub((float)y, c.cy);
                const float dxy = __fsqrt_rn(ffma(ex, ex, fmul(ey, ey)));
                const float t = fmul(fmul(dxy, norm_xy), weight);
                const float cd = __fsqrt_rn(ffma(dcolor, dcolor, fmul(t, t)));
                if (cd < dist) { dist = cd; minidx = c.id; }
            }
        }
    if (minidx >= 0) idx[y * w + x] = minidx;
}

// Update_Cluster_Center_device + Finalize_Reduction_Result_device (GPU.cu:260-369, shared.h:153-175), parity mode.
// Of the 256 slots of a 16x16 sub-block only 28 reach thread 0's result in the compiled reference (SURVEY Q10):
// slots k, k+128, k+64, k+192 for k in {0, 32, 16, 8, 4, 2, 1}, summed as ((o_k + o_k+128) + (o_k+64 + o_k+192)) and then
// chained in that order of k.  One warp per superpixel: lane 4*q + part loads slot (k_q, part); two xor-shuffles
// form the four-slot sums with exactly that association (float addition is commutative), lane 0 chains the seven of
// them and accumulates over the sub-blocks in order.
__global__ void slic_update_parity_kernel(const float4 *__restrict__ lab, const int *__restrict__ idx,
                                          SpixelInfo *__restrict__ sp, int mw, int mh, int w, int h, int size,
                                          int nblocks, int nbpl) {
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= mw * mh) return;  // whole warps
    const int sx = s % mw, sy = s / mw;
    const int x_start = sx * size - size, y_start = sy * size - size;
    const int q = lane >> 2, part = lane & 3;
    const int kq = q == 0 ? 0 : (64 >> q);                          // 0, 32, 16, 8, 4, 2, 1 (q = 7: unused lanes)
    const int off = part == 0 ? 0 : (part == 1 ? 128 : (part == 2 ? 64 : 192));
    const int id = kq + off;
    float ccx = 0.f, ccy = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f;
    int count = 0;
    for (int z = 0; z < nblocks; z++) {
        const int bx = z % nbpl, by = z / nbpl;
        float o[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        int hit = 0;
        const int xo = bx * 16 + (id & 15), yo = by * 16 + (id >> 4);
        if (q < 7 && xo < size * 3 && yo < size * 3) {
            const int xi = x_start + xo, yi = y_start + yo;
            if (xi >= 0 && xi < w && yi >= 0 && yi < h && idx[yi * w + xi] == s) {
                const float4 c = lab[yi * w + xi];
                o[0] = c.x; o[1] = c.y; o[2] = c.z; o[3] = (float)xi; o[4] = (float)yi;
                hit = 1;
            }
        }
        count += __popc(__ballot_sync(0xffffffffu, hit));
#pragma unroll
        for (int e = 0; e < 5; e++) {
            float v = fadd(o[e], __shfl_xor_sync(0xffffffffu, o[e], 1));   // (o_k + o_k+128) | (o_k+64 + o_k+192)
            v = fadd(v, __shfl_xor_sync(0xffffffffu, v, 2));               // S[q] on every lane of the group
            float a = v;                                                   // lane 0: S[0]
#pragma unroll
            for (int g = 1; g < 7; g++) a = fadd(a, __shfl_sync(0xffffffffu, v, 4 * g));
            o[e] = a;                                                      // meaningful on lane 0
        }
        c0 = fadd(c0, o[0]); c1 = fadd(c1, o[1]); c2 = fadd(c2, o[2]);
        ccx = fadd(ccx, o[3]); ccy = fadd(ccy, o[4]);
    }
    if (lane != 0) return;
    SpixelInfo out = sp[s];
    out.no_pixels = count;
    if (count != 0) {
        const float n = (float)count;
        out.cx = fdiv(ccx, n); out.cy = fdiv(ccy, n);
        out.color = make_float4(fdiv(c0, n), fdiv(c1, n), fdiv(c2, n), 0.f);
    } else {
        out.cx = 0.f; out.cy = 0.f; out.color = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    sp[s] = out;
}

// complete sums over the 3*size window: one warp per superpixel, shuffle reduction (not the parity mode)
__global__ void slic_update_full_kernel(const float4 *__restrict__ lab, const int *__restrict__ idx,
                                        SpixelInfo *__restrict__ sp, int mw, int mh, int w, int h, int size) {
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= mw * mh) return;
    const int sx = s % mw, sy = s / mw, win = 3 * size;
    const int x_start = sx * size - size, y_start = sy * size - size;
    float a[5] = {0, 0, 0, 0, 0};
    int cnt = 0;
    for (int t = lane; t < win * win; t += 32) {
        const int xi = x_start + t % win, yi = y_start + t / win;
        if (xi >= 0 && xi < w && yi >= 0 && yi < h && idx[yi * w + xi] == s) {
            const float4 c = lab[yi * w + xi];
            a[0] += c.x; a[1] += c.y; a[2] += c.z; a[3] += (float)xi; a[4] += (float)yi; cnt++;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int e = 0; e < 5; e++) a[e] += __shfl_down_sync(0xffffffffu, a[e], o);
        cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    }
    if (lane == 0) {
        SpixelInfo out = sp[s];
        out.no_pixels = cnt;
        if (cnt) { const float n = (float)cnt; out.cx = a[3] / n; out.cy = a[4] / n; out.color = make_float4(a[0] / n, a[1] / n, a[2] / n, 0.f); }
        else { out.cx = out.cy = 0.f; out.color = make_float4(0.f, 0.f, 0.f, 0.f); }
        sp[s] = out;
    }
}

// supress_local_lable (shared.h:177-205)
__global__ void slic_enforce_kernel(const int *__restrict__ in, int *__restrict__ out, int w, int h) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const int c = in[y * w + x];
    if (x <= 1 || y <= 1 || x >= w - 2 || y >= h - 2) { out[y * w + x] = c; return; }
    int diff = 0, dl = -1;
    for (int j = -2; j <= 2; j++)
        for (int i = -2; i <= 2; i++) {
            const int n = in[(y + j) * w + x + i];
            if (n != c) { dl = n; diff++; }
        }
    out[y * w + x] = diff >= 16 ? dl : c;
}

// seg_engine::Perform_Segmentation (gSLICr_seg_engine.cpp:30-46) + Get_Seg_Mask.  Returns a tsar_status; the message of a
// failure goes to hc.err.
static inline int slic_run(HandleCore &hc, SlicState &st, const unsigned char *bgrx, const tsar_slic_settings &cfg,
                           int *labels_out, cudaStream_t stream, int *n_launches) {
    *n_launches = 0;
    const int w = cfg.img_w, h = cfg.img_h, size = cfg.spixel_size;
    if (w <= 0 || h <= 0 || size <= 0 || cfg.no_iters < 0) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: bad settings");
    const int mw = w / size, mh = h / size;  // (int)ceil(int/int): the division truncates first (GPU.cu:74-75)
    if (mw < 1 || mh < 1) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: image smaller than one superpixel");
    const int npx = w * h, nsp = mw * mh;
    st.last_nsp = nsp;
    TSAR_CK(&hc, st.d_in.reserve(npx));
    TSAR_CK(&hc, st.d_lab.reserve(npx));
    TSAR_CK(&hc, st.d_idx.reserve(npx));
    TSAR_CK(&hc, st.d_tmp.reserve(npx));
    TSAR_CK(&hc, st.d_sp.reserve(nsp));
    const int nblocks = (int)ceilf((float)(size * size * 9) / 256.0f);  // no_grid_per_center (GPU.cu:80-82)
    const int nbpl = size * 3 / 16;                                     // no_blocks_per_line (GPU.cu:160)
    if (nbpl < 1) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: spixel_size below 6 is not supported by the reference's block tiling");
    const float norm_xy = 1.0f / size;                                  // max_xy_dist (GPU.cu:88)
    if (cudaMemcpyAsync(st.d_in.get(), bgrx, (size_t)npx * 4, cudaMemcpyHostToDevice, stream)) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: H2D failed");
    cudaMemsetAsync(st.d_idx.get(), 0, (size_t)npx * 4, stream);
    dim3 b(16, 16), gp((w + 15) / 16, (h + 15) / 16), gm((mw + 15) / 16, (mh + 15) / 16);
    slic_cvt_lab_kernel<<<gp, b, 0, stream>>>(st.d_in.get(), st.d_lab.get(), w, h);
    slic_init_centers_kernel<<<gm, b, 0, stream>>>(st.d_lab.get(), st.d_sp.get(), mw, mh, w, h, size);
    slic_assign_kernel<<<gp, b, 0, stream>>>(st.d_lab.get(), st.d_sp.get(), st.d_idx.get(), mw, mh, w, h, size, cfg.coh_weight, norm_xy);
    *n_launches += 3;
    for (int it = 0; it < cfg.no_iters; it++) {
        if (cfg.correct_reduction)
            slic_update_full_kernel<<<(nsp * 32 + 127) / 128, 128, 0, stream>>>(st.d_lab.get(), st.d_idx.get(), st.d_sp.get(), mw, mh, w, h, size);
        else
            slic_update_parity_kernel<<<(nsp * 32 + 127) / 128, 128, 0, stream>>>(st.d_lab.get(), st.d_idx.get(), st.d_sp.get(), mw, mh, w, h, size, nblocks, nbpl);
        slic_assign_kernel<<<gp, b, 0, stream>>>(st.d_lab.get(), st.d_sp.get(), st.d_idx.get(), mw, mh, w, h, size, cfg.coh_weight, norm_xy);
        *n_launches += 2;
    }
    if (cfg.do_enforce_connectivity) {
        slic_enforce_kernel<<<gp, b, 0, stream>>>(st.d_idx.get(), st.d_tmp.get(), w, h);
        slic_enforce_kernel<<<gp, b, 0, stream>>>(st.d_tmp.get(), st.d_idx.get(), w, h);
        *n_launches += 2;
    }
    if (cudaGetLastError() != cudaSuccess) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: kernel launch failed");
    if (cudaMemcpyAsync(labels_out, st.d_idx.get(), (size_t)npx * 4, cudaMemcpyDeviceToHost, stream)) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: D2H failed");
    if (cudaStreamSynchronize(stream) != cudaSuccess) TSAR_FAIL(&hc, TSAR_ERR_CUDA, "tsar_slic: execution failed");
    return TSAR_OK;
}

}  // namespace tsar
