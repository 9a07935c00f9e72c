/*
 * oracle/fusion_cpu.c -- TEST INFRASTRUCTURE, not product code.
 *
 * Plain-C, single-threaded restatement of the multi-view fusion rule of DESIGN.md section 4.6, the independent check of
 * tsar-mvs_b200/csrc/fusion.cu.  Built like oracle_cpu.c with -ffp-contract=off, so every float operation below is one
 * IEEE operation in the written order, as the kernels spell them with explicit-rounding intrinsics.
 */
#include <math.h>
#include <stdlib.h>

#include "../include/tsar_b200.h" /* tsar_view_camera, tsar_fusion_params */

/* The rule written literally: masks, the view loop and the raster loop.  Shares no logic with the parallel resolution
 * of fusion.cu.  The three output arrays are malloc'ed; release them with oc_free. */
typedef struct { float K[9], Kinv[9], R[9], t[3]; } oc_fcam;

static float oc_dot3s(float a0, float b0, float a1, float b1, float a2, float b2) { return a0 * b0 + a1 * b1 + a2 * b2; }
static int oc_valid_depth(float d) { return d > 0.0f && d <= 3.402823466e38f; }

static void oc_backproject(const oc_fcam *c, float x, float y, float d, float *X) {
    const float rx = c->Kinv[0] * x + c->Kinv[1] * y + c->Kinv[2];
    const float ry = c->Kinv[3] * x + c->Kinv[4] * y + c->Kinv[5];
    const float rz = c->Kinv[6] * x + c->Kinv[7] * y + c->Kinv[8];
    const float cx = d * rx - c->t[0], cy = d * ry - c->t[1], cz = d * rz - c->t[2];
    X[0] = oc_dot3s(c->R[0], cx, c->R[3], cy, c->R[6], cz);
    X[1] = oc_dot3s(c->R[1], cx, c->R[4], cy, c->R[7], cz);
    X[2] = oc_dot3s(c->R[2], cx, c->R[5], cy, c->R[8], cz);
}

static void oc_project(const oc_fcam *c, const float *X, float *px, float *py, float *z) {
    const float cx = oc_dot3s(c->R[0], X[0], c->R[1], X[1], c->R[2], X[2]) + c->t[0];
    const float cy = oc_dot3s(c->R[3], X[0], c->R[4], X[1], c->R[5], X[2]) + c->t[1];
    const float cz = oc_dot3s(c->R[6], X[0], c->R[7], X[1], c->R[8], X[2]) + c->t[2];
    *z = cz;
    *px = oc_dot3s(c->K[0], cx, c->K[1], cy, c->K[2], cz) / cz;
    *py = oc_dot3s(c->K[3], cx, c->K[4], cy, c->K[5], cz) / cz;
}

static float oc_norm3(const float *n) { return sqrtf(oc_dot3s(n[0], n[0], n[1], n[1], n[2], n[2])); }

long long oc_fuse(int n_views, int W, int H, const tsar_view_camera *cams, const float *const *depth,
                  const float *const *normals, const unsigned char *const *bgr, const int *const *neighbours,
                  const int *n_neighbours, const tsar_fusion_params *prm, float **xyz_out, float **nrm_out,
                  unsigned char **rgb_out) {
    const size_t P = (size_t)W * H;
    oc_fcam *fc = (oc_fcam *)malloc(sizeof(oc_fcam) * (size_t)n_views);
    unsigned char *mask = (unsigned char *)calloc((size_t)n_views * P, 1);
    size_t cap = 1024, n = 0;
    float *xyz = (float *)malloc(cap * 12), *nrm = (float *)malloc(cap * 12);
    unsigned char *rgb = (unsigned char *)malloc(cap * 3);
    for (int v = 0; v < n_views; ++v) {
        double m[9], a[9];
        for (int i = 0; i < 9; ++i) m[i] = cams[v].K[i];
        a[0] = m[4] * m[8] - m[5] * m[7]; a[1] = m[2] * m[7] - m[1] * m[8]; a[2] = m[1] * m[5] - m[2] * m[4];
        a[3] = m[5] * m[6] - m[3] * m[8]; a[4] = m[0] * m[8] - m[2] * m[6]; a[5] = m[2] * m[3] - m[0] * m[5];
        a[6] = m[3] * m[7] - m[4] * m[6]; a[7] = m[1] * m[6] - m[0] * m[7]; a[8] = m[0] * m[4] - m[1] * m[3];
        const double det = m[0] * a[0] + m[1] * a[3] + m[2] * a[6];
        for (int i = 0; i < 9; ++i) {
            fc[v].K[i] = cams[v].K[i];
            fc[v].Kinv[i] = (float)(a[i] / det);
            fc[v].R[i] = cams[v].R[i];
        }
        for (int i = 0; i < 3; ++i) fc[v].t[i] = cams[v].t[i];
    }
    const float cos_n = (float)cos((double)prm->max_normal_deg * (3.14159265358979323846 / 180.0));
    int E_j[TSAR_FUSION_MAX_NEIGHBOURS], E_q[TSAR_FUSION_MAX_NEIGHBOURS];
    for (int v = 0; v < n_views; ++v) {
        const int *S = neighbours[v];
        const int nS = n_neighbours[v];
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x) {
                const size_t p = (size_t)y * W + x;
                const float d = depth[v][p];
                if (mask[(size_t)v * P + p] || !oc_valid_depth(d)) continue;
                const float *nv = normals[v] + 3 * p;
                float X[3];
                oc_backproject(&fc[v], (float)x, (float)y, d, X);
                int nE = 0;
                for (int j = 0; j < nS; ++j) {
                    const int u = S[j];
                    float px, py, z;
                    oc_project(&fc[u], X, &px, &py, &z);
                    if (!(z > 0.0f)) continue;
                    const float qx = floorf(px + 0.5f), qy = floorf(py + 0.5f);
                    if (!(qx >= 0.0f && qx < (float)W && qy >= 0.0f && qy < (float)H)) continue;
                    const size_t q = (size_t)qy * W + (size_t)qx;
                    if (mask[(size_t)u * P + q] || !oc_valid_depth(depth[u][q])) continue;
                    const float *nu = normals[u] + 3 * q;
                    float Y[3], rx, ry, rz;
                    oc_backproject(&fc[u], qx, qy, depth[u][q], Y);
                    oc_project(&fc[v], Y, &rx, &ry, &rz);
                    const float dx = rx - (float)x, dy = ry - (float)y;
                    if (!(sqrtf(dx * dx + dy * dy) < prm->max_reproj_px)) continue;
                    if (!(fabsf(rz - d) < prm->max_rel_depth * d)) continue;
                    if (!(oc_dot3s(nv[0], nu[0], nv[1], nu[1], nv[2], nu[2]) >= cos_n * oc_norm3(nv) * oc_norm3(nu))) continue;
                    E_j[nE] = j;
                    E_q[nE] = (int)q;
                    ++nE;
                }
                if (nE < prm->min_consistent) continue;
                float s[3] = {X[0], X[1], X[2]}, ns[3] = {nv[0], nv[1], nv[2]};
                int col[3] = {bgr[v][3 * p], bgr[v][3 * p + 1], bgr[v][3 * p + 2]};
                for (int e = 0; e < nE; ++e) {
                    const int u = S[E_j[e]], q = E_q[e];
                    float Y[3];
                    mask[(size_t)u * P + q] = 1;
                    oc_backproject(&fc[u], (float)(q % W), (float)(q / W), depth[u][q], Y);
                    for (int i = 0; i < 3; ++i) {
                        s[i] = s[i] + Y[i];
                        ns[i] = ns[i] + normals[u][3 * (size_t)q + i];
                        col[i] += bgr[u][3 * (size_t)q + i];
                    }
                }
                if (n == cap) {
                    cap *= 2;
                    xyz = (float *)realloc(xyz, cap * 12);
                    nrm = (float *)realloc(nrm, cap * 12);
                    rgb = (unsigned char *)realloc(rgb, cap * 3);
                }
                const int k = nE + 1;
                const float len = oc_norm3(ns);
                const int usable = len > 0.0f && len <= 3.402823466e38f;
                for (int i = 0; i < 3; ++i) {
                    xyz[3 * n + i] = s[i] / (float)k;
                    nrm[3 * n + i] = usable ? ns[i] / len : 0.0f;
                    rgb[3 * n + i] = (unsigned char)((2 * col[2 - i] + k) / (2 * k));
                }
                ++n;
            }
    }
    free(fc);
    free(mask);
    *xyz_out = xyz;
    *nrm_out = nrm;
    *rgb_out = rgb;
    return (long long)n;
}

void oc_free(void *p) { free(p); }
