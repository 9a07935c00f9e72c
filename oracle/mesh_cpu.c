/*
 * oracle/mesh_cpu.c -- TEST INFRASTRUCTURE, not product code.
 *
 * Plain-C restatement of the mesh rule of DESIGN.md section 4.8 (TSDF integration + marching tetrahedra on the
 * Freudenthal split), the independent check of tsar-mvs_b200/csrc/mesh.cu.  Built like fusion_cpu.c with
 * -ffp-contract=off, so every float operation below is one IEEE operation in the written order.  Integration is
 * parallel over grid points (OpenMP); each point's view loop is sequential.  Extraction is a literal sequential loop.
 * Nothing is shared with mesh.cu but the header; the tetrahedra and their triangles are derived here from the axis
 * permutations and the even-permutation rule, not from a table.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../include/tsar_b200.h" /* tsar_view_camera, tsar_mesh_grid */

static float oc_dot3s(float a0, float b0, float a1, float b1, float a2, float b2) { return a0 * b0 + a1 * b1 + a2 * b2; }
static int oc_valid_depth(float d) { return d > 0.0f && d <= 3.402823466e38f; }

static void oc_project(const tsar_view_camera *c, const float *X, float *px, float *py, float *z) {
    const float cx = oc_dot3s(c->R[0], X[0], c->R[1], X[1], c->R[2], X[2]) + c->t[0];
    const float cy = oc_dot3s(c->R[3], X[0], c->R[4], X[1], c->R[5], X[2]) + c->t[1];
    const float cz = oc_dot3s(c->R[6], X[0], c->R[7], X[1], c->R[8], X[2]) + c->t[2];
    *z = cz;
    *px = oc_dot3s(c->K[0], cx, c->K[1], cy, c->K[2], cz) / cz;
    *py = oc_dot3s(c->K[3], cx, c->K[4], cy, c->K[5], cz) / cz;
}

static float oc_coord(const tsar_mesh_grid *g, int axis, int i) { return g->origin[axis] + ((float)i + 0.5f) * g->voxel; }

/* The field: F = S / W where W >= 1 (else 0), W, Wc and the B, G, R sums of every grid point. */
void oc_mesh_field(int n_views, int Wd, int Hd, const tsar_view_camera *cams, const float *const *depth,
                   const unsigned char *const *bgr, const tsar_mesh_grid *g, float trunc, float *F, uint16_t *Wt,
                   uint16_t *Wc, uint32_t *sum) {
    const int nx = g->dims[0], ny = g->dims[1], nz = g->dims[2];
    const long long n = (long long)nx * ny * nz;
#pragma omp parallel for schedule(dynamic, 4096)
    for (long long p = 0; p < n; ++p) {
        const int i = (int)(p % nx), j = (int)(p / nx % ny), k = (int)(p / ((long long)nx * ny));
        const float X[3] = {oc_coord(g, 0, i), oc_coord(g, 1, j), oc_coord(g, 2, k)};
        float S = 0.0f;
        unsigned w = 0, wc = 0, s[3] = {0, 0, 0};
        for (int v = 0; v < n_views; ++v) {
            float px, py, z;
            oc_project(&cams[v], X, &px, &py, &z);
            if (!(z > 0.0f)) continue;
            const float qx = floorf(px + 0.5f), qy = floorf(py + 0.5f);
            if (!(qx >= 0.0f && qx < (float)Wd && qy >= 0.0f && qy < (float)Hd)) continue;
            const size_t q = (size_t)qy * Wd + (size_t)qx;
            const float D = depth[v][q];
            if (!oc_valid_depth(D)) continue;
            const float sdf = D - z;
            if (sdf < -trunc) continue;
            S = S + fminf(1.0f, sdf / trunc);
            w += 1;
            if (sdf <= trunc) {
                for (int c = 0; c < 3; ++c) s[c] += bgr[v][3 * q + c];
                wc += 1;
            }
        }
        F[p] = w >= 1 ? S / (float)w : 0.0f;
        Wt[p] = (uint16_t)w;
        Wc[p] = (uint16_t)wc;
        for (int c = 0; c < 3; ++c) sum[3 * p + c] = s[c];
    }
}

typedef struct {
    const tsar_mesh_grid *g;
    int min_weight;
    const float *F;
    const uint16_t *W;
} oc_field;

static long long oc_index(const oc_field *f, int i, int j, int k) {
    return ((long long)k * f->g->dims[1] + j) * f->g->dims[0] + i;
}
static int oc_in_grid(const oc_field *f, int i, int j, int k) {
    return i >= 0 && j >= 0 && k >= 0 && i < f->g->dims[0] && j < f->g->dims[1] && k < f->g->dims[2];
}
static int oc_defined(const oc_field *f, long long p) { return f->W[p] >= f->min_weight; }
static int oc_inside(const oc_field *f, long long p) { return oc_defined(f, p) && f->F[p] < 0.0f; }

/* Cell (i, j, k) exists and its 8 corners are defined. */
static int oc_complete(const oc_field *f, int i, int j, int k) {
    if (!oc_in_grid(f, i, j, k) || !oc_in_grid(f, i + 1, j + 1, k + 1)) return 0;
    for (int dz = 0; dz <= 1; ++dz)
        for (int dy = 0; dy <= 1; ++dy)
            for (int dx = 0; dx <= 1; ++dx)
                if (!oc_defined(f, oc_index(f, i + dx, j + dy, k + dz))) return 0;
    return 1;
}

static const int OC_DELTA[7][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {1, 1, 0}, {1, 0, 1}, {0, 1, 1}, {1, 1, 1}};
static const int OC_PERM[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};  /* xyz ... zyx */

static int oc_even(const int *p, int n) {
    int inv = 0;
    for (int a = 0; a < n; ++a)
        for (int b = a + 1; b < n; ++b) inv += p[a] > p[b];
    return inv % 2 == 0;
}

/* Orders the corners of a tetrahedron as (lead..., rest...): `lead` in the given order, then the first ordering of
 * the remaining corners in lexicographic order for which the whole sequence is an even permutation of (0, 1, 2, 3). */
static void oc_even_order(const int *lead, int n_lead, int *out) {
    int rest[4], nr = 0;
    for (int c = 0; c < 4; ++c) {
        int used = 0;
        for (int l = 0; l < n_lead; ++l) used |= lead[l] == c;
        if (!used) rest[nr++] = c;
    }
    for (int l = 0; l < n_lead; ++l) out[l] = lead[l];
    /* nr <= 3: orderings of rest in lexicographic order (rest is ascending) */
    static const int ORD3[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
    static const int ORD2[2][2] = {{0, 1}, {1, 0}};
    const int n_ord = nr == 3 ? 6 : 2;
    for (int o = 0; o < n_ord; ++o) {
        for (int r = 0; r < nr; ++r) out[n_lead + r] = rest[nr == 3 ? ORD3[o][r] : ORD2[o][r]];
        if (oc_even(out, 4)) return;
    }
}

long long oc_mesh_extract(const tsar_mesh_grid *g, int min_weight, const float *F, const uint16_t *W, const uint16_t *Wc,
                          const uint32_t *sum, float **xyz_out, unsigned char **rgb_out, int **tri_out,
                          long long *n_tri_out) {
    const oc_field f = {g, min_weight, F, W};
    const int nx = g->dims[0], ny = g->dims[1], nz = g->dims[2];
    const long long n = (long long)nx * ny * nz;
    int *vid = (int *)malloc(sizeof(int) * 7 * (size_t)n);
    size_t vcap = 1024, nv = 0, tcap = 1024, nt = 0;
    float *xyz = (float *)malloc(vcap * 12);
    unsigned char *rgb = (unsigned char *)malloc(vcap * 3);
    int *tri = (int *)malloc(tcap * 12);
    /* vertices: lattice points in linear order, then delta in order */
    for (int k = 0; k < nz; ++k)
        for (int j = 0; j < ny; ++j)
            for (int i = 0; i < nx; ++i) {
                const long long a = oc_index(&f, i, j, k);
                for (int d = 0; d < 7; ++d) {
                    vid[7 * a + d] = -1;
                    const int bi = i + OC_DELTA[d][0], bj = j + OC_DELTA[d][1], bk = k + OC_DELTA[d][2];
                    if (!oc_in_grid(&f, bi, bj, bk)) continue;
                    const long long b = oc_index(&f, bi, bj, bk);
                    if (oc_inside(&f, a) + oc_inside(&f, b) != 1) continue;
                    int edge_of_complete_cell = 0;
                    for (int ck = k - 1; ck <= k; ++ck)
                        for (int cj = j - 1; cj <= j; ++cj)
                            for (int ci = i - 1; ci <= i; ++ci)
                                if (ci <= bi && bi <= ci + 1 && cj <= bj && bj <= cj + 1 && ck <= bk && bk <= ck + 1 &&
                                    oc_complete(&f, ci, cj, ck))
                                    edge_of_complete_cell = 1;
                    if (!edge_of_complete_cell) continue;
                    if (nv == vcap) {
                        vcap *= 2;
                        xyz = (float *)realloc(xyz, vcap * 12);
                        rgb = (unsigned char *)realloc(rgb, vcap * 3);
                    }
                    const float Fa = F[a], Fb = F[b];
                    const float t = Fa / (Fa - Fb);
                    const int ia[3] = {i, j, k}, ib[3] = {bi, bj, bk};
                    for (int ax = 0; ax < 3; ++ax) {
                        const float pa = oc_coord(g, ax, ia[ax]), pb = oc_coord(g, ax, ib[ax]);
                        xyz[3 * nv + ax] = pa + t * (pb - pa);
                    }
                    long long src = a;
                    if (Wc[a] == 0 || (Wc[b] > 0 && fabsf(Fb) < fabsf(Fa))) src = b;
                    const unsigned wc = Wc[src];
                    rgb[3 * nv] = (unsigned char)((2 * sum[3 * src + 2] + wc) / (2 * wc));
                    rgb[3 * nv + 1] = (unsigned char)((2 * sum[3 * src + 1] + wc) / (2 * wc));
                    rgb[3 * nv + 2] = (unsigned char)((2 * sum[3 * src] + wc) / (2 * wc));
                    vid[7 * a + d] = (int)nv;
                    ++nv;
                }
            }
    /* triangles: complete cells in linear order, tetrahedra in permutation order */
    int bad = 0;
    for (int k = 0; k + 1 < nz; ++k)
        for (int j = 0; j + 1 < ny; ++j)
            for (int i = 0; i + 1 < nx; ++i) {
                if (!oc_complete(&f, i, j, k)) continue;
                for (int t = 0; t < 6; ++t) {
                    int corner[4][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {1, 1, 1}};
                    corner[1][OC_PERM[t][0]] = 1;
                    corner[2][OC_PERM[t][0]] = 1;
                    corner[2][OC_PERM[t][1]] = 1;
                    const int odd = !oc_even(OC_PERM[t], 3);
                    int in[4], n_in = 0;
                    for (int r = 0; r < 4; ++r) {
                        in[r] = oc_inside(&f, oc_index(&f, i + corner[r][0], j + corner[r][1], k + corner[r][2]));
                        n_in += in[r];
                    }
                    if (n_in == 0 || n_in == 4) continue;
                    int e[4][2], ne = 0, ord[4];  /* polygon as a cycle of tetrahedron edges */
                    if (n_in == 1 || n_in == 3) {
                        int s = 0;
                        while (in[s] != (n_in == 1)) ++s;   /* the corner alone on its side */
                        oc_even_order(&s, 1, ord);
                        const int c1 = n_in == 1 ? ord[2] : ord[3], c2 = n_in == 1 ? ord[3] : ord[2];
                        e[0][0] = s; e[0][1] = ord[1];
                        e[1][0] = s; e[1][1] = c1;
                        e[2][0] = s; e[2][1] = c2;
                        ne = 3;
                    } else {
                        int lead[2], nl = 0;
                        for (int r = 0; r < 4; ++r)
                            if (in[r]) lead[nl++] = r;
                        oc_even_order(lead, 2, ord);     /* (i, j, k, l): i < j inside */
                        e[0][0] = ord[0]; e[0][1] = ord[2];
                        e[1][0] = ord[0]; e[1][1] = ord[3];
                        e[2][0] = ord[1]; e[2][1] = ord[3];
                        e[3][0] = ord[1]; e[3][1] = ord[2];
                        ne = 4;
                    }
                    int id[4];
                    for (int q = 0; q < ne; ++q) {
                        const int *u = corner[e[q][0]], *w = corner[e[q][1]];
                        const int u_low = u[0] + u[1] + u[2] < w[0] + w[1] + w[2];
                        const int *lo = u_low ? u : w, *hi = u_low ? w : u;
                        int d = 0;
                        while (!(OC_DELTA[d][0] == hi[0] - lo[0] && OC_DELTA[d][1] == hi[1] - lo[1] && OC_DELTA[d][2] == hi[2] - lo[2])) ++d;
                        id[q] = vid[7 * oc_index(&f, i + lo[0], j + lo[1], k + lo[2]) + d];
                        bad |= id[q] < 0;
                    }
                    for (int s2 = 0; s2 + 2 < ne; ++s2) {  /* fan from q0: (q0, q1, q2), (q0, q2, q3) */
                        if (nt == tcap) {
                            tcap *= 2;
                            tri = (int *)realloc(tri, tcap * 12);
                        }
                        tri[3 * nt] = id[0];
                        tri[3 * nt + 1] = odd ? id[s2 + 2] : id[s2 + 1];
                        tri[3 * nt + 2] = odd ? id[s2 + 1] : id[s2 + 2];
                        ++nt;
                    }
                }
            }
    free(vid);
    *xyz_out = xyz;
    *rgb_out = rgb;
    *tri_out = tri;
    *n_tri_out = bad ? -1 : (long long)nt;
    return (long long)nv;
}

long long oc_mesh(int n_views, int Wd, int Hd, const tsar_view_camera *cams, const float *const *depth,
                  const unsigned char *const *bgr, const tsar_mesh_grid *g, float trunc, int min_weight, float **xyz_out,
                  unsigned char **rgb_out, int **tri_out, long long *n_tri_out) {
    const size_t n = (size_t)g->dims[0] * g->dims[1] * g->dims[2];
    float *F = (float *)malloc(n * sizeof(float));
    uint16_t *Wt = (uint16_t *)malloc(n * sizeof(uint16_t)), *Wc = (uint16_t *)malloc(n * sizeof(uint16_t));
    uint32_t *sum = (uint32_t *)malloc(3 * n * sizeof(uint32_t));
    oc_mesh_field(n_views, Wd, Hd, cams, depth, bgr, g, trunc, F, Wt, Wc, sum);
    const long long nv = oc_mesh_extract(g, min_weight, F, Wt, Wc, sum, xyz_out, rgb_out, tri_out, n_tri_out);
    free(F);
    free(Wt);
    free(Wc);
    free(sum);
    return nv;
}

void oc_free(void *p) { free(p); }
