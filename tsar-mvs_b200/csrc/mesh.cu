// mesh.cu -- a coloured triangle mesh from the per-view depth maps: TSDF integration on a dense voxel grid, then marching
// tetrahedra on the Freudenthal split (DESIGN.md section 4.8).
//
//   1. mesh_integrate_kernel  one thread per grid point (CTA = 8 x 8 x 4 points), the views in order, cameras staged in
//                             shared memory 64 at a time; one 8-byte gather (depth + BGRx) per point and view.
//   2. mesh_cells_kernel      per cell: complete (all 8 corners defined) and the number of triangles of its 6 tetrahedra.
//   3. mesh_vmask_kernel      per lattice point a: bit d set when the edge a -> a + delta_d carries a vertex.
//   4. two CUB exclusive scans give every lattice point its first vertex id and every cell its first triangle.
//   5. mesh_vertices_kernel / mesh_triangles_kernel write the mesh at those offsets, so the output order is the rule's
//      and no atomic decides it.
// Every rounding step is spelled with an explicit-rounding intrinsic so that oracle/mesh_cpu.c, compiled with
// -ffp-contract=off, performs the same operations in the same order.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cub/device/device_scan.cuh>
#include <memory>
#include <string>
#include <thrust/iterator/transform_iterator.h>
#include <vector>

#include "../../include/tsar_b200.h"
#include "dev_mem.h"
#include "pm_math.cuh"
#include "view_project.cuh"

using namespace tsar;

namespace {

struct MeshCam {
    float K[9], R[9], t[3];
};
constexpr int kCamFloats = 21;
constexpr int kCamChunk = 64;
constexpr int kTX = 8, kTY = 8, kTZ = 4;
constexpr int kIntThreads = kTX * kTY * kTZ;
constexpr int kThreads = 256;
constexpr int kMaxDim = 1 << 23;                 // (float)i + 0.5f is exact below 2^23
constexpr long long kMaxPoints = (1LL << 31) - 1;  // grid points and vertices: int32 indices
constexpr unsigned char kComplete = 0x80;        // cell byte: complete flag | number of triangles (0..12)

struct GridArgs {
    float ox, oy, oz, s;
    int nx, ny, nz;
    long long n;
};

// Lattice edges a -> a + delta, delta in the rule's order 100, 010, 001, 110, 101, 011, 111 (bit 0 = x, 1 = y, 2 = z).
__constant__ unsigned char c_delta[7] = {1, 2, 4, 3, 5, 6, 7};
__constant__ unsigned char c_delta_index[8] = {0, 0, 1, 3, 2, 4, 5, 6};  // delta bits -> position in that order
// The six tetrahedra of a cell, one per axis permutation (a, b, c) in the order xyz, xzy, yxz, yzx, zxy, zyx: corners
// 000, e_a, e_a + e_b, 111 (cell corner index = x + 2y + 4z).  Parity = sign of the permutation = sign of the volume.
__constant__ unsigned char c_tet[6][4] = {{0, 1, 3, 7}, {0, 1, 5, 7}, {0, 2, 3, 7}, {0, 2, 6, 7}, {0, 4, 5, 7}, {0, 4, 6, 7}};
__constant__ bool c_tet_odd[6] = {false, true, true, false, false, true};
// Triangles of a positively oriented tetrahedron by inside mask (bit r = corner r inside), as edges (r, s) packed r*4+s;
// their right-hand normal points from the inside corners to the outside ones.  One inside corner i: the edges from i to
// the opposite face in its outward order; three: the same for the outside corner, reversed; two (i, j inside, k, l
// outside, (i, j, k, l) an even permutation): the quad (ik, il, jl, jk), split as (q0, q1, q2), (q0, q2, q3).  An odd
// tetrahedron swaps the last two edges of every triangle.
__constant__ unsigned char c_ntri[16] = {0, 1, 1, 2, 1, 2, 2, 1, 1, 2, 2, 1, 2, 1, 1, 0};
__constant__ unsigned char c_tri[16][2][3] = {
    {{0, 0, 0}, {0, 0, 0}},
    {{1, 2, 3}, {0, 0, 0}},          // {0}:       01 02 03
    {{4, 7, 6}, {0, 0, 0}},          // {1}:       10 13 12
    {{2, 3, 7}, {2, 7, 6}},          // {0,1}:     02 03 13 12
    {{8, 9, 11}, {0, 0, 0}},         // {2}:       20 21 23
    {{3, 1, 9}, {3, 9, 11}},         // {0,2}:     03 01 21 23
    {{4, 7, 11}, {4, 11, 8}},        // {1,2}:     10 13 23 20
    {{12, 13, 14}, {0, 0, 0}},       // {0,1,2}:   30 31 32
    {{12, 14, 13}, {0, 0, 0}},       // {3}:       30 32 31
    {{1, 2, 14}, {1, 14, 13}},       // {0,3}:     01 02 32 31
    {{6, 4, 12}, {6, 12, 14}},       // {1,3}:     12 10 30 32
    {{8, 11, 9}, {0, 0, 0}},         // {0,1,3}:   20 23 21
    {{8, 9, 13}, {8, 13, 12}},       // {2,3}:     20 21 31 30
    {{4, 6, 7}, {0, 0, 0}},          // {0,2,3}:   10 12 13
    {{1, 3, 2}, {0, 0, 0}},          // {1,2,3}:   01 03 02
    {{0, 0, 0}, {0, 0, 0}}};

__device__ __forceinline__ float grid_coord(float o, int i, float s) { return fadd(o, fmul(fadd((float)i, 0.5f), s)); }
__device__ __forceinline__ bool defined(unsigned wts, int min_weight) { return (int)(wts & 0xffffu) >= min_weight; }

__global__ void mesh_pack_kernel(const float *__restrict__ depth, const unsigned char *__restrict__ bgr, size_t P,
                                 uint2 *__restrict__ out) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    out[p] = make_uint2(__float_as_uint(depth[p]), bgr[3 * p] | (unsigned)bgr[3 * p + 1] << 8 | (unsigned)bgr[3 * p + 2] << 16);
}

__global__ void __launch_bounds__(kIntThreads) mesh_integrate_kernel(GridArgs g, int n_views, int W, int H, float trunc,
                                                                     const MeshCam *__restrict__ cams,
                                                                     const uint2 *__restrict__ views, float *__restrict__ F,
                                                                     unsigned *__restrict__ wts, unsigned *__restrict__ csum) {
    __shared__ MeshCam sc[kCamChunk];
    const long long tiles_x = (g.nx + kTX - 1) / kTX, tiles_y = (g.ny + kTY - 1) / kTY;
    const long long tile = blockIdx.x;
    const int i = (int)(tile % tiles_x) * kTX + threadIdx.x % kTX;
    const int j = (int)(tile / tiles_x % tiles_y) * kTY + threadIdx.x / kTX % kTY;
    const int k = (int)(tile / (tiles_x * tiles_y)) * kTZ + threadIdx.x / (kTX * kTY);
    const bool in = i < g.nx && j < g.ny && k < g.nz;
    const float3 X = make_float3(grid_coord(g.ox, i, g.s), grid_coord(g.oy, j, g.s), grid_coord(g.oz, k, g.s));
    const size_t P = (size_t)W * H;
    const float neg_trunc = -trunc;
    float S = 0.0f;
    unsigned w = 0, wc = 0, cb = 0, cg = 0, cr = 0;
    for (int v0 = 0; v0 < n_views; v0 += kCamChunk) {
        const int nc = min(kCamChunk, n_views - v0);
        __syncthreads();
        for (int f = threadIdx.x; f < nc * kCamFloats; f += blockDim.x)
            reinterpret_cast<float *>(sc)[f] = reinterpret_cast<const float *>(cams + v0)[f];
        __syncthreads();
        if (!in) continue;
        for (int c = 0; c < nc; ++c) {
            float px, py, z;
            project(sc[c], X, px, py, z);
            if (!(z > 0.0f)) continue;
            const float qx = floorf(fadd(px, 0.5f)), qy = floorf(fadd(py, 0.5f));
            if (!(qx >= 0.0f && qx < (float)W && qy >= 0.0f && qy < (float)H)) continue;
            const uint2 pix = views[(size_t)(v0 + c) * P + (size_t)qy * W + (size_t)qx];
            const float D = __uint_as_float(pix.x);
            if (!valid_depth(D)) continue;
            const float sdf = fsub(D, z);
            if (sdf < neg_trunc) continue;
            S = fadd(S, fminf(1.0f, fdiv(sdf, trunc)));
            ++w;
            if (sdf <= trunc) {
                cb += pix.y & 255u;
                cg += pix.y >> 8 & 255u;
                cr += pix.y >> 16 & 255u;
                ++wc;
            }
        }
    }
    if (!in) return;
    const size_t p = ((size_t)k * g.ny + j) * g.nx + i;
    F[p] = w ? fdiv(S, (float)w) : 0.0f;
    wts[p] = w | wc << 16;
    csum[3 * p] = cb;
    csum[3 * p + 1] = cg;
    csum[3 * p + 2] = cr;
}

__device__ __forceinline__ long long corner_offset(const GridArgs &g, int c) {
    return (c & 1) + ((c >> 1) & 1) * (long long)g.nx + ((c >> 2) & 1) * (long long)g.nx * g.ny;
}

// Cell p (its 000 corner is grid point p): kComplete | triangles when all 8 corners are defined, else 0.
__global__ void __launch_bounds__(kThreads) mesh_cells_kernel(GridArgs g, int min_weight, const float *__restrict__ F,
                                                              const unsigned *__restrict__ wts, unsigned char *__restrict__ cell) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.n) return;
    const int i = (int)(p % g.nx), j = (int)(p / g.nx % g.ny), k = (int)(p / ((long long)g.nx * g.ny));
    unsigned char out = 0;
    if (i < g.nx - 1 && j < g.ny - 1 && k < g.nz - 1) {
        bool complete = true;
        unsigned inside = 0;
        for (int c = 0; c < 8; ++c) {
            const long long q = p + corner_offset(g, c);
            complete = complete && defined(wts[q], min_weight);
            inside |= (F[q] < 0.0f ? 1u : 0u) << c;
        }
        if (complete) {
            int nt = 0;
            for (int t = 0; t < 6; ++t) {
                unsigned m = 0;
                for (int r = 0; r < 4; ++r) m |= (inside >> c_tet[t][r] & 1u) << r;
                nt += c_ntri[m];
            }
            out = kComplete | nt;
        }
    }
    cell[p] = out;
}

// Bit d of vmask[a]: the edge a -> a + delta_d has exactly one inside endpoint and is an edge of a complete cell.  The
// Freudenthal split makes every monotone pair of corners of a cell an edge, so the cells of that edge are the cells that
// contain both endpoints: corner index a along the axes delta_d moves, a - 1 or a along the others.  A complete cell has
// defined corners, so F < 0 is the rule's inside test at both endpoints.
__global__ void __launch_bounds__(kThreads) mesh_vmask_kernel(GridArgs g, const float *__restrict__ F,
                                                              const unsigned char *__restrict__ cell,
                                                              unsigned char *__restrict__ vmask) {
    const long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= g.n) return;
    const int i = (int)(a % g.nx), j = (int)(a / g.nx % g.ny), k = (int)(a / ((long long)g.nx * g.ny));
    const bool ia = F[a] < 0.0f;
    unsigned mask = 0;
    for (int d = 0; d < 7; ++d) {
        const int db = c_delta[d], di = db & 1, dj = db >> 1 & 1, dk = db >> 2 & 1;
        if (i + di >= g.nx || j + dj >= g.ny || k + dk >= g.nz) continue;
        if ((F[a + corner_offset(g, db)] < 0.0f) == ia) continue;
        bool used = false;
        for (int m = 0; m < 8 && !used; ++m) {
            if (m & db) continue;                      // no step back along an axis the edge moves along
            const int ci = i - (m & 1), cj = j - (m >> 1 & 1), ck = k - (m >> 2 & 1);
            if (ci < 0 || cj < 0 || ck < 0) continue;  // cells past the last plane are stored as 0
            used = cell[((long long)ck * g.ny + cj) * g.nx + ci] & kComplete;
        }
        if (used) mask |= 1u << d;
    }
    vmask[a] = (unsigned char)mask;
}

struct PopCount {
    __device__ long long operator()(unsigned char m) const { return __popc(m); }
};
struct CellTriangles {
    __device__ long long operator()(unsigned char c) const { return c & 0x7f; }
};

__global__ void mesh_totals_kernel(long long n, const unsigned char *__restrict__ vmask, const long long *__restrict__ voff,
                                   const unsigned char *__restrict__ cell, const long long *__restrict__ toff,
                                   long long *__restrict__ tot) {
    tot[0] = voff[n - 1] + PopCount()(vmask[n - 1]);
    tot[1] = toff[n - 1] + CellTriangles()(cell[n - 1]);
}

// The vertices owned by lattice point a, in delta order.  t = Fa / (Fa - Fb); position pa + t (pb - pa) per axis.
// Colour: the endpoint with the smaller |F| among those with Wc > 0, ties to a.  Wc > 0 holds at the inside endpoint:
// F < 0 needs S < 0, so some view added d = fminf(1, sdf / trunc) < 0, i.e. sdf < 0; it also passed sdf >= -trunc, so
// that view had -trunc <= sdf <= trunc and added to Wc.  Hence the chosen endpoint always has Wc >= 1.
__global__ void __launch_bounds__(kThreads) mesh_vertices_kernel(GridArgs g, const float *__restrict__ F,
                                                                 const unsigned *__restrict__ wts,
                                                                 const unsigned *__restrict__ csum,
                                                                 const unsigned char *__restrict__ vmask,
                                                                 const long long *__restrict__ voff,
                                                                 float *__restrict__ xyz, unsigned char *__restrict__ rgb) {
    const long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= g.n) return;
    const unsigned mask = vmask[a];
    if (!mask) return;
    const int i = (int)(a % g.nx), j = (int)(a / g.nx % g.ny), k = (int)(a / ((long long)g.nx * g.ny));
    const float Fa = F[a];
    const float pax = grid_coord(g.ox, i, g.s), pay = grid_coord(g.oy, j, g.s), paz = grid_coord(g.oz, k, g.s);
    const unsigned wca = wts[a] >> 16;
    long long id = voff[a];
    for (int d = 0; d < 7; ++d) {
        if (!(mask >> d & 1u)) continue;
        const int db = c_delta[d], di = db & 1, dj = db >> 1 & 1, dk = db >> 2 & 1;
        const long long b = a + corner_offset(g, db);
        const float Fb = F[b];
        const float t = fdiv(Fa, fsub(Fa, Fb));
        xyz[3 * id] = fadd(pax, fmul(t, fsub(grid_coord(g.ox, i + di, g.s), pax)));
        xyz[3 * id + 1] = fadd(pay, fmul(t, fsub(grid_coord(g.oy, j + dj, g.s), pay)));
        xyz[3 * id + 2] = fadd(paz, fmul(t, fsub(grid_coord(g.oz, k + dk, g.s), paz)));
        const unsigned wcb = wts[b] >> 16;
        const bool use_b = wca == 0 || (wcb > 0 && fabsf(Fb) < fabsf(Fa));
        const long long src = use_b ? b : a;
        const unsigned wc = use_b ? wcb : wca;
        for (int ch = 0; ch < 3; ++ch)   // sums are B, G, R; the output is R, G, B
            rgb[3 * id + ch] = (unsigned char)((2 * csum[3 * src + 2 - ch] + wc) / (2 * wc));
        ++id;
    }
}

// The triangles of cell p, tetrahedron after tetrahedron, at toff[p].  A vertex on the edge between cell corners u, w
// (a monotone pair: one corner's bits contain the other's) is owned by the lower corner and found by the rank of the
// edge's delta among the vertices that corner owns.
__global__ void __launch_bounds__(kThreads) mesh_triangles_kernel(GridArgs g, const float *__restrict__ F,
                                                                  const unsigned char *__restrict__ cell,
                                                                  const unsigned char *__restrict__ vmask,
                                                                  const long long *__restrict__ voff,
                                                                  const long long *__restrict__ toff, int *__restrict__ tri) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.n || !(cell[p] & 0x7f)) return;
    unsigned inside = 0;
    for (int c = 0; c < 8; ++c) inside |= (F[p + corner_offset(g, c)] < 0.0f ? 1u : 0u) << c;
    long long out = toff[p];
    for (int t = 0; t < 6; ++t) {
        unsigned m = 0;
        for (int r = 0; r < 4; ++r) m |= (inside >> c_tet[t][r] & 1u) << r;
        for (int n = 0; n < c_ntri[m]; ++n) {
            int ids[3];
            for (int e = 0; e < 3; ++e) {
                const int edge = c_tri[m][n][e];
                const int u = c_tet[t][edge >> 2], w = c_tet[t][edge & 3];
                const int lo = (u & w) == u ? u : w, hi = u ^ w ^ lo;
                const long long owner = p + corner_offset(g, lo);
                const unsigned below = (1u << c_delta_index[lo ^ hi]) - 1u;
                ids[e] = (int)(voff[owner] + __popc(vmask[owner] & below));
            }
            const bool odd = c_tet_odd[t];
            tri[3 * out] = ids[0];
            tri[3 * out + 1] = ids[odd ? 2 : 1];
            tri[3 * out + 2] = ids[odd ? 1 : 2];
            ++out;
        }
    }
}

unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace

struct tsar_mesh : HandleCore {
    int n_views = 0, W = 0, H = 0;
    size_t P = 0;
    std::vector<char> view_set;
    // resident views: 8 B per pixel and view (depth + BGRx), and the staging buffers of one upload
    DeviceBuf<MeshCam> d_cams;
    DeviceBuf<uint2> d_views;
    DeviceBuf<float> d_stage_depth;
    DeviceBuf<unsigned char> d_stage_bgr;
    // the field: 20 B per grid point
    DeviceBuf<float> d_F;
    DeviceBuf<unsigned> d_wts, d_csum;
    // extraction scratch: 18 B per grid point plus the scan's temporary storage
    DeviceBuf<unsigned char> d_cell, d_vmask, d_cub;
    DeviceBuf<long long> d_voff, d_toff, d_tot;
    // the mesh of the last run
    DeviceBuf<float> d_xyz;
    DeviceBuf<unsigned char> d_rgb;
    DeviceBuf<int> d_tri;
    PinnedBuf<long long> h_tot;
    long long n_field = 0, n_vertices = 0, n_triangles = 0;
    // CUDA events around the integration and the extraction of the last tsar_mesh_run (tsar_mesh_dbg_times)
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    bool timed = false;
    ~tsar_mesh() {
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
    }
};

static const char *check_grid(const tsar_mesh_grid *g, GridArgs *out) {
    if (!g) return "null grid";
    for (int a = 0; a < 3; ++a)
        if (!isfinite(g->origin[a])) return "grid origin is not finite";
    if (!(g->voxel > 0.0f) || !isfinite(g->voxel)) return "voxel must be finite and > 0";
    for (int a = 0; a < 3; ++a)
        if (g->dims[a] < 2 || g->dims[a] > kMaxDim) return "each grid dimension must be in [2, 2^23]";
    const long long n = (long long)g->dims[0] * g->dims[1] * g->dims[2];
    if (n > kMaxPoints) return "the grid has more than 2^31 - 1 points";
    *out = GridArgs{g->origin[0], g->origin[1], g->origin[2], g->voxel, g->dims[0], g->dims[1], g->dims[2], n};
    return nullptr;
}

// Cells, vertex masks, scans and the mesh from the field in d_F / d_wts / d_csum.
static int extract(tsar_mesh *m, const GridArgs &g, int min_weight, long long *n_vertices, long long *n_triangles) {
    const long long n = g.n;
    TSAR_CK(m, m->d_cell.reserve(n));
    TSAR_CK(m, m->d_vmask.reserve(n));
    TSAR_CK(m, m->d_voff.reserve(n));
    TSAR_CK(m, m->d_toff.reserve(n));
    const auto vcount = thrust::make_transform_iterator(m->d_vmask.get(), PopCount());
    const auto tcount = thrust::make_transform_iterator(m->d_cell.get(), CellTriangles());
    size_t tmp_v = 0, tmp_t = 0;
    TSAR_CK(m, cub::DeviceScan::ExclusiveSum(nullptr, tmp_v, vcount, m->d_voff.get(), (int)n, m->stream));
    TSAR_CK(m, cub::DeviceScan::ExclusiveSum(nullptr, tmp_t, tcount, m->d_toff.get(), (int)n, m->stream));
    size_t tmp = std::max(tmp_v, tmp_t);
    TSAR_CK(m, m->d_cub.reserve(tmp));
    const unsigned nb = blocks_for(n, kThreads);
    mesh_cells_kernel<<<nb, kThreads, 0, m->stream>>>(g, min_weight, m->d_F.get(), m->d_wts.get(), m->d_cell.get());
    mesh_vmask_kernel<<<nb, kThreads, 0, m->stream>>>(g, m->d_F.get(), m->d_cell.get(), m->d_vmask.get());
    TSAR_CK(m, cudaGetLastError());
    TSAR_CK(m, cub::DeviceScan::ExclusiveSum(m->d_cub.get(), tmp, vcount, m->d_voff.get(), (int)n, m->stream));
    tmp = m->d_cub.capacity();
    TSAR_CK(m, cub::DeviceScan::ExclusiveSum(m->d_cub.get(), tmp, tcount, m->d_toff.get(), (int)n, m->stream));
    mesh_totals_kernel<<<1, 1, 0, m->stream>>>(n, m->d_vmask.get(), m->d_voff.get(), m->d_cell.get(), m->d_toff.get(), m->d_tot.get());
    TSAR_CK(m, cudaGetLastError());
    TSAR_CK(m, cudaMemcpyAsync(m->h_tot.get(), m->d_tot.get(), 2 * sizeof(long long), cudaMemcpyDeviceToHost, m->stream));
    TSAR_CK(m, cudaStreamSynchronize(m->stream));
    const long long nv = m->h_tot.get()[0], nt = m->h_tot.get()[1];
    m->n_vertices = m->n_triangles = 0;
    if (nv > kMaxPoints) TSAR_FAIL(m, TSAR_ERR_NOMEM, "tsar_mesh_run: more than 2^31 - 1 vertices (int32 indices)");
    TSAR_CK(m, m->d_xyz.reserve(3 * (size_t)std::max(nv, 1LL)));
    TSAR_CK(m, m->d_rgb.reserve(3 * (size_t)std::max(nv, 1LL)));
    TSAR_CK(m, m->d_tri.reserve(3 * (size_t)std::max(nt, 1LL)));
    mesh_vertices_kernel<<<nb, kThreads, 0, m->stream>>>(g, m->d_F.get(), m->d_wts.get(), m->d_csum.get(), m->d_vmask.get(),
                                                         m->d_voff.get(), m->d_xyz.get(), m->d_rgb.get());
    mesh_triangles_kernel<<<nb, kThreads, 0, m->stream>>>(g, m->d_F.get(), m->d_cell.get(), m->d_vmask.get(), m->d_voff.get(),
                                                          m->d_toff.get(), m->d_tri.get());
    TSAR_CK(m, cudaGetLastError());
    TSAR_CK(m, cudaStreamSynchronize(m->stream));
    m->n_vertices = nv;
    m->n_triangles = nt;
    if (n_vertices) *n_vertices = nv;
    if (n_triangles) *n_triangles = nt;
    return TSAR_OK;
}

static int reserve_field(tsar_mesh *m, long long n) {
    TSAR_CK(m, m->d_F.reserve(n));
    TSAR_CK(m, m->d_wts.reserve(n));
    TSAR_CK(m, m->d_csum.reserve(3 * (size_t)n));
    return TSAR_OK;
}

extern "C" {

int tsar_mesh_create(int device, void *stream, int n_views, int W, int H, tsar_mesh **out) {
    if (!out) return TSAR_ERR_ARG;
    *out = nullptr;
    if (n_views < 1 || n_views > 65535 || W < 1 || H < 1) return TSAR_ERR_ARG;
    std::unique_ptr<tsar_mesh> m(new tsar_mesh);
    if (int rc = m->open(device, stream)) return rc;
    m->n_views = n_views;
    m->W = W;
    m->H = H;
    m->P = (size_t)W * H;
    m->view_set.assign(n_views, 0);
    TSAR_CK(m, m->d_cams.reserve(n_views));
    TSAR_CK(m, m->d_views.reserve((size_t)n_views * m->P));
    TSAR_CK(m, m->d_stage_depth.reserve(m->P));
    TSAR_CK(m, m->d_stage_bgr.reserve(3 * m->P));
    TSAR_CK(m, m->d_tot.reserve(2));
    TSAR_CK(m, m->h_tot.reserve(2));
    for (cudaEvent_t &e : m->ev) TSAR_CK(m, cudaEventCreate(&e));
    *out = m.release();
    return TSAR_OK;
}

int tsar_mesh_destroy(tsar_mesh *m) {
    if (!m) return TSAR_OK;
    cudaSetDevice(m->device);
    cudaStreamSynchronize(m->stream);
    delete m;
    return TSAR_OK;
}

const char *tsar_mesh_last_error(const tsar_mesh *m) { return m ? m->err.c_str() : "null mesh handle"; }

int tsar_mesh_set_view(tsar_mesh *m, int view, const tsar_view_camera *cam, const float *depth, const unsigned char *bgr) {
    if (!m) return TSAR_ERR_ARG;
    if (view < 0 || view >= m->n_views) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_set_view: view index out of range");
    if (!cam || !depth || !bgr) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_set_view: null pointer");
    MeshCam c;
    memcpy(c.K, cam->K, sizeof c.K);
    memcpy(c.R, cam->R, sizeof c.R);
    memcpy(c.t, cam->t, sizeof c.t);
    TSAR_CK(m, cudaSetDevice(m->device));
    const size_t P = m->P;
    TSAR_CK(m, cudaMemcpyAsync(m->d_stage_depth.get(), depth, P * sizeof(float), cudaMemcpyHostToDevice, m->stream));
    TSAR_CK(m, cudaMemcpyAsync(m->d_stage_bgr.get(), bgr, 3 * P, cudaMemcpyHostToDevice, m->stream));
    mesh_pack_kernel<<<blocks_for((long long)P, kThreads), kThreads, 0, m->stream>>>(m->d_stage_depth.get(), m->d_stage_bgr.get(), P,
                                                                                    m->d_views.get() + (size_t)view * P);
    TSAR_CK(m, cudaGetLastError());
    TSAR_CK(m, cudaMemcpyAsync(m->d_cams.get() + view, &c, sizeof c, cudaMemcpyHostToDevice, m->stream));
    TSAR_CK(m, cudaStreamSynchronize(m->stream));
    m->view_set[view] = 1;
    return TSAR_OK;
}

int tsar_mesh_run(tsar_mesh *m, const tsar_mesh_grid *grid, const tsar_mesh_params *prm, long long *n_vertices,
                  long long *n_triangles) {
    if (!m) return TSAR_ERR_ARG;
    GridArgs g;
    if (const char *why = check_grid(grid, &g)) {
        m->err = std::string("tsar_mesh_run: ") + why;
        return TSAR_ERR_ARG;
    }
    if (!prm) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_run: null parameters");
    if (!(prm->trunc > 0.0f) || !isfinite(prm->trunc))
        TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_run: trunc must be finite and > 0");
    if (prm->min_weight < 1 || prm->min_weight > 65535) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_run: min_weight must be in [1, 65535]");
    for (int v = 0; v < m->n_views; ++v)
        if (!m->view_set[v]) {
            char buf[128];
            snprintf(buf, sizeof buf, "tsar_mesh_run: view %d was not set", v);
            TSAR_FAIL(m, TSAR_ERR_ARG, buf);
        }
    TSAR_CK(m, cudaSetDevice(m->device));
    m->n_field = 0;
    m->timed = false;
    if (int rc = reserve_field(m, g.n)) return rc;
    TSAR_CK(m, cudaEventRecord(m->ev[0], m->stream));
    const long long tiles = (long long)((g.nx + kTX - 1) / kTX) * ((g.ny + kTY - 1) / kTY) * ((g.nz + kTZ - 1) / kTZ);
    mesh_integrate_kernel<<<(unsigned)tiles, kIntThreads, 0, m->stream>>>(g, m->n_views, m->W, m->H, prm->trunc, m->d_cams.get(),
                                                                        m->d_views.get(), m->d_F.get(), m->d_wts.get(),
                                                                        m->d_csum.get());
    TSAR_CK(m, cudaGetLastError());
    TSAR_CK(m, cudaEventRecord(m->ev[1], m->stream));
    m->n_field = g.n;
    if (int rc = extract(m, g, prm->min_weight, n_vertices, n_triangles)) return rc;
    TSAR_CK(m, cudaEventRecord(m->ev[2], m->stream));
    TSAR_CK(m, cudaEventSynchronize(m->ev[2]));
    m->timed = true;
    return TSAR_OK;
}

int tsar_mesh_get(tsar_mesh *m, float *xyz, unsigned char *rgb, long long vertex_capacity, int *triangles,
                  long long triangle_capacity) {
    if (!m) return TSAR_ERR_ARG;
    if (vertex_capacity < m->n_vertices || triangle_capacity < m->n_triangles)
        TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_get: capacity is smaller than the mesh");
    if ((m->n_vertices && (!xyz || !rgb)) || (m->n_triangles && !triangles)) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_get: null pointer");
    TSAR_CK(m, cudaSetDevice(m->device));
    const size_t nv = (size_t)m->n_vertices, nt = (size_t)m->n_triangles;
    if (nv) {
        TSAR_CK(m, cudaMemcpyAsync(xyz, m->d_xyz.get(), 3 * nv * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
        TSAR_CK(m, cudaMemcpyAsync(rgb, m->d_rgb.get(), 3 * nv, cudaMemcpyDeviceToHost, m->stream));
    }
    if (nt) TSAR_CK(m, cudaMemcpyAsync(triangles, m->d_tri.get(), 3 * nt * sizeof(int), cudaMemcpyDeviceToHost, m->stream));
    TSAR_CK(m, cudaStreamSynchronize(m->stream));
    return TSAR_OK;
}

int tsar_mesh_dbg_extract(tsar_mesh *m, const tsar_mesh_grid *grid, int min_weight, const float *F, const uint16_t *W,
                          const uint16_t *Wc, const uint32_t *bgr_sum, long long *n_vertices, long long *n_triangles) {
    if (!m) return TSAR_ERR_ARG;
    GridArgs g;
    if (const char *why = check_grid(grid, &g)) {
        m->err = std::string("tsar_mesh_dbg_extract: ") + why;
        return TSAR_ERR_ARG;
    }
    if (!F || !W || !Wc || !bgr_sum) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_dbg_extract: null pointer");
    if (min_weight < 1 || min_weight > 65535) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_dbg_extract: min_weight must be in [1, 65535]");
    std::vector<unsigned> wts((size_t)g.n);
    for (long long p = 0; p < g.n; ++p) {
        // what integration guarantees and the colour rule relies on: a defined inside point has Wc >= 1
        if (W[p] >= min_weight && F[p] < 0.0f && Wc[p] == 0)
            TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_dbg_extract: a defined point with F < 0 has Wc = 0");
        wts[p] = W[p] | (unsigned)Wc[p] << 16;
    }
    TSAR_CK(m, cudaSetDevice(m->device));
    m->n_field = 0;
    if (int rc = reserve_field(m, g.n)) return rc;
    TSAR_CK(m, cudaMemcpyAsync(m->d_F.get(), F, g.n * sizeof(float), cudaMemcpyHostToDevice, m->stream));
    TSAR_CK(m, cudaMemcpyAsync(m->d_wts.get(), wts.data(), g.n * sizeof(unsigned), cudaMemcpyHostToDevice, m->stream));
    TSAR_CK(m, cudaMemcpyAsync(m->d_csum.get(), bgr_sum, 3 * g.n * sizeof(unsigned), cudaMemcpyHostToDevice, m->stream));
    m->n_field = g.n;
    return extract(m, g, min_weight, n_vertices, n_triangles);
}

int tsar_mesh_dbg_times(tsar_mesh *m, float *integrate_ms, float *extract_ms) {
    if (!m) return TSAR_ERR_ARG;
    if (!integrate_ms || !extract_ms) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_dbg_times: null pointer");
    if (!m->timed) TSAR_FAIL(m, TSAR_ERR_STATE, "tsar_mesh_dbg_times: no completed tsar_mesh_run");
    TSAR_CK(m, cudaEventElapsedTime(integrate_ms, m->ev[0], m->ev[1]));
    TSAR_CK(m, cudaEventElapsedTime(extract_ms, m->ev[1], m->ev[2]));
    return TSAR_OK;
}

int tsar_mesh_dbg_field(tsar_mesh *m, float *F, uint16_t *W, uint16_t *Wc, uint32_t *bgr_sum) {
    if (!m) return TSAR_ERR_ARG;
    if (!F || !W || !Wc || !bgr_sum) TSAR_FAIL(m, TSAR_ERR_ARG, "tsar_mesh_dbg_field: null pointer");
    const size_t n = (size_t)m->n_field;
    if (!n) TSAR_FAIL(m, TSAR_ERR_STATE, "tsar_mesh_dbg_field: no field (call tsar_mesh_run first)");
    TSAR_CK(m, cudaSetDevice(m->device));
    std::vector<unsigned> wts(n);
    TSAR_CK(m, cudaMemcpyAsync(F, m->d_F.get(), n * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    TSAR_CK(m, cudaMemcpyAsync(wts.data(), m->d_wts.get(), n * sizeof(unsigned), cudaMemcpyDeviceToHost, m->stream));
    TSAR_CK(m, cudaMemcpyAsync(bgr_sum, m->d_csum.get(), 3 * n * sizeof(unsigned), cudaMemcpyDeviceToHost, m->stream));
    TSAR_CK(m, cudaStreamSynchronize(m->stream));
    for (size_t p = 0; p < n; ++p) {
        W[p] = (uint16_t)(wts[p] & 0xffffu);
        Wc[p] = (uint16_t)(wts[p] >> 16);
    }
    return TSAR_OK;
}

}  // extern "C"
