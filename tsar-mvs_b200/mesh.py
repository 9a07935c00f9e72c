"""A coloured triangle mesh from per-view depth maps (DESIGN.md section 4.8) on top of the tsar_mesh_* entry points of
libtsar_b200.so: TSDF integration on a dense voxel grid, then marching tetrahedra.

A view is a dict: K, R, t (world -> camera, as in cams/*_cam.txt with cam_scale applied), depth (H x W float32, camera
z, 0 = none) and bgr (H x W x 3 uint8); other keys are ignored.  Views are integrated in list order.  A grid is a dict:
origin (3 floats), voxel (> 0) and dims (nx, ny, nz); grid point (i, j, k) sits at origin + (i + 0.5, j + 0.5, k + 0.5)
* voxel.
"""
import ctypes as C
import math

import numpy as np

from . import _lib as L
from .engine import TsarError
from .fusion import view_camera

MAX_POINTS = 2 ** 31 - 1     # grid points and vertices (int32 indices)
MAX_DIM = 2 ** 23            # per axis: (float)i + 0.5f is exact
DEFAULT_MIN_WEIGHT = 3
TRUNC_VOXELS = 4.0           # default trunc, in voxels
SAMPLE_STRIDE = 8            # default_grid back-projects every 8th pixel of each axis


def make_grid(grid):
    g = L.TsarMeshGrid()
    g.origin[:] = [float(np.float32(v)) for v in grid["origin"]]
    g.voxel = float(np.float32(grid["voxel"]))
    g.dims[:] = [int(v) for v in grid["dims"]]
    return g


def depth_samples(view, stride=SAMPLE_STRIDE):
    """World points (float64, X = C + D R^T K^-1 (x, y, 1)) and D / f_x of every `stride`-th pixel (both axes) with a
    finite depth > 0."""
    K, R, t = (np.asarray(view[k], np.float64) for k in ("K", "R", "t"))
    d = np.asarray(view["depth"], np.float64)[::stride, ::stride]
    ys, xs = np.mgrid[0:view["depth"].shape[0]:stride, 0:view["depth"].shape[1]:stride]
    ok = np.isfinite(d) & (d > 0)
    rays = np.stack([xs[ok], ys[ok], np.ones(ok.sum())], -1) @ np.linalg.inv(K).T
    C_ = -R.T @ t.reshape(3)
    return C_ + d[ok, None] * (rays @ R), d[ok] / K[0, 0]


def box_grid(lo, hi, voxel):
    """The grid whose points cover the box [lo, hi] at spacing `voxel` (at least 2 points per axis).  Raises a one-line
    ValueError when it has more than 2^31 - 1 points or an axis more than 2^23."""
    voxel = float(np.float32(voxel))
    if not (math.isfinite(voxel) and voxel > 0):
        raise ValueError(f"bad voxel size {voxel!r} (need a finite value > 0)")
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    dims = [max(2, int(math.ceil((h - l) / voxel))) for l, h in zip(lo, hi)]
    n = dims[0] * dims[1] * dims[2]
    if n > MAX_POINTS or max(dims) > MAX_DIM:
        raise ValueError(f"the mesh grid would have {n} voxels ({dims[0]} x {dims[1]} x {dims[2]} at voxel {voxel:g}), more "
                         f"than 2^31 - 1 (or 2^23 per axis): choose a larger -mesh_voxel or a smaller -mesh_bbox")
    return dict(origin=[float(np.float32(v)) for v in lo], voxel=voxel, dims=dims)


def default_voxel(ratios):
    """2 x the median of the D / f_x of depth_samples, rounded to float32."""
    if len(ratios) == 0:
        raise ValueError("no valid depth in any view: cannot place a mesh grid")
    return float(np.float32(2.0 * np.median(ratios)))


def grid_from_samples(points, ratios, voxel=None, margin=None):
    """default_grid from depth_samples: voxel = default_voxel(ratios); the box is the per-axis 0.001 / 0.999 quantile
    (method "lower") of the points, widened by `margin` (default: the default trunc, 4 voxels)."""
    voxel = default_voxel(ratios) if voxel is None else float(np.float32(voxel))
    margin = TRUNC_VOXELS * voxel if margin is None else float(margin)
    lo = np.quantile(points, 0.001, axis=0, method="lower") - margin
    hi = np.quantile(points, 0.999, axis=0, method="lower") + margin
    return box_grid(lo, hi, voxel)


def default_grid(views, voxel=None, margin=None):
    """A grid around what the views see (host side, deterministic): see grid_from_samples."""
    s = [depth_samples(v) for v in views]
    return grid_from_samples(np.concatenate([p for p, _ in s]), np.concatenate([r for _, r in s]), voxel, margin)


class MeshEngine:
    """One tsar_mesh handle: n_views views of W x H resident on one GPU; run() may be called again with another grid or
    other parameters."""

    def __init__(self, n_views, W, H, device=0, stream=None):
        self.lib = L.load()
        h = C.c_void_p()
        rc = self.lib.tsar_mesh_create(int(device), C.c_void_p(stream) if stream else None, int(n_views), int(W), int(H),
                                       C.byref(h))
        if rc != 0:
            raise TsarError(f"tsar_mesh_create(device={device}, {n_views} views of {W}x{H}) failed with {rc}")
        self.h, self.n_views, self.W, self.H = h, int(n_views), int(W), int(H)
        self.counts = (0, 0)

    def _check(self, rc, what):
        if rc != 0:
            raise TsarError(f"{what} failed with {rc}: {self.lib.tsar_mesh_last_error(self.h).decode()}")

    def set_view(self, view, K, R, t, depth, bgr):
        shape = (self.H, self.W)
        depth = np.ascontiguousarray(depth, np.float32)
        bgr = np.ascontiguousarray(bgr, np.uint8)
        if depth.shape != shape or bgr.shape != shape + (3,):
            raise ValueError(f"view {view}: depth / bgr must be {shape}, {shape + (3,)}; got {depth.shape}, {bgr.shape}")
        self._check(self.lib.tsar_mesh_set_view(self.h, int(view), C.byref(view_camera(K, R, t)), depth.ctypes.data,
                                                bgr.ctypes.data), f"tsar_mesh_set_view(view {view})")

    def run(self, grid, trunc=None, min_weight=DEFAULT_MIN_WEIGHT, fetch=True):
        """Integrates and extracts; returns get() (or (n_vertices, n_triangles) with fetch=False, the mesh staying on
        the device).  trunc defaults to 4 voxels."""
        trunc = TRUNC_VOXELS * float(np.float32(grid["voxel"])) if trunc is None else trunc
        p = L.TsarMeshParams(float(np.float32(trunc)), int(min_weight))
        nv, nt = C.c_longlong(), C.c_longlong()
        self._check(self.lib.tsar_mesh_run(self.h, C.byref(make_grid(grid)), C.byref(p), C.byref(nv), C.byref(nt)),
                    "tsar_mesh_run")
        self.counts = (nv.value, nt.value)
        return self.get() if fetch else self.counts

    def get(self):
        """(xyz [n][3] float32, rgb [n][3] uint8, triangles [m][3] int32) of the last run."""
        nv, nt = self.counts
        xyz, rgb, tri = np.empty((nv, 3), np.float32), np.empty((nv, 3), np.uint8), np.empty((nt, 3), np.int32)
        self._check(self.lib.tsar_mesh_get(self.h, xyz.ctypes.data, rgb.ctypes.data, nv, tri.ctypes.data, nt), "tsar_mesh_get")
        return xyz, rgb, tri

    def dbg_extract(self, grid, min_weight, F, W, Wc, bgr_sum):
        """Extraction alone, from a given field (arrays of nx*ny*nz points in grid order; bgr_sum 3 per point)."""
        a = [np.ascontiguousarray(x, dt) for x, dt in ((F, np.float32), (W, np.uint16), (Wc, np.uint16), (bgr_sum, np.uint32))]
        nv, nt = C.c_longlong(), C.c_longlong()
        self._check(self.lib.tsar_mesh_dbg_extract(self.h, C.byref(make_grid(grid)), int(min_weight), *[x.ctypes.data for x in a],
                                                   C.byref(nv), C.byref(nt)), "tsar_mesh_dbg_extract")
        self.counts = (nv.value, nt.value)
        return self.get()

    def dbg_times(self):
        """(integration ms, extraction ms) of the last run, from CUDA events on the handle's stream."""
        a, b = C.c_float(), C.c_float()
        self._check(self.lib.tsar_mesh_dbg_times(self.h, C.byref(a), C.byref(b)), "tsar_mesh_dbg_times")
        return a.value, b.value

    def dbg_field(self, grid):
        """(F, W, Wc, bgr_sum) of the last run, shaped (nz, ny, nx) (bgr_sum: (nz, ny, nx, 3))."""
        shape = tuple(int(v) for v in grid["dims"])[::-1]
        F, W, Wc = np.empty(shape, np.float32), np.empty(shape, np.uint16), np.empty(shape, np.uint16)
        S = np.empty(shape + (3,), np.uint32)
        self._check(self.lib.tsar_mesh_dbg_field(self.h, F.ctypes.data, W.ctypes.data, Wc.ctypes.data, S.ctypes.data),
                    "tsar_mesh_dbg_field")
        return F, W, Wc, S

    def close(self):
        if getattr(self, "h", None):
            self.lib.tsar_mesh_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def mesh(views, grid=None, trunc=None, min_weight=DEFAULT_MIN_WEIGHT, device=0):
    """Triangle mesh of `views` (see the module docstring): (xyz, rgb, triangles).  grid defaults to
    default_grid(views), trunc to 4 voxels."""
    if not views:
        raise ValueError("mesh: no views")
    grid = default_grid(views) if grid is None else grid
    H, W = np.shape(views[0]["depth"])
    with MeshEngine(len(views), W, H, device=device) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        return eng.run(grid, trunc, min_weight)
