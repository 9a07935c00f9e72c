"""Multi-view fusion of per-view depth maps into one coloured point cloud (DESIGN.md section 4.6) on top of the
tsar_fusion_* entry points of libtsar_b200.so.

A view is a dict: K, R, t (world -> camera, as in cams/*_cam.txt with cam_scale applied), depth (H x W float32, camera
z, 0 = none), normals (H x W x 3 float32, world frame), bgr (H x W x 3 uint8) and neighbours (1..32 indices of other
views, pair.txt order).  Views are fused in list order.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .engine import TsarError

MAX_NEIGHBOURS = 32   # TSAR_FUSION_MAX_NEIGHBOURS
DEFAULT_PARAMS = dict(max_reproj_px=2.0, max_rel_depth=0.01, max_normal_deg=10.0, min_consistent=2)


def make_params(**overrides):
    """tsar_fusion_params: DEFAULT_PARAMS with the given fields replaced."""
    unknown = set(overrides) - set(DEFAULT_PARAMS)
    if unknown:
        raise TypeError(f"unknown fusion parameters {sorted(unknown)}")
    p = dict(DEFAULT_PARAMS, **overrides)
    return L.TsarFusionParams(p["max_reproj_px"], p["max_rel_depth"], p["max_normal_deg"], int(p["min_consistent"]))


def view_camera(K, R, t):
    cam = L.TsarViewCamera()
    cam.K[:] = [float(v) for v in np.asarray(K, np.float32).reshape(9)]
    cam.R[:] = [float(v) for v in np.asarray(R, np.float32).reshape(9)]
    cam.t[:] = [float(v) for v in np.asarray(t, np.float32).reshape(3)]
    return cam


class FusionEngine:
    """One tsar_fusion handle: n_views views of W x H resident on one GPU; run() may be called again with other
    parameters."""

    def __init__(self, n_views, W, H, device=0, stream=None):
        self.lib = L.load()
        h = C.c_void_p()
        rc = self.lib.tsar_fusion_create(int(device), C.c_void_p(stream) if stream else None, int(n_views), int(W), int(H),
                                         C.byref(h))
        if rc != 0:
            raise TsarError(f"tsar_fusion_create(device={device}, {n_views} views of {W}x{H}) failed with {rc}")
        self.h, self.n_views, self.W, self.H = h, int(n_views), int(W), int(H)

    def _check(self, rc, what):
        if rc != 0:
            raise TsarError(f"{what} failed with {rc}: {self.lib.tsar_fusion_last_error(self.h).decode()}")

    def set_view(self, view, K, R, t, depth, normals, bgr, neighbours):
        shape = (self.H, self.W)
        depth = np.ascontiguousarray(depth, np.float32)
        normals = np.ascontiguousarray(normals, np.float32)
        bgr = np.ascontiguousarray(bgr, np.uint8)
        if depth.shape != shape or normals.shape != shape + (3,) or bgr.shape != shape + (3,):
            raise ValueError(f"view {view}: depth / normals / bgr must be {shape}, {shape + (3,)}, {shape + (3,)}; got "
                             f"{depth.shape}, {normals.shape}, {bgr.shape}")
        nb = (C.c_int * max(1, len(neighbours)))(*[int(k) for k in neighbours])
        self._check(self.lib.tsar_fusion_set_view(self.h, int(view), C.byref(view_camera(K, R, t)), depth.ctypes.data,
                                                  normals.ctypes.data, bgr.ctypes.data, nb, len(neighbours)),
                    f"tsar_fusion_set_view(view {view})")

    def run(self, params=None):
        """Returns (xyz [n][3] float32, normals [n][3] float32, rgb [n][3] uint8)."""
        p = params if isinstance(params, L.TsarFusionParams) else make_params(**(params or {}))
        n = C.c_longlong()
        self._check(self.lib.tsar_fusion_run(self.h, C.byref(p), C.byref(n)), "tsar_fusion_run")
        xyz, nrm, rgb = np.empty((n.value, 3), np.float32), np.empty((n.value, 3), np.float32), np.empty((n.value, 3), np.uint8)
        self._check(self.lib.tsar_fusion_points(self.h, xyz.ctypes.data, nrm.ctypes.data, rgb.ctypes.data, n.value),
                    "tsar_fusion_points")
        return xyz, nrm, rgb

    def rounds(self):
        """(most resolution rounds one view needed, rounds summed over the views) of the last run."""
        mx, tot = C.c_int(), C.c_longlong()
        self._check(self.lib.tsar_fusion_dbg_rounds(self.h, C.byref(mx), C.byref(tot)), "tsar_fusion_dbg_rounds")
        return mx.value, tot.value

    def close(self):
        if getattr(self, "h", None):
            self.lib.tsar_fusion_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def fuse(views, params=None, device=0):
    """Fused point cloud of `views` (see the module docstring): (xyz, normals, rgb).  params: dict of
    tsar_fusion_params fields overriding DEFAULT_PARAMS."""
    if not views:
        raise ValueError("fuse: no views")
    H, W = np.shape(views[0]["depth"])
    with FusionEngine(len(views), W, H, device=device) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], v["neighbours"])
        return eng.run(params)
