"""ctypes binding of oracle/liboracle_cpu.so (C restatement) -- TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "liboracle_cpu.so")


def build():
    src = os.path.join(_HERE, "oracle_cpu.c")
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "oracle_cpu.h"))):
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-fopenmp", "-o", LIB, src, "-lm"])
    return LIB


class CpuOracle:
    def __init__(self, camera_struct_type, params_struct_type, images, cams_struct, subset, params, cam_f):
        self.lib = C.CDLL(build())
        vp, i = C.c_void_p, C.c_int
        L = self.lib
        L.oc_create.restype = vp
        L.oc_create.argtypes = [i, i, i, C.POINTER(vp), C.POINTER(camera_struct_type), C.c_float, C.POINTER(i), i,
                                C.POINTER(params_struct_type)]
        L.oc_destroy.argtypes = [vp]
        for n in ("oc_planes", "oc_costs", "oc_beview"):
            getattr(L, n).restype = vp
            getattr(L, n).argtypes = [vp]
        L.oc_evals.restype = C.c_longlong
        L.oc_evals.argtypes = [vp]
        L.oc_xorwow_row.argtypes = [C.c_uint64, i, i, vp]
        L.oc_tex.restype = C.c_float
        L.oc_tex.argtypes = [vp, i, i, C.c_float, C.c_float]
        L.oc_eval_planes.argtypes = [vp, i, vp, vp, i, vp, vp, vp]
        L.oc_eval_views.argtypes = [vp, i, vp, vp, i, vp, vp]
        L.oc_init.argtypes = [vp, C.c_uint64]
        L.oc_init_planes_only.argtypes = [vp, C.c_uint64]
        L.oc_spatial.argtypes = [vp, i]
        L.oc_refine.argtypes = [vp, i, C.c_uint64]
        L.oc_iterate.argtypes = [vp, i, C.c_uint64]
        L.oc_output.argtypes = [vp, vp]
        imgs = [np.ascontiguousarray(im, np.float32) for im in images]
        self.H, self.W = imgs[0].shape
        self.V = len(subset)
        ptrs = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
        sub = (C.c_int * len(subset))(*[int(s) for s in subset])
        self.h = C.c_void_p(L.oc_create(self.W, self.H, len(imgs), ptrs, cams_struct, float(cam_f), sub, len(subset), C.byref(params)))

    def close(self):
        if self.h:
            self.lib.oc_destroy(self.h)
            self.h = None

    def _arr(self, ptr, shape, dt):
        n = int(np.prod(shape))
        buf = (C.c_byte * (n * np.dtype(dt).itemsize)).from_address(ptr)
        return np.frombuffer(buf, dt).reshape(shape).copy()

    def planes(self): return self._arr(self.lib.oc_planes(self.h), (self.H, self.W, 4), np.float32)
    def costs(self): return self._arr(self.lib.oc_costs(self.h), (self.H, self.W), np.float32)
    def beview(self): return self._arr(self.lib.oc_beview(self.h), (self.H, self.W), np.int32)
    def evals(self): return self.lib.oc_evals(self.h)

    def set_state(self, planes, costs):
        C.memmove(self.lib.oc_planes(self.h), np.ascontiguousarray(planes, np.float32).ctypes.data, self.W * self.H * 16)
        C.memmove(self.lib.oc_costs(self.h), np.ascontiguousarray(costs, np.float32).ctypes.data, self.W * self.H * 4)

    def eval_planes(self, xy, planes, wrapper_rounding=False):
        xy = np.ascontiguousarray(xy, np.int32).reshape(-1, 2)
        planes = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
        n = len(xy)
        cost, bv, ratio = np.empty(n, np.float32), np.empty(n, np.int32), np.empty(n, np.float32)
        self.lib.oc_eval_planes(self.h, n, xy.ctypes.data, planes.ctypes.data, int(wrapper_rounding), cost.ctypes.data,
                                bv.ctypes.data, ratio.ctypes.data)
        return cost, bv, ratio

    def eval_views(self, xy, planes, wrapper_rounding=False):
        """[n][V] pmCost of each selected view (subset order) for each pair, and [n][V] float64 relative variance
        var / E[src^2] of that view's bilateral-weighted source samples."""
        xy = np.ascontiguousarray(xy, np.int32).reshape(-1, 2)
        planes = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
        out = np.empty((len(xy), self.V), np.float32)
        rel = np.empty((len(xy), self.V), np.float64)
        self.lib.oc_eval_views(self.h, len(xy), xy.ctypes.data, planes.ctypes.data, int(wrapper_rounding), out.ctypes.data,
                               rel.ctypes.data)
        return out, rel

    def init_planes(self, seed): self.lib.oc_init(self.h, int(seed))
    def init_planes_only(self, seed): self.lib.oc_init_planes_only(self.h, int(seed))
    def spatial(self, colour): self.lib.oc_spatial(self.h, int(colour))
    def refine(self, colour, seed): self.lib.oc_refine(self.h, int(colour), int(seed))
    def iterate(self, iters, seed0): self.lib.oc_iterate(self.h, int(iters), int(seed0))

    def output(self):
        out = np.empty((self.H, self.W, 4), np.float32)
        self.lib.oc_output(self.h, out.ctypes.data)
        return out

    def xorwow_row(self, seed, y, n):
        out = np.empty(n, np.uint32)
        self.lib.oc_xorwow_row(int(seed), int(y), int(n), out.ctypes.data)
        return out

    def tex(self, img, x, y):
        img = np.ascontiguousarray(img, np.float32)
        return self.lib.oc_tex(img.ctypes.data, img.shape[1], img.shape[0], float(x), float(y))


def fit_region_plane(camera_struct_type, cam0_struct, cam_f, depth, scale, canny, region, region_size, rnd, plane0):
    """C restatement of the reference's per-region RANSAC (main.cpp:1520-1730) for one region."""
    lib = C.CDLL(build())
    lib.oc_fit_region_plane.argtypes = [C.c_int, C.c_int, C.POINTER(camera_struct_type), C.c_float, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
    depth, scale, canny = (np.ascontiguousarray(a, np.float32) for a in (depth, scale, canny))
    rnd = np.ascontiguousarray(rnd, np.uint32)
    plane = np.ascontiguousarray(plane0, np.float32).copy()
    H, W = depth.shape
    used = lib.oc_fit_region_plane(W, H, C.byref(cam0_struct), float(cam_f), depth.ctypes.data, scale.ctypes.data,
                                   canny.ctypes.data, int(region), float(region_size), rnd.ctypes.data, plane.ctypes.data)
    return plane, used
