"""ctypes binding of oracle/libmesh_cpu.so (C restatement of the mesh rule) -- TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libmesh_cpu.so")


class Grid(C.Structure):
    """tsar_mesh_grid."""
    _fields_ = [("origin", C.c_float * 3), ("voxel", C.c_float), ("dims", C.c_int * 3)]


class ViewCamera(C.Structure):
    """tsar_view_camera."""
    _fields_ = [("K", C.c_float * 9), ("R", C.c_float * 9), ("t", C.c_float * 3)]


def build():
    src = os.path.join(_HERE, "mesh_cpu.c")
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-fopenmp", "-o", LIB, src, "-lm"])
    return LIB


def _lib():
    lib = C.CDLL(build())
    vp, ll, i, f = C.c_void_p, C.c_longlong, C.c_int, C.c_float
    lib.oc_mesh_field.restype = None
    lib.oc_mesh_field.argtypes = [i, i, i, vp, vp, vp, vp, f, vp, vp, vp, vp]
    lib.oc_mesh_extract.restype = ll
    lib.oc_mesh_extract.argtypes = [vp, i, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.oc_free.argtypes = [vp]
    return lib


def make_grid(grid):
    """grid: dict origin (3), voxel, dims (nx, ny, nz)."""
    g = Grid()
    g.origin[:] = [float(np.float32(v)) for v in grid["origin"]]
    g.voxel = float(np.float32(grid["voxel"]))
    g.dims[:] = [int(v) for v in grid["dims"]]
    return g


def field(views, grid, trunc):
    """oc_mesh_field: (F, W, Wc, bgr_sum) as arrays of shape (nz, ny, nx) (bgr_sum: (nz, ny, nx, 3))."""
    lib = _lib()
    g = make_grid(grid)
    n_views = len(views)
    H, W = np.shape(views[0]["depth"])
    cams = (ViewCamera * n_views)()
    for k, v in enumerate(views):
        cams[k].K[:] = [float(x) for x in np.asarray(v["K"], np.float32).reshape(9)]
        cams[k].R[:] = [float(x) for x in np.asarray(v["R"], np.float32).reshape(9)]
        cams[k].t[:] = [float(x) for x in np.asarray(v["t"], np.float32).reshape(3)]
    keep = [(np.ascontiguousarray(v["depth"], np.float32), np.ascontiguousarray(v["bgr"], np.uint8)) for v in views]
    depth = (C.c_void_p * n_views)(*[d.ctypes.data for d, _ in keep])
    bgr = (C.c_void_p * n_views)(*[b.ctypes.data for _, b in keep])
    shape = tuple(int(v) for v in grid["dims"])[::-1]
    F, Wt, Wc = np.empty(shape, np.float32), np.empty(shape, np.uint16), np.empty(shape, np.uint16)
    S = np.empty(shape + (3,), np.uint32)
    lib.oc_mesh_field(n_views, W, H, cams, depth, bgr, C.byref(g), float(np.float32(trunc)), F.ctypes.data, Wt.ctypes.data,
                      Wc.ctypes.data, S.ctypes.data)
    return F, Wt, Wc, S


def extract(grid, min_weight, F, W, Wc, bgr_sum):
    """oc_mesh_extract on a given field: (xyz [n][3] float32, rgb [n][3] uint8, triangles [m][3] int32).  Raises when a
    triangle would use a vertex the rule does not create."""
    lib = _lib()
    g = make_grid(grid)
    arrs = [np.ascontiguousarray(a, dt) for a, dt in ((F, np.float32), (W, np.uint16), (Wc, np.uint16), (bgr_sum, np.uint32))]
    out = [C.c_void_p() for _ in range(3)]
    n_tri = C.c_longlong()
    nv = lib.oc_mesh_extract(C.byref(g), int(min_weight), *[a.ctypes.data for a in arrs], *[C.byref(o) for o in out],
                             C.byref(n_tri))
    res = []
    for o, dt, n in zip(out, (np.float32, np.uint8, np.int32), (nv, nv, max(n_tri.value, 0))):
        a = np.frombuffer((C.c_byte * (n * 3 * np.dtype(dt).itemsize)).from_address(o.value), dt).reshape(n, 3).copy() \
            if n else np.empty((0, 3), dt)
        lib.oc_free(o)
        res.append(a)
    if n_tri.value < 0:
        raise AssertionError("oc_mesh_extract: a triangle uses an edge without a vertex")
    return tuple(res)


def mesh(views, grid, trunc, min_weight):
    """oc_mesh: the whole rule (DESIGN.md section 4.8) on views as tsar-mvs_b200/mesh.py takes them."""
    return extract(grid, min_weight, *field(views, grid, trunc))
