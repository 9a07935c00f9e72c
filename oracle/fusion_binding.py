"""ctypes binding of oracle/libfusion_cpu.so (C restatement of the fusion rule) -- TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libfusion_cpu.so")


def build():
    src = os.path.join(_HERE, "fusion_cpu.c")
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-o", LIB, src, "-lm"])
    return LIB


def fuse(view_camera_type, params_struct, views):
    """C restatement of the sequential fusion rule (oc_fuse, DESIGN.md section 4.6); views as tsar-mvs_b200/fusion.py
    takes them.  Returns (xyz, normals, rgb)."""
    lib = C.CDLL(build())
    vp = C.c_void_p
    lib.oc_fuse.restype = C.c_longlong
    lib.oc_fuse.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.oc_free.argtypes = [vp]
    n_views = len(views)
    H, W = np.shape(views[0]["depth"])
    cams = (view_camera_type * n_views)()
    for k, v in enumerate(views):
        cams[k].K[:] = [float(x) for x in np.asarray(v["K"], np.float32).reshape(9)]
        cams[k].R[:] = [float(x) for x in np.asarray(v["R"], np.float32).reshape(9)]
        cams[k].t[:] = [float(x) for x in np.asarray(v["t"], np.float32).reshape(3)]
    keep = [np.ascontiguousarray(v[key], dt) for v in views for key, dt in (("depth", np.float32), ("normals", np.float32), ("bgr", np.uint8))]
    depth, nrm, bgr = ((C.c_void_p * n_views)(*[keep[3 * k + i].ctypes.data for k in range(n_views)]) for i in range(3))
    nbs = [np.ascontiguousarray(v["neighbours"], np.int32) for v in views]
    nb_ptr = (C.c_void_p * n_views)(*[a.ctypes.data for a in nbs])
    nb_len = (C.c_int * n_views)(*[len(a) for a in nbs])
    out = [C.c_void_p() for _ in range(3)]
    n = lib.oc_fuse(n_views, W, H, cams, depth, nrm, bgr, nb_ptr, nb_len, C.byref(params_struct), *[C.byref(o) for o in out])
    res = []
    for o, dt in zip(out, (np.float32, np.float32, np.uint8)):
        a = np.frombuffer((C.c_byte * (n * 3 * np.dtype(dt).itemsize)).from_address(o.value), dt).reshape(n, 3).copy() if n else np.empty((0, 3), dt)
        lib.oc_free(o)
        res.append(a)
    return tuple(res)
