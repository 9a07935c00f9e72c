"""ctypes binding of oracle/_ref/libtsar_ref*.so -- TEST INFRASTRUCTURE ONLY.

Drives the reference's own kernels (gipuma.cu compiled unmodified by oracle/build_ref.sh) with the
same method names as tsar-mvs_b200/engine.py so parity tests can run both side by side.  Only
tests/, __graft_entry__.smoke() and bench.py (--impl reference / cpu_baseline) may import this.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(_HERE, "_ref")

F_NORM4, F_COST, F_DEPTH, F_FAKEDEPTH, F_SCALE, F_CANNY, F_RATIO, F_BEVIEW, F_LRDIFF, F_CONFID, \
    F_REGION_TEXT, F_REGION_NORM4 = range(12)
_DT = {F_NORM4: (np.float32, 4), F_BEVIEW: (np.int32, 1), F_REGION_NORM4: (np.float32, 4)}


# 'asis': gipuma.cu unmodified; 'snapshot': the race-free twin (2-line store redirection); 'snapshot_init': the twin with
# gipuma_WMF's / gipuma_WMF_Final's norm_mid zero-initialised (defined where the reference reads it uninitialised)
_LIB_OF = {"asis": "libtsar_ref.so", "snapshot": "libtsar_ref_snap.so", "snapshot_init": "libtsar_ref_snapinit.so"}


def available(variant="asis"):
    return os.path.exists(os.path.join(REF_DIR, _LIB_OF[variant]))


class RefEngine:
    """variant: 'asis' (the reference as written, racy same-colour reads, SURVEY Q3) or
    'snapshot' (2-line build-time patch: deterministic pre-launch-snapshot semantics)."""

    def __init__(self, camera_struct_type, params_struct_type, variant="asis"):
        name = _LIB_OF[variant]
        self.lib = C.CDLL(os.path.join(REF_DIR, name))
        self.variant = variant
        self.Cam, self.Par = camera_struct_type, params_struct_type
        self.h = None
        vp, i, u64 = C.c_void_p, C.c_int, C.c_uint64
        L = self.lib
        L.ref_variant.restype = C.c_char_p
        L.ref_create.restype = i
        L.ref_create.argtypes = [i, i, i, C.POINTER(vp), C.POINTER(self.Cam), C.c_float, C.POINTER(i), i,
                                 C.POINTER(self.Par), C.POINTER(vp)]
        L.ref_destroy.argtypes = [vp]
        L.ref_set_regions.argtypes = [vp, i, vp, vp]
        L.ref_upload.argtypes = [vp, i, vp, C.c_size_t]
        L.ref_download.argtypes = [vp, i, vp, C.c_size_t]
        L.ref_init.argtypes = [vp, u64]
        L.ref_launch.argtypes = [vp, i, u64]
        L.ref_iterate.argtypes = [vp, i, u64]
        for n in ("ref_lrdiff", "ref_getview", "ref_get_disp", "ref_update_scale_2", "ref_update_scale", "ref_compute_disp"):
            getattr(L, n).argtypes = [vp]
        L.ref_wmf.argtypes = [vp, i]
        L.ref_wmf_final.argtypes = [vp, i]
        L.ref_eval_planes.argtypes = [vp, i, vp, vp, vp, vp, vp]
        L.ref_depthmap.argtypes = [vp, u64, i, i, C.POINTER(C.c_float)]
        assert L.ref_variant().decode() == variant

    def _ck(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"[ref:{self.variant}] {what} failed ({rc})")

    def create(self, images, cams_struct, subset, params, cam_f):
        imgs = [np.ascontiguousarray(im, np.float32) for im in images]
        self.H, self.W = imgs[0].shape
        ptrs = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
        sub = (C.c_int * len(subset))(*[int(s) for s in subset])
        h = C.c_void_p()
        self._ck(self.lib.ref_create(self.W, self.H, len(imgs), ptrs, cams_struct, float(cam_f), sub, len(subset),
                                     C.byref(params), C.byref(h)), "ref_create")
        self.h = h
        self.iterations = params.iterations

    def close(self):
        if self.h:
            self.lib.ref_destroy(self.h)
            self.h = None

    def set_regions(self, text, norm4):
        text = np.ascontiguousarray(text, np.float32)
        norm4 = np.ascontiguousarray(norm4, np.float32).reshape(-1, 4)
        self.n_regions = len(text)
        self._ck(self.lib.ref_set_regions(self.h, len(text), text.ctypes.data, norm4.ctypes.data), "ref_set_regions")

    def init_planes(self, seed): self._ck(self.lib.ref_init(self.h, int(seed)), "ref_init")
    def launch(self, kind, seed=0): self._ck(self.lib.ref_launch(self.h, int(kind), int(seed)), "ref_launch")
    def iterate(self, iters, seed0): self._ck(self.lib.ref_iterate(self.h, int(iters), int(seed0)), "ref_iterate")
    def lrdiff(self): self._ck(self.lib.ref_lrdiff(self.h), "ref_lrdiff")
    def getview(self): self._ck(self.lib.ref_getview(self.h), "ref_getview")
    def get_disp(self): self._ck(self.lib.ref_get_disp(self.h), "ref_get_disp")
    def update_scale_2(self): self._ck(self.lib.ref_update_scale_2(self.h), "ref_update_scale_2")
    def update_scale(self): self._ck(self.lib.ref_update_scale(self.h), "ref_update_scale")
    def compute_disp(self): self._ck(self.lib.ref_compute_disp(self.h), "ref_compute_disp")
    def wmf(self, it): self._ck(self.lib.ref_wmf(self.h, int(it)), "ref_wmf")
    def wmf_final(self, it): self._ck(self.lib.ref_wmf_final(self.h, int(it)), "ref_wmf_final")

    def eval_planes(self, xy, planes):
        xy = np.ascontiguousarray(xy, np.int32).reshape(-1, 2)
        planes = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
        n = len(xy)
        cost, bv, ratio = np.empty(n, np.float32), np.empty(n, np.int32), np.empty(n, np.float32)
        self._ck(self.lib.ref_eval_planes(self.h, n, xy.ctypes.data, planes.ctypes.data, cost.ctypes.data,
                                          bv.ctypes.data, ratio.ctypes.data), "ref_eval_planes")
        return cost, bv, ratio

    def depthmap(self, seed0, iters=None, prefetch=False):
        ms = C.c_float(0)
        self._ck(self.lib.ref_depthmap(self.h, int(seed0), int(self.iterations if iters is None else iters),
                                       int(prefetch), C.byref(ms)), "ref_depthmap")
        return ms.value

    def download(self, field):
        dt, ch = _DT.get(field, (np.float32, 1))
        if field in (F_REGION_TEXT, F_REGION_NORM4):
            shape = (self.n_regions,) if ch == 1 else (self.n_regions, ch)
        else:
            shape = (self.H, self.W) if ch == 1 else (self.H, self.W, ch)
        out = np.empty(shape, dt)
        self._ck(self.lib.ref_download(self.h, field, out.ctypes.data, out.nbytes), "ref_download")
        return out

    def upload(self, field, arr):
        dt, _ = _DT.get(field, (np.float32, 1))
        arr = np.ascontiguousarray(arr, dt)
        self._ck(self.lib.ref_upload(self.h, field, arr.ctypes.data, arr.nbytes), "ref_upload")


def ref_slic(bgrx, spixel_size=20, no_iters=5, coh_weight=5.0, enforce_connectivity=False):
    """The reference's gSLICr GPU engine (gSLICr_seg_engine_GPU.cu unmodified) on a [h][w][4] uint8 image.
    Returns (labels int32 [h][w], ms)."""
    lib = C.CDLL(os.path.join(REF_DIR, "libgslic_ref.so"))
    lib.ref_slic.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p,
                             C.POINTER(C.c_float)]
    bgrx = np.ascontiguousarray(bgrx, np.uint8)
    h, w = bgrx.shape[:2]
    labels = np.empty((h, w), np.int32)
    ms = C.c_float(0)
    rc = lib.ref_slic(bgrx.ctypes.data, w, h, int(spixel_size), int(no_iters), float(coh_weight), int(enforce_connectivity),
                      labels.ctypes.data, C.byref(ms))
    if rc != 0:
        raise RuntimeError(f"ref_slic failed ({rc})")
    return labels, ms.value


def slic_last_lab(n):
    """CIELab image [n][4] of the last ref_slic call (the reference engine's own buffer)."""
    lib = C.CDLL(os.path.join(REF_DIR, "libgslic_ref.so"))
    lib.ref_slic_last_lab.restype = C.c_longlong
    lib.ref_slic_last_lab.argtypes = [C.c_void_p, C.c_longlong]
    out = np.empty((n, 4), np.float32)
    lib.ref_slic_last_lab(out.ctypes.data, n)
    return out


def slic_last_centres(nsp):
    """Superpixel records [nsp][8] (centre, colour, count) of the last ref_slic call."""
    lib = C.CDLL(os.path.join(REF_DIR, "libgslic_ref.so"))
    out = np.zeros((nsp, 8), np.float32)
    lib.ref_slic_last_centres(out.ctypes.data_as(C.c_void_p), nsp)
    return out
