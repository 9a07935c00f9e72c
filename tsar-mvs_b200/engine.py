"""Host-side mirror of the reference's depthmap entry points on top of the C ABI.

`DepthmapEngine` is what a user of the reference's firstcuda/sliccuda/fakecuda/fillcuda
(gipuma.h:2-5) + gSLICr core_engine (gSLICr_core_engine.h:11-33) drives instead; method names follow
the reference kernels they stand for.  All compute happens in libtsar_b200.so (hand-written sm_100a
CUDA); this module only marshals numpy arrays / device pointers.
"""
import ctypes as C

import numpy as np

from . import _lib as L

FIELD_DTYPE = {
    L.F_NORM4: (np.float32, 4), L.F_COST: (np.float32, 1), L.F_DEPTH: (np.float32, 1),
    L.F_FAKEDEPTH: (np.float32, 1), L.F_SCALE: (np.float32, 1), L.F_CANNY: (np.float32, 1),
    L.F_RATIO: (np.float32, 1), L.F_BEVIEW: (np.int32, 1), L.F_LRDIFF: (np.float32, 1),
    L.F_CONFID: (np.float32, 1), L.F_REGION_TEXT: (np.float32, 1), L.F_REGION_NORM4: (np.float32, 4),
}


class TsarError(RuntimeError):
    pass


def make_params(box=11, iterations=8, n_best=1, cost_comb=1, min_disparity=0.0, max_disparity=256.0, color_processing=0):
    """AlgorithmParameters as the run scripts set them (scripts/pipes.sh:10-15)."""
    return L.TsarParams(box, box, iterations, n_best, cost_comb, min_disparity, max_disparity, int(color_processing))


def cameras_to_struct(cams):
    """cams: list of dicts with the tsar_camera fields (see scene.make_cameras)."""
    arr = (L.TsarCamera * len(cams))()
    for i, c in enumerate(cams):
        for name in ("K", "K_inv", "R", "R_orig", "R_orig_inv", "M_inv"):
            getattr(arr[i], name)[:] = [float(v) for v in np.asarray(c[name], np.float32).reshape(9)]
        for name in ("t4", "P_col34", "C4"):
            getattr(arr[i], name)[:] = [float(v) for v in np.asarray(c[name], np.float32).reshape(3)]
        for name in ("fx", "fy", "f", "alpha", "baseline", "depthMin", "depthMax"):
            setattr(arr[i], name, float(np.float32(c[name])))
    return arr


class DepthmapEngine:
    """One reference view in flight on one GPU (reference: one gipuma process per view)."""

    def __init__(self, device=0, stream=None):
        self.lib = L.load()
        h = C.c_void_p()
        rc = self.lib.tsar_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise TsarError(f"tsar_create(device={device}) failed with {rc}: no usable sm_100 GPU (there is no CPU path)")
        self.h = h
        self.W = self.H = 0
        self._keep = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.tsar_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise TsarError(f"{what} failed ({rc}): {self.lib.tsar_last_error(self.h).decode()}")

    # -- inputs ----------------------------------------------------------------------------------
    def set_views(self, images, cams, subset, cam_f=None):
        """images: [n][H][W] float32 numpy (host) -- image 0 is the reference view."""
        imgs = [np.ascontiguousarray(im, np.float32) for im in images]
        H, W = imgs[0].shape
        ptrs = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
        cs = cameras_to_struct(cams) if not isinstance(cams, C.Array) else cams
        sub = (C.c_int * len(subset))(*[int(s) for s in subset])
        f = float(cam_f if cam_f is not None else cs[0].f)
        self._ck(self.lib.tsar_set_views(self.h, W, H, len(imgs), ptrs, 0, cs, f, sub, len(subset)), "tsar_set_views")
        self.W, self.H = W, H
        self._keep = (imgs, cs, sub)

    def set_views_device(self, dev_ptrs, W, H, cams, subset, cam_f=None):
        """Same, from device pointers (e.g. torch tensors already resident in HBM)."""
        ptrs = (C.c_void_p * len(dev_ptrs))(*[int(p) for p in dev_ptrs])
        cs = cameras_to_struct(cams) if not isinstance(cams, C.Array) else cams
        sub = (C.c_int * len(subset))(*[int(s) for s in subset])
        f = float(cam_f if cam_f is not None else cs[0].f)
        self._ck(self.lib.tsar_set_views(self.h, W, H, len(dev_ptrs), ptrs, 1, cs, f, sub, len(subset)), "tsar_set_views")
        self.W, self.H = W, H
        self._keep = (cs, sub)

    def set_params(self, params):
        self.params = params
        self._ck(self.lib.tsar_set_params(self.h, C.byref(params)), "tsar_set_params")

    def set_regions(self, text, norm4):
        text = np.ascontiguousarray(text, np.float32)
        norm4 = np.ascontiguousarray(norm4, np.float32).reshape(-1, 4)
        self._ck(self.lib.tsar_set_regions(self.h, len(text), text.ctypes.data, norm4.ctypes.data), "tsar_set_regions")

    def set_labels_quarter(self, labels_q):
        """lines->canny from the quarter-resolution region labels of texture.detect (main.cpp:558-568), expanded on
        the device."""
        lab = np.ascontiguousarray(labels_q, np.int32)
        self._ck(self.lib.tsar_set_labels_quarter(self.h, lab.ctypes.data, lab.shape[1], lab.shape[0]), "tsar_set_labels_quarter")

    def scale_from_confidence(self, threshold=0.8):
        """lines->scale = (confid > threshold): stands in for APD's weak.png when PatchMatch runs in the library."""
        self._ck(self.lib.tsar_scale_from_confidence(self.h, float(threshold)), "tsar_scale_from_confidence")

    def scale_from_weak_png(self, bgr):
        """lines->scale from the decoded APD/<view>/weak.png (H x W x 3 uint8, BGR): main.cpp:1499-1514."""
        bgr = np.ascontiguousarray(bgr, np.uint8)
        if bgr.shape != (self.H, self.W, 3):
            raise TsarError(f"weak.png is {bgr.shape}, expected {(self.H, self.W, 3)}")
        self._ck(self.lib.tsar_scale_from_weak_png(self.h, bgr.ctypes.data), "tsar_scale_from_weak_png")

    def download_outputs(self, depth=None, normals=None, confid=None):
        """File payloads after compute_disp: depth [H][W], normals [H][W][3], confidence [H][W] (numpy arrays or raw
        addresses of host buffers of those sizes; missing ones are allocated).  Returns (depth, normals, confid)."""
        def buf(a, shape):
            return np.empty(shape, np.float32) if a is None else a
        depth, normals, confid = buf(depth, (self.H, self.W)), buf(normals, (self.H, self.W, 3)), buf(confid, (self.H, self.W))
        ptr = lambda a: a if isinstance(a, int) else a.ctypes.data
        self._ck(self.lib.tsar_download_outputs(self.h, ptr(depth), ptr(normals), ptr(confid)), "tsar_download_outputs")
        return depth, normals, confid

    def fit_region_planes(self, region_text, region_size, rnd, region_norm4, seed=None):
        """Per-region RANSAC plane fit (main.cpp:1520-1730) for regions with text == -1.  rnd: [n_regions][46000] uint32
        (the values rand() would return), or None to let the device generate the stream of `seed`
        (tsar_fit_region_planes_seeded).  Returns the updated [n_regions][4] planes."""
        text = np.ascontiguousarray(region_text, np.float32)
        size = np.ascontiguousarray(region_size, np.float32)
        planes = np.ascontiguousarray(region_norm4, np.float32).reshape(len(text), 4).copy()
        if rnd is None:
            self._ck(self.lib.tsar_fit_region_planes_seeded(self.h, len(text), text.ctypes.data, size.ctypes.data, int(seed or 0),
                                                            planes.ctypes.data), "tsar_fit_region_planes_seeded")
            return planes
        per = self.lib.tsar_ransac_rand_per_region()
        rnd = np.ascontiguousarray(rnd, np.uint32).reshape(len(text), per)
        self._ck(self.lib.tsar_fit_region_planes(self.h, len(text), text.ctypes.data, size.ctypes.data, rnd.ctypes.data,
                                                 planes.ctypes.data), "tsar_fit_region_planes")
        return planes

    def ransac_rand_stream(self, seed, region):
        """The device stream of tsar_fit_region_planes_seeded for one region (host restatement, for checkers)."""
        per = self.lib.tsar_ransac_rand_per_region()
        z = (np.uint64(seed) ^ (np.uint64(region) << np.uint64(32)) ^ np.arange(per, dtype=np.uint64)) + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
        return (z >> np.uint64(33)).astype(np.uint32)

    # -- PatchMatch path ---------------------------------------------------------------------------
    def init_planes(self, seed):                      # gipuma_init_cu2
        self._ck(self.lib.tsar_init_planes(self.h, int(seed)), "tsar_init_planes")

    def load_planes(self, norm4, cost=None):
        norm4 = np.ascontiguousarray(norm4, np.float32)
        cost = None if cost is None else np.ascontiguousarray(cost, np.float32)
        self._ck(self.lib.tsar_load_planes(self.h, norm4.ctypes.data, cost.ctypes.data if cost is not None else None),
                 "tsar_load_planes")

    def launch(self, kind, seed=0):                   # one checkerboard half-step
        self._ck(self.lib.tsar_launch(self.h, int(kind), int(seed)), "tsar_launch")

    def iterate(self, iters, seed0, refine_seeds=None):
        arr = None
        if refine_seeds is not None:
            arr = (C.c_uint64 * len(refine_seeds))(*[int(s) for s in refine_seeds])
        self._ck(self.lib.tsar_iterate(self.h, int(iters), int(seed0), arr), "tsar_iterate")

    def eval_planes(self, xy, planes, wrapper_rounding=False):   # pmCostMultiview_cu on explicit pairs
        self._ck(self.lib.tsar_dbg_eval_rounding(self.h, int(bool(wrapper_rounding))), "tsar_dbg_eval_rounding")
        xy = np.ascontiguousarray(xy, np.int32).reshape(-1, 2)
        planes = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
        n = len(xy)
        cost = np.empty(n, np.float32)
        bv = np.empty(n, np.int32)
        ratio = np.empty(n, np.float32)
        self._ck(self.lib.tsar_eval_planes(self.h, n, xy.ctypes.data, planes.ctypes.data, cost.ctypes.data,
                                           bv.ctypes.data, ratio.ctypes.data), "tsar_eval_planes")
        return cost, bv, ratio

    def lrdiff(self): self._ck(self.lib.tsar_lrdiff(self.h), "tsar_lrdiff")                      # gipuma_getlrdiff
    def getview(self): self._ck(self.lib.tsar_getview(self.h), "tsar_getview")                   # gipuma_getview
    def get_disp(self): self._ck(self.lib.tsar_get_disp(self.h), "tsar_get_disp")                # gipuma_get_disp
    def update_scale_2(self): self._ck(self.lib.tsar_update_scale_2(self.h), "tsar_update_scale_2")
    def update_scale(self): self._ck(self.lib.tsar_update_scale(self.h), "tsar_update_scale")
    def compute_disp(self): self._ck(self.lib.tsar_compute_disp(self.h), "tsar_compute_disp")
    def wmf(self, it): self._ck(self.lib.tsar_wmf(self.h, int(it)), "tsar_wmf")
    def wmf_final(self, it): self._ck(self.lib.tsar_wmf_final(self.h, int(it)), "tsar_wmf_final")

    def depthmap(self, seed0, timed=True):
        """init -> iterations -> lrdiff -> getview -> compute_disp, resident. Returns CUDA-event ms."""
        ms = C.c_float(0)
        self._ck(self.lib.tsar_depthmap(self.h, int(seed0), C.byref(ms) if timed else None), "tsar_depthmap")
        return ms.value

    def depthmap_host(self, images, cams, subset, params, seed0, want_norm4=True, want_confid=True, cam_f=None,
                      out_norm4=None, out_confid=None):
        """The end-to-end call: host images in, host depth/normal/confidence out."""
        imgs = [np.ascontiguousarray(im, np.float32) for im in images]
        H, W = imgs[0].shape
        ptrs = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
        cs = cameras_to_struct(cams) if not isinstance(cams, C.Array) else cams
        sub = (C.c_int * len(subset))(*[int(s) for s in subset])
        f = float(cam_f if cam_f is not None else cs[0].f)
        if out_norm4 is None and want_norm4:
            out_norm4 = np.empty((H, W, 4), np.float32)
        if out_confid is None and want_confid:
            out_confid = np.empty((H, W), np.float32)
        self._ck(self.lib.tsar_depthmap_host(self.h, W, H, len(imgs), ptrs, cs, f, sub, len(subset), C.byref(params),
                                             int(seed0), out_norm4.ctypes.data if out_norm4 is not None else None,
                                             out_confid.ctypes.data if out_confid is not None else None),
                 "tsar_depthmap_host")
        self.W, self.H = W, H
        self.params = params
        return out_norm4, out_confid

    # -- state -----------------------------------------------------------------------------------
    def download(self, field, n_regions=None):
        dt, ch = FIELD_DTYPE[field]
        if field in (L.F_REGION_TEXT, L.F_REGION_NORM4):
            shape = (n_regions,) if ch == 1 else (n_regions, ch)
        else:
            shape = (self.H, self.W) if ch == 1 else (self.H, self.W, ch)
        out = np.empty(shape, dt)
        self._ck(self.lib.tsar_download(self.h, field, out.ctypes.data, out.nbytes), "tsar_download")
        return out

    def upload(self, field, arr):
        dt, _ = FIELD_DTYPE[field]
        arr = np.ascontiguousarray(arr, dt)
        self._ck(self.lib.tsar_upload(self.h, field, arr.ctypes.data, arr.nbytes), "tsar_upload")

    def sync(self):
        self._ck(self.lib.tsar_sync(self.h), "tsar_sync")

    def launch_count(self, reset=False):
        n = C.c_longlong(0)
        self._ck(self.lib.tsar_launch_count(self.h, C.byref(n), int(reset)), "tsar_launch_count")
        return n.value

    def eval_count(self, iters):
        n = C.c_longlong(0)
        self._ck(self.lib.tsar_eval_count(self.h, int(iters), C.byref(n)), "tsar_eval_count")
        return n.value

    def profile(self, enable=True):
        self._ck(self.lib.tsar_profile(self.h, int(enable)), "tsar_profile")

    def profile_read(self):
        """(summed CUDA-event ms of the checkerboard kernels, number of launches) since profiling was enabled."""
        ms, n = C.c_float(0), C.c_int(0)
        self._ck(self.lib.tsar_profile_read(self.h, C.byref(ms), C.byref(n)), "tsar_profile_read")
        return ms.value, n.value

    def profile_read_launches(self, cap=4096):
        """CUDA-event ms of each checkerboard launch since profiling was enabled (consumes them, as profile_read)."""
        ms, n = (C.c_float * cap)(), C.c_int(0)
        self._ck(self.lib.tsar_profile_read_launches(self.h, ms, int(cap), C.byref(n)), "tsar_profile_read_launches")
        return [ms[k] for k in range(min(n.value, cap))]

    def quad_sampling(self, checker_launches):
        """tsar_dbg_quad_sampling: < 0 off; >= 0 init and the first checker_launches checkerboard launches."""
        self._ck(self.lib.tsar_dbg_quad_sampling(self.h, int(checker_launches)), "tsar_dbg_quad_sampling")

    def candidate_stats(self, colour):
        """Counters of the propagation candidates the checkerboard launch of `colour` would try on the current state
        (tsar_dbg_candidate_stats): dict of counts + histogram of distinct candidates per pixel."""
        out = (C.c_ulonglong * 22)()
        self._ck(self.lib.tsar_dbg_candidate_stats(self.h, int(colour), out), "tsar_dbg_candidate_stats")
        names = ("pixels", "behind_border_guards", "in_depth_range", "dup_of_own_plane", "dup_of_earlier_candidate", "distinct",
                 "warp_rounds_as_written", "warp_rounds_lane_lists", "warp_rounds_packed", "warps", "distinct_without_own_rule",
                 "warp_rounds_lane_lists_without_own_rule", "warp_rounds_packed_without_own_rule")
        d = {n: int(out[k]) for k, n in enumerate(names)}
        d["pixels_by_distinct"] = [int(out[13 + k]) for k in range(9)]
        return d

    def peaks(self):
        """Issue-rate microbenchmarks: (FP32 FFMA TFLOP/s, MUFU Gop/s, bilinear texture Gsamples/s)."""
        out = (C.c_float * 3)()
        self._ck(self.lib.tsar_dbg_peaks(self.h, out), "tsar_dbg_peaks")
        return out[0], out[1], out[2]

    # -- gSLICr ------------------------------------------------------------------------------------
    def slic(self, bgrx, spixel_size=20, no_iters=5, coh_weight=5.0, enforce_connectivity=False,
             correct_reduction=False):
        """core_engine::Process_Frame + Get_Seg_Res. bgrx: [h][w][4] uint8 (B,G,R,x). Returns int32 labels."""
        bgrx = np.ascontiguousarray(bgrx, np.uint8)
        h, w = bgrx.shape[:2]
        s = L.TsarSlicSettings(w, h, spixel_size, no_iters, coh_weight, int(enforce_connectivity), int(correct_reduction))
        labels = np.empty((h, w), np.int32)
        self._ck(self.lib.tsar_slic(self.h, bgrx.ctypes.data, C.byref(s), labels.ctypes.data), "tsar_slic")
        return labels
