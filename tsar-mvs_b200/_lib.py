"""ctypes binding of the C ABI in include/tsar_b200.h (libtsar_b200.so, built in-tree by `make`).

There is no Python or CPU fallback: if the CUDA library is missing the import of the engine fails
loudly with build instructions.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtsar_b200.so")

TSAR_MAX_VIEWS = 32


class TsarCamera(C.Structure):
    """tsar_camera (include/tsar_b200.h) == value fields of Camera_cu (reference camera.h:7-65)."""
    _fields_ = [
        ("K", C.c_float * 9), ("K_inv", C.c_float * 9), ("R", C.c_float * 9), ("R_orig", C.c_float * 9),
        ("R_orig_inv", C.c_float * 9), ("M_inv", C.c_float * 9), ("t4", C.c_float * 3),
        ("P_col34", C.c_float * 3), ("C4", C.c_float * 3),
        ("fx", C.c_float), ("fy", C.c_float), ("f", C.c_float), ("alpha", C.c_float), ("baseline", C.c_float),
        ("depthMin", C.c_float), ("depthMax", C.c_float),
    ]


class TsarParams(C.Structure):
    """tsar_params == hot fields of AlgorithmParameters (reference algorithmparameters.h:19-89)."""
    _fields_ = [
        ("box_hsize", C.c_int), ("box_vsize", C.c_int), ("iterations", C.c_int), ("n_best", C.c_int),
        ("cost_comb", C.c_int), ("min_disparity", C.c_float), ("max_disparity", C.c_float),
        ("color_processing", C.c_int),
    ]


class TsarSlicSettings(C.Structure):
    """tsar_slic_settings == gSLICr::objects::settings (reference gSLICr_settings.h:10-21)."""
    _fields_ = [
        ("img_w", C.c_int), ("img_h", C.c_int), ("spixel_size", C.c_int), ("no_iters", C.c_int),
        ("coh_weight", C.c_float), ("do_enforce_connectivity", C.c_int), ("correct_reduction", C.c_int),
    ]


class TsarViewCamera(C.Structure):
    """tsar_view_camera: world -> camera K, R, t of one view (row-major)."""
    _fields_ = [("K", C.c_float * 9), ("R", C.c_float * 9), ("t", C.c_float * 3)]


class TsarFusionParams(C.Structure):
    """tsar_fusion_params (DESIGN.md section 4.6)."""
    _fields_ = [("max_reproj_px", C.c_float), ("max_rel_depth", C.c_float), ("max_normal_deg", C.c_float),
                ("min_consistent", C.c_int)]


class TsarMeshGrid(C.Structure):
    """tsar_mesh_grid (DESIGN.md section 4.8): grid point (i, j, k) at origin + ((float)i + 0.5f, ...) * voxel."""
    _fields_ = [("origin", C.c_float * 3), ("voxel", C.c_float), ("dims", C.c_int * 3)]


class TsarMeshParams(C.Structure):
    """tsar_mesh_params (DESIGN.md section 4.8)."""
    _fields_ = [("trunc", C.c_float), ("min_weight", C.c_int)]


# tsar_field
F_NORM4, F_COST, F_DEPTH, F_FAKEDEPTH, F_SCALE, F_CANNY, F_RATIO, F_BEVIEW, F_LRDIFF, F_CONFID, \
    F_REGION_TEXT, F_REGION_NORM4 = range(12)
# launch kinds
BLACK_SPATIAL, BLACK_REFINE, RED_SPATIAL, RED_REFINE = range(4)

EXPORTS = [
    "tsar_create", "tsar_destroy", "tsar_last_error", "tsar_sync", "tsar_set_views", "tsar_set_params",
    "tsar_init_planes", "tsar_load_planes", "tsar_launch", "tsar_iterate", "tsar_eval_planes", "tsar_lrdiff",
    "tsar_getview", "tsar_get_disp", "tsar_update_scale_2", "tsar_update_scale", "tsar_compute_disp", "tsar_wmf",
    "tsar_wmf_final", "tsar_set_regions", "tsar_fit_region_planes", "tsar_fit_region_planes_seeded", "tsar_ransac_rand_value", "tsar_ransac_rand_per_region", "tsar_upload", "tsar_download", "tsar_device_ptr", "tsar_depthmap",
    "tsar_depthmap_host", "tsar_slic", "tsar_launch_count", "tsar_eval_count", "tsar_version", "tsar_dbg_tex_sample", "tsar_dbg_peaks", "tsar_dbg_eval_rounding", "tsar_dbg_quad_sampling", "tsar_dbg_candidate_stats", "tsar_dbg_tex_formats", "tsar_profile", "tsar_profile_read", "tsar_profile_read_launches",
    "tsar_weak_edges", "tsar_weak_connect", "tsar_weak_boundary", "tsar_weak_close_border", "tsar_weak_regions", "tsar_set_labels_quarter", "tsar_scale_from_weak_png", "tsar_scale_from_confidence", "tsar_download_outputs",
    "tsar_fusion_create", "tsar_fusion_set_view", "tsar_fusion_run", "tsar_fusion_points", "tsar_fusion_destroy",
    "tsar_fusion_last_error", "tsar_fusion_dbg_rounds",
    "tsar_eval_create", "tsar_eval_run", "tsar_eval_destroy", "tsar_eval_last_error", "tsar_eval_dbg_visits",
    "tsar_mesh_create", "tsar_mesh_set_view", "tsar_mesh_run", "tsar_mesh_get", "tsar_mesh_destroy", "tsar_mesh_last_error",
    "tsar_mesh_dbg_extract", "tsar_mesh_dbg_field", "tsar_mesh_dbg_times",
]


class LibraryMissing(RuntimeError):
    pass


_lib = None


def load():
    """Load libtsar_b200.so (RTLD_GLOBAL so profilers see its kernels). Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} not found: build the CUDA library first (`make` at the repo root, or "
            f"`python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i, u64 = C.c_void_p, C.c_int, C.c_uint64
    fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int)
    sig = {
        "tsar_create": (i, [i, vp, C.POINTER(vp)]),
        "tsar_destroy": (i, [vp]),
        "tsar_last_error": (C.c_char_p, [vp]),
        "tsar_sync": (i, [vp]),
        "tsar_set_views": (i, [vp, i, i, i, C.POINTER(vp), i, C.POINTER(TsarCamera), C.c_float, ip, i]),
        "tsar_set_params": (i, [vp, C.POINTER(TsarParams)]),
        "tsar_init_planes": (i, [vp, u64]),
        "tsar_load_planes": (i, [vp, vp, vp]),
        "tsar_launch": (i, [vp, i, u64]),
        "tsar_iterate": (i, [vp, i, u64, C.POINTER(u64)]),
        "tsar_eval_planes": (i, [vp, i, vp, vp, vp, vp, vp]),
        "tsar_lrdiff": (i, [vp]), "tsar_getview": (i, [vp]), "tsar_get_disp": (i, [vp]),
        "tsar_update_scale_2": (i, [vp]), "tsar_update_scale": (i, [vp]), "tsar_compute_disp": (i, [vp]),
        "tsar_wmf": (i, [vp, i]), "tsar_wmf_final": (i, [vp, i]),
        "tsar_set_regions": (i, [vp, i, vp, vp]),
        "tsar_fit_region_planes": (i, [vp, i, vp, vp, vp, vp]),
        "tsar_fit_region_planes_seeded": (i, [vp, i, vp, vp, u64, vp]),
        "tsar_ransac_rand_value": (C.c_uint32, [u64, i, i]),
        "tsar_ransac_rand_per_region": (i, []),
        "tsar_upload": (i, [vp, i, vp, C.c_size_t]),
        "tsar_download": (i, [vp, i, vp, C.c_size_t]),
        "tsar_device_ptr": (i, [vp, i, C.POINTER(vp)]),
        "tsar_depthmap": (i, [vp, u64, fp]),
        "tsar_depthmap_host": (i, [vp, i, i, i, C.POINTER(vp), C.POINTER(TsarCamera), C.c_float, ip, i,
                                   C.POINTER(TsarParams), u64, vp, vp]),
        "tsar_slic": (i, [vp, vp, C.POINTER(TsarSlicSettings), vp]),
        "tsar_launch_count": (i, [vp, C.POINTER(C.c_longlong), i]),
        "tsar_eval_count": (i, [vp, i, C.POINTER(C.c_longlong)]),
        "tsar_version": (C.c_char_p, []),
        "tsar_dbg_tex_sample": (i, [vp, i, i, vp, vp]),
        "tsar_dbg_peaks": (i, [vp, fp]),
        "tsar_dbg_eval_rounding": (i, [vp, i]),
        "tsar_dbg_quad_sampling": (i, [vp, i]),
        "tsar_dbg_candidate_stats": (i, [vp, i, vp]),
        "tsar_dbg_tex_formats": (i, [vp, i, i, vp, vp, vp]),
        "tsar_profile": (i, [vp, i]),
        "tsar_profile_read": (i, [vp, fp, ip]),
        "tsar_profile_read_launches": (i, [vp, fp, i, ip]),
        "tsar_weak_edges": (i, [vp, i, i, i, vp]),
        "tsar_weak_connect": (i, [vp, i, i, vp, vp, i, ip]),
        "tsar_weak_boundary": (i, [vp, i, i, i, vp]),
        "tsar_weak_close_border": (i, [vp, i, i]),
        "tsar_weak_regions": (i, [vp, i, i, vp, i, i, i, vp, vp, vp, vp]),
        "tsar_set_labels_quarter": (i, [vp, vp, i, i]),
        "tsar_scale_from_weak_png": (i, [vp, vp]),
        "tsar_scale_from_confidence": (i, [vp, C.c_float]),
        "tsar_download_outputs": (i, [vp, vp, vp, vp]),
        "tsar_fusion_create": (i, [i, vp, i, i, i, C.POINTER(vp)]),
        "tsar_fusion_set_view": (i, [vp, i, C.POINTER(TsarViewCamera), vp, vp, vp, ip, i]),
        "tsar_fusion_run": (i, [vp, C.POINTER(TsarFusionParams), C.POINTER(C.c_longlong)]),
        "tsar_fusion_points": (i, [vp, vp, vp, vp, C.c_longlong]),
        "tsar_fusion_destroy": (i, [vp]),
        "tsar_fusion_last_error": (C.c_char_p, [vp]),
        "tsar_fusion_dbg_rounds": (i, [vp, ip, C.POINTER(C.c_longlong)]),
        "tsar_eval_create": (i, [i, vp, C.POINTER(vp)]),
        "tsar_eval_run": (i, [vp, vp, C.c_longlong, vp, C.c_longlong, vp, i, C.c_float, vp, vp, vp, vp]),
        "tsar_eval_destroy": (i, [vp]),
        "tsar_eval_last_error": (C.c_char_p, [vp]),
        "tsar_eval_dbg_visits": (i, [vp, vp, vp]),
        "tsar_mesh_create": (i, [i, vp, i, i, i, C.POINTER(vp)]),
        "tsar_mesh_set_view": (i, [vp, i, C.POINTER(TsarViewCamera), vp, vp]),
        "tsar_mesh_run": (i, [vp, C.POINTER(TsarMeshGrid), C.POINTER(TsarMeshParams), C.POINTER(C.c_longlong),
                              C.POINTER(C.c_longlong)]),
        "tsar_mesh_get": (i, [vp, vp, vp, C.c_longlong, vp, C.c_longlong]),
        "tsar_mesh_destroy": (i, [vp]),
        "tsar_mesh_last_error": (C.c_char_p, [vp]),
        "tsar_mesh_dbg_extract": (i, [vp, C.POINTER(TsarMeshGrid), i, vp, vp, vp, vp, C.POINTER(C.c_longlong),
                                      C.POINTER(C.c_longlong)]),
        "tsar_mesh_dbg_field": (i, [vp, vp, vp, vp, vp]),
        "tsar_mesh_dbg_times": (i, [vp, fp, fp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
