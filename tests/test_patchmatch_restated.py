"""The PatchMatch core on the GPU against the C restatement (oracle/oracle_cpu.c, `CpuOracle`) at any shape.

The recorded-digest tests (test_parity_gpu.py) hold the product to the reference build at the calls that were recorded;
they cannot check a new configuration.  Here both sides run on the same images, cameras and parameters, with no
reference checkout and no digests: the product through `DepthmapEngine`, the checker through `CpuOracle`.  Covered:
1..32 source views, n_best up to V with both cost combinations, square windows 3..27 (even ones too), rectangular windows
up to the largest the shared-memory weight table takes, 8-bit and fp32 textures, pinhole and skewed intrinsics, image
widths 1 and 31 (mod 32), heights 32 m + 1 (rows past the checkerboard grid), and a C5-size scene at its last columns.

Tolerances.  The GPU takes expf (bilateral weights) and rsqrtf (normals) from the MUFU unit, the oracle from libm, so
costs agree to TOL where the window is well conditioned.  A pair is ill-conditioned when its window touches the scene's
textureless facet (grey levels 128/129; dilated by the window radius), or when the float64 relative variance
var / E[v^2] of the bilateral-weighted samples is below REL_VAR_MIN on the reference side or in the source window of any
view (the oracle reports the latter): the fp32 variance E[v^2] - E[v]^2 then cancels to a few significant bits in any
implementation, and the `var < 1e-5` test of pmCost (cost 2) flips on rounding noise.  Source windows are degenerate
where they fall into the textureless facet of a source view or far outside it (every sample clamped to one border
texel), which random and hostile planes do often.  Those pairs get the loose bound and are counted.  Accept / reject
decisions of the checkerboard launches flip on near-ties, so launches are compared by invariants (see
test_checkerboard_launches_match_restatement), and the pixels where the product's choice is worse than the oracle's are
counted.  Every count goes to pc.record.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.ndimage import maximum_filter

from tests import parity_common as pc
from tests.test_quad_sampling import _compare_run, _hostile_planes

pytestmark = pytest.mark.gpu

TOL = 5e-5             # cost, well-conditioned window (test_cpu.test_oracle_cost_matches_reference_build)
LOOSE = 5e-2           # cost, ill-conditioned window
REL_VAR_MIN = 1e-2     # var / E[v^2] of a reference or source window below this: ill-conditioned
PLANE_RTOL = 2e-5      # refined normals pass through rsqrtf
SEED = 6060
TSAR_ERR_ARG = -1      # include/tsar_b200.h
# Bounds set from one run of this file on an NVIDIA B200 at its 1000 W power limit, measured figure in brackets:
#  - ill-conditioned pairs beyond LOOSE: 5 % of them per configuration (at most 1.3 %; 48.7 % of the 133 536 pairs of
#    the pair tests are ill-conditioned, the largest well-conditioned difference is 3.4e-5);
#  - launch pixels (well-conditioned) whose plane is worse than the oracle's choice by more than 2 TOL, as a fraction
#    of the launch's pixels: propagation 0 (0), refinement 0.2 % (0.03 %: 1 pixel), fused iteration 0.5 % (0.08 %);
#  - 8-iteration depth map, V = 32, 11 x 7 window: textured pixels within 1 % of the true depth >= 0.90 (0.932).
WORSE_BOUND = {"spatial": 0.0, "refine": 0.002, "fused": 0.005}
GT_FLOOR = 0.90


# ---- scenes ------------------------------------------------------------------------------------------------
# Two shapes: W = 97 = 1 (mod 32) with H = 65, and W = 95 = 31 (mod 32) with H = 97; both H = 32 m + 1, so the last row
# lies beyond the checkerboard grid (y_limit = 64 and 96).  33 images each, so any V <= 32 selects a prefix.
SHAPES = {"A": (97, 65), "B": (95, 97)}


def _y_limit(H):
    return min(H, 32 * ((H // 2 + 15) // 16))


def _skewed_cameras(pkg, cams):
    """The same poses with skewed intrinsics, and focal lengths of their own in every source view: the homography takes
    its general form (no zero-skew pinhole shortcut)."""
    Ks = []
    for i, c in enumerate(cams):
        K = np.array(c["K"], float)
        K[0, 1] = 0.02 * K[0, 0]
        if i:
            K[0, 0] *= 1.0 + 0.004 * i
            K[1, 1] *= 1.0 - 0.003 * i
        Ks.append(K)
    Rs = [c["_R_world"] for c in cams]
    ts = [-c["_R_world"] @ c["_C_world"] for c in cams]
    return pkg.scene.cameras_from_krt(Ks, Rs, ts, cams[0]["depthMin"], cams[0]["depthMax"])


_SCENES = {}


def _scene(pkg, shape, fp32=False, skew=False):
    """fp32: images that are not 8-bit valued (the library then samples fp32 textures)."""
    key = (shape, fp32, skew)
    if key not in _SCENES:
        W, H = SHAPES[shape]
        s = pkg.scene.make_scene(dict(W=W, H=H, n_images=33, V=32, fx=3.2 * W, radius=1.5, arc_deg=30.0), seed=W * H)
        if fp32:
            s["images"] = [im * np.float32(0.8125) + np.float32(0.3) for im in s["images"]]
        if skew:
            s["cams"] = _skewed_cameras(pkg, s["cams"])
        _SCENES[key] = s
    return _SCENES[key]


def _params(pkg, scene, box, n_best, cost_comb, iterations=8):
    hs, vs = box
    return pkg._lib.TsarParams(hs, vs, iterations, n_best, cost_comb, scene["min_disparity"], scene["max_disparity"], 0)


def _pair(pkg, scene, V, params):
    """(product engine, oracle) on the first V source views of the scene."""
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    subset = list(range(1, V + 1))
    eng = pkg.DepthmapEngine(0)
    eng.set_views(scene["images"], cams, subset, cam_f=scene["cam_f"])
    eng.set_params(params)
    ora = cb.CpuOracle(pkg._lib.TsarCamera, pkg._lib.TsarParams, scene["images"], cams, subset, params, scene["cam_f"])
    return eng, ora


# ---- pairs and their conditioning -------------------------------------------------------------------------------
def _planes_at(scene, xy, rng):
    """A plane through a random depth of the range at each pixel, normal facing the camera (as pc.random_planes)."""
    cam = scene["cams"][0]
    n = len(xy)
    depth = rng.uniform(cam["depthMin"], cam["depthMax"], n)
    nrm = rng.normal(size=(n, 3))
    nrm[:, 2] = -np.abs(nrm[:, 2]) - 0.3
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    X = (np.asarray(cam["K_inv"], float) @ np.stack([xy[:, 0], xy[:, 1], np.ones(n)]).astype(float)).T * depth[:, None]
    return np.concatenate([nrm, -np.sum(nrm * X, axis=1)[:, None]], axis=1).astype(np.float32)


def _pairs(scene, n=2400, n_hostile=600, seed=11):
    """Random pixels (an eighth forced onto each border band by pc.random_planes), the four corners and their
    neighbours, and hostile planes (zero / huge / tiny / grazing normals, offsets 0, +-1e30, inf, NaN)."""
    rng = np.random.RandomState(seed)
    W, H = scene["W"], scene["H"]
    xy, pl = pc.random_planes(scene, n, seed=seed)
    cxy = np.array([[0, 0], [W - 1, 0], [0, H - 1], [W - 1, H - 1], [1, 1], [W - 2, 1], [1, H - 2], [W - 2, H - 2]] * 4,
                   np.int32)
    idx = rng.choice(W * H, n_hostile, replace=False)
    hxy = np.stack([idx % W, idx // W], axis=1).astype(np.int32)
    hpl = _hostile_planes(scene, seed).reshape(-1, 4)[idx]
    return np.concatenate([xy, cxy, hxy]), np.concatenate([pl, _planes_at(scene, cxy, rng), hpl])


def _ill_conditioned(scene, xy, hr, vr):
    """Pairs whose window touches the textureless facet, or whose reference side has relative variance below
    REL_VAR_MIN (float64, the bilateral weights of pmCost).  Returns (mask, relative variance)."""
    ref = np.asarray(scene["images"][0], np.float64)
    H, W = ref.shape
    flat = scene["region_text"][scene["labels"]] < 0
    near_flat = maximum_filter(flat, size=(2 * vr + 1, 2 * hr + 1), mode="nearest")
    di, dj = np.meshgrid(np.arange(-hr, hr + 1, 2), np.arange(-vr, vr + 1, 2), indexing="ij")
    di, dj = di.reshape(-1), dj.reshape(-1)
    x, y = xy[:, 0].astype(np.int64), xy[:, 1].astype(np.int64)
    r = ref[np.clip(y[:, None] + dj, 0, H - 1), np.clip(x[:, None] + di, 0, W - 1)]
    cen = ref[y, x][:, None]
    w = np.exp(-np.sqrt(di * di + dj * dj) / 50.0 - np.abs(r - cen) / 18.0)
    m1 = (w * r).sum(1) / w.sum(1)
    m2 = (w * r * r).sum(1) / w.sum(1)
    rel = (m2 - m1 * m1) / m2
    return near_flat[y, x] | (rel < REL_VAR_MIN), rel


def _check_costs(gpu, ora, views, ill, V, what, cond=None):
    """gpu / ora: (cost, best view, ratio) of the same pairs; views: the oracle's [n][V] per-view costs.
    Cost within TOL (well-conditioned) or LOOSE (counted); best view equal unless the oracle's two smallest view costs
    are within 2 TOL; ratio within the error TOL implies for cv0 / cv1; with one view the ratio is exactly 0."""
    c_g, b_g, r_g = gpu
    c_o, b_o, r_o = ora
    well = ~ill
    d = np.abs(c_g.astype(np.float64) - c_o)
    sv = np.sort(np.minimum(views.astype(np.float64), 2.0), axis=1)
    tie = (sv[:, 1] - sv[:, 0] <= 2 * TOL) if V > 1 else np.zeros(len(d), bool)
    if V > 1:
        cv0, cv1 = sv[:, 0], sv[:, 1]
        r_tol = np.where(cv1 > 2 * TOL, TOL * (1.0 + r_o) / np.maximum(cv1 - TOL, TOL) + 1e-6, np.inf)
        r_bad = well & ~(np.abs(r_g.astype(np.float64) - r_o) <= r_tol)
    else:
        r_bad = ~((r_g == 0) & (r_o == 0))
    stats = dict(what=what, n=int(len(d)), ill=int(ill.sum()), well_over_tol=int((well & ~(d <= TOL)).sum()),
                 max_d_well=float(d[well].max()) if well.any() else 0.0,
                 ill_over_tol=int((ill & ~(d <= TOL)).sum()), ill_over_loose=int((ill & ~(d <= LOOSE)).sum()),
                 ties=int(tie.sum()), beview_diff=int((well & ~tie & (b_g != b_o)).sum()), ratio_bad=int(r_bad.sum()),
                 ratio_v1_nonzero=int((r_g != 0).sum()) if V == 1 else 0)
    if cond is not None:   # the worst well-conditioned pairs: (cost difference, smallest relative variance)
        k = np.argsort(np.where(well, d, -1.0))[::-1][:5]
        stats["worst_well"] = [(float(d[i]), float(cond[i])) for i in k if well[i]]
    return stats


def _assert_costs(stats, ill_loose_frac=0.05):
    s = stats
    assert s["ratio_v1_nonzero"] == 0, f"{s['what']}: with one view the ratio must be exactly 0: {s}"
    assert s["well_over_tol"] == 0, f"{s['what']}: cost beyond {TOL} on well-conditioned windows: {s}"
    assert s["beview_diff"] == 0, f"{s['what']}: best view differs away from ties: {s}"
    assert s["ratio_bad"] == 0, f"{s['what']}: ratio beyond its bound: {s}"
    assert s["ill_over_loose"] <= ill_loose_frac * max(1, s["ill"]), f"{s['what']}: ill-conditioned beyond {LOOSE}: {s}"


def _oracle_views(ora, scene, xy, planes, hr, vr, wrapper_rounding=False):
    """The oracle's per-view costs of the pairs and their ill-conditioned mask (reference side and every source view)."""
    ill, ref_rel = _ill_conditioned(scene, xy, hr, vr)
    views, src_rel = ora.eval_views(xy, planes, wrapper_rounding=wrapper_rounding)
    return views, ill | (src_rel < REL_VAR_MIN).any(axis=1), np.minimum(ref_rel, src_rel.min(axis=1))


def _compare_pairs(eng, ora, scene, V, box, xy, planes, wrapper_rounding, what):
    views, ill, cond = _oracle_views(ora, scene, xy, planes, (box[0] - 1) // 2, (box[1] - 1) // 2, wrapper_rounding)
    gpu = eng.eval_planes(xy, planes, wrapper_rounding=wrapper_rounding)
    ref = ora.eval_planes(xy, planes, wrapper_rounding=wrapper_rounding)
    return _check_costs(gpu, ref, views, ill, V, what, cond)


# ---- 1. cost of explicit pairs -------------------------------------------------------------------------------
# (V, n_best, cost_comb, (box_hsize, box_vsize), fp32 texels, skewed intrinsics, shape): every V, n_best in {1, 2, 3, V}
# with both combinations, every window, both texel formats and both camera models appear; V = 1 runs in the 11 x 11 and
# 19 x 19 two-best variants and in the generic one (ratio exactly 0 in all of them).
COST_CONFIGS = [
    (1, 1, 1, (11, 11), False, False, "A"),
    (1, 3, 1, (5, 5), False, False, "B"),
    (1, 1, 0, (19, 19), True, True, "A"),
    (1, 2, 1, (11, 5), False, True, "B"),
    (1, 1, 1, (19, 19), False, True, "B"),
    (2, 1, 1, (19, 19), False, False, "A"),
    (2, 2, 1, (3, 3), True, False, "B"),
    (2, 2, 0, (12, 12), False, True, "A"),
    (2, 3, 1, (25, 25), False, False, "B"),
    (2, 1, 1, (217, 3), True, False, "A"),
    (21, 3, 1, (5, 19), False, False, "A"),
    (21, 21, 0, (11, 11), True, True, "B"),
    (21, 1, 1, (27, 27), False, False, "B"),
    (21, 2, 1, (11, 11), False, True, "A"),
    (21, 21, 1, (19, 19), False, False, "A"),
    (32, 32, 1, (19, 11), False, False, "A"),
    (32, 32, 0, (3, 217), False, False, "B"),
    (32, 1, 1, (11, 11), True, False, "B"),
    (32, 2, 0, (25, 25), False, True, "A"),
    (32, 3, 0, (12, 12), True, True, "B"),
]


def _cfg_id(c):
    V, nb, comb, box, fp32, skew, shape = c
    return f"V{V}-nb{nb}-comb{comb}-{box[0]}x{box[1]}-{'f32' if fp32 else 'u8'}-{'skew' if skew else 'pin'}-{shape}"


@pytest.mark.parametrize("cfg", COST_CONFIGS, ids=_cfg_id)
def test_eval_planes_matches_restatement(pkg, cfg):
    V, nb, comb, box, fp32, skew, shape = cfg
    scene = _scene(pkg, shape, fp32, skew)
    eng, ora = _pair(pkg, scene, V, _params(pkg, scene, box, nb, comb))
    try:
        xy, planes = _pairs(scene)
        out = [_compare_pairs(eng, ora, scene, V, box, xy, planes, wr, f"{_cfg_id(cfg)} pxf={int(wr)}") for wr in (True, False)]
    finally:
        eng.close(); ora.close()
    pc.record(f"restated_eval_{_cfg_id(cfg)}.json", out)
    for s in out:
        _assert_costs(s)


def test_eval_planes_one_view_ratio_is_zero(pkg):
    """DESIGN Q8: with one source view the second-best cost is +inf, so the ratio is 0 in every variant (the 11 x 11 and
    19 x 19 two-best kernels, and the generic kernel for any other window, n_best >= 3 or cost_comb = 0)."""
    scene = _scene(pkg, "A")
    xy, planes = _pairs(scene, n=1000, n_hostile=200)
    for box, nb, comb in (((11, 11), 1, 1), ((19, 19), 2, 1), ((7, 7), 1, 1), ((11, 11), 3, 1), ((11, 11), 1, 0), ((9, 5), 2, 1)):
        eng = pkg.DepthmapEngine(0)
        try:
            from tsar_mvs_b200.engine import cameras_to_struct
            eng.set_views(scene["images"], cameras_to_struct(scene["cams"]), [1], cam_f=scene["cam_f"])
            eng.set_params(_params(pkg, scene, box, nb, comb))
            for wr in (True, False):
                _, _, ratio = eng.eval_planes(xy, planes, wrapper_rounding=wr)
                assert (ratio == 0).all(), f"{box} n_best={nb} cost_comb={comb}: {int((ratio != 0).sum())} non-zero ratios"
        finally:
            eng.close()


def test_eval_planes_c5_last_columns(pkg):
    """C5 (6048 x 4032, 20 source views): pixels in the last columns and rows, where texture coordinates exceed 4096."""
    import torch
    s = pkg.scene.make_scene("C5", backend="torch", device="cuda:0")
    s["images"] = [t.cpu().numpy() for t in s["images"]]
    torch.cuda.empty_cache()
    W, H, V = s["W"], s["H"], 20
    rng = np.random.RandomState(5)
    xy = np.concatenate([np.stack([rng.randint(W - 48, W, 600), rng.randint(0, H, 600)], 1),
                         np.stack([rng.randint(4096, W, 400), rng.randint(H - 48, H, 400)], 1),
                         np.stack([rng.randint(W - 8, W, 200), rng.randint(H - 8, H, 200)], 1)]).astype(np.int32)
    planes = _planes_at(s, xy, rng)
    out = []
    for box, nb, comb in (((11, 11), 1, 1), ((19, 11), 3, 0)):
        eng, ora = _pair(pkg, s, V, _params(pkg, s, box, nb, comb))
        try:
            out += [_compare_pairs(eng, ora, s, V, box, xy, planes, wr, f"C5 {box} pxf={int(wr)}") for wr in (True, False)]
        finally:
            eng.close(); ora.close()
    pc.record("restated_eval_C5.json", out)
    for st in out:
        _assert_costs(st)


# ---- 2. initialisation ---------------------------------------------------------------------------------------
INIT_CONFIGS = [
    (32, 1, 1, (11, 11), "A"),
    (21, 1, 1, (27, 27), "B"),
    (5, 3, 0, (5, 19), "A"),
    (2, 2, 1, (12, 12), "B"),
    (3, 1, 1, (12, 7), "A"),
]


@pytest.mark.parametrize("cfg", INIT_CONFIGS, ids=lambda c: f"V{c[0]}-nb{c[1]}-comb{c[2]}-{c[3][0]}x{c[3][1]}-{c[4]}")
def test_init_planes_match_restatement(pkg, cfg):
    """gipuma_init_cu2: planes bit-identical on >= 99.9 % of the pixels (rsqrtf only decides a sign), costs within the
    bar of the pair test.  The init window is box / 2, not (box - 1) / 2: even boxes tell them apart."""
    V, nb, comb, box, shape = cfg
    scene = _scene(pkg, shape)
    L = pkg._lib
    eng, ora = _pair(pkg, scene, V, _params(pkg, scene, box, nb, comb))
    try:
        eng.init_planes(SEED)
        p_g, c_g = eng.download(L.F_NORM4), eng.download(L.F_COST)
        ora.init_planes(SEED)
        p_o, c_o = ora.planes(), ora.costs()
    finally:
        eng.close(); ora.close()
    same = pc.bits_equal(p_g, p_o).all(axis=-1)
    H, W = same.shape
    yy, xx = np.mgrid[0:H, 0:W]
    xy = np.stack([xx[same], yy[same]], 1).astype(np.int32)
    odd = (2 * (box[0] // 2) + 1, 2 * (box[1] // 2) + 1)     # its (box - 1) / 2 is the init window box / 2
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    ora_w = cb.CpuOracle(L.TsarCamera, L.TsarParams, scene["images"], cameras_to_struct(scene["cams"]),
                         list(range(1, V + 1)), _params(pkg, scene, odd, nb, comb), scene["cam_f"])
    try:
        _, ill, cond = _oracle_views(ora_w, scene, xy, p_g[same], box[0] // 2, box[1] // 2)
    finally:
        ora_w.close()
    d = np.abs(c_g[same].astype(np.float64) - c_o[same])
    st = dict(cfg=str(cfg), planes_bit_identical=float(same.mean()), ill=int(ill.sum()), well_over_tol=int((~ill & ~(d <= TOL)).sum()),
              max_d_well=float(d[~ill].max()), ill_over_loose=int((ill & ~(d <= LOOSE)).sum()),
              worst_well=sorted(zip(np.where(ill, -1.0, d).tolist(), cond.tolist()), reverse=True)[:5])
    pc.record(f"restated_init_V{V}_{box[0]}x{box[1]}.json", st)
    assert same.mean() >= 0.999, st
    assert st["well_over_tol"] == 0, st
    assert st["ill_over_loose"] <= 0.05 * max(1, st["ill"]), st


# ---- 3. single launches from one loaded state ------------------------------------------------------------------
def _offsets():
    """(dy, dx) of every neighbour a propagation step may take its plane from (gipuma.cu:888-1042, oc_spatial)."""
    o = []
    for i in range(11):
        k = 3 + 2 * i
        o += [(-k, 0), (k, 0), (0, -k), (0, k)]
    o += [(-1, 0), (1, 0), (0, -1), (0, 1)]
    for i in range(3):
        o += [(-(2 + i), -i), (-(2 + i), i), (2 + i, -i), (2 + i, i), (-i, -(2 + i)), (i, -(2 + i)), (-i, 2 + i), (i, 2 + i)]
    return sorted(set(o))


def _from_neighbour(pre, post):
    """True where post's plane is bitwise the pre-launch plane of some propagation neighbour (or the pixel's own)."""
    H, W = pre.shape[:2]
    pu, qu = pre.view(np.uint32), post.view(np.uint32)
    ok = (pu == qu).all(-1)
    for dy, dx in _offsets():
        ys, xs = slice(max(0, -dy), min(H, H - dy)), slice(max(0, -dx), min(W, W - dx))
        src = pu[max(0, dy):min(H, H + dy), max(0, dx):min(W, W + dx)]
        ok[ys, xs] |= (src == qu[ys, xs]).all(-1)
    return ok


def _state(pkg, eng):
    L = pkg._lib
    return dict(plane=eng.download(L.F_NORM4), cost=eng.download(L.F_COST), ratio=eng.download(L.F_RATIO),
                beview=eng.download(L.F_BEVIEW))


def _oracle_costs_of(ora, scene, box, V, xy, planes, ratio, beview, cost, what):
    views, ill, cond = _oracle_views(ora, scene, xy, planes, (box[0] - 1) // 2, (box[1] - 1) // 2)
    ref = ora.eval_planes(xy, planes)
    st = _check_costs((cost, beview, ratio), ref, views, ill, V, what, cond)
    return st, ref[0], ill


LAUNCH_CONFIGS = [
    (21, 3, 1, (11, 5), False, "A"),
    (32, 1, 1, (11, 11), False, "A"),
    (5, 2, 1, (19, 19), True, "B"),
    (1, 1, 0, (12, 12), False, "A"),
]


@pytest.mark.parametrize("cfg", LAUNCH_CONFIGS, ids=lambda c: f"V{c[0]}-nb{c[1]}-comb{c[2]}-{c[3][0]}x{c[3][1]}-{'skew' if c[4] else 'pin'}-{c[5]}")
def test_checkerboard_launches_match_restatement(pkg, cfg):
    """tsar_load_planes, then each of BLACK_SPATIAL, RED_SPATIAL, BLACK_REFINE, RED_REFINE and one fused iterate(1) from
    that same state, with the oracle's oc_spatial / oc_refine / oc_iterate on the same seeds.  Invariants:
      - pixels of the other colour and rows >= y_limit are bit-unchanged (plane, cost, ratio, best view);
      - a pixel whose cost did not change keeps its plane, ratio and best view bit for bit;
      - a changed pixel's cost, best view and ratio are the oracle's for the plane stored there (the pair bar);
      - propagation: the plane is bitwise a pre-launch plane of a propagation neighbour, and the oracle's cost of it is
        at most the oracle's own choice + 2 TOL; refinement: the same bound where the planes differ beyond PLANE_RTOL.
    Pixels that break the last bound are counted (near-ties, then different refinement paths)."""
    V, nb, comb, box, skew, shape = cfg
    scene = _scene(pkg, shape, skew=skew)
    L = pkg._lib
    H, W = scene["H"], scene["W"]
    yl = _y_limit(H)
    yy, xx = np.mgrid[0:H, 0:W]
    eng, ora = _pair(pkg, scene, V, _params(pkg, scene, box, nb, comb))
    records = []
    try:
        eng.init_planes(SEED)
        p0 = eng.download(L.F_NORM4)
        eng.load_planes(p0)                     # costs of the loaded planes: pm_cost_of_state_kernel
        c0 = eng.download(L.F_COST)
        allxy = np.stack([xx.ravel(), yy.ravel()], 1).astype(np.int32)
        st, _, _ = _oracle_costs_of(ora, scene, box, V, allxy, p0.reshape(-1, 4), np.zeros(H * W, np.float32),
                                    np.zeros(H * W, np.int32), c0.ravel(), "cost of loaded state")
        st["beview_diff"] = st["ratio_bad"] = st["ratio_v1_nonzero"] = 0   # only the cost is stored
        records.append(st)
        _assert_costs(st)
        r0, b0 = np.full((H, W), -1.5, np.float32), np.full((H, W), -7, np.int32)

        def run(kind):
            eng.load_planes(p0, c0)
            eng.upload(L.F_RATIO, r0); eng.upload(L.F_BEVIEW, b0)
            ora.set_state(p0, c0)
            if kind == "fused":
                eng.iterate(1, SEED + 100)
                ora.iterate(1, SEED + 100)
                return None
            colour = 0 if kind in (L.BLACK_SPATIAL, L.BLACK_REFINE) else 1
            eng.launch(kind, SEED + 10 + kind)
            if kind in (L.BLACK_SPATIAL, L.RED_SPATIAL):
                ora.spatial(colour)
            else:
                ora.refine(colour, SEED + 10 + kind)
            return colour

        names = {L.BLACK_SPATIAL: "black spatial", L.RED_SPATIAL: "red spatial", L.BLACK_REFINE: "black refine",
                 L.RED_REFINE: "red refine", "fused": "fused iteration"}
        for kind in (L.BLACK_SPATIAL, L.RED_SPATIAL, L.BLACK_REFINE, L.RED_REFINE, "fused"):
            colour = run(kind)
            g = _state(pkg, eng)
            p_o, c_o = ora.planes(), ora.costs()
            what = f"{cfg} {names[kind]}"
            mine = (yy < yl) & (((xx + yy) & 1) == colour) if colour is not None else (yy < yl)
            bits = lambda a, b: pc.bits_equal(a, b) if a.ndim == 2 else pc.bits_equal(a, b).all(-1)
            for f, a0 in (("plane", p0), ("cost", c0), ("ratio", r0), ("beview", b0)):
                assert bits(g[f], a0)[~mine].all(), f"{what}: {f} changed outside the launch's pixels"
            changed = mine & ~pc.bits_equal(g["cost"], c0)
            assert (g["cost"][changed] < c0[changed]).all(), f"{what}: a changed cost did not decrease"
            for f, a0 in (("plane", p0), ("ratio", r0), ("beview", b0)):
                assert bits(g[f], a0)[mine & ~changed].all(), f"{what}: {f} changed where the cost did not"
            # changed pixels: stored cost / best view / ratio are those of the stored plane
            cxy = np.stack([xx[changed], yy[changed]], 1).astype(np.int32)
            if len(cxy):
                st, _, _ = _oracle_costs_of(ora, scene, box, V, cxy, g["plane"][changed], g["ratio"][changed],
                                            g["beview"][changed], g["cost"][changed], what + " (changed pixels)")
                records.append(st)
                _assert_costs(st)
            # as good as the oracle's choice
            mxy = np.stack([xx[mine], yy[mine]], 1).astype(np.int32)
            ill = _oracle_views(ora, scene, mxy, g["plane"][mine], (box[0] - 1) // 2, (box[1] - 1) // 2)[1]
            ill |= _oracle_views(ora, scene, mxy, p_o[mine], (box[0] - 1) // 2, (box[1] - 1) // 2)[1]
            c_of_mine = ora.eval_planes(mxy, g["plane"][mine])[0].astype(np.float64)
            worse = c_of_mine > c_o[mine].astype(np.float64) + 2 * TOL
            differ = np.ones(len(mxy), bool)
            if kind in (L.BLACK_REFINE, L.RED_REFINE):
                differ = ~np.isclose(g["plane"][mine], p_o[mine], rtol=PLANE_RTOL, atol=PLANE_RTOL * 0.1).all(-1)
            if kind in (L.BLACK_SPATIAL, L.RED_SPATIAL):
                assert _from_neighbour(p0, g["plane"])[mine].all(), f"{what}: a plane that is no pre-launch neighbour's"
            rec = dict(what=what, pixels=int(mine.sum()), changed=int(changed.sum()),
                       planes_bit_equal_oracle=float(pc.bits_equal(g["plane"], p_o).all(-1)[mine].mean()),
                       differ=int(differ.sum()), worse_well=int((worse & differ & ~ill).sum()),
                       worse_ill=int((worse & differ & ill).sum()), ill=int(ill.sum()))
            records.append(rec)
            bound = WORSE_BOUND["fused" if kind == "fused" else ("spatial" if kind in (L.BLACK_SPATIAL, L.RED_SPATIAL) else "refine")]
            assert rec["worse_well"] <= bound * rec["pixels"], f"{what}: worse than the oracle's choice: {rec}"
    finally:
        eng.close(); ora.close()
        pc.record(f"restated_launch_V{V}_{box[0]}x{box[1]}.json", records)



# ---- 4. whole depth map at the new corners ------------------------------------------------------------------------
def test_depthmap_all_views_rectangular_window(pkg):
    """V = 32, n_best = 32, cost_comb = 0, an 11 x 7 window, 8 iterations on a 320 x 240 scene: close to the ground truth
    on textured pixels, and deterministic."""
    scene = pkg.scene.make_scene(dict(W=320, H=240, n_images=33, V=32, fx=800.0, radius=1.0, arc_deg=30.0))
    from tsar_mvs_b200.engine import cameras_to_struct
    L = pkg._lib
    outs = []
    for _ in range(2):
        eng = pkg.DepthmapEngine(0)
        try:
            eng.set_views(scene["images"], cameras_to_struct(scene["cams"]), scene["subset"], cam_f=scene["cam_f"])
            eng.set_params(_params(pkg, scene, (11, 7), 32, 0, iterations=8))
            eng.depthmap(SEED)
            outs.append((eng.download(L.F_NORM4), eng.download(L.F_COST)))
        finally:
            eng.close()
    agree = pc.gt_agreement(outs[0][0], scene)
    pc.record("restated_depthmap_V32.json", agree)
    assert outs[0][0].tobytes() == outs[1][0].tobytes() and outs[0][1].tobytes() == outs[1][1].tobytes(), "not deterministic"
    assert agree["frac_within_1pct_textured"] >= GT_FLOOR, agree



def test_quad_sampling_32_views(pkg):
    """Quad-cooperative sampling on and off give bit-identical state at V = 32 with the 11 x 11 window."""
    scene = pkg.scene.make_scene(dict(W=203, H=97, n_images=33, V=32, fx=600.0, radius=1.5, arc_deg=30.0), seed=32)
    _compare_run(pkg, scene)


# ---- 5. window limits ----------------------------------------------------------------------------------------------
# The weight table of a 128-thread CTA takes ns * 1028 bytes for ns window samples, within 220 KB: ns <= 219, where the
# init window (box / 2) is the larger one.  27 x 27 -> 14 x 14 = 196; 3 x 217 -> 2 x 109 = 218; 1 x 437 -> 1 x 219.
ACCEPTED = [(27, 27), (3, 217), (217, 3), (1, 437)]
REFUSED = [(28, 28), (29, 29), (3, 218), (218, 3), (1, 438)]


@pytest.mark.parametrize("box", ACCEPTED, ids=lambda b: f"{b[0]}x{b[1]}")
def test_largest_windows_launch_and_match(pkg, box):
    scene = _scene(pkg, "A")
    V = 4
    eng, ora = _pair(pkg, scene, V, _params(pkg, scene, box, 1, 1))
    L = pkg._lib
    try:
        xy, planes = _pairs(scene, n=800, n_hostile=100)
        out = [_compare_pairs(eng, ora, scene, V, box, xy, planes, wr, f"{box} pxf={int(wr)}") for wr in (True, False)]
        eng.init_planes(SEED)
        for kind in (L.BLACK_SPATIAL, L.RED_SPATIAL, L.BLACK_REFINE, L.RED_REFINE):
            eng.launch(kind, SEED + kind)
        eng.iterate(1, SEED)
        eng.sync()
        assert np.isfinite(eng.download(L.F_COST)).all()
    finally:
        eng.close(); ora.close()
    pc.record(f"restated_window_{box[0]}x{box[1]}.json", out)
    for s in out:
        _assert_costs(s)


@pytest.mark.parametrize("box", REFUSED, ids=lambda b: f"{b[0]}x{b[1]}")
def test_window_one_size_up_is_refused(pkg, box):
    scene = _scene(pkg, "A")
    from tsar_mvs_b200.engine import cameras_to_struct
    eng = pkg.DepthmapEngine(0)
    try:
        eng.set_views(scene["images"], cameras_to_struct(scene["cams"]), [1, 2], cam_f=scene["cam_f"])
        rc = eng.lib.tsar_set_params(eng.h, C.byref(_params(pkg, scene, box, 1, 1)))
        assert rc == TSAR_ERR_ARG, rc
        assert b"window too large" in eng.lib.tsar_last_error(eng.h)
    finally:
        eng.close()
