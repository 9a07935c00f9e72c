"""Quad-cooperative sampling (pm_core.cuh, view_cost_quad; DESIGN.md 4.2) against the per-lane sampling loop.

The quad path only changes which lane fetches a source sample, so the PatchMatch state must be bit-identical with the
switch on and off: planes, costs, ratio and best view after the initialisation, after every single launch (fused,
propagation-only and refinement-only kernels) and after a full 8-iteration sequence.  Scenes: the small test scene,
sizes whose width is not a multiple of 4 or 32 and whose checkerboard grid stops short of the last row (helper lanes
outside the image or past y_limit), hostile planes that put lanes of the exact-division path and of the fast path into
one quad, and a C2-size scene.
"""
import numpy as np
import pytest

from tests import parity_common as pc

pytestmark = pytest.mark.gpu
SEED = 4242
ALL = 1 << 30


def _engine(pkg, scene, quad):
    from tsar_mvs_b200.engine import cameras_to_struct
    params = pkg.make_params(box=11, iterations=8, n_best=1, cost_comb=1, min_disparity=scene["min_disparity"],
                             max_disparity=scene["max_disparity"])
    eng = pkg.DepthmapEngine(0)
    if isinstance(scene["images"][0], np.ndarray):
        eng.set_views(scene["images"], cameras_to_struct(scene["cams"]), scene["subset"], cam_f=scene["cam_f"])
    else:   # torch tensors on the device
        eng.set_views_device([t.data_ptr() for t in scene["images"]], scene["W"], scene["H"], cameras_to_struct(scene["cams"]),
                             scene["subset"], cam_f=scene["cam_f"])
    eng.set_params(params)
    eng.quad_sampling(ALL if quad else -1)
    return eng


def _state(pkg, eng):
    L = pkg._lib
    return [eng.download(f) for f in (L.F_NORM4, L.F_COST, L.F_RATIO, L.F_BEVIEW)]


def _assert_same(pkg, a, b, what):
    for name, x, y in zip(("planes", "costs", "ratio", "best view"), _state(pkg, a), _state(pkg, b)):
        assert x.tobytes() == y.tobytes(), f"{what}: {name} differ at {int((x.view(np.uint8) != y.view(np.uint8)).sum())} bytes"


def _hostile_planes(scene, seed):
    """Planes of tools/gpu_cost_sweep.py's hostile mix on every pixel (grazing, zero, huge and tiny normals, offsets
    0 / +-1e-30 / +-1e30 / inf / NaN), interleaved with well-behaved planes so that quads mix both."""
    rng = np.random.RandomState(seed)
    H, W = scene["H"], scene["W"]
    n = W * H
    xy, good = pc.random_planes(scene, n, seed=seed, border=False)
    nrm = rng.normal(size=(n, 3)).astype(np.float32)
    mode = rng.randint(0, 8, n)
    unit = mode < 5
    nrm[unit] /= np.linalg.norm(nrm[unit], axis=1, keepdims=True)
    nrm[mode == 5, 2] = rng.uniform(-1e-4, 1e-4, int((mode == 5).sum()))
    nrm[mode == 6] = 0.0
    nrm[mode == 7] *= rng.choice(np.array([1e-20, 1e20, 3.0], np.float32), int((mode == 7).sum()))[:, None]
    d = rng.uniform(-3, 3, n).astype(np.float32)
    special = rng.rand(n) < 0.25
    d[special] = rng.choice(np.array([0.0, -0.0, 1e-30, -1e-30, 1e-10, 1e30, -1e30, np.inf, -np.inf, np.nan], np.float32),
                            int(special.sum()))
    hostile = np.concatenate([nrm, d[:, None]], 1).astype(np.float32)
    # the planes of random_planes belong to random pixels; for "well-behaved at this pixel" re-derive d at each pixel
    cam = scene["cams"][0]
    yy, xx = np.divmod(np.arange(n), W)
    depth = rng.uniform(cam["depthMin"], cam["depthMax"], n)
    X = (np.asarray(cam["K_inv"], float) @ np.stack([xx, yy, np.ones(n)]).astype(float)).T * depth[:, None]
    good[:, 3] = -np.sum(good[:, :3].astype(float) * X, axis=1)
    pick = rng.rand(n) < 0.5
    return np.where(pick[:, None], hostile, good).reshape(H, W, 4).astype(np.float32)


def _compare_run(pkg, scene, load=None):
    L = pkg._lib
    on, off = _engine(pkg, scene, True), _engine(pkg, scene, False)
    try:
        for e in (on, off):
            if load is None:
                e.init_planes(SEED)
            else:
                e.load_planes(load)
        _assert_same(pkg, on, off, "initial state")
        # single propagation-only and refinement-only launches (tsar_launch), both colours
        for k, kind in enumerate((L.BLACK_SPATIAL, L.BLACK_REFINE, L.RED_SPATIAL, L.RED_REFINE)):
            for e in (on, off):
                e.launch(kind, SEED + 10 + k)
            _assert_same(pkg, on, off, f"launch kind {kind}")
        # fused launches, one iteration (two launches) at a time
        for it in range(3):
            for e in (on, off):
                e.iterate(1, SEED + 100 * it)
            _assert_same(pkg, on, off, f"fused iteration {it}")
        # a full 8-iteration sequence from a fresh start
        for e in (on, off):
            if load is None:
                e.init_planes(SEED + 1)
            else:
                e.load_planes(load)
            e.iterate(8, SEED + 7)
        _assert_same(pkg, on, off, "8 iterations")
    finally:
        on.close(); off.close()


def test_quad_sampling_small_scene(pkg):
    _compare_run(pkg, pkg.scene.make_scene("small"))


@pytest.mark.parametrize("W,H", [(203, 97), (61, 33), (130, 161)])
def test_quad_sampling_helper_lanes(pkg, W, H):
    """Widths not a multiple of 4 or 32; H = 32 m + 1 leaves the last row beyond the checkerboard grid (y_limit < H)."""
    scene = pkg.scene.make_scene(dict(W=W, H=H, n_images=6, V=5, fx=300.0, radius=1.5, arc_deg=20.0), seed=W * H)
    y_limit = min(H, 32 * ((H // 2 + 15) // 16))
    assert W % 4 and y_limit < H
    _compare_run(pkg, scene)


def test_quad_sampling_hostile_planes(pkg):
    """Exact-division lanes next to fast lanes in one quad: the quad fetches for its fast lanes, the others divide."""
    scene = pkg.scene.make_scene(dict(W=190, H=129, n_images=5, V=4, fx=250.0, radius=2.0, arc_deg=25.0), seed=77)
    _compare_run(pkg, scene, load=_hostile_planes(scene, 5))


def test_quad_sampling_c2_size(pkg):
    """The benchmark's shape: 3100 x 2050, 10 source views, init + 8 iterations."""
    scene = pkg.scene.make_scene("C2", backend="torch", device="cuda:0")
    on, off = _engine(pkg, scene, True), _engine(pkg, scene, False)
    try:
        for e in (on, off):
            e.init_planes(SEED)
        _assert_same(pkg, on, off, "C2 init")
        for it in range(8):
            for e in (on, off):
                e.iterate(1, SEED + it)
            _assert_same(pkg, on, off, f"C2 iteration {it}")
    finally:
        on.close(); off.close()
