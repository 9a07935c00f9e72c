"""GPU parity tests (pytest -m gpu, on a B200).  Every product call goes through the C ABI
(libtsar_b200.so); the checker is the reference's own gipuma.cu rebuilt for sm_100 (oracle/_ref), or, where that
build is absent, its results recorded as digests (oracle/recorded.py, tests/golden/reference_digests.json):
  * 'asis'     -- exactly as written (same-colour reads race, SURVEY Q3: not run-to-run reproducible);
  * 'snapshot' -- 2-line build-time patch giving deterministic pre-launch-snapshot semantics.
Bar: bit-exact against the snapshot build (integer/float bits identical); against the racy as-is build
we report agreement next to the build's own run-to-run noise floor and require ours to be no further
from it than the snapshot build is.
"""
import os

import numpy as np
import pytest

from tests import parity_common as pc

pytestmark = pytest.mark.gpu
SEED = 20240601


@pytest.fixture(scope="module")
def env():
    return pc.load_pkg(), pc.ref_binding()


@pytest.fixture(scope="module")
def small(env):
    pkg, _ = env
    return pkg.scene.make_scene("small")


@pytest.mark.parametrize("box,n_best,cost_comb", [(11, 1, 1), (11, 2, 1), (19, 1, 1), (7, 3, 1), (9, 2, 0)])
def test_pmcost_multiview_bit_exact(env, small, box, n_best, cost_comb):
    """pmCostMultiview_cu (gipuma.cu:456-518) on 50k random (pixel, plane) pairs incl. image borders."""
    pkg, rb = env
    params, mine, refs = pc.make_engines(pkg, small, box=box, n_best=n_best, cost_comb=cost_comb, variants=("asis",))
    xy, planes = pc.random_planes(small, 50000)
    c_m, b_m, r_m = mine.eval_planes(xy, planes, wrapper_rounding=True)
    c_r, b_r, r_r = refs["asis"].eval_planes(xy, planes)
    mine.close(); refs["asis"].close()
    assert pc.frac_bit_exact(c_m, c_r) == 1.0
    assert (b_m == b_r).all()
    assert pc.frac_bit_exact(r_m, r_r) == 1.0


def test_init_same_seed_bit_exact(env, small):
    """gipuma_init_cu2 (gipuma.cu:679-729): same XORWOW streams, planes and costs from the reference's seed."""
    pkg, rb = env
    params, mine, refs = pc.make_engines(pkg, small, variants=("asis",))
    mine.init_planes(SEED); refs["asis"].init_planes(SEED)
    n_m, c_m = mine.download(pkg._lib.F_NORM4), mine.download(pkg._lib.F_COST)
    n_r, c_r = refs["asis"].download(rb.F_NORM4), refs["asis"].download(rb.F_COST)
    mine.close(); refs["asis"].close()
    assert pc.frac_bit_exact(n_m, n_r) == 1.0
    assert pc.frac_bit_exact(c_m, c_r) == 1.0
    assert len(np.unique(n_m[..., 0])) > 1000  # really random


def test_single_half_steps_bit_exact(env, small):
    """Each checkerboard half-step from the reference's initial planes (tsar_load_planes)."""
    pkg, rb = env
    L = pkg._lib
    params, mine, refs = pc.make_engines(pkg, small, variants=("asis", "snapshot"))
    asis, snap = refs["asis"], refs["snapshot"]
    asis.init_planes(SEED)
    n0, c0 = asis.download(rb.F_NORM4), asis.download(rb.F_COST)
    for kind in (L.BLACK_REFINE, L.RED_REFINE):  # refinement touches only the pixel itself: no race in the reference
        asis.upload(rb.F_NORM4, n0); asis.upload(rb.F_COST, c0); asis.launch(kind, SEED + 1)
        mine.load_planes(n0, c0); mine.launch(kind, SEED + 1)
        assert pc.frac_bit_exact(mine.download(L.F_NORM4), asis.download(rb.F_NORM4)) == 1.0
        assert pc.frac_bit_exact(mine.download(L.F_COST), asis.download(rb.F_COST)) == 1.0
        assert (mine.download(L.F_BEVIEW) == asis.download(rb.F_BEVIEW)).all()
        assert pc.frac_bit_exact(mine.download(L.F_RATIO), asis.download(rb.F_RATIO)) == 1.0
    for kind in (L.BLACK_SPATIAL, L.RED_SPATIAL):
        snap.upload(rb.F_NORM4, n0); snap.upload(rb.F_COST, c0); snap.launch(kind)
        mine.load_planes(n0, c0); mine.launch(kind)
        assert pc.frac_bit_exact(mine.download(L.F_NORM4), snap.download(rb.F_NORM4)) == 1.0
        assert pc.frac_bit_exact(mine.download(L.F_COST), snap.download(rb.F_COST)) == 1.0
        changed = 1.0 - pc.frac_bit_exact(mine.download(L.F_COST), c0)
        assert changed > 0.2  # the step really propagated planes
    for e in (mine, asis, snap):
        e.close()


@pytest.mark.parametrize("cfg,iters", [("small", 8), ("tiny", 3)])
def test_full_sequence_vs_reference(env, cfg, iters):
    """init -> iters x (bSP,bPR,rSP,rPR) -> getlrdiff -> getview -> compute_disp (gipuma.cu:1741-1761)."""
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene(cfg)
    params, mine, refs = pc.make_engines(pkg, scene, iterations=iters, variants=("asis", "snapshot"))
    asis, snap = refs["asis"], refs["snapshot"]
    mine.depthmap(SEED)
    o_m, conf_m = mine.download(L.F_NORM4), mine.download(L.F_CONFID)
    snap.depthmap(SEED, iters=iters)
    o_s, conf_s = snap.download(rb.F_NORM4), snap.download(rb.F_CONFID)
    asis.depthmap(SEED, iters=iters); o_a = asis.download(rb.F_NORM4)
    asis.depthmap(SEED, iters=iters); o_a2 = asis.download(rb.F_NORM4)
    for e in (mine, asis, snap):
        e.close()
    # deterministic reference build: identical bits, so trivially inside the north-star tolerance
    a = pc.output_agreement(o_m, o_s)
    assert a["bit_exact"] == 1.0, a
    assert a["frac_ok"] >= pc.GATE_FRACTION
    assert pc.frac_bit_exact(conf_m, conf_s) == 1.0
    # racy as-written build: we must be as close to it as its race-free twin is (its own noise floor is
    # reported for the record and is below the 99 % gate on these scenes -- see DESIGN.md)
    ours, twin, floor = pc.output_agreement(o_m, o_a), pc.output_agreement(o_s, o_a), pc.output_agreement(o_a2, o_a)
    print(f"\n[{cfg}] ours-vs-asis {ours['frac_ok']:.4f} (depth {ours['frac_depth_ok']:.4f}), "
          f"snapshot-vs-asis {twin['frac_ok']:.4f}, asis-vs-asis {floor['frac_ok']:.4f} (depth {floor['frac_depth_ok']:.4f})")
    assert ours["frac_ok"] == twin["frac_ok"] and ours["frac_depth_ok"] == twin["frac_depth_ok"]


@pytest.mark.parametrize("box,n_best,cost_comb", [(19, 1, 1), (7, 3, 1), (9, 2, 0), (11, 2, 1), (5, 1, 1), (25, 1, 1), (12, 1, 1), (11, 3, 0)])
def test_full_sequence_other_windows_and_view_combinations(env, box, n_best, cost_comb):
    """The 19x19 kernel variant, the runtime-window variant (any other blocksize) and the n_best > 1 / cost_comb
    paths of the propagation + refinement kernel, through the whole per-view sequence."""
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene("tiny")
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, box=box, n_best=n_best, cost_comb=cost_comb, variants=("snapshot",))
    snap = refs["snapshot"]
    mine.depthmap(SEED); snap.depthmap(SEED, iters=2)
    o_m, o_s = mine.download(L.F_NORM4), snap.download(rb.F_NORM4)
    c_m, c_s = mine.download(L.F_COST), snap.download(rb.F_COST)
    v_m, v_s = mine.download(L.F_BEVIEW), snap.download(rb.F_BEVIEW)
    mine.close(); snap.close()
    assert pc.frac_bit_exact(o_m, o_s) == 1.0
    assert pc.frac_bit_exact(c_m, c_s) == 1.0
    assert (v_m == v_s).all()


@pytest.mark.parametrize("box", [11, 19])
def test_fused_equals_unfused(env, small, monkeypatch, box):
    """Fusing spatial propagation + refinement of one colour into one kernel changes nothing.  Runs every instantiation of the
    checkerboard kernel of a window variant in ONE process (fused, propagation-only, refinement-only; 8-bit and fp32 source
    textures; pinhole and general intrinsics): with the 19x19 window each of them needs its own opt-in to more than 48 KB
    of shared memory."""
    pkg, rb = env
    outs, counts = [], []
    for envs in ((), (("TSAR_B200_UNFUSED", "1"),), (("TSAR_B200_NO_U8", "1"),), (("TSAR_B200_NO_U8", "1"), ("TSAR_B200_UNFUSED", "1")),
                 (("TSAR_B200_NO_PINHOLE_FASTPATH", "1"),), (("TSAR_B200_NO_PINHOLE_FASTPATH", "1"), ("TSAR_B200_UNFUSED", "1"))):
        for k, v in envs:
            monkeypatch.setenv(k, v)
        params, eng, _ = pc.make_engines(pkg, small, box=box, iterations=3 if box == 11 else 1, variants=())
        eng.depthmap(SEED)
        outs.append(eng.download(pkg._lib.F_NORM4))
        counts.append(eng.launch_count())
        eng.close()
        for k, _ in envs:
            monkeypatch.delenv(k)
    for o in outs[1:]:
        assert pc.frac_bit_exact(outs[0], o) == 1.0
    assert counts[1] > counts[0] > 0


def test_general_intrinsics_instantiation_matches(env, small, monkeypatch):
    """The homography instantiation for arbitrary intrinsic matrices (selected automatically when some K has skew or
    a non-unit last row; forced here) and the zero-skew pinhole one give the same bits, and both equal the reference."""
    pkg, rb = env
    L = pkg._lib
    params, fast, refs = pc.make_engines(pkg, small, iterations=2, variants=("snapshot",))
    fast.depthmap(SEED)
    o_f = fast.download(L.F_NORM4)
    monkeypatch.setenv("TSAR_B200_NO_PINHOLE_FASTPATH", "1")
    params, general, _ = pc.make_engines(pkg, small, iterations=2, variants=())
    general.depthmap(SEED)
    o_g = general.download(L.F_NORM4)
    monkeypatch.delenv("TSAR_B200_NO_PINHOLE_FASTPATH")
    refs["snapshot"].depthmap(SEED, iters=2)
    o_r = refs["snapshot"].download(rb.F_NORM4)
    for e in (fast, general, refs["snapshot"]):
        e.close()
    assert pc.frac_bit_exact(o_f, o_g) == 1.0
    assert pc.frac_bit_exact(o_g, o_r) == 1.0


def test_run_is_deterministic(env, small):
    pkg, rb = env
    params, mine, _ = pc.make_engines(pkg, small, iterations=2, variants=())
    mine.depthmap(SEED); a = mine.download(pkg._lib.F_NORM4)
    mine.depthmap(SEED); b = mine.download(pkg._lib.F_NORM4)
    mine.depthmap(SEED + 5); c = mine.download(pkg._lib.F_NORM4)
    mine.close()
    assert pc.frac_bit_exact(a, b) == 1.0
    assert pc.frac_bit_exact(a, c) < 0.9  # a different seed gives different planes


def test_glue_and_depth_completion_bit_exact(env, small):
    """getlrdiff/getview/get_disp/update_scale(_2)/compute_disp (gipuma.cu:732-755, 810-844, 1161-1292)."""
    pkg, rb = env
    L = pkg._lib
    scene = small
    params, mine, refs = pc.make_engines(pkg, scene, variants=("snapshot",))
    ref = refs["snapshot"]
    ref.init_planes(SEED); ref.iterate(2, SEED)
    n0, c0 = ref.download(rb.F_NORM4), ref.download(rb.F_COST)
    mine.load_planes(n0, c0)
    mine.upload(L.F_BEVIEW, ref.download(rb.F_BEVIEW)); mine.upload(L.F_RATIO, ref.download(rb.F_RATIO))
    ref.lrdiff(); mine.lrdiff()
    assert pc.frac_bit_exact(mine.download(L.F_LRDIFF), ref.download(rb.F_LRDIFF)) == 1.0
    ref.getview(); mine.getview()
    assert pc.frac_bit_exact(mine.download(L.F_CONFID), ref.download(rb.F_CONFID)) == 1.0
    assert pc.frac_bit_exact(mine.download(L.F_DEPTH), ref.download(rb.F_DEPTH)) == 1.0
    for e in (mine, ref):
        e.set_regions(scene["region_text"], scene["region_norm4"])
    mine.upload(L.F_CANNY, scene["canny"]); ref.upload(rb.F_CANNY, scene["canny"])
    ref.update_scale_2(); mine.update_scale_2()
    assert pc.frac_bit_exact(mine.download(L.F_FAKEDEPTH), ref.download(rb.F_FAKEDEPTH)) == 1.0
    ref.update_scale(); mine.update_scale()
    for fm, fr in ((L.F_NORM4, rb.F_NORM4), (L.F_COST, rb.F_COST), (L.F_SCALE, rb.F_SCALE), (L.F_DEPTH, rb.F_DEPTH)):
        assert pc.frac_bit_exact(mine.download(fm), ref.download(fr)) == 1.0
    filled = mine.download(L.F_SCALE)
    assert 0.05 < filled.mean() < 0.5  # the textureless facet was completed
    ref.compute_disp(); mine.compute_disp()
    out = mine.download(L.F_NORM4)
    assert pc.frac_bit_exact(out, ref.download(rb.F_NORM4)) == 1.0
    # depth completion really put the region plane there: GT agreement inside the textureless facet
    flat = scene["labels"] == 4
    rel = np.abs(out[..., 3] - scene["gt_depth"]) / scene["gt_depth"]
    assert np.median(rel[flat]) < 0.05
    wn = out.copy()
    dsp = np.where(wn[..., 3] > 0, scene["cam_f"] / np.maximum(wn[..., 3], 1e-6), 1.0).astype(np.float32)
    for e, f_n, f_d in ((mine, L.F_NORM4, L.F_DEPTH), (ref, rb.F_NORM4, rb.F_DEPTH)):
        e.upload(f_n, wn); e.upload(f_d, dsp)
    ref.get_disp(); mine.get_disp()
    assert pc.frac_bit_exact(mine.download(L.F_NORM4), ref.download(rb.F_NORM4)) == 1.0
    mine.close(); ref.close()


def test_reliable_flags_and_output_payloads(env, small):
    """lines->scale from APD's weak.png (main.cpp:1499-1514: white, green and red pixels are reliable) and from the
    confidence map; tsar_download_outputs hands out exactly the payloads of TSAR_disp.dmb / TSAR_normals.dmb."""
    pkg, rb = env
    L = pkg._lib
    params, mine, _ = pc.make_engines(pkg, small, iterations=2, variants=())
    H, W = small["H"], small["W"]
    rng = np.random.RandomState(3)
    bgr = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
    kinds = np.array([[255, 255, 255], [0, 255, 0], [0, 0, 255], [255, 0, 0], [0, 255, 255], [254, 255, 255], [0, 0, 0]], np.uint8)
    pick = rng.randint(0, len(kinds) + 3, (H, W))
    for k, col in enumerate(kinds):
        bgr[pick == k] = col
    want = ((bgr == [255, 255, 255]).all(-1) | (bgr == [0, 255, 0]).all(-1) | (bgr == [0, 0, 255]).all(-1)).astype(np.float32)
    assert 0.2 < want.mean() < 0.5
    mine.scale_from_weak_png(bgr)
    assert np.array_equal(mine.download(L.F_SCALE), want)
    mine.depthmap(SEED)
    out4, confid = mine.download(L.F_NORM4), mine.download(L.F_CONFID)
    mine.scale_from_confidence(0.8)
    assert np.array_equal(mine.download(L.F_SCALE), (confid > 0.8).astype(np.float32))
    depth, normals, cf = mine.download_outputs()
    assert pc.frac_bit_exact(depth, out4[..., 3]) == 1.0 and pc.frac_bit_exact(normals, np.ascontiguousarray(out4[..., :3])) == 1.0
    assert pc.frac_bit_exact(cf, confid) == 1.0
    mine.close()


def test_edge_cases(env):
    """Odd sizes (last row outside the reference's checkerboard grid), V = 1 and V = 2, tiny images."""
    pkg, rb = env
    L = pkg._lib
    for W, H in ((67, 33), (261, 9), (9, 261), (33, 34), (64, 32)):   # odd, very wide, very tall, tile-aligned
        cfg = dict(W=W, H=H, n_images=3, V=2, fx=150.0, radius=1.0, arc_deg=14.0)
        scene = pkg.scene.make_scene(cfg)
        params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot",))
        ref = refs["snapshot"]
        mine.depthmap(SEED); ref.depthmap(SEED, iters=2)
        assert pc.frac_bit_exact(mine.download(L.F_NORM4), ref.download(rb.F_NORM4)) == 1.0, (W, H)
        assert pc.frac_bit_exact(mine.download(L.F_COST), ref.download(rb.F_COST)) == 1.0, (W, H)
        mine.close(); ref.close()


def test_non_8bit_images_use_fp32_textures(env):
    """Images that are not 8-bit valued (e.g. rescaled inputs) cannot use the 8-bit texture copies; the library
    detects that on upload and samples the fp32 arrays like the reference: still bit-exact."""
    pkg, rb = env
    L = pkg._lib
    scene = dict(pkg.scene.make_scene("tiny"))
    scene["images"] = [(im * np.float32(0.731) + np.float32(0.2)).astype(np.float32) for im in scene["images"]]
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot",))
    ref = refs["snapshot"]
    mine.depthmap(SEED); ref.depthmap(SEED, iters=2)
    assert pc.frac_bit_exact(mine.download(L.F_NORM4), ref.download(rb.F_NORM4)) == 1.0
    assert pc.frac_bit_exact(mine.download(L.F_CONFID), ref.download(rb.F_CONFID)) == 1.0
    mine.close(); ref.close()


def test_randomized_configurations_bit_exact(env):
    """Differential sweep against the race-free reference build: random image sizes (odd ones included), view
    counts, windows, view combinations and depth ranges; the whole per-view sequence must agree bit for bit."""
    pkg, rb = env
    L = pkg._lib
    rng = np.random.RandomState(20240601)
    for trial in range(8):
        W, H = int(rng.randint(40, 200)), int(rng.randint(34, 140))
        V = int(rng.randint(1, 6))
        box = int(rng.choice([5, 7, 9, 11, 11, 13, 15, 19]))
        n_best = int(rng.randint(1, min(V, 3) + 1))
        cost_comb = int(rng.choice([0, 1]))
        cfg = dict(W=W, H=H, n_images=V + 1, V=V, fx=float(rng.uniform(120, 400)), radius=float(rng.uniform(0.8, 3.0)),
                   arc_deg=float(rng.uniform(8, 24)))
        scene = pkg.scene.make_scene(cfg, seed=int(rng.randint(1, 1000)))
        iters = int(rng.randint(1, 3))
        params, mine, refs = pc.make_engines(pkg, scene, iterations=iters, box=box, n_best=n_best, cost_comb=cost_comb, variants=("snapshot",))
        ref = refs["snapshot"]
        seed = int(rng.randint(1, 2 ** 31))
        mine.depthmap(seed); ref.depthmap(seed, iters=iters)
        tag = dict(trial=trial, W=W, H=H, V=V, box=box, n_best=n_best, cost_comb=cost_comb, iters=iters)
        assert pc.frac_bit_exact(mine.download(L.F_NORM4), ref.download(rb.F_NORM4)) == 1.0, tag
        assert pc.frac_bit_exact(mine.download(L.F_CONFID), ref.download(rb.F_CONFID)) == 1.0, tag
        assert (mine.download(L.F_BEVIEW) == ref.download(rb.F_BEVIEW)).all(), tag
        mine.close(); ref.close()


def test_color_processing_is_the_grey_path_on_channel_x(env):
    """`-color_processing`: the reference uploads BGRA float4 textures and instantiates its kernels for float4, but they
    still sample with tex2D<float> (gipuma.cu:247,262,265), i.e. the first component.  The reference build run that way
    (channel x = the image, other channels different data) must equal our path fed with channel x."""
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene("tiny")
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot",), color_processing=1)
    ref = refs["snapshot"]
    mine.depthmap(SEED); ref.depthmap(SEED, iters=2)
    assert pc.frac_bit_exact(mine.download(L.F_NORM4), ref.download(rb.F_NORM4)) == 1.0
    assert pc.frac_bit_exact(mine.download(L.F_CONFID), ref.download(rb.F_CONFID)) == 1.0
    # and it is the same result as the grey build on that image
    params, grey, _ = pc.make_engines(pkg, scene, iterations=2, variants=())
    grey.depthmap(SEED)
    assert pc.frac_bit_exact(mine.download(L.F_NORM4), grey.download(L.F_NORM4)) == 1.0
    for e in (mine, ref, grey):
        e.close()


def test_context_reuse_across_sizes_and_view_counts(env):
    """One context processes views of different sizes / view counts / windows one after the other (what a multi-view
    driver does); every result equals a fresh context's."""
    pkg, rb = env
    L = pkg._lib
    from tsar_mvs_b200.engine import cameras_to_struct
    cases = [("tiny", 11, 2), (dict(W=150, H=90, n_images=6, V=5, fx=260.0, radius=1.5, arc_deg=18.0), 19, 1),
             (dict(W=67, H=33, n_images=3, V=2, fx=150.0, radius=1.0, arc_deg=14.0), 7, 2), ("tiny", 11, 2)]
    shared = pkg.DepthmapEngine(0)
    for cfg, box, iters in cases:
        scene = pkg.scene.make_scene(cfg)
        params = pkg.make_params(box=box, iterations=iters, min_disparity=scene["min_disparity"], max_disparity=scene["max_disparity"])
        outs = []
        for eng in (shared, pkg.DepthmapEngine(0)):
            eng.set_views(scene["images"], cameras_to_struct(scene["cams"]), scene["subset"], cam_f=scene["cam_f"])
            eng.set_params(params)
            eng.depthmap(SEED)
            outs.append((eng.download(L.F_NORM4), eng.download(L.F_CONFID)))
            if eng is not shared:
                eng.close()
        assert pc.frac_bit_exact(outs[0][0], outs[1][0]) == 1.0 and pc.frac_bit_exact(outs[0][1], outs[1][1]) == 1.0, cfg
    shared.close()


def test_host_entry_matches_resident_path(env, small):
    """tsar_depthmap_host (host buffers in/out, the e2e path) == set_views + depthmap + download."""
    pkg, rb = env
    L = pkg._lib
    params, mine, _ = pc.make_engines(pkg, small, iterations=2, variants=())
    mine.depthmap(SEED)
    a, ca = mine.download(L.F_NORM4), mine.download(L.F_CONFID)
    e2 = pkg.DepthmapEngine(0)
    b, cb = e2.depthmap_host(small["images"], small["cams"], small["subset"], params, SEED, cam_f=small["cam_f"])
    mine.close(); e2.close()
    assert pc.frac_bit_exact(a, b) == 1.0 and pc.frac_bit_exact(ca, cb) == 1.0


def test_errors_are_codes_not_exits(env, small):
    pkg, rb = env
    e = pkg.DepthmapEngine(0)
    with pytest.raises(pkg.TsarError):
        e.init_planes(1)  # no views yet
    with pytest.raises(pkg.TsarError):
        e.set_views(small["images"], small["cams"], list(range(40)))  # V > 32 (SURVEY Q8)
    e.close()


def test_smoke_entry(env):
    import __graft_entry__ as g
    g.smoke()


@pytest.mark.parametrize("cfg,size,enforce", [("small", 20, False), ("small", 12, True), ("C1", 20, False)])
def test_slic_labels_bit_exact(env, cfg, size, enforce):
    """gSLICr (7 kernels, GPU.cu:213-379; settings of main.cpp:608-615): labels identical to the reference build,
    including its as-compiled partial warp-tail reduction (SURVEY Q10) and window tiling (Q11)."""
    pkg, rb = env
    scene = pkg.scene.make_scene(cfg, with_colour=True)
    bgrx = pkg.scene.box_downsample4(scene["bgr"]) if cfg == "C1" else np.concatenate(
        [scene["bgr"], np.zeros(scene["bgr"].shape[:2] + (1,), np.uint8)], axis=-1)
    eng = pkg.DepthmapEngine(0)
    mine = eng.slic(bgrx, spixel_size=size, no_iters=5, coh_weight=5.0, enforce_connectivity=enforce)
    ref, _ = rb.ref_slic(bgrx, spixel_size=size, no_iters=5, coh_weight=5.0, enforce_connectivity=enforce)
    full = eng.slic(bgrx, spixel_size=size, correct_reduction=True)
    eng.close()
    assert mine.shape == ref.shape
    assert (mine == ref).all(), f"{(mine != ref).mean():.4%} of labels differ"
    assert len(np.unique(mine)) > 4
    assert (full >= 0).all() and full.max() < (bgrx.shape[0] // size) * (bgrx.shape[1] // size)


def test_slic_stages_bit_exact_and_exact_ties(env):
    """Beyond the final labels (tools/gpu_slic_stages.py): rgb2CIELab over its whole input domain -- every 24-bit colour
    once -- and the superpixel records (centre, colour, count) after every iteration, bit for bit against the reference
    engine, on a piecewise-constant image: there the distances of a pixel to two centres tie exactly and the last ulp of
    the compiled contraction decides the label (found in round 2: 0.1 % of the labels of one such image differed)."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tools", "gpu_slic_stages.py")], capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0 and "ALL EXACT" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


def test_gslicr_core_engine_drop_in(env, tmp_path):
    """gSLICr::engines::core_engine exported by libtsar_b200.so under the reference's mangled names, driven by a harness
    compiled against the REFERENCE's own gSLICr / ORUtils headers that plays gslic() (main.cpp:598-660): labels equal the
    reference's GPU engine, Draw_Segmentation_Result marks label boundaries, Write_Seg_Res_To_PGM writes the 16-bit map."""
    import ctypes as C
    pkg, rb = env
    so = os.path.join(pc.ROOT, "oracle", "_ref", "libgslicr_harness.so")
    if not os.path.exists(so):
        pytest.skip("the harness compiles against the reference checkout's own gSLICr headers (`make oracle` where it exists)")
    h = C.CDLL(so)
    scene = pkg.scene.make_scene("C1", with_colour=True)
    rgbx = pkg.scene.box_downsample4(scene["bgr"])
    hh, ww = rgbx.shape[:2]
    labels = np.zeros((hh, ww), np.int32)
    drawn = np.zeros((hh, ww, 4), np.uint8)
    pgm = str(tmp_path / "seg.pgm")
    rc = h.gslicr_harness_run(rgbx.ctypes.data_as(C.c_void_p), ww, hh, 20, 5, C.c_float(5.0), 0, labels.ctypes.data_as(C.c_void_p),
                              drawn.ctypes.data_as(C.c_void_p), pgm.encode())
    assert rc == 0
    ref, _ = rb.ref_slic(rgbx, spixel_size=20, no_iters=5, coh_weight=5.0, enforce_connectivity=False)
    assert (labels == ref).all(), f"{(labels != ref).mean():.4%} of labels differ"
    inner = np.zeros((hh, ww), bool)
    inner[1:-1, 1:-1] = True
    edge = np.zeros((hh, ww), bool)
    edge[1:-1, 1:-1] = ((labels[1:-1, 1:-1] != labels[1:-1, 2:]) | (labels[1:-1, 1:-1] != labels[1:-1, :-2]) |
                        (labels[1:-1, 1:-1] != labels[:-2, 1:-1]) | (labels[1:-1, 1:-1] != labels[2:, 1:-1]))
    assert (drawn[edge] == np.array([0, 0, 255, 0], np.uint8)).all()
    assert (drawn[inner & ~edge] == rgbx[inner & ~edge]).all()
    assert (drawn[~inner] == 7).all()                       # border pixels are not written (GPU.cu:229)
    raw = open(pgm, "rb").read()
    head = f"P5\n{ww} {hh}\n65535\n".encode()
    assert raw.startswith(head) and len(raw) == len(head) + 2 * ww * hh
    assert np.array_equal(np.frombuffer(raw[len(head):], ">u2").reshape(hh, ww), labels.astype(np.uint16))


def test_reference_entry_points_drop_in(env, small):
    """firstcuda / sliccuda / fakecuda / fillcuda (gipuma.h:2-5) exported by libtsar_b200.so, driven by a harness that
    plays the reference's host program (managed GlobalState with the reference's layout, float textures in
    cudaArrays): (a) north-star PatchMatch mode == the engine's own sequence, (b) shipped flow == reference build."""
    import ctypes as C
    import os
    pkg, rb = env
    L = pkg._lib
    scene = small
    so = os.path.join(pc.ROOT, "tests", "libshim_harness.so")
    assert os.path.exists(so), "tests/libshim_harness.so missing: run `make oracle`"
    h = C.CDLL(so)
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    params = pkg.make_params(box=11, iterations=2, min_disparity=scene["min_disparity"], max_disparity=scene["max_disparity"])
    imgs = [np.ascontiguousarray(im, np.float32) for im in scene["images"]]
    ptrs = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
    sub = (C.c_int * len(scene["subset"]))(*scene["subset"])
    H, W = imgs[0].shape
    n = W * H

    def run(shipped, imp_n4=None, imp_disp=None):
        o_n4, o_cf = np.zeros((H, W, 4), np.float32), np.zeros((H, W), np.float32)
        o_fd, o_sc = np.zeros((H, W), np.float32), np.zeros((H, W), np.float32)
        imp_n4 = np.zeros((H, W, 4), np.float32) if imp_n4 is None else np.ascontiguousarray(imp_n4, np.float32)
        imp_disp = np.zeros((H, W), np.float32) if imp_disp is None else np.ascontiguousarray(imp_disp, np.float32)
        rc = h.shim_harness_run(W, H, len(imgs), ptrs, cams, C.c_float(scene["cam_f"]), sub, len(scene["subset"]), C.byref(params),
                                scene["canny"].ctypes.data_as(C.c_void_p), len(scene["region_text"]),
                                scene["region_text"].ctypes.data_as(C.c_void_p), scene["region_norm4"].ctypes.data_as(C.c_void_p),
                                int(shipped), imp_n4.ctypes.data_as(C.c_void_p), imp_disp.ctypes.data_as(C.c_void_p),
                                o_n4.ctypes.data_as(C.c_void_p), o_cf.ctypes.data_as(C.c_void_p), o_fd.ctypes.data_as(C.c_void_p),
                                o_sc.ctypes.data_as(C.c_void_p))
        assert rc == 0
        return o_n4, o_cf, o_fd, o_sc

    # (a) north-star mode through the reference's entry points == engine sequence
    os.environ["TSAR_B200_PATCHMATCH"] = "1"
    os.environ["TSAR_B200_SEED"] = str(SEED)
    try:
        s_n4, s_cf, s_fd, s_sc = run(False)
    finally:
        del os.environ["TSAR_B200_PATCHMATCH"]
    _, eng, _ = pc.make_engines(pkg, scene, iterations=2, variants=())
    eng.set_regions(scene["region_text"], scene["region_norm4"])
    eng.upload(L.F_CANNY, scene["canny"])
    eng.init_planes(SEED); eng.iterate(2, SEED); eng.lrdiff(); eng.getview()
    cf = eng.download(L.F_CONFID)
    eng.update_scale_2(); eng.update_scale(); eng.compute_disp()
    assert pc.frac_bit_exact(s_cf, cf) == 1.0
    # the same through BGRA float4 arrays (color_processing): the shim takes channel x, as the kernels would
    params_grey = params
    params = pkg.make_params(box=11, iterations=2, min_disparity=scene["min_disparity"], max_disparity=scene["max_disparity"],
                             color_processing=1)
    os.environ["TSAR_B200_PATCHMATCH"] = "1"
    try:
        c_n4, c_cf, _, _ = run(False)
    finally:
        del os.environ["TSAR_B200_PATCHMATCH"]
    params = params_grey
    assert pc.frac_bit_exact(c_n4, s_n4) == 1.0 and pc.frac_bit_exact(c_cf, s_cf) == 1.0
    assert pc.frac_bit_exact(s_n4, eng.download(L.F_NORM4)) == 1.0
    assert pc.frac_bit_exact(s_fd, eng.download(L.F_FAKEDEPTH)) == 1.0
    assert pc.frac_bit_exact(s_sc, eng.download(L.F_SCALE)) == 1.0
    eng.close()
    # (b) shipped flow (imported normals + disparities -> get_disp -> getview -> fake -> fill) == reference build
    rng = np.random.RandomState(3)
    wn = rng.normal(size=(H, W, 4)).astype(np.float32)
    wn[..., :3] /= np.linalg.norm(wn[..., :3], axis=-1, keepdims=True)
    disp = (scene["cam_f"] / scene["gt_depth"]).astype(np.float32)
    s_n4, s_cf, s_fd, s_sc = run(True, wn, disp)
    _, _, refs = pc.make_engines(pkg, scene, iterations=2, variants=("asis",))
    ref = refs["asis"]
    ref.set_regions(scene["region_text"], scene["region_norm4"])
    ref.upload(rb.F_CANNY, scene["canny"])
    ref.upload(rb.F_NORM4, wn); ref.upload(rb.F_COST, np.ones((H, W), np.float32)); ref.upload(rb.F_DEPTH, disp)
    ref.get_disp(); ref.getview()
    assert pc.frac_bit_exact(s_cf, ref.download(rb.F_CONFID)) == 1.0
    ref.update_scale_2(); ref.update_scale(); ref.compute_disp()
    assert pc.frac_bit_exact(s_n4, ref.download(rb.F_NORM4)) == 1.0
    assert pc.frac_bit_exact(s_fd, ref.download(rb.F_FAKEDEPTH)) == 1.0
    assert pc.frac_bit_exact(s_sc, ref.download(rb.F_SCALE)) == 1.0
    ref.close()
    # (c) TSAR_B200_WMF=1: the weighted-median stages at the launch sites where the reference has them commented out
    # (gipuma_WMF x 4 at the end of sliccuda, gipuma_WMF_Final x 6 in fillcuda; gipuma.cu:1809-1812, 1844-1847), fed with the
    # reliable flags main() takes from weak.png before sliccuda == the engine running the same sequence
    reliable = (rng.rand(H, W) < 0.6).astype(np.float32)
    h.shim_harness_set_reliable(reliable.ctypes.data_as(C.c_void_p))
    os.environ["TSAR_B200_WMF"] = "1"
    try:
        w_n4, w_cf, w_fd, w_sc = run(True, wn, disp)
    finally:
        del os.environ["TSAR_B200_WMF"]
        h.shim_harness_set_reliable(None)
    _, eng, _ = pc.make_engines(pkg, scene, iterations=2, variants=())
    eng.set_regions(scene["region_text"], scene["region_norm4"])
    eng.upload(L.F_CANNY, scene["canny"])
    eng.upload(L.F_NORM4, wn); eng.upload(L.F_COST, np.ones((H, W), np.float32)); eng.upload(L.F_DEPTH, disp)
    eng.get_disp(); eng.getview()
    eng.upload(L.F_SCALE, reliable)
    for it in range(4):
        eng.wmf(it)
    eng.update_scale_2(); eng.update_scale()
    for it in range(6):
        eng.wmf_final(it)
    eng.compute_disp()
    assert pc.frac_bit_exact(w_cf, s_cf) == 1.0                         # the confidence map is computed before the filter
    assert pc.frac_bit_exact(w_n4, eng.download(L.F_NORM4)) == 1.0
    assert pc.frac_bit_exact(w_fd, eng.download(L.F_FAKEDEPTH)) == 1.0
    assert pc.frac_bit_exact(w_sc, eng.download(L.F_SCALE)) == 1.0
    assert pc.frac_bit_exact(w_n4, s_n4) < 0.999                        # and the filter changed the result
    eng.close()


@pytest.mark.parametrize("variant", ["snapshot_init", "snapshot"])
def test_wmf_and_wmf_final_bit_exact(env, small, variant):
    """gipuma_WMF x4 and gipuma_WMF_Final x6 (gipuma.cu:1500-1698, 1295-1497; launch sites 1809-1812, 1844-1847)
    against the race-free reference build: scale after every consistency level, then planes/disparities/flags after
    every fill level.  Includes the reference's bubble-sort off-by-one (dummy element, largest element dropped).
    When a weighted median is never reached (tiny neighbour lists) the reference reads its `float4 norm_mid` uninitialised
    (gipuma.cu:1423, 1625), i.e. is undefined there.  Variant 'snapshot_init' is the twin with that ONE variable
    zero-initialised at build time (oracle/build_ref.sh 2b): against it every pixel of every level must agree, 100 %.
    Against the twin as written the same comparison may differ on the undefined pixels only (bounded, < 5e-4)."""
    pkg, rb = env
    L = pkg._lib
    scene = small
    params, mine, refs = pc.make_engines(pkg, scene, iterations=3, variants=(variant,))
    ref = refs[variant]
    bound = 0.0 if variant == "snapshot_init" else 5e-4
    ref.init_planes(SEED); ref.iterate(3, SEED); ref.lrdiff(); ref.getview()
    n0, c0, d0 = ref.download(rb.F_NORM4), ref.download(rb.F_COST), ref.download(rb.F_DEPTH)
    reliable = (c0 < 0.25).astype(np.float32)          # stands in for APD's weak.png (main.cpp:1499-1514)
    assert 0.2 < reliable.mean() < 0.98
    mine.load_planes(n0, c0); mine.upload(L.F_DEPTH, d0); mine.upload(L.F_SCALE, reliable)
    ref.upload(rb.F_SCALE, reliable)
    # Bar: identical except where the reference itself is undefined -- when a weighted median is never reached
    # (tiny neighbour lists) it reads an uninitialised norm_mid component (gipuma.cu:1625-1649).  Each level starts
    # from the reference's state so levels are judged independently; mismatches are counted and bounded.
    changed, worst = 0.0, 0.0
    for it in range(4):
        mine.upload(L.F_SCALE, ref.download(rb.F_SCALE))
        ref.wmf(it); mine.wmf(it)
        s_m, s_r = mine.download(L.F_SCALE), ref.download(rb.F_SCALE)
        worst = max(worst, float((s_m != s_r).mean()))
        changed = max(changed, float((s_r != reliable).mean()))
    print(f"\n[wmf] worst per-level label mismatch {worst:.5%}")
    assert worst <= bound
    assert changed > 0.01                                # the filter really re-classified pixels
    for e in (mine, ref):
        e.set_regions(scene["region_text"], scene["region_norm4"])
    mine.upload(L.F_CANNY, scene["canny"]); ref.upload(rb.F_CANNY, scene["canny"])
    before = ref.download(rb.F_SCALE).copy()
    for it in range(6):
        for fm, fr in ((L.F_NORM4, rb.F_NORM4), (L.F_DEPTH, rb.F_DEPTH), (L.F_SCALE, rb.F_SCALE)):
            mine.upload(fm, ref.download(fr))
        ref.wmf_final(it); mine.wmf_final(it)
        for fm, fr in ((L.F_NORM4, rb.F_NORM4), (L.F_DEPTH, rb.F_DEPTH), (L.F_SCALE, rb.F_SCALE)):
            a, b = mine.download(fm), ref.download(fr)
            miss = 1 - pc.frac_bit_exact(a, b)
            worst = max(worst, miss)
            assert miss <= bound, f"WMF_Final level {it} field {fm}: {miss:.4%} differ"
    print(f"[wmf_final] worst per-level mismatch {worst:.5%}")
    assert (ref.download(rb.F_SCALE) != before).mean() > 0.001   # pixels were filled
    mine.close(); ref.close()


@pytest.mark.parametrize("density", [0.9, 0.03])
def test_wmf_cooperative_equals_per_thread(env, monkeypatch, density):
    """The warp-cooperative gipuma_WMF (bitonic sort of (key, slot) composites, sequential sums by one lane) and the
    per-thread implementation (merge sort in local memory) give identical flags on every level, on an image with
    borders, unreliable areas and ties (propagated planes are exact copies) -- and on a SPARSE reliable mask (3 %), where
    most pixels have one or two reliable neighbours and the bubble sort's dummy element is the one that reaches half the
    weight: the reference then takes pixel (0, 0) as the median's pixel (found by tools/gpu_wmf_sweep.py in round 2: the
    cooperative kernel got that case wrong, up to 12 % of the flags of such a level)."""
    pkg, rb = env
    L = pkg._lib
    cfg = dict(W=333, H=201, n_images=3, V=2, fx=400.0, radius=2.0, arc_deg=12.0)
    scene = pkg.scene.make_scene(cfg)
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot_init",))
    ref = refs["snapshot_init"]
    mine.depthmap(SEED)
    mine.init_planes(SEED); mine.iterate(2, SEED); mine.lrdiff(); mine.getview()
    cost = mine.download(L.F_COST)
    rng = np.random.RandomState(4)
    reliable = ((cost < (0.3 if density > 0.5 else 3.0)) & (rng.rand(*cost.shape) < density)).astype(np.float32)
    reliable[:, :40] = 0                                   # a band with (almost) no reliable neighbours
    reliable[60:64, 100:104] = 1
    # the same state on the reference twin (zero-initialised norm_mid: defined everywhere)
    ref.upload(rb.F_NORM4, mine.download(L.F_NORM4)); ref.upload(rb.F_COST, cost); ref.upload(rb.F_DEPTH, mine.download(L.F_DEPTH))
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("TSAR_B200_WMF_PER_THREAD", mode)
        mine.upload(L.F_SCALE, reliable)
        levels = []
        for it in range(4):
            mine.wmf(it)
            levels.append(mine.download(L.F_SCALE).copy())
        outs[mode] = levels
    monkeypatch.delenv("TSAR_B200_WMF_PER_THREAD")
    ref.upload(rb.F_SCALE, reliable)
    ref_levels = []
    for it in range(4):
        ref.wmf(it)
        ref_levels.append(ref.download(rb.F_SCALE).copy())
    mine.close(); ref.close()
    for it in range(4):
        assert np.array_equal(outs["0"][it], outs["1"][it]), (it, float((outs["0"][it] != outs["1"][it]).mean()))
        assert np.array_equal(outs["0"][it], ref_levels[it]), (it, float((outs["0"][it] != ref_levels[it]).mean()))
    if density > 0.5:
        assert 0.05 < outs["0"][3].mean() < 0.999


def test_region_plane_fit_matches_reference_code(env, small):
    """Per-region RANSAC plane fit on the device (one cooperative kernel, loop termination on the device) against the
    reference's OWN loop -- main.cpp:1520-1730 cut out of the checkout and compiled by oracle/build_ref.sh
    (oracle/_ref/libtsar_ref_host.so) -- fed with the same rand() stream; both sides are IEEE double without contraction:
    bit-exact bar.  Also: the C restatement agrees, the fit is geometrically right, the seeded device stream reproduces,
    and a second call on the same context (persistent scratch) gives the same planes."""
    pkg, rb = env
    L = pkg._lib
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    rh = pc.ref_host()
    scene = small
    params, mine, _ = pc.make_engines(pkg, scene, variants=())
    H, W = scene["H"], scene["W"]
    rng = np.random.RandomState(9)
    # disparities of the true surface + noise + 20 % gross outliers; every second pixel "reliable"
    disp = (scene["cam_f"] / scene["gt_depth"]).astype(np.float32)
    disp *= (1 + 0.0005 * rng.normal(size=disp.shape)).astype(np.float32)
    out = rng.rand(H, W) < 0.2
    disp[out] *= rng.uniform(0.8, 1.2, out.sum()).astype(np.float32)
    scale = (rng.rand(H, W) < 0.5).astype(np.float32)
    text = scene["region_text"].copy()
    text[1] = -1.0                                         # a second region to fit, besides the textureless facet
    size = np.array([(scene["labels"] == r).sum() / 16.0 for r in range(len(text))], np.float32)
    per = mine.lib.tsar_ransac_rand_per_region()
    rnd = rng.randint(0, 2 ** 31 - 1, size=(len(text), per)).astype(np.uint32)
    mine.upload(L.F_DEPTH, disp); mine.upload(L.F_SCALE, scale); mine.upload(L.F_CANNY, scene["canny"])
    p0 = np.tile(np.array([0, 0, 1, -1], np.float32), (len(text), 1))
    fitted = mine.fit_region_planes(text, size, rnd, p0)
    again = mine.fit_region_planes(text, size, rnd, p0)
    assert pc.frac_bit_exact(fitted, again) == 1.0
    stream = np.concatenate([rnd[r] for r in range(len(text)) if text[r] == -1])
    ref, used = rh.fit_regions(scene["cams"][0], scene["cam_f"], disp, scale, scene["canny"], text, size, stream, p0)
    assert used == len(stream)
    assert pc.frac_bit_exact(fitted, ref) == 1.0, (fitted, ref)
    cams = cameras_to_struct(scene["cams"])
    for r in range(len(text)):
        if text[r] != -1:
            assert np.array_equal(fitted[r], p0[r])
            continue
        want, n_used = cb.fit_region_plane(pkg._lib.TsarCamera, cams[0], scene["cam_f"], disp, scale, scene["canny"], r, size[r], rnd[r], p0[r])
        assert n_used > 1000
        assert pc.frac_bit_exact(fitted[r], want) == 1.0, (r, fitted[r], want)
        # the fitted plane is the facet's true plane (n.X + d = 0 in the reference frame), up to sign
        true = scene["region_norm4"][r].astype(np.float64)   # generator planes carry a small perturbation
        cosang = abs(np.dot(fitted[r][:3], true[:3]) / np.linalg.norm(fitted[r][:3]) / np.linalg.norm(true[:3]))
        assert cosang > np.cos(np.radians(8.0)), (r, fitted[r], true)
    # device-generated stream (tsar_fit_region_planes_seeded) == the reference's loop fed with that stream
    seeded = mine.fit_region_planes(text, size, None, p0, seed=77)
    with np.errstate(over="ignore"):
        stream = np.concatenate([mine.ransac_rand_stream(77, r) for r in range(len(text)) if text[r] == -1])
    ref2, _ = rh.fit_regions(scene["cams"][0], scene["cam_f"], disp, scale, scene["canny"], text, size, stream, p0)
    assert pc.frac_bit_exact(seeded, ref2) == 1.0, (seeded, ref2)
    assert mine.lib.tsar_ransac_rand_value(77, 4, 5) == int(stream[per + 5])
    # edge cases: a region without any reliable pixel keeps its plane; a one-region table
    scale0 = scale.copy()
    scale0[scene["labels"] == 1] = 0
    mine.upload(L.F_SCALE, scale0)
    kept = mine.fit_region_planes(text, size, rnd, p0)
    assert np.array_equal(kept[1], p0[1]) and pc.frac_bit_exact(kept[4], fitted[4]) == 1.0
    mine.close()


def test_c1_shape_many_views_bit_exact(env):
    """BASELINE config C1 (640x480, 15 source views): exercises V > 10 and the reference's launch geometry."""
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene("C1")
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot",))
    ref = refs["snapshot"]
    mine.depthmap(SEED); ref.depthmap(SEED, iters=2)
    a = pc.output_agreement(mine.download(L.F_NORM4), ref.download(rb.F_NORM4))
    assert a["bit_exact"] == 1.0, a
    assert pc.frac_bit_exact(mine.download(L.F_CONFID), ref.download(rb.F_CONFID)) == 1.0
    assert mine.eval_count(8) == 519628800   # exact border-guard count; BASELINE.md's interior approximation: 0.521 G
    mine.close(); ref.close()


FULL_SIZE_CASES = {
    # BASELINE.json configs at their full sizes, 8 iterations, blocksize 11 (the run scripts' settings)
    "C2": "C2",                                                                                     # 3100x2050, V = 10
    "C4": "C4",                                                                                     # 1920x1080, V = 10
    "C5": "C5",                                                                                     # 6048x4032, V = 20 (about 30 s)
    "C5crop": dict(W=1512, H=1008, n_images=21, V=20, fx=3410.0, radius=6.0, arc_deg=40.0),         # C5's cameras and V = 20 on a crop
}


@pytest.mark.parametrize("case", ["C2", "C4", "C5crop", "C5"])
def test_baseline_size_bit_exact_vs_reference(env, case):
    """The whole per-view sequence (gipuma.cu:1741-1761: init, 8 x (bSP, bPR, rSP, rPR), getlrdiff, getview, compute_disp)
    at BASELINE sizes against the reference's own kernels (race-free twin): depth, normals, confidence, best view and
    cost bit for bit.  The reference needs about 2 s per C2 depthmap on a B200."""
    import torch
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene(FULL_SIZE_CASES[case], backend="torch", device="cuda:0")
    scene["images"] = [im.cpu().numpy() for im in scene["images"]]
    torch.cuda.empty_cache()
    params, mine, refs = pc.make_engines(pkg, scene, iterations=8, variants=("snapshot",))
    snap = refs["snapshot"]
    mine.depthmap(SEED)
    snap.depthmap(SEED, iters=8)
    res = {"case": case, "W": scene["W"], "H": scene["H"], "V": len(scene["subset"])}
    for name, fm, fr in (("output", L.F_NORM4, rb.F_NORM4), ("confidence", L.F_CONFID, rb.F_CONFID), ("cost", L.F_COST, rb.F_COST),
                         ("lrdiff", L.F_LRDIFF, rb.F_LRDIFF), ("ratio", L.F_RATIO, rb.F_RATIO)):
        res[name] = pc.frac_bit_exact(mine.download(fm), snap.download(fr))
    res["best_view"] = float((mine.download(L.F_BEVIEW) == snap.download(rb.F_BEVIEW)).mean())
    out = mine.download(L.F_NORM4)
    res["gt"] = pc.gt_agreement(out, scene)
    mine.close(); snap.close()
    pc.record(f"full_size_parity_{case}.json", res)
    print("\n", res)
    for k in ("output", "confidence", "cost", "lrdiff", "ratio", "best_view"):
        assert res[k] == 1.0, res
    assert res["gt"]["frac_within_1pct_textured"] > 0.95, res   # and it converged to the true surface


def test_c2_agreement_with_reference_as_written(env):
    """C2, 8 iterations, against the reference build AS WRITTEN (its propagation launch races on same-colour pixels,
    SURVEY Q3, so it does not reproduce itself): ours must be exactly as far from it as its race-free twin is, and the
    north-star tolerance figures are recorded next to the build's own run-to-run figures (depth and normals, textured
    and untextured pixels).  Writes the record that profiles/r02_agreement_with_asis_reference_C2.json is copied from."""
    import torch
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene("C2", backend="torch", device="cuda:0")
    scene["images"] = [im.cpu().numpy() for im in scene["images"]]
    torch.cuda.empty_cache()
    params, mine, refs = pc.make_engines(pkg, scene, iterations=8, variants=("asis", "snapshot"))
    asis, snap = refs["asis"], refs["snapshot"]
    mine.depthmap(SEED); o_m = mine.download(L.F_NORM4); mine.close()
    snap.depthmap(SEED, iters=8); o_s = snap.download(rb.F_NORM4); snap.close()
    asis.depthmap(SEED, iters=8); o_a = asis.download(rb.F_NORM4)
    asis.depthmap(SEED, iters=8); o_a2 = asis.download(rb.F_NORM4); asis.close()
    tex = scene["region_text"][scene["labels"]] > 0

    def masked(a, b, m):
        return pc.output_agreement(a[m][None], b[m][None])

    res = {"config": "C2", "iterations": 8, "ours_vs_snapshot_bit_exact": pc.frac_bit_exact(o_m, o_s),
           "ours_vs_asis": pc.output_agreement(o_m, o_a), "snapshot_vs_asis": pc.output_agreement(o_s, o_a),
           "asis_vs_asis": pc.output_agreement(o_a2, o_a),
           "ours_vs_asis_textured": masked(o_m, o_a, tex), "asis_vs_asis_textured": masked(o_a2, o_a, tex),
           "ours_vs_asis_untextured": masked(o_m, o_a, ~tex), "asis_vs_asis_untextured": masked(o_a2, o_a, ~tex),
           "gt_ours": pc.gt_agreement(o_m, scene), "gt_asis": pc.gt_agreement(o_a, scene), "textured_fraction": float(tex.mean())}
    pc.record("agreement_with_asis_reference_C2.json", res)
    print("\n", {k: (v if not isinstance(v, dict) else {q: round(w, 4) for q, w in v.items()}) for k, v in res.items()})
    assert res["ours_vs_snapshot_bit_exact"] == 1.0
    for k in ("frac_ok", "frac_depth_ok", "frac_angle_ok"):
        assert res["ours_vs_asis"][k] == res["snapshot_vs_asis"][k]      # ours == twin in distance to the racy build
    assert res["ours_vs_asis_textured"]["frac_depth_ok"] > 0.99           # depth of textured pixels inside the gate
    assert abs(res["gt_ours"]["frac_within_1pct_textured"] - res["gt_asis"]["frac_within_1pct_textured"]) < 0.005


def test_full_size_properties(env, monkeypatch):
    """Size-independent properties at BASELINE config C2 (3100x2050, 10 source views): determinism, 8-bit vs fp32 source
    textures identical, evaluation count."""
    import torch
    pkg, rb = env
    L = pkg._lib
    scene = pkg.scene.make_scene("C2", backend="torch", device="cuda:0")
    imgs = [im.contiguous() for im in scene["images"]]
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    params = pkg.make_params(box=11, iterations=8, min_disparity=scene["min_disparity"], max_disparity=scene["max_disparity"])

    def run(env_pairs=()):
        for k, v in env_pairs:
            monkeypatch.setenv(k, v)
        eng = pkg.DepthmapEngine(0)
        eng.set_views_device([t.data_ptr() for t in imgs], scene["W"], scene["H"], cams, scene["subset"], cam_f=scene["cam_f"])
        eng.set_params(params)
        eng.depthmap(SEED)
        out = eng.download(L.F_NORM4)
        n_ev = eng.eval_count(8)
        eng.close()
        for k, _ in env_pairs:
            monkeypatch.delenv(k)
        return out, n_ev

    a, n_ev = run()
    b, _ = run()
    assert pc.frac_bit_exact(a, b) == 1.0                                   # deterministic
    c, _ = run((("TSAR_B200_NO_U8", "1"),))
    assert pc.frac_bit_exact(a, c) == 1.0                                   # 8-bit textures == fp32 textures
    gt = pc.gt_agreement(a, scene)
    assert gt["frac_within_1pct_textured"] > 0.95, gt                       # converged to the true surface
    assert 6.6e9 < n_ev < 6.8e9                                             # 6.67 G pmCost evaluations per depthmap as written
    del imgs
    torch.cuda.empty_cache()


def test_cli_end_to_end_on_synthetic_dataset(env, tmp_path):
    """tsar_cli.py with the reference's flags on a dataset in the reference's folder layout: writes TSAR_disp.dmb /
    TSAR_normals.dmb (fileIoUtils.h:333-381) identical to driving the engine directly."""
    import subprocess
    import sys
    pkg, rb = env
    L = pkg._lib
    root = str(tmp_path / "ds") + "/"
    cmd = [sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "--synthetic=tiny", "-mslp_folder", root, "-krt_file", "x",
           "-no_display", "--cam_scale=1", "--iterations=3", "--blocksize=11", "--cost_comb=best_n", "--n_best=1",
           "--min_angle=", "--max_angle=", f"--seed={SEED}"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    from tsar_mvs_b200 import dmb
    depth = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
    normal = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_normals.dmb"))
    scene = pkg.scene.make_scene("tiny")
    params, mine, _ = pc.make_engines(pkg, scene, iterations=3, variants=())
    mine.depthmap(SEED)
    out = mine.download(L.F_NORM4)
    mine.close()
    assert depth.shape == (scene["H"], scene["W"]) and normal.shape == (scene["H"], scene["W"], 3)
    assert pc.frac_bit_exact(depth, out[..., 3]) == 1.0
    assert pc.frac_bit_exact(normal, np.ascontiguousarray(out[..., :3])) == 1.0


def test_cli_all_views_resident_pool(env, tmp_path):
    """`-all_views`: every image is the reference view once, images resident on the GPU, two pipelined contexts.
    View 0 must equal the one-view command line bit for bit; every view must produce its three files."""
    import subprocess
    import sys
    pkg, rb = env
    from tsar_mvs_b200 import dmb
    root = str(tmp_path / "ds") + "/"
    common = ["-mslp_folder", root, "-krt_file", "x", "-no_display", "--cam_scale=1", "--iterations=2", "--blocksize=11",
              "--cost_comb=best_n", "--n_best=1", f"--seed={SEED}"]
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "--synthetic=tiny"] + common,
                       capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    one = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
    one_n = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_normals.dmb"))
    os.remove(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "-all_views", "-images_folder", root + "images/"] + common,
                       capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    n = pkg.scene.CONFIGS["tiny"]["n_images"]
    assert f"{n} of {n} reference views" in r.stdout
    for v in range(n):
        d = dmb.read_dmb(os.path.join(root, "APD", f"{v:08d}", "TSAR_disp.dmb"))
        assert d.shape == one.shape and np.isfinite(d).all() and (d > 0).mean() > 0.5
        assert os.path.exists(os.path.join(root, "APD", f"{v:08d}", "TSAR_confidence.dmb"))
    assert pc.frac_bit_exact(dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb")), one) == 1.0
    assert pc.frac_bit_exact(dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_normals.dmb")), one_n) == 1.0
    # the persistent driver (contexts and pinned buffers kept between passes, as the benchmark's passes do): a warm-up
    # pass over two views and two full passes in this process write the same files again
    import shutil
    ref_files = {v: dmb.read_dmb(os.path.join(root, "APD", f"{v:08d}", "TSAR_normals.dmb")) for v in range(n)}
    opt = pkg.cli.parse_args(["-all_views", "-images_folder", root + "images/"] + common)
    pkg.cli.run_all_views(dict(opt, views_per_rank=2), root, quiet=True, persistent=True)
    for _ in range(2):
        shutil.rmtree(os.path.join(root, "APD"))
        res = pkg.cli.run_all_views(opt, root, quiet=True, persistent=True)
        assert res["views"] == n and res["gpu_launches"] > 0
        for v in range(n):
            assert pc.frac_bit_exact(dmb.read_dmb(os.path.join(root, "APD", f"{v:08d}", "TSAR_normals.dmb")), ref_files[v]) == 1.0
    assert len(pkg.cli._LANE_POOL) == 1
    pkg.cli.release_lanes()
    assert not pkg.cli._LANE_POOL
    # -resume: only the views whose outputs are missing (or incomplete: a .part file does not count) are computed again
    os.remove(os.path.join(root, "APD", "00000001", "TSAR_normals.dmb"))
    os.rename(os.path.join(root, "APD", "00000002", "TSAR_disp.dmb"), os.path.join(root, "APD", "00000002", "TSAR_disp.dmb.part"))
    res = pkg.cli.run_all_views(dict(opt, resume=True), root, quiet=True)
    assert res["views"] == 2 and res["skipped"] == n - 2
    for v in range(n):
        assert pc.frac_bit_exact(dmb.read_dmb(os.path.join(root, "APD", f"{v:08d}", "TSAR_normals.dmb")), ref_files[v]) == 1.0
    res = pkg.cli.run_all_views(dict(opt, resume=True), root, quiet=True)
    assert res["views"] == 0 and res["skipped"] == n


def test_labels_quarter_expansion_on_device(env):
    """lines->canny from the quarter-resolution region labels (main.cpp:558-568), expanded by a kernel: equals the
    plain-Python restatement, including the stepped-back last column/row of sizes that are not multiples of 4."""
    pkg, rb = env
    L = pkg._lib
    from oracle import weak_texture_ref as wr
    cfg = dict(W=67, H=33, n_images=2, V=1, fx=150.0, radius=1.0, arc_deg=14.0)
    scene = pkg.scene.make_scene(cfg)
    params, mine, _ = pc.make_engines(pkg, scene, variants=())
    lab = np.random.RandomState(2).randint(0, 9, size=(33 // 2 // 2, 67 // 2 // 2)).astype(np.int32)
    mine.set_labels_quarter(lab)
    got = mine.download(L.F_CANNY)
    assert np.array_equal(got, wr.expand(lab, 67, 33))
    assert np.array_equal(got, pkg.texture.expand_labels(lab, 67, 33))
    with pytest.raises(Exception):
        mine.set_labels_quarter(lab[:, :5])
    mine.close()


def test_cli_full_tsar_flow_with_detector(env, tmp_path):
    """The whole TSAR flow from files: weak-texture detector (texture.py) -> PatchMatch -> confidence -> per-region
    RANSAC plane on the device -> depth completion -> .dmb.  The untextured facet must end up closer to the ground
    truth than without completion (`-no_weak_texture`)."""
    import subprocess
    import sys
    pkg, rb = env
    from tsar_mvs_b200 import dmb
    root = str(tmp_path / "ds") + "/"
    common = ["-mslp_folder", root, "-krt_file", "x", "-no_display", "--cam_scale=1", "--iterations=4", "--blocksize=11",
              "--cost_comb=best_n", "--n_best=1", f"--seed={SEED}"]
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "--synthetic=mid"] + common,
                       capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "weakly textured" in r.stdout
    with_fill = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
    names = sorted(os.listdir(root + "images"))
    r2 = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py")] + names + ["-images_folder", root + "images/", "-no_weak_texture"] + common,
                        capture_output=True, text=True, cwd=pc.ROOT)
    assert r2.returncode == 0, r2.stderr[-2000:]
    without = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
    cfg = pkg.scene.CONFIGS["mid"]
    cams = pkg.scene.make_cameras(cfg["W"], cfg["H"], cfg["n_images"], cfg["fx"], cfg["radius"], cfg["arc_deg"])
    _, gt, labels = pkg.scene.Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"]).render(cams[0], cfg["W"], cfg["H"])
    flat = labels == 4
    err_fill = np.abs(with_fill - gt)[flat] / gt[flat]
    err_raw = np.abs(without - gt)[flat] / gt[flat]
    print(f"\n[facet] median rel. depth error: completed {np.median(err_fill):.4f}, PatchMatch only {np.median(err_raw):.4f}; "
          f"within 2 %: {np.mean(err_fill < 0.02):.3f} vs {np.mean(err_raw < 0.02):.3f}\n{r.stdout[-400:]}")
    assert np.mean(err_fill < 0.02) > 0.9 > np.mean(err_raw < 0.02)
    assert np.median(err_fill) < 0.01
    ground = (labels == 0) & (without > 0)
    assert np.mean(with_fill[ground] == without[ground]) > 0.95   # textured regions are left as PatchMatch found them
    # -all_views runs the same whole flow (detector, gSLICr, PatchMatch, RANSAC, completion) for every view: view 0 must
    # give the same files as the one-view command, bit for bit -- without and with the weighted-median stages (-wmf)
    for extra in ([], ["-wmf"]):
        r1 = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py")] + names + ["-images_folder", root + "images/"] + common + extra,
                            capture_output=True, text=True, cwd=pc.ROOT)
        assert r1.returncode == 0, r1.stderr[-2000:]
        one = {f: open(os.path.join(root, "APD", "00000000", f), "rb").read() for f in ("TSAR_disp.dmb", "TSAR_normals.dmb", "TSAR_confidence.dmb")}
        for f in one:
            os.remove(os.path.join(root, "APD", "00000000", f))
        r3 = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "-all_views", "-images_folder", root + "images/"] + common + extra,
                            capture_output=True, text=True, cwd=pc.ROOT)
        assert r3.returncode == 0, r3.stderr[-2000:]
        assert f"{len(names)} of {len(names)} reference views" in r3.stdout
        for f, want in one.items():
            assert open(os.path.join(root, "APD", "00000000", f), "rb").read() == want, (extra, f)
        if not extra:
            assert one["TSAR_disp.dmb"][16:] == with_fill.tobytes()      # and the completion really ran in both
        else:
            wmf_depth = dmb.read_dmb(os.path.join(root, "APD", "00000000", "TSAR_disp.dmb"))
            assert (wmf_depth != with_fill).mean() > 1e-4               # the weighted-median fill changed pixels


def test_cli_shipped_flow_from_an_apd_folder(env, tmp_path):
    """`-import_apd`: the flow the reference ships (main.cpp:1459-1783) from files -- planes from APD/<view>/depths_geom.dmb +
    normals.dmb, reliable pixels from APD/<view>/weak.png (white, green or red, main.cpp:1499-1514), detector, per-region
    RANSAC, completion -- against the same flow assembled from the reference's own pieces: its kernels (oracle/_ref
    libtsar_ref.so: get_disp, getview, update_scale_2, update_scale, compute_disp) and its own RANSAC loop
    (libtsar_ref_host.so) fed with the random stream the command line uses.  Output files bit for bit."""
    import subprocess
    import sys
    import cv2
    pkg, rb = env
    from tsar_mvs_b200 import cli, dmb, texture
    from tsar_mvs_b200.engine import cameras_to_struct
    rh = pc.ref_host()
    root = str(tmp_path / "ds") + "/"
    common = ["-mslp_folder", root, "-krt_file", "x", "-no_display", "--cam_scale=1", "--iterations=2", "--blocksize=11",
              "--cost_comb=best_n", "--n_best=1", f"--seed={SEED}"]
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py"), "--synthetic=mid"] + common,
                       capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    apd = os.path.join(root, "APD", "00000000")
    # what APD / Fusion would have left in the folder: a depth map, a normal map and weak.png
    cfg = pkg.scene.CONFIGS["mid"]
    H, W = cfg["H"], cfg["W"]
    rng = np.random.RandomState(11)
    depth_in = dmb.read_dmb(os.path.join(apd, "TSAR_disp.dmb")).astype(np.float32)
    depth_in[depth_in <= 0] = 1.0
    normal_in = dmb.read_dmb(os.path.join(apd, "TSAR_normals.dmb")).astype(np.float32)
    dmb.write_dmb(os.path.join(apd, "depths_geom.dmb"), depth_in)
    dmb.write_dmb(os.path.join(apd, "normals.dmb"), normal_in)
    colours = np.array([[255, 255, 255], [0, 255, 0], [0, 0, 255], [0, 0, 0], [255, 0, 0], [254, 255, 255]], np.uint8)   # BGR
    # 20 % reliable pixels: the facet's region stays below the 50 000 points beyond which the reference cuts the list to a
    # clock-seeded random subset (main.cpp:1541-1549), which nothing can reproduce
    weak = colours[rng.choice(len(colours), size=(H, W), p=[0.12, 0.04, 0.04, 0.5, 0.15, 0.15])]
    cv2.imwrite(os.path.join(apd, "weak.png"), weak)
    names = sorted(os.listdir(root + "images"))
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tsar_cli.py")] + names + ["-images_folder", root + "images/", "-import_apd"] + common,
                       capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "not found" not in r.stderr
    got_d = dmb.read_dmb(os.path.join(apd, "TSAR_disp.dmb"))
    got_n = dmb.read_dmb(os.path.join(apd, "TSAR_normals.dmb"))

    # the same flow from the reference's pieces
    images = [cli._imread_gray(os.path.join(root, "images", n)) for n in names]
    krt = [cli.read_cam_txt(os.path.join(root, "cams", f"{n[:8]}_cam.txt")) for n in names]
    cams = pkg.scene.cameras_from_krt([k[0] for k in krt], [k[1] for k in krt], [k[2] for k in krt], krt[0][3], krt[0][4])
    subset = [s_ for s_ in cli.read_pair_subset(os.path.join(root, "pair.txt"), 0) if s_ < len(names)]
    f = float(np.float32(cams[0]["f"]))
    params = pkg.make_params(box=11, iterations=2, n_best=1, cost_comb=1, min_disparity=float(np.float32(f / np.float32(krt[0][4]))),
                             max_disparity=float(np.float32(f / np.float32(krt[0][3]))))
    det = texture.detect(images[0].astype(np.uint8))
    text, size = det["text"], det["size"]
    weak_regions = [r_ for r_ in range(len(text)) if text[r_] == -1]
    assert weak_regions, "the detector must flag the textureless facet"
    canny = texture.expand_labels(det["labels_q"], W, H)
    ref = rb.RefEngine(pkg._lib.TsarCamera, pkg._lib.TsarParams, variant="asis")
    ref.create(images, cameras_to_struct(cams), subset, params, f)
    ref.upload(rb.F_CANNY, canny)
    ref.upload(rb.F_NORM4, np.concatenate([normal_in, np.zeros((H, W, 1), np.float32)], axis=-1))
    ref.upload(rb.F_COST, np.ones((H, W), np.float32))
    ref.upload(rb.F_DEPTH, (np.float32(f) / depth_in).astype(np.float32))
    ref.get_disp(); ref.getview()
    reliable = ((weak == [255, 255, 255]).all(-1) | (weak == [0, 255, 0]).all(-1) | (weak == [0, 0, 255]).all(-1)).astype(np.float32)
    assert 0.18 < reliable.mean() < 0.22
    assert max(int(((canny == r_) & (reliable == 1)).sum()) for r_ in weak_regions) < 50000
    ref.upload(rb.F_SCALE, reliable)
    probe = pkg.DepthmapEngine(0)
    with np.errstate(over="ignore"):
        stream = np.concatenate([probe.ransac_rand_stream(SEED, r_) for r_ in weak_regions])
    probe.close()
    p0 = np.tile(np.array([0, 0, 1, -1], np.float32), (len(text), 1))
    planes, used = rh.fit_regions(cams[0], f, ref.download(rb.F_DEPTH), reliable, canny, text, size, stream, p0)
    assert used == len(stream)
    ref.set_regions(text, planes)
    ref.update_scale_2(); ref.update_scale(); ref.compute_disp()
    want = ref.download(rb.F_NORM4)
    ref.close()
    assert pc.frac_bit_exact(got_d, want[..., 3]) == 1.0
    assert pc.frac_bit_exact(got_n, np.ascontiguousarray(want[..., :3])) == 1.0
    assert (got_d != depth_in).mean() > 0.01                      # and the completion rewrote the facet


def test_every_kernel_and_variant_in_one_process(env):
    """tools/gpu_sanitize.py drives every kernel of the library -- all window variants (11x11, 19x19, run-time windows, n_best
    2 / 3, COMB_ALL), fused and unfused launches, odd image sizes, glue, weighted-median stages, region fit (host and device
    stream), reliable-pixel sources, gSLICr modes, the host entry point -- inside ONE process, which is where per-process state
    (kernel attributes, persistent scratch, context reuse) can go wrong.  (It is also the script to put under a memory
    checker where one is available.)"""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tools", "gpu_sanitize.py")], capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    assert "SANITIZE-SCRIPT-DONE" in r.stdout


@pytest.mark.parametrize("script,args", [("gpu_cost_sweep.py", ["4", "30000"]), ("gpu_glue_sweep.py", ["8"]), ("gpu_slic_sweep.py", ["45"]),
                                         ("gpu_wmf_sweep.py", ["8"]), ("gpu_ransac_sweep.py", ["8"])])
def test_differential_sweeps(env, script, args):
    """Short runs of the differential sweeps (tools/README.md): every component against the reference's own code on random and
    adversarial inputs -- hostile planes for the cost (exact-division path, NaN / inf), NaN / inf state for the per-pixel
    kernels, piecewise-constant images for gSLICr (exact ties), sparse reliable masks for the weighted medians (dummy-element
    medians), degenerate and collinear regions for the RANSAC fit (NaN planes).  Each script exits non-zero on the first
    configuration that is not bit-exact; the long runs are recorded under profiles/r02_*_sweep.json."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(pc.ROOT, "tools", script)] + args, capture_output=True, text=True, cwd=pc.ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])


def test_plain_c_program_runs_a_depthmap(env, tmp_path):
    """examples/c_abi_check.c: a C11 program drives tsar_depthmap_host through the C ABI and recovers a known plane."""
    import subprocess
    from tests.test_cpu import _build_c_abi_check
    exe = _build_c_abi_check(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert "interior pixels" in r.stdout
