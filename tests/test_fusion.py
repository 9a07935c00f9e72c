"""Multi-view fusion (DESIGN.md section 4.6): the C restatement oc_fuse pinned on hand-built cases (CPU), and the CUDA
fusion (tsar_fusion_*) bit-exact against it on rendered rigs, the real -all_views output, adversarial maps and
production sizes (GPU).  TSAR_FUSION_SEED picks other random inputs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import fusion_binding

SEED = int(os.environ.get("TSAR_FUSION_SEED", "20261020"))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_fuse(pkg, views, **params):
    return fusion_binding.fuse(pkg._lib.TsarViewCamera, pkg.fusion.make_params(**params), views)


def flat_view(W, H, K=None, R=None, t=(0, 0, 0), depth=1.0, normal=(0, 0, 1), bgr=(10, 20, 30), neighbours=(1,)):
    """A view of an exact-arithmetic rig: K = I unless given, so a pixel's coordinates are camera x, y at depth 1."""
    return dict(K=np.eye(3) if K is None else np.asarray(K, float), R=np.eye(3) if R is None else np.asarray(R, float),
                t=np.asarray(t, float), depth=np.full((H, W), depth, np.float32),
                normals=np.tile(np.asarray(normal, np.float32), (H, W, 1)), bgr=np.tile(np.asarray(bgr, np.uint8), (H, W, 1)),
                neighbours=list(neighbours))


HALF = np.diag([0.5, 0.5, 1.0])                       # pixel x at depth 1 -> source pixel floor(x/2 + 1/2)
HALF_SHIFTED = [[0.5, 0, 0.5], [0, 0.5, 0], [0, 0, 1]]  # -> floor(x/2 + 1)


def chain_views():
    """Row of 8 pixels, S_0 = [A, D], min_consistent = 2.  A pairs pixels {0}, {1,2}, {3,4}, {5,6}, {7}; D pairs {0,1},
    {2,3}, {4,5}, {6,7}.  Pixel 0 fuses and takes D1, so pixel 1 (A1, D1) drops and pixel 2 takes A1 and fuses: a chain
    that runs through the whole row."""
    return [flat_view(8, 1, neighbours=[1, 2]), flat_view(8, 1, K=HALF, neighbours=[0]),
            flat_view(8, 1, K=HALF_SHIFTED, neighbours=[0])]


# ---- oc_fuse on hand-built cases --------------------------------------------------------------------------------
def test_masks_across_views(pkg):
    # three coincident cameras: view 0 takes every pixel of view 1; view 1 is then skipped as a reference; view 2 finds
    # view 1's pixels taken, but view 0's own pixels were never masked (the reference pixel is not masked, as in ACMM)
    views = [flat_view(4, 3, neighbours=[1]), flat_view(4, 3, neighbours=[0, 2]), flat_view(4, 3, neighbours=[1])]
    xyz, _, _ = oracle_fuse(pkg, views, min_consistent=1)
    assert len(xyz) == 12                               # view 0 only: view 1 masked, view 2's sources masked
    views[2]["neighbours"] = [0]
    xyz, _, _ = oracle_fuse(pkg, views, min_consistent=1)
    assert len(xyz) == 24                               # view 0, then view 2 on view 0's unmasked pixels
    y, x = np.mgrid[0:3, 0:4]
    px = np.stack([x, y, np.ones_like(x)], -1).reshape(-1, 3).astype(np.float32)
    assert np.array_equal(xyz, np.concatenate([px, px]))


def test_first_pixel_in_raster_order_takes_a_shared_source(pkg):
    views = [flat_view(4, 1, neighbours=[1]), flat_view(4, 1, K=HALF, neighbours=[0])]
    xyz, _, _ = oracle_fuse(pkg, views, min_consistent=1)
    # x = 1 and x = 2 both land on source pixel 1 (back at x = 2): x = 1 takes it, x = 2 is left without a source;
    # view 1's pixel 3 projects outside view 0
    assert xyz.tolist() == [[0, 0, 1], [1.5, 0, 1], [3.5, 0, 1]]


def test_chain_first_taker_drops_second_fuses(pkg):
    xyz, _, _ = oracle_fuse(pkg, chain_views(), min_consistent=2)
    assert [round(float(v), 4) for v in xyz[:, 0] * 3] == [0 + 0 + 1, 2 + 2 + 3, 4 + 4 + 5, 6 + 6 + 7]
    xyz1, _, _ = oracle_fuse(pkg, chain_views(), min_consistent=1)
    assert len(xyz1) == 8                               # with one source pixel enough, every pixel fuses


@pytest.mark.parametrize("bad", [0.0, -1.0, np.nan, np.inf])
def test_invalid_depths(pkg, bad):
    views = [flat_view(5, 1, neighbours=[1]), flat_view(5, 1, neighbours=[0])]
    views[0]["depth"][0, 1] = bad                       # as a reference pixel: skipped
    views[1]["depth"][0, 3] = bad                       # as a source pixel: no candidate
    xyz, _, _ = oracle_fuse(pkg, views, min_consistent=1)
    # view 0 fuses x = 0, 2, 4; view 1's pixel 1 finds view 0's pixel 1 invalid, pixel 3 is itself invalid
    assert xyz[:, 0].tolist() == [0, 2, 4]


def test_point_behind_the_source_camera(pkg):
    turned = np.diag([-1.0, 1.0, -1.0])                # looks the other way: camera z = -1 for every point
    views = [flat_view(3, 1, neighbours=[1]), flat_view(3, 1, R=turned, neighbours=[0])]
    # without the z > 0 test x would map to itself and pass: reprojection 0, |z' - D| = 2 < 3 * D, equal normals
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=3.0)[0]) == 0
    views[1]["R"] = np.eye(3)
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=3.0)[0]) == 3


@pytest.mark.parametrize("cx, n_points, last_x", [(-0.5, 2, 1.25), (-0.6, 1, 0.8)])
def test_border_rounding(pkg, cx, n_points, last_x):
    # pixel 0 lands at x = cx in view 1: floor(-0.5 + 0.5) = 0 is inside, floor(-0.6 + 0.5) = -1 is outside (int() would
    # truncate both to column 0)
    views = [flat_view(2, 1, neighbours=[1]), flat_view(2, 1, K=[[1, 0, cx], [0, 1, 0], [0, 0, 1]], neighbours=[0])]
    xyz, _, _ = oracle_fuse(pkg, views, min_consistent=1)
    assert len(xyz) == n_points
    # pixel 1 lands at 1 + cx: on source pixel 1 (back at 1.5) for -0.5, on source pixel 0 (back at 0.6) for -0.6
    assert xyz[-1, 0] == pytest.approx(last_x, abs=1e-6)


def test_reprojection_threshold_is_strict(pkg):
    # view 1 shifted by 2: pixel 2 -> source pixel 0, whose depth 0.5 puts it back at x = 4: error exactly 2
    views = [flat_view(3, 1, neighbours=[1]), flat_view(3, 1, t=(-2, 0, 0), depth=0.5, neighbours=[0])]
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=1.0, max_reproj_px=2.0)[0]) == 0
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=1.0, max_reproj_px=2.0001)[0]) == 1


def test_depth_threshold_is_strict(pkg):
    views = [flat_view(3, 1, neighbours=[1]), flat_view(3, 1, depth=0.75, neighbours=[0])]   # |0.75 - 1| = 0.25 * 1
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=0.25)[0]) == 0
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_rel_depth=0.2501)[0]) == 3


def _cos_threshold(deg):
    """(cos(deg) rounded to float) * |n_v| * |n_u| for n_v = (0, 0, 1), n_u = (0, 0.75, 1) (|n_u| = 1.25), in float32."""
    c = np.float32(np.cos(np.float64(np.float32(deg)) * (np.pi / 180.0)))
    return np.float32(np.float32(c * np.float32(1.0)) * np.float32(1.25))


def test_normal_threshold_is_inclusive(pkg):
    eq = np.degrees(np.arccos(0.8))                     # n_v . n_u = 1 = 0.8 * 1 * 1.25
    assert _cos_threshold(eq) == np.float32(1.0)
    tighter = np.float32(eq)
    while _cos_threshold(tighter) <= 1.0:
        tighter = np.nextafter(tighter, np.float32(0))
    views = [flat_view(3, 1, normal=(0, 0, 1), neighbours=[1]), flat_view(3, 1, normal=(0, 0.75, 1), neighbours=[0])]
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_normal_deg=float(np.float32(eq)))[0]) == 3
    assert len(oracle_fuse(pkg, views, min_consistent=1, max_normal_deg=float(tighter))[0]) == 0


def test_summation_order(pkg):
    rng = np.random.RandomState(SEED)
    W = 64
    views = [flat_view(W, 1, neighbours=[1, 2]), flat_view(W, 1, neighbours=[0, 2]), flat_view(W, 1, neighbours=[0, 1])]
    for v in views:
        v["depth"][:] = rng.uniform(0.8, 1.2, (1, W)).astype(np.float32)
        n = np.concatenate([rng.uniform(-0.3, 0.3, (1, W, 2)), np.ones((1, W, 1))], -1)
        v["normals"][:] = (n * rng.uniform(0.5, 3.0, (1, W, 1))).astype(np.float32)
        v["bgr"][:] = rng.randint(0, 256, (1, W, 3)).astype(np.uint8)
    xyz, nrm, rgb = oracle_fuse(pkg, views, min_consistent=2, max_rel_depth=1.0, max_normal_deg=60.0)
    assert len(xyz) == W                                # every pixel of view 0 takes both sources
    f = np.float32
    x = np.arange(W, dtype=f)
    X = [np.stack([v["depth"][0] * x, np.zeros(W, f), v["depth"][0]], -1) for v in views]
    want = ((X[0] + X[1]) + X[2]) / f(3)
    assert np.array_equal(xyz, want)
    assert not np.array_equal(((X[2] + X[1]) + X[0]) / f(3), want)
    ns = (views[0]["normals"][0] + views[1]["normals"][0]) + views[2]["normals"][0]
    length = np.sqrt((ns[:, 0] * ns[:, 0] + ns[:, 1] * ns[:, 1]) + ns[:, 2] * ns[:, 2])
    assert np.array_equal(nrm, ns / length[:, None])
    col = sum(v["bgr"][0].astype(np.int64) for v in views)[:, ::-1]
    assert np.array_equal(rgb, ((2 * col + 3) // 6).astype(np.uint8))
    assert np.array_equal(rgb, np.floor(col / 3.0 + 0.5).astype(np.uint8))


def test_fused_ply_round_trip(pkg, tmp_path):
    rng = np.random.RandomState(SEED)
    xyz, nrm = rng.randn(100, 3).astype(np.float32), rng.randn(100, 3).astype(np.float32)
    rgb = rng.randint(0, 256, (100, 3)).astype(np.uint8)
    path = str(tmp_path / "TSAR_fused.ply")
    pkg.dmb.write_fused_ply(path, xyz, nrm, rgb)
    p, n, c = pkg.dmb.read_model_ply(path)
    assert np.array_equal(p, xyz) and np.array_equal(n, nrm) and np.array_equal(c, rgb)
    pkg.dmb.write_fused_ply(path, xyz[:0], nrm[:0], rgb[:0])
    assert len(pkg.dmb.read_model_ply(path)[0]) == 0


def test_fuse_flag_is_boolean(pkg):
    opt = pkg.cli.parse_args(["-fuse", "-mslp_folder", "data/", "-all_views"])
    assert opt["fuse"] is True and opt["all_views"] is True and opt["mslp_folder"] == "data/" and opt["images"] == []
    assert pkg.cli.parse_args(["-mslp_folder", "data/"])["fuse"] is False


def test_fuse_names_missing_views(pkg, tmp_path):
    import cv2
    root = str(tmp_path) + "/"
    os.makedirs(root + "images")
    for i in range(3):
        cv2.imwrite(root + f"images/{i:08d}.png", np.zeros((4, 4, 3), np.uint8))
    os.makedirs(root + "APD/00000001")
    pkg.dmb.write_dmb(root + "APD/00000001/TSAR_disp.dmb", np.ones((4, 4), np.float32))
    with pytest.raises(FileNotFoundError, match="00000000, 00000001, 00000002"):
        pkg.cli.read_fusion_views(pkg.cli.parse_args(["-fuse", "-mslp_folder", root]), root)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tsar_cli.py"), "-fuse", "-mslp_folder", root],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode != 0 and "00000000, 00000001, 00000002" in r.stderr


def test_fuse_reports_bad_datasets(pkg, tmp_path):
    import cv2
    root = str(tmp_path) + "/"
    os.makedirs(root + "images")
    cli = [sys.executable, os.path.join(ROOT, "tsar_cli.py"), "-fuse", "-mslp_folder", root]
    r = subprocess.run(cli, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 1 and "no images" in r.stderr and "Traceback" not in r.stderr
    n = 34
    for i in range(n):
        cv2.imwrite(root + f"images/{i:08d}.png", np.zeros((4, 4, 3), np.uint8))
        os.makedirs(root + f"APD/{i:08d}")
        pkg.dmb.write_dmb(root + f"APD/{i:08d}/TSAR_disp.dmb", np.ones((4, 4), np.float32))
        pkg.dmb.write_dmb(root + f"APD/{i:08d}/TSAR_normals.dmb", np.ones((4, 4, 3), np.float32))
    # view 0: 33 neighbours; view 1: only a camera that is not in the dataset; the others: view 0
    pkg.cli.write_pair_txt(root + "pair.txt", [list(range(1, n)), [n + 5]] + [[0]] * (n - 2))
    r = subprocess.run(cli, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 1 and "view(s) 00000000 (33), 00000001 (0) " in r.stderr and "Traceback" not in r.stderr


def test_fuse_refuses_several_ranks(pkg, tmp_path):
    env = dict(os.environ, WORLD_SIZE="2", RANK="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tsar_cli.py"), "-all_views", "-fuse", "-mslp_folder", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, env=env)
    assert r.returncode != 0 and "single process" in r.stderr


# ---- the CUDA fusion against oc_fuse --------------------------------------------------------------------------------
def assert_same_points(got, want):
    assert len(got[0]) == len(want[0]), (len(got[0]), len(want[0]))
    for g, w in zip(got, want):
        assert g.tobytes() == w.tobytes()


def gpu_vs_oracle(pkg, views, **params):
    got = pkg.fusion.fuse(views, params)
    want = oracle_fuse(pkg, views, **params)
    assert_same_points(got, want)
    return got


def rig_views(pkg, cfg, noise=0.0, seed=SEED, quarter=(), backend="numpy", device=None):
    """Views of a scene.make_rig rig with ground-truth depth (times 1 + noise * N(0, 1)) and the facets' world normals;
    views listed in `quarter` get K / 4 (sixteen pixels of a full-K view compete for each of their pixels)."""
    sc_mod = pkg.scene
    K, Rs, Cs, neighbours = sc_mod.make_rig(cfg)
    sc = sc_mod.Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"], seed=1234)
    normals = np.array([f["n"] for f in sc.facets], np.float32)
    rng = np.random.RandomState(seed)
    views = []
    for i, (R, C) in enumerate(zip(Rs, Cs)):
        Ki = K.copy()
        if i in quarter:
            Ki[:2] /= 4.0
        cam = dict(K_inv=np.linalg.inv(Ki), _R_world=R, _C_world=C)
        if backend == "torch":
            img, depth, label = (a.cpu().numpy() for a in sc.render_torch(cam, cfg["W"], cfg["H"], device))
        else:
            img, depth, label = sc.render(cam, cfg["W"], cfg["H"])
        depth = depth.astype(np.float32)
        if noise:
            depth = (depth * (1.0 + noise * rng.randn(*depth.shape))).astype(np.float32)
        img = img.astype(np.uint8)
        bgr = np.stack([img, np.roll(img, 3, axis=1), np.roll(img, 5, axis=0)], -1)
        views.append(dict(K=Ki, R=R, t=-R @ C, depth=depth, normals=normals[label], bgr=bgr, neighbours=neighbours[i]))
    return views, sc


def facet_distance(sc, X):
    """Distance of world points to the nearest facet plane of the scene."""
    X = np.asarray(X, np.float64)
    return np.min([np.abs((X - f["p0"]) @ f["n"]) for f in sc.facets], axis=0)


@pytest.mark.gpu
def test_gpu_rig_ground_truth(pkg):
    cfg = pkg.scene.CONFIGS["C3small"]
    views, sc = rig_views(pkg, cfg)
    xyz, nrm, rgb = gpu_vs_oracle(pkg, views)
    assert len(xyz) > cfg["W"] * cfg["H"]
    Cs = np.array([-v["R"].T @ v["t"] for v in views])
    cam_dist = np.min(np.linalg.norm(xyz[:, None, :].astype(np.float64) - Cs[None], axis=-1), axis=1)
    assert (facet_distance(sc, xyz) <= 1e-4 * cam_dist).all()


@pytest.mark.gpu
def test_gpu_fused_cloud_no_less_accurate_than_its_inputs(pkg):
    views, sc = rig_views(pkg, pkg.scene.CONFIGS["C3small"], noise=1e-3)
    xyz, _, _ = gpu_vs_oracle(pkg, views)
    per_view = []
    for v in views:
        H, W = v["depth"].shape
        y, x = np.mgrid[0:H, 0:W]
        ray = np.stack([x, y, np.ones_like(x)], -1).reshape(-1, 3) @ np.linalg.inv(v["K"]).T
        per_view.append(((v["depth"].reshape(-1, 1) * ray) - v["t"]) @ v["R"])
    d_in = np.median(facet_distance(sc, np.concatenate(per_view)))
    d_out = np.median(facet_distance(sc, xyz))
    print(f"[fusion] median facet distance: per-view maps {d_in:.3e}, fused cloud {d_out:.3e} ({len(xyz)} points)")
    assert d_out <= d_in


@pytest.mark.gpu
def test_gpu_all_views_then_fuse(pkg, tmp_path):
    root = str(tmp_path / "c3small") + "/"
    cli = [sys.executable, os.path.join(ROOT, "tsar_cli.py")]
    r = subprocess.run(cli + ["--synthetic=C3small", "-mslp_folder", root, "-all_views", "-fuse", "--iterations=2"],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    ply = os.path.join(root, "TSAR_fused.ply")
    first = open(ply, "rb").read()
    views = pkg.cli.read_fusion_views(pkg.cli.parse_args(["-fuse", "-mslp_folder", root]), root)
    xyz, nrm, rgb = gpu_vs_oracle(pkg, views)
    assert len(xyz) > 0
    pkg.dmb.write_fused_ply(str(tmp_path / "api.ply"), xyz, nrm, rgb)
    assert open(str(tmp_path / "api.ply"), "rb").read() == first
    os.remove(ply)
    r = subprocess.run(cli + ["-fuse", "-mslp_folder", root], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert open(ply, "rb").read() == first             # a separate -fuse over the same files, and a second run


@pytest.mark.gpu
@pytest.mark.parametrize("min_consistent", [1, 2, 3])
def test_gpu_adversarial_maps(pkg, min_consistent):
    rng = np.random.RandomState(SEED + min_consistent)
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], quarter=(1,))
    for k, v in enumerate(views):
        H, W = v["depth"].shape
        d = v["depth"]
        if k % 2:                                       # noise maps on half of the views
            d *= rng.uniform(0.97, 1.03, d.shape).astype(np.float32)
            v["normals"] = (v["normals"] + rng.normal(0, 0.1, v["normals"].shape)).astype(np.float32)
        bad = rng.rand(H, W) < 0.05
        d[bad] = rng.choice(np.array([0.0, -1.0, np.nan, np.inf, -0.0], np.float32), bad.sum())
        v["normals"][rng.rand(H, W) < 0.01] = np.nan
        v["bgr"] = rng.randint(0, 256, v["bgr"].shape).astype(np.uint8)
    gpu_vs_oracle(pkg, views, min_consistent=min_consistent, max_rel_depth=0.02)


@pytest.mark.gpu
def test_gpu_quarter_k_neighbour(pkg):
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], quarter=(1,))
    for v in views:
        if 1 in v["neighbours"]:
            v["neighbours"] = [1] + [k for k in v["neighbours"] if k != 1]
    xyz, _, _ = gpu_vs_oracle(pkg, views, min_consistent=1, max_reproj_px=8.0, max_rel_depth=0.05)
    assert len(xyz) > 0


@pytest.mark.gpu
def test_gpu_chain_takes_several_rounds(pkg):
    views = chain_views()
    with pkg.fusion.FusionEngine(3, 8, 1) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], v["neighbours"])
        got = eng.run(dict(min_consistent=2))
        assert eng.rounds()[0] > 1
    assert_same_points(got, oracle_fuse(pkg, views, min_consistent=2))
    assert len(got[0]) == 4


@pytest.mark.gpu
@pytest.mark.parametrize("n_neighbours", [1, 32])
def test_gpu_neighbour_list_lengths(pkg, n_neighbours):
    cfg = dict(W=96, H=64, n_images=33, V=n_neighbours, fx=180.0, radius=1.0, arc_deg=30.0, rig="two_arcs")
    views, _ = rig_views(pkg, cfg, noise=2e-3)
    assert all(len(v["neighbours"]) == n_neighbours for v in views)
    for mc in (1, 2):
        gpu_vs_oracle(pkg, views, min_consistent=mc, max_reproj_px=1.5)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(12, 1920, 1080, 4), (4, 3100, 2050, 3)])
def test_gpu_production_sizes(pkg, shape):
    n, W, H, V = shape
    cfg = dict(W=W, H=H, n_images=n, V=V, fx=1160.0 if W == 1920 else 1750.0, radius=4.0, arc_deg=20.0, rig="sequence")
    views, _ = rig_views(pkg, cfg, noise=2e-3, backend="torch", device="cuda:0")
    xyz, _, _ = gpu_vs_oracle(pkg, views)
    assert len(xyz) > W * H // 2


@pytest.mark.gpu
def test_gpu_second_run_other_parameters(pkg):
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], noise=2e-3)
    H, W = views[0]["depth"].shape
    with pkg.fusion.FusionEngine(len(views), W, H) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], v["neighbours"])
        first = eng.run()
        second = eng.run(dict(max_reproj_px=1.0, max_rel_depth=0.003, max_normal_deg=5.0, min_consistent=3))
        again = eng.run()
    assert_same_points(first, oracle_fuse(pkg, views))
    assert_same_points(second, oracle_fuse(pkg, views, max_reproj_px=1.0, max_rel_depth=0.003, max_normal_deg=5.0, min_consistent=3))
    assert_same_points(again, first)
    assert len(second[0]) < len(first[0])


@pytest.mark.gpu
def test_gpu_rejects_bad_arguments(pkg):
    v = flat_view(4, 1, neighbours=[1])
    with pkg.fusion.FusionEngine(3, 4, 1) as eng:
        for nb in ([], [0], [1, 1], [3], list(range(33))):
            with pytest.raises(pkg.TsarError):
                eng.set_view(0, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], nb)
        eng.set_view(0, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], [1])
        with pytest.raises(pkg.TsarError, match="not set"):
            eng.run()
        for k in (1, 2):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], [0])
        import ctypes as C
        n = C.c_longlong()
        assert eng.lib.tsar_fusion_run(eng.h, C.byref(pkg.fusion.make_params(min_consistent=1)), C.byref(n)) == 0
        assert n.value == 8                             # view 0 takes view 1's pixels; view 2 fuses with view 0's
        buf = np.empty((4, 3), np.float32)
        assert eng.lib.tsar_fusion_points(eng.h, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, 3) == -1
