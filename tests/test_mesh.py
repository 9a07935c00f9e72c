"""Mesh extraction (DESIGN.md section 4.8): the C restatement oc_mesh pinned on hand-built exact rigs and its
tetrahedron rule checked by the topology of analytic fields (CPU); the CUDA mesh (tsar_mesh_*) byte for byte against it
on rendered rigs, the real -all_views output, adversarial maps and production sizes, plus geometry and memory (GPU).
TSAR_MESH_SEED picks other random inputs."""
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

from oracle import mesh_binding
from tests.test_device_memory import interposer, run_scenario  # noqa: F401  (fixture)
from tests.test_fusion import rig_views

SEED = int(os.environ.get("TSAR_MESH_SEED", "20261022"))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = [sys.executable, os.path.join(ROOT, "tsar_cli.py")]


# ---- exact rigs ---------------------------------------------------------------------------------------------------
def plane_view(depth=2.0, bgr=(10, 20, 30), R=None, W=64, H=64):
    """A camera at the origin looking along +z (K: f = 8, centre 32) at a fronto-parallel plane z = depth."""
    return dict(K=np.array([[8.0, 0, 32.0], [0, 8.0, 32.0], [0, 0, 1]]), R=np.eye(3) if R is None else np.asarray(R, float),
                t=np.zeros(3), depth=np.full((H, W), depth, np.float32), bgr=np.tile(np.asarray(bgr, np.uint8), (H, W, 1)))


def column_grid(z0, nz=3, n=3, s=0.25):
    """n x n x nz points at x, y in {-0.25, 0, 0.25} (n = 3) and z = z0, z0 + s, ..."""
    return dict(origin=(-0.375, -0.375, z0 - 0.5 * s), voxel=s, dims=(n, n, nz))


def field(views, grid, trunc):
    return mesh_binding.field(views, grid, trunc)


def test_trunc_boundary_integrates(pkg):
    # plane at 2: layers z = 2.25, 2.5, 2.75 have sdf = -0.25, -0.5 (= -trunc: integrates, d = -1), -0.75 (skipped)
    F, W, Wc, S = field([plane_view()], column_grid(2.25), 0.5)
    assert W[:, 1, 1].tolist() == [1, 1, 0]
    assert F[:, 1, 1].tolist() == [-0.5, -1.0, 0.0]
    # sdf = +trunc still adds colour, above it only weight: z = 1.5 (sdf 0.5) and 1.25 (sdf 0.75, d = min(1, 1.5))
    F, W, Wc, S = field([plane_view()], column_grid(1.25, nz=2), 0.5)
    assert W[:, 1, 1].tolist() == [1, 1] and Wc[:, 1, 1].tolist() == [0, 1] and F[:, 1, 1].tolist() == [1.0, 1.0]
    assert S[1, 1, 1].tolist() == [10, 20, 30] and S[0, 1, 1].tolist() == [0, 0, 0]


def test_zero_is_outside_and_vertex_order(pkg):
    # layers z = 1.75, 2, 2.25 at a plane z = 2: F = 0.5, 0, -0.5.  F = 0 is outside, so the surface crosses between the
    # layers 2 and 2.25 only, at t = 0 / (0 - (-0.5)) = 0: every vertex sits on its owner in layer 2, four per owner
    # (delta 001, 101, 011, 111 where they stay in the grid), in lattice order
    grid = column_grid(1.75)
    xyz, rgb, tri = mesh_binding.mesh([plane_view()], grid, 0.5, 1)
    want, vid = [], {}
    for j in range(3):
        for i in range(3):
            for d in ((0, 0, 1), (1, 0, 1), (0, 1, 1), (1, 1, 1)):
                if i + d[0] < 3 and j + d[1] < 3:
                    vid[i, j, d] = len(want)
                    want.append([-0.25 + 0.25 * i, -0.25 + 0.25 * j, 2.0])
    assert xyz.tolist() == want
    assert rgb.tolist() == [[30, 20, 10]] * len(want)
    # each of the 4 cells between the layers 2 and 2.25 gives its tetrahedra xyz .. zyx 1, 2, 1, 2, 1, 1 triangles
    assert len(tri) == 4 * 8 and sorted(np.unique(tri).tolist()) == list(range(len(want)))
    # first cell: tetrahedron xyz (000, 100, 110, 111; only 111 inside) gives (E30, E32, E31); xzy (000, 100, 101, 111,
    # odd; 101 and 111 inside) gives (E20, E21, E31), (E20, E31, E30) with the last two vertices swapped
    e30, e32, e31 = vid[0, 0, (1, 1, 1)], vid[1, 1, (0, 0, 1)], vid[1, 0, (0, 1, 1)]
    e20, e21 = vid[0, 0, (1, 0, 1)], vid[1, 0, (0, 0, 1)]
    assert tri[:3].tolist() == [[e30, e32, e31], [e20, e31, e21], [e20, e30, e31]]
    # inside is z > 2, the camera side z < 2: normals point to -z (some triangles are degenerate: t = 0 everywhere)
    P = xyz[tri].astype(np.float64)
    n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    assert (n[:, 2] <= 0).all() and (n[:, 2] < 0).any()


def test_min_weight_gating_and_no_orphans(pkg):
    # a second view has no depth left of column 32: grid points at x = -0.5, -0.25 project to columns <= 31 from every
    # layer, those at x = 0, 0.25 to columns >= 32
    v1 = plane_view()
    v1["depth"][:, :32] = 0.0
    grid = dict(origin=(-0.625, -0.375, 1.625), voxel=0.25, dims=(4, 3, 3))
    F, W, _, _ = field([plane_view(), v1], grid, 0.5)
    assert W[:, :, :2].max() == 1 and W[:, :, 2:].min() == 2
    xyz1, _, tri1 = mesh_binding.mesh([plane_view(), v1], grid, 0.5, 1)
    xyz2, _, tri2 = mesh_binding.mesh([plane_view(), v1], grid, 0.5, 2)
    assert len(xyz2) < len(xyz1) and len(tri2) < len(tri1)
    assert (xyz2[:, 0] >= 0).all() and (xyz1[:, 0] < 0).any()   # cells with a corner at x < 0 are incomplete
    for xyz, tri in ((xyz1, tri1), (xyz2, tri2)):
        assert sorted(np.unique(tri).tolist()) == list(range(len(xyz)))
    assert len(mesh_binding.mesh([plane_view(), v1], grid, 0.5, 3)[0]) == 0


def test_colour_rounding_preference_and_ties(pkg):
    # two views of colour B = 10 and 11: mean 10.5 rounds half up to 11
    xyz, rgb, _ = mesh_binding.mesh([plane_view(bgr=(10, 20, 30)), plane_view(bgr=(11, 21, 31))], column_grid(1.75), 0.5, 1)
    assert rgb.tolist() == [[31, 21, 11]] * len(xyz)
    # hand-built field on 2 x 2 x 2 points: the lower layer inside (F = -0.5, colour A), the upper one outside
    grid = dict(origin=(0, 0, 0), voxel=1.0, dims=(2, 2, 2))
    A, B = [100, 0, 0], [0, 0, 200]

    def run(Fb, Wcb):
        F = np.array([-0.5] * 4 + [Fb] * 4, np.float32)
        W = np.full(8, 3, np.uint16)
        Wc = np.array([1] * 4 + [Wcb] * 4, np.uint16)
        S = np.array([A] * 4 + [[c * max(Wcb, 1) for c in B]] * 4, np.uint32)
        return mesh_binding.extract(grid, 1, F, W, Wc, S)[1]
    assert (run(0.25, 1) == [200, 0, 0]).all()         # |Fb| < |Fa|: colour of b
    assert (run(0.5, 1) == [0, 0, 100]).all()          # tie: colour of a
    assert (run(0.75, 1) == [0, 0, 100]).all()
    assert (run(0.25, 0) == [0, 0, 100]).all()         # b has no colour: a


def test_behind_the_camera_and_outside_the_image(pkg):
    turned = np.diag([-1.0, 1.0, -1.0])               # looks along -z: every grid point has z < 0
    F, W, _, _ = field([plane_view(R=turned)], column_grid(1.75), 0.5)
    assert W.max() == 0
    far = dict(origin=(100.0, 0, 1.875), voxel=0.25, dims=(2, 2, 2))   # px = 8 * 100 / 2 + 32, far right of the image
    assert field([plane_view()], far, 0.5)[1].max() == 0


@pytest.mark.parametrize("bad", [np.nan, 0.0, -1.0, np.inf])
def test_invalid_depths(pkg, bad):
    v = plane_view()
    v["depth"][:] = bad
    assert field([v, plane_view()], column_grid(1.75), 0.5)[1].max() == 1   # only the second view counts


# ---- topology of the tetrahedron rule on analytic fields -----------------------------------------------------------
def sign_field(values, weight=None):
    F = np.asarray(values, np.float32)
    W = np.full(F.shape, 4, np.uint16) if weight is None else np.asarray(weight, np.uint16)
    Wc = np.full(F.shape, 2, np.uint16)
    S = np.stack([np.full(F.shape, v, np.uint32) for v in (20, 40, 60)], -1)
    return F, W, Wc, S


def lattice(n):
    z, y, x = np.mgrid[0:n, 0:n, 0:n] + 0.5
    return x, y, z


def sphere_field(n=24, r=7.3):
    x, y, z = lattice(n)
    c = n / 2
    return dict(origin=(0, 0, 0), voxel=1.0, dims=(n, n, n)), sign_field(np.sqrt((x - c) ** 2 + (y - c) ** 2 + (z - c) ** 2) - r)


def torus_field(n=24, R=7.0, r=2.5):
    x, y, z = lattice(n)
    c = n / 2
    return dict(origin=(0, 0, 0), voxel=1.0, dims=(n, n, n)), sign_field(np.sqrt((np.sqrt((x - c) ** 2 + (y - c) ** 2) - R) ** 2 + (z - c) ** 2) - r)


def random_field(seed, shape=(10, 11, 13), undefined=0.0):
    rng = np.random.RandomState(seed)
    F = rng.randn(*shape).astype(np.float32)
    W = np.where(rng.rand(*shape) < undefined, 0, 4)
    return dict(origin=(0.5, -1.0, 2.0), voxel=0.5, dims=shape[::-1]), sign_field(F, W)


def edge_counts(tri):
    e = np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]]).tolist()
    return Counter(map(tuple, e)), Counter(tuple(sorted(k)) for k in e)


def assert_oriented_manifold(tri, n_vertices, closed=True):
    directed, undirected = edge_counts(tri)
    assert all(c == 1 for c in directed.values()), "an edge is used twice in the same direction"
    if closed:
        assert all(c == 2 for c in undirected.values())
        assert all((b, a) in directed for (a, b) in directed)
    else:
        assert all(c <= 2 for c in undirected.values())
    assert sorted(np.unique(tri).tolist()) == list(range(n_vertices)), "orphan vertex"
    return n_vertices - len(undirected) + len(tri)


def test_sphere_is_closed_oriented_and_faces_outwards(pkg):
    grid, f = sphere_field()
    xyz, _, tri = mesh_binding.extract(grid, 1, *f)
    assert assert_oriented_manifold(tri, len(xyz)) == 2
    P = xyz[tri].astype(np.float64)
    n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    assert ((n * (P.mean(1) - 12.0)).sum(-1) > 0).all()


def test_torus_has_euler_characteristic_zero(pkg):
    grid, f = torus_field()
    xyz, _, tri = mesh_binding.extract(grid, 1, *f)
    assert assert_oriented_manifold(tri, len(xyz)) == 0


@pytest.mark.parametrize("k", range(4))
def test_random_sign_fields_are_oriented_manifolds(pkg, k):
    grid, (F, W, Wc, S) = random_field(SEED + k, undefined=0.1 * k)
    xyz, _, tri = mesh_binding.extract(grid, 1, F, W, Wc, S)
    assert len(tri) > 0
    # a border of outside points closes the surface when every point is defined
    closed = k == 0
    if closed:
        F[0], F[-1], F[:, 0], F[:, -1], F[:, :, 0], F[:, :, -1] = 1, 1, 1, 1, 1, 1
        xyz, _, tri = mesh_binding.extract(grid, 1, F, W, Wc, S)
    assert_oriented_manifold(tri, len(xyz), closed=closed)


# ---- files, grid and command line -----------------------------------------------------------------------------------
def test_mesh_ply_round_trip(pkg, tmp_path):
    rng = np.random.RandomState(SEED)
    xyz = rng.randn(50, 3).astype(np.float32)
    rgb = rng.randint(0, 256, (50, 3)).astype(np.uint8)
    tri = rng.randint(0, 50, (80, 3)).astype(np.int32)
    path = str(tmp_path / "TSAR_mesh.ply")
    pkg.dmb.write_mesh_ply(path, xyz, rgb, tri)
    p, c, t = pkg.dmb.read_mesh_ply(path)
    assert np.array_equal(p, xyz) and np.array_equal(c, rgb) and np.array_equal(t, tri)
    assert np.array_equal(pkg.dmb.read_ply_points(path), xyz)
    head = open(path, "rb").read(400)
    assert b"element face 80\nproperty list uchar int vertex_indices\nend_header\n" in head
    assert os.path.getsize(path) == len(head.split(b"end_header\n")[0]) + len(b"end_header\n") + 50 * 15 + 80 * 13
    pkg.dmb.write_mesh_ply(path, xyz[:0], rgb[:0], tri[:0])
    assert all(len(a) == 0 for a in pkg.dmb.read_mesh_ply(path))


def test_default_grid_is_deterministic(pkg):
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"])
    g1, g2 = pkg.mesh.default_grid(views), pkg.mesh.default_grid(views)
    assert g1 == g2
    ratios = np.concatenate([pkg.mesh.depth_samples(v)[1] for v in views])
    assert g1["voxel"] == float(np.float32(2 * np.median(ratios)))
    g3 = pkg.mesh.default_grid(views, voxel=0.01)
    assert g3["voxel"] == float(np.float32(0.01)) and all(a < b for a, b in zip(g3["dims"], g1["dims"]))
    with pytest.raises(ValueError, match="voxels .* -mesh_voxel .* -mesh_bbox"):
        pkg.mesh.default_grid(views, voxel=1e-5)


def test_mesh_flags(pkg):
    opt = pkg.cli.parse_args(["-mesh", "-mesh_voxel", "0.01", "-mesh_bbox", "0,0,0,1,1,1", "-mesh_trunc", "0.04",
                              "-mesh_min_weight", "2", "-mslp_folder", "d/"])
    assert opt["mesh"] is True and opt["mslp_folder"] == "d/"
    voxel, box, trunc, mw = pkg.cli.parse_mesh_options(opt)
    assert voxel == 0.01 and box == ([0, 0, 0], [1, 1, 1]) and trunc == 0.04 and mw == 2
    assert pkg.cli.parse_mesh_options(pkg.cli.parse_args([])) == (None, None, None, 3)


def write_small_dataset(pkg, root, n=3, W=16, H=12, with_maps=True):
    import cv2
    os.makedirs(root + "images")
    os.makedirs(root + "cams")
    for i in range(n):
        cv2.imwrite(root + f"images/{i:08d}.png", np.full((H, W, 3), 50 * i, np.uint8))
        pkg.cli.write_cam_txt(root + f"cams/{i:08d}_cam.txt", [[10.0, 0, W / 2], [0, 10.0, H / 2], [0, 0, 1]], np.eye(3),
                              [0.1 * i, 0, 0], 0.5, 2.0)
        if with_maps:
            os.makedirs(root + f"APD/{i:08d}")
            pkg.dmb.write_dmb(root + f"APD/{i:08d}/TSAR_disp.dmb", np.ones((H, W), np.float32))


def test_mesh_grid_placement(pkg, monkeypatch):
    rng = np.random.RandomState(SEED)
    points = rng.uniform(-1, 1, (5000, 3))
    ratios = np.full(5000, 0.01)
    lo = np.quantile(points, 0.001, axis=0, method="lower")
    g = pkg.cli.mesh_grid(points, ratios, None, None, None)          # default: widened by 4 voxels = the default trunc
    assert g["voxel"] == float(np.float32(0.02)) and g["origin"] == [float(np.float32(v)) for v in lo - 4 * g["voxel"]]
    g = pkg.cli.mesh_grid(points, ratios, None, None, 0.3)           # -mesh_trunc widens the box by trunc
    assert g["origin"] == [float(np.float32(v)) for v in lo - 0.3]
    # a -mesh_bbox grid at the default voxel does not depend on the default box, even when that box is too large
    monkeypatch.setattr(pkg.mesh, "MAX_POINTS", 1000)
    with pytest.raises(ValueError, match="voxels"):
        pkg.cli.mesh_grid(points, ratios, None, None, None)
    g = pkg.cli.mesh_grid(points, ratios, None, ([0, 0, 0], [0.09, 0.09, 0.09]), None)
    assert g == dict(origin=[0.0, 0.0, 0.0], voxel=float(np.float32(0.02)), dims=[5, 5, 5])


def write_wide_dataset(pkg, root, n=3, W=64, H=48):
    """A plane at depth 1 whose depth samples (every 8th pixel) include four at depth 1e5: the box of what the views see
    has far more than 2^31 - 1 points at the default voxel (2 x median(D / f_x) = 0.2)."""
    import cv2
    os.makedirs(root + "images")
    os.makedirs(root + "cams")
    for i in range(n):
        cv2.imwrite(root + f"images/{i:08d}.png", np.full((H, W, 3), 60 + 40 * i, np.uint8))
        pkg.cli.write_cam_txt(root + f"cams/{i:08d}_cam.txt", [[10.0, 0, W / 2], [0, 10.0, H / 2], [0, 0, 1]], np.eye(3),
                              [0.01 * i, 0, 0], 0.5, 2.0)
        depth = np.ones((H, W), np.float32)
        depth[0, 0] = depth[8, 0] = depth[40, 56] = depth[32, 56] = 1e5
        os.makedirs(root + f"APD/{i:08d}")
        pkg.dmb.write_dmb(root + f"APD/{i:08d}/TSAR_disp.dmb", depth)


def test_mesh_bbox_without_voxel_ignores_the_default_box(pkg, tmp_path):
    root = str(tmp_path) + "/"
    write_wide_dataset(pkg, root)
    one_line_error(mesh_cli(root), "-mesh_voxel or a smaller -mesh_bbox")
    r = mesh_cli(root, "-mesh_bbox", "-0.5,-0.5,0.5,0.5,0.5,1.5")
    assert "voxels" not in r.stderr and "Traceback" not in r.stderr, r.stderr
    # without a GPU the command stops at the device; with one it writes the mesh (test_gpu_mesh_bbox_without_voxel)
    assert r.returncode == 0 or "tsar_mesh_create" in r.stderr, r.stderr


@pytest.mark.gpu
def test_gpu_mesh_bbox_without_voxel(pkg, tmp_path):
    root = str(tmp_path) + "/"
    write_wide_dataset(pkg, root)
    r = mesh_cli(root, "-mesh_bbox", "-0.5,-0.5,0.5,0.5,0.5,1.5")
    assert r.returncode == 0, r.stderr
    xyz, _, tri = pkg.dmb.read_mesh_ply(root + "TSAR_mesh.ply")
    assert len(tri) > 0 and np.allclose(xyz[:, 2], 1.0, atol=0.2)


def mesh_cli(root, *extra, env=None):
    return subprocess.run(CLI + ["-mesh", "-mslp_folder", root, *extra], capture_output=True, text=True, cwd=ROOT, env=env)


def one_line_error(r, needle):
    assert r.returncode == 1, (r.returncode, r.stderr)
    assert needle in r.stderr and "Traceback" not in r.stderr and len(r.stderr.strip().splitlines()) == 1, r.stderr


def test_mesh_names_missing_views(pkg, tmp_path):
    root = str(tmp_path) + "/"
    write_small_dataset(pkg, root, n=3, with_maps=False)
    os.makedirs(root + "APD/00000001")
    pkg.dmb.write_dmb(root + "APD/00000001/TSAR_disp.dmb", np.ones((12, 16), np.float32))
    one_line_error(mesh_cli(root), "view(s) 00000000, 00000002:")


def test_mesh_reports_bad_datasets_and_options(pkg, tmp_path):
    empty = str(tmp_path / "empty") + "/"
    os.makedirs(empty + "images")
    one_line_error(mesh_cli(empty), "no images")
    root = str(tmp_path / "d") + "/"
    write_small_dataset(pkg, root)
    for opts, needle in ((["-mesh_bbox", "0,0,0,1,1"], "-mesh_bbox: bad box"),
                         (["-mesh_bbox", "0,0,1,1,1,0"], "-mesh_bbox: bad box"),
                         (["-mesh_bbox", "0,0,0,1,nan,1"], "-mesh_bbox: bad box"),
                         (["-mesh_voxel", "0"], "-mesh_voxel: bad value"),
                         (["-mesh_voxel", "-1"], "-mesh_voxel: bad value"),
                         (["-mesh_voxel", "abc"], "-mesh_voxel: bad value"),
                         (["-mesh_trunc", "inf"], "-mesh_trunc: bad value"),
                         (["-mesh_min_weight", "0"], "-mesh_min_weight: bad value"),
                         (["-mesh_voxel", "1e-6", "-mesh_bbox", "0,0,0,1,1,1"], "-mesh_voxel or a smaller -mesh_bbox")):
        one_line_error(mesh_cli(root, *opts), needle)


def test_mesh_refuses_several_ranks(pkg, tmp_path):
    env = dict(os.environ, WORLD_SIZE="2", RANK="0")
    for extra in ([], ["-all_views"]):
        r = mesh_cli(str(tmp_path), *extra, env=env)
        assert r.returncode == 2 and "single process" in r.stderr


# ---- the CUDA mesh against oc_mesh ----------------------------------------------------------------------------------
def assert_same_mesh(got, want):
    assert [len(a) for a in got] == [len(a) for a in want], ([len(a) for a in got], [len(a) for a in want])
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and g.tobytes() == w.tobytes()


def gpu_vs_oracle(pkg, views, grid, trunc=None, min_weight=3):
    trunc = 4.0 * float(np.float32(grid["voxel"])) if trunc is None else trunc
    got = pkg.mesh.mesh(views, grid, trunc, min_weight)
    want = mesh_binding.mesh(views, grid, trunc, min_weight)
    assert_same_mesh(got, want)
    return got


def coarse_grid(pkg, views, factor=3.0):
    g = pkg.mesh.default_grid(views)
    return pkg.mesh.default_grid(views, voxel=g["voxel"] * factor)


def exact_rig(case):
    """(views, grid, trunc, min_weights) of the hand-built exact rigs above."""
    masked = plane_view()
    masked["depth"][:, :32] = 0.0
    gating_grid = dict(origin=(-0.625, -0.375, 1.625), voxel=0.25, dims=(4, 3, 3))
    turned = plane_view(R=np.diag([-1.0, 1.0, -1.0]))
    bad = {k: plane_view() for k in ("nan", "zero", "negative", "inf")}
    for k, v in zip(bad, (np.nan, 0.0, -1.0, np.inf)):
        bad[k]["depth"][:, ::2] = v                    # every other column: grid points on both kinds of pixel
    cases = {
        "trunc_boundary": ([plane_view()], column_grid(2.25), 0.5, [1]),      # sdf = -0.25, -0.5 (= -trunc), -0.75
        "trunc_colour": ([plane_view()], column_grid(1.25, nz=2), 0.5, [1]),  # sdf = 0.75, 0.5 (= +trunc)
        "zero_is_outside": ([plane_view()], column_grid(1.75), 0.5, [1]),      # F = 0.5, 0, -0.5
        "min_weight": ([plane_view(), masked], gating_grid, 0.5, [1, 2, 3]),
        "colour_rounding": ([plane_view(bgr=(10, 20, 30)), plane_view(bgr=(11, 21, 31)), plane_view(bgr=(11, 22, 33))],
                            column_grid(1.75), 0.5, [1, 2]),
        "behind_the_camera": ([turned, plane_view()], column_grid(1.75), 0.5, [1, 2]),
        "outside_the_image": ([plane_view()], dict(origin=(3.5, -0.375, 1.625), voxel=0.25, dims=(6, 3, 3)), 0.5, [1]),
    }
    for k, v in bad.items():
        cases["depth_" + k] = ([v, plane_view(bgr=(200, 100, 50))], dict(column_grid(1.75), dims=(9, 3, 3)), 0.5, [1, 2])
    return cases[case]


EXACT_RIGS = ["trunc_boundary", "trunc_colour", "zero_is_outside", "min_weight", "colour_rounding", "behind_the_camera",
              "outside_the_image", "depth_nan", "depth_zero", "depth_negative", "depth_inf"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EXACT_RIGS)
def test_gpu_exact_rigs(pkg, case):
    """The hand-built rigs of the CPU tests on the GPU: field and mesh byte for byte against oc_mesh, so the rule's
    boundaries (sdf = -trunc, sdf = +trunc, F = 0, min_weight, colour rounding, z <= 0, out of image, invalid depths)
    are held in the kernels, not only in the restatement."""
    views, grid, trunc, min_weights = exact_rig(case)
    want_field = mesh_binding.field(views, grid, trunc)
    with pkg.mesh.MeshEngine(len(views), 64, 64) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        for mw in min_weights:
            got = eng.run(grid, trunc, mw)
            for g, w in zip(eng.dbg_field(grid), want_field):
                assert g.tobytes() == w.tobytes()
            assert_same_mesh(got, mesh_binding.mesh(views, grid, trunc, mw))


def tie_field(seed, shape=(7, 9, 11)):
    """A field of exact values: F in {-1, -0.5, -0.25, 0, 0.25, 0.5, 1} (so F = 0 and |Fa| = |Fb| are common), W in
    0..3, Wc in 0..3 (at least 1 where F < 0, as integration guarantees) and distinct colour sums per point."""
    rng = np.random.RandomState(seed)
    F = rng.choice(np.array([-1, -0.5, -0.25, 0, 0.25, 0.5, 1], np.float32), shape)
    W = rng.randint(0, 4, shape).astype(np.uint16)
    Wc = rng.randint(0, 4, shape).astype(np.uint16)
    Wc[(F < 0) & (Wc == 0)] = 1
    S = (rng.randint(0, 256, shape + (3,)) * Wc[..., None] + rng.randint(0, 2, shape + (3,)) * (Wc[..., None] > 1)).astype(np.uint32)
    return dict(origin=(-1.0, 0.5, 0.25), voxel=0.125, dims=shape[::-1]), (F, W, Wc, S)


def test_tie_field_exercises_the_boundaries(pkg):
    grid, (F, W, Wc, S) = tie_field(SEED)
    xyz, rgb, tri = mesh_binding.extract(grid, 1, F, W, Wc, S)
    assert len(tri) > 100 and assert_oriented_manifold(tri, len(xyz), closed=False) is not None
    assert (F == 0).sum() > 50 and len(np.unique(rgb, axis=0)) > 50


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_gpu_extract_ties_and_colours(pkg, seed):
    grid, f = tie_field(SEED + seed)
    with pkg.mesh.MeshEngine(1, 1, 1) as eng:
        for mw in (1, 2, 3):
            assert_same_mesh(eng.dbg_extract(grid, mw, *f), mesh_binding.extract(grid, mw, *f))


@pytest.mark.gpu
def test_gpu_rig_ground_truth(pkg):
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"])
    grid = pkg.mesh.default_grid(views)
    xyz, rgb, tri = gpu_vs_oracle(pkg, views, grid)
    print(f"[mesh] C3small default grid {grid['dims']} voxel {grid['voxel']:.4g}: {len(xyz)} vertices, {len(tri)} triangles")
    assert len(tri) > 10000


@pytest.mark.gpu
def test_gpu_field_matches_oracle(pkg):
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], noise=2e-3)
    grid = coarse_grid(pkg, views)
    trunc = 4.0 * grid["voxel"]
    H, W = views[0]["depth"].shape
    with pkg.mesh.MeshEngine(len(views), W, H) as eng:
        for k, v in enumerate(views):
            eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        eng.run(grid, trunc, 2)
        got = eng.dbg_field(grid)
    for g, w in zip(got, mesh_binding.field(views, grid, trunc)):
        assert g.tobytes() == w.tobytes()


@pytest.mark.gpu
def test_gpu_all_views_then_mesh(pkg, tmp_path):
    root = str(tmp_path / "c3small") + "/"
    r = subprocess.run(CLI + ["--synthetic=C3small", "-mslp_folder", root, "-all_views", "-fuse", "-mesh", "--iterations=2"],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    ply = os.path.join(root, "TSAR_mesh.ply")
    first = open(ply, "rb").read()
    assert os.path.exists(os.path.join(root, "TSAR_fused.ply"))
    opt = pkg.cli.parse_args(["-mesh", "-mslp_folder", root])
    _, names, load = pkg.cli.dataset_views(opt, root, ("TSAR_disp.dmb",))
    views = [load(k) for k in range(len(names))]
    xyz, rgb, tri = gpu_vs_oracle(pkg, views, pkg.mesh.default_grid(views))
    assert len(tri) > 0
    pkg.dmb.write_mesh_ply(str(tmp_path / "api.ply"), xyz, rgb, tri)
    assert open(str(tmp_path / "api.ply"), "rb").read() == first
    os.remove(ply)
    r = subprocess.run(CLI + ["-mesh", "-mslp_folder", root], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert open(ply, "rb").read() == first


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["noise", "one_view", "nx2", "odd_dims", "partly_outside"])
def test_gpu_adversarial_maps(pkg, case):
    rng = np.random.RandomState(SEED + len(case))
    views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], noise=3e-3)
    for v in views:
        H, W = v["depth"].shape
        bad = rng.rand(H, W) < 0.05
        v["depth"][bad] = rng.choice(np.array([0.0, -1.0, np.nan, np.inf, -0.0], np.float32), bad.sum())
        v["bgr"] = rng.randint(0, 256, v["bgr"].shape).astype(np.uint8)
    grid = coarse_grid(pkg, views)
    o, s, d = np.array(grid["origin"]), grid["voxel"], list(grid["dims"])
    if case == "one_view":
        views = views[:1]
    elif case == "nx2":
        grid = dict(origin=list(o + [s * d[0] / 2, 0, 0]), voxel=s, dims=[2, d[1], d[2]])
    elif case == "odd_dims":
        grid = dict(origin=list(o), voxel=s, dims=[d[0] - (d[0] % 8 == 0) * 3, d[1] | 1, d[2] - (d[2] % 4 == 0)])
    elif case == "partly_outside":
        grid = dict(origin=list(o - [s * d[0] / 2, 0, s * d[2] / 2]), voxel=s, dims=d)
    for mw in range(1, len(views) + 1, 2 if case == "noise" else len(views)):
        gpu_vs_oracle(pkg, views, grid, min_weight=mw)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(12, 1920, 1080), (4, 3100, 2050)])
def test_gpu_production_sizes(pkg, shape):
    n, W, H = shape
    cfg = dict(W=W, H=H, n_images=n, V=3, fx=1160.0 if W == 1920 else 1750.0, radius=4.0, arc_deg=20.0, rig="sequence")
    views, _ = rig_views(pkg, cfg, noise=2e-3, backend="torch", device="cuda:0")
    grid = pkg.mesh.default_grid(views)
    while np.prod(grid["dims"]) < 1e8:
        grid = pkg.mesh.default_grid(views, voxel=grid["voxel"] * 0.8)
    xyz, _, tri = gpu_vs_oracle(pkg, views, grid)
    print(f"[mesh] {n} x {W}x{H}: grid {grid['dims']} ({np.prod(grid['dims'])} points): {len(xyz)} vertices, {len(tri)} triangles")
    assert len(tri) > 100000


@pytest.mark.gpu
@pytest.mark.parametrize("make", [sphere_field, torus_field, lambda: random_field(SEED, undefined=0.1),
                                  lambda: random_field(SEED + 1, shape=(17, 9, 33))])
def test_gpu_extract_matches_oracle(pkg, make):
    grid, f = make()
    with pkg.mesh.MeshEngine(1, 1, 1) as eng:
        got = eng.dbg_extract(grid, 1, *f)
        assert_same_mesh(got, mesh_binding.extract(grid, 1, *f))
        W = f[1].copy()
        W[W > 0] = 3
        assert_same_mesh(eng.dbg_extract(grid, 4, f[0], W, f[2], f[3]), (np.empty((0, 3), np.float32),
                                                                          np.empty((0, 3), np.uint8), np.empty((0, 3), np.int32)))


def sphere_views(pkg, n_cams=20, W=160, H=160, f=120.0, dist=3.0, r=1.0):
    """Depth maps of the unit sphere at the origin, exact ray / sphere intersections in float64; 0 off the sphere."""
    K = np.array([[f, 0, (W - 1) / 2], [0, f, (H - 1) / 2], [0, 0, 1]])
    ys, xs = np.mgrid[0:H, 0:W]
    rays_cam = np.stack([xs, ys, np.ones_like(xs)], -1).reshape(-1, 3).astype(np.float64) @ np.linalg.inv(K).T
    views = []
    for i in range(n_cams):                            # a Fibonacci spiral of directions, away from the y axis poles
        y = 0.9 * (1 - 2 * (i + 0.5) / n_cams)
        a = i * np.pi * (3 - np.sqrt(5))
        C = dist * np.array([np.sqrt(1 - y * y) * np.cos(a), y, np.sqrt(1 - y * y) * np.sin(a)])
        R = pkg.scene._look_at(C, np.zeros(3))
        d = rays_cam @ R                               # world directions with camera z = 1
        b, c = d @ C, C @ C - r * r
        aa = (d * d).sum(-1)
        disc = b * b - aa * c
        lam = np.where(disc >= 0, (-b - np.sqrt(np.maximum(disc, 0))) / aa, 0.0)
        views.append(dict(K=K, R=R, t=-R @ C, depth=lam.reshape(H, W).astype(np.float32),
                          bgr=np.full((H, W, 3), (40 + 10 * i) % 256, np.uint8)))
    return views


@pytest.mark.gpu
def test_gpu_sphere_geometry(pkg):
    views = sphere_views(pkg)
    voxel = 0.04
    grid = pkg.mesh.box_grid([-1.3] * 3, [1.3] * 3, voxel)
    xyz, _, tri = gpu_vs_oracle(pkg, views, grid, min_weight=1)
    chi = assert_oriented_manifold(tri, len(xyz))
    err = np.abs(np.linalg.norm(xyz.astype(np.float64), axis=1) - 1.0)
    print(f"[mesh] sphere: {len(xyz)} vertices, {len(tri)} triangles, chi {chi}, max |r - 1| = {err.max():.4g} "
          f"({err.max() / voxel:.3f} voxels)")
    assert chi == 2 and err.max() <= voxel
    P = xyz[tri].astype(np.float64)
    n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    assert ((n * P.mean(1)).sum(-1) > 0).all()


@pytest.mark.gpu
def test_gpu_c3small_accuracy(pkg):
    cfg = pkg.scene.CONFIGS["C3small"]
    views, _ = rig_views(pkg, cfg, noise=1e-3)
    grid = pkg.mesh.default_grid(views)
    xyz, _, _ = pkg.mesh.mesh(views, grid)
    gt = pkg.scene.rig_ground_truth_points(cfg, 2, grid["voxel"] / 2)
    tau = 2 * grid["voxel"]
    res = pkg.cloud_eval.evaluate(xyz, gt, [tau])
    print(f"[mesh] C3small: {len(xyz)} vertices, accuracy at 2 voxels ({tau:.4g}) {res['accuracy'][0]:.4f}, "
          f"completeness {res['completeness'][0]:.4f}")
    assert res["accuracy"][0] >= ACCURACY_FLOOR


ACCURACY_FLOOR = 0.89   # measured 0.948 on a B200 (completeness 0.886), floor 0.05 below


@pytest.mark.gpu
def test_gpu_second_run_allocates_nothing(interposer):  # noqa: F811
    run_scenario(interposer, """
        sys.path.insert(0, ROOT)
        from tests.test_fusion import rig_views
        from tests.test_mesh import coarse_grid
        views, _ = rig_views(pkg, pkg.scene.CONFIGS["C3small"], noise=2e-3)
        H, W = views[0]["depth"].shape
        small = coarse_grid(pkg, views, 4.0)
        large = coarse_grid(pkg, views, 2.0)
        me = pkg.mesh.MeshEngine(len(views), W, H)
        for k, v in enumerate(views):
            me.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        first = me.run(small)
        before = counts()
        again = me.run(small)
        assert calls_since(before) == {}, ("MeshEngine", calls_since(before))
        assert all(a.tobytes() == b.tobytes() for a, b in zip(first, again))
        big = me.run(large)
        assert len(big[2]) > len(first[2])
        before = counts()
        third = me.run(small)
        assert calls_since(before) == {}, ("MeshEngine after a larger grid", calls_since(before))
        assert all(a.tobytes() == b.tobytes() for a, b in zip(first, third))
        fresh = pkg.mesh.mesh(views, large)
        assert all(a.tobytes() == b.tobytes() for a, b in zip(big, fresh))
        me.close()
        print("ok")
    """)


@pytest.mark.gpu
def test_gpu_rejects_bad_arguments(pkg):
    import ctypes as C
    v = plane_view()
    L = pkg._lib
    lib = L.load()
    h = C.c_void_p()
    assert lib.tsar_mesh_create(0, None, 0, 4, 4, C.byref(h)) == -1
    assert lib.tsar_mesh_create(0, None, 65536, 4, 4, C.byref(h)) == -1
    grid = column_grid(1.75)
    with pkg.mesh.MeshEngine(2, 64, 64) as eng:
        with pytest.raises(pkg.TsarError, match="no completed tsar_mesh_run"):
            eng.dbg_times()
        eng.set_view(0, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        with pytest.raises(pkg.TsarError, match="view 1 was not set"):
            eng.run(grid, 0.5, 1)
        eng.set_view(1, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        for g, trunc, mw in ((dict(grid, voxel=0.0), 0.5, 1), (dict(grid, voxel=float("nan")), 0.5, 1),
                             (dict(grid, dims=(1, 3, 3)), 0.5, 1), (dict(grid, dims=(2, 2, 2 ** 23 + 1)), 0.5, 1),
                             (dict(grid, dims=(2 ** 11, 2 ** 11, 2 ** 10)), 0.5, 1), (grid, 0.0, 1), (grid, float("inf"), 1),
                             (grid, 0.5, 0), (grid, 0.5, 65536)):
            with pytest.raises(pkg.TsarError):
                eng.run(g, trunc, mw)
        xyz, _, tri = eng.run(grid, 0.5, 1)
        assert len(xyz) > 0 and len(tri) > 0
        integrate_ms, extract_ms = eng.dbg_times()
        assert integrate_ms > 0 and extract_ms > 0
        buf = np.empty((len(xyz), 3), np.float32)
        assert lib.tsar_mesh_get(eng.h, buf.ctypes.data, buf.ctypes.data, len(xyz) - 1, buf.ctypes.data, len(tri)) == -1
        assert lib.tsar_mesh_get(eng.h, None, None, len(xyz), None, len(tri)) == -1
