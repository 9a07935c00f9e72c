"""Shared helpers of the parity tests, smoke() and the GPU probe scripts (test infrastructure).

The checker side is oracle/ (reference kernels rebuilt for sm_100, and the CPU restatement); the
product side is always driven through the C ABI (tsar-mvs_b200/engine.py -> libtsar_b200.so).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# tolerance of the north-star parity gate (BASELINE.json): at least 99 % of pixels within 1e-3 relative
# depth and 1 degree normal angle of the reference build, from a shared initialisation
REL_DEPTH_TOL = 1e-3
ANGLE_TOL_DEG = 1.0
GATE_FRACTION = 0.99


def load_pkg():
    import __graft_entry__ as g
    return g.load_package()


def ref_binding():
    """The reference's own kernels (oracle/_ref, built by `make oracle` where the reference checkout exists), else their
    recorded results (oracle/recorded.py).  With TSAR_RECORD_REFERENCE_DIGESTS set, the reference build's results are
    recorded; that needs the build."""
    from oracle import recorded, ref_binding as rb
    built = all(rb.available(v) for v in ("asis", "snapshot", "snapshot_init")) and os.path.exists(os.path.join(rb.REF_DIR, "libgslic_ref.so"))
    if os.environ.get("TSAR_RECORD_REFERENCE_DIGESTS"):
        assert built, "recording reference results needs the reference build (oracle/_ref: `make oracle` with the reference checkout)"
        return recorded.recording()
    return rb if built else recorded


def ref_host():
    """The reference's own host code (oracle/_ref/libtsar_ref_host.so), else its recorded results."""
    from oracle import recorded, ref_host_binding as rh
    if os.environ.get("TSAR_RECORD_REFERENCE_DIGESTS"):
        assert rh.available(), "recording reference results needs the reference build (oracle/_ref/libtsar_ref_host.so)"
        return recorded.recording_host()
    return rh if rh.available() else recorded.host


def record(name, obj):
    """Writes a JSON record of a sweep or a full-size comparison into $TSAR_RECORD_DIR (default: a directory of the user's
    under the system's temporary directory); returns its path."""
    import json
    import tempfile
    out = os.environ.get("TSAR_RECORD_DIR") or os.path.join(tempfile.gettempdir(), f"tsar-mvs_b200-records-{os.getuid()}")
    os.makedirs(out, exist_ok=True)
    path = os.path.join(out, name)
    with open(path, "w") as f:
        json.dump(obj, f, indent=1)
    return path


def make_engines(pkg, scene, box=11, iterations=8, n_best=1, cost_comb=1, variants=("asis",), device=0, color_processing=0, rb=None):
    """Returns (params, mine, {variant: RefEngine}) on the same scene."""
    rb = rb or ref_binding()
    params = pkg.make_params(box=box, iterations=iterations, n_best=n_best, cost_comb=cost_comb,
                             min_disparity=scene["min_disparity"], max_disparity=scene["max_disparity"],
                             color_processing=color_processing)
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    mine = pkg.DepthmapEngine(device)
    mine.set_views(scene["images"], cams, scene["subset"], cam_f=scene["cam_f"])
    mine.set_params(params)
    refs = {}
    for v in variants:
        r = rb.RefEngine(pkg._lib.TsarCamera, pkg._lib.TsarParams, variant=v)
        r.create(scene["images"], cams, scene["subset"], params, scene["cam_f"])
        refs[v] = r
    return params, mine, refs


def random_planes(scene, n, seed=7, border=True):
    """n random (pixel, plane) pairs: depth uniform in the range, normal facing the camera."""
    rng = np.random.RandomState(seed)
    W, H = scene["W"], scene["H"]
    cam = scene["cams"][0]
    xy = np.stack([rng.randint(0, W, n), rng.randint(0, H, n)], axis=1).astype(np.int32)
    if border:  # force a share of the samples onto the image border (clamp addressing)
        k = n // 8
        xy[:k, 0] = rng.choice([0, 1, 2, W - 3, W - 2, W - 1], k)
        xy[k:2 * k, 1] = rng.choice([0, 1, 2, H - 3, H - 2, H - 1], k)
    depth = rng.uniform(cam["depthMin"], cam["depthMax"], n)
    nrm = rng.normal(size=(n, 3))
    nrm[:, 2] = -np.abs(nrm[:, 2]) - 0.3
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    Kinv = np.asarray(cam["K_inv"], float)
    X = (Kinv @ np.stack([xy[:, 0], xy[:, 1], np.ones(n)]).astype(float)).T * depth[:, None]
    d = -np.sum(nrm * X, axis=1)
    planes = np.concatenate([nrm, d[:, None]], axis=1).astype(np.float32)
    return xy, planes


def bits_equal(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.view(np.uint32 if a.dtype.itemsize == 4 else np.uint8) == b.view(np.uint32 if b.dtype.itemsize == 4 else np.uint8)


def frac_bit_exact(a, b):
    eq = bits_equal(a, b)
    if eq.ndim > 2:
        eq = eq.all(axis=-1)
    return float(eq.mean())


def output_agreement(out_a, out_b):
    """out_*: [H][W][4] in gipuma_compute_disp layout (xyz = world normal, w = depth).
    Returns dict with the fraction of pixels inside the north-star tolerance."""
    za, zb = out_a[..., 3].astype(np.float64), out_b[..., 3].astype(np.float64)
    na, nb = out_a[..., :3].astype(np.float64), out_b[..., :3].astype(np.float64)
    valid = (zb != 0)
    rel = np.abs(za - zb) / np.where(valid, np.abs(zb), 1.0)
    cosang = np.sum(na * nb, axis=-1) / np.maximum(np.linalg.norm(na, axis=-1) * np.linalg.norm(nb, axis=-1), 1e-30)
    ang = np.degrees(np.arccos(np.clip(cosang, -1, 1)))
    both_invalid = (~valid) & (za == 0)
    ok = (valid & (rel <= REL_DEPTH_TOL) & (ang <= ANGLE_TOL_DEG)) | both_invalid
    return dict(frac_ok=float(ok.mean()), frac_depth_ok=float(((rel <= REL_DEPTH_TOL) & valid | both_invalid).mean()),
                frac_angle_ok=float(((ang <= ANGLE_TOL_DEG) & valid | both_invalid).mean()),
                frac_valid=float(valid.mean()), median_rel=float(np.median(rel[valid])) if valid.any() else 0.0,
                bit_exact=frac_bit_exact(out_a, out_b))


def gt_agreement(out, scene, tol=0.01):
    z = out[..., 3].astype(np.float64)
    gt = scene["gt_depth"].astype(np.float64)
    tex = scene["region_text"][scene["labels"]] > 0
    rel = np.abs(z - gt) / gt
    return dict(frac_within_1pct_textured=float((rel[tex] <= tol).mean()), frac_within_1pct_all=float((rel <= tol).mean()))


def run_smoke_check(pkg):
    """One tiny depthmap through the C ABI on cuda:0, checked against the reference-kernel oracle when it
    travelled with the repo (oracle/_ref), else against the committed golden output."""
    scene = pkg.scene.make_scene("tiny")
    from oracle import ref_binding as rb
    variants = ("snapshot",) if rb.available("snapshot") else ()
    params, mine, refs = make_engines(pkg, scene, iterations=2, variants=variants, rb=rb)
    xy, planes = random_planes(scene, 2000)
    c_m, b_m, r_m = mine.eval_planes(xy, planes, wrapper_rounding=True)
    ms = mine.depthmap(20240601)
    out = mine.download(pkg._lib.F_NORM4)
    assert np.isfinite(out).all(), "non-finite output"
    assert mine.launch_count() > 0
    if refs:
        ref = refs["snapshot"]
        c_r, b_r, r_r = ref.eval_planes(xy, planes)
        fe = frac_bit_exact(c_m, c_r)
        ref.depthmap(20240601, iters=2)
        agree = output_agreement(out, ref.download(rb.F_NORM4))
        print(f"[smoke] eval cost bit-exact {fe:.4f}; depthmap agreement {agree}; {ms:.2f} ms")
        assert fe >= 0.999, f"pmCostMultiview parity broken: {fe}"
        assert agree["frac_ok"] >= GATE_FRACTION, agree
        ref.close()
    else:
        gold = np.load(os.path.join(ROOT, "tests", "golden", "tiny_eval.npz"))
        c_g = gold["cost"]
        fe = frac_bit_exact(c_m, c_g)
        print(f"[smoke] eval cost vs golden bit-exact {fe:.4f}; {ms:.2f} ms")
        assert fe >= 0.999, f"pmCostMultiview parity vs golden vectors broken: {fe}"
    mine.close()
    print("[smoke] ok")
