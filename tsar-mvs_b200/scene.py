"""Deterministic synthetic multi-view scenes of the shapes named in BASELINE.json.

The reference has no data-independent test inputs (SURVEY section 4); this module supplies them:
an analytic piecewise-planar scene (tilted background + three slanted facets + one textureless
facet), a 3-D procedural texture I(X) evaluated at the exact ray/plane intersection of every pixel
(no resampling, so all views are photo-consistent), pin-hole cameras on an arc, and the camera
quantities getCameraParameters(transformP=true) would produce (cameraGeometryUtils.h:174-364;
formulas restated in SURVEY section 3.4).  Everything is computed in float64 with numpy and rounded
once to float32 / uint8, so both the reference build and this library receive identical bits.
"""
import numpy as np

# name -> (W, H, n_images, V, fx, radius)   (SURVEY section 8, row d)
CONFIGS = {
    "C1": dict(W=640, H=480, n_images=16, V=15, fx=3310.0, radius=0.65, arc_deg=45.0),     # dinoSparseRing-shaped
    "C2": dict(W=3100, H=2050, n_images=11, V=10, fx=1750.0, radius=4.0, arc_deg=30.0),    # ETH3D pipes-shaped
    "C4": dict(W=1920, H=1080, n_images=11, V=10, fx=1160.0, radius=5.0, arc_deg=30.0),    # Tanks&Temples-shaped
    "C5": dict(W=6048, H=4032, n_images=21, V=20, fx=3410.0, radius=6.0, arc_deg=40.0),    # full-resolution stress
    # multi-view datasets: a fixed set of reference views, each paired with its 10 nearest cameras (pair.txt)
    "C3": dict(W=3100, H=2050, n_images=38, V=10, fx=1750.0, radius=4.0, arc_deg=44.0, rig="two_arcs"),   # ETH3D courtyard-shaped
    "C4seq": dict(W=1920, H=1080, n_images=300, V=10, fx=1160.0, radius=5.0, arc_deg=60.0, rig="sequence"),  # Tanks&Temples-shaped
    "C3small": dict(W=320, H=240, n_images=8, V=4, fx=800.0, radius=1.0, arc_deg=24.0, rig="two_arcs"),      # tests
    "mid": dict(W=1280, H=960, n_images=5, V=4, fx=720.0, radius=4.0, arc_deg=16.0),       # detector + completion tests
    "tiny": dict(W=96, H=64, n_images=4, V=3, fx=180.0, radius=1.0, arc_deg=16.0),         # unit tests / golden
    "small": dict(W=320, H=240, n_images=6, V=5, fx=800.0, radius=1.0, arc_deg=20.0),      # GPU parity tests
}


def _look_at(C, target):
    z = target - C
    z = z / np.linalg.norm(z)
    up = np.array([0.0, -1.0, 0.0])
    x = np.cross(-up, z)  # image x to the right when y points down
    x = x / np.linalg.norm(x)
    y = np.cross(z, x)
    return np.stack([x, y, z])  # rows: world -> camera


def cameras_from_krt(Ks, Rs, ts, depth_min, depth_max):
    """Camera_cu fields as getCameraParameters(transformP=true) fills them (cameraGeometryUtils.h:174-364; SURVEY 3.4)
    from per-image K, world->camera R and t; image 0 is the reference.  Note the reference's choices that are kept:
    every P uses the intrinsics of camera 0, baseline is hard-coded to 1, fx/fy/f/alpha come from K_0."""
    Ks = [np.asarray(K, float) for K in Ks]
    Rs = [np.asarray(R, float) for R in Rs]
    ts = [np.asarray(t, float).reshape(3) for t in ts]
    R0, t0, K0 = Rs[0], ts[0], Ks[0]
    cams = []
    for K, R, t in zip(Ks, Rs, ts):
        Rp = R @ R0.T                          # cameraGeometryUtils.h:113-139
        tp = t - Rp @ t0
        P = K0 @ np.concatenate([Rp, tp[:, None]], axis=1)
        cams.append(dict(
            K=K, K_inv=np.linalg.inv(K), R=Rp, R_orig=R, R_orig_inv=np.linalg.inv(R), M_inv=np.linalg.inv(P[:, :3]),
            t4=tp, P_col34=P[:, 3], C4=-Rp.T @ tp, fx=K0[0, 0], fy=K0[1, 1], f=K0[0, 0], alpha=K0[0, 0] / K0[1, 1],
            baseline=1.0, depthMin=depth_min, depthMax=depth_max))
    return cams


def make_cameras(W, H, n_images, fx, radius, arc_deg, depth_range=(0.7, 1.45), ref_index=0):
    """Cameras on an arc, sorted by baseline from the middle one.  Camera `ref_index` of that list becomes
    the reference (index 0 of the returned list); the others keep their order."""
    K = np.array([[fx, 0, (W - 1) / 2.0], [0, fx, (H - 1) / 2.0], [0, 0, 1.0]])
    target = np.zeros(3)
    half = np.deg2rad(arc_deg) / 2.0
    # angles: 0 for the reference, the others alternate left/right with growing baseline
    angs = [0.0]
    k = 1
    while len(angs) < n_images:
        step = half * (int((k + 1) / 2) / np.ceil((n_images - 1) / 2.0))
        angs.append(step if k % 2 else -step)
        k += 1
    Rs, ts, Cs = [], [], []
    for i, a in enumerate(angs):
        elev = 0.06 * np.sin(2.3 * i)  # small vertical parallax as well
        C = radius * np.array([np.sin(a), elev, -np.cos(a)])
        R = _look_at(C, target)
        Rs.append(R)
        Cs.append(C)
        ts.append(-R @ C)
    order = [ref_index % n_images] + [i for i in range(n_images) if i != ref_index % n_images]
    Rs, ts, Cs = [Rs[i] for i in order], [ts[i] for i in order], [Cs[i] for i in order]
    cams = cameras_from_krt([K] * n_images, Rs, ts, depth_range[0] * radius, depth_range[1] * radius)
    for c, R, C in zip(cams, Rs, Cs):
        c["_R_world"], c["_C_world"] = R, C
    return cams


def make_rig(cfg):
    """World cameras of a multi-view dataset (every image is a reference view once, scripts/pipes.sh:30-49):
      two_arcs  n/2 cameras on each of two arcs at different heights (ETH3D courtyard-shaped: a photographer walking
                along the scene twice);
      sequence  n cameras along one arc with a slow vertical wave (Tanks&Temples-shaped video sequence).
    Returns (K, [R], [C], neighbours) with neighbours[i] = the V cameras nearest to camera i, nearest first (pair.txt)."""
    W, H, n, fx, radius = cfg["W"], cfg["H"], cfg["n_images"], cfg["fx"], cfg["radius"]
    K = np.array([[fx, 0, (W - 1) / 2.0], [0, fx, (H - 1) / 2.0], [0, 0, 1.0]])
    half = np.deg2rad(cfg["arc_deg"]) / 2.0
    Cs = []
    if cfg["rig"] == "two_arcs":
        per = (n + 1) // 2
        for i in range(n):
            row, k = divmod(i, per)
            a = -half + 2 * half * (k + 0.5 * row) / max(per - 1 + 0.5, 1)
            Cs.append(radius * np.array([np.sin(a), (-0.10 if row == 0 else 0.12), -np.cos(a)]))
    else:
        for i in range(n):
            a = -half + 2 * half * i / max(n - 1, 1)
            Cs.append(radius * np.array([np.sin(a), 0.08 * np.sin(0.21 * i), -np.cos(a)]))
    Rs = [_look_at(C, np.zeros(3)) for C in Cs]
    P = np.stack(Cs)
    d = np.linalg.norm(P[:, None, :] - P[None, :, :], axis=-1)
    neighbours = [[int(j) for j in np.argsort(d[i], kind="stable") if j != i][:cfg["V"]] for i in range(n)]
    return K, Rs, Cs, neighbours


def render_rig(cfg, seed=1234, backend="numpy", device=None, depth_range=(0.7, 1.45)):
    """Images of all cameras of a rig (uint8), generator of (index, image).  Depth range as make_cameras."""
    K, Rs, Cs, _ = make_rig(cfg)
    sc = Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"], seed=seed)
    Kinv = np.linalg.inv(K)
    for i, (R, C) in enumerate(zip(Rs, Cs)):
        cam = dict(K_inv=Kinv, _R_world=R, _C_world=C)
        if backend == "torch":
            img = sc.render_torch(cam, cfg["W"], cfg["H"], device)[0].cpu().numpy().astype(np.uint8)
        else:
            img = sc.render(cam, cfg["W"], cfg["H"])[0]
        yield i, img


def rig_ground_truth_points(cfg, stride, spacing, backend="numpy", device=None):
    """The visible ground truth of a rig as a point cloud ([n][3] float32): every `stride`-th pixel (both axes) of the
    rendered ground-truth depth of every view is back-projected in float64 (X = C + depth * R^T K^-1 (x, y, 1)), then
    thinned to one point per voxel of size `spacing` (voxel = floor(X / spacing)): the first point in view order, then
    raster order, is kept.  Deterministic.  The facets are not sampled directly because facet 0 is unbounded; what the
    cameras see bounds it."""
    K, Rs, Cs, _ = make_rig(cfg)
    sc = Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"], seed=1234)
    Kinv = np.linalg.inv(K)
    ys, xs = np.mgrid[0:cfg["H"]:stride, 0:cfg["W"]:stride]
    rays = np.stack([xs, ys, np.ones_like(xs)], -1).reshape(-1, 3).astype(np.float64) @ Kinv.T
    pts = []
    for R, C in zip(Rs, Cs):
        cam = dict(K_inv=Kinv, _R_world=R, _C_world=C)
        if backend == "torch":
            depth = sc.render_torch(cam, cfg["W"], cfg["H"], device)[1].cpu().numpy().astype(np.float64)
        else:
            depth = sc.render(cam, cfg["W"], cfg["H"])[1]
        d = depth[::stride, ::stride].reshape(-1)
        ok = np.isfinite(d)
        pts.append(C + d[ok, None] * (rays[ok] @ R))
    X = np.concatenate(pts)
    vox = np.floor(X / spacing).astype(np.int64)
    _, first = np.unique(vox, axis=0, return_index=True)
    return X[np.sort(first)].astype(np.float32)


class Scene:
    """Piecewise-planar scene in world coordinates, sized to the reference camera's frustum."""

    def __init__(self, W, H, fx, radius, seed=1234):
        rng = np.random.RandomState(seed)
        hw = 0.5 * W / fx * radius  # half-extent of the frustum at the look-at distance
        hh = 0.5 * H / fx * radius
        self.radius = radius

        def unit(v):
            v = np.asarray(v, float)
            return v / np.linalg.norm(v)

        # facets: (point, normal, u half-extent, v half-extent, textured?)   index = region label
        self.facets = [
            dict(p0=np.array([0, 0, 0.22 * radius]), n=unit([0.12, 0.08, -1]), hu=np.inf, hv=np.inf, textured=True),
            dict(p0=np.array([-0.45 * hw, -0.40 * hh, 0.02 * radius]), n=unit([0.35, 0.05, -1]), hu=0.36 * hw, hv=0.40 * hh, textured=True),
            dict(p0=np.array([0.50 * hw, -0.35 * hh, -0.06 * radius]), n=unit([-0.30, 0.20, -1]), hu=0.34 * hw, hv=0.42 * hh, textured=True),
            dict(p0=np.array([-0.40 * hw, 0.50 * hh, -0.02 * radius]), n=unit([0.05, -0.40, -1]), hu=0.42 * hw, hv=0.32 * hh, textured=True),
            dict(p0=np.array([0.45 * hw, 0.45 * hh, 0.06 * radius]), n=unit([-0.10, -0.12, -1]), hu=0.45 * hw, hv=0.42 * hh, textured=False),
        ]
        for f in self.facets:
            u = np.cross(f["n"], [0.0, 1.0, 0.0])
            f["u"] = u / np.linalg.norm(u)
            f["v"] = np.cross(f["n"], f["u"])
        # procedural 3-D texture: 12 sinusoids, wavelengths 5..80 pixels at the look-at distance
        px = radius / fx
        lam = np.exp(rng.uniform(np.log(5 * px), np.log(80 * px), size=12))
        dirs = rng.normal(size=(12, 3))
        dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
        self.omega = dirs * (2 * np.pi / lam)[:, None]
        self.phase = rng.uniform(0, 2 * np.pi, size=12)
        self.amp = 45.0 / np.sqrt(np.arange(1, 13))
        self.flat_omega = unit(rng.normal(size=3)) * (2 * np.pi / (3.1 * px))

    def intensity(self, X, textured):
        val = 127.5 + np.tensordot(np.sin(np.tensordot(X, self.omega.T, axes=1) + self.phase), self.amp, axes=1)
        flat = 128.0 + (np.sin(np.tensordot(X, self.flat_omega, axes=1)) > 0.3)  # constant +- 1 grey level
        return np.where(textured, np.clip(val, 0, 255), flat)

    def render(self, cam, W, H, rows=None):
        """Returns (uint8 image, depth along the camera z axis, facet label) for one camera."""
        R, C = cam["_R_world"], cam["_C_world"]
        Kinv = np.asarray(cam["K_inv"], float)
        ys = np.arange(H) if rows is None else np.arange(rows[0], rows[1])
        xx, yy = np.meshgrid(np.arange(W, dtype=float), ys.astype(float))
        d_cam = np.stack([Kinv[0, 0] * xx + Kinv[0, 2], Kinv[1, 1] * yy + Kinv[1, 2], np.ones_like(xx)], axis=-1)
        d = d_cam @ R  # world direction per unit camera depth (R^T d_cam)
        best_t = np.full(xx.shape, np.inf)
        label = np.zeros(xx.shape, np.int32)
        for idx, f in enumerate(self.facets):
            denom = d @ f["n"]
            with np.errstate(divide="ignore", invalid="ignore"):
                t = (f["n"] @ (f["p0"] - C)) / denom
            X = C + t[..., None] * d
            rel = X - f["p0"]
            ok = (t > 0) & np.isfinite(t)
            if np.isfinite(f["hu"]):
                ok &= (np.abs(rel @ f["u"]) <= f["hu"]) & (np.abs(rel @ f["v"]) <= f["hv"])
            upd = ok & (t < best_t)
            best_t = np.where(upd, t, best_t)
            label = np.where(upd, idx, label)
        X = C + best_t[..., None] * d
        textured = np.array([f["textured"] for f in self.facets])[label]
        img = np.rint(self.intensity(X, textured)).astype(np.uint8)
        return img, best_t, label

    def render_torch(self, cam, W, H, device):
        """Same renderer with torch (float64) so large bench scenes are rendered on the GPU in < 1 s.
        sin() may differ from numpy in the last bit, i.e. +-1 grey level in rare pixels: fine for the
        benchmark (both arms get the same images); parity fixtures always use the numpy path."""
        import torch
        dt = torch.float64
        tt = lambda a: torch.as_tensor(np.asarray(a, float), dtype=dt, device=device)
        R, C, Kinv = tt(cam["_R_world"]), tt(cam["_C_world"]), tt(cam["K_inv"])
        img = torch.empty((H, W), dtype=torch.float32, device=device)
        depth = torch.empty((H, W), dtype=torch.float32, device=device)
        label = torch.empty((H, W), dtype=torch.int32, device=device)
        omega, phase, amp, fomega = tt(self.omega), tt(self.phase), tt(self.amp), tt(self.flat_omega)
        step = max(1, (1 << 22) // W)
        xs = torch.arange(W, dtype=dt, device=device)
        for r0 in range(0, H, step):
            r1 = min(H, r0 + step)
            ys = torch.arange(r0, r1, dtype=dt, device=device)
            yy, xx = torch.meshgrid(ys, xs, indexing="ij")
            d_cam = torch.stack([Kinv[0, 0] * xx + Kinv[0, 2], Kinv[1, 1] * yy + Kinv[1, 2], torch.ones_like(xx)], dim=-1)
            d = d_cam @ R
            best_t = torch.full(xx.shape, float("inf"), dtype=dt, device=device)
            lab = torch.zeros(xx.shape, dtype=torch.int32, device=device)
            for idx, f in enumerate(self.facets):
                n, p0 = tt(f["n"]), tt(f["p0"])
                t = (n @ (p0 - C)) / (d @ n)
                rel = C + t[..., None] * d - p0
                ok = (t > 0) & torch.isfinite(t)
                if np.isfinite(f["hu"]):
                    ok &= ((rel @ tt(f["u"])).abs() <= f["hu"]) & ((rel @ tt(f["v"])).abs() <= f["hv"])
                upd = ok & (t < best_t)
                best_t = torch.where(upd, t, best_t)
                lab = torch.where(upd, torch.full_like(lab, idx), lab)
            X = C + best_t[..., None] * d
            textured = torch.as_tensor([f["textured"] for f in self.facets], device=device)[lab.long()]
            val = 127.5 + torch.sin(X @ omega.T + phase) @ amp
            flat = 128.0 + (torch.sin(X @ fomega) > 0.3).to(dt)
            v = torch.where(textured, val.clamp(0, 255), flat)
            img[r0:r1] = torch.round(v).to(torch.float32)
            depth[r0:r1] = best_t.to(torch.float32)
            label[r0:r1] = lab
        return img, depth, label

    def region_planes(self, cam0, perturb=0.0):
        """Per-facet plane (n, d) with n.X + d = 0 in the reference camera frame (linestate.h:12)."""
        R, C = cam0["_R_world"], cam0["_C_world"]
        out = []
        for i, f in enumerate(self.facets):
            n = R @ f["n"]
            p = R @ (f["p0"] - C)
            if perturb:
                n = n + perturb * np.array([0.3, -0.2, 0.1]) * (1 + i % 3)
                n = n / np.linalg.norm(n)
            out.append(np.concatenate([n, [-n @ p]]))
        return np.array(out)


def reorder_reference(cams_world, ref_index):
    """Camera list with camera `ref_index` moved to the front (it becomes the reference view)."""
    order = [ref_index] + [i for i in range(len(cams_world)) if i != ref_index]
    return order


def make_scene(name_or_cfg, seed=1234, with_colour=False, ref_index=0, backend="numpy", device=None):
    """Builds a full test case: images (float32 0..255, image 0 = reference), cameras, view subset,
    algorithm parameters, ground-truth depth / facet labels of the reference view, region table."""
    cfg = CONFIGS[name_or_cfg] if isinstance(name_or_cfg, str) else dict(name_or_cfg)
    W, H, n, V = cfg["W"], cfg["H"], cfg["n_images"], cfg["V"]
    cams = make_cameras(W, H, n, cfg["fx"], cfg["radius"], cfg["arc_deg"], ref_index=ref_index)
    sc = Scene(W, H, cfg["fx"], cfg["radius"], seed=seed)
    images = []
    gt_depth = labels = None
    for i, cam in enumerate(cams):
        if backend == "torch":
            im, dep, lab = sc.render_torch(cam, W, H, device)
            images.append(im)  # stays a torch tensor (on `device`)
            if i == 0:
                gt_depth, labels = dep.cpu().numpy(), lab.cpu().numpy()
            continue
        parts = []
        step = max(1, (1 << 21) // W)  # render in row bands to bound memory
        for r0 in range(0, H, step):
            parts.append(sc.render(cam, W, H, rows=(r0, min(H, r0 + step))))
        img = np.concatenate([p[0] for p in parts], axis=0)
        if i == 0:
            gt_depth = np.concatenate([p[1] for p in parts], axis=0).astype(np.float32)
            labels = np.concatenate([p[2] for p in parts], axis=0)
        images.append(img.astype(np.float32))  # uint8 -> float32 as main.cpp:1423
    f = float(np.float32(cams[0]["f"]))
    dmin, dmax = float(np.float32(cams[0]["depthMin"])), float(np.float32(cams[0]["depthMax"]))
    # disparityDepthConversion(f, baseline, depth) in float (main.cpp:1393-1398)
    min_disp = float(np.float32(np.float32(f * np.float32(1.0)) / np.float32(dmax)))
    max_disp = float(np.float32(np.float32(f * np.float32(1.0)) / np.float32(dmin)))
    planes = sc.region_planes(cams[0], perturb=0.02).astype(np.float32)
    text = np.array([1.0 if fct["textured"] else -1.0 for fct in sc.facets], np.float32)
    out = dict(W=W, H=H, images=images, cams=cams, subset=list(range(1, V + 1)), cam_f=f,
               min_disparity=min_disp, max_disparity=max_disp, gt_depth=gt_depth, labels=labels,
               region_text=text, region_norm4=planes, canny=labels.astype(np.float32))
    if with_colour:
        ref = images[0] if backend == "numpy" else images[0].cpu().numpy()
        g = np.roll(ref, 3, axis=1)
        r = np.roll(ref, 5, axis=0)
        out["bgr"] = np.stack([ref, g, r], axis=-1).astype(np.uint8)
    return out


def box_downsample4(bgr):
    """Quarter-resolution colour image for gSLICr (stands in for the two pyrDown of main.cpp:621-622;
    the same routine feeds the reference kernels and ours).  Returns [h/4][w/4][4] uint8 (B,G,R,0)."""
    h, w = bgr.shape[0] // 4 * 4, bgr.shape[1] // 4 * 4
    x = bgr[:h, :w].astype(np.uint32).reshape(h // 4, 4, w // 4, 4, 3).sum(axis=(1, 3))
    out = np.zeros((h // 4, w // 4, 4), np.uint8)
    out[..., :3] = ((x + 8) // 16).astype(np.uint8)
    return out
