#!/usr/bin/env python3
"""One-off adversarial stress of pmCostMultiview against the reference's own function (unmodified build) on explicit
(pixel, plane) pairs: the parity test uses well-behaved planes (depth in range, normal facing the camera); here the planes
are hostile -- offsets 0, +-1e-30 ... +-1e30, normals at grazing angles, through the camera centre, behind the camera,
non-unit and zero normals, NaN / inf components -- so that the window crosses z = 0, divisors leave the range of the
branch-free refined division (the kernel must take its exact IEEE path), samples fall far outside the image, variances
vanish.  Windows 5..25, 1..10 views, n_best 1..3, both combinations, 8-bit and fp32 texels.  Cost, best view and ratio
must agree bit for bit (NaN counts as equal to NaN; the ratio is not compared for V = 1, where the reference reads an
uninitialised slot, SURVEY Q8).

    python tools/gpu_cost_sweep.py [configs] [pairs]   ->  $TSAR_RECORD_DIR/cost_sweep.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

NCFG = int(sys.argv[1]) if len(sys.argv) > 1 else 16
NP = int(sys.argv[2]) if len(sys.argv) > 2 else 60000
pkg = pc.load_pkg()
rng = np.random.RandomState(int(os.environ.get("TSAR_SWEEP_SEED", "1618")))   # TSAR_SWEEP_SEED: another campaign
rows, bad = [], 0


def eq(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind == "f":
        return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    return a == b


for trial in range(NCFG):
    W, H = int(rng.randint(48, 400)), int(rng.randint(40, 300))
    V = int(rng.randint(1, 11))
    box = int(rng.choice([5, 7, 11, 11, 12, 19, 25]))
    n_best = int(rng.randint(1, min(V, 3) + 1))
    cost_comb = int(rng.choice([0, 1]))
    cfg = dict(W=W, H=H, n_images=V + 1, V=V, fx=float(rng.uniform(120, 500)), radius=float(rng.uniform(0.8, 3.0)), arc_deg=float(rng.uniform(6, 30)))
    scene = pkg.scene.make_scene(cfg, seed=int(rng.randint(1, 100000)))
    if trial % 2:
        scene["images"] = [np.ascontiguousarray(im + rng.uniform(0, 0.9, im.shape).astype(np.float32)) for im in scene["images"]]
    params, mine, refs = pc.make_engines(pkg, scene, box=box, n_best=n_best, cost_comb=cost_comb, variants=("asis",))
    ref = refs["asis"]
    xy = np.stack([rng.randint(0, W, NP), rng.randint(0, H, NP)], 1).astype(np.int32)
    k = NP // 6
    xy[:k, 0] = rng.choice([0, 1, W - 2, W - 1], k); xy[k:2 * k, 1] = rng.choice([0, 1, H - 2, H - 1], k)
    nrm = rng.normal(size=(NP, 3)).astype(np.float32)
    mode = rng.randint(0, 8, NP)
    unit = mode < 5
    nrm[unit] /= np.linalg.norm(nrm[unit], axis=1, keepdims=True)
    nrm[mode == 5, 2] = rng.uniform(-1e-4, 1e-4, int((mode == 5).sum()))          # grazing
    nrm[mode == 6] = 0.0
    nrm[mode == 7] *= rng.choice(np.array([1e-20, 1e20, 3.0], np.float32), int((mode == 7).sum()))[:, None]
    d = rng.uniform(-3, 3, NP).astype(np.float32)
    special = rng.rand(NP) < 0.25
    d[special] = rng.choice(np.array([0.0, -0.0, 1e-30, -1e-30, 1e-10, 1e30, -1e30, np.inf, -np.inf, np.nan], np.float32), int(special.sum()))
    bad_n = rng.rand(NP) < 0.01
    nrm[bad_n, int(rng.randint(0, 3))] = rng.choice(np.array([np.nan, np.inf], np.float32), int(bad_n.sum()))
    planes = np.concatenate([nrm, d[:, None]], 1).astype(np.float32)
    c_m, b_m, r_m = mine.eval_planes(xy, planes, wrapper_rounding=True)
    c_r, b_r, r_r = ref.eval_planes(xy, planes)
    e_c, e_b, e_r = eq(c_m, c_r), eq(b_m, b_r), eq(r_m, r_r)
    if V == 1:      # SURVEY Q8: with one view the reference's ratio = costVector[0] / costVector[1] reads an uninitialised slot
        e_r = np.ones_like(e_r)
    ok = bool(e_c.all() and e_b.all() and e_r.all())
    row = dict(trial=trial, W=W, H=H, V=V, box=box, n_best=n_best, cost_comb=cost_comb, texels="fp32" if trial % 2 else "u8", pairs=NP,
               cost=float(e_c.mean()), best_view=float(e_b.mean()), ratio=float(e_r.mean()), nan_costs=int(np.isnan(c_r).sum()),
               maxcost=int((c_r == 2.0).sum()))
    if not ok:
        i = int(np.argmin(e_c & e_b & e_r))
        row["first_bad"] = dict(xy=xy[i].tolist(), plane=[float(v) for v in planes[i]], mine=[float(c_m[i]), int(b_m[i]), float(r_m[i])], ref=[float(c_r[i]), int(b_r[i]), float(r_r[i])])
    mine.close(); ref.close()
    bad += 0 if ok else 1
    rows.append(row)
    print(("ok  " if ok else "FAIL"), json.dumps(row), flush=True)
pc.record("cost_sweep.json", dict(configs=NCFG, exact_configs=NCFG - bad, rows=rows))
print(f"{NCFG - bad} of {NCFG} configurations exact")
sys.exit(1 if bad else 0)
