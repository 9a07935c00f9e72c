#!/usr/bin/env python3
"""One-off differential stress of the per-region RANSAC plane fit against the reference's own loop (main.cpp:1520-1730 in
oracle/_ref/libtsar_ref_host.so) on region tables the parity test does not reach: regions with 1, 2, 3, 5, 20, 300, 5000
reliable points (degenerate triples: every hypothesis is 0/0 = NaN and, ties replacing the best, NaN becomes the plane),
exactly collinear points, outlier fractions 0 ... 60 %, several weak regions per view, random streams, both the
host-supplied and the device-generated stream.  Planes must agree bit for bit (a NaN on both sides counts as equal).
Regions without any reliable point are left out: the reference divides by zero there (rand() % 0).

    python tools/gpu_ransac_sweep.py [N]   ->  $TSAR_RECORD_DIR/ransac_sweep.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 30
pkg = pc.load_pkg()
rh = pc.ref_host()
L = pkg._lib
rng = np.random.RandomState(int(os.environ.get("TSAR_SWEEP_SEED", "2718")))   # TSAR_SWEEP_SEED: another campaign
rows, bad = [], 0
scene = pkg.scene.make_scene("small")
H, W = scene["H"], scene["W"]
params, mine, _ = pc.make_engines(pkg, scene, variants=())
per = mine.lib.tsar_ransac_rand_per_region()
labels = scene["labels"]
nreg = len(scene["region_text"])


def same(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


for trial in range(N):
    disp = (scene["cam_f"] / scene["gt_depth"]).astype(np.float32)
    disp *= (1 + 0.0005 * rng.normal(size=disp.shape)).astype(np.float32)
    out_frac = float(rng.choice([0.0, 0.05, 0.2, 0.6]))
    out = rng.rand(H, W) < out_frac
    disp[out] *= rng.uniform(0.7, 1.3, int(out.sum())).astype(np.float32)
    text = np.ones(nreg, np.float32)
    weak = rng.choice(nreg, size=int(rng.randint(1, nreg + 1)), replace=False)
    text[weak] = -1.0
    scale = np.zeros((H, W), np.float32)
    counts = {}
    for r in weak:
        ys, xs = np.nonzero(labels == r)
        want = int(rng.choice([1, 2, 3, 5, 20, 300, 5000]))
        want = min(want, len(ys))
        if trial % 5 == 4 and want >= 3:        # exactly collinear: one image row
            row = ys[len(ys) // 2]
            sel = np.nonzero(ys == row)[0][:want]
        else:
            sel = rng.choice(len(ys), size=want, replace=False)
        scale[ys[sel], xs[sel]] = 1.0
        counts[int(r)] = int(len(sel))
    size = np.array([(labels == r).sum() / 16.0 for r in range(nreg)], np.float32)
    rnd = rng.randint(0, 2 ** 31 - 1, size=(nreg, per)).astype(np.uint32)
    mine.upload(L.F_DEPTH, disp); mine.upload(L.F_SCALE, scale); mine.upload(L.F_CANNY, scene["canny"])
    p0 = np.tile(np.array([0, 0, 1, -1], np.float32), (nreg, 1))
    fitted = mine.fit_region_planes(text, size, rnd, p0)
    stream = np.concatenate([rnd[r] for r in range(nreg) if text[r] == -1])
    ref, used = rh.fit_regions(scene["cams"][0], scene["cam_f"], disp, scale, scene["canny"], text, size, stream, p0)
    seed = int(rng.randint(1, 2 ** 31))
    seeded = mine.fit_region_planes(text, size, None, p0, seed=seed)
    with np.errstate(over="ignore"):
        stream2 = np.concatenate([mine.ransac_rand_stream(seed, r) for r in range(nreg) if text[r] == -1])
    ref2, _ = rh.fit_regions(scene["cams"][0], scene["cam_f"], disp, scale, scene["canny"], text, size, stream2, p0)
    ok = same(fitted, ref) and same(seeded, ref2) and used == len(stream)
    row = dict(trial=trial, weak_regions=counts, outlier_fraction=out_frac, collinear=bool(trial % 5 == 4), host_stream_equal=same(fitted, ref),
               device_stream_equal=same(seeded, ref2), rand_values_used=int(used), nan_planes=int(np.isnan(ref).any(axis=1).sum()))
    if not ok:
        row["mine"] = fitted.tolist(); row["ref"] = ref.tolist()
    bad += 0 if ok else 1
    rows.append(row)
    print(("ok  " if ok else "FAIL"), json.dumps({k: v for k, v in row.items() if k not in ("mine", "ref")}), flush=True)
mine.close()
pc.record("ransac_sweep.json", dict(trials=N, exact_trials=N - bad, rows=rows))
print(f"{N - bad} of {N} trials exact")
sys.exit(1 if bad else 0)
