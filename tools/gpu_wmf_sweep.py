#!/usr/bin/env python3
"""One-off differential stress of the weighted-median kernels (gipuma_WMF x 4 levels, gipuma_WMF_Final x 6 levels) against
the reference twin whose `norm_mid` is zero-initialised (oracle/build_ref.sh 2b: the reference as written reads that
variable uninitialised when a median is never reached): random sizes, reliable-pixel densities from 3 % to 97 % (sparse
masks give the tiny neighbour lists where medians are not reached), random region tables, planes straight from a short
PatchMatch run.  Every level starts from the reference's state; flags, planes and disparities must agree on 100 % of the pixels.

    python tools/gpu_wmf_sweep.py [N]   ->  $TSAR_RECORD_DIR/wmf_sweep.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 24
pkg = pc.load_pkg()
L = pkg._lib
rb = pc.ref_binding()
rng = np.random.RandomState(int(os.environ.get("TSAR_SWEEP_SEED", "31337")))   # TSAR_SWEEP_SEED: another campaign
rows, bad = [], 0
for trial in range(N):
    W, H = int(rng.randint(60, 420)), int(rng.randint(50, 300))
    V = int(rng.randint(2, 5))
    cfg = dict(W=W, H=H, n_images=V + 1, V=V, fx=float(rng.uniform(150, 600)), radius=float(rng.uniform(0.8, 3.0)), arc_deg=float(rng.uniform(8, 24)))
    scene = pkg.scene.make_scene(cfg, seed=int(rng.randint(1, 100000)))
    params, mine, refs = pc.make_engines(pkg, scene, iterations=2, variants=("snapshot_init",))
    ref = refs["snapshot_init"]
    seed = int(rng.randint(1, 2 ** 31))
    ref.init_planes(seed); ref.iterate(2, seed); ref.lrdiff(); ref.getview()
    n0, c0, d0 = ref.download(rb.F_NORM4), ref.download(rb.F_COST), ref.download(rb.F_DEPTH)
    density = float(rng.choice([0.03, 0.1, 0.3, 0.5, 0.8, 0.97]))
    reliable = (rng.rand(H, W) < density).astype(np.float32)
    mine.load_planes(n0, c0); mine.upload(L.F_DEPTH, d0); mine.upload(L.F_SCALE, reliable)
    ref.upload(rb.F_SCALE, reliable)
    worst = 0.0
    for it in range(4):
        mine.upload(L.F_SCALE, ref.download(rb.F_SCALE))
        ref.wmf(it); mine.wmf(it)
        worst = max(worst, float((mine.download(L.F_SCALE) != ref.download(rb.F_SCALE)).mean()))
    nreg = len(scene["region_text"])
    text = rng.choice(np.array([1.0, 1.0, -1.0], np.float32), size=nreg)
    for e in (mine, ref):
        e.set_regions(text, scene["region_norm4"])
    mine.upload(L.F_CANNY, scene["canny"]); ref.upload(rb.F_CANNY, scene["canny"])
    ref.upload(rb.F_SCALE, reliable)          # the fill starts from the sparse mask again
    worst_final = 0.0
    for it in range(6):
        for fm, fr in ((L.F_NORM4, rb.F_NORM4), (L.F_DEPTH, rb.F_DEPTH), (L.F_SCALE, rb.F_SCALE)):
            mine.upload(fm, ref.download(fr))
        ref.wmf_final(it); mine.wmf_final(it)
        for fm, fr in ((L.F_NORM4, rb.F_NORM4), (L.F_DEPTH, rb.F_DEPTH), (L.F_SCALE, rb.F_SCALE)):
            worst_final = max(worst_final, 1 - pc.frac_bit_exact(mine.download(fm), ref.download(fr)))
    filled = float((ref.download(rb.F_SCALE) != reliable).mean())
    mine.close(); ref.close()
    row = dict(trial=trial, W=W, H=H, V=V, reliable_density=density, wmf_worst_mismatch=worst, wmf_final_worst_mismatch=worst_final, pixels_filled=filled)
    ok = worst == 0.0 and worst_final == 0.0
    bad += 0 if ok else 1
    rows.append(row)
    print(("ok  " if ok else "FAIL"), json.dumps(row), flush=True)
pc.record("wmf_sweep.json", dict(trials=N, exact_trials=N - bad, rows=rows))
print(f"{N - bad} of {N} trials exact")
sys.exit(1 if bad else 0)
