#!/usr/bin/env python3
"""One-off differential stress of the per-pixel kernels around PatchMatch -- gipuma_getlrdiff, gipuma_getview,
gipuma_update_scale_2, gipuma_update_scale, gipuma_compute_disp, gipuma_get_disp -- against the reference's own kernels on
ADVERSARIAL state: random planes (incl. degenerate normals and plane offsets of either sign, zero and tiny), costs on and
around the thresholds (0, 2.0 = MAXCOST), random best views, random reliable flags, random region labels and region tables
whose planes include zeros, on random sizes and camera rigs.  Every field is compared bit for bit (NaN payloads included).

    python tools/gpu_glue_sweep.py [N]   ->  $TSAR_RECORD_DIR/glue_sweep.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 40
pkg = pc.load_pkg()
L = pkg._lib
rb = pc.ref_binding()
rng = np.random.RandomState(int(os.environ.get("TSAR_SWEEP_SEED", "99")))   # TSAR_SWEEP_SEED: another campaign
FIELDS = (("norm4", L.F_NORM4, rb.F_NORM4), ("cost", L.F_COST, rb.F_COST), ("depth", L.F_DEPTH, rb.F_DEPTH),
          ("fakedepth", L.F_FAKEDEPTH, rb.F_FAKEDEPTH), ("scale", L.F_SCALE, rb.F_SCALE), ("lrdiff", L.F_LRDIFF, rb.F_LRDIFF),
          ("confid", L.F_CONFID, rb.F_CONFID))
rows, bad = [], 0


def pick(shape, values, p_special, base):
    out = base.astype(np.float32)
    m = rng.rand(*shape) < p_special
    out[m] = rng.choice(np.array(values, np.float32), size=int(m.sum()))
    return out


for trial in range(N):
    W, H = int(rng.randint(40, 300)), int(rng.randint(34, 220))
    V = int(rng.randint(1, 7))
    cfg = dict(W=W, H=H, n_images=V + 1, V=V, fx=float(rng.uniform(120, 500)), radius=float(rng.uniform(0.8, 3.0)), arc_deg=float(rng.uniform(6, 30)))
    scene = pkg.scene.make_scene(cfg, seed=int(rng.randint(1, 100000)))
    params, mine, refs = pc.make_engines(pkg, scene, iterations=1, variants=("asis",))
    ref = refs["asis"]
    nrm = rng.normal(size=(H, W, 3)).astype(np.float32)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=-1, keepdims=True), 1e-6)
    nrm[rng.rand(H, W) < 0.02] = 0.0                                              # degenerate normals
    d = pick((H, W), [0.0, -0.0, 1e-30, -1e-30, 1e30, -1.0, 1.0], 0.05, rng.uniform(-3, 3, (H, W)))
    n4 = np.concatenate([nrm, d[..., None]], -1).astype(np.float32)
    cost = pick((H, W), [0.0, 2.0, 1.9999999, 2.0000002, 1.0], 0.2, rng.uniform(0, 2, (H, W)))
    beview = rng.randint(1, V + 1, (H, W)).astype(np.int32)   # camera ids of the source views (the reference indexes its camera
                                                               # table with this value: -1 is an out-of-bounds read there)
    ratio = pick((H, W), [0.0, 1.0, np.inf], 0.1, rng.uniform(0, 1, (H, W)))
    depth = pick((H, W), [0.0, -1.0, 1e-20, 1e20], 0.05, rng.uniform(0.1, 20, (H, W)))
    scale = (rng.rand(H, W) < 0.5).astype(np.float32)
    nreg = int(rng.randint(1, 12))
    canny = rng.randint(0, nreg, (H, W)).astype(np.float32)
    text = rng.choice(np.array([-1.0, 1.0, 0.0], np.float32), size=nreg)
    planes = rng.normal(size=(nreg, 4)).astype(np.float32)
    planes[rng.rand(nreg) < 0.2] = 0.0
    for e, fn, fc, fb, fr, fd, fs, fca in ((mine, L.F_NORM4, L.F_COST, L.F_BEVIEW, L.F_RATIO, L.F_DEPTH, L.F_SCALE, L.F_CANNY),
                                           (ref, rb.F_NORM4, rb.F_COST, rb.F_BEVIEW, rb.F_RATIO, rb.F_DEPTH, rb.F_SCALE, rb.F_CANNY)):
        if e is mine:
            e.load_planes(n4, cost)
        else:
            e.upload(fn, n4); e.upload(fc, cost)
        e.upload(fb, beview); e.upload(fr, ratio); e.upload(fd, depth); e.upload(fs, scale); e.upload(fca, canny)
        e.set_regions(text, planes)
    row = dict(trial=trial, W=W, H=H, V=V, regions=nreg, stages={})
    ok = True
    for stage in ("lrdiff", "getview", "update_scale_2", "update_scale", "compute_disp", "get_disp"):
        getattr(mine, stage)(); getattr(ref, stage)()
        worst = {}
        for name, fm, fr in FIELDS:
            f = pc.frac_bit_exact(mine.download(fm), ref.download(fr))
            if f != 1.0:
                worst[name] = f
        row["stages"][stage] = worst or "bit-exact"
        ok = ok and not worst
    mine.close(); ref.close()
    bad += 0 if ok else 1
    rows.append(row)
    print(("ok  " if ok else "FAIL"), json.dumps(row), flush=True)
pc.record("glue_sweep.json", dict(trials=N, bit_exact_trials=N - bad, rows=rows))
print(f"{N - bad} of {N} trials bit-exact")
sys.exit(1 if bad else 0)
