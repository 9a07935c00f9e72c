#!/usr/bin/env python3
"""One-off differential stress of the gSLICr kernels against the reference engine (gSLICr_seg_engine_GPU.cu unmodified):
random image sizes (incl. sizes that are not multiples of the superpixel size), superpixel sizes, iteration counts,
coherence weights, with and without the connectivity pass, on structured and on noise images.  Labels must be identical.

    python tools/gpu_slic_sweep.py [N]   ->  $TSAR_RECORD_DIR/slic_sweep.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 150
pkg = pc.load_pkg()
rb = pc.ref_binding()
rng = np.random.RandomState(int(os.environ.get("TSAR_SWEEP_SEED", "777")))   # TSAR_SWEEP_SEED: another campaign
eng = pkg.DepthmapEngine(0)
rows, bad = [], 0
for trial in range(N):
    size = int(rng.choice([8, 10, 12, 16, 20, 20, 24, 32]))
    w, h = int(rng.randint(4 * size, 900)), int(rng.randint(4 * size, 600))
    iters = int(rng.randint(1, 8))
    coh = float(rng.choice([0.5, 1.0, 5.0, 5.0, 10.0, 40.0]))
    enforce = bool(rng.randint(0, 2))
    kind = trial % 3
    if kind == 0:      # smooth colour structure + noise
        yy, xx = np.mgrid[0:h, 0:w]
        base = np.stack([127 + 100 * np.sin(xx / rng.uniform(9, 60) + yy / rng.uniform(9, 60)), 127 + 100 * np.cos(xx / rng.uniform(9, 60)),
                         127 + 100 * np.sin(yy / rng.uniform(9, 60))], -1)
        img = np.clip(base + rng.normal(0, 6, base.shape), 0, 255).astype(np.uint8)
    elif kind == 1:    # pure noise
        img = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
    else:              # piecewise constant blocks (many exact ties in the colour distance)
        blk = rng.randint(0, 256, (h // 16 + 1, w // 16 + 1, 3)).astype(np.uint8)
        img = np.repeat(np.repeat(blk, 16, 0), 16, 1)[:h, :w]
    bgrx = np.concatenate([img, np.zeros((h, w, 1), np.uint8)], -1)
    mine = eng.slic(bgrx, spixel_size=size, no_iters=iters, coh_weight=coh, enforce_connectivity=enforce)
    ref, _ = rb.ref_slic(bgrx, spixel_size=size, no_iters=iters, coh_weight=coh, enforce_connectivity=enforce)
    same = float((mine == ref).mean())
    row = dict(trial=trial, w=w, h=h, spixel_size=size, no_iters=iters, coh_weight=coh, enforce_connectivity=enforce,
               image=("structured", "noise", "blocks")[kind], labels_identical=same)
    bad += 0 if same == 1.0 else 1
    rows.append(row)
    print(("ok  " if same == 1.0 else "FAIL"), json.dumps(row), flush=True)
eng.close()
pc.record("slic_sweep.json", dict(trials=N, identical_trials=N - bad, rows=rows))
print(f"{N - bad} of {N} configurations identical")
sys.exit(1 if bad else 0)
