#!/usr/bin/env python3
"""Stage-by-stage comparison of the gSLICr kernels with the reference engine, beyond the final labels:
  * rgb2CIELab over its WHOLE input domain: a 4096 x 4096 image holding every 24-bit colour once, Lab bit for bit;
  * superpixel records (centre, colour, pixel count) after 0..5 iterations on a piecewise-constant image (exact ties
    in the distance, where a last-ulp difference decides) and on a noise image, bit for bit.

    python tools/gpu_slic_stages.py   ->  $TSAR_RECORD_DIR/slic_stages.json
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

pkg = pc.load_pkg()
rb = pc.ref_binding()
eng = pkg.DepthmapEngine(0)
eng.lib.tsar_dbg_slic_lab.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
res = {}

# every colour once
n = 4096
v = np.arange(n * n, dtype=np.uint32)
img = np.zeros((n, n, 4), np.uint8)
img[..., 0] = (v & 255).reshape(n, n); img[..., 1] = ((v >> 8) & 255).reshape(n, n); img[..., 2] = ((v >> 16) & 255).reshape(n, n)
mine_lab = np.empty((n, n, 4), np.float32)
lm = eng.slic(img, spixel_size=20, no_iters=0)
eng._ck(eng.lib.tsar_dbg_slic_lab(eng.h, mine_lab.ctypes.data, n * n), "lab")
lr, _ = rb.ref_slic(img, spixel_size=20, no_iters=0)
ref_lab = rb.slic_last_lab(n * n).reshape(n, n, 4)
eq = (mine_lab[..., :3].view(np.uint32) == ref_lab[..., :3].view(np.uint32)).all(-1)
res["rgb2CIELab_all_16777216_colours_bit_exact"] = float(eq.mean())
res["labels_on_that_image_identical"] = float((lm == lr).mean())
print("Lab over all colours:", eq.mean(), "labels", (lm == lr).mean(), flush=True)

rng = np.random.RandomState(5)
for name in ("blocks", "noise"):
    w, h, size = 897, 584, 10
    if name == "blocks":
        blk = rng.randint(0, 256, (h // 16 + 1, w // 16 + 1, 3)).astype(np.uint8)
        im = np.repeat(np.repeat(blk, 16, 0), 16, 1)[:h, :w]
    else:
        im = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
    bgrx = np.concatenate([im, np.zeros((h, w, 1), np.uint8)], -1)
    nsp = (w // size) * (h // size)
    rows = []
    for it in range(6):
        m = eng.slic(bgrx, spixel_size=size, no_iters=it, coh_weight=10.0)
        mc = np.zeros((nsp, 8), np.float32); cnt = C.c_int(0)
        eng._ck(eng.lib.tsar_dbg_slic_centres(eng.h, mc.ctypes.data_as(C.c_void_p), nsp, C.byref(cnt)), "centres")
        r, _ = rb.ref_slic(bgrx, spixel_size=size, no_iters=it, coh_weight=10.0)
        rc = rb.slic_last_centres(nsp)
        sel = [0, 1, 2, 3, 4, 6, 7]          # colour w is not defined by the reference's conversion
        rows.append(dict(iterations=it, labels_identical=float((m == r).mean()),
                         records_bit_exact=float((mc.view(np.uint32)[:, sel] == rc.view(np.uint32)[:, sel]).all(1).mean())))
        print(name, rows[-1], flush=True)
    res[name] = rows
eng.close()
pc.record("slic_stages.json", res)
ok = res["rgb2CIELab_all_16777216_colours_bit_exact"] == 1.0 and all(r["labels_identical"] == 1.0 and r["records_bit_exact"] == 1.0 for k in ("blocks", "noise") for r in res[k])
print("ALL EXACT" if ok else "MISMATCH")
sys.exit(0 if ok else 1)
