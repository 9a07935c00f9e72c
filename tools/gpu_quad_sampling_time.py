#!/usr/bin/env python3
"""Per-launch time of the PatchMatch kernels with quad-cooperative sampling on and off (DESIGN.md 4.4).

In one process: for each configuration, two contexts on the same scene -- one with quad sampling in every launch, one
with the per-lane loop everywhere (tsar_dbg_quad_sampling) -- run the benchmark's sequence (pm_init_kernel, then 8
fused red/black iterations = 16 pm_checker_kernel launches) alternately, REPS times each.  pm_init_kernel is timed by
CUDA events around tsar_init_planes (which also clears the state and draws one XORWOW table, the same in both modes),
every checkerboard launch by the library's own event pair (tsar_profile_read_launches).  Nsight Compute is not used:
the argument rests on launch times, not on texture wavefront counts.  The 19 x 19 window has no quad path; its two
contexts run the same kernels, which shows the spread of the measurement.

    python tools/gpu_quad_sampling_time.py [configs]   ->  $TSAR_RECORD_DIR/quad_sampling_<config>.json
    configs: comma-separated NAME or NAME/BOX (default C2,C1,C4,C5,C1/19,C4/19); env TSAR_QUAD_REPS (default 5)
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import parity_common as pc  # noqa: E402

SEED = 20240601
ITERS = 8
ALL = 1 << 30


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


def run_config(pkg, name, box, reps):
    import torch
    from tsar_mvs_b200.engine import cameras_to_struct
    cfg = pkg.scene.CONFIGS[name]
    scene = pkg.scene.make_scene(name, backend="torch", device="cuda:0")
    params = pkg.make_params(box=box, iterations=ITERS, n_best=1, cost_comb=1, min_disparity=scene["min_disparity"],
                             max_disparity=scene["max_disparity"])
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    engines = {}
    for mode, k in (("per_lane", -1), ("quad", ALL)):
        e = pkg.DepthmapEngine(0, stream=stream.cuda_stream)
        e.set_views_device([t.data_ptr() for t in scene["images"]], cfg["W"], cfg["H"], cameras_to_struct(scene["cams"]),
                           scene["subset"], cam_f=scene["cam_f"])
        e.set_params(params)
        e.quad_sampling(k)
        e.init_planes(SEED); e.iterate(ITERS, SEED)      # warm-up: modules, attributes, tables
        engines[mode] = e
    torch.cuda.synchronize()
    samples = {m: dict(init=[], launches=[]) for m in engines}
    for r in range(reps):
        for mode in (("per_lane", "quad") if r % 2 == 0 else ("quad", "per_lane")):
            e = engines[mode]
            e.profile(True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); e.init_planes(SEED + r); b.record()
            e.iterate(ITERS, SEED + r)
            torch.cuda.synchronize()
            samples[mode]["init"].append(a.elapsed_time(b))
            samples[mode]["launches"].append(e.profile_read_launches())
            e.profile(False)
    for e in engines.values():
        e.close()
    res = {}
    for mode, s in samples.items():
        L = np.asarray(s["launches"])          # [reps][16]
        tot = L.sum(1) + np.asarray(s["init"])
        res[mode] = dict(init_ms_median=float(np.median(s["init"])), init_ms=[round(v, 4) for v in s["init"]],
                         launch_ms_median=[round(float(v), 4) for v in np.median(L, 0)],
                         launch_ms_min=[round(float(v), 4) for v in L.min(0)], launch_ms_max=[round(float(v), 4) for v in L.max(0)],
                         init_plus_checker_ms_median=float(np.median(tot)), init_plus_checker_ms=[round(float(v), 3) for v in tot])
    p, q = res["per_lane"], res["quad"]
    res["quad_over_per_lane"] = dict(init=q["init_ms_median"] / p["init_ms_median"],
                                     launches=[round(b / a, 4) for a, b in zip(p["launch_ms_median"], q["launch_ms_median"])],
                                     init_plus_checker=q["init_plus_checker_ms_median"] / p["init_plus_checker_ms_median"])
    return res


def main():
    import torch
    names = (sys.argv[1] if len(sys.argv) > 1 else "C2,C1,C4,C5,C1/19,C4/19").split(",")
    reps = int(os.environ.get("TSAR_QUAD_REPS", "5"))
    pkg = pc.load_pkg()
    info = gpu_info()
    info["torch_device"] = torch.cuda.get_device_name(0)
    for item in names:
        name, box = (item.split("/") + ["11"])[:2]
        res = run_config(pkg, name, int(box), reps)
        rec = dict(config=name, box=int(box), reps=reps, iterations=ITERS, gpu=info, gpu_after=gpu_info(),
                   method="CUDA events; modes alternate; pm_init_kernel timed with tsar_init_planes (memsets + one RNG table "
                          "included in both modes); no Nsight Compute on this machine, so wavefronts per quad are not re-measured",
                   **res)
        tag = f"{name}" + ("" if box == "11" else f"_box{box}")
        path = pc.record(f"quad_sampling_{tag}.json", rec)
        r = res["quad_over_per_lane"]
        print(f"{tag}: init {res['per_lane']['init_ms_median']:.3f} -> {res['quad']['init_ms_median']:.3f} ms; "
              f"init+checker {res['per_lane']['init_plus_checker_ms_median']:.2f} -> {res['quad']['init_plus_checker_ms_median']:.2f} ms "
              f"({r['init_plus_checker']:.4f}); per launch quad/per-lane {r['launches']}  [{path}]", flush=True)


if __name__ == "__main__":
    main()
