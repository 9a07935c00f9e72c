"""Timing of the mesh extraction (tsar_mesh_*, DESIGN.md section 4.8) on one GPU.

    python tools/gpu_mesh_time.py --out profiles/r03_mesh_timing.json [--configs C3,C4seq] [--repeat 3]

For each rig (C3: 38 views of 3100x2050, C4seq: 300 views of 1920x1080) the views are the noisy ground-truth maps of
tools/gpu_fusion_time.py (depth times 1 + 1e-3 N(0, 1), rendered on the GPU) on the default grid (mesh.default_grid,
trunc 4 voxels, min_weight 3); where the default grid has more than 2^31 - 1 points the voxel is raised by factors of
1.25 until it fits, and the default grid's size is recorded.  Reported:
  * the whole run: CUDA events on the handle's stream around tsar_mesh_run (integration + extraction, which ends in a
    synchronise; the mesh stays on the device), best and median of --repeat runs;
  * per kernel: torch.profiler with CUDA activities over one further run (repeated while its trace lacks the integration
    kernel, up to 3 windows);
  * integration and extraction separately from CUDA events recorded by the library (tsar_mesh_dbg_times), best of the
    same runs; point-view updates per second from the integration time;
  * grid points, vertices, triangles;
  * device memory from shapes (views 8 B per pixel, field 20 B and extraction scratch 18 B per grid point, mesh 15 B per
    vertex and 12 B per triangle).
The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import __graft_entry__ as g  # noqa: E402
from gpu_fusion_time import gpu_info, render_views  # noqa: E402


def time_config(pkg, name, repeat):
    cfg = pkg.scene.CONFIGS[name]
    W, H, N = cfg["W"], cfg["H"], cfg["n_images"]
    stream = torch.cuda.Stream(device=0)
    eng = pkg.mesh.MeshEngine(N, W, H, device=0, stream=stream.cuda_stream)
    t = time.perf_counter()
    points, ratios = [], []
    for k, v in enumerate(render_views(pkg, cfg)):
        eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["bgr"])
        p, r = pkg.mesh.depth_samples(v)
        points.append(p)
        ratios.append(r)
    points, ratios = np.concatenate(points), np.concatenate(ratios)
    # the default grid, or when it has more than 2^31 - 1 points, the default voxel times 1.25^k for the smallest k that fits
    default_error, factor = None, 1.0
    voxel = float(np.float32(2.0 * np.median(ratios)))
    while True:
        try:
            grid = pkg.mesh.grid_from_samples(points, ratios, voxel * factor)
            break
        except ValueError as e:
            default_error = default_error or str(e)
            factor *= 1.25
    setup_s = time.perf_counter() - t
    n_grid = int(np.prod(grid["dims"]))
    nv, nt = eng.run(grid, fetch=False)                  # warm-up (module load, allocation)
    ms, int_ev, ext_ev = [], [], []
    for _ in range(repeat):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.run(grid, fetch=False)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
        a, b = eng.dbg_times()
        int_ev.append(a)
        ext_ev.append(b)
    from torch.profiler import ProfilerActivity, profile
    # one run per profiler window; a window whose trace lacks the integration kernel's record (seen once at C4seq, where
    # that kernel runs for about a second) is repeated, up to 3 windows
    for windows in range(1, 4):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.run(grid, fetch=False)
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.key_averages():
            m = re.search(r"mesh_\w+_kernel|DeviceScan\w*Kernel", ev.key)
            if m:
                k = kernels.setdefault(m.group(0), dict(calls=0, total_ms=0.0))
                k["calls"] += ev.count
                k["total_ms"] = round(k["total_ms"] + ev.device_time_total / 1e3, 3)
        if "mesh_integrate_kernel" in kernels:
            break
    t = time.perf_counter()
    xyz, _, tri = eng.get()
    get_s = time.perf_counter() - t
    eng.close()
    updates = n_grid * N
    int_ms = kernels.get("mesh_integrate_kernel", {}).get("total_ms")
    extract_ms = round(sum(v["total_ms"] for k, v in kernels.items() if k != "mesh_integrate_kernel" and k != "mesh_pack_kernel"), 3)
    mem = dict(views=8 * W * H * N, field=20 * n_grid, scratch=18 * n_grid, mesh=15 * nv + 12 * nt)
    res = dict(config=name, W=W, H=H, views=N, default_voxel=voxel, default_grid_error=default_error, voxel_factor=factor,
               grid_dims=list(grid["dims"]), voxel=grid["voxel"], trunc=4 * grid["voxel"],
               min_weight=3, grid_points=n_grid, vertices=int(nv), triangles=int(nt), setup_s=round(setup_s, 2),
               run_ms_best=round(min(ms), 2), run_ms_median=round(float(np.median(ms)), 2), kernels=kernels, profiler_windows=windows,
               integrate_ms=int_ms, extract_ms=extract_ms, get_s=round(get_s, 3), point_view_updates=updates,
               device_bytes_from_shapes=mem, device_gb_total=round(sum(mem.values()) / 1e9, 2))
    res["integrate_ms_events_best"] = round(min(int_ev), 3)
    res["extract_ms_events_best"] = round(min(ext_ev), 3)
    res["point_view_updates_per_s"] = round(updates / (min(int_ev) / 1e3), 1)
    assert len(xyz) == nv and len(tri) == nt
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="C3,C4seq")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    pkg = g.load_package()
    out = dict(gpu=gpu_info(), torch=torch.__version__, mesh=[])
    for name in a.configs.split(","):
        out["mesh"].append(time_config(pkg, name, a.repeat))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
