"""Timing of the cloud-to-cloud evaluation (tsar_eval_*, DESIGN.md section 4.7) on one GPU.

    python tools/gpu_eval_time.py --out profiles/r03_eval_timing.json [--configs C3,C4seq] [--tau-max 0.05,0.5]

For each rig the reconstruction is the fused cloud of its noisy ground-truth maps (depth x (1 + 1e-3 N(0, 1)), as
tools/gpu_fusion_time.py makes it) and the ground truth is scene.rig_ground_truth_points(cfg, 8, 0.005).  Per tau_max:
  * the whole tsar_eval_run (upload, both indexes, both query directions, counts, distances not copied back): CUDA
    events on the handle's stream, best of --repeat;
  * index build and query time: torch.profiler with CUDA activities over one further run, kernels summed by stage
    (index = box, keys, radix sort, gather, leaves, merges; query = eval_query_kernel);
  * queries per second of the query kernel (n + m queries over its time);
  * tree leaves visited per query, mean and max, per direction (tsar_eval_dbg_visits).
For scale, scipy.spatial.cKDTree on the host with all cores (workers=-1): tree build on the ground truth and a query of
--kdtree-sample reconstruction points at distance_upper_bound = tau_max; at C3 also the tree over the reconstruction
and a sample of ground-truth queries.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402

GT_STRIDE, GT_SPACING = 8, 0.005
THRESHOLDS = {0.05: [0.005, 0.01, 0.02, 0.05], 0.5: [0.01, 0.02, 0.05, 0.1, 0.2, 0.5]}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def fused_cloud(pkg, cfg, seed=7):
    K, Rs, Cs, neighbours = pkg.scene.make_rig(cfg)
    sc = pkg.scene.Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"], seed=1234)
    normals = torch.tensor(np.array([f["n"] for f in sc.facets], np.float32), device="cuda:0")
    gen = torch.Generator(device="cuda:0").manual_seed(seed)
    Kinv = np.linalg.inv(K)
    with pkg.fusion.FusionEngine(cfg["n_images"], cfg["W"], cfg["H"]) as eng:
        for i, (R, C) in enumerate(zip(Rs, Cs)):
            img, depth, label = sc.render_torch(dict(K_inv=Kinv, _R_world=R, _C_world=C), cfg["W"], cfg["H"], "cuda:0")
            depth = depth * (1.0 + 1e-3 * torch.randn(depth.shape, generator=gen, device="cuda:0"))
            u8 = img.to(torch.uint8)
            bgr = torch.stack([u8, torch.roll(u8, 3, 1), torch.roll(u8, 5, 0)], -1)
            eng.set_view(i, K, R, -R @ C, depth.cpu().numpy(), normals[label.long()].cpu().numpy(), bgr.cpu().numpy(),
                         neighbours[i])
        return eng.run()[0]


def stage(name):
    if "eval_query_kernel" in name:
        return "query"
    if re.search(r"eval_(bbox|key|gather|leaf|merge)_kernel|DeviceRadixSort|Onesweep|RadixSort", name):
        return "index"
    return None


def time_gpu(pkg, recon, gt, tau_max, repeat):
    thr = THRESHOLDS[tau_max]
    stream = torch.cuda.Stream(device=0)
    with pkg.cloud_eval.EvalEngine(0, stream=stream.cuda_stream) as eng:
        res = eng.run(recon, gt, thr, tau_max=tau_max)          # warm-up: module load, scratch allocation
        ms = []
        for _ in range(repeat):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            eng.run(recon, gt, thr, tau_max=tau_max)
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        tot, mx = eng.visits()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.run(recon, gt, thr, tau_max=tau_max)
            torch.cuda.synchronize()
    stages, kernels = {"index": 0.0, "query": 0.0}, {}
    for ev in prof.key_averages():
        s = stage(ev.key)
        if s:
            stages[s] += ev.device_time_total / 1e3
            kernels[ev.key[:80]] = dict(calls=ev.count, total_ms=round(ev.device_time_total / 1e3, 3))
    n, m = len(recon), len(gt)
    out = dict(tau_max=tau_max, thresholds=thr, eval_ms_best=round(min(ms), 2), eval_ms_all=[round(x, 2) for x in ms],
               index_ms=round(stages["index"], 2), query_ms=round(stages["query"], 2),
               queries_per_s=round((n + m) / (stages["query"] / 1e3), 1) if stages["query"] else None,
               visits_mean=[round(tot[0] / max(n, 1), 2), round(tot[1] / max(m, 1), 2)], visits_max=mx,
               accuracy=res["accuracy"], completeness=res["completeness"], fscore=res["fscore"], kernels=kernels)
    print(json.dumps({k: v for k, v in out.items() if k != "kernels"}), flush=True)
    return out


def time_kdtree(index, queries, tau_max, n_sample, seed=3):
    from scipy.spatial import cKDTree
    t = time.perf_counter()
    tree = cKDTree(index.astype(np.float64))
    build = time.perf_counter() - t
    sel = np.random.RandomState(seed).choice(len(queries), min(n_sample, len(queries)), replace=False)
    Q = queries[sel].astype(np.float64)
    t = time.perf_counter()
    tree.query(Q, k=1, distance_upper_bound=tau_max, workers=-1)
    q = time.perf_counter() - t
    return dict(index_points=len(index), build_s=round(build, 2), sampled_queries=len(sel), query_s=round(q, 2),
                queries_per_s=round(len(sel) / q, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="C3,C4seq")
    ap.add_argument("--tau-max", default="0.05,0.5")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--kdtree-sample", type=int, default=2000000)
    a = ap.parse_args()
    pkg = g.load_package()
    out = dict(gpu=gpu_info(), torch=torch.__version__, host_cores=os.cpu_count(), runs=[])
    for name in a.configs.split(","):
        cfg = pkg.scene.CONFIGS[name]
        t = time.perf_counter()
        recon = fused_cloud(pkg, cfg)
        gt = pkg.scene.rig_ground_truth_points(cfg, GT_STRIDE, GT_SPACING, backend="torch", device="cuda:0")
        run = dict(config=name, n_recon=len(recon), n_gt=len(gt), gt_stride=GT_STRIDE, gt_spacing=GT_SPACING,
                   setup_s=round(time.perf_counter() - t, 1), gpu=[], kdtree=[])
        print(json.dumps({k: v for k, v in run.items() if k not in ("gpu", "kdtree")}), flush=True)
        for tau in [float(x) for x in a.tau_max.split(",")]:
            run["gpu"].append(time_gpu(pkg, recon, gt, tau, a.repeat))
            kd = dict(tau_max=tau, direction="recon -> gt", **time_kdtree(gt, recon, tau, a.kdtree_sample))
            print(json.dumps(kd), flush=True)
            run["kdtree"].append(kd)
            if name == "C3" and not any(k["direction"] == "gt -> recon" for k in run["kdtree"]):
                kd = dict(tau_max=tau, direction="gt -> recon", **time_kdtree(recon, gt, tau, a.kdtree_sample))
                print(json.dumps(kd), flush=True)
                run["kdtree"].append(kd)
        out["runs"].append(run)
        del recon, gt
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
