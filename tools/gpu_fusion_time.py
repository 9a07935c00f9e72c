"""Timing of the multi-view fusion (tsar_fusion_*, DESIGN.md section 4.6) on one GPU.

    python tools/gpu_fusion_time.py --out profiles/r03_fusion_timing.json [--configs C3,C4seq] [--repeat 3]

For each rig (C3: 38 views of 3100x2050, C4seq: 300 views of 1920x1080, 10 pair.txt neighbours each) the views are
rendered on the GPU (scene.render_torch): ground-truth depth times (1 + 1e-3 N(0, 1)), the facets' world normals and the
rendered image as colour.  Reported:
  * fusion alone: CUDA events on the handle's stream around tsar_fusion_run (which ends in a synchronise), best and
    median of --repeat runs, and per view;
  * per kernel: torch.profiler with CUDA activities over one further run;
  * from shapes: candidate checks (pixel x neighbour) per second of the candidate kernel, and the bytes that kernel
    gathers (the reference pixel's float4 + mask, per neighbour one float4 + one mask byte, one int written) over its
    time, against 7.7 TB/s of HBM3e (the data sheet figure; the gathers mostly hit L2);
  * the whole `tsar_cli.py -fuse` command on C3 files (JPEG images + .dmb maps in a temporary directory), wall clock;
  * oc_fuse (the single-threaded C restatement) on the first 3 views of C3 for scale.
The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402

HBM_TBPS = 7.7


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def render_views(pkg, cfg, seed=7):
    """Generator of view dicts (numpy) of a rig, rendered on cuda:0."""
    K, Rs, Cs, neighbours = pkg.scene.make_rig(cfg)
    sc = pkg.scene.Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"], seed=1234)
    normals = torch.tensor(np.array([f["n"] for f in sc.facets], np.float32), device="cuda:0")
    gen = torch.Generator(device="cuda:0").manual_seed(seed)
    Kinv = np.linalg.inv(K)
    for i, (R, C) in enumerate(zip(Rs, Cs)):
        img, depth, label = sc.render_torch(dict(K_inv=Kinv, _R_world=R, _C_world=C), cfg["W"], cfg["H"], "cuda:0")
        depth = depth * (1.0 + 1e-3 * torch.randn(depth.shape, generator=gen, device="cuda:0"))
        u8 = img.to(torch.uint8)
        bgr = torch.stack([u8, torch.roll(u8, 3, 1), torch.roll(u8, 5, 0)], -1)
        yield dict(K=K, R=R, t=-R @ C, depth=depth.cpu().numpy(), normals=normals[label.long()].cpu().numpy(),
                   bgr=bgr.cpu().numpy(), neighbours=neighbours[i])


def time_config(pkg, name, repeat):
    cfg = pkg.scene.CONFIGS[name]
    W, H, N = cfg["W"], cfg["H"], cfg["n_images"]
    P = W * H
    stream = torch.cuda.Stream(device=0)
    eng = pkg.fusion.FusionEngine(N, W, H, device=0, stream=stream.cuda_stream)
    t = time.perf_counter()
    n_src = []
    for k, v in enumerate(render_views(pkg, cfg)):
        eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], v["neighbours"])
        n_src.append(len(v["neighbours"]))
    setup_s = time.perf_counter() - t
    eng.run()                                   # warm-up (module load, scratch allocation)
    ms, wall = [], []
    for _ in range(repeat):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t = time.perf_counter()
        xyz, _, _ = eng.run()
        wall.append(time.perf_counter() - t)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    rounds = eng.rounds()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.run()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        m = re.search(r"fusion_\w+_kernel", ev.key)
        if m:
            kernels[m.group(0)] = dict(calls=ev.count, total_ms=round(ev.device_time_total / 1e3, 3))
    eng.close()
    checks = int(P * sum(n_src))
    cand_ms = kernels.get("fusion_candidates_kernel", {}).get("total_ms")
    gathered = int(N * P * (17 + 1) + checks * (16 + 1 + 4))
    res = dict(config=name, W=W, H=H, views=N, neighbours_per_view=float(np.mean(n_src)), points=int(len(xyz)),
               rounds_max=rounds[0], rounds_total=rounds[1], setup_s=round(setup_s, 2),
               fusion_ms_best=round(min(ms), 2), fusion_ms_median=round(float(np.median(ms)), 2),
               fusion_ms_per_view=round(min(ms) / N, 3), fusion_wall_s_best=round(min(wall), 3), kernels=kernels,
               candidate_checks=checks, candidate_bytes=gathered)
    if cand_ms:
        res["candidate_checks_per_s"] = round(checks / (cand_ms / 1e3), 1)
        res["candidate_bytes_per_s"] = round(gathered / (cand_ms / 1e3), 1)
        res["candidate_share_of_hbm_bandwidth"] = round(gathered / (cand_ms / 1e3) / (HBM_TBPS * 1e12), 4)
    print(json.dumps(res), flush=True)
    return res


def time_cli_fuse(pkg):
    """The whole -fuse command (read cams, pair.txt, JPEGs and .dmb maps, fuse, write the PLY) on C3 files."""
    cfg = pkg.scene.CONFIGS["C3"]
    root = tempfile.mkdtemp(prefix="tsar_fuse_C3_") + "/"
    try:
        names = pkg.cli.write_rig_dataset("C3", root, backend="torch", device="cuda:0")
        for n, v in zip(names, render_views(pkg, cfg)):
            d = os.path.join(root, "APD", n[:8])
            os.makedirs(d, exist_ok=True)
            pkg.dmb.write_dmb(os.path.join(d, "TSAR_disp.dmb"), v["depth"])
            pkg.dmb.write_dmb(os.path.join(d, "TSAR_normals.dmb"), v["normals"])
        walls = []
        for _ in range(2):
            t = time.perf_counter()
            rc = pkg.cli.run(["-fuse", "-mslp_folder", root])
            walls.append(time.perf_counter() - t)
            assert rc == 0
        n_points = len(pkg.dmb.read_model_ply(os.path.join(root, "TSAR_fused.ply"))[0])
        res = dict(config="C3", command="tsar_cli.py -fuse", wall_s=[round(w, 2) for w in walls], points=n_points,
                   ply_bytes=os.path.getsize(os.path.join(root, "TSAR_fused.ply")))
    finally:
        shutil.rmtree(root, ignore_errors=True)
    print(json.dumps(res), flush=True)
    return res


def time_oracle(pkg, n_views=3):
    from oracle import fusion_binding
    views = []
    for k, v in enumerate(render_views(pkg, pkg.scene.CONFIGS["C3"])):
        if k == n_views:
            break
        views.append(v)
    for k, v in enumerate(views):
        v["neighbours"] = [j for j in range(n_views) if j != k]
    t = time.perf_counter()
    xyz, _, _ = fusion_binding.fuse(pkg._lib.TsarViewCamera, pkg.fusion.make_params(), views)
    dt = time.perf_counter() - t
    P = views[0]["depth"].size
    res = dict(config=f"C3, first {n_views} views, each other's neighbours", threads=1, seconds=round(dt, 2), points=int(len(xyz)),
               candidate_checks_per_s=round(n_views * P * (n_views - 1) / dt, 1))
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="C3,C4seq")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--no-cli", action="store_true")
    a = ap.parse_args()
    pkg = g.load_package()
    out = dict(gpu=gpu_info(), torch=torch.__version__, fusion=[], cli=None, oracle=None)
    for name in a.configs.split(","):
        out["fusion"].append(time_config(pkg, name, a.repeat))
    if not a.no_cli:
        out["cli"] = time_cli_fuse(pkg)
    out["oracle"] = time_oracle(pkg)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
