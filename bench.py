#!/usr/bin/env python3
"""bench.py -- depthmaps/s of the TSAR-MVS per-reference-view depthmap path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one reference view of a synthetic scene of the named shape
(BASELINE.json configs; default C2 = ETH3D-pipes-shaped 3100x2050, 10 source views, full TSAR path):
  gSLICr segmentation -> random plane init -> 8 x red/black (propagation + refinement) -> left/right
  cost check -> confidence -> textureless-region depth completion (update_scale_2, update_scale) ->
  output layout (compute_disp).
`value` times that with every input resident in HBM; `e2e` times the same work through the public host
API (host images in, host depth/normal/confidence/labels out, copies inside the timed region).
Reference views are independent: with N GPUs each rank processes its own reference views (weak scaling,
no collective on the data path).

--impl reference runs the reference's own CUDA kernels rebuilt for sm_100 (oracle/_ref: gipuma.cu and
gSLICr unmodified, managed memory and a device sync after every kernel, as the reference is written) on
the same workload.  The reference has no CPU implementation of this path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SEED = 20240601
FLOPS_PER_EVAL = 1590.0      # BASELINE.md section 3: 40*S + 150 at S = 36 (as written in pmCost)
FLOPS_PER_EVAL_19 = 4150.0   # S = 100
FP32_NOMINAL_TFLOPS = 74.5   # 148 SM x 128 lanes x 2 x 1.965 GHz

# stdout carries the ONE JSON line and nothing else: libraries write there too (NCCL prints its version line on stdout, the
# reference's kernels printf debug lines, gipuma.cu:1043-1045), so file descriptor 1 is pointed at stderr for the whole run
# and the line goes to a duplicate of the real stdout.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    line = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--blocksize", type=int, default=11, help="NCC window (the run scripts use 11; the reference's built-in default is 19)")
    ap.add_argument("--mode", default="auto", choices=["auto", "engine", "driver"],
                    help="engine: one reference-view stream per GPU, inputs resident (C1, C2, C4, C5); driver: a fixed view set through the "
                         "multi-view file driver (C3, C4 = 300 views); auto: driver for C3 / C4, engine otherwise")
    ap.add_argument("--lanes", type=int, default=2, help="pipelined contexts per GPU of the multi-view driver (--config C3 / C4)")
    ap.add_argument("--io_threads", type=int, default=6, help="decoder / writer threads per rank of the multi-view driver")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what the last timed step computed as DIR/<name>.npy (per-view path, "
                         "rank 0): depth, normals and confidence at a fixed sample of pixels, and the superpixel labels")
    return ap.parse_args()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md): one streaming
    `nvidia-smi -lms 100` process, lines collected by a reader thread between __enter__ and __exit__."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        self.index, self.rows, self.proc, self.th, self.enabled = index, [], None, None, enabled

    def _run(self):
        for line in self.proc.stdout:
            cols = [c.strip() for c in line.strip().split(",")]
            if len(cols) >= 7:
                self.rows.append(cols)

    def __enter__(self):
        if not self.enabled:       # only rank 0 reports clocks; 8 pollers on one node would only add noise
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
            time.sleep(0.25)  # let the first sample arrive before the timed region starts
            self.rows.clear()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.th.join(timeout=5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}

        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        sm = sorted(v for v in (num(r[0]) for r in self.rows) if v is not None)
        mx = [v for v in (num(r[1]) for r in self.rows) if v is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in self.rows)]
        pw = [v for v in (num(r[2]) for r in self.rows) if v is not None]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version / debug lines must not precede the JSON line on stdout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def shutdown(world):
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def max_over_ranks(x, world):
    import torch
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def workload_name(cfg_name, cfg, iters, box=11):
    shape = {"C1": "Middlebury dinoSparseRing-shaped", "C2": "ETH3D pipes-shaped", "C4": "Tanks&Temples-shaped",
             "C5": "full-resolution ETH3D-shaped"}.get(cfg_name, "synthetic")
    return (f"{cfg_name}: synthetic {shape} scene {cfg['W']}x{cfg['H']}, {cfg['V']} source views, one reference view per step, "
            f"blocksize {box}, {iters} iterations, n_best 1; full TSAR path (gSLICr + checkerboard PatchMatch + L/R check + "
            f"confidence + textureless depth completion)")


def config_dict(cfg_name, cfg, iters, box, world):
    """`config` of the JSON line: the SAME dict in both arms (the driver compares them key by key)."""
    work_bytes = (cfg["n_images"] * 5 + 72) * cfg["W"] * cfg["H"]
    timing = (f"inputs_larger_than_l2 ({work_bytes / 1e6:.0f} MB of views + state per step)" if work_bytes >= (512 << 20)
              else "l2_flush (256 MB overwritten between timed steps)")
    return {"workload": workload_name(cfg_name, cfg, iters, box), "timing": timing, "reference_views_per_gpu_per_step": 1,
            "parallelism": f"views sharded over {world} GPU(s), one reference-view stream per GPU, no collective on the data path"}


def build_scene(pkg, cfg_name, rank, device):
    import torch
    scene = pkg.scene.make_scene(cfg_name, with_colour=True, ref_index=rank, backend="torch", device=device)
    imgs_dev = [im.contiguous() for im in scene["images"]]
    imgs_host = [torch.empty(im.shape, dtype=torch.float32).pin_memory() for im in imgs_dev]
    for h, d in zip(imgs_host, imgs_dev):
        h.copy_(d)
    bgrx = pkg.scene.box_downsample4(scene["bgr"])
    return scene, imgs_dev, imgs_host, bgrx


def cpu_baseline(pkg, cfg, evals_per_depthmap):
    """Single-threaded C restatement of cost + propagation + refinement (oracle/oracle_cpu.c) on a bounded
    sample: a 128x96 scene with the config's number of source views, init + 1 iteration."""
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    small = dict(W=128, H=96, n_images=cfg["V"] + 1, V=cfg["V"], fx=cfg["fx"] * 128.0 / cfg["W"], radius=cfg["radius"],
                 arc_deg=cfg["arc_deg"])
    sc = pkg.scene.make_scene(small)
    params = pkg.make_params(box=11, iterations=1, min_disparity=sc["min_disparity"], max_disparity=sc["max_disparity"])
    o = cb.CpuOracle(pkg._lib.TsarCamera, pkg._lib.TsarParams, sc["images"], cameras_to_struct(sc["cams"]), sc["subset"], params, sc["cam_f"])
    t = time.time()
    o.init_planes(SEED)
    o.iterate(1, SEED)
    dt = time.time() - t
    ev = o.evals()
    o.close()
    return {"value": (ev / dt) / evals_per_depthmap, "unit": "depthmaps/s", "cores": 1, "kind": "port",
            "sample": f"128x96 scene, V={cfg['V']}, init + 1 red/black iteration = {ev} pmCost evaluations in {dt:.1f} s "
                      f"({ev / dt / 1e6:.3f} M evals/s), scaled by {evals_per_depthmap} evaluations per depthmap",
            "host_cores_available": os.cpu_count()}


def dump_outputs(out_dir, norm4, confid, labels, n_sample=1 << 20):
    """What a caller of the per-view path receives, as float32 / float64 .npy files (31 MB at C2): depth, normals and
    confidence at n_sample pixels drawn with a fixed seed (the full C2 maps would be 127 MB), and the superpixel labels
    in full."""
    os.makedirs(out_dir, exist_ok=True)
    H, W = confid.shape
    idx = np.sort(np.random.RandomState(0).choice(H * W, min(n_sample, H * W), replace=False))
    n4 = norm4.reshape(H * W, 4)[idx]
    arrays = {"pixel_index": idx.astype(np.float64), "depth": n4[:, 3], "normals": n4[:, :3], "confidence": confid.reshape(-1)[idx],
              "superpixel_labels": labels.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


def run_ours(args):
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    L = pkg._lib
    rank, world, local = dist_setup(args.gpus)
    cfg = pkg.scene.CONFIGS[args.config]
    iters = 8
    scene, imgs_dev, imgs_host, bgrx = build_scene(pkg, args.config, rank, f"cuda:{local}")
    W, H, V = cfg["W"], cfg["H"], cfg["V"]
    params = pkg.make_params(box=args.blocksize, iterations=iters, n_best=1, cost_comb=1, min_disparity=scene["min_disparity"],
                             max_disparity=scene["max_disparity"])
    # our kernels run on a torch side stream made current below, so torch.cuda.Event brackets exactly them
    tstream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(tstream)
    eng = pkg.DepthmapEngine(local, stream=tstream.cuda_stream)
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    eng.set_views_device([t.data_ptr() for t in imgs_dev], W, H, cams, scene["subset"], cam_f=scene["cam_f"])
    eng.set_params(params)
    eng.set_regions(scene["region_text"], scene["region_norm4"])
    canny = torch.from_numpy(np.ascontiguousarray(scene["canny"], np.float32)).pin_memory().numpy()   # pinned: e2e uploads it every step
    eng.upload(L.F_CANNY, canny)            # region labels of the reference view (caller input, resident)

    def step_resident(seed):
        labels = eng.slic(bgrx)             # quarter-resolution colour image of the reference view
        eng.init_planes(seed)
        eng.iterate(iters, seed)
        eng.lrdiff(); eng.getview()
        eng.update_scale_2(); eng.update_scale(); eng.compute_disp()
        return labels

    n_evals = eng.eval_count(iters)
    for _ in range(args.warmup):
        step_resident(SEED)
    eng.launch_count(reset=True)
    eng.profile(True)
    barrier(world)
    # L2 rule: C2/C5 stream far more than the 126 MB L2 per step (views + state); for the small configs a 256 MB
    # buffer is overwritten between the timed steps, outside the per-step event pairs
    work_bytes = (cfg["n_images"] * 5 + 72) * W * H
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}") if work_bytes < (512 << 20) else None
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local, enabled=(rank == 0)) as clk:
        for k in range(args.steps):
            if flush is not None:
                flush.fill_(k)
            evs[k][0].record()
            labels = step_resident(SEED + 100 * k)
            evs[k][1].record()
        torch.cuda.synchronize()
    if args.dump_outputs and rank == 0 and args.steps > 0:
        dump_outputs(args.dump_outputs, eng.download(L.F_NORM4), eng.download(L.F_CONFID), labels)
    ms_local = sum(a.elapsed_time(b) for a, b in evs)
    barrier(world)
    ms = max_over_ranks(ms_local, world)
    launches = eng.launch_count(reset=True)
    chk_ms, chk_n = eng.profile_read()
    eng.profile(False)
    value = world * args.steps / (ms * 1e-3)

    # ---- end to end through the host API: pinned host images in, host results out, every step.  Two contexts on two
    # streams are driven by two host threads (ctypes releases the GIL), so the upload of the next reference view
    # overlaps the kernels of the current one -- what a multi-view driver does (SURVEY section 8e: ">= 2 streams").
    import concurrent.futures as cf
    host_np = [t.numpy() for t in imgs_host]
    lanes = []
    for lane in range(2):
        st = torch.cuda.Stream(device=local)
        e = pkg.DepthmapEngine(local, stream=st.cuda_stream)
        e.set_params(params)
        lanes.append(dict(eng=e, stream=st, n4=torch.empty((H, W, 4), dtype=torch.float32).pin_memory(),
                          cf=torch.empty((H, W), dtype=torch.float32).pin_memory()))

    def step_e2e(lane, seed):
        e = lane["eng"]
        labels = e.slic(bgrx)
        e.set_views(host_np, cams, scene["subset"], cam_f=scene["cam_f"])  # H2D of every view
        e.set_regions(scene["region_text"], scene["region_norm4"])
        e.upload(L.F_CANNY, canny)
        e.init_planes(seed)
        e.iterate(iters, seed)
        e.lrdiff(); e.getview()
        e.update_scale_2(); e.update_scale(); e.compute_disp()
        e.lib.tsar_download(e.h, L.F_NORM4, lane["n4"].numpy().ctypes.data, lane["n4"].numel() * 4)   # D2H
        e.lib.tsar_download(e.h, L.F_CONFID, lane["cf"].numpy().ctypes.data, lane["cf"].numel() * 4)
        return labels

    for lane in lanes:
        step_e2e(lane, SEED)
    barrier(world)
    t0 = time.perf_counter()
    def lane_worker(j):                     # one host thread per lane: a context is never used by two threads
        for k in range(j, args.steps, 2):
            step_e2e(lanes[j], SEED + 100 * k)

    with cf.ThreadPoolExecutor(2) as pool:
        for f in [pool.submit(lane_worker, j) for j in range(2)]:
            f.result()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    h2d = (V + 1) * W * H * 4 + bgrx.nbytes + canny.nbytes
    d2h = W * H * 20 + bgrx.shape[0] * bgrx.shape[1] * 4
    e2e = {"value": world * args.steps / e2e_s, "unit": "depthmaps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "pipelining": "2 contexts / 2 streams / 2 host threads per GPU"}
    launches_e2e = sum(l["eng"].launch_count() for l in lanes)

    if rank != 0:
        shutdown(world)
        return
    # ---- roofline of the dominant kernel (fused checkerboard propagation + refinement), timed live with CUDA events
    ffma_tf, mufu_g, tex_g = eng.peaks()
    evals_checker = (n_evals - V * W * H) / (2.0 * iters)           # pmCost evaluations per checkerboard launch
    avg_ms = chk_ms / max(chk_n, 1)
    n_samp = ((args.blocksize - 1) // 2 + 1) ** 2                   # S = (hRad + 1)^2 window samples, stride 2
    flops_eval = 40.0 * n_samp + 150.0                              # BASELINE.md section 3 (1590 at S = 36)
    achieved = evals_checker * flops_eval / (avg_ms * 1e-3) / 1e12
    traffic = None
    for tname in ("r02_dominant_kernel_dram_bytes.json", "r01_dominant_kernel_dram_bytes.json"):   # one ncu --set full capture per round
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(args.config)
            except Exception:
                traffic = None
            break
    peaks_file = {}
    try:
        peaks_file = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks_file.get("hbm_gbs", 6650.0)
    alg_bytes = (W * H / 2.0) * (4 * (1 + V) * 4 + 40)               # compulsory bytes of one launch (BASELINE.md section 3)
    roofline = {
        "bound": "fp32", "kernel": "pm_checker_kernel (fused red/black propagation + refinement)",
        "achieved": achieved, "peak": ffma_tf, "unit": "TFLOP/s", "frac": achieved / ffma_tf if ffma_tf else None,
        "peak_source": "FP32 FFMA issue microbenchmark measured live in this run (tsar_dbg_peaks; MEASURED_PEAKS.json has no FP32 entry); "
                       f"recorded with clocks in profiles/r02_fp32_peaks.json; nominal {FP32_NOMINAL_TFLOPS} TFLOP/s",
        "frac_of_nominal": achieved / FP32_NOMINAL_TFLOPS,
        "algorithmic_flops_per_launch": evals_checker * flops_eval, "avg_launch_ms": avg_ms, "launches_timed": chk_n,
        "kernel_share_of_step": chk_ms / ms_local if ms_local else None,
        "gevals_per_s": evals_checker / (avg_ms * 1e-3) / 1e9,
        "tex_gsamples_per_s": evals_checker * n_samp / (avg_ms * 1e-3) / 1e9, "tex_peak_gsamples_per_s": tex_g,
        "tex_frac": (evals_checker * n_samp / (avg_ms * 1e-3) / 1e9) / tex_g if tex_g else None,
        "mufu_peak_gops_measured": mufu_g, "mufu_peak_gops_nominal": 148 * 16 * 1.965,
        # SFU view (SURVEY section 8d): 4*S + 12 MUFU per evaluation as written in pmCost (two rcp, one rsq, one ex2 per
        # sample); this kernel issues S + 12 (one reciprocal per sample, reference-image terms hoisted)
        "sfu": {"as_written_gops": evals_checker * (4 * n_samp + 12) / (avg_ms * 1e-3) / 1e9,
                "executed_gops": evals_checker * (n_samp + 12) / (avg_ms * 1e-3) / 1e9, "peak_gops": mufu_g,
                "frac_as_written": evals_checker * (4 * n_samp + 12) / (avg_ms * 1e-3) / 1e9 / mufu_g if mufu_g else None,
                "frac_executed": evals_checker * (n_samp + 12) / (avg_ms * 1e-3) / 1e9 / mufu_g if mufu_g else None},
        "hbm": {"bound": "hbm", "achieved": alg_bytes / (avg_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": alg_bytes / (avg_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks_file else "fallback"},
        "traffic": traffic,
    }
    if args.blocksize == 11:
        # texture-pipe view (the tighter bound, DESIGN.md section 4.4): one wavefront per clock per SM; 9.64 wavefronts per
        # warp-wide bilinear fetch measured by ncu (profiles/r01_variants_C2.json, independent of locality)
        sm_count, clk_hz, wf_per_fetch = 148, 1.965e9, 9.64   # profiles/r02_ncu_full_pm_checker_C2.csv: 4483.5 M wavefronts / 465.3 M fetches
        tex_bound_ms = evals_checker * n_samp / 32.0 * wf_per_fetch / (sm_count * clk_hz) * 1e3
        roofline["texture"] = {"bound": "texture wavefronts", "bound_ms": tex_bound_ms, "achieved_ms": avg_ms,
                               "frac": tex_bound_ms / avg_ms if avg_ms else None, "wavefronts_per_fetch": wf_per_fetch,
                               "ncu_data_pipe_pct_of_sustained_peak": 91.5}
    out = {
        "metric": "depthmaps/s", "value": value, "unit": "depthmaps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "ours",
        "config": config_dict(args.config, cfg, iters, args.blocksize, world),
        "gevals_per_s": world * args.steps * n_evals / (ms * 1e-3) / 1e9, "evals_per_depthmap": n_evals,
        "roofline": roofline, "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches), "gpu_launches_e2e": int(launches_e2e),
    }
    # executed evaluations counted on the device (debug counter, tools/gpu_cand_stats.py) next to the as-written closed form
    spath = os.path.join(ROOT, "profiles", f"r02_candidate_stats_{args.config}.json")
    if os.path.exists(spath) and args.blocksize == 11:
        try:
            st = json.load(open(spath))
            out["evals_executed"] = {"as_written_closed_form": st["closed_form_evaluations"], "executed_device_counter": st["executed_evaluations_as_written"],
                                     "distinct_hypotheses_only": st["executed_evaluations_skipping_duplicates"],
                                     "roofline_frac_on_executed": roofline["frac"] * st["executed_evaluations_as_written"] / st["closed_form_evaluations"]
                                     if roofline["frac"] else None, "source": os.path.relpath(spath, ROOT)}
        except Exception:
            pass
    if world == 1 and not args.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_baseline(pkg, cfg, n_evals)
        except Exception as e:  # the baseline must not take the bench down
            out["cpu_baseline"] = {"error": repr(e)}
    emit(out)
    shutdown(world)


PRODUCT_CONFIGS = {"C3": "C3", "C4": "C4seq", "C3small": "C3small"}


def run_product(args):
    """BASELINE configs 3 and 4: a FIXED set of reference views (C3: 38 cameras on two arcs, C4: a 300-frame sequence; each
    view paired with its 10 nearest cameras) through the product's multi-view driver (tsar_cli -all_views: resident image
    pool, shared view queue, pipelined lanes) with image decoding and .dmb writing INSIDE the timed region.  Strong scaling:
    the view set is sharded round-robin over the ranks, no collective on the data path.  A step = one pass over the set."""
    import shutil
    import tempfile
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    rank, world, local = dist_setup(args.gpus)
    name = PRODUCT_CONFIGS[args.config]
    cfg = pkg.scene.CONFIGS[name]
    base = os.environ.get("TSAR_BENCH_TMP") or tempfile.gettempdir()
    root = os.path.join(base, f"tsar_bench_{name}_{os.environ.get('MASTER_PORT', '0')}") + "/"
    t_gen = time.perf_counter()
    if rank == 0:                                # the dataset is generated once, outside the timed region
        shutil.rmtree(root, ignore_errors=True)
        pkg.cli.write_rig_dataset(name, root, backend="torch", device=f"cuda:{local}")
    barrier(world)
    t_gen = time.perf_counter() - t_gen
    argv = ["-all_views", "-mslp_folder", root, "-images_folder", root + "images/", "-krt_file", "x", "-no_display", "--cam_scale=1",
            "--iterations=8", f"--blocksize={args.blocksize}", "--cost_comb=best_n", "--n_best=1", f"--seed={SEED}", f"--lanes={args.lanes}",
            f"--io_threads={args.io_threads}"]
    opt = pkg.cli.parse_args(argv)
    os.environ["LOCAL_RANK"] = str(local)
    results = []
    for _ in range(max(args.warmup, 1) if args.warmup else 0):
        # warm-up: two views per rank; the driver is persistent (contexts and pinned buffers stay alive between passes)
        pkg.cli.run_all_views(dict(opt, views_per_rank=2), root, quiet=True, persistent=True)
    secs = []
    with ClockSampler(local, enabled=(rank == 0)) as clk:
        for k in range(args.steps):
            shutil.rmtree(os.path.join(root, "APD"), ignore_errors=True) if rank == 0 else None
            barrier(world)
            t0 = time.perf_counter()
            res = pkg.cli.run_all_views(opt, root, quiet=True, persistent=True)
            torch.cuda.synchronize()
            dt_local = time.perf_counter() - t0
            barrier(world)
            secs.append(max_over_ranks(dt_local, world))
            results.append(res)
    n_views = cfg["n_images"]
    total_s = sum(secs)
    value = args.steps * n_views / total_s
    mine_views = results[-1]["views"]
    host = results[-1]["host_seconds"]
    if rank == 0:
        per_gpu_views = -(-n_views // world)
        out = {
            "metric": "depthmaps/s", "value": value, "unit": "depthmaps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_s * 1e3 / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "ours",
            "config": {"workload": f"{args.config}: fixed set of {n_views} reference views {cfg['W']}x{cfg['H']}, each with its {cfg['V']} nearest "
                                   f"cameras ({cfg['rig']} rig), blocksize {args.blocksize}, 8 iterations, n_best 1; whole TSAR flow per view "
                                   f"(weak-texture detector, gSLICr, checkerboard PatchMatch, L/R check, confidence, region RANSAC, depth "
                                   f"completion) through the -all_views driver",
                       "timing": "wall clock per pass over the view set, max over ranks; PNG decoding, H2D, kernels, D2H and .dmb writes inside the timed region; "
                                 f"inputs_larger_than_l2 ({n_views * cfg['W'] * cfg['H'] * 4 / 1e6:.0f} MB image pool)",
                       "parallelism": f"views sharded round-robin over {world} GPU(s), {args.lanes} pipelined contexts per GPU, no collective on the data path",
                       "output_folder": base},
            "e2e": {"value": value, "unit": "depthmaps/s", "h2d_bytes_per_step": int(n_views * cfg["W"] * cfg["H"] * 4),
                    "d2h_bytes_per_step": int(n_views * cfg["W"] * cfg["H"] * 20), "note": "this configuration IS the end-to-end product path (files in, files out)"},
            "gpu_launches": int(sum(r["gpu_launches"] for r in results)),
            "limiter": {"views_per_gpu_max": per_gpu_views, "imbalance_bound": n_views / (world * per_gpu_views),
                        "rank0_views": mine_views, "rank0_host_seconds_summed_over_threads": host,
                        "rank0_bytes_decoded": results[-1]["bytes_decoded"], "rank0_bytes_written": results[-1]["bytes_written"],
                        "per_pass_seconds": secs, "dataset_generation_s": t_gen, "host_cores": os.cpu_count()},
            "clocks": clk.summary(),
        }
        emit(out)
    pkg.cli.release_lanes()
    barrier(world)
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
    shutdown(world)


def run_reference(args):
    """The reference's own kernels (oracle/_ref) on the same workload.  The reference's execution model is one process
    per reference view on one GPU (scripts/pipes.sh:30-49), so under torchrun EVERY rank runs its own stream of reference
    views on its own GPU, exactly like our arm; the time is the max over ranks and rank 0 prints the line.  Nothing of
    libtsar_b200.so is loaded here: struct layouts and the closed-form evaluation count are pure Python."""
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    from oracle import ref_binding as rb
    rank, world, local = dist_setup(args.gpus)
    if not rb.available("asis"):
        if rank == 0:
            emit({"impl": "reference", "unavailable": "oracle/_ref/libtsar_ref.so missing (run `make oracle` where the reference checkout exists)"})
        shutdown(world)
        return
    cfg = pkg.scene.CONFIGS[args.config]
    iters = 8
    scene, imgs_dev, imgs_host, bgrx = build_scene(pkg, args.config, rank, f"cuda:{local}")
    del imgs_dev
    torch.cuda.empty_cache()
    from tsar_mvs_b200.engine import cameras_to_struct
    cams = cameras_to_struct(scene["cams"])
    params = pkg.make_params(box=args.blocksize, iterations=iters, n_best=1, cost_comb=1, min_disparity=scene["min_disparity"],
                             max_disparity=scene["max_disparity"])
    ref = rb.RefEngine(pkg._lib.TsarCamera, pkg._lib.TsarParams, variant="asis")
    ref.create([t.numpy() for t in imgs_host], cams, scene["subset"], params, scene["cam_f"])
    ref.set_regions(scene["region_text"], scene["region_norm4"])
    ref.upload(rb.F_CANNY, scene["canny"])

    def step(seed):
        rb.ref_slic(bgrx)
        ref.init_planes(seed)
        ref.iterate(iters, seed)
        ref.lrdiff(); ref.getview()
        ref.update_scale_2(); ref.update_scale(); ref.compute_disp()

    for _ in range(args.warmup):
        step(SEED)
    barrier(world)
    # the reference launches on the legacy default stream, which is torch's current stream here
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local, enabled=(rank == 0)) as clk:
        e0.record()
        for k in range(args.steps):
            step(SEED + 100 * k)
        e1.record()
        torch.cuda.synchronize()
    ms_local = e0.elapsed_time(e1)
    barrier(world)
    ms = max_over_ranks(ms_local, world)
    ref.close()
    torch.cuda.synchronize()
    if rank != 0:
        shutdown(world)
        return
    value = world * args.steps / (ms * 1e-3)
    n_evals = pkg.counts.eval_count(cfg["W"], cfg["H"], cfg["V"], iters, scene["max_disparity"])
    out = {
        "metric": "depthmaps/s", "value": value, "unit": "depthmaps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "reference",
        "config": config_dict(args.config, cfg, iters, args.blocksize, world),
        "reference_note": "reference CUDA kernels rebuilt for sm_100a (gipuma.cu + gSLICr unmodified), managed memory, device sync after "
                          "every kernel, warm (pages resident after warm-up); one process + one GPU per reference-view stream as in "
                          "scripts/pipes.sh; the reference has no CPU path",
        "gevals_per_s": world * args.steps * n_evals / (ms * 1e-3) / 1e9, "evals_per_depthmap": n_evals,
        "cpu_baseline": {"value": value, "unit": "depthmaps/s", "cores": 0, "kind": "reference",
                         "sample": f"{args.steps} full depthmaps of the workload per GPU on {world} B200 (the reference implements this path in CUDA only)"},
        "e2e": {"value": value, "unit": "depthmaps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "clocks": clk.summary(),
    }
    emit(out)
    shutdown(world)


if __name__ == "__main__":
    a = parse()
    capture_stdout()
    driver = a.config in PRODUCT_CONFIGS and a.mode != "engine"
    if a.mode == "driver" and a.config not in PRODUCT_CONFIGS:
        sys.exit(f"--mode driver needs one of {sorted(PRODUCT_CONFIGS)}")
    if a.dump_outputs and (a.impl == "reference" or driver):
        sys.exit("--dump-outputs writes the outputs of the per-view path (--impl ours, per-view configs or --mode engine)")
    if a.impl == "reference" and driver:
        if int(os.environ.get("RANK", "0")) == 0:
            emit({"impl": "reference", "unavailable": "the reference has no multi-view driver (one process per view, scripts/pipes.sh); "
                                                      "its per-view rate is measured by --config C2 --impl reference"})
    elif a.impl == "reference":
        run_reference(a)
    elif driver:
        run_product(a)
    else:
        run_ours(a)
