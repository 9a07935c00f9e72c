"""CPU-only tests (pytest -m "not gpu"): the C oracle against golden vectors produced by the reference's own
kernels on a B200 (tests/golden/, tools/make_golden.py), the host-side logic, and the C ABI surface.
No compute call is made on the CUDA library here (no GPU in this environment)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import parity_common as pc

ROOT = pc.ROOT
GOLD = os.path.join(ROOT, "tests", "golden")
SEED = 20240601


@pytest.fixture(scope="module")
def tiny(pkg):
    return pkg.scene.make_scene("tiny")


@pytest.fixture(scope="module")
def oracle(pkg, tiny):
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    params = pkg.make_params(box=11, iterations=3, min_disparity=tiny["min_disparity"], max_disparity=tiny["max_disparity"])
    o = cb.CpuOracle(pkg._lib.TsarCamera, pkg._lib.TsarParams, tiny["images"], cameras_to_struct(tiny["cams"]), tiny["subset"],
                     params, tiny["cam_f"])
    yield o
    o.close()


# ---- the C ABI ---------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "tsar_b200.h")).read()
    declared = set(re.findall(r"\b(tsar_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"tsar_status", "tsar_field"}
    assert len(declared) >= 30
    lib = C.CDLL(pkg._lib.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, f"declared in include/tsar_b200.h but not exported: {missing}"
    assert set(pkg._lib.EXPORTS) <= declared


def test_library_exports_the_reference_entry_points(pkg):
    """gipuma.h:2-5: `int firstcuda(GlobalState&)` ... with the reference's C++ linkage (global namespace), so the
    reference's main.cpp links against the library unchanged."""
    out = subprocess.run("nm -D --defined-only '%s' | c++filt" % pkg._lib.LIB_PATH, shell=True, capture_output=True, text=True).stdout
    for fn in ("firstcuda", "sliccuda", "fakecuda", "fillcuda"):
        assert f" T {fn}(GlobalState&)" in out, fn


def test_no_cpu_fallback(pkg):
    """Without a GPU the product path must fail loudly, not fall back to the oracle."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg.TsarError):
        pkg.DepthmapEngine(0)
    src = "".join(open(os.path.join(ROOT, "tsar-mvs_b200", f)).read() for f in os.listdir(os.path.join(ROOT, "tsar-mvs_b200")) if f.endswith(".py"))
    assert "oracle" not in src.replace("the oracle", "").replace("oracle's", ""), "product package must not import oracle/"


def test_struct_sizes_match_header(pkg):
    code = '#include "include/tsar_b200.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu\\n",sizeof(tsar_camera),sizeof(tsar_params),sizeof(tsar_slic_settings));return 0;}'
    exe = os.path.join(ROOT, "build", "sizes_test")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", ROOT, "-o", exe], input=code.encode(), cwd=ROOT, check=True)
    sizes = [int(v) for v in subprocess.run([exe], capture_output=True, text=True).stdout.split()]
    assert sizes == [C.sizeof(pkg._lib.TsarCamera), C.sizeof(pkg._lib.TsarParams), C.sizeof(pkg._lib.TsarSlicSettings)]


# ---- the scene generator ---------------------------------------------------------------------------------
def test_scene_matches_golden_images(tiny):
    g = np.load(os.path.join(GOLD, "tiny_scene.npz"))
    imgs = np.stack(tiny["images"]).astype(np.uint8)
    assert (np.abs(imgs.astype(int) - g["images"].astype(int)) <= 1).all()   # sin() last-bit differences at most
    assert (imgs != g["images"]).mean() < 1e-3
    assert np.allclose(tiny["gt_depth"], g["gt_depth"], rtol=1e-6)


def test_cameras_are_photo_consistent(pkg):
    """The plane-induced homography built from the camera fields (SURVEY 3.4) maps a reference pixel onto the
    pixel of the same 3-D point in a source view: checks make_cameras against the scene renderer."""
    s = pkg.scene.make_scene("tiny")
    ref, src = s["cams"][0], s["cams"][2]
    planes = s["region_norm4"]  # per facet (n, d) in the reference frame (slightly perturbed) -> use exact ones
    from tsar_mvs_b200.scene import Scene, CONFIGS
    cfg = CONFIGS["tiny"]
    sc = Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"])
    exact = sc.region_planes(ref)
    ys, xs = np.mgrid[8:56:6, 8:88:6]
    for x, y in zip(xs.ravel(), ys.ravel()):
        lab = s["labels"][y, x]
        n, d = exact[lab][:3], exact[lab][3]
        H = np.asarray(src["K"]) @ (np.asarray(src["R"]) - np.outer(src["t4"], n) / d) @ np.asarray(ref["K_inv"])
        q = H @ np.array([x, y, 1.0])
        q = q[:2] / q[2]
        # same 3-D point through explicit geometry
        X = np.asarray(ref["K_inv"]) @ np.array([x, y, 1.0]) * s["gt_depth"][y, x]
        p = np.asarray(src["K"]) @ (np.asarray(src["R"]) @ X + np.asarray(src["t4"]))
        assert np.allclose(q, p[:2] / p[2], atol=1e-3), (x, y, q, p[:2] / p[2])


def test_reference_reordering(pkg):
    a = pkg.scene.make_scene("tiny")
    b = pkg.scene.make_scene("tiny", ref_index=2)
    assert np.array_equal(b["images"][0], a["images"][2])
    assert np.allclose(b["cams"][0]["R"], np.eye(3), atol=1e-12) and np.allclose(b["cams"][0]["t4"], 0, atol=1e-12)


# ---- the C oracle pinned against the reference build's output ---------------------------------------------
def test_oracle_xorwow_and_init_planes_match_reference_build(oracle):
    """Init planes depend on cuRAND XORWOW streams (curand_init(seed, y, x)), Marsaglia sampling, the view vector
    and getD_cu: all IEEE operations except one rsqrtf whose result only decides a sign.  Bit-exact bar."""
    g = np.load(os.path.join(GOLD, "tiny_steps.npz"))
    oracle.init_planes_only(SEED)
    mine = oracle.planes()
    eq = pc.bits_equal(mine, g["init_norm4"]).all(axis=-1)
    assert eq.mean() > 0.999, f"only {eq.mean():.4f} of the init planes are bit-identical"


def test_oracle_texture_model_matches_hardware_samples(oracle, tiny):
    g = np.load(os.path.join(GOLD, "tiny_tex.npz"))
    img = tiny["images"][1]
    got = np.array([oracle.tex(img, x, y) for x, y in g["xy"][:3000]], np.float32)
    assert np.array_equal(got, g["out"][:3000])


def test_oracle_texture_model_tie_rule(oracle, tiny):
    """Hardware samples at coordinates i + 0.5 + k/512: every step of the 8-bit weight grid and every exact tie between two
    steps (k odd), where the rule -- round half up -- cannot be seen with random coordinates (tools/gpu_tex_ties.py pinned
    it on a B200: half-up 100 %, half-to-even 53 % on 131 000 ties)."""
    g = np.load(os.path.join(GOLD, "tiny_tex_ties.npz"))
    img = tiny["images"][1]
    got = np.array([oracle.tex(img, x, y) for x, y in g["xy"]], np.float32)
    assert np.array_equal(got, g["out"])


def test_oracle_cost_matches_reference_build(oracle, tiny):
    """pmCostMultiview on 2000 (pixel, plane) pairs.  Not bit-reproducible on a CPU by construction (MUFU.EX2 inside
    CUDA's expf, <= 2 ulp on every bilateral weight).  Tolerance: 5e-5 absolute on a cost in [0, 2] where the window is
    textured; inside the textureless facet (grey levels 128/129) the variance is a difference of two numbers ~16384,
    so the cost is ill-conditioned at the 1e-2 level for ANY fp32 implementation: 5e-2 there."""
    g = np.load(os.path.join(GOLD, "tiny_eval.npz"))
    yy, xx = np.mgrid[0:tiny["H"], 0:tiny["W"]]
    flat = tiny["labels"] == 4
    from scipy.ndimage import binary_dilation
    near_flat = binary_dilation(flat, iterations=6)[g["xy"][:, 1], g["xy"][:, 0]]
    for key, wrapper in (("cost", True), ("cost_kernel_rounding", False)):
        c, bv, ratio = oracle.eval_planes(g["xy"], g["planes"], wrapper_rounding=wrapper)
        d = np.abs(c.astype(np.float64) - g[key])
        assert d[~near_flat].max() < 5e-5, (key, d[~near_flat].max())
        assert d[near_flat].max() < 5e-2, (key, d[near_flat].max())
        assert np.median(d) < 2e-6
    c, bv, ratio = oracle.eval_planes(g["xy"], g["planes"], wrapper_rounding=True)
    assert (bv == g["beview"]).mean() > 0.995   # ties between views can flip at the 1e-7 level


def test_oracle_half_steps_match_reference_build(oracle):
    """One black propagation + one black refinement from the reference build's initial state."""
    g = np.load(os.path.join(GOLD, "tiny_steps.npz"))
    oracle.set_state(g["init_norm4"], g["init_cost"])
    oracle.spatial(0)
    same = pc.bits_equal(oracle.planes(), g["sp_norm4"]).all(axis=-1)
    assert same.mean() > 0.97, same.mean()          # a 1e-7 cost difference flips a few accept decisions
    dc = np.abs(oracle.costs() - g["sp_cost"])[same]
    assert np.quantile(dc, 0.9) < 2e-5 and dc.max() < 5e-2   # the max sits in the ill-conditioned textureless facet
    oracle.set_state(g["sp_norm4"], g["sp_cost"])
    oracle.refine(0, SEED + 1)
    # refined normals pass through rsqrtf (MUFU.RSQ on the GPU, 1/sqrtf here): equal to a few ulp, not bit-equal
    close = np.isclose(oracle.planes(), g["pr_norm4"], rtol=2e-5, atol=2e-6).all(axis=-1)
    assert close.mean() > 0.95, close.mean()


def test_oracle_full_sequence_statistics(oracle, tiny):
    g = np.load(os.path.join(GOLD, "tiny_full.npz"))
    oracle.init_planes(SEED)
    oracle.iterate(3, SEED)
    out = oracle.output()
    a = pc.output_agreement(out, g["out"])
    assert a["frac_depth_ok"] > 0.80, a              # chaotic after 3 iterations of a 96x64 scene: statistical bar
    assert abs(pc.gt_agreement(out, tiny)["frac_within_1pct_all"] - pc.gt_agreement(g["out"], tiny)["frac_within_1pct_all"]) < 0.1


# ---- host logic ------------------------------------------------------------------------------------------
def test_dmb_roundtrip(tmp_path, pkg):
    from tsar_mvs_b200 import dmb
    rng = np.random.RandomState(0)
    d, n = rng.rand(7, 9).astype(np.float32), rng.rand(7, 9, 3).astype(np.float32)
    dmb.write_dmb(tmp_path / "d.dmb", d)
    dmb.write_dmb(tmp_path / "n.dmb", n)
    assert np.array_equal(dmb.read_dmb(tmp_path / "d.dmb"), d) and np.array_equal(dmb.read_dmb(tmp_path / "n.dmb"), n)
    raw = open(tmp_path / "n.dmb", "rb").read()
    assert np.frombuffer(raw[:16], np.int32).tolist() == [1, 7, 9, 3] and len(raw) == 16 + 7 * 9 * 3 * 4
    open(tmp_path / "bad.dmb", "wb").write(raw[:40])
    with pytest.raises(ValueError):
        dmb.read_dmb(tmp_path / "bad.dmb")


def test_view_sharding_partitions(pkg):
    from tsar_mvs_b200 import shard
    for n, w in ((38, 8), (300, 8), (5, 8), (0, 2), (7, 1)):
        parts = [shard.views_for_rank(n, r, w) for r in range(w)]
        assert sorted(sum(parts, [])) == list(range(n))
        assert max(map(len, parts)) - min(map(len, parts)) <= 1
        blocks = [shard.block_for_rank(n, r, w) for r in range(w)]
        assert sum(blocks, []) == list(range(n))                                  # contiguous, in order
        assert max(map(len, blocks)) - min(map(len, blocks)) <= 1
    with pytest.raises(ValueError):
        shard.views_for_rank(3, 2, 2)
    with pytest.raises(ValueError):
        shard.block_for_rank(3, 2, 2)
    # blocks keep a rank's image pool small: 38 courtyard views on 8 ranks, 10 nearest neighbours each
    K, Rs, Cs, nb = pkg.scene.make_rig(pkg.scene.CONFIGS["C3"])
    need_block = max(len(set(b) | {j for i in b for j in nb[i]}) for b in (shard.block_for_rank(38, r, 8) for r in range(8)))
    need_rr = max(len(set(b) | {j for i in b for j in nb[i]}) for b in (shard.views_for_rank(38, r, 8) for r in range(8)))
    assert need_block <= 26 and need_rr >= 36


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    pkg = g.load_package()
    from tsar_mvs_b200 import shard
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    local = shard.run_sharded(7, rank, world, lambda v: np.full((2, 2), v, np.float32))
    allres = shard.gather_results(local, world)
    dist.barrier()
    if rank == 0:
        q.put(sorted(allres.keys()) == list(range(7)) and all((allres[v] == v).all() for v in allres))
    dist.destroy_process_group()


def test_sharded_run_world_size_2_gloo():
    """The N > 1 path on CPU: two ranks, views sharded round-robin, results gathered on rank 0 (gloo)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    ok = q.get(timeout=120)
    for p in ps:
        p.join(timeout=60)
    assert ok and all(p.exitcode == 0 for p in ps)


def test_bench_reference_arm_contract():
    """bench.py parses; --impl reference without a GPU is out of scope here (needs the B200), but the ratio inputs
    (metric, unit, higher_is_better) must be identical strings in both arms."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    # three emitters: our arm, the reference arm, the multi-view product driver (--config C3 / C4)
    assert src.count('"metric": "depthmaps/s"') == 3 and src.count('"higher_is_better": True') == 3
    assert src.count('"config": config_dict(args.config, cfg, iters, args.blocksize, world)') == 2   # identical dicts in both arms
    ref_arm = src[src.index("def run_reference(args):"):src.index('if __name__ == "__main__":')]
    assert "DepthmapEngine" not in ref_arm and "_lib.load" not in ref_arm   # the product library stays out of the reference arm


# Layouts of the reference's types that include/tsar_gipuma_abi.h and include/tsar_gslicr_abi.h mirror: per type, the mirror's
# name and {reference member: mirror member}.  tests/golden/abi_layout.json stores sizeof, alignof and every offsetof as the
# reference's headers give them; the mirrors are compiled alone against those numbers, and the reference's headers are
# compiled against them too where a checkout of the reference is named by TSAR_REFERENCE_DIR.
GIPUMA_ABI_FIELDS = {
    "Camera_cu": "P P_col34 P_inv M_inv R R_orig R_orig_inv t4 C4 fx fy f alpha baseline reference depthMin depthMax id K K_inv",
    "CameraParameters_cu": "f rectified cameras idRef cols rows viewSelectionSubset viewSelectionSubsetNumber",
    "LineState": "norm4 c depth fakedepth resize4 canny cenxi cenyi nein neip nump eacp ranp pind borlen depdif scale ransa "
                 "text XYZ ratio beview lrdiff confid ranumax size n s l",
    "AlgorithmParameters": "algorithm max_disparity min_disparity box_hsize box_vsize tau_color tau_gradient alpha gamma "
                           "border_value iterations color_processing dispTol normTol census_epsilon self_similarity_n cam_scale "
                           "num_img_processed costThresh good_factor n_best cost_comb viewSelection depthMin depthMax min_angle "
                           "max_angle no_texture_sim no_texture_per max_views cols rows thres",
    "GlobalState": "cameras lines cannylines cs params col row imgs cuArray",
}
GSLICR_ABI_FIELDS = {
    "gSLICr::objects::settings": ("tsar_gslicr_abi::SettingsMirror", {
        "img_size": "img_w", "no_segs": "no_segs", "spixel_size": "spixel_size", "no_iters": "no_iters", "coh_weight": "coh_weight",
        "do_enforce_connectivity": "do_enforce_connectivity", "color_space": "color_space", "seg_method": "seg_method"}),
    "ORUtils::Image<int>": ("tsar_gslicr_abi::ImageMirror", {
        "isAllocated_CPU": "isAllocated_CPU", "data_cpu": "data_cpu", "data_cuda": "data_cuda", "dataSize": "dataSize", "noDims": "dims_x"}),
}
# values of the reference's gSLICr headers the shim relies on without a mirror (the enums it reads as ints, the class size)
GSLICR_REFERENCE_VALUES = ("sizeof(gSLICr::engines::core_engine)", "gSLICr::CIELAB", "gSLICr::GIVEN_NUM", "gSLICr::GIVEN_SIZE")


def _abi_golden():
    import json
    return json.load(open(os.path.join(GOLD, "abi_layout.json")))


def _reference_dir(probe):
    ref = os.environ.get("TSAR_REFERENCE_DIR")
    return ref if ref and os.path.exists(os.path.join(ref, probe)) else None


def _layout(tmp_path, headers, include_dirs, types, values=()):
    """Compiles and runs a host program printing {label: [sizeof, alignof, {member label: offsetof}]} for
    types = {label: (C++ type, {member label: member})}, and {expression: value} for values."""
    import json
    q = '\\"'
    out = []
    for label, (ty, members) in types.items():
        fmt = ", ".join(f"{q}{m}{q}: %zu" for m in members)
        args = "".join(f", (size_t)offsetof({ty}, {m})" for m in members.values())
        out.append(f'std::printf("{q}{label}{q}: [%zu, %zu, {{{fmt}}}], ", sizeof({ty}), alignof({ty}){args});')
    for v in values:
        out.append(f'std::printf("{q}{v}{q}: %zu, ", (size_t)({v}));')
    src = "\n".join([f'#include "{h}"' for h in headers] + ["#include <cstddef>", "#include <cstdio>", "int main() {", 'std::printf("{");']
                    + out + ['std::printf("}\\n");', "return 0;", "}"])
    cu = tmp_path / "layout.cu"
    cu.write_text(src)
    exe = str(tmp_path / "layout")
    inc = sum((["-I", d] for d in include_dirs + [os.path.join(ROOT, "include")]), [])
    r = subprocess.run(["/usr/local/cuda/bin/nvcc", "-std=c++14", "-w", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-Wno-invalid-offsetof",
                        str(cu), "-o", exe] + inc, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    text = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.strip()
    return json.loads(text[:-3] + "}" if text.endswith(", }") else text)


def test_abi_layout_matches_reference(tmp_path):
    """include/tsar_gipuma_abi.h against the reference's own headers (globalstate.h and what it includes): sizeof, alignof
    and every field offset of the five types, against the stored numbers and, where the checkout exists, against the
    headers themselves."""
    want = _abi_golden()["gipuma"]
    mirror = {t: (f"tsar_abi::{t}", {f: f for f in fs.split()}) for t, fs in GIPUMA_ABI_FIELDS.items()}
    assert _layout(tmp_path, ["tsar_gipuma_abi.h"], [], mirror) == want
    ref = _reference_dir("globalstate.h")
    if ref:
        theirs = {t: (f"::{t}", {f: f for f in fs.split()}) for t, fs in GIPUMA_ABI_FIELDS.items()}
        assert _layout(tmp_path, ["globalstate.h"], [os.path.join(ROOT, "oracle", "stubs"), ref], theirs) == want


def test_gslicr_shim_layout_matches_reference(tmp_path, pkg):
    """include/tsar_gslicr_abi.h against the reference's gSLICr / ORUtils headers (settings, Image<T>), and the drop-in
    class members exported under the reference's mangled names (gSLICr_core_engine.h:11-33)."""
    out = subprocess.run("nm -D --defined-only '%s' | c++filt" % pkg._lib.LIB_PATH, shell=True, capture_output=True, text=True).stdout
    for member in ("core_engine(gSLICr::objects::settings const&)", "~core_engine()",
                   "Process_Frame(ORUtils::Image<ORUtils::Vector4<unsigned char> >*, GlobalState*)", "Get_Seg_Res()",
                   "Draw_Segmentation_Result(ORUtils::Image<ORUtils::Vector4<unsigned char> >*)", "Write_Seg_Res_To_PGM(char const*)"):
        assert f" T gSLICr::engines::core_engine::{member}" in out, member
    golden = _abi_golden()
    mirror = {t: (m, {a: b for a, b in fields.items()}) for t, (m, fields) in GSLICR_ABI_FIELDS.items()}
    assert _layout(tmp_path, ["tsar_gslicr_abi.h"], [], mirror) == golden["gslicr"]
    assert golden["gslicr_reference_values"]["sizeof(gSLICr::engines::core_engine)"] == C.sizeof(C.c_void_p)   # one pointer
    ref = _reference_dir(os.path.join("gSLICr_Lib", "gSLICr.h"))
    if ref:
        theirs = {t: (t, {a: a for a in fields}) for t, (_, fields) in GSLICR_ABI_FIELDS.items()}
        got = _layout(tmp_path, ["gSLICr_Lib/gSLICr.h"], [os.path.join(ROOT, "oracle", "stubs"), ref], theirs, GSLICR_REFERENCE_VALUES)
        assert {t: got[t] for t in theirs} == golden["gslicr"]
        assert {v: got[v] for v in GSLICR_REFERENCE_VALUES} == golden["gslicr_reference_values"]


def test_cli_flag_parsing_matches_run_scripts(pkg):
    """The command line the reference's scripts build (scripts/pipes.sh:45), incl. its empty and unknown flags."""
    from tsar_mvs_b200 import cli
    argv = ("00000003.jpg 00000000.jpg 00000001.jpg -mslp_folder ./data/TRAIN/pipes/ -images_folder data/TRAIN/pipes/images/ "
            "-krt_file data/x.txt -output_folder results/pipes/ -no_display --cam_scale=1 --iterations=8 --blocksize=11 "
            "--cost_gamma=10 --cost_comb=best_n --n_best=1 --min_angle= --max_angle= --bogus=3").split()
    o = cli.parse_args(argv)
    assert o["images"] == ["00000003.jpg", "00000000.jpg", "00000001.jpg"]
    assert (o["blocksize"], o["iterations"], o["n_best"], o["cost_comb"], o["cam_scale"]) == (11, 8, 1, 1, 1.0)
    assert o["mslp_folder"] == "./data/TRAIN/pipes/" and o["no_display"] is True


def test_dataset_readers_roundtrip(tmp_path, pkg, tiny):
    """cams/<id>_cam.txt and pair.txt as the reference reads them (fileIoUtils.h:111-163, main.cpp:1351-1376)."""
    from tsar_mvs_b200 import cli, scene
    sc, names = cli.write_synthetic_dataset("tiny", str(tmp_path))
    Ks, Rs, ts = [], [], []
    for n in names:
        K, R, t, dmin, dmax = cli.read_cam_txt(str(tmp_path / "cams" / f"{n[:8]}_cam.txt"))
        Ks.append(K); Rs.append(R); ts.append(t)
    cams = scene.cameras_from_krt(Ks, Rs, ts, dmin, dmax)
    for a, b in zip(cams, tiny["cams"]):
        for k in ("K", "R", "t4", "M_inv", "C4", "P_col34", "R_orig"):
            assert np.array_equal(np.asarray(a[k], np.float32), np.asarray(b[k], np.float32)), k
    # reference view = image 2: the list is [2, 0, 1, 3]; pair.txt lists neighbours 0, 1, 3 -> list positions 1, 2, 3
    assert cli.read_pair_subset(str(tmp_path / "pair.txt"), 2) == [1, 2, 3]
    assert cli.read_pair_subset(str(tmp_path / "pair.txt"), 0) == [1, 2, 3]
    assert cli.read_pair_neighbours(str(tmp_path / "pair.txt"), 2) == [0, 1, 3]
    assert cli.parse_args(["-all_views", "-mslp_folder", "x/"])["all_views"] is True
    import cv2
    im = cv2.imread(str(tmp_path / "images" / names[1]), cv2.IMREAD_GRAYSCALE)
    assert np.array_equal(im.astype(np.float32), tiny["images"][1])


# ---- weak-texture region detector (SURVEY section 8 row f3): host functions vs the plain-Python restatement ----------
def _detector_inputs():
    rng = np.random.RandomState(5)
    yy, xx = np.mgrid[0:38, 0:53]
    smooth = (120 + 60 * np.sin(xx / 7.0) * np.cos(yy / 5.0)).astype(np.uint8)
    noisy = smooth.copy()
    noisy[:, 20:40] = rng.randint(0, 256, (38, 20))                       # a textured band between two flat areas
    hard = np.where((xx + yy) % 2 == 0, 0, 255).astype(np.uint8)          # magnitudes >= 256: the low-byte quirk
    hard[10:20, 10:30] = 200
    steps = (np.arange(53)[None, :] * np.ones((38, 1))).astype(np.uint8)  # magnitude sqrt(2) everywhere
    steps[5:30, 8:45] = (181 * ((xx[5:30, 8:45] + yy[5:30, 8:45]) % 2)).astype(np.uint8)  # t1+t2 = 2*181^2 = 65522 / 0
    stripes = (255 * (xx % 2)).astype(np.uint8)                           # magnitude 360 -> stored as 104
    stripes[20:22, 30:32] = [[255, 0], [30, 0]]                           # 255^2 + 30^2 = 65925 -> 256 -> stored as 0
    return [smooth, noisy, hard, steps, stripes]


def test_weak_texture_stages_match_restatement(pkg):
    """tsar_weak_* (libtsar_b200.so host functions) against oracle/weak_texture_ref.py: Roberts + threshold, the
    two-pass labelling with the reference's own equivalence table (order dependent), boundary images, border closing,
    region statistics and the weak decision, the label expansion to full resolution."""
    from oracle import weak_texture_ref as wr
    from tsar_mvs_b200 import texture as tx
    rng = np.random.RandomState(11)
    for gray in _detector_inputs():
        for thr in (4, 40):
            e = tx.edges(gray, thr)
            assert np.array_equal(e, wr.roberts_threshold(gray, thr))
    assert tx.edges(_detector_inputs()[4], 4)[20, 30] == 0 and tx.edges(_detector_inputs()[4], 4)[5, 5] == 255
    # labelling: random edge maps of several densities provoke every branch, including lost equivalences
    split_seen = False
    for density in (0.15, 0.3, 0.45, 0.6):
        for trial in range(3):
            e = np.where(rng.rand(31, 44) < density, 255, 0).astype(np.uint8)
            lab, cnt = tx.connect(e)
            lab_r, cnt_r = wr.connect(e)
            assert np.array_equal(lab, lab_r) and np.array_equal(cnt, cnt_r)
            assert cnt.sum() == e.size and cnt[0] == (e == 255).sum()
            from scipy import ndimage
            true_n = ndimage.label(e == 0)[1]
            assert len(cnt) - 1 >= true_n            # never fewer labels than true 4-connected components ...
            split_seen |= (len(cnt) - 1 > true_n)    # ... and sometimes more: the table loses equivalences
            k = int(np.argmax(cnt[1:])) + 1
            assert np.array_equal(tx.boundary(lab, k), wr.boundary(lab_r, k))
            assert np.array_equal(tx.close_border(e), wr.close_border(e))
            for weaktextnum in (5, 60):
                got = tx.regions(lab, cnt, weaktextnum, 2)
                want = wr.regions(lab_r, cnt_r, weaktextnum, 2)
                for g, w_ in zip(got, want):
                    assert np.array_equal(g, w_)
            assert np.array_equal(tx.expand_labels(lab, 4 * 44 + 3, 4 * 31 + 2), wr.expand(lab_r, 4 * 44 + 3, 4 * 31 + 2))
    assert split_seen, "test inputs never exercised the order-dependent equivalence table"


def test_weak_texture_detector_finds_the_textureless_facet(pkg):
    """texture() end to end (cv2 for pyrDown / HoughLinesP / line, as the reference uses OpenCV): on the synthetic
    scene the untextured facet must come out as a weakly textured region (text = -1), the label map must cover the
    image, and textured ground must not be flagged."""
    pytest.importorskip("cv2")
    from tsar_mvs_b200 import scene, texture as tx
    cfg = dict(W=1280, H=960, n_images=2, V=1, fx=720.0, radius=4.0, arc_deg=10.0)
    cams = scene.make_cameras(cfg["W"], cfg["H"], cfg["n_images"], cfg["fx"], cfg["radius"], cfg["arc_deg"])
    sc = scene.Scene(cfg["W"], cfg["H"], cfg["fx"], cfg["radius"])
    img, _, labels = sc.render(cams[0], cfg["W"], cfg["H"])
    det = tx.detect(img.astype(np.uint8), min_pixels=2000)
    lab = det["labels_q"]
    assert lab.shape == (240, 320) and det["label_count"].sum() == lab.size
    facet_q = labels[::4, ::4][:240, :320] == 4                 # generator label of the untextured facet
    weak = det["text"][lab] == -1.0
    assert weak[facet_q].mean() > 0.7, weak[facet_q].mean()     # most of the facet is inside a weak region
    assert weak[~facet_q].mean() < 0.2, weak[~facet_q].mean()   # and weak regions are mostly the facet
    k = int(np.bincount(lab[facet_q]).argmax())
    assert det["text"][k] == -1.0 and det["size"][k] > 50
    cx, cy = det["cenxi"][k], det["cenyi"][k]
    assert labels[min(cy, cfg["H"] - 1), min(cx, cfg["W"] - 1)] == 4   # centroid (full-resolution pixels) lies on the facet
    full = tx.expand_labels(lab, cfg["W"], cfg["H"])
    assert full.shape == (cfg["H"], cfg["W"]) and full[5, 7] == lab[1, 1]


# ---- rows f1 / f3 pinned to the reference's OWN host code (oracle/_ref/libtsar_ref_host.so = main.cpp line ranges compiled by
# oracle/build_ref.sh; OpenCV library calls served by cv2), or to its recorded results where that build is absent -------
def _ref_host():
    return pc.ref_host()


def test_weak_texture_stages_match_reference_code(pkg):
    """tsar_weak_edges / tsar_weak_connect against roberts() and Connect() as the reference wrote them
    (main.cpp:214-362), on the inputs that provoke the (uchar)sqrt low-byte quirk and lost label equivalences."""
    import cv2
    rh = _ref_host()
    from tsar_mvs_b200 import texture as tx
    for gray in _detector_inputs():
        rob = rh.roberts(gray)
        for thr in (4, 40):
            assert np.array_equal(tx.edges(gray, thr), cv2.threshold(rob, thr, 255, cv2.THRESH_BINARY)[1])
    rng = np.random.RandomState(11)
    for density in (0.1, 0.15, 0.3, 0.45, 0.6, 0.8):
        for trial in range(4):
            e = np.where(rng.rand(31 + trial, 44 + 3 * trial) < density, 255, 0).astype(np.uint8)
            lab, cnt = tx.connect(e)
            lab_r, cnt_r, weak_r = rh.connect(e)
            assert np.array_equal(lab, lab_r) and np.array_equal(cnt, cnt_r)
            assert list(weak_r) == [k for k in range(1, len(cnt)) if cnt[k] > 5000]


@pytest.mark.parametrize("size,seed", [((1280, 960), 1234), ((1000, 750), 7), ((643, 481), 3)])
def test_weak_texture_detector_matches_reference_texture_function(pkg, size, seed):
    """texture.detect (product: tsar_weak_* + cv2) against the reference's whole texture() (main.cpp:365-596): the full-
    resolution label map lines->canny, the region count and cannylines->text / cenxi / cenyi / size, on rendered views
    (one with sizes that are not multiples of 4: the stepped-back last column / row)."""
    rh = _ref_host()
    from tsar_mvs_b200 import scene, texture as tx
    W, H = size
    cams = scene.make_cameras(W, H, 2, 0.5625 * W, 4.0, 10.0)
    img = scene.Scene(W, H, 0.5625 * W, 4.0, seed=seed).render(cams[0], W, H)[0].astype(np.uint8)
    if seed != 1234:                                # a painted flat area, large enough to be a weak label
        img[40:H - 60, 60:W - 110] = 90
    ref = rh.texture(img)
    det = tx.detect(img)
    assert np.array_equal(tx.expand_labels(det["labels_q"], W, H), ref["canny"])
    for k in ("text", "cenxi", "cenyi", "size"):
        assert np.array_equal(det[k], ref[k]), k
    assert (ref["text"] == -1).sum() >= 1           # the untextured facet (and the painted area) are found


def test_region_plane_fit_restatement_matches_reference_code(pkg):
    """oracle_cpu.c's restatement of the per-region RANSAC against the reference's own loop (main.cpp:1520-1730) fed with
    the same rand() stream: bit-exact planes.  (The device implementation is compared with the same library in the GPU
    suite.)"""
    rh = _ref_host()
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    scene = pkg.scene.make_scene("small")
    H, W = scene["H"], scene["W"]
    rng = np.random.RandomState(9)
    disp = (scene["cam_f"] / scene["gt_depth"]).astype(np.float32)
    disp *= (1 + 0.0005 * rng.normal(size=disp.shape)).astype(np.float32)
    out = rng.rand(H, W) < 0.2
    disp[out] *= rng.uniform(0.8, 1.2, out.sum()).astype(np.float32)
    scale = (rng.rand(H, W) < 0.5).astype(np.float32)
    text = scene["region_text"].copy()
    text[1] = -1.0
    size = np.array([(scene["labels"] == r).sum() / 16.0 for r in range(len(text))], np.float32)
    rnd = rng.randint(0, 2 ** 31 - 1, size=(len(text), 46000)).astype(np.uint32)
    p0 = np.tile(np.array([0, 0, 1, -1], np.float32), (len(text), 1))
    stream = np.concatenate([rnd[r] for r in range(len(text)) if text[r] == -1])
    ref, used = rh.fit_regions(scene["cams"][0], scene["cam_f"], disp, scale, scene["canny"], text, size, stream, p0)
    assert used == 46000 * int((text == -1).sum())  # the reference draws exactly 3 x 10 000 + 4 x 4 x 1000 values per region
    cams = cameras_to_struct(scene["cams"])
    for r in range(len(text)):
        if text[r] != -1:
            assert np.array_equal(ref[r], p0[r])
            continue
        want, n = cb.fit_region_plane(pkg._lib.TsarCamera, cams[0], scene["cam_f"], disp, scale, scene["canny"], r, size[r], rnd[r], p0[r])
        assert n > 1000 and pc.frac_bit_exact(want, ref[r]) == 1.0, (r, want, ref[r])


def test_model_ply_writer(tmp_path, pkg, tiny):
    """TSAR_model.ply (displayUtils.h:77-158): header, column-major vertex order, world points that reproject onto
    their pixel at their depth with the untransformed camera (cameraGeometryUtils.h:53-65)."""
    from tsar_mvs_b200 import dmb
    cam = tiny["cams"][0]
    H, W = tiny["H"], tiny["W"]
    depth = tiny["gt_depth"].astype(np.float32)
    depth[3, 5] = np.inf                                            # a non-finite point is written as the origin
    normals = np.zeros((H, W, 3), np.float32); normals[..., 2] = -1
    R, C = cam["_R_world"], cam["_C_world"]
    t = -R @ C
    path = str(tmp_path / "TSAR_model.ply")
    dmb.write_model_ply(path, depth, normals, tiny["images"][0], cam["K"], R, t)
    head = open(path, "rb").read(400).decode("latin1")
    assert head.startswith("ply\nformat binary_little_endian 1.0\n") and f"element vertex {H * W}\n" in head
    pts, nrm, col = dmb.read_model_ply(path)
    assert pts.shape == (H * W, 3) and os.path.getsize(path) == head.index("end_header\n") + 11 + 27 * H * W
    P = cam["K"] @ np.concatenate([R, t[:, None]], 1)
    for (x, y) in ((0, 0), (10, 7), (W - 1, H - 1), (50, 33)):
        X = pts[x * H + y].astype(np.float64)                       # x outer, y inner
        p = P @ np.append(X, 1.0)
        assert abs(p[2] - depth[y, x]) < 1e-3 * depth[y, x]
        assert abs(p[0] / p[2] - x) < 1e-2 and abs(p[1] / p[2] - y) < 1e-2
        assert col[x * H + y].tolist() == [int(tiny["images"][0][y, x])] * 3
    assert np.array_equal(pts[5 * H + 3], np.zeros(3, np.float32))
    assert np.array_equal(nrm[7], normals[7, 0])


def _build_c_abi_check(tmp_path):
    import subprocess
    exe = str(tmp_path / "c_abi_check")
    pkgdir = os.path.join(ROOT, "tsar-mvs_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "c_abi_check.c"), "-L" + pkgdir, "-ltsar_b200", "-Wl,-rpath," + pkgdir, "-lm", "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_header_is_plain_c_and_fails_loudly_without_a_device(tmp_path, pkg):
    """include/tsar_b200.h compiles as C11 (-Wall -Wextra -Werror) and links against the library from a C program;
    on a machine without an sm_100 device tsar_create reports TSAR_ERR_NODEVICE -- there is no CPU path."""
    import subprocess
    import torch
    exe = _build_c_abi_check(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked twin of this test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "TSAR_ERR_NODEVICE" in r.stdout and "no CPU path" in r.stderr
