"""Command line of the reference (`gipuma <ref image> <other images...> flags`, main.cpp:708-1009, run scripts
scripts/*.sh) on top of libtsar_b200.so.

    python -m tsar_cli 00000000.jpg 00000001.jpg ... -mslp_folder data/TRAIN/pipes/ -images_folder data/TRAIN/pipes/images/ \
        -krt_file x -output_folder results/pipes/ -no_display --cam_scale=1 --iterations=8 --blocksize=11 \
        --cost_gamma=10 --cost_comb=best_n --n_best=1 --min_angle= --max_angle=

Kept from the reference: positional arguments are image names, the first one is the reference view; `--key=value`
numeric flags, `-key value` path flags, `-color_processing` / `-view_selection` booleans; unknown flags only warn
(main.cpp:941-945) -- the scripts pass an unknown `-no_display` and empty `--min_angle=`/`--max_angle=` (SURVEY Q16);
`-krt_file` merely selects the MVSNet-style reader, its value is ignored (fileIoUtils.h:111-118); cameras come from
`<mslp>/cams/<8-digit stem>_cam.txt`, the source views from `<mslp>/pair.txt` (main.cpp:1351-1376, camera id =
atoi(name[4:8])); results go to `<mslp>/APD/<stem>/TSAR_disp.dmb` and `TSAR_normals.dmb` (main.cpp:1807-1861).

Flows:
  * default (north-star): random initialisation + red/black PatchMatch + L/R check + confidence + output layout;
  * `-import_apd`: the shipped flow -- planes imported from `<mslp>/APD/<stem>/depths_geom.dmb` + `normals.dmb`
    (main.cpp:1459-1490) then gipuma_get_disp / getview / output.
Textureless-region completion: the weak-texture detector of main.cpp:365-596 (texture.py; cv2 for pyrDown /
HoughLinesP / line as the reference uses OpenCV) labels the reference view; regions it flags get a plane from
tsar_fit_region_planes and are completed by update_scale(_2).  `-no_weak_texture` skips it; `-regions_file labels.npy`
(+ `-regions_text text.npy`) supplies a precomputed label map instead.
`-write_ply` also writes `TSAR_model.ply` (displayUtils.h:77-158).
`-fuse` fuses every view's `APD/<stem>/TSAR_disp.dmb` + `TSAR_normals.dmb` with the colour images, cams and pair.txt
into one point cloud, `<mslp>/TSAR_fused.ply` (fusion.py, DESIGN.md section 4.6; one GPU, views in dataset order).
With `-all_views` it runs after the last view (single process only: fusion reads every view's output).
`-eval <gt.ply>` scores `<mslp>/TSAR_fused.ply` against a ground-truth cloud (cloud_eval.py, DESIGN.md section 4.7):
accuracy, completeness and F-score per threshold (`-eval_thresholds 0.01,0.02,...`, scene units; default
0.01,0.02,0.05,0.1,0.2,0.5), one table line each, and `<mslp>/TSAR_eval.json`.  It runs alone on an existing
TSAR_fused.ply or after `-fuse` / `-all_views -fuse` in the same call.
Extra: `--synthetic=<C1|C2|small|tiny>` first writes a synthetic dataset in the reference's folder layout.

`-all_views` replaces the per-view process loop of the run scripts (scripts/pipes.sh:30-49): every image of the
dataset becomes the reference view once.  All images are decoded and uploaded ONCE and stay resident in HBM; each
reference view binds itself + its pair.txt neighbours from that pool (device-to-device), two contexts on two streams
pipeline view r+1 behind view r, results are written by a writer pool.  Under torchrun the views are sharded in
contiguous blocks over the ranks (shard.py), one GPU per rank, no collective.  `-resume` skips the views whose three
output files are already complete (an interrupted run continues where it stopped; files are written under a temporary
name and renamed, so a partial file never counts).
"""
import itertools
import math
import os
import sys

import numpy as np

from . import dmb, scene
from .engine import DepthmapEngine, make_params

NUMERIC = {"blocksize", "iterations", "n_best", "cost_gamma", "depth_min", "depth_max", "max_views", "min_angle", "max_angle",
           "cam_scale", "cost_tau_color", "cost_tau_gradient", "cost_alpha", "disp_tol", "normal_tol", "census_epsilon",
           "self_similarity_n", "good_factor", "num_img_processed", "seed", "synthetic", "device", "lanes", "io_threads"}
PATHS = {"images_folder", "mslp_folder", "krt_file", "output_folder", "p_folder", "camera_folder", "calib_file", "pmvs_folder",
         "bounding_folder", "regions_file", "regions_text", "regions_size", "eval", "eval_thresholds"}
BOOLS = {"color_processing", "view_selection", "import_apd", "no_display", "all_views", "no_weak_texture", "write_ply", "wmf", "no_slic", "no_write", "resume", "fuse"}


def parse_args(argv):
    """getParametersFromCommandLine (main.cpp:708-1009), tolerant in the same places."""
    opt = dict(images=[], blocksize=19, iterations=8, n_best=2, cost_comb=1, cam_scale=1.0, depth_min=-1.0, depth_max=-1.0,
               seed=20240601, device=0, images_folder="", mslp_folder="", output_folder="", synthetic=None,
               color_processing=False, import_apd=False, all_views=False, no_weak_texture=False, write_ply=False, wmf=False, no_slic=False, no_write=False, resume=False, fuse=False,
               regions_file=None, regions_text=None, regions_size=None, lanes=2, io_threads=4, eval=None, eval_thresholds=None)
    i = 0
    while i < len(argv):
        a = argv[i]
        if a.startswith("--"):
            key, _, val = a[2:].partition("=")
            if key == "cost_comb":
                opt["cost_comb"] = {"all": 0, "best_n": 1, "angle": 2, "good": 3}.get(val, opt["cost_comb"])
            elif key == "synthetic":
                opt["synthetic"] = val
            elif key in NUMERIC:
                if val != "":  # the scripts pass `--min_angle=` with an empty value
                    opt[key] = float(val) if "." in val or key in ("cam_scale", "depth_min", "depth_max") else int(val)
            else:
                print(f"[tsar_cli] warning: unknown option {a}", file=sys.stderr)
        elif a.startswith("-") and len(a) > 1 and not a[1].isdigit():
            key = a[1:]
            if key in BOOLS:
                opt[key] = True
            elif key in PATHS:
                i += 1
                opt[key] = argv[i] if i < len(argv) else ""
            else:
                print(f"[tsar_cli] warning: unknown option {a}", file=sys.stderr)
        else:
            opt["images"].append(a)
        i += 1
    return opt


# ---- dataset I/O -------------------------------------------------------------------------------------------
def read_cam_txt(path):
    """MVSNet-style camera file as readKRtFileMiddlebury reads it (fileIoUtils.h:111-163): 'extrinsic', 4x4 [R|t],
    'intrinsic', 3x3 K, then depth_min interval depth_num depth_max."""
    tok = open(path).read().split()
    assert tok[0] == "extrinsic", path
    E = np.array(tok[1:17], float).reshape(4, 4)
    assert tok[17] == "intrinsic", path
    K = np.array(tok[18:27], float).reshape(3, 3)
    tail = [float(v) for v in tok[27:31]]
    depth_min, depth_max = tail[0], tail[3]
    return K, E[:3, :3], E[:3, 3], depth_min, depth_max


def write_cam_txt(path, K, R, t, depth_min, depth_max, interval=0.0, depth_num=0):
    E = np.eye(4)
    E[:3, :3], E[:3, 3] = R, t
    with open(path, "w") as f:
        f.write("extrinsic\n" + "\n".join(" ".join(repr(float(v)) for v in row) for row in E) + "\n\nintrinsic\n")
        f.write("\n".join(" ".join(repr(float(v)) for v in row) for row in np.asarray(K, float)) + "\n\n")
        f.write(f"{depth_min!r} {interval!r} {depth_num} {depth_max!r}\n")


def read_pair_subset(path, camera_id):
    """Source views of camera `camera_id` as indices into the command-line image list (main.cpp:1351-1376): the list is
    [reference, all other images in order], so image k maps to k+1 if k < camera_id else k."""
    lines = open(path).read().split("\n")
    line = lines[2 * camera_id + 2].split()  # 1 header line, then per camera: id line + neighbour line
    n = int(line[0])
    subset = []
    for j in range(n):
        k = int(line[1 + 2 * j])
        subset.append(k if k > camera_id else k + 1)
    return subset


def write_pair_txt(path, neighbours):
    with open(path, "w") as f:
        f.write(f"{len(neighbours)}\n")
        for i, nb in enumerate(neighbours):
            f.write(f"{i}\n{len(nb)} " + " ".join(f"{k} 1.0" for k in nb) + "\n")


def _imread_gray(path, colour=False):
    """Grey image (cv::imread IMREAD_GRAYSCALE, main.cpp:1302).  With -color_processing the reference uploads the
    BGRA image instead and its kernels sample the first component (tex2D<float>, gipuma.cu:247,262,265): blue."""
    if path.endswith(".npy"):
        return np.load(path).astype(np.float32)
    import cv2  # image decoding only
    im = cv2.imread(path, cv2.IMREAD_COLOR if colour else cv2.IMREAD_GRAYSCALE)
    if im is None:
        raise FileNotFoundError(path)
    return (im[..., 0] if colour else im).astype(np.float32)


def write_synthetic_dataset(cfg_name, root):
    """Writes a synthetic scene in the reference's folder layout: <root>/images/%08d.png, <root>/cams/%08d_cam.txt,
    <root>/pair.txt.  Returns (scene dict, list of image names)."""
    import cv2
    sc = scene.make_scene(cfg_name)
    os.makedirs(os.path.join(root, "images"), exist_ok=True)
    os.makedirs(os.path.join(root, "cams"), exist_ok=True)
    names = []
    n = len(sc["images"])
    for i, (im, cam) in enumerate(zip(sc["images"], sc["cams"])):
        name = f"{i:08d}.png"
        cv2.imwrite(os.path.join(root, "images", name), im.astype(np.uint8))
        R, C = cam["_R_world"], cam["_C_world"]
        write_cam_txt(os.path.join(root, "cams", f"{i:08d}_cam.txt"), cam["K"], R, -R @ C, cam["depthMin"], cam["depthMax"])
        names.append(name)
    write_pair_txt(os.path.join(root, "pair.txt"), [[k for k in range(n) if k != i] for i in range(n)])
    return sc, names


def write_rig_dataset(cfg_name, root, backend="numpy", device=None, jpeg_quality=95):
    """A multi-view synthetic dataset (scene.make_rig: C3 = 38 cameras on two arcs, C4seq = 300-frame sequence) in the
    reference's folder layout, images as JPEG files like the ETH3D / Tanks&Temples originals (scripts/*.sh list
    %08d.jpg names); pair.txt lists every camera's 10 nearest neighbours.  Returns the image names."""
    import cv2
    cfg = scene.CONFIGS[cfg_name]
    K, Rs, Cs, neighbours = scene.make_rig(cfg)
    os.makedirs(os.path.join(root, "images"), exist_ok=True)
    os.makedirs(os.path.join(root, "cams"), exist_ok=True)
    names = []
    for i, img in scene.render_rig(cfg, backend=backend, device=device):
        name = f"{i:08d}.jpg"
        cv2.imwrite(os.path.join(root, "images", name), img, [cv2.IMWRITE_JPEG_QUALITY, int(jpeg_quality)])
        R, C = Rs[i], Cs[i]
        write_cam_txt(os.path.join(root, "cams", f"{i:08d}_cam.txt"), K, R, -R @ C, 0.7 * cfg["radius"], 1.45 * cfg["radius"])
        names.append(name)
    write_pair_txt(os.path.join(root, "pair.txt"), neighbours)
    return names


# ---- one reference view: the TSAR flow of runGipuma (main.cpp:1268-1866) -----------------------------------------
def _load_image_bytes(bgr_quarter):
    """UChar4Image as load_image fills it (main.cpp:190-201): OpenCV's B goes to `.b` (byte 2), G to byte 1, R to `.r`
    (byte 0)."""
    h, w = bgr_quarter.shape[:2]
    out = np.zeros((h, w, 4), np.uint8)
    out[..., 0], out[..., 1], out[..., 2] = bgr_quarter[..., 2], bgr_quarter[..., 1], bgr_quarter[..., 0]
    return out


def quarter_colour(bgr_full):
    """main.cpp:619-622: two pyrDown with explicit halved sizes on the colour image."""
    import cv2
    c2 = cv2.pyrDown(bgr_full, dstsize=(bgr_full.shape[1] // 2, bgr_full.shape[0] // 2))
    return cv2.pyrDown(c2, dstsize=(c2.shape[1] // 2, c2.shape[0] // 2))


def run_view(eng, opt, view, outputs=None):
    """The whole per-view flow on a context whose views and parameters are already set: texture() -> gslic() -> firstcuda
    -> [weak.png] -> sliccuda -> per-region RANSAC -> fakecuda -> fillcuda (main.cpp:1893-1896, 1459-1783).
    view: dict(gray_u8 = reference image (H x W uint8) for the detector, bgr = colour reference image or None, apd_dir,
    seed).  outputs: optional (depth, normals, confid) host buffers (arrays or raw addresses).  Returns
    (depth, normals, confid, info)."""
    from . import _lib as L
    info = {}
    H, W = eng.H, eng.W
    text = size = None
    if opt["regions_file"]:
        labels = np.load(opt["regions_file"]).astype(np.float32)
        text = np.load(opt["regions_text"]).astype(np.float32)
        size = np.load(opt["regions_size"]).astype(np.float32) if opt["regions_size"] else \
            np.array([(labels == r).sum() / 16.0 for r in range(len(text))], np.float32)
        eng.upload(L.F_CANNY, labels)
    elif not opt["no_weak_texture"]:            # texture() runs first in the reference's main (main.cpp:1893)
        import time
        from . import texture
        t_det = time.perf_counter()
        det = texture.detect(view["gray_u8"])
        info["detect_s"] = time.perf_counter() - t_det
        info["regions"], info["weak_regions"] = len(det["text"]) - 1, int((det["text"] == -1).sum())
        text, size = det["text"], det["size"]
        eng.set_labels_quarter(det["labels_q"])
    if view.get("bgr") is not None and not opt["no_slic"] and min(H, W) >= 4 * 20:   # gslic() (main.cpp:598-660): superpixels of
        info["slic_labels"] = eng.slic(_load_image_bytes(quarter_colour(view["bgr"])))  # size 20 on the quarter-size image; debug output only
    if opt["import_apd"]:                       # shipped flow, main.cpp:1459-1490
        f = float(np.float32(view["cam_f"]))
        depth = dmb.read_dmb(os.path.join(view["apd_dir"], "depths_geom.dmb"))
        normal = dmb.read_dmb(os.path.join(view["apd_dir"], "normals.dmb"))
        eng.upload(L.F_NORM4, np.concatenate([normal, np.zeros((H, W, 1), np.float32)], axis=-1))
        eng.upload(L.F_COST, np.ones((H, W), np.float32))
        eng.upload(L.F_DEPTH, (np.float32(f) / depth).astype(np.float32))
        eng.get_disp()
    else:                                       # the block the reference has commented out (gipuma.cu:1741-1758)
        eng.init_planes(int(view["seed"]))
        eng.iterate(opt["iterations"], int(view["seed"]))
        eng.lrdiff()
    eng.getview()
    n_weak = int((text == -1).sum()) if text is not None else 0
    if text is not None and (n_weak or opt["wmf"]):
        weak_png = os.path.join(view["apd_dir"], "weak.png")
        if opt["import_apd"] and os.path.exists(weak_png):     # reliable pixels: main.cpp:1499-1514
            import cv2
            eng.scale_from_weak_png(cv2.imread(weak_png, cv2.IMREAD_COLOR))
        else:
            if opt["import_apd"]:
                print(f"[tsar_cli] {weak_png} not found: reliable pixels taken from the confidence map", file=sys.stderr)
            eng.scale_from_confidence(0.8)      # stands in for APD's weak.png
        if opt["wmf"]:                          # gipuma_WMF x 4 (gipuma.cu:1809-1812)
            for it in range(4):
                eng.wmf(it)
        planes = np.tile(np.array([0, 0, 1, -1], np.float32), (len(text), 1))
        if n_weak:                              # main.cpp:1520-1730
            planes = eng.fit_region_planes(text, size, None, planes, seed=int(view["seed"]))
        eng.set_regions(text, planes)
        if n_weak:
            eng.update_scale_2()                # fakecuda
            eng.update_scale()                  # fillcuda
        if opt["wmf"]:                          # gipuma_WMF_Final x 6 (gipuma.cu:1844-1847)
            for it in range(6):
                eng.wmf_final(it)
    eng.compute_disp()
    bufs = outputs if outputs is not None else (None, None, None)
    depth, normals, confid = eng.download_outputs(*bufs)
    return depth, normals, confid, info


# ---- the driver ---------------------------------------------------------------------------------------------
def run(argv):
    opt = parse_args(argv)
    mslp = opt["mslp_folder"]
    if opt["synthetic"]:
        mslp = mslp or "./synthetic_" + opt["synthetic"] + "/"
        if "rig" in scene.CONFIGS.get(opt["synthetic"], {}):
            names = write_rig_dataset(opt["synthetic"], mslp)
        else:
            _, names = write_synthetic_dataset(opt["synthetic"], mslp)
        opt["images"] = opt["images"] or names
        opt["images_folder"] = os.path.join(mslp, "images/")
    if opt["all_views"]:
        if opt["fuse"] and int(os.environ.get("WORLD_SIZE", "1")) > 1:
            print("[tsar_cli] -fuse runs on one GPU (view v depends on the views before it): run -all_views under several "
                  "ranks without -fuse, then `tsar_cli.py -fuse -mslp_folder ...` as a single process", file=sys.stderr)
            return 2
        if opt["eval"] and int(os.environ.get("WORLD_SIZE", "1")) > 1:
            print("[tsar_cli] -eval runs in a single process: run -all_views under several ranks without it, then "
                  "`tsar_cli.py -fuse -eval <gt.ply> -mslp_folder ...`", file=sys.stderr)
            return 2
        run_all_views(opt, mslp)
        if opt["fuse"]:
            rc = run_fuse(opt, mslp)
            if rc or not opt["eval"]:
                return rc
        if opt["eval"]:
            return run_eval(opt, mslp)
        return 0
    if opt["fuse"]:
        rc = run_fuse(opt, mslp)
        if rc or not opt["eval"]:
            return rc
    if opt["eval"]:
        return run_eval(opt, mslp)
    if not opt["images"]:
        print(__doc__)
        return 2
    names = opt["images"]
    stem = names[0][:8]                         # main.cpp:1462: numind = imgname.substr(0, 8)
    camera_id = int(names[0][4:8])              # main.cpp:1347-1349: atoi(name.substr(4, 8)) (sic: 4 characters)
    images = [_imread_gray(os.path.join(opt["images_folder"], n), opt["color_processing"]) for n in names]
    Ks, Rs, ts, dmin, dmax = [], [], [], None, None
    for i, n in enumerate(names):
        K, R, t, a, b = read_cam_txt(os.path.join(mslp, "cams", f"{n[:8]}_cam.txt"))
        K = K.copy()
        K[:2] /= opt["cam_scale"]               # scaleK (cameraGeometryUtils.h:141-151)
        Ks.append(K); Rs.append(R); ts.append(t)
        if i == 0:
            dmin, dmax = a, b                   # depth range of the reference view (fileIoUtils.h:145-153)
    if opt["depth_min"] > 0:
        dmin = opt["depth_min"]
    if opt["depth_max"] > 0:
        dmax = opt["depth_max"]
    cams = scene.cameras_from_krt(Ks, Rs, ts, dmin, dmax)
    subset = read_pair_subset(os.path.join(mslp, "pair.txt"), camera_id)
    subset = [s for s in subset if s < len(names)]
    f = float(np.float32(cams[0]["f"]))
    params = make_params(box=opt["blocksize"], iterations=opt["iterations"], n_best=opt["n_best"], cost_comb=opt["cost_comb"],
                         min_disparity=float(np.float32(f / np.float32(dmax))), max_disparity=float(np.float32(f / np.float32(dmin))))
    eng = DepthmapEngine(int(opt["device"]))
    eng.set_views(images, cams, subset, cam_f=f)
    eng.set_params(params)
    out_dir = os.path.join(mslp, "APD", stem)
    H, W = images[0].shape
    bgr = None
    if not opt["no_slic"] and not names[0].endswith(".npy"):
        import cv2
        bgr = cv2.imread(os.path.join(opt["images_folder"], names[0]), cv2.IMREAD_COLOR)
    view = dict(gray_u8=_imread_gray(os.path.join(opt["images_folder"], names[0])).astype(np.uint8) if opt["color_processing"] else images[0].astype(np.uint8),
                bgr=bgr, apd_dir=out_dir, seed=int(opt["seed"]), cam_f=f)
    depth, normals, confid, info = run_view(eng, opt, view)
    if "regions" in info:
        print(f"[tsar_cli] weak-texture detector: {info['regions']} regions, {info['weak_regions']} weakly textured")
    os.makedirs(out_dir, exist_ok=True)
    dmb.write_dmb(os.path.join(out_dir, "TSAR_disp.dmb"), depth)
    dmb.write_dmb(os.path.join(out_dir, "TSAR_normals.dmb"), normals)
    dmb.write_dmb(os.path.join(out_dir, "TSAR_confidence.dmb"), confid)   # computed but never written by the reference
    if opt["write_ply"]:                        # main.cpp:1836-1843 (always on there; 27 B per pixel, so opt-in here)
        dmb.write_model_ply(os.path.join(out_dir, "TSAR_model.ply"), depth, normals, images[0], Ks[0], Rs[0], ts[0])
    print(f"[tsar_cli] {stem}: {W}x{H}, {len(subset)} source views -> {out_dir}/TSAR_disp.dmb, TSAR_normals.dmb")
    eng.close()
    return 0


def read_pair_neighbours(path, camera_id):
    """Camera ids of the source views of `camera_id` in pair.txt order (main.cpp:1351-1376)."""
    lines = open(path).read().split("\n")
    line = lines[2 * camera_id + 2].split()
    return [int(line[1 + 2 * j]) for j in range(int(line[0]))]


def read_pair_table(path):
    """pair.txt parsed once: {camera id: [neighbour camera ids in file order]} (main.cpp:1351-1376)."""
    lines = open(path).read().split("\n")
    n = int(lines[0].split()[0])
    table = {}
    for k in range(n):
        cam = int(lines[2 * k + 1].split()[0])
        tok = lines[2 * k + 2].split()
        table[cam] = [int(tok[1 + 2 * j]) for j in range(int(tok[0]))]
    return table


def read_fusion_views(opt, mslp, lazy=False):
    """The inputs of fusion.fuse for every image of the dataset (names as -all_views lists them): depth and normals from
    APD/<stem>/, K R t from cams/ (cam_scale applied), the colour image, and the pair.txt neighbours that exist in the
    dataset.  Raises FileNotFoundError naming every view whose outputs are missing, ValueError when there is no image or
    naming every view with no neighbour in the dataset or more than 32.  lazy=True returns (number of views, generator
    of the views) so that only one view is held in host memory at a time."""
    import cv2
    from .fusion import MAX_NEIGHBOURS
    folder = opt["images_folder"] or os.path.join(mslp, "images/")
    names = opt["images"] or sorted(n for n in os.listdir(folder) if n.lower().endswith((".jpg", ".jpeg", ".png", ".npy")))
    if not names:
        raise ValueError(f"no images in {folder}")
    apd = [os.path.join(mslp, "APD", n[:8]) for n in names]
    missing = [n[:8] for n, d in zip(names, apd) if not all(os.path.exists(os.path.join(d, f)) for f in ("TSAR_disp.dmb", "TSAR_normals.dmb"))]
    if missing:
        raise FileNotFoundError(f"no TSAR_disp.dmb / TSAR_normals.dmb under {os.path.join(mslp, 'APD')} for view(s) {', '.join(missing)}: "
                                f"compute them first (-all_views)")
    ids = [int(n[4:8]) for n in names]
    by_id = {c: k for k, c in enumerate(ids)}
    pairs = read_pair_table(os.path.join(mslp, "pair.txt"))
    neighbours = [[by_id[c] for c in pairs.get(i, []) if c in by_id] for i in ids]
    bad = [f"{n[:8]} ({len(nb)})" for n, nb in zip(names, neighbours) if not 1 <= len(nb) <= MAX_NEIGHBOURS]
    if bad:
        raise ValueError(f"fusion needs 1..{MAX_NEIGHBOURS} pair.txt neighbours present in the dataset per view; "
                         f"view(s) {', '.join(bad)} have not")

    def load(k):
        n = names[k]
        K, R, t, _, _ = read_cam_txt(os.path.join(mslp, "cams", f"{n[:8]}_cam.txt"))
        K = K.copy()
        K[:2] /= opt["cam_scale"]
        path = os.path.join(folder, n)
        if n.endswith(".npy"):
            bgr = np.repeat(np.clip(np.load(path), 0, 255).astype(np.uint8)[..., None], 3, axis=-1)
        else:
            bgr = cv2.imread(path, cv2.IMREAD_COLOR)
            if bgr is None:
                raise FileNotFoundError(path)
        return dict(K=K, R=R, t=t, depth=dmb.read_dmb(os.path.join(apd[k], "TSAR_disp.dmb")),
                    normals=dmb.read_dmb(os.path.join(apd[k], "TSAR_normals.dmb")), bgr=bgr,
                    neighbours=neighbours[k])

    if lazy:
        return len(names), (load(k) for k in range(len(names)))
    return [load(k) for k in range(len(names))]


def run_fuse(opt, mslp, quiet=False):
    """-fuse: every view's depth + normal maps -> <mslp>/TSAR_fused.ply.  Returns the exit code."""
    import time
    from . import fusion
    t0 = time.perf_counter()
    from .engine import TsarError
    try:
        n_views, views = read_fusion_views(opt, mslp, lazy=True)
        first = next(views)
        H, W = first["depth"].shape
        with fusion.FusionEngine(n_views, W, H, device=int(opt["device"])) as eng:
            for k, v in enumerate(itertools.chain([first], views)):
                eng.set_view(k, v["K"], v["R"], v["t"], v["depth"], v["normals"], v["bgr"], v["neighbours"])
            xyz, nrm, rgb = eng.run()
    except (FileNotFoundError, ValueError, TsarError) as e:    # set_view names the view (index in dataset order)
        print(f"[tsar_cli] -fuse: {e}", file=sys.stderr)
        return 1
    out = os.path.join(mslp, "TSAR_fused.ply")
    dmb.write_fused_ply(out, xyz, nrm, rgb)
    if not quiet:
        print(f"[tsar_cli] fused {n_views} views ({W}x{H}) into {len(xyz)} points in {time.perf_counter() - t0:.2f} s -> {out}")
    return 0


def parse_thresholds(text):
    """-eval_thresholds: comma-separated finite values > 0.  Raises ValueError naming the bad item."""
    from .cloud_eval import MAX_THRESHOLDS
    items = [t.strip() for t in (text or "").split(",") if t.strip()]
    if not items:
        raise ValueError("-eval_thresholds: empty threshold list")
    if len(items) > MAX_THRESHOLDS:
        raise ValueError(f"-eval_thresholds: at most {MAX_THRESHOLDS} thresholds")
    out = []
    for t in items:
        try:
            v = float(t)
        except ValueError:
            v = math.nan
        if not (math.isfinite(v) and v > 0 and math.isfinite(np.float32(v)) and np.float32(v) > 0):
            raise ValueError(f"-eval_thresholds: bad threshold {t!r} (need finite values > 0)")
        out.append(v)
    return out


def run_eval(opt, mslp, quiet=False):
    """-eval: <mslp>/TSAR_fused.ply against the ground-truth cloud -> table + <mslp>/TSAR_eval.json.  Returns the exit
    code."""
    import json
    from . import cloud_eval
    from .engine import TsarError
    recon_path, gt_path = os.path.join(mslp, "TSAR_fused.ply"), opt["eval"]
    try:
        thresholds = parse_thresholds(opt["eval_thresholds"]) if opt["eval_thresholds"] is not None \
            else list(cloud_eval.DEFAULT_THRESHOLDS)
        recon = dmb.read_ply_points(recon_path)
        gt = dmb.read_ply_points(gt_path)
        res = cloud_eval.evaluate(recon, gt, thresholds, device=int(opt["device"]))
    except (ValueError, TsarError) as e:
        print(f"[tsar_cli] -eval: {e}", file=sys.stderr)
        return 1
    if not quiet:
        print(f"[tsar_cli] -eval {recon_path} ({res['n_recon']} points) against {gt_path} ({res['n_gt']} points)")
        for i, t in enumerate(res["thresholds"]):
            print(f"[tsar_cli]   tau {t:g}: accuracy {res['accuracy'][i]:.4f} ({res['within_recon'][i]}), completeness "
                  f"{res['completeness'][i]:.4f} ({res['within_gt'][i]}), F {res['fscore'][i]:.4f}")
    out = {k: v for k, v in res.items()}
    for k in ("accuracy", "completeness", "fscore"):      # JSON has no NaN: an empty cloud's fractions are null
        out[k] = [None if math.isnan(v) else v for v in out[k]]
    out = dict(recon=os.path.abspath(recon_path), gt=os.path.abspath(gt_path), **out)
    with open(os.path.join(mslp, "TSAR_eval.json"), "w") as f:
        json.dump(out, f, indent=1)
    return 0


_LANE_POOL = {}   # (device, W, H) -> lanes kept alive between run_all_views calls of one process (persistent=True)


def release_lanes():
    """Closes the contexts a persistent driver kept (run_all_views(..., persistent=True))."""
    for lanes in _LANE_POOL.values():
        for lane in lanes:
            if lane.get("eng") is not None:
                lane["eng"].close()
    _LANE_POOL.clear()


def run_all_views(opt, mslp, quiet=False, persistent=False):
    """Persistent multi-view driver (SURVEY section 8 rows e/f4), the replacement of the per-view process loop of
    scripts/pipes.sh:30-49.  Every reference view of this rank runs the whole TSAR flow (run_view).  Host side:
      * a decoder pool reads the images this rank needs (its views + their pair.txt neighbours) in parallel, while the
        first views already run; decoded images go to HBM once and stay there;
      * `lanes` contexts (own stream, own host thread) take views from a shared queue, so a view's host stages (cameras,
        weak-texture detector, file hand-over) overlap the kernels of the other lane;
      * results arrive in pinned buffers that already carry the .dmb header and are written by a writer pool.
    Returns a dict with the throughput and where the time went."""
    import concurrent.futures as cf
    import itertools
    import threading
    import time

    import torch

    from .engine import cameras_to_struct
    from .shard import block_for_rank
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise RuntimeError("tsar_cli -all_views needs a CUDA device (no CPU path)")
    dev = int(os.environ.get("LOCAL_RANK", opt["device"])) % ndev
    folder = opt["images_folder"] or os.path.join(mslp, "images/")
    names = opt["images"] or sorted(n for n in os.listdir(folder) if n.lower().endswith((".jpg", ".jpeg", ".png", ".npy")))
    ids = [int(n[4:8]) for n in names]                          # camera id of each image (main.cpp:1347-1349)
    by_id = {c: k for k, c in enumerate(ids)}
    t0 = time.perf_counter()
    krt = [read_cam_txt(os.path.join(mslp, "cams", f"{n[:8]}_cam.txt")) for n in names]
    pairs = read_pair_table(os.path.join(mslp, "pair.txt"))
    mine = block_for_rank(len(names), rank, world)      # contiguous blocks: neighbouring views share their source images
    if opt.get("views_per_rank"):                        # warm-up pass of the benchmark: the first few views of each rank
        mine = mine[:int(opt["views_per_rank"])]
    skipped = []
    if opt.get("resume"):                                # views whose outputs are complete are not computed again
        def complete(r):
            d = os.path.join(mslp, "APD", names[r][:8])
            return all(os.path.exists(os.path.join(d, f)) for f in ("TSAR_disp.dmb", "TSAR_normals.dmb", "TSAR_confidence.dmb"))
        skipped = [r for r in mine if complete(r)]
        mine = [r for r in mine if r not in set(skipped)]
    if not mine:                                         # nothing (left) to do on this rank
        if not quiet:
            print(f"[tsar_cli] rank {rank}/{world}: 0 of {len(names)} reference views to compute ({len(skipped)} already complete)")
        return dict(rank=rank, world=world, views=0, skipped=len(skipped), images=len(names), seconds=0.0, depthmaps_per_s=0.0, gpu_launches=0,
                    host_seconds={}, bytes_decoded=0, bytes_written=0, weak_regions=0)
    neigh = {r: [by_id[c] for c in pairs.get(ids[r], []) if c in by_id] for r in mine}
    needed = sorted(set(mine) | {i for r in mine for i in neigh[r]})
    want_colour = not opt["no_slic"]
    stats = dict(decode_s=0.0, detect_s=0.0, gpu_wait_s=0.0, write_s=0.0, setup_s=0.0)
    stats_lock = threading.Lock()

    def add(key, dt):
        with stats_lock:
            stats[key] += dt

    # ---- decoder pool: grey image of every needed view (+ colour for this rank's reference views) ------------------
    def decode(i):
        t = time.perf_counter()
        path = os.path.join(folder, names[i])
        grey = _imread_gray(path, opt["color_processing"])
        u8 = grey.astype(np.uint8) if not opt["color_processing"] else _imread_gray(path).astype(np.uint8)
        bgr = None
        if want_colour and i in mine_set and not path.endswith(".npy"):
            import cv2
            bgr = cv2.imread(path, cv2.IMREAD_COLOR)
        add("decode_s", time.perf_counter() - t)
        return grey, u8, bgr

    mine_set = set(mine)
    io_pool = cf.ThreadPoolExecutor(max(1, int(opt["io_threads"])))
    order = list(itertools.chain.from_iterable([r] + neigh[r] for r in mine))   # decode in the order the lanes ask
    seen, decode_order = set(), []
    for i in order:
        if i not in seen:
            seen.add(i); decode_order.append(i)
    fut = {i: io_pool.submit(decode, i) for i in decode_order}
    resident, resident_lock = {}, {i: threading.Lock() for i in needed}

    def device_image(i):
        with resident_lock[i]:
            if i not in resident:
                grey = fut[i].result()[0]
                resident[i] = torch.from_numpy(np.ascontiguousarray(grey, np.float32)).to(f"cuda:{dev}")   # resident, once
            return resident[i]

    H, W = fut[decode_order[0]].result()[0].shape
    npx = W * H

    def out_buffers():
        """pinned buffers holding header + payload of the three output files of one view"""
        bufs = []
        for nb in (1, 3, 1):
            t = torch.empty(16 + npx * nb * 4, dtype=torch.uint8).pin_memory()
            t.numpy()[:16].view(np.int32)[:] = [1, H, W, nb]            # fileIoUtils.h:333-381
            bufs.append(t)
        return bufs

    # Lanes (context + stream + pinned output sets) are created by their own host thread while the decoder pool is already
    # working, and the 127 MB-per-set pinned buffers (C2 size) only when a view first needs one: nothing of that sits in
    # front of the first view.  A persistent driver (persistent=True: a service processing dataset after dataset, and the
    # benchmark's passes after its warm-up pass) keeps them between calls.
    n_lanes = max(1, min(int(opt["lanes"]), len(mine)))
    pool_key = (dev, W, H)
    lanes = _LANE_POOL.get(pool_key, []) if persistent else []
    while len(lanes) < n_lanes:
        lanes.append(dict(eng=None, stream=None, free=__import__("queue").Queue(), sets=0))
    if persistent:
        _LANE_POOL[pool_key] = lanes
    launches0 = sum(lane["eng"].launch_count() for lane in lanes[:n_lanes] if lane["eng"] is not None)

    def lane_ready(lane):
        if lane["eng"] is None:
            lane["stream"] = torch.cuda.Stream(device=dev)
            lane["eng"] = DepthmapEngine(dev, stream=lane["stream"].cuda_stream)

    def take_buffers(lane):
        """two sets per lane: one being written while the next view runs; blocks only when both are still in the writer pool"""
        if lane["free"].empty() and lane["sets"] < 2:
            lane["sets"] += 1
            return out_buffers()
        return lane["free"].get()

    add("setup_s", time.perf_counter() - t0)
    done, writes, infos = [], [], {}
    marks = dict(first_view_start=None, last_view_done=None)

    def write_view(out_dir, bufs, free):
        t = time.perf_counter()
        os.makedirs(out_dir, exist_ok=True)
        for name, b in zip(("TSAR_disp.dmb", "TSAR_normals.dmb", "TSAR_confidence.dmb"), bufs):
            tmp = os.path.join(out_dir, name + ".part")
            with open(tmp, "wb", buffering=0) as f:
                f.write(memoryview(b.numpy()))
            os.replace(tmp, os.path.join(out_dir, name))     # a file under its final name is always complete (-resume)
        free.put(bufs)
        add("write_s", time.perf_counter() - t)

    def process(k, lane):
        eng = lane["eng"]
        r = mine[k]
        sel = [r] + neigh[r]
        Ks = []
        for i in sel:
            K = krt[i][0].copy()
            K[:2] /= opt["cam_scale"]
            Ks.append(K)
        dmin = opt["depth_min"] if opt["depth_min"] > 0 else krt[r][3]
        dmax = opt["depth_max"] if opt["depth_max"] > 0 else krt[r][4]
        cams = scene.cameras_from_krt(Ks, [krt[i][1] for i in sel], [krt[i][2] for i in sel], dmin, dmax)
        f = float(np.float32(cams[0]["f"]))
        params = make_params(box=opt["blocksize"], iterations=opt["iterations"], n_best=opt["n_best"], cost_comb=opt["cost_comb"],
                             min_disparity=float(np.float32(f / np.float32(dmax))), max_disparity=float(np.float32(f / np.float32(dmin))))
        eng.set_views_device([device_image(i).data_ptr() for i in sel], W, H, cameras_to_struct(cams), list(range(1, len(sel))), cam_f=f)
        eng.set_params(params)
        _, u8, bgr = fut[r].result()
        out_dir = os.path.join(mslp, "APD", names[r][:8])
        bufs = take_buffers(lane)
        view = dict(gray_u8=u8, bgr=bgr, apd_dir=out_dir, seed=int(opt["seed"]) + r, cam_f=f)
        t = time.perf_counter()
        with stats_lock:
            if marks["first_view_start"] is None:
                marks["first_view_start"] = t - t0
        _, _, _, info = run_view(eng, opt, view, outputs=tuple(b.data_ptr() + 16 for b in bufs))
        add("detect_s", info.get("detect_s", 0.0))      # host stage of run_view (weak-texture detector)
        add("gpu_wait_s", time.perf_counter() - t - info.get("detect_s", 0.0))
        infos[r] = {k_: v for k_, v in info.items() if k_ != "slic_labels"}
        if opt["no_write"]:
            lane["free"].put(bufs)
        else:
            writes.append(io_pool.submit(write_view, out_dir, bufs, lane["free"]))
        done.append(r)
        marks["last_view_done"] = time.perf_counter() - t0
        return r

    ticket, ticket_lock = itertools.count(), threading.Lock()

    def lane_worker(j):     # one host thread per lane (a context is never shared); views are taken from a shared queue,
        lane_ready(lanes[j])
        while True:         # so lanes stay balanced when the views' neighbour counts differ (SURVEY section 8e)
            with ticket_lock:
                k = next(ticket)
            if k >= len(mine):
                return
            process(k, lanes[j])

    with cf.ThreadPoolExecutor(n_lanes) as ex:
        for fu in [ex.submit(lane_worker, j) for j in range(n_lanes)]:
            fu.result()
    for w in writes:
        w.result()
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    launches = sum(lane["eng"].launch_count() for lane in lanes[:n_lanes]) - launches0
    if not persistent:
        for lane in lanes:
            lane["eng"].close()
    io_pool.shutdown()
    stats["until_first_view_s"] = marks["first_view_start"] or 0.0      # timeline of the pass (not summed over threads)
    stats["after_last_view_s"] = dt - (marks["last_view_done"] or dt)
    res = dict(rank=rank, world=world, views=len(done), skipped=len(skipped), images=len(names), W=W, H=H, seconds=dt, depthmaps_per_s=len(done) / dt,
               lanes=n_lanes, io_threads=int(opt["io_threads"]), gpu_launches=int(launches),
               host_seconds={k: round(v, 3) for k, v in stats.items()},
               bytes_decoded=int(sum(os.path.getsize(os.path.join(folder, names[i])) for i in needed)),
               bytes_written=0 if opt["no_write"] else int(len(done) * (48 + 20 * npx)),
               weak_regions=int(sum(v.get("weak_regions", 0) for v in infos.values())))
    if not quiet:
        print(f"[tsar_cli] rank {rank}/{world}: {len(done)} of {len(names)} reference views ({W}x{H}) in {dt:.2f} s "
              f"({len(done) / dt:.2f} depthmaps/s incl. decoding and .dmb writing) -> {os.path.join(mslp, 'APD')}\n"
              f"[tsar_cli] host seconds (summed over threads): {res['host_seconds']}")
    return res


if __name__ == "__main__":
    sys.exit(run(sys.argv[1:]))
