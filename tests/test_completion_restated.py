"""The stages after PatchMatch against independent restatements, on fresh inputs at production sizes:
  * per-region RANSAC fit (tsar_fit_region_planes) vs the C restatement oc_fit_region_plane (oracle/oracle_cpu.c), bit-exact;
  * gipuma_WMF (cooperative and per-thread kernels) and gipuma_WMF_Final vs a float64 restatement (oracle/completion_ref.py);
  * the per-pixel completion kernels vs float64 restatements (same module).
No digest and no reference build is involved, so every input is new: TSAR_COMPLETION_SEED picks another campaign.
The hand-built cases at the end pin the weighted-median restatement itself and run without a GPU."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import completion_ref as cr

SEED = int(os.environ.get("TSAR_COMPLETION_SEED", "20261020"))
REL = 1e-5


def _same_or_nan(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def _close(got, want, mag=None):
    """float32 result within REL of max(|want|, mag); NaN only where NaN is expected, infinities equal."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = np.abs(want) if mag is None else np.maximum(np.abs(want), mag)
    with np.errstate(invalid="ignore"):
        ok = np.abs(got - want) <= REL * scale
    return ok | (np.isnan(got) & np.isnan(want)) | (np.isinf(want) & (got == want))


def _engine(pkg, W, H, fx, min_disp, max_disp, rng):
    """A context on a two-image rig of size W x H; the reference image has continuous (non-8-bit) values."""
    cams = pkg.scene.make_cameras(W, H, 2, fx, 4.0, 6.0)
    cam_f = float(np.float32(cams[0]["f"]))
    y, x = np.mgrid[0:H, 0:W]
    img = (128 + 50 * np.sin(x / 7.0) * np.cos(y / 11.0) + 20 * rng.rand(H, W)).astype(np.float32)
    eng = pkg.DepthmapEngine(0)
    eng.set_views([img, img[:, ::-1].copy()], cams, [1], cam_f=cam_f)
    eng.set_params(pkg.make_params(box=11, iterations=1, min_disparity=min_disp, max_disparity=max_disp))
    return eng, cams, cam_f, img


# ---- 1. region fit at production sizes ------------------------------------------------------------------------------
RF_W, RF_H = 1600, 1200
BIG = {0: 1_000_000, 1: 120_000, 2: 49_998, 3: 49_999, 4: 50_000, 5: 50_001}
SKIPPED = {6: (1.0, 100_000), 7: (0.0, 60_000)}   # large regions that are not weak: never fitted
N_SMALL = 340                                       # weak regions of 1...60 points: more than the 296 CTAs of the grid
N_EMPTY = 8                                         # weak regions without any reliable point
N_LATER = 100                                       # small regions that only the second call fits (regrows the scratch)


def _fit_maps(pkg, rng):
    cams = pkg.scene.make_cameras(RF_W, RF_H, 2, 1400.0, 4.0, 6.0)
    cam_f = float(np.float32(cams[0]["f"]))
    first_small = 8
    first_empty = first_small + N_SMALL
    first_later = first_empty + N_EMPTY
    n_reg = first_later + N_LATER
    rel = np.zeros(n_reg, np.int64)
    unrel = np.zeros(n_reg, np.int64)
    for r, n in BIG.items():
        rel[r], unrel[r] = n, n // 20
    for r, (_, n) in SKIPPED.items():
        rel[r] = n
    small = rng.randint(3, 61, N_SMALL)
    small[:12] = [1, 2] * 6                          # degenerate triples: NaN planes
    rel[first_small:first_empty] = small
    unrel[first_empty:first_later] = 300
    rel[first_later:] = rng.randint(1, 61, N_LATER)
    n_px = RF_W * RF_H
    lab = np.concatenate([np.repeat(np.arange(n_reg), rel), np.repeat(np.arange(n_reg), unrel)])
    sc = np.concatenate([np.ones(rel.sum()), rng.choice([0.0, 0.5, 2.0], unrel.sum())])
    rest = n_px - len(lab)
    assert rest > 0
    lab = np.concatenate([lab, np.full(rest, -1)])  # unlabelled pixels, reliable or not
    sc = np.concatenate([sc, (rng.rand(rest) < 0.5).astype(np.float64)])
    perm = rng.permutation(n_px)
    lab, sc = lab[perm].reshape(RF_H, RF_W), sc[perm].reshape(RF_H, RF_W)
    canny = lab.astype(np.float32)
    frac = (lab >= first_small) & (rng.rand(RF_H, RF_W) < 0.5)
    canny[frac] += np.float32(0.5)                   # C truncation: r + 0.5 is region r ...
    zero = np.nonzero((lab == 0).ravel())[0][:1000]
    canny.ravel()[zero] = np.float32(-0.5)           # ... and -0.5 is region 0
    # a plane per region, facing the camera, through a point at depth 3...5 on the optical axis
    nrm = np.stack([rng.uniform(-0.4, 0.4, n_reg), rng.uniform(-0.4, 0.4, n_reg), -np.ones(n_reg)], axis=1)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    d = -nrm[:, 2] * rng.uniform(3.0, 5.0, n_reg)
    Kinv = np.asarray(cams[0]["K_inv"], np.float64)
    y, x = np.mgrid[0:RF_H, 0:RF_W].astype(np.float64)
    ray = np.stack([x, y, np.ones_like(x)], axis=-1) @ Kinv.T
    li = np.maximum(lab, 0)
    z = -d[li] / np.sum(nrm[li] * ray, axis=-1)
    z = np.where(lab >= 0, z, rng.uniform(3.0, 6.0, z.shape))
    disp = cam_f / z * (1 + 0.0005 * rng.normal(size=z.shape))
    out = rng.rand(RF_H, RF_W) < 0.2
    disp[out] *= rng.uniform(0.8, 1.2, int(out.sum()))
    text = np.ones(n_reg, np.float32)
    text[:6] = -1.0
    for r, (t, _) in SKIPPED.items():
        text[r] = t
    text[first_small:first_later] = -1.0
    size = (np.bincount(lab[lab >= 0], minlength=n_reg) / 16.0).astype(np.float32)
    return dict(cams=cams, cam_f=cam_f, disp=disp.astype(np.float32), scale=sc.astype(np.float32), canny=canny,
                text=text, size=size, normal=nrm, n_reg=n_reg, rel=rel, later=np.arange(first_later, n_reg),
                empty=np.arange(first_empty, first_later))


@pytest.mark.gpu
def test_region_fit_at_production_sizes_matches_restatement(pkg):
    """tsar_fit_region_planes on 1600 x 1200 maps against oc_fit_region_plane region by region, bit-exact (NaN = NaN):
    regions of 49 998 ... 50 001, 120 000 and 1 000 000 reliable points (lists of up to 50 000 points are used whole,
    longer ones are cut to an evenly strided 49 999), 340 small weak regions (more than the cooperative grid has CTAs),
    weak regions without reliable points (plane kept), large regions that are not weak (skipped); host-supplied and
    device-generated streams; a second call with more weak regions (regrows the scratch) and a third with fewer."""
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    L = pkg._lib
    rng = np.random.RandomState(SEED)
    m = _fit_maps(pkg, rng)
    n_reg, text = m["n_reg"], m["text"]
    cams = cameras_to_struct(m["cams"])
    eng = pkg.DepthmapEngine(0)
    eng.set_views([np.zeros((RF_H, RF_W), np.float32)] * 2, cams, [1], cam_f=m["cam_f"])
    eng.set_params(pkg.make_params())
    eng.upload(L.F_DEPTH, m["disp"]); eng.upload(L.F_SCALE, m["scale"]); eng.upload(L.F_CANNY, m["canny"])
    per = eng.lib.tsar_ransac_rand_per_region()
    rnd = rng.randint(0, 2 ** 31 - 1, size=(n_reg, per)).astype(np.uint32)
    p0 = np.tile(np.array([0, 0, 1, -1], np.float32), (n_reg, 1))
    p0[:, 3] -= np.arange(n_reg, dtype=np.float32)   # a distinct starting plane per region
    seed = int(rng.randint(1, 2 ** 31))
    cb.build()
    cache = {}

    def oracle(regions, stream):
        todo = [r for r in regions if (stream, r) not in cache]
        def one(r):
            with np.errstate(over="ignore"):
                s = rnd[r] if stream == "host" else eng.ransac_rand_stream(seed, r)
            return r, cb.fit_region_plane(L.TsarCamera, cams[0], m["cam_f"], m["disp"], m["scale"], m["canny"], r,
                                          m["size"][r], s, p0[r])
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
            for r, res in ex.map(one, todo):
                cache[(stream, r)] = res
        return {r: cache[(stream, r)] for r in regions}

    def check(fitted, txt, stream):
        weak = [r for r in range(n_reg) if txt[r] == -1]
        want = oracle(weak, stream)
        for r in range(n_reg):
            if txt[r] != -1:
                assert np.array_equal(fitted[r], p0[r]), (r, fitted[r])
                continue
            plane, used = want[r]
            assert used == (m["rel"][r] if m["rel"][r] <= 50000 else 49999), (r, used)
            assert _same_or_nan(fitted[r], plane).all(), (stream, r, m["rel"][r], fitted[r], plane)
        return weak

    t0 = text.copy()
    t0[m["later"]] = 1.0
    fitted = eng.fit_region_planes(t0, m["size"], rnd, p0)
    weak = check(fitted, t0, "host")
    assert len(weak) > 296
    assert np.isnan(fitted[:, 0]).sum() >= 6                      # 1-point regions: every triple is 0/0
    for r in m["empty"]:
        assert np.array_equal(fitted[r], p0[r])
    for r in BIG:                                                  # the geometry is right, up to sign
        cosang = abs(np.dot(fitted[r][:3].astype(np.float64), m["normal"][r])) / np.linalg.norm(fitted[r][:3])
        assert cosang > np.cos(np.radians(3.0)), (r, fitted[r], m["normal"][r])
    seeded = eng.fit_region_planes(t0, m["size"], None, p0, seed=seed)
    check(seeded, t0, "seeded")
    assert not _same_or_nan(seeded[:6], fitted[:6]).all()
    grown = eng.fit_region_planes(text, m["size"], rnd, p0)        # more weak regions: the scratch grows
    check(grown, text, "host")
    fl = int(m["later"][0])
    assert _same_or_nan(grown[:fl], fitted[:fl]).all()
    fewer = text.copy()
    fewer[:2] = 1.0
    fewer[8:200] = 1.0
    again = eng.fit_region_planes(fewer, m["size"], rnd, p0)
    check(again, fewer, "host")
    eng.close()


# ---- 2. weighted-median stages ----------------------------------------------------------------------------------------
PALETTE_N = np.array([[-0.0, 0.0, -1.0], [0.0, -0.0, -1.0], [-0.0, 0.28, -0.96], [0.6, -0.0, -0.8],
                      [-0.28, 0.0, -0.96], [0.2, -0.2, -0.959166], [-0.3, -0.3, -0.905539], [0.1, 0.15, -0.983298]])


def _wmf_state(g, W, H, rng):
    """Tie-rich planes (blocks of a palette of 8, -0.0 components), disparities from the planes (some perturbed, some
    from a palette of 4), reliable densities 3 % / 30 % / 97 % by row thirds and a band of columns with none."""
    pal = PALETTE_N.astype(np.float32)
    pal_w = (-pal[:, 2].astype(np.float64) * rng.uniform(3.5, 5.0, len(pal))).astype(np.float32)
    blk = rng.randint(0, len(pal), ((H + 47) // 48, (W + 47) // 48))
    idx = np.kron(blk, np.ones((48, 48), np.int64))[:H, :W]
    plane = np.concatenate([pal[idx], pal_w[idx][..., None]], axis=-1)
    pert = rng.rand(H, W) < 0.3
    n = plane[pert, :3].astype(np.float64) + rng.uniform(-0.08, 0.08, (int(pert.sum()), 3))
    plane[pert, :3] = (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32)
    x, y = cr.pixel_grid(H, W)
    dep, _ = g.plane_depth(plane, x, y)
    disp = g.fb / dep
    odd = rng.rand(H, W)
    disp = np.where(odd < 0.15, disp * rng.uniform(0.85, 1.15, (H, W)), disp)
    disp = np.where(odd > 0.95, rng.choice(g.fb / np.array([3.0, 4.0, 4.5, 6.0]), (H, W)), disp)
    density = np.where(y < H / 3, 0.03, np.where(y < 2 * H / 3, 0.30, 0.97))
    scale = (rng.rand(H, W) < density).astype(np.float32)
    b0 = int(W * 0.55)
    scale[:, b0:b0 + max(1, min(200, W // 5))] = 0.0
    return plane, disp.astype(np.float32), scale


def _counts(mask, radius, gap):
    """Reliable lattice neighbours of every pixel."""
    H, W = mask.shape
    pad = np.pad(mask.astype(np.int32), radius)
    out = np.zeros((H, W), np.int32)
    for i in range(-radius, radius + 1, gap):
        for j in range(-radius, radius + 1, gap):
            out += pad[radius + j:radius + j + H, radius + i:radius + i + W]
    return out


def _sample(H, W, counts, extra, n, rng):
    """Every pixel of small images; else the first and last 8 columns, border rows, pixels with 0, 1 or 2 reliable
    neighbours (and those of `extra`), and random ones up to about n."""
    if n is None or H * W <= n:
        y, x = np.mgrid[0:H, 0:W]
        return x.ravel(), y.ravel()
    keep = np.zeros((H, W), bool)
    keep[:, :8] = keep[:, -8:] = True
    keep[[0, 1, H - 2, H - 1], :] = True
    for k in (0, 1, 2):
        ids = np.flatnonzero(counts == k)
        keep.ravel()[rng.choice(ids, min(len(ids), 3000), replace=False)] = True
    if extra is not None:
        ids = np.flatnonzero(extra)
        keep.ravel()[rng.choice(ids, min(len(ids), 8000), replace=False)] = True
    more = n - int(keep.sum())
    if more > 0:
        keep.ravel()[rng.choice(H * W, more, replace=False)] = True
    y, x = np.nonzero(keep)
    return x, y


def _chunks(f, xs, ys, size=8000):
    parts = [f(xs[k:k + size], ys[k:k + size]) for k in range(0, len(xs), size)]
    return [np.concatenate([p[i] for p in parts]) for i in range(len(parts[0]))]


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,n", [(1920, 1080, 50000), (1917, 1079, 50000), (261, 9, None), (9, 261, None), (67, 33, None)])
def test_weighted_median_stages_match_float64_restatement(pkg, monkeypatch, W, H, n):
    """gipuma_WMF (cooperative kernel and TSAR_B200_WMF_PER_THREAD=1) levels 0..3 and gipuma_WMF_Final levels 0..5, each
    level judged on its own from the library's state before it: flags and the median choice identical on every decided
    pixel, planes and disparities within 1e-5; undecided pixels (near-ties of running sums or bounds) below 0.1 %."""
    L = pkg._lib
    rng = np.random.RandomState(SEED + W * 7 + H)
    fx = float(max(W, H))
    eng, cams, cam_f, img = _engine(pkg, W, H, fx, fx / 9.0, fx / 4.0, rng)
    params = eng.params
    g = cr.Glue(cams[0], cam_f, params.min_disparity, params.max_disparity)
    plane, disp, scale0 = _wmf_state(g, W, H, rng)
    blk = rng.randint(0, 10 ** 6, ((H + 63) // 64, (W + 63) // 64))
    canny = (np.kron(blk, np.ones((64, 64), np.int64))[:H, :W] % 40).astype(np.float32)
    canny[rng.rand(H, W) < 0.05] = -1.0
    text = rng.choice(np.array([1.0, 1.0, -1.0, 0.0], np.float32), 40)
    text[:3] = [1.0, -1.0, 0.0]
    eng.set_regions(text, np.zeros((40, 4), np.float32))
    eng.upload(L.F_CANNY, canny)
    eng.upload(L.F_NORM4, plane); eng.upload(L.F_DEPTH, disp)
    stats = dict(px=0, undecided=0, changed=0, dummy_px=0)
    cache = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("TSAR_B200_WMF_PER_THREAD", mode)
        eng.upload(L.F_SCALE, scale0)
        for it in range(4):
            po = 1 << it
            s_in = eng.download(L.F_SCALE)
            eng.wmf(it)
            s_out = eng.download(L.F_SCALE)
            key = (it, s_in.tobytes())
            if key not in cache:
                cnt = _counts(s_in == 1.0, 80 // po, 16 // po)
                xs, ys = _sample(H, W, cnt, None, n, rng)
                flag, und = _chunks(lambda a, b: cr.wmf(g, img, plane, disp, s_in, it, a, b), xs, ys)
                cache[key] = (xs, ys, flag, und, cnt[ys, xs])
            xs, ys, flag, und, cnt = cache[key]
            bad = ~und & (s_out[ys, xs] != flag)
            assert not bad.any(), (mode, it, int(bad.sum()), list(zip(xs[bad][:5], ys[bad][:5])), cnt[bad][:5])
            stats["px"] += len(xs); stats["undecided"] += int(und.sum())
            stats["changed"] += int((flag != s_in[ys, xs]).sum()); stats["dummy_px"] += int((cnt <= 2).sum())
    monkeypatch.delenv("TSAR_B200_WMF_PER_THREAD")
    eng.upload(L.F_SCALE, scale0)
    for it in range(6):
        po = 1 << it
        p_in, d_in, s_in = eng.download(L.F_NORM4), eng.download(L.F_DEPTH), eng.download(L.F_SCALE)
        eng.wmf_final(it)
        p_out, d_out, s_out = eng.download(L.F_NORM4), eng.download(L.F_DEPTH), eng.download(L.F_SCALE)
        cnt = _counts(s_in == 1.0, 5 * po, po)
        reg = cr.region_of(canny, len(text))
        cand = (reg >= 0) & (s_in == 0.0) & (text[np.maximum(reg, 0)] == 1.0)
        xs, ys = _sample(H, W, np.where(cand, cnt, -1), cand & (np.abs(cnt - 32 // po) <= 1), n, rng)
        filled, nm, mag_w, dd, sc, und = _chunks(
            lambda a, b: cr.wmf_final(g, img, p_in, d_in, s_in, canny, text, it, a, b), xs, ys)
        keep = ~filled & ~und
        assert _same_or_nan(p_out[ys, xs][keep], p_in[ys, xs][keep]).all(), (it, "plane of an unfilled pixel changed")
        assert _same_or_nan(d_out[ys, xs][keep], d_in[ys, xs][keep]).all() and np.array_equal(s_out[ys, xs][keep], s_in[ys, xs][keep])
        f = filled & ~und
        got = p_out[ys, xs][f]
        assert np.array_equal(s_out[ys, xs][f], sc[f].astype(np.float32)), (it, "flags")
        assert _close(got[:, :3], nm[f][:, :3]).all(), (it, "median normal")
        assert _close(got[:, 3], nm[f][:, 3], mag_w[f]).all(), (it, "plane offset")
        assert _close(d_out[ys, xs][f], dd[f]).all(), (it, "disparity")
        stats["px"] += len(xs); stats["undecided"] += int(und.sum()); stats["changed"] += int(f.sum())
        stats[f"final{it}_filled"] = int(f.sum())
        stats[f"final{it}_at_bound"] = int((f & (cnt[ys, xs] == 32 // po)).sum())
        stats["clamped"] = stats.get("clamped", 0) + int((f & (sc == 0)).sum())
    eng.close()
    frac = stats["undecided"] / stats["px"]
    print(f"\n[wmf {W}x{H}] {stats}; undecided fraction {frac:.5%}")
    assert frac < 1e-3
    assert stats["changed"] > 0.01 * stats["px"]
    if n is not None:
        assert stats["dummy_px"] > 1000 and stats["final0_at_bound"] > 0 and stats["final4_at_bound"] > 0
        assert 0 < stats["clamped"] < sum(stats[f"final{it}_filled"] for it in range(6))


# ---- 3. per-pixel completion kernels ----------------------------------------------------------------------------------
C2_W, C2_H = 3100, 2050


@pytest.mark.gpu
def test_completion_kernels_at_c2_size_match_float64_restatement(pkg):
    """get_disp, getview, scale_from_confidence, scale_from_weak_png, update_scale_2, update_scale and compute_disp on
    3100 x 2050 maps with a 3 300-entry region table (text -1 / 1 / 0, planes facing towards and away from the camera, a
    NaN plane), labels -1, >= n_regions and fractional (C truncation), NaN pixel planes and costs equal to MAXCOST.
    Replaced pixels, costs and flags exact; floats within 1e-5; near-singular pixels excluded and counted."""
    L = pkg._lib
    rng = np.random.RandomState(SEED + 3)
    W, H = C2_W, C2_H
    eng, cams, cam_f, _ = _engine(pkg, W, H, 1750.0, 1750.0 / 9.0, 1750.0 / 2.0, rng)
    g = cr.Glue(cams[0], cam_f, eng.params.min_disparity, eng.params.max_disparity)
    x, y = cr.pixel_grid(H, W)
    view = g.view_vector(x, y)
    excluded = np.zeros((H, W), bool)

    # per-pixel planes facing the camera; a few degenerate ones (zero normal) and NaN offsets (depth 1000)
    n = -view + rng.uniform(-0.35, 0.35, (H, W, 3))
    n /= np.linalg.norm(n, axis=-1, keepdims=True)
    w = np.sum(n * view, axis=-1) * -rng.uniform(3.0, 6.0, (H, W))
    plane = np.concatenate([n, w[..., None]], axis=-1).astype(np.float32)
    plane[rng.rand(H, W) < 0.005, 3] = np.nan
    plane[rng.rand(H, W) < 0.0005, :3] = 0.0
    cost = rng.uniform(0, 2, (H, W)).astype(np.float32)
    cost[rng.rand(H, W) < 0.05] = np.float32(cr.MAXCOST)
    lrdiff = rng.uniform(0, 1, (H, W)).astype(np.float32)

    # get_disp: imported world normals and disparities
    wn = plane.copy()
    wn[..., :3] = (plane[..., :3].astype(np.float64) @ g.Rorig_inv.T).astype(np.float32)
    wdisp = (g.fb / rng.uniform(3.0, 6.0, (H, W))).astype(np.float32)
    eng.upload(L.F_NORM4, wn); eng.upload(L.F_DEPTH, wdisp)
    eng.get_disp()
    got = eng.download(L.F_NORM4)
    want, mag_n, mag_d = cr.get_disp(g, wn, wdisp)
    assert _close(got[..., :3], want[..., :3], mag_n).all()
    assert _close(got[..., 3], want[..., 3], mag_d).all()

    # getview: confidence and disparity
    eng.upload(L.F_NORM4, plane); eng.upload(L.F_COST, cost); eng.upload(L.F_LRDIFF, lrdiff)
    eng.getview()
    confid, gdisp = eng.download(L.F_CONFID), eng.download(L.F_DEPTH)
    w_conf, w_disp, sing = cr.getview(g, plane, cost, lrdiff)
    excluded |= sing
    assert _close(confid, w_conf).all()
    assert _close(gdisp, w_disp)[~sing].all()
    assert (gdisp[np.isnan(plane[..., 3])] == np.float32(g.fb / 1000.0)).all()

    # reliable flags
    eng.scale_from_confidence(0.6)
    assert np.array_equal(eng.download(L.F_SCALE), cr.scale_from_confidence(confid, 0.6))
    prior = rng.choice(np.array([0.0, 0.5, 1.0, 7.0], np.float32), (H, W))
    kinds = np.array([[255, 255, 255], [0, 255, 0], [0, 0, 255], [255, 0, 0], [0, 255, 255], [254, 255, 255]], np.uint8)
    bgr = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
    pick = rng.randint(0, len(kinds) + 2, (H, W))
    for k, col in enumerate(kinds):
        bgr[pick == k] = col
    eng.upload(L.F_SCALE, prior)
    eng.scale_from_weak_png(bgr)
    assert np.array_equal(eng.download(L.F_SCALE), cr.scale_from_weak_png(bgr, prior))

    # region table: 3 300 regions, planes towards and away from the camera, one NaN plane
    n_reg = 3300
    rn = np.stack([rng.uniform(-0.45, 0.45, n_reg), rng.uniform(-0.45, 0.45, n_reg), rng.choice([-1.0, 1.0], n_reg)], axis=1)
    rn /= np.linalg.norm(rn, axis=1, keepdims=True)
    rw = -rn[:, 2] * rng.uniform(3.0, 6.0, n_reg)
    rplane = np.concatenate([rn, rw[:, None]], axis=1).astype(np.float32)
    text = rng.choice(np.array([-1.0, 1.0, 0.0], np.float32), n_reg, p=[0.5, 0.3, 0.2])
    text[:4] = -1.0
    rplane[1, 3] = np.nan
    blk = rng.randint(0, n_reg, ((H + 36) // 37, (W + 36) // 37))
    canny = np.kron(blk, np.ones((37, 37), np.int64))[:H, :W].astype(np.float32)
    u = rng.rand(H, W)
    canny[u < 0.02] = -1.0
    canny[(u >= 0.02) & (u < 0.03)] = n_reg
    canny[(u >= 0.03) & (u < 0.04)] = n_reg + 17
    canny[(u >= 0.04) & (u < 0.05)] = 3.7                         # -> region 3
    canny[(u >= 0.05) & (u < 0.06)] = -0.5                        # -> region 0
    canny[(u >= 0.06) & (u < 0.07)] += np.float32(0.25)
    eng.set_regions(text, rplane)
    eng.upload(L.F_CANNY, canny)
    fake0 = rng.uniform(1, 9, (H, W)).astype(np.float32)
    eng.upload(L.F_FAKEDEPTH, fake0)
    eng.update_scale_2()
    fake, rep, und = cr.update_scale_2(g, fake0, canny, text, rplane)
    excluded |= und
    got = eng.download(L.F_FAKEDEPTH)
    assert _close(got, fake)[~und].all()
    assert np.array_equal(got[~rep], fake0[~rep])
    assert rep.mean() > 0.2 and (rep & (canny == 3.7)).any() and (rep & (canny == -0.5)).any()

    # update_scale: state from before the stage
    scale_in = eng.download(L.F_SCALE)
    eng.upload(L.F_NORM4, plane); eng.upload(L.F_COST, cost)
    eng.update_scale()
    w_pl, w_cost, w_scale, w_disp, rep2, und = cr.update_scale(g, plane, cost, scale_in, canny, text, rplane)
    excluded |= und
    assert np.array_equal(rep, rep2)
    got_pl, got_cost, got_scale, got_disp = (eng.download(f) for f in (L.F_NORM4, L.F_COST, L.F_SCALE, L.F_DEPTH))
    assert np.array_equal(got_cost, w_cost.astype(np.float32)) and np.array_equal(got_scale, w_scale.astype(np.float32))
    assert _same_or_nan(got_pl, w_pl.astype(np.float32))[~und].all()
    assert _close(got_disp, w_disp)[~und].all()
    reg = cr.region_of(canny, n_reg)
    flipped = rep & (np.sum(rplane[np.maximum(reg, 0)][..., :3] * view, axis=-1) > 0)
    assert flipped.mean() > 0.05 and (rep & ~flipped).mean() > 0.05
    assert (reg[rep] == 1).any()                                  # the NaN region plane was spread (depth 1000)

    # compute_disp: state from before the stage (costs of MAXCOST kept outside the replaced pixels)
    pl_in, cost_in = eng.download(L.F_NORM4), eng.download(L.F_COST)
    assert (cost_in == np.float32(cr.MAXCOST)).sum() > 1000
    eng.compute_disp()
    out = eng.download(L.F_NORM4)
    want, mag, sing = cr.compute_disp(g, pl_in, cost_in)
    excluded |= sing
    assert _close(out[..., :3], want[..., :3], mag).all()
    assert _close(out[..., 3], want[..., 3])[~sing].all()
    assert (out[..., 3][cost_in == np.float32(cr.MAXCOST)] == 0).all()
    eng.close()
    print(f"\n[completion] excluded {excluded.mean():.6%} of {W}x{H} pixels")
    assert excluded.mean() < 1e-3


# ---- restatement pinned by hand (no GPU) ------------------------------------------------------------------------------
def _lists(entries):
    """One row of weighted_medians inputs from {slot: (weight, depth, nx, ny, nz)}."""
    w, valid = np.zeros((1, cr.N_SLOTS)), np.zeros((1, cr.N_SLOTS), bool)
    keys = [np.zeros((1, cr.N_SLOTS)) for _ in range(4)]
    for s, (wt, *k) in entries.items():
        w[0, s], valid[0, s] = wt, True
        for q in range(4):
            keys[q][0, s] = k[q]
    return w, keys, valid


def test_restated_median_one_neighbour_is_the_dummy():
    """One reliable neighbour of positive depth: the sorted list is (dummy, neighbour), only position 0 counts, wSum = 0,
    so the dummy reaches half -- for the depth and for every component the neighbour exceeds (0 < 0.3)."""
    hit, num, und, alt = cr.weighted_medians(*_lists({17: (0.7, 40.0, 0.3, -0.3, -0.9)}))
    assert num[0] == 1 and not und[0] and alt[0] == -2
    assert list(hit[:, 0]) == [cr.N_SLOTS, cr.N_SLOTS, 17, 17]


def test_restated_median_equal_keys_first_slot_wins():
    entries = {1: (1.0, 4.0, 0, 0, -1), 3: (2.0, 5.0, 0, 0, -1), 7: (1.0, 5.0, 0, 0, -1), 9: (1.5, 5.0, 0, 0, -1),
               20: (1.0, 6.0, 0, 0, -1)}
    hit, _, und, alt = cr.weighted_medians(*_lists(entries))
    # depth order: dummy, 1, 3, 7, 9, (20 dropped) -> wSum 5.5, half 2.75, sums 0, 1, 3 -> slot 3 (ties in reverse slot
    # order would give 0, 1, 2.5, 3.5 -> slot 7)
    assert hit[0, 0] == 3 and not und[0] and alt[0] == -2


def test_restated_median_drops_the_largest_element():
    hit, _, und, alt = cr.weighted_medians(*_lists({0: (1.2, 1.0, 0, 0, -1), 1: (1.0, 2.0, 0, 0, -1), 2: (10.0, 3.0, 0, 0, -1)}))
    # with the heavy largest element the median would be slot 2; it drops out: wSum = 2.2, half 1.1 -> slot 0
    assert hit[0, 0] == 0 and not und[0] and alt[0] == -2


def test_restated_median_negative_zero_ties_with_zero():
    """x keys +0.0 (slot 2), -0.0 (slot 5), the dummy's 0, 0.5, 0.7: -0 equals +0, so slot 2 stays first and the running
    sum reaches half (1.5) at slot 5; ordering -0 below +0 would pick slot 2."""
    entries = {2: (1.0, 1.0, 0.0, 0, -1), 5: (1.0, 2.0, -0.0, 0, -1), 8: (1.0, 3.0, 0.5, 0, -1), 11: (1.0, 4.0, 0.7, 0, -1)}
    hit, _, und, alt = cr.weighted_medians(*_lists(entries))
    assert hit[1, 0] == 5 and not und[0] and alt[0] == -2


def _tiny_glue(pkg, W, H):
    cams = pkg.scene.make_cameras(W, H, 2, 40.0, 4.0, 6.0)
    return cr.Glue(cams[0], float(np.float32(cams[0]["f"])), 40.0 / 9.0, 10.0)


def _tiny_state(g, W, H):
    plane = np.tile(np.array([0.0, 0.0, -1.0, 5.0], np.float32), (H, W, 1))   # disparity 8
    x, y = cr.pixel_grid(H, W)
    disp = (g.fb / g.plane_depth(plane, x, y)[0]).astype(np.float32)
    ref = (100.0 + (np.arange(H * W) * 0.618) % 7.0).reshape(H, W).astype(np.float32)   # no two weights alike
    return ref, plane, disp


def test_restated_wmf_no_neighbour_gives_flag_0_and_dummy_uses_pixel_0_0(pkg):
    W, H = 40, 40
    g = _tiny_glue(pkg, W, H)
    ref, plane, disp = _tiny_state(g, W, H)
    scale = np.zeros((H, W), np.float32)
    flag, und = cr.wmf(g, ref, plane, disp, scale, 3, [20], [20])
    assert flag[0] == 0.0 and not und[0]
    # one reliable neighbour: the dummy is the depth median -> the offset comes from pixel (0, 0) and its disparity
    scale[22, 20] = 1.0
    nm, _, num, und, _, _, has_alt = cr._median_plane(g, ref, plane, disp, scale, np.array([20]), np.array([20]), 10, 2, 1.0)
    assert num[0] == 1 and not und[0] and not has_alt[0]
    want, _ = g.plane_d(nm[0, :3], 0.0, 0.0, g.fb / float(disp[0, 0]))
    assert nm[0, 3] == want
    disp[0, 0] *= 2
    nm2 = cr._median_plane(g, ref, plane, disp, scale, np.array([20]), np.array([20]), 10, 2, 1.0)[0]
    assert nm2[0, 3] != nm[0, 3]


def test_restated_wmf_final_needs_enough_neighbours(pkg):
    """Level 0 fills only with at least 32 reliable neighbours (radius 5, gap 1); with 31 the pixel stays unchanged."""
    W, H = 30, 30
    g = _tiny_glue(pkg, W, H)
    ref, plane, disp = _tiny_state(g, W, H)
    canny = np.zeros((H, W), np.float32)
    text = np.array([1.0], np.float32)
    ys, xs = np.mgrid[10:21, 10:21]
    ring = [(yy, xx) for yy, xx in zip(ys.ravel(), xs.ravel()) if (yy, xx) != (15, 15)]
    for k, filled_want in ((31, False), (32, True)):
        scale = np.zeros((H, W), np.float32)
        for yy, xx in ring[:k]:
            scale[yy, xx] = 1.0
        filled, nm, _, _, sc, und = cr.wmf_final(g, ref, plane, disp, scale, canny, text, 0, [15], [15])
        assert filled[0] == filled_want and not und[0]
    assert np.allclose(nm[0, :3], [0, 0, -1]) and sc[0] == 1.0
    # not textured (text 0 or -1) or already reliable: never filled
    for t, s in ((0.0, 0.0), (-1.0, 0.0), (1.0, 1.0)):
        scale[15, 15] = s
        assert not cr.wmf_final(g, ref, plane, disp, scale, canny, np.array([t], np.float32), 0, [15], [15])[0][0]


def test_region_fit_restatement_uses_lists_of_50000_points_whole(pkg):
    """oc_fit_region_plane follows the library's rule: up to 50 000 reliable points are used whole (main.cpp:1541),
    longer lists are cut to 49 999 (main.cpp:1547-1549)."""
    from oracle import cpu_binding as cb
    from tsar_mvs_b200.engine import cameras_to_struct
    W, H = 400, 300
    cams = pkg.scene.make_cameras(W, H, 2, 350.0, 4.0, 6.0)
    cs = cameras_to_struct(cams)
    rng = np.random.RandomState(SEED)
    disp = rng.uniform(60, 120, (H, W)).astype(np.float32)
    canny = np.zeros((H, W), np.float32)
    rnd = rng.randint(0, 2 ** 31 - 1, 46000).astype(np.uint32)
    for n, used_want in ((50000, 50000), (50001, 49999)):
        scale = np.zeros(H * W, np.float32)
        scale[rng.choice(H * W, n, replace=False)] = 1.0
        _, used = cb.fit_region_plane(pkg._lib.TsarCamera, cs[0], float(np.float32(cams[0]["f"])), disp,
                                      scale.reshape(H, W), canny, 0, 5000.0, rnd, np.array([0, 0, 1, -1], np.float32))
        assert used == used_want
