"""TEST INFRASTRUCTURE -- float64 restatements of the stages after PatchMatch: the per-pixel completion kernels
(gipuma_get_disp, gipuma_getview, gipuma_update_scale_2, gipuma_update_scale, gipuma_compute_disp; gipuma.cu:732-755,
810-844, 1189-1292), the reliable flags (main.cpp:1499-1514) and the weighted-median stages gipuma_WMF /
gipuma_WMF_Final (gipuma.cu:1500-1698, 1295-1497).  Only tests/ may import this.

Written from the reference's semantics (DESIGN.md 4.5 and the kernel header comments), not ported from the kernels:
numpy, vectorised over pixels, every quantity in float64 from the float32 inputs.  Each function also says where float32
arithmetic may legitimately decide otherwise:
  * `singular` -- a depth denominator (or a plane offset from a cancelling sum) below 1e-3 of the sum of its terms'
    magnitudes, or a view-vector dot product within 1e-6 of 0 (the flip of a region plane);
  * `undecided` (weighted medians) -- a running weight sum within 1e-5 * wSum of half where the other candidate for the
    median would change the result, or a threshold / clamp comparison within 1e-5 of its bound (relative to the larger
    of the bound and the compared values).
Float results carry a magnitude `mag` (sum of the magnitudes of the terms that formed them): a float32 result is judged
within 1e-5 of max(|value|, mag)."""
import numpy as np

MAXCOST = 2.0
SING = 1e-3        # relative size below which a denominator counts as near-singular
FLIP_EPS = 1e-6    # |view . normal| below which the flip of a region plane is undecided
TIE = 1e-5         # relative window of running sums and threshold / clamp comparisons
N_SLOTS = 121      # 11 x 11 lattice neighbours; slot 121 is the dummy element


class Glue:
    """The reference camera's constants as the library receives them (float32 values, held as float64)."""

    def __init__(self, cam0, cam_f, min_disp, max_disp):
        f = lambda v: np.asarray(np.float32(v), np.float64)
        a = lambda k: np.asarray(cam0[k], np.float32).astype(np.float64)
        K = a("K").reshape(9)
        self.Minv, self.Rorig, self.Rorig_inv = a("M_inv").reshape(3, 3), a("R_orig").reshape(3, 3), a("R_orig_inv").reshape(3, 3)
        self.Pc, self.C = a("P_col34").reshape(3), a("C4").reshape(3)
        self.fx, self.alpha, self.cx, self.cy = f(cam0["fx"]), f(cam0["alpha"]), K[2], K[5]
        self.fb = f(np.float32(cam_f) * np.float32(cam0["baseline"]))
        self.min_disp, self.max_disp = f(min_disp), f(max_disp)

    def plane_depth(self, pl, x, y):
        """getDepthFromPlane3_cu (gipuma.cu:436-453): depth along the pixel ray; 1000 for a NaN offset.
        Returns (depth, singular)."""
        pl = np.asarray(pl, np.float64)
        t1 = pl[..., 2] * self.fx
        t2 = pl[..., 0] * (x - self.cx)
        t3 = self.alpha * (pl[..., 1] * (y - self.cy))
        den = t1 + t2 + t3
        nan_w = np.isnan(pl[..., 3])
        with np.errstate(divide="ignore", invalid="ignore"):
            dep = pl[..., 3] * -self.fx / den
        dep = np.where(nan_w, 1000.0, dep)
        singular = ~nan_w & (np.abs(den) <= SING * (np.abs(t1) + np.abs(t2) + np.abs(t3)))
        return dep, singular

    def plane_d(self, n, x, y, depth):
        """getD_cu (gipuma.cu:71-86): offset of the plane with normal n through the pixel's point at `depth`.
        Returns (d, mag)."""
        n = np.asarray(n, np.float64)
        pt = np.stack([x * depth - self.Pc[0], y * depth - self.Pc[1], depth - self.Pc[2]], axis=-1)
        mpt = np.stack([np.abs(x * depth) + abs(self.Pc[0]), np.abs(y * depth) + abs(self.Pc[1]),
                        np.abs(depth) + abs(self.Pc[2])], axis=-1)
        X = pt @ self.Minv.T
        mX = mpt @ np.abs(self.Minv).T
        return -np.sum(n * X, axis=-1), np.sum(np.abs(n) * mX, axis=-1)

    def view_vector(self, x, y):
        """getViewVector_cu (gipuma.cu:97-105), unit length."""
        pt = np.stack([x - self.Pc[0], y - self.Pc[1], np.full(np.shape(x), 1.0 - self.Pc[2])], axis=-1)
        v = pt @ self.Minv.T - self.C
        return v / np.linalg.norm(v, axis=-1, keepdims=True)

    def disparity(self, depth):
        with np.errstate(divide="ignore"):
            return self.fb / depth


def pixel_grid(H, W):
    y, x = np.mgrid[0:H, 0:W]
    return x.astype(np.float64), y.astype(np.float64)


# ---- per-pixel completion kernels -------------------------------------------------------------------------------
def get_disp(g, world_norm4, disp):
    """gipuma_get_disp: world normal -> reference frame; offset from the imported disparity.  Returns (plane, mag_xyz, mag_w)."""
    H, W = disp.shape
    x, y = pixel_grid(H, W)
    n = world_norm4[..., :3].astype(np.float64)
    nr = n @ g.Rorig.T
    mag_n = np.abs(n) @ np.abs(g.Rorig).T
    d, mag_d = g.plane_d(nr, x, y, g.disparity(disp.astype(np.float64)))
    return np.concatenate([nr, d[..., None]], axis=-1), mag_n, mag_d


def getview(g, plane, cost, lrdiff):
    """gipuma_getview: confidence ((2 - c) / 2 + (1 - lrdiff)) / 2 and the disparity of the plane.
    Returns (confid, disp, singular)."""
    H, W = cost.shape
    x, y = pixel_grid(H, W)
    confid = ((2.0 - cost.astype(np.float64)) / 2.0 + (1.0 - lrdiff.astype(np.float64))) / 2.0
    dep, sing = g.plane_depth(plane, x, y)
    return confid, g.disparity(dep), sing


def region_of(canny, n_regions):
    """Region index of each pixel: C truncation of the float label; -1 outside the table."""
    r = np.trunc(canny.astype(np.float64)).astype(np.int64)
    return np.where((r >= 0) & (r < n_regions), r, -1)


def _flipped_region_planes(g, canny, text, region_plane):
    """Pixels of textureless regions (text == -1) and their region plane turned to face the camera.
    Returns (replaced mask, plane per pixel, flip undecided mask)."""
    H, W = canny.shape
    reg = region_of(canny, len(text))
    rep = reg >= 0
    rep[rep] = np.asarray(text, np.float32)[reg[rep]] == -1.0
    pl = np.asarray(region_plane, np.float64)[np.where(rep, reg, 0)]
    x, y = pixel_grid(H, W)
    dot = np.sum(pl[..., :3] * g.view_vector(x, y), axis=-1)
    flip = dot > 0
    pl = np.where(flip[..., None], -pl, pl)
    return rep, pl, rep & (np.abs(dot) < FLIP_EPS)


def update_scale_2(g, fakedepth, canny, text, region_plane):
    """gipuma_update_scale_2: fakedepth <- depth of the (flipped) region plane in textureless regions.
    Returns (fakedepth, replaced, singular)."""
    H, W = canny.shape
    rep, pl, undecided = _flipped_region_planes(g, canny, text, region_plane)
    x, y = pixel_grid(H, W)
    dep, sing = g.plane_depth(pl, x, y)
    return np.where(rep, dep, fakedepth.astype(np.float64)), rep, undecided | (rep & sing)


def update_scale(g, plane, cost, scale, canny, text, region_plane):
    """gipuma_update_scale: textureless pixels take the flipped region plane, cost 0 and scale 1; every pixel gets the
    disparity of its plane.  Returns (plane, cost, scale, disp, replaced, singular)."""
    H, W = canny.shape
    rep, rpl, undecided = _flipped_region_planes(g, canny, text, region_plane)
    pl = np.where(rep[..., None], rpl, plane.astype(np.float64))
    x, y = pixel_grid(H, W)
    dep, sing = g.plane_depth(pl, x, y)
    return (pl, np.where(rep, 0.0, cost), np.where(rep, 1.0, scale), g.disparity(dep), rep, undecided | sing)


def compute_disp(g, plane, cost):
    """gipuma_compute_disp: world normal in xyz, depth in w (0 where the cost is MAXCOST).
    Returns (out, mag_xyz, singular)."""
    H, W = cost.shape
    x, y = pixel_grid(H, W)
    n = plane[..., :3].astype(np.float64)
    dep, sing = g.plane_depth(plane, x, y)
    keep = cost != np.float32(MAXCOST)
    out = np.concatenate([n @ g.Rorig_inv.T, np.where(keep, dep, 0.0)[..., None]], axis=-1)
    return out, np.abs(n) @ np.abs(g.Rorig_inv).T, keep & sing


def scale_from_confidence(confid, thr):
    """lines->scale = 1 where confid > thr (float32 comparison)."""
    return (np.asarray(confid, np.float32) > np.float32(thr)).astype(np.float32)


def scale_from_weak_png(bgr, scale):
    """main.cpp:1499-1514: white, green (0,255,0) and red (0,0,255) BGR pixels are reliable; others keep their value."""
    b, gr, r = (bgr[..., k].astype(np.int64) for k in range(3))
    hit = ((b == 255) & (gr == 255) & (r == 255)) | ((b == 0) & (gr == 255) & (r == 0)) | ((b == 0) & (gr == 0) & (r == 255))
    return np.where(hit, np.float32(1.0), scale).astype(np.float32)


# ---- weighted medians --------------------------------------------------------------------------------------------
def weighted_medians(w, keys, valid):
    """Weighted medians of one list per row, as gipuma_WMF(_Final) form them.

    w: [P, 121] weights; keys: four [P, 121] arrays (depth, nx, ny, nz); valid: [P, 121] -- slot c of a row is neighbour c
    of the reference's list order (x offset outer, y offset inner).  The valid slots plus a dummy (value 0, weight 0) after
    them are sorted stably per key (-0 equal to +0); only positions 0..num-1 are scanned, so the largest element drops out.
    half = half the weight sum in depth order; a key's median is the first position whose running sum reaches half.
    Returns (hit [4, P] slot of each median: 0..120, 121 for the dummy, -1 if never reached; num [P]; undecided [P];
    alt [P] the slot float32 sums could pick for the depth median instead, -2 where the depth median is decided)."""
    P = w.shape[0]
    rows = np.arange(P)
    num = valid.sum(axis=1)
    Wt = np.concatenate([np.where(valid, w, 0.0), np.zeros((P, 1))], axis=1)
    inpos = np.arange(N_SLOTS + 1)[None, :] < num[:, None]
    hit = np.full((4, P), -1, np.int64)
    undecided = np.zeros(P, bool)
    alt = np.full(P, -2, np.int64)
    half = wsum = None
    for q, key in enumerate(keys):
        k = np.concatenate([np.where(valid, np.asarray(key, np.float64) + 0.0, np.inf), np.zeros((P, 1))], axis=1)
        order = np.argsort(k, axis=1, kind="stable")
        S = np.cumsum(np.take_along_axis(Wt, order, axis=1), axis=1)
        if q == 0:
            wsum = np.where(num > 0, S[rows, np.maximum(num - 1, 0)], 0.0)
            half = wsum * 0.5
        reach = (S >= half[:, None]) & inpos
        first = np.argmax(reach, axis=1)
        hit[q] = np.where(reach.any(axis=1), order[rows, first], -1)
        # a running sum near half lets position j or j + 1 take the median.  For the depth the element itself matters
        # (its pixel gives the plane offset); for a normal component only its value does (ties of equal values are moot).
        near = (np.abs(S - half[:, None]) < TIE * wsum[:, None]) & inpos
        if q == 0:
            jn = np.argmax(near, axis=1)
            pos = np.where(jn < first, jn, first + 1)
            alt = np.where(near.any(axis=1), np.where(pos < num, order[rows, np.minimum(pos, N_SLOTS)], -1), -2)
            undecided |= alt == -1
            continue
        else:
            ks = np.take_along_axis(k, order, axis=1)
            ks = np.where(inpos, ks, 0.0)                  # past position num - 1: never reached, component 0
            v = np.where(hit[q] >= 0, ks[rows, first], 0.0)[:, None]
            near &= (ks != v) | (np.concatenate([ks[:, 1:], np.zeros((P, 1))], axis=1) != v)
        undecided |= near.any(axis=1)
    return hit, num, undecided, alt


def _lattice(xs, ys, W, H, radius, gap):
    """Lattice neighbours of pixels (xs, ys) in list order: offsets i (x, outer) and j (y, inner) of each slot."""
    steps = -radius + gap * np.arange(11)
    i = np.repeat(steps, 11)
    j = np.tile(steps, 11)
    nx, ny = xs[:, None] + i[None, :], ys[:, None] + j[None, :]
    inside = (nx >= 0) & (nx < W) & (ny >= 0) & (ny < H)
    return i, j, np.clip(nx, 0, W - 1), np.clip(ny, 0, H - 1), inside


def _offset(g, depth, n, nx, ny, dp, hd):
    """Plane offset from getD at the pixel of depth-median slot hd (the dummy: pixel (0, 0) and its disparity)."""
    rows = np.arange(len(hd))
    dummy = hd == N_SLOTS
    hs = np.clip(hd, 0, N_SLOTS - 1)
    mx = np.where(dummy, 0, nx[rows, hs]).astype(np.float64)
    my = np.where(dummy, 0, ny[rows, hs]).astype(np.float64)
    dmid = np.where(dummy, float(depth[0, 0]), dp[rows, hs])
    with np.errstate(divide="ignore", invalid="ignore"):
        return g.plane_d(n, mx, my, g.disparity(dmid))


def _median_plane(g, ref, plane, depth, scale, xs, ys, radius, gap, scale_div):
    """Gather + weighted medians + the median plane (normal normalised, offset from getD at the median's pixel).
    Returns (norm_mid [P, 4], mag_w, num, undecided, singular, alt_mid [P, 4] with the offset of the alternative depth
    median, has_alt [P])."""
    H, W = depth.shape
    i, j, nx, ny, inside = _lattice(xs, ys, W, H, radius, gap)
    valid = inside & (scale[ny, nx] == 1.0)
    spatial = np.sqrt((i * i + j * j).astype(np.float64)) / scale_div
    dref = np.abs(ref[ny, nx].astype(np.float64) - ref[ys, xs].astype(np.float64)[:, None])
    w = np.exp(-spatial / 4.0)[None, :] * np.exp(-dref / 9.0)
    pl = plane[ny, nx].astype(np.float64)
    dp = depth[ny, nx].astype(np.float64)
    hit, num, undecided, alt = weighted_medians(w, [dp, pl[..., 0], pl[..., 1], pl[..., 2]], valid)
    P = len(xs)
    rows = np.arange(P)
    comp = []
    for q in range(1, 4):
        h = hit[q]
        comp.append(np.where((h >= 0) & (h < N_SLOTS), pl[rows, np.clip(h, 0, N_SLOTS - 1), q - 1], 0.0))
    raw = np.stack(comp, axis=-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        n = raw / np.linalg.norm(raw, axis=-1, keepdims=True)
    reached = hit[0] >= 0
    d, mag_w = _offset(g, depth, n, nx, ny, dp, hit[0])
    d = np.where(reached, d, 0.0)
    n = np.where(reached[:, None], n, raw)
    d_alt, _ = _offset(g, depth, n, nx, ny, dp, np.maximum(alt, 0))
    singular = reached & np.isfinite(d) & (np.abs(d) <= SING * mag_w)
    return (np.concatenate([n, d[:, None]], axis=-1), mag_w, num, undecided, singular,
            np.concatenate([n, d_alt[:, None]], axis=-1), alt >= 0)


def wmf(g, ref, plane, depth, scale, it, xs, ys):
    """gipuma_WMF level `it` (0..3) at pixels (xs, ys): radius 80/2^it, gap 16/2^it, spatial divisor 2^(3-it); flag 0
    when the disparity of the weighted-median plane differs from the pixel's own by more than 24/2^it, or when no
    neighbour is reliable.  Every pixel reads the pre-launch state.  Returns (flag, undecided)."""
    po = 1 << it
    xs, ys = np.asarray(xs, np.int64), np.asarray(ys, np.int64)
    nm, _, num, undecided, singular, nm_alt, has_alt = _median_plane(g, ref, plane, depth, scale, xs, ys, 80 // po, 16 // po,
                                                                     float(1 << (3 - it)))
    fx, fy = xs.astype(np.float64), ys.astype(np.float64)
    dep_org, s2 = g.plane_depth(plane[ys, xs], fx, fy)
    ths = float(24 // po)

    def flag_of(pl):
        dep_now, s1 = g.plane_depth(pl, fx, fy)
        with np.errstate(invalid="ignore", divide="ignore"):
            dn, do = g.disparity(dep_now), g.disparity(dep_org)
            diff = np.abs(dn - do)
            near = np.abs(diff - ths) < TIE * np.maximum(ths, np.maximum(np.abs(dn), np.abs(do)))
        return np.where(diff > ths, 0.0, 1.0), s1 | near

    flag, und1 = flag_of(nm)
    flag_alt, und_alt = flag_of(nm_alt)
    has = num > 0
    flag = np.where(has, flag, 0.0)
    moot = ~has_alt | ((flag_alt == flag) & ~und_alt)      # the alternative depth median gives the same flag
    return flag, has & (undecided | singular | s2 | und1 | ~moot)


def wmf_final(g, ref, plane, depth, scale, canny, text, it, xs, ys):
    """gipuma_WMF_Final level `it` (0..5) at pixels (xs, ys): only unreliable pixels (scale 0) of textured regions
    (text == 1) with at least 32/2^it reliable neighbours (radius 5*2^it, gap 2^it, spatial divisor 2^it) are filled:
    plane = weighted-median plane, disparity of that plane clamped (outside (min, max) -> min_disp, scale 0; else scale 1).
    Returns (filled, plane [P, 4], mag_w, disp, scale, undecided)."""
    po = 1 << it
    xs, ys = np.asarray(xs, np.int64), np.asarray(ys, np.int64)
    reg = region_of(canny[ys, xs], len(text))
    cand = (reg >= 0) & (scale[ys, xs] == 0.0)
    cand[cand] = np.asarray(text, np.float32)[reg[cand]] == 1.0
    nm, mag_w, num, undecided, singular, nm_alt, has_alt = _median_plane(g, ref, plane, depth, scale, xs, ys, 5 * po, po,
                                                                         float(po))
    filled = cand & (num >= 32 // po)

    def fill_of(pl):
        dep, s1 = g.plane_depth(pl, xs.astype(np.float64), ys.astype(np.float64))
        with np.errstate(invalid="ignore", divide="ignore"):
            d = g.disparity(dep)
            out = (d <= g.min_disp) | (d >= g.max_disp)
            near = (np.abs(d - g.min_disp) < TIE * np.maximum(np.abs(d), g.min_disp)) | \
                   (np.abs(d - g.max_disp) < TIE * np.maximum(np.abs(d), g.max_disp))
        return np.where(out, g.min_disp, d), np.where(out, 0.0, 1.0), s1 | near

    d, sc, und1 = fill_of(nm)
    d_alt, sc_alt, und_alt = fill_of(nm_alt)
    with np.errstate(invalid="ignore"):
        same = (np.abs(nm_alt[:, 3] - nm[:, 3]) <= 0.1 * TIE * np.maximum(np.abs(nm[:, 3]), mag_w)) & \
               (np.abs(d_alt - d) <= 0.1 * TIE * np.abs(d)) & (sc_alt == sc) & ~und_alt
    moot = ~has_alt | same                                   # the alternative depth median gives the same fill
    return filled, nm, mag_w, d, sc, filled & (undecided | singular | und1 | ~moot)
