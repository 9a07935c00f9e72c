"""`.dmb` depth / normal maps as the reference writes them (fileIoUtils.h:333-381): int32 type (1 = float),
int32 height, int32 width, int32 channels, then h*w*channels float32 row-major.  Fusion.exe and the TSAR
scripts consume TSAR_disp.dmb (1 channel) and TSAR_normals.dmb (3 channels) (main.cpp:1807-1861)."""
import numpy as np

PLY_VERTEX = [("p", "<f4", 3), ("n", "<f4", 3), ("c", "u1", 3)]   # float x y z, float nx ny nz, uchar red green blue


def write_dmb(path, arr):
    a = np.ascontiguousarray(arr, np.float32)
    if a.ndim == 2:
        a = a[..., None]
    h, w, nb = a.shape
    with open(path, "wb") as f:
        np.array([1, h, w, nb], np.int32).tofile(f)
        a.tofile(f)


def read_dmb(path):
    with open(path, "rb") as f:
        t, h, w, nb = np.fromfile(f, np.int32, 4)
        if t != 1:
            raise ValueError(f"{path}: unsupported dmb type {t} (only float32 = 1 is written by the reference)")
        data = np.fromfile(f, np.float32, int(h) * int(w) * int(nb))
    if data.size != int(h) * int(w) * int(nb):
        raise ValueError(f"{path}: truncated dmb ({data.size} of {int(h) * int(w) * int(nb)} values)")
    a = data.reshape(int(h), int(w), int(nb))
    return a[..., 0] if nb == 1 else a


def write_outputs(folder, out_norm4):
    """TSAR_disp.dmb + TSAR_normals.dmb from the gipuma_compute_disp layout (xyz = world normal, w = depth)."""
    import os
    os.makedirs(folder, exist_ok=True)
    write_dmb(os.path.join(folder, "TSAR_disp.dmb"), out_norm4[..., 3])
    write_dmb(os.path.join(folder, "TSAR_normals.dmb"), out_norm4[..., :3])


def write_model_ply(path, depth, normals, gray, K, R, t):
    """TSAR_model.ply as storePlyFileBinary writes it (displayUtils.h:77-158, call site main.cpp:1836-1843): binary
    little-endian, one vertex per pixel -- float x y z (get3Dpoint with the UNtransformed camera P = K[R|t],
    cameraGeometryUtils.h:53-65: X = M^-1 (depth*(x,y,1) - p4)), float nx ny nz, uchar grey x3 -- pixels visited
    column by column (x outer, y inner; the reference's OpenMP loop writes them in a thread-dependent order, this is
    its sequential order).  Non-finite points become (0,0,0)."""
    depth = np.asarray(depth, np.float32)
    H, W = depth.shape
    P = (np.asarray(K, np.float64) @ np.concatenate([np.asarray(R, np.float64), np.asarray(t, np.float64).reshape(3, 1)], 1)).astype(np.float32)
    Minv = np.linalg.inv(P[:, :3].astype(np.float64)).astype(np.float32)
    xs, ys = np.meshgrid(np.arange(W, dtype=np.float32), np.arange(H, dtype=np.float32), indexing="ij")   # [x][y]
    d = depth.T
    rhs = np.stack([d * xs - P[0, 3], d * ys - P[1, 3], d - P[2, 3]], -1).astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        X = (rhs @ Minv.T).astype(np.float32)
    bad = ~np.isfinite(X).all(-1)
    X[bad] = 0.0
    rec = np.zeros(W * H, dtype=PLY_VERTEX)
    rec["p"] = X.reshape(-1, 3)
    rec["n"] = np.asarray(normals, np.float32).transpose(1, 0, 2).reshape(-1, 3)
    rec["c"] = np.asarray(gray).astype(np.uint8).T.reshape(-1, 1)
    _write_vertices(path, rec)


def write_fused_ply(path, xyz, normals, rgb):
    """The fused point cloud (fusion.fuse) in the vertex layout of TSAR_model.ply; read_model_ply reads it back."""
    rec = np.zeros(len(np.asarray(xyz).reshape(-1, 3)), dtype=PLY_VERTEX)
    rec["p"], rec["n"], rec["c"] = (np.asarray(a, dt).reshape(-1, 3) for a, dt in ((xyz, np.float32), (normals, np.float32), (rgb, np.uint8)))
    _write_vertices(path, rec)


def _write_vertices(path, rec):
    with open(path, "wb") as f:
        f.write(("ply\nformat binary_little_endian 1.0\n" + f"element vertex {len(rec)}\n" +
                 "property float x\nproperty float y\nproperty float z\nproperty float nx\nproperty float ny\nproperty float nz\n"
                 "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n").encode())
        rec.tofile(f)


def read_model_ply(path):
    """Reader for TSAR_model.ply and TSAR_fused.ply: returns (points [n][3], normals, colour)."""
    with open(path, "rb") as f:
        n = None
        while True:
            line = f.readline().decode().strip()
            if line.startswith("element vertex"):
                n = int(line.split()[-1])
            if line == "end_header":
                break
        rec = np.fromfile(f, dtype=PLY_VERTEX, count=n)
    return rec["p"], rec["n"], rec["c"]


PLY_SCALARS = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2", "ushort": "u2",
               "uint16": "u2", "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4", "float": "f4", "float32": "f4",
               "double": "f8", "float64": "f8"}


def read_ply_points(path):
    """xyz of the vertex element of a PLY file ([n][3] float32; double coordinates are rounded once).  Reads
    binary_little_endian and ascii files with any scalar property types and any extra properties (TSAR_fused.ply and
    typical ground-truth scans); elements before the vertex element are skipped when they have no list property.
    Anything else raises a one-line ValueError naming the file and the reason."""
    def fail(reason):
        return ValueError(f"{path}: {reason}")
    try:
        f = open(path, "rb")
    except OSError as e:
        raise fail(f"cannot open ({e.strerror})") from None
    with f:
        if f.readline().strip() != b"ply":
            raise fail("not a PLY file")
        fmt, elements = None, []                     # elements: [name, count, [(name, dtype or None for a list)]]
        while True:
            raw = f.readline()
            if not raw:
                raise fail("header has no end_header")
            tok = raw.decode("ascii", "replace").split()
            if not tok or tok[0] in ("comment", "obj_info"):
                continue
            if tok[0] == "end_header":
                break
            if tok[0] == "format" and len(tok) >= 2:
                fmt = tok[1]
            elif tok[0] == "element" and len(tok) == 3:
                elements.append([tok[1], int(tok[2]), []])
            elif tok[0] == "property" and elements and len(tok) >= 3:
                if tok[1] == "list":
                    elements[-1][2].append((tok[-1], None))
                elif tok[1] in PLY_SCALARS:
                    elements[-1][2].append((tok[2], PLY_SCALARS[tok[1]]))
                else:
                    raise fail(f"unknown property type {tok[1]}")
            else:
                raise fail(f"malformed header line {raw.strip()[:60]!r}")
        if fmt not in ("binary_little_endian", "ascii"):
            raise fail(f"unsupported format {fmt} (binary_little_endian or ascii only)")
        names = [e[0] for e in elements]
        if "vertex" not in names:
            raise fail("no vertex element")
        k = names.index("vertex")
        for e in elements[:k + 1]:
            if any(dt is None for _, dt in e[2]):
                raise fail(f"list property in element {e[0]} (cannot locate the vertices)")
        props = [p for p, _ in elements[k][2]]
        if not all(c in props for c in "xyz"):
            raise fail("vertex element has no x, y, z properties")
        n = elements[k][1]
        if fmt == "ascii":
            for e in elements[:k]:
                for _ in range(e[1]):
                    f.readline()
            lines = [f.readline() for _ in range(n)]
            try:
                rows = np.array([ln.split() for ln in lines], np.float64).reshape(n, len(props))
            except ValueError:
                raise fail(f"vertex data is not {n} rows of {len(props)} numbers") from None
            return np.stack([rows[:, props.index(c)] for c in "xyz"], -1).astype(np.float32)
        for e in elements[:k]:
            f.seek(e[1] * np.dtype([(p, "<" + dt) for p, dt in e[2]]).itemsize, 1)
        dt = np.dtype([(p, "<" + t) for p, t in elements[k][2]])
        rec = np.fromfile(f, dtype=dt, count=n)
        if len(rec) != n:
            raise fail(f"truncated vertex data ({len(rec)} of {n} vertices)")
        return np.stack([rec[c] for c in "xyz"], -1).astype(np.float32)
