"""Recorded outputs of the reference build -- TEST INFRASTRUCTURE ONLY.

The parity tests compare the library with the reference's own code: its kernels (oracle/ref_binding.py) and its host
functions (oracle/ref_host_binding.py), both built into oracle/_ref/ by `make oracle` where a checkout of the reference
exists.  Where that build is absent, this module takes their place with the same names.  Each result is computed by the
library (or, for the region fit, by the C restatement oracle/oracle_cpu.c) and checked against the SHA-256 digest of the
result the reference build gave at the same call of the same test, stored in tests/golden/reference_digests.json.  A
result that differs raises, so every comparison of the tests keeps its bar: bit for bit.  The stored digests were
taken from the library at a commit where each of these results was bit-identical to the reference build's
(tests/golden/MANIFEST.json).

The reference as written races on same-colour pixels (variant 'asis'), so its results after a propagation step differ
from run to run.  The recording holds the race-free twin's results in their place: in this mode the tests' comparisons
with the as-written build (ours as far from it as the twin is, thresholds on the agreement) are dropped, and only the
bit-exact comparisons remain.

Recording needs the reference build: with TSAR_RECORD_REFERENCE_DIGESTS=<json path>, tests/parity_common.py hands the
tests recording() / recording_host(), which wrap oracle/ref_binding.py / oracle/ref_host_binding.py and store the digest
of every result those return, so a new or changed test cannot record the library's own output as the reference's.
Digests are keyed by test id and call order: a renamed or reparametrised test, or a sweep script run with other
arguments or another TSAR_SWEEP_SEED, finds no recording and fails until it is recorded from the reference build.
"""
import hashlib
import json
import os
import sys
import types

import numpy as np

from oracle.ref_binding import (F_BEVIEW, F_CANNY, F_CONFID, F_COST, F_DEPTH, F_FAKEDEPTH, F_LRDIFF, F_NORM4,  # noqa: F401
                                F_RATIO, F_REGION_NORM4, F_REGION_TEXT, F_SCALE)

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIGESTS = os.path.join(_ROOT, "tests", "golden", "reference_digests.json")
_RECORD = os.environ.get("TSAR_RECORD_REFERENCE_DIGESTS")
_table = None
_calls = {}


def available(variant="asis"):
    return os.path.exists(DIGESTS)


def _pkg():
    if _ROOT not in sys.path:
        sys.path.insert(0, _ROOT)
    import __graft_entry__ as g
    return g.load_package()


def _key():
    """The test that asks (pytest's node id) and, for a script the test runs, the script and its arguments."""
    node = os.environ.get("PYTEST_CURRENT_TEST", "").rsplit(" (", 1)[0]
    node = os.path.basename(node.split("::", 1)[0]) + node[len(node.split("::", 1)[0]):]   # independent of pytest's rootdir
    if "pytest" in sys.modules:
        return node
    return node + "|" + " ".join([os.path.basename(sys.argv[0])] + sys.argv[1:])


def digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:24]


def _record(*arrays):
    key = _key()
    for a in arrays:
        i = _calls.get(key, 0)
        _calls[key] = i + 1
        table = json.load(open(_RECORD)) if os.path.exists(_RECORD) else {}
        table[key] = table.get(key, [])[:i] + [digest(a)]
        with open(_RECORD, "w") as f:
            json.dump(table, f, indent=0, sort_keys=True)
    return arrays if len(arrays) > 1 else arrays[0]


def _check(*arrays):
    global _table
    key = _key()
    for a in arrays:
        i = _calls.get(key, 0)
        _calls[key] = i + 1
        d = digest(a)
        if _table is None:
            _table = json.load(open(DIGESTS))
        want = _table.get(key, [])
        assert i < len(want), f"no recorded reference result #{i} for {key!r} in {DIGESTS}"
        assert want[i] == d, f"result #{i} of {key!r} ({a.dtype} {a.shape}) differs from the reference build's recorded result"
    return arrays if len(arrays) > 1 else arrays[0]


class RefEngine:
    """ref_binding.RefEngine's methods on a library context; every result handed out is checked against the recording."""

    def __init__(self, camera_struct_type, params_struct_type, variant="asis"):
        self.variant = variant
        self.eng = _pkg().DepthmapEngine(0)
        self.n_regions = 0

    def create(self, images, cams_struct, subset, params, cam_f):
        self.eng.set_views(images, cams_struct, subset, cam_f=cam_f)
        self.eng.set_params(params)
        self.params = params

    def close(self):
        self.eng.close()

    def set_regions(self, text, norm4):
        self.n_regions = len(text)
        self.eng.set_regions(text, norm4)

    def depthmap(self, seed0, iters=None, prefetch=False):
        if iters is not None and iters != self.params.iterations:
            self.params = type(self.params).from_buffer_copy(self.params)
            self.params.iterations = int(iters)
            self.eng.set_params(self.params)
        return self.eng.depthmap(seed0)

    def eval_planes(self, xy, planes):
        return _check(*self.eng.eval_planes(xy, planes, wrapper_rounding=True))

    def download(self, field):
        return _check(self.eng.download(field, self.n_regions))

    def __getattr__(self, name):   # init_planes, launch, iterate, upload and the per-pixel stages
        return getattr(self.eng, name)


_slic_eng = None


def ref_slic(bgrx, spixel_size=20, no_iters=5, coh_weight=5.0, enforce_connectivity=False):
    global _slic_eng
    if _slic_eng is None:
        _slic_eng = _pkg().DepthmapEngine(0)
    labels = _slic_eng.slic(bgrx, spixel_size=spixel_size, no_iters=no_iters, coh_weight=coh_weight,
                            enforce_connectivity=enforce_connectivity)
    return _check(labels), 0.0


def slic_last_lab(n):
    """CIELab image [n][4] of the last ref_slic call."""
    import ctypes as C
    out = np.empty((n, 4), np.float32)
    _slic_eng.lib.tsar_dbg_slic_lab.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    _slic_eng._ck(_slic_eng.lib.tsar_dbg_slic_lab(_slic_eng.h, out.ctypes.data, n), "lab")
    return _check(out)


def slic_last_centres(nsp):
    """Superpixel records [nsp][8] (centre, colour, count) of the last ref_slic call."""
    import ctypes as C
    out = np.zeros((nsp, 8), np.float32)
    cnt = C.c_int(0)
    _slic_eng._ck(_slic_eng.lib.tsar_dbg_slic_centres(_slic_eng.h, out.ctypes.data_as(C.c_void_p), nsp, C.byref(cnt)), "centres")
    return _check(out)


class host:
    """ref_host_binding's functions (the reference's host code: roberts, Connect, texture, the per-region RANSAC)."""

    @staticmethod
    def available():
        return os.path.exists(DIGESTS)

    @staticmethod
    def roberts(gray):
        g = np.asarray(gray, np.int64)
        mag = np.full(g.shape, 100 * 50 * 2, np.int64)
        t1 = (g[1:-1, 1:-1] - g[2:, 2:]) ** 2
        t2 = (g[2:, 1:-1] - g[1:-1, 2:]) ** 2
        mag[1:-1, 1:-1] = t1 + t2
        return _check((np.sqrt(mag.astype(np.float64)).astype(np.int64) & 0xFF).astype(np.uint8))

    @staticmethod
    def connect(edges):
        from tsar_mvs_b200 import texture as tx
        _pkg()
        lab, cnt = tx.connect(edges)
        weak = np.array([k for k in range(1, len(cnt)) if cnt[k] > 5000], np.int32)
        return _check(np.asarray(lab, np.int32), np.asarray(cnt, np.int32), weak)

    @staticmethod
    def texture(gray_full):
        from tsar_mvs_b200 import texture as tx
        _pkg()
        h, w = gray_full.shape
        det = tx.detect(np.ascontiguousarray(gray_full, np.uint8))
        out = dict(canny=tx.expand_labels(det["labels_q"], w, h).astype(np.float32), text=np.asarray(det["text"], np.float32),
                   cenxi=np.asarray(det["cenxi"], np.int32), cenyi=np.asarray(det["cenyi"], np.int32),
                   size=np.asarray(det["size"], np.float32))
        _check(*out.values())
        return out

    @staticmethod
    def fit_regions(cam0, cam_f, depth, scale, canny, text, size, rnd_stream, planes0, cenxi=None, cenyi=None):
        from oracle import cpu_binding as cb
        pkg = _pkg()
        from tsar_mvs_b200.engine import cameras_to_struct
        per = 46000                     # rand() values the reference draws per fitted region: 3 x 10 000 + 4 x 4 x 1000
        stream = np.ascontiguousarray(rnd_stream, np.uint32).ravel()
        planes = np.ascontiguousarray(planes0, np.float32).reshape(len(text), 4).copy()
        cam = cameras_to_struct([cam0])[0]
        used = 0
        for r in range(len(text)):
            if text[r] == -1:
                planes[r], _ = cb.fit_region_plane(pkg._lib.TsarCamera, cam, cam_f, depth, scale, canny, r, size[r],
                                                   stream[used:used + per], planes[r])
                used += per
        return _check(planes), used


# ---- recording from the reference build ----------------------------------------------------------------------------
class _RecordingRefEngine:
    """ref_binding.RefEngine recording every result it hands out; the as-written variant is served by the race-free twin."""

    def __init__(self, camera_struct_type, params_struct_type, variant="asis"):
        from oracle import ref_binding as rb
        self.ref = rb.RefEngine(camera_struct_type, params_struct_type, "snapshot" if variant == "asis" else variant)

    def eval_planes(self, xy, planes):
        return _record(*self.ref.eval_planes(xy, planes))

    def download(self, field):
        return _record(self.ref.download(field))

    def __getattr__(self, name):
        return getattr(self.ref, name)


def recording():
    """oracle/ref_binding.py with every result recorded to $TSAR_RECORD_REFERENCE_DIGESTS."""
    from oracle import ref_binding as rb
    ns = types.SimpleNamespace(**{k: getattr(rb, k) for k in dir(rb) if k.startswith("F_")})
    ns.available, ns.RefEngine = rb.available, _RecordingRefEngine

    def ref_slic(*args, **kw):
        labels, ms = rb.ref_slic(*args, **kw)
        return _record(labels), ms
    ns.ref_slic = ref_slic
    ns.slic_last_lab = lambda n: _record(rb.slic_last_lab(n))
    ns.slic_last_centres = lambda nsp: _record(rb.slic_last_centres(nsp))
    return ns


def recording_host():
    """oracle/ref_host_binding.py with every result recorded to $TSAR_RECORD_REFERENCE_DIGESTS."""
    from oracle import ref_host_binding as rh

    def texture(gray_full):
        out = rh.texture(gray_full)
        _record(*out.values())
        return out

    def fit_regions(*args, **kw):
        planes, used = rh.fit_regions(*args, **kw)
        return _record(planes), used
    return types.SimpleNamespace(available=rh.available, roberts=lambda gray: _record(rh.roberts(gray)),
                                 connect=lambda edges: _record(*rh.connect(edges)), texture=texture, fit_regions=fit_regions)
