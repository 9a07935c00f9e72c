"""Who owns the library's CUDA memory (csrc/dev_mem.h), observed from outside (pytest -m gpu, on a B200).

libtsar_b200.so links libcudart.so.12 dynamically, so an LD_PRELOAD interposer sees every cudaMalloc / cudaFree,
cudaMallocArray / cudaFreeArray and cudaMallocHost / cudaFreeHost it makes.  Each scenario runs in a subprocess that
imports the package (not torch, whose own allocations would be counted too) with the interposer preloaded:
  * steady state: a handle driven again at sizes it has seen allocates and frees nothing (DESIGN.md 4.4: an allocation
    or a free synchronises the whole device and serialised the two pipelined contexts of the file driver);
  * no leaks: small -> large -> small, then destroy, frees every allocation of each kind;
  * a failed allocation returns TSAR_ERR_NOMEM and leaves no pending error behind for the next call on the handle.
"""
import os
import subprocess
import sys
import textwrap

import pytest

from tests import parity_common as pc

pytestmark = pytest.mark.gpu

INTERPOSER = r"""
#define _GNU_SOURCE
#include <dlfcn.h>
#include <stddef.h>

typedef int err_t;
enum { MALLOC, FREE, MALLOC_ARRAY, FREE_ARRAY, MALLOC_HOST, FREE_HOST, N_KINDS };
static long long calls[N_KINDS];
static unsigned long long bytes[N_KINDS];
static size_t armed;   /* the next cudaMalloc of exactly this many bytes asks for 2^62 instead */

/* ctypes loads the library RTLD_LOCAL, where dlsym(RTLD_NEXT) finds nothing: look the symbol up in the runtime itself */
static void *real(const char *name) {
    void *h = dlopen("libcudart.so.12", RTLD_NOLOAD | RTLD_LAZY);
    void *f = h ? dlsym(h, name) : NULL;
    return f ? f : dlsym(RTLD_NEXT, name);
}

#define REAL(fn) static __typeof__(&fn) f; if (!f) f = (__typeof__(&fn))real(#fn)

err_t cudaMalloc(void **p, size_t n) {
    REAL(cudaMalloc);
    calls[MALLOC]++; bytes[MALLOC] += n;
    if (armed && n == armed) { armed = 0; n = (size_t)1 << 62; }
    return f(p, n);
}
err_t cudaFree(void *p) { REAL(cudaFree); calls[FREE]++; return f(p); }
err_t cudaMallocArray(void **a, const void *desc, size_t w, size_t h, unsigned flags) {
    REAL(cudaMallocArray);
    calls[MALLOC_ARRAY]++; bytes[MALLOC_ARRAY] += w * h;
    return f(a, desc, w, h, flags);
}
err_t cudaFreeArray(void *a) { REAL(cudaFreeArray); calls[FREE_ARRAY]++; return f(a); }
err_t cudaMallocHost(void **p, size_t n) {
    REAL(cudaMallocHost);
    calls[MALLOC_HOST]++; bytes[MALLOC_HOST] += n;
    return f(p, n);
}
err_t cudaFreeHost(void *p) { REAL(cudaFreeHost); calls[FREE_HOST]++; return f(p); }

void count_arm(size_t n) { armed = n; }
long long count_calls(int kind) { return calls[kind]; }
unsigned long long count_bytes(int kind) { return bytes[kind]; }
"""

PRELUDE = r"""
import ctypes as C
import sys
import numpy as np
sys.path.insert(0, ROOT)
import __graft_entry__ as g
pkg = g.load_package()
L = pkg._lib
lib = L.load()
assert "torch" not in sys.modules
I = C.CDLL(INTERPOSER)
I.count_arm.argtypes = [C.c_size_t]
I.count_calls.restype = C.c_longlong
I.count_bytes.restype = C.c_ulonglong
KINDS = ("cudaMalloc", "cudaFree", "cudaMallocArray", "cudaFreeArray", "cudaMallocHost", "cudaFreeHost")
NOMEM = -4


def counts():
    return {k: (I.count_calls(i), I.count_bytes(i)) for i, k in enumerate(KINDS)}


def calls_since(before):
    now = counts()
    return {k: now[k][0] - before[k][0] for k in KINDS if now[k][0] != before[k][0]}


def depthmap_pass(eng, s, seed=20240601):
    eng.set_views(s["images"], s["cams"], s["subset"], cam_f=s["cam_f"])
    eng.set_params(pkg.make_params(iterations=2, min_disparity=s["min_disparity"], max_disparity=s["max_disparity"]))
    ref = s["images"][0].astype(np.uint8)
    eng.slic(np.ascontiguousarray(np.stack([ref, ref, ref, ref], axis=-1)))
    eng.depthmap(seed)
    eng.scale_from_confidence(0.5)
    eng.upload(L.F_CANNY, s["canny"])
    text, planes = s["region_text"], s["region_norm4"]
    size = (np.bincount(s["labels"].ravel(), minlength=len(text)) / 16.0).astype(np.float32)
    rnd = np.random.RandomState(7).randint(0, 2 ** 31 - 1, (len(text), lib.tsar_ransac_rand_per_region())).astype(np.uint32)
    eng.fit_region_planes(text, size, rnd, planes)
    eng.fit_region_planes(text, size, None, planes, seed=seed)
    eng.set_regions(text, planes)
    eng.wmf(0)
    eng.wmf_final(0)
    eng.download_outputs()


def tex_formats(eng, image=0, n=64, xy=True):
    pts = (np.random.RandomState(3).rand(n, 2) * [eng.W, eng.H]).astype(np.float32)
    out, rate = np.empty(4 * max(n, 1), np.float32), np.empty(4, np.float32)
    return lib.tsar_dbg_tex_formats(eng.h, image, n, pts.ctypes.data if xy else None, out.ctypes.data, rate.ctypes.data)


def fusion_views(W, H, n_views, seed=5):
    rng = np.random.RandomState(seed)
    K = np.array([[200.0, 0, W / 2], [0, 200.0, H / 2], [0, 0, 1]], np.float32)
    views = []
    for v in range(n_views):
        normals = np.zeros((H, W, 3), np.float32)
        normals[..., 2] = -1.0
        views.append(dict(K=K, R=np.eye(3, dtype=np.float32), t=np.array([0.02 * v, 0, 0], np.float32),
                          depth=(2.0 + 0.001 * rng.rand(H, W)).astype(np.float32), normals=normals,
                          bgr=rng.randint(0, 256, (H, W, 3)).astype(np.uint8)))
    return views


def fusion_engine(views, n_neighbours):
    H, W = views[0]["depth"].shape
    eng = pkg.fusion.FusionEngine(len(views), W, H)
    for v, d in enumerate(views):
        nb = [u for u in range(len(views)) if u != v][:n_neighbours]
        eng.set_view(v, d["K"], d["R"], d["t"], d["depth"], d["normals"], d["bgr"], nb)
    return eng


def cloud(n, seed):
    return np.random.RandomState(seed).rand(n, 3).astype(np.float32)
"""


@pytest.fixture(scope="module")
def interposer(tmp_path_factory):
    d = tmp_path_factory.mktemp("count_alloc")
    so = str(d / "libcount_alloc.so")
    subprocess.run(["gcc", "-x", "c", "-shared", "-fPIC", "-O2", "-", "-o", so, "-ldl"], input=INTERPOSER.encode(),
                   check=True)
    return so


def run_scenario(interposer, body):
    """Runs PRELUDE + body in a fresh interpreter with the interposer preloaded; the body asserts what it checks."""
    code = f"ROOT = {pc.ROOT!r}\nINTERPOSER = {interposer!r}\n" + PRELUDE + textwrap.dedent(body)
    env = dict(os.environ, LD_PRELOAD=interposer)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=pc.ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return r.stdout


def test_no_allocation_in_steady_state(interposer):
    out = run_scenario(interposer, """
        s = pkg.scene.make_scene("small")
        eng = pkg.DepthmapEngine(0)
        depthmap_pass(eng, s)
        before = counts()
        depthmap_pass(eng, s)
        assert calls_since(before) == {}, ("DepthmapEngine", calls_since(before))

        views = fusion_views(160, 120, 4)
        fe = fusion_engine(views, 3)
        fe.run()
        before = counts()
        fe.run()
        assert calls_since(before) == {}, ("FusionEngine", calls_since(before))

        ee = pkg.cloud_eval.EvalEngine(0)
        ee.run(cloud(50000, 1), cloud(40000, 2), distances=True)
        before = counts()
        ee.run(cloud(50000, 3), cloud(40000, 4), distances=True)
        assert calls_since(before) == {}, ("EvalEngine", calls_since(before))
        print("ok")
    """)
    assert "ok" in out


def test_every_allocation_is_freed(interposer):
    run_scenario(interposer, """
        def balanced(what, before):
            d = calls_since(before)
            for a, f in (("cudaMalloc", "cudaFree"), ("cudaMallocArray", "cudaFreeArray"), ("cudaMallocHost", "cudaFreeHost")):
                assert d.get(a, 0) == d.get(f, 0), (what, d)
            assert d.get("cudaMalloc", 0) > 0, (what, d)

        tiny, small = pkg.scene.make_scene("tiny"), pkg.scene.make_scene("small")
        before = counts()
        eng = pkg.DepthmapEngine(0)
        for s in (tiny, small, tiny):
            depthmap_pass(eng, s)
            assert tex_formats(eng) == 0
        eng.close()
        balanced("DepthmapEngine", before)

        views = fusion_views(96, 64, 5)
        before = counts()
        fe = fusion_engine(views, 1)
        fe.run()
        for v, d in enumerate(views):   # more neighbours: the scratch grows
            fe.set_view(v, d["K"], d["R"], d["t"], d["depth"], d["normals"], d["bgr"], [u for u in range(5) if u != v])
        fe.run()
        fe.close()
        balanced("FusionEngine", before)

        before = counts()
        ee = pkg.cloud_eval.EvalEngine(0)
        for n in (1000, 200000, 1000):
            ee.run(cloud(n, n), cloud(n // 2 + 1, n + 1))
        ee.close()
        balanced("EvalEngine", before)
    """)


def test_failed_allocation_does_not_poison_the_next_call(interposer):
    """A scratch growth refused by the runtime returns TSAR_ERR_NOMEM; the runtime's last error is cleared, so the next
    call on the same handle (which allocates a smaller buffer) succeeds and computes what a fresh handle computes."""
    run_scenario(interposer, """
        s = pkg.scene.make_scene("small")
        W, H = s["W"], s["H"]

        def prepared():
            eng = pkg.DepthmapEngine(0)
            eng.set_views(s["images"], s["cams"], s["subset"], cam_f=s["cam_f"])
            eng.set_params(pkg.make_params(iterations=2, min_disparity=s["min_disparity"], max_disparity=s["max_disparity"]))
            eng.depthmap(20240601)
            eng.scale_from_confidence(0.5)
            eng.upload(L.F_CANNY, s["canny"])
            eng.set_regions(s["region_text"], s["region_norm4"])
            return eng

        eng = prepared()
        I.count_arm(W * H * 24)   # the tsar_wmf_final scratch
        assert lib.tsar_wmf_final(eng.h, 0) == NOMEM
        assert b"out of memory" in lib.tsar_last_error(eng.h), lib.tsar_last_error(eng.h)
        eng.wmf(0)
        fresh = prepared()
        fresh.wmf(0)
        assert np.array_equal(eng.download(L.F_SCALE), fresh.download(L.F_SCALE))
        eng.close(); fresh.close()

        views = fusion_views(96, 64, 4)
        fe = fusion_engine(views, 3)
        I.count_arm(3 * 96 * 64 * 4)   # the candidate scratch of tsar_fusion_run
        p = pkg.fusion.make_params()
        n = C.c_longlong()
        assert lib.tsar_fusion_run(fe.h, C.byref(p), C.byref(n)) == NOMEM
        got = fe.run()
        ref = fusion_engine(views, 3)
        want = ref.run()
        assert len(got[0]) > 0 and all(np.array_equal(a, b) for a, b in zip(got, want))
        fe.close(); ref.close()
    """)


def test_tex_formats_rejects_bad_arguments(interposer):
    run_scenario(interposer, """
        s = pkg.scene.make_scene("tiny")
        eng = pkg.DepthmapEngine(0)
        eng.set_views(s["images"], s["cams"], s["subset"], cam_f=s["cam_f"])
        eng.set_params(pkg.make_params())
        assert tex_formats(eng, image=len(s["images"])) == -1
        assert tex_formats(eng, image=-1) == -1
        assert tex_formats(eng, n=0) == -1
        assert tex_formats(eng, xy=False) == -1
        assert tex_formats(eng) == 0
        eng.close()
    """)
