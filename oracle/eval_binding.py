"""ctypes binding of oracle/libeval_cpu.so (C restatement of the cloud evaluation rule) -- TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libeval_cpu.so")


def build():
    src = os.path.join(_HERE, "eval_cpu.c")
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-fopenmp", "-o", LIB, src, "-lm"])
    return LIB


def evaluate(recon, gt, thresholds, tau_max=None):
    """oc_eval (DESIGN.md section 4.7) on [n][3] / [m][3] float32 clouds.  tau_max defaults to the largest threshold.
    Returns (within_recon [k] int64, within_gt [k] int64, dist_recon [n] float32, dist_gt [m] float32)."""
    lib = C.CDLL(build())
    vp, ll = C.c_void_p, C.c_longlong
    lib.oc_eval.restype = None
    lib.oc_eval.argtypes = [vp, ll, vp, ll, vp, C.c_int, C.c_float, vp, vp, vp, vp]
    R = np.ascontiguousarray(np.asarray(recon, np.float32).reshape(-1, 3))
    G = np.ascontiguousarray(np.asarray(gt, np.float32).reshape(-1, 3))
    thr = np.ascontiguousarray(thresholds, np.float32).reshape(-1)
    tau = np.float32(thr.max() if tau_max is None else tau_max)
    wR, wG = np.zeros(len(thr), np.int64), np.zeros(len(thr), np.int64)
    dR, dG = np.empty(len(R), np.float32), np.empty(len(G), np.float32)
    lib.oc_eval(R.ctypes.data, len(R), G.ctypes.data, len(G), thr.ctypes.data, len(thr), float(tau),
                wR.ctypes.data, wG.ctypes.data, dR.ctypes.data, dG.ctypes.data)
    return wR, wG, dR, dG
