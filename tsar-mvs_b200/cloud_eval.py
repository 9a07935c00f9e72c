"""Nearest-neighbour cloud-to-cloud evaluation (DESIGN.md section 4.7) on top of the tsar_eval_* entry points of
libtsar_b200.so: accuracy, completeness and F-score of a reconstruction against a ground-truth cloud.

For a threshold tau: accuracy = the fraction of reconstruction points whose nearest ground-truth point lies within tau,
completeness = the fraction of ground-truth points whose nearest reconstruction point lies within tau, F = their
harmonic mean.  Distances are float32, pinned to one operation order, and found by an exact tree search on the GPU.
This is not the ETH3D or Tanks and Temples evaluator (no cropping, alignment, masks or density handling): its numbers
cannot be compared with their leaderboards.
"""
import ctypes as C
import math

import numpy as np

from . import _lib as L
from .engine import TsarError

MAX_THRESHOLDS = 64   # TSAR_EVAL_MAX_THRESHOLDS
DEFAULT_THRESHOLDS = (0.01, 0.02, 0.05, 0.1, 0.2, 0.5)   # scene units


def fraction(count, total):
    """count / total; NaN over an empty cloud."""
    return count / total if total else math.nan


def fscore(accuracy, completeness):
    """Harmonic mean: NaN if either input is NaN, 0 if both are 0."""
    if math.isnan(accuracy) or math.isnan(completeness):
        return math.nan
    if accuracy + completeness == 0:
        return 0.0
    return 2.0 * accuracy * completeness / (accuracy + completeness)


def _cloud(a, name):
    a = np.ascontiguousarray(np.asarray(a, np.float32))
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError(f"{name} must be [n][3] xyz, got shape {a.shape}")
    return a


class EvalEngine:
    """One tsar_eval handle on one GPU; run() may be called again (its device scratch only grows)."""

    def __init__(self, device=0, stream=None):
        self.lib = L.load()
        h = C.c_void_p()
        rc = self.lib.tsar_eval_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise TsarError(f"tsar_eval_create(device={device}) failed with {rc}")
        self.h = h

    def run(self, recon, gt, thresholds=DEFAULT_THRESHOLDS, tau_max=None, distances=False):
        """Returns a dict: thresholds, tau_max, n_recon, n_gt, within_recon / within_gt (counts per threshold),
        accuracy / completeness / fscore (per threshold), and with distances=True dist_recon / dist_gt (float32 per
        point, input order, +inf beyond tau_max).  tau_max defaults to the largest threshold."""
        R, G = _cloud(recon, "recon"), _cloud(gt, "gt")
        thr = np.ascontiguousarray(thresholds, np.float32).reshape(-1)
        if len(thr) == 0:
            raise ValueError("no thresholds")
        tau = np.float32(thr.max() if tau_max is None else tau_max)
        wR, wG = np.zeros(len(thr), np.int64), np.zeros(len(thr), np.int64)
        dR = np.empty(len(R), np.float32) if distances else None
        dG = np.empty(len(G), np.float32) if distances else None
        rc = self.lib.tsar_eval_run(self.h, R.ctypes.data, len(R), G.ctypes.data, len(G), thr.ctypes.data, len(thr),
                                    float(tau), wR.ctypes.data, wG.ctypes.data,
                                    dR.ctypes.data if distances else None, dG.ctypes.data if distances else None)
        if rc != 0:
            raise TsarError(f"tsar_eval_run failed with {rc}: {self.lib.tsar_eval_last_error(self.h).decode()}")
        acc = [fraction(int(c), len(R)) for c in wR]
        comp = [fraction(int(c), len(G)) for c in wG]
        res = dict(thresholds=[float(t) for t in thr], tau_max=float(tau), n_recon=len(R), n_gt=len(G),
                   within_recon=[int(c) for c in wR], within_gt=[int(c) for c in wG], accuracy=acc, completeness=comp,
                   fscore=[fscore(a, c) for a, c in zip(acc, comp)])
        if distances:
            res["dist_recon"], res["dist_gt"] = dR, dG
        return res

    def visits(self):
        """Tree leaves visited in the last run per direction (recon -> gt, gt -> recon): (totals, per-query maxima)."""
        tot, mx = (C.c_longlong * 2)(), (C.c_int * 2)()
        rc = self.lib.tsar_eval_dbg_visits(self.h, tot, mx)
        if rc != 0:
            raise TsarError(f"tsar_eval_dbg_visits failed with {rc}")
        return list(tot), list(mx)

    def close(self):
        if getattr(self, "h", None):
            self.lib.tsar_eval_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def evaluate(recon, gt, thresholds=DEFAULT_THRESHOLDS, device=0, distances=False, tau_max=None):
    """Scores `recon` ([n][3]) against `gt` ([m][3]) at each threshold; see EvalEngine.run for the result."""
    with EvalEngine(device) as eng:
        return eng.run(recon, gt, thresholds, tau_max=tau_max, distances=distances)
