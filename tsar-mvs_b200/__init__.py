"""tsar-mvs_b200: B200-native (sm_100a) implementation of TSAR-MVS's per-reference-view depthmap path.

The product is libtsar_b200.so (hand-written CUDA behind the C ABI of include/tsar_b200.h); this
package is the thin host-side mirror of the reference's entry points plus the synthetic-scene and
file-format helpers the tests and the benchmark use.  The directory name carries a hyphen (as the
task names it); import it through `__graft_entry__.load_package()` or importlib.
"""
from . import _lib  # noqa: F401
from .engine import DepthmapEngine, TsarError, make_params  # noqa: F401
from . import scene  # noqa: F401
from . import dmb, shard, cli, texture, counts, fusion, cloud_eval, mesh  # noqa: F401

__all__ = ["DepthmapEngine", "TsarError", "make_params", "scene", "dmb", "shard", "fusion", "cloud_eval", "mesh"]
