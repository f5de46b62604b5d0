"""rrt_b200 -- a B200-native (sm_100a) path-tracing core behind rogerallen/rrt's renderer seam.

The product is the CUDA library rrt_b200/librrtb200.so (C ABI: include/rrtb.h, sources rrt_b200/csrc) and
the drop-in `rrt` executable (rrt_b200/host).  This package is the thin ctypes binding over the C ABI
(the reference's "add pybind11" to-do, README.md:66) used by the tests and bench.py.
"""
from .api import Context, PinnedBuffer, Rrt, Scene, SceneError, camera_derive, render_group, tonemap, write_pfm, write_png  # noqa: F401
from ._lib import RrtbError, LIB_PATH  # noqa: F401
from .types import SceneArrays, RenderParams, Stats  # noqa: F401
