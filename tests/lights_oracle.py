"""ctypes wrapper of the CPU oracle WITH LIGHTS (tests/oracle_lights/lights.h): diffuse_light emitters and a constant
background over the unchanged oracle/rrt_oracle*.c, for the checks of tests/test_lights.py and tests/test_gpu_lights.py.

Test infrastructure only: nothing under rrt_b200/ imports this module.  The library is compiled on first use, with the
oracle's own compiler and flags (oracle/Makefile), into the temporary directory: the repository tree is never written.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle_lib import ORACLE_DIR, Counters, Oracle, _OrcBvh

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_lights")
SOURCES = [os.path.join(HERE, f) for f in ("lights_f32.c", "lights_f64.c")]
DEPS = SOURCES + [os.path.join(HERE, "lights.h")] + [os.path.join(ORACLE_DIR, f) for f in ("rrt_oracle.c", "rrt_oracle_f64.c", "rrt_oracle.h")]
DEPS.append(os.path.join(os.path.dirname(ORACLE_DIR), "include", "rrtb.h"))

_lib = None


def build_lights_oracle():
    h = hashlib.sha256()
    for p in DEPS:
        h.update(open(p, "rb").read())
    so = os.path.join(tempfile.gettempdir(), "rrtb_oracle_lights_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-fopenmp", "-o", tmp] + SOURCES + ["-lm"])
        os.replace(tmp, so)  # atomic: concurrent test processes see a whole library or none
    return so


def lights_lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build_lights_oracle())
        _lib.orc_bvh_build.restype = C.POINTER(_OrcBvh)
    return _lib


class LitOracle(Oracle):
    """The CPU oracle bound to one scene, emitters and the scene's background (SceneArrays.background) included.  The
    LBVH, trace and camera hooks are the oracle's own (the library holds the same code); render, render_f64, scatter
    and scatter_f64 add the emitted and background terms."""

    def __init__(self, scene):
        super().__init__(scene)
        self.lib = lights_lib()
        bg = getattr(scene, "background", None)
        self._bg = None if bg is None else np.ascontiguousarray(bg, dtype=np.float32).reshape(3)

    def _bgp(self):
        return None if self._bg is None else C.c_void_p(self._bg.ctypes.data)

    def render(self, W, H, spp, max_depth=50, seed=1984, use_bvh=True, rank=0, world=1, shard_mode=0):
        out = np.zeros((H, W, 3), np.float32)
        fixed = np.zeros((H, W, 3), np.uint64)
        cnt = Counters()
        self.lib.orc_l_render(C.byref(self._s), self._bgp(), self.bvh() if use_bvh else None, W, H, spp, max_depth,
                              C.c_uint64(seed), rank, world, shard_mode, C.c_void_p(out.ctypes.data),
                              C.c_void_p(fixed.ctypes.data), C.byref(cnt))
        return out, fixed, cnt.as_dict()

    def render_f64(self, W, H, spp, max_depth=50, seed=1984, use_bvh=True):
        out = np.zeros((H, W, 3), np.float64)
        fixed = np.zeros((H, W, 3), np.uint64)
        cnt = Counters()
        self.lib.orc_l_d_render(C.byref(self._s), self._bgp(), self.bvh() if use_bvh else None, W, H, spp, max_depth,
                                C.c_uint64(seed), C.c_void_p(out.ctypes.data), C.c_void_p(fixed.ctypes.data), C.byref(cnt))
        return out, fixed, cnt.as_dict()

    def scatter(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float32)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32)
        out = np.zeros((len(in16), 8), np.float32)
        self.lib.orc_l_scatter(C.byref(self._s), C.c_void_p(in16.ctypes.data), C.c_void_p(rnd4.ctypes.data), len(in16),
                               C.c_void_p(out.ctypes.data))
        return out

    def scatter_f64(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float64)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32)
        out = np.zeros((len(in16), 8), np.float64)
        self.lib.orc_l_d_scatter(C.byref(self._s), C.c_void_p(in16.ctypes.data), C.c_void_p(rnd4.ctypes.data), len(in16),
                                 C.c_void_p(out.ctypes.data))
        return out
