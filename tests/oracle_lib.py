"""ctypes wrappers for the CHECKERS: oracle/liboracle.so (our C restatement) and
oracle/_ref/libref_{f,d}.so (the unmodified reference behind oracle/ref_harness.cpp).

Test infrastructure only: nothing under rrt_b200/ imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from rrt_b200.types import (
    SceneArrays,
    camera_dtype,
    material_dtype,
    msphere_dtype,
    sphere_dtype,
    triangle_dtype,
)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
GOLDEN_SCENES = os.path.join(ROOT, "tests", "golden", "scenes")


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


# ------------------------------------------------------------------------------------------------
# oracle/liboracle.so
# ------------------------------------------------------------------------------------------------
class _OrcScene(C.Structure):
    _fields_ = [
        ("cam", C.c_float * 24),
        ("materials", C.c_void_p), ("n_materials", C.c_int),
        ("spheres", C.c_void_p), ("n_spheres", C.c_int),
        ("mspheres", C.c_void_p), ("n_mspheres", C.c_int),
        ("triangles", C.c_void_p), ("n_triangles", C.c_int),
        ("mtriangles", C.c_void_p), ("n_mtriangles", C.c_int),
    ]


class _OrcBvh(C.Structure):
    _fields_ = [
        ("n", C.c_int),
        ("morton", C.POINTER(C.c_uint32)),
        ("perm", C.POINTER(C.c_uint32)),
        ("left", C.POINTER(C.c_int32)),
        ("right", C.POINTER(C.c_int32)),
        ("parent", C.POINTER(C.c_int32)),
        ("node_box", C.POINTER(C.c_float)),
        ("prim_box", C.POINTER(C.c_float)),
        ("pad", C.c_float),
    ]


class Counters(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("rays", "box_tests", "sphere_tests", "msphere_tests", "triangle_tests", "hits", "paths")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def build_oracle():
    if os.environ.get("RRTB_ORACLE_LIB"):  # e.g. oracle/liboracle_ubsan.so (`make -C oracle ubsan`): the checker under UBSan
        return os.environ["RRTB_ORACLE_LIB"]
    so = os.path.join(ORACLE_DIR, "liboracle.so")
    src = [os.path.join(ORACLE_DIR, f) for f in ("rrt_oracle.c", "rrt_oracle_f64.c", "rrt_oracle.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
    return so


_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        _oracle = C.CDLL(build_oracle())
        _oracle.orc_bvh_build.restype = C.POINTER(_OrcBvh)
        _oracle.orc_u01.restype = C.c_float
        _oracle.orc_u01.argtypes = [C.c_uint32]
    return _oracle


class Oracle:
    """The CPU oracle bound to one scene."""

    def __init__(self, scene: SceneArrays):
        self.lib = oracle_lib()
        self.scene = scene
        s = _OrcScene()
        C.memmove(s.cam, scene.camera.ctypes.data, 96)
        s.materials, s.n_materials = scene.materials.ctypes.data, len(scene.materials)
        s.spheres, s.n_spheres = scene.spheres.ctypes.data, len(scene.spheres)
        s.mspheres, s.n_mspheres = scene.mspheres.ctypes.data, len(scene.mspheres)
        s.triangles, s.n_triangles = scene.triangles.ctypes.data, len(scene.triangles)
        s.mtriangles, s.n_mtriangles = scene.mtriangles.ctypes.data, len(scene.mtriangles)
        self._s = s
        self._bvh = None

    def __del__(self):
        if getattr(self, "_bvh", None):
            self.lib.orc_bvh_free(self._bvh)

    # -- LBVH --
    def bvh(self):
        if self._bvh is None:
            self._bvh = self.lib.orc_bvh_build(C.byref(self._s))
        return self._bvh

    def bvh_arrays(self):
        b = self.bvh().contents
        n = b.n
        ni = max(n - 1, 0)
        g = lambda ptr, cnt, dt: np.ctypeslib.as_array(ptr, shape=(max(cnt, 1),))[:cnt].astype(dt, copy=True)
        return dict(
            morton=g(b.morton, n, np.uint32),
            perm=g(b.perm, n, np.uint32),
            left=g(b.left, ni, np.int32),
            right=g(b.right, ni, np.int32),
            parent=g(b.parent, 2 * n - 1, np.int32),
            node_box=g(b.node_box, 6 * ni, np.float32).reshape(-1, 6),
            prim_box=g(b.prim_box, 6 * n, np.float32).reshape(-1, 6),
            pad=float(b.pad),
        )

    # -- rays --
    def camera_rays(self, W, H, pixels, sample, seed):
        pixels = np.asarray(pixels, dtype=np.int32)
        out = np.zeros((len(pixels), 7), np.float32)
        cam = self.scene.camera
        f = self.lib.orc_camera_ray
        for k, p in enumerate(pixels):
            f(C.c_void_p(cam.ctypes.data), W, H, int(p), int(sample), C.c_uint64(seed), C.c_void_p(out[k].ctypes.data))
        return out

    def trace(self, rays7, t_min=0.001, mode="scan", want_rec=False, counters=False):
        rays7 = np.ascontiguousarray(rays7, dtype=np.float32)
        n = len(rays7)
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        rec = np.zeros((n, 7), np.float32) if want_rec else None
        recp = C.c_void_p(rec.ctypes.data) if want_rec else None
        cnt = Counters()
        if mode == "scan":
            self.lib.orc_trace_scan(C.byref(self._s), C.c_void_p(rays7.ctypes.data), n, C.c_float(t_min),
                                    C.c_void_p(ids.ctypes.data), C.c_void_p(t.ctypes.data), recp)
        else:
            self.lib.orc_trace_bvh(C.byref(self._s), self.bvh(), C.c_void_p(rays7.ctypes.data), n, C.c_float(t_min),
                                   C.c_void_p(ids.ctypes.data), C.c_void_p(t.ctypes.data), recp, C.byref(cnt))
        res = [ids, t]
        if want_rec:
            res.append(rec)
        if counters:
            res.append(cnt.as_dict())
        return tuple(res)

    def hit_object(self, obj, ray7, t_min=0.001, t_max=np.inf):
        ray7 = np.ascontiguousarray(ray7, dtype=np.float32)
        t = C.c_float()
        rec = np.zeros(7, np.float32)
        ok = self.lib.orc_hit_object(C.byref(self._s), int(obj), C.c_void_p(ray7.ctypes.data), C.c_float(t_min),
                                     C.c_float(t_max), C.byref(t), C.c_void_p(rec.ctypes.data))
        return bool(ok), t.value, rec

    def scatter(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float32)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32)
        out = np.zeros((len(in16), 8), np.float32)
        self.lib.orc_scatter(C.byref(self._s), C.c_void_p(in16.ctypes.data), C.c_void_p(rnd4.ctypes.data), len(in16),
                             C.c_void_p(out.ctypes.data))
        return out

    def render(self, W, H, spp, max_depth=50, seed=1984, use_bvh=True, rank=0, world=1, shard_mode=0):
        out = np.zeros((H, W, 3), np.float32)
        fixed = np.zeros((H, W, 3), np.uint64)
        cnt = Counters()
        self.lib.orc_render(C.byref(self._s), self.bvh() if use_bvh else None, W, H, spp, max_depth, C.c_uint64(seed),
                            rank, world, shard_mode, C.c_void_p(out.ctypes.data), C.c_void_p(fixed.ctypes.data),
                            C.byref(cnt))
        return out, fixed, cnt.as_dict()

    # -- the double integrator (oracle/rrt_oracle_f64.c) --
    def camera_rays_f64(self, W, H, pixels, sample, seed):
        pixels = np.asarray(pixels, dtype=np.int32)
        out = np.zeros((len(pixels), 7), np.float64)
        f = self.lib.orc_d_camera_ray
        for k, p in enumerate(pixels):
            f(C.c_void_p(self.scene.camera.ctypes.data), W, H, int(p), int(sample), C.c_uint64(seed), C.c_void_p(out[k].ctypes.data))
        return out

    def trace_f64(self, rays7, t_min=0.001, mode="scan", want_rec=False):
        rays7 = np.ascontiguousarray(rays7, dtype=np.float64)
        n = len(rays7)
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        rec = np.zeros((n, 7), np.float64) if want_rec else None
        self.lib.orc_d_trace(C.byref(self._s), self.bvh() if mode == "bvh" else None, C.c_void_p(rays7.ctypes.data), n,
                             C.c_double(t_min), C.c_void_p(ids.ctypes.data), C.c_void_p(t.ctypes.data),
                             C.c_void_p(rec.ctypes.data) if want_rec else None)
        return (ids, t, rec) if want_rec else (ids, t)

    def scatter_f64(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float64)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32)
        out = np.zeros((len(in16), 8), np.float64)
        self.lib.orc_d_scatter(C.byref(self._s), C.c_void_p(in16.ctypes.data), C.c_void_p(rnd4.ctypes.data), len(in16),
                               C.c_void_p(out.ctypes.data))
        return out

    def render_f64(self, W, H, spp, max_depth=50, seed=1984, use_bvh=True):
        out = np.zeros((H, W, 3), np.float64)
        fixed = np.zeros((H, W, 3), np.uint64)
        cnt = Counters()
        self.lib.orc_d_render(C.byref(self._s), self.bvh() if use_bvh else None, W, H, spp, max_depth, C.c_uint64(seed),
                              C.c_void_p(out.ctypes.data), C.c_void_p(fixed.ctypes.data), C.byref(cnt))
        return out, fixed, cnt.as_dict()

    def tonemap(self, rgb_sum, spp):
        rgb_sum = np.ascontiguousarray(rgb_sum, dtype=np.float32)
        H, W, _ = rgb_sum.shape
        out = np.zeros((H, W, 3), np.uint8)
        self.lib.orc_tonemap_rgb8(C.c_void_p(rgb_sum.ctypes.data), W, H, spp, C.c_void_p(out.ctypes.data))
        return out


def philox(ctr4, key0, key1):
    lib = oracle_lib()
    ctr4 = np.ascontiguousarray(ctr4, dtype=np.uint32).reshape(-1, 4)
    out = np.zeros_like(ctr4)
    key = (C.c_uint32 * 2)(key0, key1)
    for i in range(len(ctr4)):
        lib.orc_philox4x32_10(C.c_void_p(ctr4[i].ctypes.data), key, C.c_void_p(out[i].ctypes.data))
    return out


def sincos2pi(u):
    lib = oracle_lib()
    c, s = C.c_float(), C.c_float()
    lib.orc_sincos2pi(C.c_float(u), C.byref(c), C.byref(s))
    return c.value, s.value


def camera_derive(lookfrom, lookat, vup, vfov, aspect, aperture, focus, t0=0.0, t1=0.0):
    lib = oracle_lib()
    out = np.zeros(1, camera_dtype)
    f3 = lambda v: (C.c_float * 3)(*[float(x) for x in v])
    lib.orc_camera_derive(f3(lookfrom), f3(lookat), f3(vup), C.c_float(vfov), C.c_float(aspect), C.c_float(aperture),
                          C.c_float(focus), C.c_float(t0), C.c_float(t1), C.c_void_p(out.ctypes.data))
    return out


# ------------------------------------------------------------------------------------------------
# oracle/_ref/libref_{f,d}.so -- the reference itself
# ------------------------------------------------------------------------------------------------
def have_ref():
    return os.path.exists(os.path.join(REF_DIR, "libref_f.so")) and os.path.exists(os.path.join(REF_DIR, "libref_d.so"))


def ref_scene_path(name):
    """The reference's scene file as staged by oracle/Makefile (oracle/_ref/scenes), else its stored stand-in
    (tests/golden/scenes): a text written from the reference parser's arrays (tests/golden/scene_*.npz) that parses
    back to exactly those arrays and counts."""
    for base in (os.path.join(REF_DIR, "scenes"), GOLDEN_SCENES):
        p = os.path.join(base, name)
        if os.path.exists(p):
            return p
    return None


_ref = {}


def ref_lib(precision="f"):
    if precision not in _ref:
        lib = C.CDLL(os.path.join(REF_DIR, "libref_%s.so" % precision))
        for fn in ("ref_scene_load", "ref_world_create", "ref_world_from_arrays", "ref_bvh_from_list", "ref_material_create"):
            getattr(lib, fn).restype = C.c_void_p
        lib.ref_reflectance.restype = C.c_double
        lib.ref_reflectance.argtypes = [C.c_double, C.c_double]
        lib.ref_random_uniform.restype = C.c_double
        _ref[precision] = lib
    return _ref[precision]


class RefScene:
    """A scene parsed by the reference's own parser (scene.h:212-452)."""

    def __init__(self, path, W, H, precision="f"):
        self.lib = ref_lib(precision)
        self.h = C.c_void_p(self.lib.ref_scene_load(path.encode(), W, H))
        cnt = (C.c_int * 6)()
        self.lib.ref_scene_counts(self.h, cnt)
        self.counts = dict(zip(("materials", "spheres", "mspheres", "triangles", "objs", "obj_insts"), list(cnt)))

    def arrays(self) -> SceneArrays:
        """The scene as float32 struct arrays (exact for the float build)."""
        c = self.counts
        lib = self.lib
        cam = np.zeros(24, np.float64)
        lib.ref_scene_camera(self.h, C.c_void_p(cam.ctypes.data))
        camera = np.zeros(1, camera_dtype)
        camera.view(np.float32)[:] = cam.astype(np.float32)
        nm = c["materials"]
        mt = np.zeros(nm, np.int32)
        mp = np.zeros((nm, 4), np.float64)
        lib.ref_scene_materials(self.h, C.c_void_p(mt.ctypes.data), C.c_void_p(mp.ctypes.data))
        mats = np.zeros(nm, material_dtype)
        mats["type"] = mt
        for i in range(nm):
            if mt[i] == 2:
                mats["param"][i] = mp[i, 0]
            else:
                mats["albedo"][i] = mp[i, :3]
                mats["param"][i] = mp[i, 3]
        ns = c["spheres"]
        s4 = np.zeros((ns, 4), np.float64)
        sm = np.zeros(ns, np.int32)
        lib.ref_scene_spheres(self.h, C.c_void_p(s4.ctypes.data), C.c_void_p(sm.ctypes.data))
        sph = np.zeros(ns, sphere_dtype)
        sph["center"], sph["radius"], sph["material"] = s4[:, :3], s4[:, 3], sm
        nms = c["mspheres"]
        m9 = np.zeros((nms, 9), np.float64)
        mm = np.zeros(nms, np.int32)
        lib.ref_scene_mspheres(self.h, C.c_void_p(m9.ctypes.data), C.c_void_p(mm.ctypes.data))
        ms = np.zeros(nms, msphere_dtype)
        ms["center0"], ms["center1"] = m9[:, :3], m9[:, 3:6]
        ms["time0"], ms["time1"], ms["radius"], ms["material"] = m9[:, 6], m9[:, 7], m9[:, 8], mm
        nt = c["triangles"]
        t9 = np.zeros((nt, 9), np.float64)
        tm = np.zeros(nt, np.int32)
        lib.ref_scene_triangles(self.h, C.c_void_p(t9.ctypes.data), C.c_void_p(tm.ctypes.data))
        tr = np.zeros(nt, triangle_dtype)
        tr["v0"], tr["v1"], tr["v2"], tr["material"] = t9[:, :3], t9[:, 3:6], t9[:, 6:9], tm
        return SceneArrays(camera, mats, sph, ms, tr)


class RefWorld:
    """The reference's hittable_list (object-id oracle) built from explicit arrays, in float or double."""

    def __init__(self, scene: SceneArrays, precision="d"):
        self.lib = ref_lib(precision)
        self.scene = scene
        d = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        i = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        m = scene.materials
        mp = np.zeros((len(m), 4), np.float64)
        for k in range(len(m)):
            if m["type"][k] == 2:
                mp[k, 0] = m["param"][k]
            else:
                mp[k, :3] = m["albedo"][k]
                mp[k, 3] = m["param"][k]
        s, ms, t = scene.spheres, scene.mspheres, scene.triangles
        s4 = d(np.concatenate([s["center"], s["radius"][:, None]], axis=1)) if len(s) else np.zeros((0, 4))
        m9 = (
            d(np.concatenate([ms["center0"], ms["center1"], ms["time0"][:, None], ms["time1"][:, None], ms["radius"][:, None]], axis=1))
            if len(ms) else np.zeros((0, 9))
        )
        t9 = d(np.concatenate([t["v0"], t["v1"], t["v2"]], axis=1)) if len(t) else np.zeros((0, 9))
        self._keep = (i(m["type"]), mp, s4, i(s["material"]), m9, i(ms["material"]), t9, i(t["material"]))
        k = self._keep
        vp = lambda a: C.c_void_p(a.ctypes.data)
        self.list = C.c_void_p(self.lib.ref_world_from_arrays(len(m), vp(k[0]), vp(k[1]), len(s), vp(k[2]), vp(k[3]),
                                                              len(ms), vp(k[4]), vp(k[5]), len(t), vp(k[6]), vp(k[7])))
        self.n = scene.n_objects

    def bvh(self):
        cam = self.scene.camera
        return C.c_void_p(self.lib.ref_bvh_from_list(self.list, C.c_double(float(cam["time0"][0])), C.c_double(float(cam["time1"][0]))))

    def trace_scan(self, rays7, t_min=0.001):
        r = np.ascontiguousarray(rays7, dtype=np.float64)
        n = len(r)
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        self.lib.ref_trace_scan(self.list, C.c_void_p(r.ctypes.data), n, C.c_double(t_min), C.c_void_p(ids.ctypes.data),
                                C.c_void_p(t.ctypes.data))
        return ids, t

    def trace_world(self, world, rays7, t_min=0.001):
        r = np.ascontiguousarray(rays7, dtype=np.float64)
        rec = np.zeros((len(r), 10), np.float64)
        self.lib.ref_trace_world(world, C.c_void_p(r.ctypes.data), len(r), C.c_double(t_min), C.c_void_p(rec.ctypes.data))
        return rec

    def hit_one(self, obj, ray7, t_min=0.001, t_max=np.inf):
        r = np.ascontiguousarray(ray7, dtype=np.float64)
        rec = np.zeros(8, np.float64)
        ok = self.lib.ref_hit_one(self.list, int(obj), C.c_void_p(r.ctypes.data), C.c_double(t_min), C.c_double(t_max),
                                  C.c_void_p(rec.ctypes.data))
        return bool(ok), rec

    def bounding_box(self, obj, time0, time1):
        out = np.zeros(6, np.float64)
        self.lib.ref_bounding_box(self.list, int(obj), C.c_double(time0), C.c_double(time1), C.c_void_p(out.ctypes.data))
        return out

    def ray_color_mean(self, world, ray7, depth, nsamples):
        r = np.ascontiguousarray(ray7, dtype=np.float64)
        out = np.zeros(3, np.float64)
        self.lib.ref_ray_color_mean(world, C.c_void_p(r.ctypes.data), depth, nsamples, C.c_void_p(out.ctypes.data))
        return out


def pinhole_rays(scene: SceneArrays, W, H, step=1):
    """Pixel-centre rays through the lens centre (no RNG): the deterministic primary-ray set used for
    hit-id / t parity (SURVEY 8c).  Same float arithmetic as camera.h:31-38 with rd = 0."""
    cam = scene.camera[0]
    jj, ii = np.meshgrid(np.arange(0, H, step), np.arange(0, W, step), indexing="ij")
    u = ((ii.astype(np.float32) + np.float32(0.5)) / np.float32(W - 1)).astype(np.float32)
    v = ((jj.astype(np.float32) + np.float32(0.5)) / np.float32(H - 1)).astype(np.float32)
    o = cam["origin"].astype(np.float32)
    d = (cam["lower_left_corner"][None, None, :] + u[..., None] * cam["horizontal"][None, None, :]).astype(np.float32)
    d = (d + v[..., None] * cam["vertical"][None, None, :]).astype(np.float32)
    d = (d - o[None, None, :]).astype(np.float32)
    rays = np.zeros((d.shape[0] * d.shape[1], 7), np.float32)
    rays[:, :3] = o
    rays[:, 3:6] = d.reshape(-1, 3)
    rays[:, 6] = cam["time0"]
    return rays


def psnr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    mse = np.mean((a - b) ** 2)
    return float("inf") if mse == 0 else 10.0 * np.log10(255.0 * 255.0 / mse)
