"""Python host-side mirror of the reference's renderer seam, over the C ABI (include/rrtb.h).

  Scene   <-> `scene` (scene.h:210-481): parsed by the C++ parser inside librrtb200.so
  Rrt     <-> `class Rrt` (rrt.h:14-48): Rrt(w, h, spp, max_depth, use_bvh, tx, ty).render(scene) -> fb
  Context  :  one GPU context; the lower-level calls the parity tests and bench.py use

Everything that computes runs in the CUDA library; numpy is only the container for host buffers.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import RrtbError
from .types import (
    RenderParams,
    SceneArrays,
    Stats,
    camera_dtype,
    material_dtype,
    msphere_dtype,
    mtriangle_dtype,
    sphere_dtype,
    triangle_dtype,
)


class SceneError(RrtbError):
    """Parse failure; `.ref_exit_code` is the exit code the reference's parser would have used
    (1 obj/arg errors, 2 cannot open, 3 unknown material type, 4 missing camera/materials/objects)."""

    def __init__(self, status, message, ref_exit_code):
        super().__init__(status, message)
        self.ref_exit_code = ref_exit_code
        self.message = message


def _vp(a):
    return C.c_void_p(a.ctypes.data) if a is not None and a.size else C.c_void_p(0)


class Scene:
    """A scene in the reference's vocabulary.  Build with Scene.from_file (reference grammar) or
    Scene.from_arrays."""

    def __init__(self, arrays: SceneArrays, n_objs=0, n_obj_insts=0):
        self.arrays = arrays
        self.n_objs = n_objs
        self.n_obj_insts = n_obj_insts

    @classmethod
    def from_arrays(cls, arrays: SceneArrays):
        return cls(arrays)

    @classmethod
    def from_file(cls, path, image_width, image_height):
        lib = _lib.load()
        h = C.c_void_p()
        code = C.c_int(0)
        err = C.create_string_buffer(512)
        rc = lib.rrtb_scene_parse_file(str(path).encode(), int(image_width), int(image_height), C.byref(h), C.byref(code), err, 512)
        if rc != 0:
            raise SceneError(rc, err.value.decode(errors="replace"), code.value)
        try:
            cnt = (C.c_int32 * 6)()
            lib.rrtb_scene_counts(h, cnt)
            nm, ns, nms, nt, nobj, ninst = list(cnt)
            bg = np.zeros(3, np.float32)

            def grab(ptr, n, dt):
                if n == 0 or not ptr:
                    return np.zeros(0, dt)
                buf = (C.c_char * (n * dt.itemsize)).from_address(ptr)
                return np.frombuffer(buf, dtype=dt, count=n).copy()

            arrays = SceneArrays(
                grab(lib.rrtb_scene_camera(h), 1, camera_dtype),
                grab(lib.rrtb_scene_materials(h), nm, material_dtype),
                grab(lib.rrtb_scene_spheres(h), ns, sphere_dtype),
                grab(lib.rrtb_scene_mspheres(h), nms, msphere_dtype),
                grab(lib.rrtb_scene_triangles(h), nt, triangle_dtype),
                grab(lib.rrtb_scene_mtriangles(h), lib.rrtb_scene_mtriangle_count(h), mtriangle_dtype),
                background=bg if lib.rrtb_scene_background(h, _vp(bg)) else None,
            )
        finally:
            lib.rrtb_scene_free(h)
        return cls(arrays, nobj, ninst)

    def counts(self):
        c = self.arrays.counts()
        c.update(objs=self.n_objs, obj_insts=self.n_obj_insts)
        return c

    def summary(self, filename):
        """The lines the reference prints to stderr after parsing (scene.h:443-451)."""
        a = self.arrays
        lines = [
            "read scene file: %s" % filename,
            "material count:  %d" % len(a.materials),
            "sphere count:    %d" % len(a.spheres),
            "msphere count:   %d" % len(a.mspheres),
            "obj count:       %d" % self.n_objs,
            "obj_inst count:  %d" % self.n_obj_insts,
        ]
        if a.camera["time0"][0] != a.camera["time1"][0]:
            lines.append("camera time:     %g - %g" % (a.camera["time0"][0], a.camera["time1"][0]))
        return "\n".join(lines)


_PRECISION = {"f32": 0, "f64": 1, 0: 0, 1: 1}
FRAME_HANDLE_BYTES = 192  # RRTB_FRAME_HANDLE_BYTES


def render_group(contexts, width, height, spp, max_depth=50, seed=1984, shard_mode=0, out=None, dtype=np.float32, precision="f32",
                 count_rays=False):
    """One process, n GPUs (the drop-in's `-G n`): contexts[0] owns the frame, every context has the scene loaded;
    shard i of len(contexts) renders on contexts[i] and lands in the owner's frame over NVLink."""
    lib = contexts[0].lib
    dtype = np.dtype(dtype) if out is None else out.dtype
    if out is None:
        out = np.empty((height, width, 3), dtype)
    p = Context.params(width, height, spp, max_depth, seed, 0, len(contexts), shard_mode, count_rays, 0, precision)
    hs = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
    st = Stats()
    rc = lib.rrtb_render_group(hs, len(contexts), C.byref(p), 1 if dtype == np.dtype(np.float64) else 0, C.c_void_p(out.ctypes.data), C.byref(st))
    if rc != 0:
        raise RrtbError(rc, lib.rrtb_last_error(contexts[0].h).decode())
    return out, st.as_dict()


class PinnedBuffer:
    """Page-locked host memory from rrtb_host_alloc as a numpy array (`.array`): device copies to / from it are DMA."""

    def __init__(self, shape, dtype=np.float32):
        self.lib = _lib.load()
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        self.ptr = self.lib.rrtb_host_alloc(n)
        if not self.ptr:
            raise MemoryError("rrtb_host_alloc(%d)" % n)
        self.array = np.frombuffer((C.c_char * n).from_address(self.ptr), dtype=dtype).reshape(shape)

    def free(self):
        if getattr(self, "ptr", None):
            self.array = None
            self.lib.rrtb_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One GPU.  Raises RrtbError(RRTB_ERR_NO_DEVICE) when there is no CUDA device: no CPU fallback."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        self.h = C.c_void_p()
        rc = self.lib.rrtb_create(C.byref(self.h), int(device))
        if rc != 0:
            raise RrtbError(rc, self.lib.rrtb_last_error(None).decode())
        self.device = device
        self.scene = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.rrtb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise RrtbError(rc, self.lib.rrtb_last_error(self.h).decode())

    def device_info(self):
        out = (C.c_int64 * 4)()
        name = C.create_string_buffer(256)
        self._check(self.lib.rrtb_device_info(self.h, out, name, 256))
        return dict(name=name.value.decode(), sm_count=out[0], clock_khz=out[1], l2_bytes=out[2], cc=out[3])

    def probe_issue_rate(self):
        """Measured FP32-issue roofline denominators on this device (lane-instructions / s)."""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.rrtb_probe_issue_rate(self.h, C.byref(a), C.byref(b)))
        return dict(ffma=a.value, ffma_fmnmx_mix=b.value)

    # -- scene ------------------------------------------------------------------------------------------
    def set_scene(self, scene, use_bvh=True):
        a = scene.arrays if isinstance(scene, Scene) else scene
        # SURVEY 8f4: moving triangles are staged, then consumed by rrtb_scene_set
        self._check(self.lib.rrtb_scene_stage_moving_triangles(self.h, _vp(a.mtriangles), len(a.mtriangles)))
        self._check(self.lib.rrtb_scene_stage_background(self.h, _vp(a.background)))  # None: the sky
        self._check(
            self.lib.rrtb_scene_set(
                self.h, _vp(a.camera), _vp(a.materials), len(a.materials), _vp(a.spheres), len(a.spheres),
                _vp(a.mspheres), len(a.mspheres), _vp(a.triangles), len(a.triangles), 1 if use_bvh else 0,
            )
        )
        self.scene = a

    def set_camera(self, camera):
        cam = np.ascontiguousarray(np.asarray(camera, dtype=camera_dtype).reshape(1))
        self._check(self.lib.rrtb_camera_set(self.h, _vp(cam)))

    # -- render -----------------------------------------------------------------------------------------
    @staticmethod
    def params(width, height, spp, max_depth=50, seed=1984, rank=0, world=1, shard_mode=0, count_rays=False, scheduler=0,
               precision="f32"):
        return RenderParams(int(width), int(height), int(spp), int(max_depth), int(seed), int(rank), int(world),
                            int(shard_mode), 1 if count_rays else 0, int(scheduler), _PRECISION[precision])

    def render(self, width, height, spp, max_depth=50, seed=1984, rank=0, world=1, shard_mode=0, count_rays=False, out=None, scheduler=0,
               dtype=np.float32, precision="f32"):
        """Host-buffer path (what Rrt::render returns): [H, W, 3] SUMS, row 0 = bottom scanline.
        dtype float32 = the `rrt` framebuffer, float64 = the `rrtd` framebuffer (rrtb_render_f64);
        precision "f32" / "f64" = the arithmetic of the integrator (the reference's rrt / rrtd builds)."""
        p = self.params(width, height, spp, max_depth, seed, rank, world, shard_mode, count_rays, scheduler, precision)
        dtype = np.dtype(dtype) if out is None else out.dtype
        assert dtype in (np.dtype(np.float32), np.dtype(np.float64))
        if out is None:
            out = np.empty((height, width, 3), dtype)
        assert out.flags.c_contiguous and out.size == 3 * width * height
        st = Stats()
        fn = self.lib.rrtb_render if dtype == np.dtype(np.float32) else self.lib.rrtb_render_f64
        self._check(fn(self.h, C.byref(p), C.c_void_p(out.ctypes.data), C.byref(st)))
        return out, st.as_dict()

    def render_aov(self, width, height, spp, seed=1984, rank=0, world=1, count_rays=False, precision="f32"):
        """First-hit AOVs (include/rrtb.h rrtb_render_aov) of tile shard (rank, world): dict of float32 MEANS albedo
        [H, W, 3], normal [H, W, 3], depth [H, W], coverage [H, W] (row 0 = bottom scanline; pixels of other shards 0),
        and the stats."""
        p = self.params(width, height, spp, 1, seed, rank, world, 0, count_rays, 0, precision)
        out = dict(albedo=np.zeros((height, width, 3), np.float32), normal=np.zeros((height, width, 3), np.float32),
                   depth=np.zeros((height, width), np.float32), coverage=np.zeros((height, width), np.float32))
        st = Stats()
        self._check(self.lib.rrtb_render_aov(self.h, C.byref(p), _vp(out["albedo"]), _vp(out["normal"]), _vp(out["depth"]),
                                             _vp(out["coverage"]), C.byref(st)))
        return out, st.as_dict()

    def render_device(self, params, accum_ptr):
        """Device-resident path: adds this shard into the uint64 accumulator at device address accum_ptr."""
        st = Stats()
        self._check(self.lib.rrtb_render_device(self.h, C.byref(params), C.c_void_p(int(accum_ptr)), C.byref(st)))
        return st.as_dict()

    def resolve_device(self, accum_ptr, out_ptr, n):
        self._check(self.lib.rrtb_resolve_device(self.h, C.c_void_p(int(accum_ptr)), C.c_void_p(int(out_ptr)), int(n)))

    def accumulate_device(self, dst_ptr, src_ptr, n):
        self._check(self.lib.rrtb_accumulate_device(self.h, C.c_void_p(int(dst_ptr)), C.c_void_p(int(src_ptr)), int(n)))

    # -- multi-GPU frame (include/rrtb.h "multi-GPU") -----------------------------------------------------
    def frame_create(self, width, height, f64=False):
        """Owner (rank 0): the frame every rank's epilogue writes its shard into."""
        self._check(self.lib.rrtb_frame_create(self.h, int(width), int(height), 1 if f64 else 0))

    def frame_export(self):
        """Owner: the bytes another PROCESS needs to map the frame (rrtb_frame_import)."""
        buf = C.create_string_buffer(FRAME_HANDLE_BYTES)
        self._check(self.lib.rrtb_frame_export(self.h, buf))
        return buf.raw

    def frame_import(self, handle):
        assert len(handle) == FRAME_HANDLE_BYTES
        self._check(self.lib.rrtb_frame_import(self.h, C.create_string_buffer(bytes(handle), FRAME_HANDLE_BYTES)))

    def frame_attach(self, owner):
        """Same process: peer access to the owner context's frame."""
        self._check(self.lib.rrtb_frame_attach(self.h, owner.h))

    def frame_detach(self):
        self._check(self.lib.rrtb_frame_detach(self.h))

    def render_shard(self, params):
        """Render shard (params.rank, params.world) and store / add it into the owner's frame."""
        st = Stats()
        self._check(self.lib.rrtb_render_shard(self.h, C.byref(params), C.byref(st)))
        return st.as_dict()

    def frame_download(self, out, shard_mode=0):
        """Owner: frame -> host array `out` ([H, W, 3] float32, or float64 for an f64 frame)."""
        assert out.flags.c_contiguous
        self._check(self.lib.rrtb_frame_download(self.h, int(shard_mode), C.c_void_p(out.ctypes.data)))
        return out

    # -- test hooks -------------------------------------------------------------------------------------
    def trace(self, rays7, t_min=0.001, mode="bvh", want_rec=False):
        rays7 = np.ascontiguousarray(rays7, dtype=np.float32).reshape(-1, 7)
        n = len(rays7)
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        rec = np.zeros((n, 7), np.float32) if want_rec else None
        self._check(self.lib.rrtb_trace_closest(self.h, _vp(rays7), n, float(t_min), 1 if mode == "bvh" else 0, _vp(ids), _vp(t),
                                                _vp(rec) if want_rec else C.c_void_p(0)))
        return (ids, t, rec) if want_rec else (ids, t)

    def camera_rays(self, width, height, pixels, sample, seed=1984):
        pixels = np.ascontiguousarray(pixels, dtype=np.int32)
        out = np.zeros((len(pixels), 7), np.float32)
        p = self.params(width, height, 1, 1, seed)
        self._check(self.lib.rrtb_camera_rays(self.h, C.byref(p), _vp(pixels), len(pixels), int(sample), _vp(out)))
        return out

    def trace_f64(self, rays7, t_min=0.001, mode="bvh", want_rec=False):
        rays7 = np.ascontiguousarray(rays7, dtype=np.float64).reshape(-1, 7)
        n = len(rays7)
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        rec = np.zeros((n, 7), np.float64) if want_rec else None
        self._check(self.lib.rrtb_trace_closest_f64(self.h, _vp(rays7), n, C.c_double(t_min), 1 if mode == "bvh" else 0, _vp(ids),
                                                    _vp(t), _vp(rec) if want_rec else C.c_void_p(0)))
        return (ids, t, rec) if want_rec else (ids, t)

    def camera_rays_f64(self, width, height, pixels, sample, seed=1984):
        pixels = np.ascontiguousarray(pixels, dtype=np.int32)
        out = np.zeros((len(pixels), 7), np.float64)
        p = self.params(width, height, 1, 1, seed)
        self._check(self.lib.rrtb_camera_rays_f64(self.h, C.byref(p), _vp(pixels), len(pixels), int(sample), _vp(out)))
        return out

    def scatter_f64(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float64).reshape(-1, 16)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32).reshape(-1, 4)
        out = np.zeros((len(in16), 8), np.float64)
        self._check(self.lib.rrtb_scatter_f64(self.h, _vp(in16), _vp(rnd4), len(in16), _vp(out)))
        return out

    def bvh_arrays(self):
        n = C.c_int32()
        self._check(self.lib.rrtb_bvh_size(self.h, C.byref(n)))
        n = n.value
        ni = max(n - 1, 0)
        morton = np.zeros(n, np.uint32)
        perm = np.zeros(n, np.uint32)
        left = np.zeros(ni, np.int32)
        right = np.zeros(ni, np.int32)
        parent = np.zeros(2 * n - 1, np.int32)
        node_box = np.zeros((ni, 6), np.float32)
        prim_box = np.zeros((n, 6), np.float32)
        self._check(self.lib.rrtb_bvh_download(self.h, _vp(morton), _vp(perm), _vp(left), _vp(right), _vp(parent), _vp(node_box), _vp(prim_box)))
        return dict(morton=morton, perm=perm, left=left, right=right, parent=parent, node_box=node_box, prim_box=prim_box)

    def wide_arrays(self):
        """The W-wide traversal tree: dict(c=[m,3,W] centres, h=[m,3,W] half extents, ref=[m,W] child refs)."""
        n, w = C.c_int32(), C.c_int32()
        self._check(self.lib.rrtb_wide_size(self.h, C.byref(n), C.byref(w)))
        n, w = n.value, w.value
        raw = np.zeros((n, 8 * w), np.float32)
        self._check(self.lib.rrtb_wide_download(self.h, _vp(raw), n))
        return dict(c=raw[:, 0:3 * w].reshape(-1, 3, w).copy(), h=raw[:, 3 * w:6 * w].reshape(-1, 3, w).copy(),
                    ref=raw[:, 6 * w:7 * w].copy().view(np.int32))

    def wide_raw(self):
        """The traversal nodes as the device holds them: [m, 24] uint32, or [m, 40] for motion nodes (include/rrtb.h
        rrtb_wide_download_raw), in the build's own node numbering."""
        n = C.c_int32()
        self._check(self.lib.rrtb_wide_size(self.h, C.byref(n), None))
        raw = np.zeros((n.value, 40), np.uint32)
        wpn = C.c_int32()
        self._check(self.lib.rrtb_wide_download_raw(self.h, _vp(raw), n.value, C.byref(wpn)))
        return raw.reshape(-1)[:n.value * wpn.value].reshape(n.value, wpn.value).copy()

    def philox(self, ctr4, key0, key1):
        ctr4 = np.ascontiguousarray(ctr4, dtype=np.uint32).reshape(-1, 4)
        out = np.zeros_like(ctr4)
        self._check(self.lib.rrtb_philox(self.h, _vp(ctr4), len(ctr4), int(key0), int(key1), _vp(out)))
        return out

    def scatter(self, in16, rnd4):
        in16 = np.ascontiguousarray(in16, dtype=np.float32).reshape(-1, 16)
        rnd4 = np.ascontiguousarray(rnd4, dtype=np.uint32).reshape(-1, 4)
        out = np.zeros((len(in16), 8), np.float32)
        self._check(self.lib.rrtb_scatter(self.h, _vp(in16), _vp(rnd4), len(in16), _vp(out)))
        return out


def camera_derive(lookfrom, lookat, vup, vfov, aspect_ratio, aperture, focus_dist, time0=0.0, time1=0.0):
    """camera.h:8-29 in the reference's float arithmetic (host code inside the library)."""
    lib = _lib.load()
    out = np.zeros(1, camera_dtype)
    f3 = lambda v: (C.c_float * 3)(*[float(x) for x in v])
    rc = lib.rrtb_camera_derive(f3(lookfrom), f3(lookat), f3(vup), vfov, aspect_ratio, aperture, focus_dist, time0, time1, _vp(out))
    if rc != 0:
        raise RrtbError(rc, "rrtb_camera_derive")
    return out


def tonemap(rgb_sum, spp):
    """color.h:8-23 + main.cpp:150-163: float sums (bottom-up) -> uint8 [H, W, 3] top-down."""
    lib = _lib.load()
    f64 = np.asarray(rgb_sum).dtype == np.float64  # the rrtd framebuffer: color.h with FP_T = double
    rgb_sum = np.ascontiguousarray(rgb_sum, dtype=np.float64 if f64 else np.float32)
    H, W, _ = rgb_sum.shape
    out = np.zeros((H, W, 3), np.uint8)
    rc = (lib.rrtb_tonemap_rgb8_f64 if f64 else lib.rrtb_tonemap_rgb8)(_vp(rgb_sum), W, H, int(spp), _vp(out))
    if rc != 0:
        raise RrtbError(rc, "rrtb_tonemap_rgb8")
    return out


def write_png(path, rgb8):
    lib = _lib.load()
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    H, W, _ = rgb8.shape
    rc = lib.rrtb_write_png(str(path).encode(), W, H, _vp(rgb8))
    if rc != 0:
        raise RrtbError(rc, "rrtb_write_png(%s)" % path)


def write_pfm(path, array):
    """rrtb_write_pfm: a float32 [H, W, 3] or [H, W] array (row 0 = bottom, the framebuffer order) as a little-endian PFM."""
    lib = _lib.load()
    a = np.ascontiguousarray(array, dtype=np.float32)
    assert a.ndim in (2, 3) and (a.ndim == 2 or a.shape[2] in (1, 3)), a.shape
    rc = lib.rrtb_write_pfm(str(path).encode(), a.shape[1], a.shape[0], 1 if a.ndim == 2 else a.shape[2], _vp(a))
    if rc != 0:
        raise RrtbError(rc, "rrtb_write_pfm(%s)" % path)


class Rrt:
    """Mirror of the reference's `class Rrt` (rrt.h:14-48; CUDA build signature with threads_x/threads_y).

    threads_x/threads_y are accepted for drop-in compatibility and ignored: the persistent kernel picks
    its own launch shape (the reference's `-tx/-ty` tuned a one-thread-per-pixel grid, rrt.cu:192-193)."""

    def __init__(self, image_width, image_height, samples_per_pixel, max_depth, use_bvh=True, threads_x=8, threads_y=8, device=0, seed=1984,
                 precision="f32"):
        self.precision = precision  # "f32" = the reference's rrt build, "f64" = rrtd (FP_T = double)
        self.image_width = image_width
        self.image_height = image_height
        self.samples_per_pixel = samples_per_pixel
        self.max_depth = max_depth
        self.bvh = use_bvh
        self.num_threads_x, self.num_threads_y = threads_x, threads_y
        self.seed = seed
        self.ctx = Context(device)
        self.fb = None
        self.stats = None

    def render(self, the_scene):
        """-> fb: FP_T [H, W, 3] (float32, or float64 for precision "f64"); fb[j, i] is the SUM over samples for
        pixel (i, j), j = 0 bottom row (the reference returns vec3* indexed j*W+i, rrt.cu:121,334)."""
        self.ctx.set_scene(the_scene, self.bvh)
        f64 = _PRECISION[self.precision] == 1
        self.fb, self.stats = self.ctx.render(self.image_width, self.image_height, self.samples_per_pixel, self.max_depth, self.seed,
                                              count_rays=True, dtype=np.float64 if f64 else np.float32, precision=self.precision)
        return self.fb

    def render_aov(self, the_scene):
        """First-hit AOVs of the scene at this renderer's size, samples, seed and precision: (dict of albedo, normal,
        depth, coverage means, as Context.render_aov), stats."""
        self.ctx.set_scene(the_scene, self.bvh)
        return self.ctx.render_aov(self.image_width, self.image_height, self.samples_per_pixel, self.seed, count_rays=True,
                                   precision=self.precision)
