"""numpy / ctypes mirrors of the C ABI structs in include/rrtb.h.

The scene vocabulary is the reference's (scene.h:43-54,183-208; camera.h:40-48): spheres, moving
spheres, world-space triangles; lambertian / metal / dielectric materials; a derived thin-lens camera.
Beyond it: diffuse_light emitters (albedo = emitted radiance) and an optional constant background.
"""
import ctypes as C

import numpy as np

LAMBERTIAN, METAL, DIELECTRIC, DIFFUSE_LIGHT = 0, 1, 2, 3
SHARD_TILES, SHARD_SAMPLES = 0, 1
SCHED_AUTO, SCHED_SIMPLE, SCHED_POOL = 0, 1, 2

camera_dtype = np.dtype(
    [
        ("origin", "<f4", 3),
        ("lower_left_corner", "<f4", 3),
        ("horizontal", "<f4", 3),
        ("vertical", "<f4", 3),
        ("u", "<f4", 3),
        ("v", "<f4", 3),
        ("w", "<f4", 3),
        ("lens_radius", "<f4"),
        ("time0", "<f4"),
        ("time1", "<f4"),
    ]
)
material_dtype = np.dtype([("type", "<i4"), ("albedo", "<f4", 3), ("param", "<f4")])
sphere_dtype = np.dtype([("center", "<f4", 3), ("radius", "<f4"), ("material", "<i4")])
msphere_dtype = np.dtype(
    [("center0", "<f4", 3), ("center1", "<f4", 3), ("time0", "<f4"), ("time1", "<f4"), ("radius", "<f4"), ("material", "<i4")]
)
triangle_dtype = np.dtype([("v0", "<f4", 3), ("v1", "<f4", 3), ("v2", "<f4", 3), ("material", "<i4")])
# SURVEY 8f4: a triangle of a moving instance (vertices at time0; until time1 vertex 0 moves by delta, vertex 1 by
# delta + extra1, vertex 2 by delta + extra2 -- extras 0 = translation, include/rrtb.h "rrtb_mtriangle")
mtriangle_dtype = np.dtype(
    [("v0", "<f4", 3), ("v1", "<f4", 3), ("v2", "<f4", 3), ("delta", "<f4", 3), ("time0", "<f4"), ("time1", "<f4"), ("material", "<i4"),
     ("extra1", "<f4", 3), ("extra2", "<f4", 3)]
)

assert camera_dtype.itemsize == 96
assert mtriangle_dtype.itemsize == 84
assert material_dtype.itemsize == 20
assert sphere_dtype.itemsize == 20
assert msphere_dtype.itemsize == 40
assert triangle_dtype.itemsize == 40


class RenderParams(C.Structure):
    """rrtb_render_params"""

    _fields_ = [
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("spp", C.c_int32),
        ("max_depth", C.c_int32),
        ("seed", C.c_uint64),
        ("rank", C.c_int32),
        ("world", C.c_int32),
        ("shard_mode", C.c_int32),
        ("count_rays", C.c_int32),
        ("scheduler", C.c_int32),
        ("precision", C.c_int32),
    ]


class Stats(C.Structure):
    """rrtb_stats"""

    _fields_ = [
        ("seconds_render", C.c_double),
        ("seconds_build", C.c_double),
        ("seconds_resolve", C.c_double),
        ("rays", C.c_uint64),
        ("paths", C.c_uint64),
        ("box_tests", C.c_uint64),
        ("sphere_tests", C.c_uint64),
        ("msphere_tests", C.c_uint64),
        ("triangle_tests", C.c_uint64),
        ("hits", C.c_uint64),
        ("kernel_launches", C.c_int32),
        ("reserved", C.c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class SceneArrays:
    """A scene as plain arrays, in the reference's object-id order (spheres, moving spheres, triangles;
    rrt.cu:151-164), then the moving triangles of SURVEY 8f4.  `background`: None renders the reference's sky,
    an RGB triple a constant background instead (include/rrtb.h rrtb_scene_stage_background)."""

    def __init__(self, camera, materials, spheres=None, mspheres=None, triangles=None, mtriangles=None, background=None):
        self.camera = np.ascontiguousarray(np.asarray(camera, dtype=camera_dtype).reshape(1))
        self.materials = np.ascontiguousarray(np.asarray(materials, dtype=material_dtype))
        self.spheres = np.ascontiguousarray(
            np.zeros(0, sphere_dtype) if spheres is None else np.asarray(spheres, dtype=sphere_dtype)
        )
        self.mspheres = np.ascontiguousarray(
            np.zeros(0, msphere_dtype) if mspheres is None else np.asarray(mspheres, dtype=msphere_dtype)
        )
        self.triangles = np.ascontiguousarray(
            np.zeros(0, triangle_dtype) if triangles is None else np.asarray(triangles, dtype=triangle_dtype)
        )
        self.mtriangles = np.ascontiguousarray(
            np.zeros(0, mtriangle_dtype) if mtriangles is None else np.asarray(mtriangles, dtype=mtriangle_dtype)
        )
        self.background = None if background is None else np.ascontiguousarray(np.asarray(background, dtype=np.float32).reshape(3))

    @property
    def n_objects(self):
        return len(self.spheres) + len(self.mspheres) + len(self.triangles) + len(self.mtriangles)

    def counts(self):
        return dict(
            materials=len(self.materials),
            spheres=len(self.spheres),
            mspheres=len(self.mspheres),
            triangles=len(self.triangles),
            mtriangles=len(self.mtriangles),
        )

    # ---- (de)serialisation used by the golden fixtures (tests/golden/*.npz) ----
    def to_npz_dict(self):
        d = dict(
            camera=self.camera.view(np.uint8),
            materials=self.materials.view(np.uint8),
            spheres=self.spheres.view(np.uint8),
            mspheres=self.mspheres.view(np.uint8),
            triangles=self.triangles.view(np.uint8),
            mtriangles=self.mtriangles.view(np.uint8),
        )
        if self.background is not None:
            d["background"] = self.background.copy()
        return d

    @classmethod
    def from_npz_dict(cls, d):
        def v(name, dt):
            if name not in d:  # fixtures written before a primitive kind existed
                return np.zeros(0, dt)
            a = np.ascontiguousarray(d[name]).view(np.uint8)
            return a.view(dt) if a.size else np.zeros(0, dt)

        return cls(
            v("camera", camera_dtype),
            v("materials", material_dtype),
            v("spheres", sphere_dtype),
            v("mspheres", msphere_dtype),
            v("triangles", triangle_dtype),
            v("mtriangles", mtriangle_dtype),
            background=np.asarray(d["background"], np.float32) if "background" in d else None,  # older fixtures: the sky
        )
