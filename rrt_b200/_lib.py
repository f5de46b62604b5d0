"""ctypes loader for rrt_b200/librrtb200.so (C ABI: include/rrtb.h).

There is no Python or CPU fallback: if the shared library has not been built this raises, and if it is
built but no CUDA device is present `Context()` raises (RRTB_ERR_NO_DEVICE).
"""
import ctypes as C
import os

from .types import RenderParams, Stats

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RRTB_LIB") or os.path.join(_HERE, "librrtb200.so")  # RRTB_LIB: tuning aid (variant builds)

# every symbol include/rrtb.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "rrtb_abi_version", "rrtb_create", "rrtb_destroy", "rrtb_last_error", "rrtb_device_info",
    "rrtb_scene_set", "rrtb_scene_stage_moving_triangles", "rrtb_scene_stage_background", "rrtb_camera_set", "rrtb_render", "rrtb_render_f64", "rrtb_render_aov", "rrtb_render_device", "rrtb_resolve_device",
    "rrtb_accumulate_device", "rrtb_frame_create", "rrtb_frame_export", "rrtb_frame_import", "rrtb_frame_attach", "rrtb_frame_detach",
    "rrtb_render_shard", "rrtb_frame_download", "rrtb_render_group", "rrtb_host_alloc", "rrtb_host_free", "rrtb_trace_closest", "rrtb_trace_closest_f64", "rrtb_camera_rays", "rrtb_camera_rays_f64",
    "rrtb_bvh_size", "rrtb_bvh_download", "rrtb_wide_size", "rrtb_wide_download", "rrtb_wide_download_raw", "rrtb_philox", "rrtb_scatter", "rrtb_scatter_f64", "rrtb_probe_issue_rate", "rrtb_scene_parse_file", "rrtb_scene_free", "rrtb_scene_counts",
    "rrtb_scene_camera", "rrtb_scene_materials", "rrtb_scene_spheres", "rrtb_scene_mspheres",
    "rrtb_scene_triangles", "rrtb_scene_mtriangle_count", "rrtb_scene_mtriangles", "rrtb_scene_background", "rrtb_scene_upload", "rrtb_camera_derive", "rrtb_tonemap_rgb8", "rrtb_tonemap_rgb8_f64", "rrtb_write_png", "rrtb_write_pfm",
]

STATUS = {0: "RRTB_OK", -1: "RRTB_ERR_INVALID", -2: "RRTB_ERR_NO_DEVICE", -3: "RRTB_ERR_CUDA", -4: "RRTB_ERR_NO_SCENE",
          -5: "RRTB_ERR_IO", -6: "RRTB_ERR_PARSE", -7: "RRTB_ERR_NOMEM"}


class RrtbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s: %s" % (STATUS.get(status, status), message))
        self.status = status


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "rrt_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_float
    P = C.POINTER
    sig = {
        "rrtb_abi_version": (C.c_int, []),
        "rrtb_create": (C.c_int, [P(vp), C.c_int]),
        "rrtb_destroy": (None, [vp]),
        "rrtb_last_error": (C.c_char_p, [vp]),
        "rrtb_device_info": (C.c_int, [vp, P(C.c_int64), C.c_char_p, C.c_int]),
        "rrtb_scene_set": (C.c_int, [vp, vp, vp, C.c_int, vp, C.c_int, vp, C.c_int, vp, C.c_int, C.c_int]),
        "rrtb_scene_stage_moving_triangles": (C.c_int, [vp, vp, C.c_int]),
        "rrtb_scene_stage_background": (C.c_int, [vp, vp]),
        "rrtb_camera_set": (C.c_int, [vp, vp]),
        "rrtb_render": (C.c_int, [vp, P(RenderParams), vp, P(Stats)]),
        "rrtb_render_f64": (C.c_int, [vp, P(RenderParams), vp, P(Stats)]),
        "rrtb_render_aov": (C.c_int, [vp, P(RenderParams), vp, vp, vp, vp, P(Stats)]),
        "rrtb_render_device": (C.c_int, [vp, P(RenderParams), vp, P(Stats)]),
        "rrtb_resolve_device": (C.c_int, [vp, vp, vp, C.c_size_t]),
        "rrtb_accumulate_device": (C.c_int, [vp, vp, vp, C.c_size_t]),
        "rrtb_frame_create": (C.c_int, [vp, C.c_int, C.c_int, C.c_int]),
        "rrtb_frame_export": (C.c_int, [vp, vp]),
        "rrtb_frame_import": (C.c_int, [vp, vp]),
        "rrtb_frame_attach": (C.c_int, [vp, vp]),
        "rrtb_frame_detach": (C.c_int, [vp]),
        "rrtb_render_shard": (C.c_int, [vp, P(RenderParams), P(Stats)]),
        "rrtb_frame_download": (C.c_int, [vp, C.c_int, vp]),
        "rrtb_render_group": (C.c_int, [P(vp), C.c_int, P(RenderParams), C.c_int, vp, P(Stats)]),
        "rrtb_host_alloc": (vp, [C.c_size_t]),
        "rrtb_host_free": (None, [vp]),
        "rrtb_trace_closest": (C.c_int, [vp, vp, C.c_int, f32, C.c_int, vp, vp, vp]),
        "rrtb_camera_rays": (C.c_int, [vp, P(RenderParams), vp, C.c_int, C.c_int, vp]),
        "rrtb_trace_closest_f64": (C.c_int, [vp, vp, C.c_int, C.c_double, C.c_int, vp, vp, vp]),
        "rrtb_camera_rays_f64": (C.c_int, [vp, P(RenderParams), vp, C.c_int, C.c_int, vp]),
        "rrtb_scatter_f64": (C.c_int, [vp, vp, vp, C.c_int, vp]),
        "rrtb_bvh_size": (C.c_int, [vp, P(i32)]),
        "rrtb_bvh_download": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp]),
        "rrtb_wide_size": (C.c_int, [vp, P(i32), P(i32)]),
        "rrtb_wide_download": (C.c_int, [vp, vp, i32]),
        "rrtb_wide_download_raw": (C.c_int, [vp, vp, i32, P(i32)]),
        "rrtb_philox": (C.c_int, [vp, vp, C.c_int, u32, u32, vp]),
        "rrtb_scatter": (C.c_int, [vp, vp, vp, C.c_int, vp]),
        "rrtb_probe_issue_rate": (C.c_int, [vp, P(C.c_double), P(C.c_double)]),
        "rrtb_scene_parse_file": (C.c_int, [C.c_char_p, C.c_int, C.c_int, P(vp), P(C.c_int), C.c_char_p, C.c_int]),
        "rrtb_scene_free": (None, [vp]),
        "rrtb_scene_counts": (C.c_int, [vp, P(i32)]),
        "rrtb_scene_camera": (vp, [vp]),
        "rrtb_scene_materials": (vp, [vp]),
        "rrtb_scene_spheres": (vp, [vp]),
        "rrtb_scene_mspheres": (vp, [vp]),
        "rrtb_scene_triangles": (vp, [vp]),
        "rrtb_scene_mtriangle_count": (C.c_int, [vp]),
        "rrtb_scene_mtriangles": (vp, [vp]),
        "rrtb_scene_background": (C.c_int, [vp, vp]),
        "rrtb_scene_upload": (C.c_int, [vp, vp, C.c_int]),
        "rrtb_camera_derive": (C.c_int, [P(f32), P(f32), P(f32), f32, f32, f32, f32, f32, f32, vp]),
        "rrtb_tonemap_rgb8": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp]),
        "rrtb_tonemap_rgb8_f64": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp]),
        "rrtb_write_png": (C.c_int, [C.c_char_p, C.c_int, C.c_int, vp]),
        "rrtb_write_pfm": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, vp]),
    }
    for name in SYMBOLS:
        fn = getattr(lib, name)  # raises AttributeError if the library does not export it
        fn.restype, fn.argtypes = sig[name]
    if lib.rrtb_abi_version() != 3:
        raise ImportError("rrt_b200: ABI version mismatch")
    _lib = lib
    return lib
