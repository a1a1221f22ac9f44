"""ctypes mirror of include/wrt_scene.h, include/wrt_host.h and include/wrt_cuda.h.

The shared libraries are built in-tree by `__graft_entry__.build()`:
  libwrt_host.so  host front-end (parser, OBJ reader, BVH build, flatten, PPM writer)
  libwrt_cuda.so  sm_100a render core
There is no CPU fallback: if libwrt_cuda.so is missing, `load_cuda()` raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
HOST_LIB = PKG / "libwrt_host.so"
CUDA_LIB = PKG / "libwrt_cuda.so"

WRT_MAX_DEPTH = 9
WRT_SOFT_SAMPLES = 50
WRT_DEFAULT_SEED = 0x5EED
WRT_REQ_SHAFT_CULL = 1          # wrt_shadow_requests_wavefront: answer soft requests with an empty shaft by the shaft test


class WrtNode(C.Structure):
    _fields_ = [("pmin", C.c_float * 3), ("link", C.c_int32), ("pmax", C.c_float * 3), ("pad", C.c_int32)]


class WrtMaterial(C.Structure):
    _fields_ = [("diffuse", C.c_float * 3), ("specular", C.c_float * 3), ("ka", C.c_float), ("kd", C.c_float),
                ("ks", C.c_float), ("n", C.c_float), ("alpha", C.c_float), ("eta", C.c_float)]


class WrtLight(C.Structure):
    _fields_ = [("pos", C.c_float * 4), ("color", C.c_float * 3), ("c1", C.c_float), ("c2", C.c_float),
                ("c3", C.c_float), ("tri", C.c_float * 9), ("pad", C.c_float)]


class WrtTexture(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("offset", C.c_int64), ("count", C.c_int64)]


class WrtSceneDesc(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_int32), ("n_prims", C.c_int32), ("n_materials", C.c_int32), ("n_lights", C.c_int32),
        ("n_textures", C.c_int32), ("n_normalmaps", C.c_int32), ("n_texels", C.c_int64),
        ("nodes", C.POINTER(WrtNode)), ("prim_geom", C.POINTER(C.c_float)), ("prim_flags", C.POINTER(C.c_uint32)),
        ("prim_material", C.POINTER(C.c_int32)), ("prim_texture", C.POINTER(C.c_int32)),
        ("prim_normalmap", C.POINTER(C.c_int32)), ("prim_object", C.POINTER(C.c_int32)),
        ("object_prim", C.POINTER(C.c_int32)), ("prim_normals", C.POINTER(C.c_float)),
        ("prim_uv", C.POINTER(C.c_float)), ("materials", C.POINTER(WrtMaterial)), ("lights", C.POINTER(WrtLight)),
        ("textures", C.POINTER(WrtTexture)), ("normalmaps", C.POINTER(WrtTexture)), ("texels", C.POINTER(C.c_float)),
        ("bkgcolor", C.c_float * 3), ("eta", C.c_float), ("shadow_type", C.c_int32), ("depth_cueing", C.c_int32),
        ("dc", C.c_float * 3), ("amin", C.c_float), ("amax", C.c_float), ("distmin", C.c_float),
        ("distmax", C.c_float), ("eye", C.c_float * 3),
    ]


class WrtCamera(C.Structure):
    _fields_ = [("eye", C.c_float * 3), ("ul", C.c_float * 3), ("delta_h", C.c_float * 3),
                ("delta_v", C.c_float * 3), ("c_off_h", C.c_float * 3), ("c_off_v", C.c_float * 3),
                ("n", C.c_float * 3), ("d", C.c_float), ("parallel", C.c_int32), ("width", C.c_int32),
                ("height", C.c_int32)]


class WrtHit(C.Structure):
    _fields_ = [("hit", C.c_int32), ("object", C.c_int32), ("t", C.c_float), ("pos", C.c_float * 3),
                ("ndir", C.c_float * 3), ("uv", C.c_float * 2), ("texture", C.c_int32), ("normalmap", C.c_int32),
                ("material", C.c_int32), ("prim", C.c_int32)]


class WrtGBuffer(C.Structure):
    _fields_ = [("hit", C.c_void_p), ("normal", C.c_void_p), ("albedo", C.c_void_p), ("shadow", C.c_void_p)]


class WrtStats(C.Structure):
    _fields_ = [("closest_rays", C.c_int64), ("shadow_rays", C.c_int64), ("rays_per_depth", C.c_int64 * 9),
                ("shadow_requests", C.c_int64), ("box_tests", C.c_int64), ("prim_tests", C.c_int64),
                ("overflow_retries", C.c_int32), ("pad", C.c_int32), ("gpu_ms", C.c_float), ("pad2", C.c_float),
                ("shaft_culled_requests", C.c_int64), ("unlit_skipped_requests", C.c_int64),
                ("shadow_rays_traced", C.c_int64)]


# numpy view of WrtHit (same layout, 60 bytes)
HIT_DTYPE = [("hit", "<i4"), ("object", "<i4"), ("t", "<f4"), ("pos", "<f4", 3), ("ndir", "<f4", 3),
             ("uv", "<f4", 2), ("texture", "<i4"), ("normalmap", "<i4"), ("material", "<i4"), ("prim", "<i4")]

# Entry points include/wrt_host.h declares (checked by tests/test_cabi_symbols.py)
HOST_SYMBOLS = [
    "wrt_scene_load", "wrt_scene_load_text", "wrt_scene_free", "wrt_scene_desc", "wrt_scene_camera",
    "wrt_scene_set_imsize", "wrt_scene_set_shadow_type", "wrt_scene_bvh_depth", "wrt_scene_upload_bytes",
    "wrt_scene_output_name", "wrt_write_ppm_p3", "wrt_host_last_error", "wrt_tile_slot_count", "wrt_tile_pixel_map",
    "wrt_scatter_tiles_host",
]
# Entry points include/wrt_cuda.h declares
CUDA_SYMBOLS = [
    "wrt_create", "wrt_destroy", "wrt_last_error", "wrt_upload_scene", "wrt_set_camera", "wrt_set_tiles",
    "wrt_set_options", "wrt_enable_kernel_timing", "wrt_trace_closest", "wrt_trace_closest_wavefront", "wrt_shadow_requests_wavefront",
    "wrt_shadow_hard", "wrt_shadow_soft", "wrt_shadow_directional",
    "wrt_render", "wrt_render_float", "wrt_render_gbuffer", "wrt_render_gbuffer_device", "wrt_render_device", "wrt_finish_device", "wrt_get_stats", "wrt_tile_pixel_count",
    "wrt_scatter_tiles", "wrt_kernel_launch_count", "wrt_get_kernel_times", "wrt_get_kernel_launches", "wrt_measure_fp32_peak",
    "wrt_multi_create", "wrt_multi_destroy", "wrt_multi_device_count", "wrt_multi_context", "wrt_multi_uses_peer_stores",
    "wrt_multi_upload_scene", "wrt_multi_set_camera", "wrt_multi_set_options", "wrt_multi_render",
]

_host = None
_cuda = None


def load_host() -> C.CDLL:
    global _host
    if _host is None:
        if not HOST_LIB.exists():
            raise RuntimeError(f"{HOST_LIB} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
        lib = C.CDLL(str(HOST_LIB))
        vp, cp, i32 = C.c_void_p, C.c_char_p, C.c_int
        lib.wrt_scene_load.argtypes = [cp, cp, cp, i32, C.POINTER(vp)]
        lib.wrt_scene_load_text.argtypes = [cp, cp, cp, i32, C.POINTER(vp)]
        lib.wrt_scene_free.argtypes = [vp]
        lib.wrt_scene_free.restype = None
        lib.wrt_scene_desc.argtypes = [vp]
        lib.wrt_scene_desc.restype = C.POINTER(WrtSceneDesc)
        lib.wrt_scene_camera.argtypes = [vp]
        lib.wrt_scene_camera.restype = C.POINTER(WrtCamera)
        lib.wrt_scene_set_imsize.argtypes = [vp, i32, i32]
        lib.wrt_scene_set_shadow_type.argtypes = [vp, i32]
        lib.wrt_scene_bvh_depth.argtypes = [vp]
        lib.wrt_scene_upload_bytes.argtypes = [vp]
        lib.wrt_scene_upload_bytes.restype = C.c_int64
        lib.wrt_scene_output_name.argtypes = [vp]
        lib.wrt_scene_output_name.restype = cp
        lib.wrt_write_ppm_p3.argtypes = [cp, i32, i32, vp]
        lib.wrt_host_last_error.restype = cp
        lib.wrt_tile_slot_count.argtypes = [i32] * 6
        lib.wrt_tile_slot_count.restype = C.c_int64
        lib.wrt_tile_pixel_map.argtypes = [i32] * 6 + [vp, C.c_int64]
        lib.wrt_scatter_tiles_host.argtypes = [i32] * 5 + [vp, C.c_int64, vp]
        _host = lib
    return _host


def load_cuda() -> C.CDLL:
    """Loads the CUDA render core.  Raises when it is not built — there is no fallback."""
    global _cuda
    if _cuda is None:
        import os
        lib_path = Path(os.environ.get("WRT_CUDA_LIB", CUDA_LIB))      # A/B builds during development
        if not lib_path.exists():
            raise RuntimeError(
                f"{CUDA_LIB} is not built (nvcc -gencode arch=compute_100a,code=sm_100a); "
                "this package has no CPU fallback — run __graft_entry__.build()")
        lib = C.CDLL(str(lib_path))
        vp, i32, i64, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32
        lib.wrt_create.argtypes = [i32, C.POINTER(vp)]
        lib.wrt_destroy.argtypes = [vp]
        lib.wrt_destroy.restype = None
        lib.wrt_last_error.restype = C.c_char_p
        lib.wrt_upload_scene.argtypes = [vp, C.POINTER(WrtSceneDesc)]
        lib.wrt_set_camera.argtypes = [vp, C.POINTER(WrtCamera)]
        lib.wrt_set_tiles.argtypes = [vp, i32, i32, i32, i32]
        lib.wrt_set_options.argtypes = [vp, i32, u32, C.c_float]
        lib.wrt_trace_closest.argtypes = [vp, vp, vp, i64, vp]
        lib.wrt_trace_closest_wavefront.argtypes = [vp, vp, vp, i64, vp]
        lib.wrt_shadow_requests_wavefront.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
        lib.wrt_shadow_hard.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.wrt_shadow_soft.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.wrt_shadow_directional.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.wrt_render.argtypes = [vp, vp, C.POINTER(WrtStats)]
        lib.wrt_render_float.argtypes = [vp, vp, vp, C.POINTER(WrtStats)]
        lib.wrt_render_gbuffer.argtypes = [vp, C.POINTER(WrtGBuffer), vp, C.POINTER(WrtStats)]
        lib.wrt_render_gbuffer_device.argtypes = [vp, C.POINTER(WrtGBuffer), vp, vp, vp]
        lib.wrt_render_device.argtypes = [vp, vp, vp]
        lib.wrt_finish_device.argtypes = [vp, C.POINTER(WrtStats)]
        lib.wrt_get_stats.argtypes = [vp, C.POINTER(WrtStats)]
        lib.wrt_tile_pixel_count.argtypes = [vp, i32, i32]
        lib.wrt_tile_pixel_count.restype = i64
        lib.wrt_scatter_tiles.argtypes = [vp, vp, i32, i64, vp, vp]
        lib.wrt_enable_kernel_timing.argtypes = [vp, i32]
        lib.wrt_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        lib.wrt_kernel_launch_count.argtypes = [vp]
        lib.wrt_kernel_launch_count.restype = i64
        lib.wrt_get_kernel_times.argtypes = [vp, vp, i32]
        lib.wrt_get_kernel_launches.argtypes = [vp, vp, i32]
        lib.wrt_multi_create.argtypes = [C.POINTER(C.c_int), i32, C.POINTER(vp)]
        lib.wrt_multi_destroy.argtypes = [vp]
        lib.wrt_multi_destroy.restype = None
        lib.wrt_multi_device_count.argtypes = [vp]
        lib.wrt_multi_context.argtypes = [vp, i32]
        lib.wrt_multi_context.restype = vp
        lib.wrt_multi_uses_peer_stores.argtypes = [vp]
        lib.wrt_multi_upload_scene.argtypes = [vp, C.POINTER(WrtSceneDesc)]
        lib.wrt_multi_set_camera.argtypes = [vp, C.POINTER(WrtCamera)]
        lib.wrt_multi_set_options.argtypes = [vp, i32, u32, C.c_float]
        lib.wrt_multi_render.argtypes = [vp, vp, C.POINTER(WrtStats)]
        _cuda = lib
    return _cuda
