"""TEST INFRASTRUCTURE: ctypes bindings for the CPU oracle (oracle/liboracle.so)
and, when it was built in the container, the unmodified-reference harness
(oracle/_ref/libwhitted_ref.so).  Only tests/, smoke() and bench.py import this."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

from whittedstyle_raytracer_b200 import cabi

REPO = Path(__file__).resolve().parent.parent
ORACLE_LIB = REPO / "oracle" / "liboracle.so"
# the same source built with -DORC_DEVICE_MATH: powf / acosf / atan2f as the render core evaluates them
ORACLE_DEVMATH_LIB = REPO / "oracle" / "liboracle_devmath.so"
REF_LIB = REPO / "oracle" / "_ref" / "libwhitted_ref.so"
REF_EXE = REPO / "oracle" / "_ref" / "whitted_ref"

_orc = {}
_ref = None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def oracle(device_math=False):
    if device_math not in _orc:
        lib = C.CDLL(str(ORACLE_DEVMATH_LIB if device_math else ORACLE_LIB))
        vp, i64, u32, i32 = C.c_void_p, C.c_int64, C.c_uint32, C.c_int
        dp = C.POINTER(cabi.WrtSceneDesc)
        lib.orc_trace_closest.argtypes = [dp, vp, vp, i64, vp]
        lib.orc_shadow_hard.argtypes = [dp, vp, vp, vp, i64, vp]
        lib.orc_shadow_soft.argtypes = [dp, vp, vp, vp, i64, vp]
        lib.orc_shadow_directional.argtypes = [dp, vp, vp, vp, i64, vp]
        lib.orc_trace_ray.argtypes = [dp, vp, vp, vp, vp, i64, u32, vp]
        lib.orc_primary_rays.argtypes = [C.POINTER(cabi.WrtCamera), vp, vp]
        lib.orc_render.argtypes = [dp, C.POINTER(cabi.WrtCamera), u32, i32, i32, i32, i32, i32, vp, vp,
                                   C.POINTER(cabi.WrtStats)]
        lib.orc_render_rect.argtypes = [dp, C.POINTER(cabi.WrtCamera), u32, i32, i32, i32, i32, i32, i32, i32, vp, vp,
                                        C.POINTER(cabi.WrtStats)]
        lib.orc_light_sample_uv.argtypes = [u32, u32, u32, u32, u32, vp]
        lib.orc_shadow_requests.argtypes = [dp, u32, vp, vp, vp, vp, vp, vp, i64, vp]
        _orc[device_math] = lib
    return _orc[device_math]


def have_reference() -> bool:
    return REF_LIB.exists()


class OracleScene:
    """The oracle over a whittedstyle_raytracer_b200.Scene.  device_math=True: the liboracle_devmath.so build, whose
    powf / acosf / atan2f are the render core's (everything else is the same source)."""

    def __init__(self, scene, device_math=False):
        self.scene = scene
        self.lib = oracle(device_math)

    def trace_closest(self, orig, dirs):
        orig, dirs = _f32(orig), _f32(dirs)
        out = np.zeros(len(orig), dtype=cabi.HIT_DTYPE)
        self.lib.orc_trace_closest(self.scene.desc_ptr, orig.ctypes.data, dirs.ctypes.data, len(orig), out.ctypes.data)
        return out

    def _shadow(self, fn, pos, ndir, lightpos):
        pos, ndir, lightpos = _f32(pos), _f32(ndir), _f32(lightpos)
        out = np.zeros(len(pos), dtype=np.float32)
        fn(self.scene.desc_ptr, pos.ctypes.data, ndir.ctypes.data, lightpos.ctypes.data, len(pos), out.ctypes.data)
        return out

    def shadow_hard(self, pos, ndir, lightpos):
        return self._shadow(self.lib.orc_shadow_hard, pos, ndir, lightpos)

    def shadow_soft(self, pos, ndir, lightpos):
        return self._shadow(self.lib.orc_shadow_soft, pos, ndir, lightpos)

    def shadow_directional(self, pos, self_object, lightdir4):
        pos, lightdir4 = _f32(pos), _f32(lightdir4)
        so = np.ascontiguousarray(self_object, dtype=np.int32)
        out = np.zeros(len(pos), dtype=np.float32)
        self.lib.orc_shadow_directional(self.scene.desc_ptr, pos.ctypes.data, so.ctypes.data, lightdir4.ctypes.data,
                                        len(pos), out.ctypes.data)
        return out

    def shadow_requests(self, pos, ndir, light, pixel, path, self_object, seed=cabi.WRT_DEFAULT_SEED):
        """What a frame stores for each shadow request (point, normal, scene light): the hard-shadow coefficient, the number
        of lit soft-shadow samples of 50 (RNG keyed on pixel and path) or the directional product."""
        pos, ndir = _f32(pos), _f32(ndir)
        li = np.ascontiguousarray(light, dtype=np.int32)
        px, pa = np.ascontiguousarray(pixel, dtype=np.uint32), np.ascontiguousarray(path, dtype=np.uint32)
        so = np.ascontiguousarray(self_object, dtype=np.int32)
        assert len(pos) == len(ndir) == len(li) == len(px) == len(pa) == len(so)
        assert ((li >= 0) & (li < self.scene.desc.n_lights)).all()
        out = np.zeros(len(pos), dtype=np.float32)
        self.lib.orc_shadow_requests(self.scene.desc_ptr, seed, pos.ctypes.data, ndir.ctypes.data, li.ctypes.data,
                                     px.ctypes.data, pa.ctypes.data, so.ctypes.data, len(pos), out.ctypes.data)
        return out

    def trace_ray(self, orig, dirs, depth=None, pixel=None, seed=cabi.WRT_DEFAULT_SEED):
        orig, dirs = _f32(orig), _f32(dirs)
        out = np.zeros((len(orig), 3), dtype=np.float32)
        dp = None if depth is None else np.ascontiguousarray(depth, dtype=np.int32)
        pp = None if pixel is None else np.ascontiguousarray(pixel, dtype=np.uint32)
        self.lib.orc_trace_ray(self.scene.desc_ptr, orig.ctypes.data, dirs.ctypes.data,
                               None if dp is None else dp.ctypes.data, None if pp is None else pp.ctypes.data,
                               len(orig), seed, out.ctypes.data)
        return out

    def primary_rays(self):
        cam = self.scene.camera
        n = cam.width * cam.height
        o = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        self.lib.orc_primary_rays(self.scene.camera_ptr, o.ctypes.data, d.ctypes.data)
        return o, d

    def render(self, seed=cabi.WRT_DEFAULT_SEED, rows=None, stride=(1, 1), threads=0, want_float=False, cols=None):
        """Whole frame, or the rectangle rows x cols of it (the rest of the returned image stays 0)."""
        cam = self.scene.camera
        y0, y1 = rows if rows else (0, cam.height)
        x0, x1 = cols if cols else (0, cam.width)
        u8 = np.zeros((cam.height, cam.width, 3), np.uint8)
        fl = np.zeros((cam.height, cam.width, 3), np.float32) if want_float else None
        st = cabi.WrtStats()
        self.lib.orc_render_rect(self.scene.desc_ptr, self.scene.camera_ptr, seed, x0, x1, y0, y1, stride[0], stride[1],
                                 threads, u8.ctypes.data, None if fl is None else fl.ctypes.data, C.byref(st))
        return (u8, fl, st) if want_float else (u8, st)


def reference():
    global _ref
    if _ref is None:
        lib = C.CDLL(str(REF_LIB))
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
        lib.ref_scene_load.argtypes = [C.c_char_p, C.c_char_p, i32]
        lib.ref_scene_load.restype = vp
        for f in ("ref_num_objects", "ref_width", "ref_height"):
            getattr(lib, f).argtypes = [vp]
        lib.ref_set_imsize.argtypes = [vp, i32, i32]
        lib.ref_set_shadow_type.argtypes = [vp, i32]
        lib.ref_bvh_leaf_order.argtypes = [vp, vp, i32, vp]
        lib.ref_trace_closest.argtypes = [vp, vp, vp, i64, vp]
        lib.ref_shadow_hard.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.ref_shadow_soft.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.ref_shadow_directional.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.ref_trace_ray.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.ref_render.argtypes = [vp, vp]
        lib.ref_render.restype = C.c_double
        lib.ref_counters_reset.argtypes = [vp]
        lib.ref_counters_get.argtypes = [vp, vp, vp]
        lib.ref_trace_pixels.argtypes = [vp, vp, vp, i64, vp]
        lib.ref_trace_pixels.restype = C.c_double
        _ref = lib
    return _ref


class ReferenceScene:
    """The UNMODIFIED reference (headers compiled where they lie) on a config in `workdir`.
    The reference resolves textures against the cwd, so loading chdirs temporarily."""

    def __init__(self, workdir, name, *, bunny=True, glass=False):
        self.lib = reference()
        old = os.getcwd()
        os.chdir(workdir)
        try:
            self.h = self.lib.ref_scene_load(f"{name}.txt".encode(), b"bunny.obj" if bunny else b"", 1 if glass else 0)
        finally:
            os.chdir(old)

    @property
    def width(self):
        return self.lib.ref_width(self.h)

    @property
    def height(self):
        return self.lib.ref_height(self.h)

    def set_imsize(self, w, h):
        self.lib.ref_set_imsize(self.h, w, h)

    def leaf_order(self):
        n = self.lib.ref_num_objects(self.h)
        out = np.zeros(max(n, 1), np.int32)
        depth = C.c_int(0)
        k = self.lib.ref_bvh_leaf_order(self.h, out.ctypes.data, n, C.byref(depth))
        return out[:k].copy(), depth.value

    def trace_closest(self, orig, dirs):
        orig, dirs = _f32(orig), _f32(dirs)
        out = np.zeros(len(orig), dtype=cabi.HIT_DTYPE)
        self.lib.ref_trace_closest(self.h, orig.ctypes.data, dirs.ctypes.data, len(orig), out.ctypes.data)
        return out

    def _shadow(self, fn, pos, ndir, lightpos):
        pos, ndir, lightpos = _f32(pos), _f32(ndir), _f32(lightpos)
        out = np.zeros(len(pos), dtype=np.float32)
        fn(self.h, pos.ctypes.data, ndir.ctypes.data, lightpos.ctypes.data, len(pos), out.ctypes.data)
        return out

    def shadow_hard(self, pos, ndir, lightpos):
        return self._shadow(self.lib.ref_shadow_hard, pos, ndir, lightpos)

    def shadow_soft(self, pos, ndir, lightpos):
        return self._shadow(self.lib.ref_shadow_soft, pos, ndir, lightpos)

    def shadow_directional(self, pos, self_object, lightdir4):
        pos, lightdir4 = _f32(pos), _f32(lightdir4)
        so = np.ascontiguousarray(self_object, dtype=np.int32)
        out = np.zeros(len(pos), dtype=np.float32)
        self.lib.ref_shadow_directional(self.h, pos.ctypes.data, so.ctypes.data, lightdir4.ctypes.data, len(pos),
                                        out.ctypes.data)
        return out

    def trace_ray(self, orig, dirs, depth=None):
        orig, dirs = _f32(orig), _f32(dirs)
        out = np.zeros((len(orig), 3), dtype=np.float32)
        dp = None if depth is None else np.ascontiguousarray(depth, dtype=np.int32)
        self.lib.ref_trace_ray(self.h, orig.ctypes.data, dirs.ctypes.data, None if dp is None else dp.ctypes.data,
                               len(orig), out.ctypes.data)
        return out

    def render(self):
        out = np.zeros((self.height, self.width, 3), np.int32)
        secs = self.lib.ref_render(self.h, out.ctypes.data)
        return out, secs

    def counters(self, reset=False):
        a, b = C.c_int64(0), C.c_int64(0)
        self.lib.ref_counters_get(self.h, C.byref(a), C.byref(b))
        if reset:
            self.lib.ref_counters_reset(self.h)
        return a.value, b.value

    def trace_pixels(self, orig, dirs):
        orig, dirs = _f32(orig), _f32(dirs)
        out = np.zeros((len(orig), 3), np.int32)
        secs = self.lib.ref_trace_pixels(self.h, orig.ctypes.data, dirs.ctypes.data, len(orig), out.ctypes.data)
        return out, secs
