"""Python host-side mirror of the reference's render interface, over the C ABI.

`CudaStrategy` is the batch form of the reference's IIntersectStrategy plugin
point (include/IIntersectStrategy.h:7-15): `UpdateInter` / `getShadowCoeffi`
keep their names and argument meaning but take N rays at once.
`Renderer.render()` replaces Renderer::render() (include/Renderer.hpp:57-137).
Everything here calls libwrt_cuda.so; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import cabi
from .scene import Scene

TRAVERSAL_EXHAUSTIVE = 0
TRAVERSAL_PRUNED = 1

KERNEL_FAMILIES = ["raygen", "trace_closest", "surface", "shadow_hard", "shadow_soft", "shadow_directional",
                   "shade", "combine", "resolve", "soft_lists", "soft_filter"]


class CudaError(RuntimeError):
    pass


def _f32(a, cols):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != cols:
        raise ValueError(f"expected an (N, {cols}) float array, got {a.shape}")
    return a


def stats_dict(st: cabi.WrtStats) -> dict:
    return {
        "closest_rays": int(st.closest_rays), "shadow_rays": int(st.shadow_rays),
        "rays": int(st.closest_rays + st.shadow_rays),
        "rays_per_depth": [int(x) for x in st.rays_per_depth],
        "shadow_requests": int(st.shadow_requests), "overflow_retries": int(st.overflow_retries),
        "gpu_ms": float(st.gpu_ms),
        # shadow requests answered without tracing (include/wrt_scene.h); shadow_rays keeps the reference's count
        "shaft_culled_requests": int(st.shaft_culled_requests),
        "unlit_skipped_requests": int(st.unlit_skipped_requests),
        "shadow_rays_traced": int(st.shadow_rays_traced),
    }


class Context:
    """One GPU's render core (wrt_create / wrt_destroy)."""

    def __init__(self, device: int = 0):
        self.lib = cabi.load_cuda()
        self.h = C.c_void_p()
        self._check(self.lib.wrt_create(device, C.byref(self.h)))
        self.scene = None

    def _check(self, rc):
        if rc != 0:
            raise CudaError(self.lib.wrt_last_error().decode(errors="replace"))

    def close(self):
        if getattr(self, "h", None):
            self.lib.wrt_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload_scene(self, scene: Scene):
        self._check(self.lib.wrt_upload_scene(self.h, scene.desc_ptr))
        self._check(self.lib.wrt_set_camera(self.h, scene.camera_ptr))
        self.scene = scene

    def set_camera(self, scene: Scene):
        self._check(self.lib.wrt_set_camera(self.h, scene.camera_ptr))

    def set_tiles(self, tile_w=8, tile_h=4, rank=0, world=1):
        self._check(self.lib.wrt_set_tiles(self.h, tile_w, tile_h, rank, world))

    def set_options(self, traversal=TRAVERSAL_PRUNED, seed=cabi.WRT_DEFAULT_SEED, queue_factor=0.0):
        self._check(self.lib.wrt_set_options(self.h, traversal, seed, queue_factor))

    def enable_kernel_timing(self, on=True):
        self._check(self.lib.wrt_enable_kernel_timing(self.h, 1 if on else 0))

    @property
    def launches(self) -> int:
        return int(self.lib.wrt_kernel_launch_count(self.h))

    def kernel_times(self) -> dict:
        ms = (C.c_float * len(KERNEL_FAMILIES))()
        n = self.lib.wrt_get_kernel_times(self.h, ms, len(KERNEL_FAMILIES))
        return {KERNEL_FAMILIES[i]: float(ms[i]) for i in range(n)}

    def kernel_launches(self) -> dict:
        n = (C.c_int32 * len(KERNEL_FAMILIES))()
        k = self.lib.wrt_get_kernel_launches(self.h, n, len(KERNEL_FAMILIES))
        return {KERNEL_FAMILIES[i]: int(n[i]) for i in range(k)}

    def measure_fp32_peak(self) -> tuple[float, float]:
        """(TFLOP/s with FFMA, TFLOP/s with separate FMUL+FADD) measured on this GPU."""
        a, b = C.c_float(0), C.c_float(0)
        self._check(self.lib.wrt_measure_fp32_peak(self.h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def tile_pixel_count(self, rank, world) -> int:
        return int(self.lib.wrt_tile_pixel_count(self.h, rank, world))


class CudaStrategy:
    """Batch IIntersectStrategy on the GPU (beside the reference's BaseInterStrategy / BVHStrategy)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def UpdateInter(self, rayOrig, rayDir) -> np.ndarray:
        """Closest hit per ray -> structured array with the fields of Intersection."""
        o, d = _f32(rayOrig, 3), _f32(rayDir, 3)
        out = np.zeros(len(o), dtype=cabi.HIT_DTYPE)
        self.ctx._check(self.ctx.lib.wrt_trace_closest(self.ctx.h, o.ctypes.data, d.ctypes.data, len(o), out.ctypes.data))
        return out

    def UpdateInterWavefront(self, rayOrig, rayDir) -> np.ndarray:
        """UpdateInter answered by the frame's own deep-level closest-hit kernel (wrt_trace_closest_wavefront)."""
        o, d = _f32(rayOrig, 3), _f32(rayDir, 3)
        out = np.zeros(len(o), dtype=cabi.HIT_DTYPE)
        self.ctx._check(self.ctx.lib.wrt_trace_closest_wavefront(self.ctx.h, o.ctypes.data, d.ctypes.data, len(o), out.ctypes.data))
        return out

    def shadowRequestsWavefront(self, pos, nDir, light, pixel, path, self_object, queue=0, flags=0) -> np.ndarray:
        """Test entry: shadow requests (point, normal, scene light index) answered by the frame's own shadow kernels of
        request queue `queue` (wrt_shadow_requests_wavefront).  Per request what the frame stores: the hard-shadow
        coefficient, the lit samples of 50 for soft shadows (RNG keyed on pixel and path), the directional product
        (self_object: the point's object).  flags: cabi.WRT_REQ_SHAFT_CULL answers empty soft shafts by the shaft test."""
        p, n = _f32(pos, 3), _f32(nDir, 3)
        li = np.ascontiguousarray(light, dtype=np.int32)
        px, pa = np.ascontiguousarray(pixel, dtype=np.uint32), np.ascontiguousarray(path, dtype=np.uint32)
        so = np.ascontiguousarray(self_object, dtype=np.int32)
        if not (len(p) == len(n) == len(li) == len(px) == len(pa) == len(so)):
            raise ValueError("shadowRequestsWavefront: arrays of different lengths")
        out = np.zeros(len(p), dtype=np.float32)
        self.ctx._check(self.ctx.lib.wrt_shadow_requests_wavefront(
            self.ctx.h, queue, flags, p.ctypes.data, n.ctypes.data, li.ctypes.data, px.ctypes.data, pa.ctypes.data,
            so.ctypes.data, len(p), out.ctypes.data))
        return out

    def getShadowCoeffi(self, pos, nDir, lightpos) -> np.ndarray:
        """Hard-shadow coefficient per (hit point, shading normal, light position)."""
        return self._shadow(self.ctx.lib.wrt_shadow_hard, pos, nDir, lightpos)

    def getSoftShadowSample(self, pos, nDir, lightpos) -> np.ndarray:
        """One soft-shadow visibility sample (0 occluded / 1 visible), Renderer.hpp:347-376."""
        return self._shadow(self.ctx.lib.wrt_shadow_soft, pos, nDir, lightpos)

    def getDirectionalShadowCoeffi(self, pos, self_object, lightDir4) -> np.ndarray:
        p, l = _f32(pos, 3), _f32(lightDir4, 4)
        so = np.ascontiguousarray(self_object, dtype=np.int32)
        out = np.zeros(len(p), dtype=np.float32)
        self.ctx._check(self.ctx.lib.wrt_shadow_directional(self.ctx.h, p.ctypes.data, so.ctypes.data, l.ctypes.data,
                                                            len(p), out.ctypes.data))
        return out

    def _shadow(self, fn, pos, nDir, lightpos):
        p, n, l = _f32(pos, 3), _f32(nDir, 3), _f32(lightpos, 3)
        out = np.zeros(len(p), dtype=np.float32)
        self.ctx._check(fn(self.ctx.h, p.ctypes.data, n.ctypes.data, l.ctypes.data, len(p), out.ctypes.data))
        return out


class Renderer:
    """Renderer(PPMGenerator*) -> render(): here Renderer(Scene) -> render() -> (H, W, 3) uint8."""

    def __init__(self, scene: Scene, device: int = 0, ctx: Context | None = None):
        self.ctx = ctx or Context(device)
        self.ctx.upload_scene(scene)
        self.scene = scene
        self.interStrategy = CudaStrategy(self.ctx)
        self.last_stats: dict = {}

    def render(self, out: np.ndarray | None = None) -> np.ndarray:
        cam = self.scene.camera
        if out is None:
            out = np.zeros((cam.height, cam.width, 3), np.uint8)
        st = cabi.WrtStats()
        self.ctx._check(self.ctx.lib.wrt_render(self.ctx.h, out.ctypes.data, C.byref(st)))
        self.last_stats = stats_dict(st)
        return out

    def render_float(self, out_f: np.ndarray | None = None, out: np.ndarray | None = None) -> tuple[np.ndarray, np.ndarray]:
        """The frame render() renders, with its unquantised colour: ((H, W, 3) float32, (H, W, 3) uint8).  The float image
        is what the 8-bit one quantises as int(255 * min(c, 1)), clamped to [0, 255]; with tiles only this rank's pixels
        are written."""
        cam = self.scene.camera
        if out_f is None:
            out_f = np.zeros((cam.height, cam.width, 3), np.float32)
        if out is None:
            out = np.zeros((cam.height, cam.width, 3), np.uint8)
        if out_f.dtype != np.float32 or out_f.shape != (cam.height, cam.width, 3) or not out_f.flags.c_contiguous:
            raise ValueError("render_float: out_f must be a C-contiguous (H, W, 3) float32 array")
        st = cabi.WrtStats()
        self.ctx._check(self.ctx.lib.wrt_render_float(self.ctx.h, out_f.ctypes.data, out.ctypes.data, C.byref(st)))
        self.last_stats = stats_dict(st)
        return out_f, out

    def render_device(self, d_ptr: int, stream: int | None = None):
        """Asynchronous render of this rank's tiles into device memory (tile order)."""
        self.ctx._check(self.ctx.lib.wrt_render_device(self.ctx.h, d_ptr, stream))

    def finish_device(self) -> dict:
        st = cabi.WrtStats()
        self.ctx._check(self.ctx.lib.wrt_finish_device(self.ctx.h, C.byref(st)))
        self.last_stats = stats_dict(st)
        return self.last_stats

    def scatter_tiles(self, d_gathered: int, world: int, stride_bytes: int, d_image: int, stream: int | None = None):
        self.ctx._check(self.ctx.lib.wrt_scatter_tiles(self.ctx.h, d_gathered, world, stride_bytes, d_image, stream))


class MultiRenderer:
    """Renderer over several GPUs of one process (wrt_multi_*): scene replicated, interleaved tiles, every GPU's
    resolve kernel stores its pixels into GPU devices[0]'s frame over NVLink.  render() -> (H, W, 3) uint8, identical to
    the single-GPU image."""

    def __init__(self, scene: Scene, devices):
        self.lib = cabi.load_cuda()
        self.h = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        self._check(self.lib.wrt_multi_create(devs, len(devices), C.byref(self.h)))
        self.scene = scene
        self._check(self.lib.wrt_multi_upload_scene(self.h, scene.desc_ptr))
        self._check(self.lib.wrt_multi_set_camera(self.h, scene.camera_ptr))
        self.last_stats: dict = {}

    def _check(self, rc):
        if rc != 0:
            raise CudaError(self.lib.wrt_last_error().decode(errors="replace"))

    @property
    def uses_peer_stores(self) -> bool:
        return bool(self.lib.wrt_multi_uses_peer_stores(self.h))

    def set_options(self, traversal=TRAVERSAL_PRUNED, seed=cabi.WRT_DEFAULT_SEED, queue_factor=0.0):
        self._check(self.lib.wrt_multi_set_options(self.h, traversal, seed, queue_factor))

    def upload(self):
        self._check(self.lib.wrt_multi_upload_scene(self.h, self.scene.desc_ptr))
        self._check(self.lib.wrt_multi_set_camera(self.h, self.scene.camera_ptr))

    def render(self, out: np.ndarray | None = None) -> np.ndarray:
        cam = self.scene.camera
        if out is None:
            out = np.zeros((cam.height, cam.width, 3), np.uint8)
        st = cabi.WrtStats()
        ptr = out.ctypes.data if isinstance(out, np.ndarray) else int(out)
        self._check(self.lib.wrt_multi_render(self.h, ptr, C.byref(st)))
        self.last_stats = stats_dict(st)
        return out

    def close(self):
        if getattr(self, "h", None):
            self.lib.wrt_multi_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
