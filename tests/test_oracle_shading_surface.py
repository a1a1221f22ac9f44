"""The shaded surface per hit record that the frame's surface planes (wrt_render_gbuffer) are held to in
tests/test_gpu_gbuffer.py: orc_shading_surface (tests/shading_surface_oracle.c, compiled here together with the oracle)
returns Od and the shading normal traceRay's shader uses at a record orc_trace_closest returns.  Checked against those
records: without texture or normal map the shading normal is the record's nDir and Od the material's diffuse colour, bit
for bit; a texel or a bumped normal is used exactly where the record carries a texture or normal map with valid uv;
misses and light avatars are not shaded (0)."""
import ctypes as C
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import load_golden_scene
from whittedstyle_raytracer_b200 import cabi

WRT_PRIM_LIGHT = 2              # include/wrt_scene.h: Object::isLight
SRC = Path(__file__).resolve().parent / "shading_surface_oracle.c"
_libs = {}


def _surface_lib(device_math):
    """The oracle with orc_shading_surface, built into a temporary directory with the oracle's own flags
    (__graft_entry__.build_oracle): -DORC_DEVICE_MATH for the build whose powf / acosf / atan2f are the device's."""
    if device_math not in _libs:
        out = Path(tempfile.mkdtemp(prefix="wrt_surface_oracle_")) / "liboracle_surface.so"
        gcc = "/usr/bin/gcc" if Path("/usr/bin/gcc").exists() else (shutil.which("gcc") or "gcc")
        base = [gcc, "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall",
                "-Wno-unknown-pragmas", *(["-DORC_DEVICE_MATH"] if device_math else []), "-shared", "-o", str(out),
                str(SRC), "-lm"]
        try:
            subprocess.run(base[:1] + ["-fopenmp"] + base[1:], check=True)
        except subprocess.CalledProcessError:
            subprocess.run(base, check=True)
        lib = C.CDLL(str(out))
        lib.orc_shading_surface.argtypes = [C.POINTER(cabi.WrtSceneDesc), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        lib.orc_shading_surface.restype = None
        _libs[device_math] = lib
    return _libs[device_math]


def shading_surface(scene, hits, device_math):
    """(shading normal, Od) of each hit record, (N, 3) float32 each."""
    hits = np.ascontiguousarray(hits, dtype=cabi.HIT_DTYPE)
    nd = np.zeros((len(hits), 3), np.float32)
    od = np.zeros((len(hits), 3), np.float32)
    _surface_lib(device_math).orc_shading_surface(scene.desc_ptr, hits.ctypes.data, len(hits), nd.ctypes.data,
                                                  od.ctypes.data)
    return nd, od


def scene_arrays(scene):
    """Per-primitive flags and per-material diffuse colour / Phong exponent of a Scene's description."""
    d = scene.desc
    flags = np.ctypeslib.as_array(d.prim_flags, (max(d.n_prims, 1),))[:d.n_prims].copy()
    mats = [d.materials[i] for i in range(d.n_materials)]
    diffuse = np.array([list(m.diffuse) for m in mats], np.float32).reshape(-1, 3)
    n_exp = np.array([m.n for m in mats], np.float32)
    return flags, diffuse, n_exp


def shaded_mask(scene, hits):
    """Hits the shader runs on: not a miss, not a light avatar."""
    flags, _, _ = scene_arrays(scene)
    if not len(flags):
        return np.zeros(len(hits), bool)
    return (hits["hit"] != 0) & ((flags[np.maximum(hits["prim"], 0)] & WRT_PRIM_LIGHT) == 0)


@pytest.mark.parametrize("name", ["parallel", "directional", "water_small", "spheres", "bump"])
def test_shading_surface_against_trace_closest(workdir, name):
    scene, _ = load_golden_scene(workdir, name)
    _, diffuse, _ = scene_arrays(scene)
    for device_math in (False, True):
        orc = ob.OracleScene(scene, device_math=device_math)
        o, d = orc.primary_rays()
        hits = orc.trace_closest(o, d)
        nd, od = shading_surface(scene, hits, device_math)
        shaded = shaded_mask(scene, hits)
        assert shaded.any() and (~shaded).any(), name
        assert not nd[~shaded].any() and not od[~shaded].any(), "unshaded records must read 0"
        texel = shaded & (hits["texture"] != -1) & (hits["uv"][:, 0] != -1) & (hits["uv"][:, 1] != -1)
        bumped = shaded & (hits["normalmap"] != -1)
        if scene.desc.n_textures == 0 and scene.desc.n_normalmaps == 0:
            assert not texel.any() and not bumped.any()
        else:
            assert texel.any(), f"{name}: no textured hit"
        plain_n, plain_d = shaded & ~bumped, shaded & ~texel
        assert np.array_equal(nd[plain_n].view(np.uint32), hits["ndir"][plain_n].view(np.uint32)), name
        assert np.array_equal(od[plain_d].view(np.uint32), diffuse[hits["material"][plain_d]].view(np.uint32)), name
        if texel.any():                                # a texel really replaces the diffuse colour somewhere
            assert not np.array_equal(od[texel], diffuse[hits["material"][texel]])
        if bumped.any():                               # a normal map really changes the normal
            assert not np.array_equal(nd[bumped], hits["ndir"][bumped])
            assert np.allclose(np.linalg.norm(nd[bumped], axis=1), 1, atol=1e-5)
