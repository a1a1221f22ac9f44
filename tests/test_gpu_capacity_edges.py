"""The render core at its fixed capacities, against the CPU oracle.

Every capacity below has a fall-back path for when it is exceeded; these scenes sit on both sides of each limit.
  * traversal-stack rows, max(reference depth, walked depth, 3 * ceil(walked depth / 2)) + 2 <= 90 (wrt_upload_scene):
    fans of triangles sharing a vertex, slivers and spheres of very mixed sizes make the device PLOC tree 45 .. 114
    levels deep; past the budget the walked tree is the host's binned-SAH tree instead (tests/test_ploc_build.py has the
    depths).  A 1500-segment fan over a floor (PLOC depth 58: 89 rows) is walked at the budget on the device tree itself.
  * WRT_SHADOW_HITS = 12 translucent blockers on one hard-shadow ray: up to 12 the product has the reference tree's
    association, bit for bit; beyond, it is multiplied in visit order, which may differ from the reference in the last
    bits: the bar there is a non-zero coefficient within k ulp of the oracle for k blockers.
  * WRT_DIR_HITS = 8 translucent hits on one directional-shadow ray: beyond, the literal O(N) loop; bit-exact either way.
  * WRT_LIST_CAP = 192 candidates per soft-shadow shaft: beyond, the per-ray walk; a build with a cap of 4 takes that
    path on almost every request and must render the same bytes.
Batch queries are compared bit for bit in both traversal modes; frames must be >= 99.99 % identical to the oracle and
within 1 LSB everywhere, with the oracle's ray counts.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import REPO, image_diff, ulp_diff
from whittedstyle_raytracer_b200 import Renderer, Scene, fixtures
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED

pytestmark = pytest.mark.gpu

MODES = (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE)

LIGHTS = {
    "hard": "light 2 8 3 1 1 1 1\n",
    "soft": "light 2 8 3 1 1 1 1\nshadow soft\n",
    "directional": "light 0.3 -1 -0.4 0 0.9 0.9 0.8\nlight 2 8 3 1 0.5 0.5 0.5\n",
}
# (geometry, material): translucent meshes (shadow rays cross one to four surfaces); opaque spheres, whose nesting would
# put more than WRT_SHADOW_HITS translucent shells on a shadow ray
DEEP = {
    "fan_1000": "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 0.6 1.2",
    "fan_2000": "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 0.6 1.2",
    "cylinder_2000": "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 0.6 1.2",
    "slivers_4000": "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 0.6 1.2",
    "mixed_radii_5000": "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1",
    "chain_30": "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1",
}
# PLOC trees that need more than 90 stack rows (host SAH instead); fan_1000 (71 rows) and chain_30 (47) keep theirs
FALLBACK = {"fan_2000", "cylinder_2000", "slivers_4000", "mixed_radii_5000"}


def _with_floor(body, y=-1.2):
    """Appends a floor quad after `body` (whose vertices come first: the faces index them from 1)."""
    nv = sum(1 for line in body.splitlines() if line.startswith("v "))
    return (body + "mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.1 10 1 1\n"
            + "".join(f"v {x} {y} {z}\n" for x, z in ((-20, 20), (20, 20), (20, -20), (-20, -20)))
            + f"f {nv + 1} {nv + 2} {nv + 3}\nf {nv + 1} {nv + 3} {nv + 4}\n")


def deep_scene(workdir, geometry, lights, body=None):
    text = ("imsize 160 120\neye 0.4 2.6 3.4\nviewdir -0.1 -0.6 -0.8\nhfov 60\nupdir 0 1 0\nbkgcolor 0.2 0.3 0.5 1\n"
            + LIGHTS[lights] + DEEP.get(geometry, DEEP["fan_1000"]) + "\n"
            + _with_floor(body if body is not None else fixtures.DEEP_TREE_GEOMETRY[geometry]()))
    return Scene(text=text, asset_dir=workdir)


def upload_verbose(scene, monkeypatch, capfd):
    """Renderer(scene) with the upload's WRT_VERBOSE line (C-level stderr) returned."""
    monkeypatch.setenv("WRT_VERBOSE", "1")
    capfd.readouterr()
    r = Renderer(scene)
    monkeypatch.delenv("WRT_VERBOSE")
    line = [ln for ln in capfd.readouterr().err.splitlines() if "[wrt] upload:" in ln]
    assert len(line) == 1, line
    return r, line[0]


def check_frames(r, scene, orc=None):
    """Both traversal modes: frame vs the oracle's, with its ray counts."""
    orc = orc or ob.OracleScene(scene)
    ref, ost = orc.render()
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        img = r.render()
        st = r.last_stats
        d = image_diff(img, ref)
        assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, (traversal, d)
        assert st["closest_rays"] == ost.closest_rays and st["shadow_rays"] == ost.shadow_rays, traversal
        assert st["rays_per_depth"] == [int(x) for x in ost.rays_per_depth], traversal
    r.ctx.set_options(traversal=TRAVERSAL_PRUNED)
    return ref


def check_closest(r, orc, o, d):
    ref = orc.trace_closest(o, d)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        for query in (r.interStrategy.UpdateInter, r.interStrategy.UpdateInterWavefront):
            h = query(o, d)
            for f in ("hit", "object", "prim"):
                assert np.array_equal(h[f], ref[f]), (f, traversal, query.__name__, int((h[f] != ref[f]).sum()))
            for f in ("t", "pos", "ndir"):
                assert np.array_equal(h[f].view(np.int32), ref[f].view(np.int32)), (f, traversal, query.__name__)
    r.ctx.set_options(traversal=TRAVERSAL_PRUNED)
    return ref


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def deep_rays(scene, rng, n=100_000):
    """Uniform rays through the scene's box (clipped to +-300), axis-parallel ones, and a quarter aimed at (0, 0, 0) —
    the vertex every fan and sliver triangle shares, where hundreds of triangles tie in t."""
    box = scene.nodes()[0]
    lo, hi = np.maximum(box[0:3], -300), np.minimum(box[4:7], 300)
    pad = 0.1 * (hi - lo) + 0.1
    o = rng.uniform(lo - pad, hi + pad, (n, 3))
    d = _unit(rng.normal(size=(n, 3)))
    d[: n // 50] = np.eye(3)[rng.integers(0, 3, n // 50)] * rng.choice([1.0, -1.0], (n // 50, 1))
    k = n // 4
    o[-k:] = _unit(rng.normal(size=(k, 3))) * rng.uniform(0.05, 3.0, (k, 1))
    d[-k:] = -o[-k:] / np.linalg.norm(o[-k:], axis=1, keepdims=True)
    return o.astype(np.float32), d.astype(np.float32)


@pytest.mark.parametrize("geometry", sorted(DEEP))
def test_deep_tree_batch_queries(workdir, monkeypatch, capfd, geometry):
    """Closest hit (batch kernel and the frame's deep-level kernel), hard, soft and directional shadows on ~1e5 rays
    through the scenes with very deep PLOC trees: the upload succeeds, on the host's SAH tree when PLOC's needs more
    than 90 stack rows, and every answer equals the oracle's bit for bit."""
    scene = deep_scene(workdir, geometry, "hard")
    r, line = upload_verbose(scene, monkeypatch, capfd)
    assert ("host SAH: the" in line) == (geometry in FALLBACK) and ("device PLOC" in line) == (geometry not in FALLBACK), line
    rows = int(re.search(r"(\d+) stack rows", line).group(1))
    assert rows <= 90, line
    orc = ob.OracleScene(scene)
    rng = np.random.default_rng(sorted(DEEP).index(geometry))
    o, d = deep_rays(scene, rng)
    ref = check_closest(r, orc, o, d)
    assert ref["hit"].mean() > 0.1
    if geometry in ("fan_1000", "fan_2000", "slivers_4000"):
        at_vertex = (ref["hit"][-len(o) // 4:] == 1) & (np.abs(ref["t"][-len(o) // 4:] - np.linalg.norm(o[-len(o) // 4:], axis=1)) < 1e-3)
        assert at_vertex.mean() > 0.2                     # the shared vertex really is hit
    # shadow queries from the surface points
    m = ref["hit"] == 1
    pos, nd, obj = ref["pos"][m], ref["ndir"][m], ref["object"][m]
    lp = np.tile(np.array([[2, 8, 3]], np.float32), (len(pos), 1))
    lp[::3] = rng.uniform(-3, 3, (len(lp[::3]), 3)).astype(np.float32)
    ldir = np.zeros((len(pos), 4), np.float32)
    ldir[:, :3] = rng.normal(size=(len(pos), 3))
    ldir[::5, 0] = 0.0
    hard, soft, dirc = orc.shadow_hard(pos, nd, lp), orc.shadow_soft(pos, nd, lp), orc.shadow_directional(pos, obj, ldir)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        assert np.array_equal(r.interStrategy.getShadowCoeffi(pos, nd, lp), hard), traversal
        assert np.array_equal(r.interStrategy.getSoftShadowSample(pos, nd, lp), soft), traversal
        assert np.array_equal(r.interStrategy.getDirectionalShadowCoeffi(pos, obj, ldir), dirc), traversal
    r.ctx.close()


@pytest.mark.parametrize("lights", sorted(LIGHTS))
@pytest.mark.parametrize("geometry", sorted(DEEP))
def test_deep_tree_frames(workdir, geometry, lights):
    scene = deep_scene(workdir, geometry, lights)
    r = Renderer(scene)
    check_frames(r, scene)
    r.ctx.close()


def test_fan_walked_at_the_stack_budget(workdir, monkeypatch, capfd):
    """A 1500-segment fan over the floor quad: PLOC depth 58 (57 for 1450 segments, 59 for 1550), the deepest walked tree
    the 90-row stack holds (3 * 29 + 2 = 89 rows).  Walked on the device tree, without the fall-back, by every
    closest-hit and shadow kernel."""
    scene = deep_scene(workdir, "fan_1500", "soft", body=fixtures.fan_geometry(1500))
    r, line = upload_verbose(scene, monkeypatch, capfd)
    depth = int(re.search(r"walked tree depth (\d+) \(device PLOC", line).group(1))
    assert depth in (57, 58) and "89 stack rows" in line, line
    orc = ob.OracleScene(scene)
    rng = np.random.default_rng(1500)
    o, d = deep_rays(scene, rng)
    ref = check_closest(r, orc, o, d)
    m = ref["hit"] == 1
    pos, nd = ref["pos"][m], ref["ndir"][m]
    lp = rng.uniform(-3, 3, (len(pos), 3)).astype(np.float32)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        assert np.array_equal(r.interStrategy.getShadowCoeffi(pos, nd, lp), orc.shadow_hard(pos, nd, lp))
        assert np.array_equal(r.interStrategy.getSoftShadowSample(pos, nd, lp), orc.shadow_soft(pos, nd, lp))
    check_frames(r, scene, orc)
    r.ctx.close()


def _row_scene(workdir, k, alphas, light):
    """k glass spheres in a row along x (y = 0, z = -2), a floor below, `light` config lines."""
    text = (f"imsize 160 120\neye 0 2.5 {k * 0.6 + 3:.1f}\nviewdir 0 -0.35 -1\nhfov 70\nupdir 0 1 0\n"
            f"bkgcolor 0.2 0.3 0.5 1\n{light}")
    for i, a in enumerate(alphas):
        text += f"mtlcolor 0.8 0.8 0.9 1 1 1 0.2 0.6 0.3 20 {a:.4f} 1.3\nsphere {i - (k - 1) / 2:.4f} 0 -2 0.42\n"
    return Scene(text=text + _with_floor("", y=-0.6), asset_dir=workdir)


def _alphas(k, kind):
    return [0.8] * k if kind == "equal" else list(np.linspace(0.05, 0.9, k))


@pytest.mark.parametrize("kind", ["distinct", "equal"])
@pytest.mark.parametrize("k", [11, 12, 13, 20])
def test_hard_shadow_crossings_around_the_association_limit(workdir, k, kind):
    """Shadow rays along a row of k glass spheres towards a point light past its end: up to WRT_SHADOW_HITS = 12
    translucent blockers the product has the reference tree's association (bit for bit); beyond, visit order: non-zero
    and within k ulp."""
    scene = _row_scene(workdir, k, _alphas(k, kind), f"light {k / 2 + 3:.1f} 0.1 -2 1 1 1 1\n")
    rng = np.random.default_rng(k)
    n = 100_000
    x0 = -k / 2 - 1
    pos = np.stack([rng.uniform(x0 - 2, x0, n), rng.uniform(-0.3, 0.3, n), rng.uniform(-2.3, -1.7, n)], 1).astype(np.float32)
    nd = _unit(rng.normal(size=(n, 3))).astype(np.float32)
    lp = np.stack([np.full(n, k / 2 + 3), rng.uniform(-0.25, 0.25, n), rng.uniform(-2.25, -1.75, n)], 1).astype(np.float32)
    orc = ob.OracleScene(scene)
    ref = orc.shadow_hard(pos, nd, lp)
    every = np.float32(1.0)
    for a in _alphas(k, kind):
        every = every * (np.float32(1.0) - np.float32(f"{a:.4f}"))
    assert (ref <= every * np.float32(1.0001)).mean() > 0.3          # most rays cross all k spheres
    assert (ref > 0).all()
    r = Renderer(scene)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        got = r.interStrategy.getShadowCoeffi(pos, nd, lp)
        if k <= 12:
            assert np.array_equal(got, ref), (traversal, int((got != ref).sum()), int(ulp_diff(got, ref).max()))
        else:
            assert (got > 0).all() and ulp_diff(got, ref).max() <= k, (traversal, int(ulp_diff(got, ref).max()))
    check_frames(r, scene, orc)
    r.ctx.close()


@pytest.mark.parametrize("k", [7, 8, 9, 30])
def test_directional_crossings_around_the_hit_limit(workdir, k):
    """Directional-shadow rays along a row of k translucent spheres: the culled walk keeps up to WRT_DIR_HITS = 8 hits
    and falls back to the literal objList loop past that; bit-exact with the oracle for every k, in both modes
    (exhaustive = the literal loop)."""
    scene = _row_scene(workdir, k, list(np.linspace(0.1, 0.7, k)), "light -1 -0.04 0.01 0 0.9 0.9 0.9\nlight 0 6 2 1 0.4 0.4 0.4\n")
    rng = np.random.default_rng(100 + k)
    n = 100_000
    x0 = -k / 2 - 1
    pos = np.stack([rng.uniform(x0 - 2, x0, n), rng.uniform(-0.3, 0.3, n), rng.uniform(-2.3, -1.7, n)], 1).astype(np.float32)
    ldir = np.zeros((n, 4), np.float32)
    ldir[:, 0] = -1.0
    ldir[:, 1:3] = rng.uniform(-0.1, 0.1, (n, 2)) / (k + 3)
    ldir[::7, 1:3] = 0.0                                              # along the axis: zero components
    ldir[1::7, 1] = -0.0
    self_obj = np.full(n, -1, np.int32)
    self_obj[::3] = k                                                 # a floor triangle (not on the ray)
    orc = ob.OracleScene(scene)
    ref = orc.shadow_directional(pos, self_obj, ldir)
    every = np.float32(1.0)
    for a in np.linspace(0.1, 0.7, k):
        every = every * (np.float32(1.0) - np.float32(f"{a:.4f}"))
    assert (ref <= every * np.float32(1.0001)).mean() > 0.3
    r = Renderer(scene)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        got = r.interStrategy.getDirectionalShadowCoeffi(pos, self_obj, ldir)
        assert np.array_equal(got, ref), (traversal, int((got != ref).sum()))
    check_frames(r, scene, orc)
    r.ctx.close()


def _slab_scene(workdir, n=5000):
    """A slab of n small spheres between the floor and the area light (a triangle about 10 units across): a shaft from
    the floor below crosses some 500 leaf boxes, far more than WRT_LIST_CAP = 192; shafts from the slab's top and from
    the floor beside it cross few."""
    rng = np.random.default_rng(192)
    text = ("imsize 120 90\neye 0 0.6 6\nviewdir 0 -0.2 -1\nhfov 70\nupdir 0 1 0\nbkgcolor 0.2 0.3 0.5 1\n"
            "light -1 7 -2 1 1 1 1\nshadow soft\nmtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1\n")
    text += "".join("sphere %.4f %.4f %.4f %.4f\n" % (x, y, z, rad) for x, y, z, rad in zip(
        rng.uniform(-2.5, 2.5, n), rng.uniform(1.5, 1.8, n), rng.uniform(-4.5, 0.5, n), rng.uniform(0.03, 0.06, n)))
    return Scene(text=text + _with_floor("", y=-1.0), asset_dir=workdir)


def test_soft_shadow_shafts_past_the_list_cap(workdir, monkeypatch):
    """Soft shadows under the sphere slab: the oracle's frame, and the same bytes with the candidate lists off."""
    scene = _slab_scene(workdir)
    r = Renderer(scene)
    check_frames(r, scene)
    img = r.render().copy()
    r.ctx.close()
    monkeypatch.setenv("WRT_SOFT_LISTS", "0")
    r = Renderer(scene)
    plain = r.render().copy()
    r.ctx.close()
    assert np.array_equal(plain, img)


_RENDER_BYTES = """
import sys; sys.path.insert(0, {repo!r}); sys.path.insert(0, {tests!r})
from pathlib import Path
import numpy as np
from whittedstyle_raytracer_b200 import Renderer, Scene, fixtures
from test_gpu_parity import MANY_LIGHTS
from test_gpu_capacity_edges import _slab_scene
wd = Path({wd!r}); fixtures.ensure_assets(wd)
fixtures.write_config(wd, "bunny_soft", fixtures.water_bunny_tex_config(200, 150, soft=True))
scenes = [Scene.from_workdir(wd, "bunny_soft"), Scene(text=MANY_LIGHTS, asset_dir=wd), _slab_scene(wd)]
out = []
for s in scenes:
    r = Renderer(s)
    out.append(r.render().copy())
    r.ctx.close()
np.savez({out!r}, *out)
"""


@pytest.fixture(scope="module")
def listcap4_lib():
    import __graft_entry__ as g
    return g.build_cuda_variant("listcap4", ["WRT_LIST_CAP=4", "WRT_DEBUG_BOUNDS"])


def test_list_cap_overflow_renders_the_same_bytes(workdir, tmp_path, listcap4_lib):
    """With a 4-entry candidate list (and every index checked) almost every soft-shadow request takes the overflow
    path to the per-ray walk: the bunny soft frame, six area lights and the sphere slab are byte-identical to the default
    build's."""
    frames = {}
    for name, lib in (("default", REPO / "whittedstyle_raytracer_b200" / "libwrt_cuda.so"), ("listcap4", listcap4_lib)):
        out = tmp_path / f"{name}.npz"
        code = _RENDER_BYTES.format(repo=str(REPO), tests=str(REPO / "tests"), wd=str(workdir), out=str(out))
        p = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, WRT_CUDA_LIB=str(lib)),
                           capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
        with np.load(out) as z:
            frames[name] = [z[f"arr_{i}"] for i in range(len(z.files))]
    assert len(frames["default"]) == 3
    for a, b in zip(frames["default"], frames["listcap4"]):
        assert a.tobytes() == b.tobytes()
