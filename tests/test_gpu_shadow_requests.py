"""The frame's own shadow kernels against the CPU oracle, request by request and bit for bit.

A frame answers its shadow requests with other code than the batch queries wrt_shadow_hard / _soft / _directional:
k_shadow_hard (octant copies, the 4-wide view, deferred leaves, lane refill, the ShadowAcc -> shadow_assoc.h association
rebuild), the soft-shadow candidate-list kernels k_soft_lists -> k_soft_filter -> k_soft_list_rays (a streaming ring of
prepared shafts, pool allocation, the edge-plane stage, compaction of the work list, 32-ray passes spanning two requests),
k_shadow_soft (light avatars, exhaustive mode, lists off), k_shadow_directional and the spawn-time shaft test.  Through an
8-bit image most of their errors are invisible: a hard-shadow product wrong in its last bits never changes a pixel, and
one lost soft sample of 50 is under 1 LSB wherever the light's term is small.  wrt_shadow_requests_wavefront queues given
requests exactly as the surface stage does and runs those kernels on the stream and grid of the chosen request queue;
its answer per request (the product, or the lit samples of 50) must equal the oracle's orc_shadow_requests bit for bit.
Bars: hard shadows bit-exact up to WRT_SHADOW_HITS = 12 translucent crossings, beyond non-zero and within k ulp for k
crossings; soft and directional shadows bit-exact; every answer independent of the batch size and of the other requests.
"""
import numpy as np
import pytest

import oracle_bindings as ob
from conftest import load_golden_scene, ulp_diff
from test_gpu_capacity_edges import _alphas, _row_scene, _slab_scene, _with_floor
from test_gpu_parity import AXIS_ALIGNED, MANY_LIGHTS
from whittedstyle_raytracer_b200 import Renderer, Scene, cabi
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED

pytestmark = pytest.mark.gpu

MODES = (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE)
SHAFT = cabi.WRT_REQ_SHAFT_CULL
RUNS = ((0, 0), (0, SHAFT), (1, 0), (2, 0))           # (request queue, flags)


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _is_point(scene):
    d = scene.desc
    return np.array([abs(d.lights[i].pos[3] - 1.0) < 1e-5 for i in range(d.n_lights)])


def _req(pos, nd, light, pixel, path, obj):
    return dict(pos=np.ascontiguousarray(pos, np.float32), nd=np.ascontiguousarray(nd, np.float32),
                light=np.ascontiguousarray(light, np.int32), pixel=np.ascontiguousarray(pixel, np.uint32),
                path=np.ascontiguousarray(path, np.uint32), obj=np.ascontiguousarray(obj, np.int32))


def _keys(rng, n, n_lights, obj):
    """Every light of the scene; pixels up to 2^25 (8K) and the extremes 0 and 2^32 - 1; paths 1 .. 511; the object the
    point lies on, and for a fifth of the requests another object or none."""
    light = rng.integers(0, n_lights, n)
    pixel = rng.integers(0, 1 << 25, n).astype(np.uint32)
    pixel[::97] = 0
    pixel[1::97] = 0xFFFFFFFF
    path = rng.integers(1, 512, n)
    obj = obj.copy()
    k = n // 5
    obj[:k] = rng.integers(-1, max(obj.max(), 0) + 1, k)
    return light, pixel, path, obj


def scene_requests(scene, orc, rng, n):
    """n requests on the oracle's closest hits of random rays through the scene's box and of the camera's primary rays,
    normals as given and flipped."""
    box = scene.nodes()[0]
    lo, hi = np.maximum(box[0:3], -50), np.minimum(box[4:7], 50)
    pos, nd, obj = [], [], []
    po, pd = orc.primary_rays()
    while sum(len(p) for p in pos) < n:
        m = n
        o = rng.uniform(lo - 0.2 * (hi - lo), hi + 0.2 * (hi - lo), (m, 3)).astype(np.float32)
        d = _unit(rng.normal(size=(m, 3))).astype(np.float32)
        pick = rng.integers(0, len(po), m // 2)
        o[: m // 2], d[: m // 2] = po[pick], pd[pick]
        h = orc.trace_closest(o, d)
        h = h[h["hit"] == 1]
        pos.append(h["pos"]), nd.append(h["ndir"]), obj.append(h["object"])
    pos, nd, obj = np.concatenate(pos)[:n], np.concatenate(nd)[:n], np.concatenate(obj)[:n]
    nd[1::2] *= -1.0
    return _req(pos, nd, *_keys(rng, n, scene.desc.n_lights, obj))


def oracle(orc, q):
    return orc.shadow_requests(q["pos"], q["nd"], q["light"], q["pixel"], q["path"], q["obj"])


def frame(r, q, queue=0, flags=0, idx=None):
    if idx is not None:
        q = {k: v[idx] for k, v in q.items()}
    return r.interStrategy.shadowRequestsWavefront(q["pos"], q["nd"], q["light"], q["pixel"], q["path"], q["obj"],
                                                   queue=queue, flags=flags)


def assert_bits(got, ref, what):
    bad = np.flatnonzero(got.view(np.int32) != ref.view(np.int32))
    assert len(bad) == 0, (what, len(bad), [(int(i), float(got[i]), float(ref[i])) for i in bad[:5]])


def check_runs(r, q, ref, what, runs=RUNS, modes=MODES):
    for traversal in modes:
        r.ctx.set_options(traversal=traversal)
        for queue, flags in runs:
            assert_bits(frame(r, q, queue, flags), ref, (what, traversal, queue, flags))
    r.ctx.set_options(traversal=TRAVERSAL_PRUNED)


# ---------------- the fixture scenes ----------------

SCENES = {          # name -> (scene builder, requests)
    "water_small": (lambda wd: load_golden_scene(wd, "water_small")[0], 1_000_000),      # glass bunny (alpha 0.2), hard
    "directional": (lambda wd: load_golden_scene(wd, "directional")[0], 1_000_000),      # point and directional lights
    "water_soft": (lambda wd: load_golden_scene(wd, "water_soft", kind="soft")[0], 200_000),
    "spheres_soft": (lambda wd: load_golden_scene(wd, "spheres_soft", kind="soft")[0], 200_000),
    "many_lights": (lambda wd: Scene(text=MANY_LIGHTS, asset_dir=wd), 200_000),   # 6 area lights: parameter bank + global
}


@pytest.mark.parametrize("name", sorted(SCENES))
def test_shadow_requests_of_the_fixture_scenes(workdir, name):
    """About 1e6 hard or 2e5 soft requests on every light of the scene, queues 0, 1 and 2, queue 0 with the spawn-time
    shaft test as well, both traversal modes."""
    build, n = SCENES[name]
    scene = build(workdir)
    orc = ob.OracleScene(scene)
    q = scene_requests(scene, orc, np.random.default_rng(len(name)), n)
    ref = oracle(orc, q)
    point = _is_point(scene)[q["light"]]
    if scene.desc.shadow_type:
        s = ref[point]
        assert ((s > 0) & (s < 50)).mean() > 0.002 and (s == 0).mean() > 0.01 and (s == 50).mean() > 0.05   # penumbra too
        assert np.array_equal(s, np.round(s))
    else:
        assert 0.01 < (ref < 1).mean() < 0.99
    if not point.all():
        assert 0.01 < (ref[~point] < 1).mean() < 0.99
    r = Renderer(scene)
    check_runs(r, q, ref, name)
    r.ctx.close()


# ---------------- the association of the hard-shadow product in k_shadow_hard ----------------

@pytest.mark.parametrize("kind", ["distinct", "equal"])
@pytest.mark.parametrize("k", [3, 6, 12, 13, 20])
def test_shadow_requests_hard_product_association(workdir, k, kind):
    """Requests beside a row of k glass spheres towards the point light past its end: up to 12 translucent blockers the
    frame kernel's product has the reference tree's association, bit for bit; beyond, non-zero and within k ulp."""
    scene = _row_scene(workdir, k, _alphas(k, kind), f"light {k / 2 + 3:.1f} 0.1 -2 1 1 1 1\n")
    rng = np.random.default_rng(300 + k)
    n = 100_000
    x0 = -k / 2 - 1
    pos = np.stack([rng.uniform(x0 - 2, x0, n), rng.uniform(-0.3, 0.3, n), rng.uniform(-2.3, -1.7, n)], 1)
    q = _req(pos, _unit(rng.normal(size=(n, 3))), *_keys(rng, n, 1, np.full(n, -1)))
    orc = ob.OracleScene(scene)
    ref = oracle(orc, q)
    every = np.float32(1.0)
    for a in _alphas(k, kind):
        every = every * (np.float32(1.0) - np.float32(f"{a:.4f}"))
    assert (ref <= every * np.float32(1.0001)).mean() > 0.3 and (ref > 0).all()
    r = Renderer(scene)
    for traversal in MODES:
        r.ctx.set_options(traversal=traversal)
        for queue in (0, 1, 2):
            got = frame(r, q, queue)
            if k <= 12:
                assert_bits(got, ref, (traversal, queue))
            else:
                assert (got > 0).all() and ulp_diff(got, ref).max() <= k, (traversal, queue, int(ulp_diff(got, ref).max()))
    r.ctx.close()


def test_shadow_requests_through_the_glass_bunny(workdir):
    """Requests behind the glass bunny (alpha 0.2), seen from its light: four and more equal factors, whose product
    already depends on the association."""
    scene, _ = load_golden_scene(workdir, "water_small")
    L = np.array(scene.desc.lights[0].pos[:3], np.float64)
    rng = np.random.default_rng(7)
    m = 200_000
    target = np.stack([rng.uniform(-1.2, 1.2, m), rng.uniform(-1.0, 1.2, m), rng.uniform(-3.2, -1.2, m)], 1)
    dirs = _unit(target - L)
    pos = target + dirs * rng.uniform(2.0, 6.0, (m, 1))
    q = _req(pos, -dirs, *_keys(rng, m, scene.desc.n_lights, np.full(m, -1)))
    q["light"][:] = 0
    orc = ob.OracleScene(scene)
    ref = oracle(orc, q)
    a4 = np.float32(0.8) ** 4
    assert ((ref > 0) & (ref <= a4)).mean() > 0.02
    r = Renderer(scene)
    check_runs(r, q, ref, "glass bunny", runs=((0, 0), (1, 0), (2, 0)))
    r.ctx.close()


# ---------------- the soft-shadow list path at its capacities ----------------

def _slab_requests(scene, rng):
    """Under the sphere slab (more than WRT_LIST_CAP = 192 candidates: the per-ray fall-back), on its top, and on the
    floor beside it (short lists that reach the edge-plane stage)."""
    n = 12_000
    under = np.stack([rng.uniform(-2.3, 2.3, n), np.full(n, -1.0), rng.uniform(-4.3, 0.3, n)], 1)
    top = np.stack([rng.uniform(-2.4, 2.4, n), rng.uniform(1.87, 1.95, n), rng.uniform(-4.4, 0.4, n)], 1)
    beside = np.stack([rng.uniform(2.6, 9.0, n), np.full(n, -1.0), rng.uniform(-8.0, 4.0, n)], 1)
    pos = np.concatenate([under, top, beside])
    nd = np.tile([[0.0, 1.0, 0.0]], (len(pos), 1))
    return _req(pos, nd, *_keys(rng, len(pos), 1, np.full(len(pos), -1)))


def _light_plane_scene(workdir):
    text = ("imsize 64 48\neye 0 6 9\nviewdir 0 -0.5 -1\nhfov 60\nupdir 0 1 0\nbkgcolor 0.2 0.3 0.5 1\n"
            "light 0 3 0 1 1 1 1\nshadow soft\nmtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1\n")
    rng = np.random.default_rng(33)
    for x, z in rng.uniform(-6, 6, (40, 2)):
        text += f"sphere {x:.3f} {3.0 + rng.uniform(-0.2, 0.2):.3f} {z:.3f} {rng.uniform(0.1, 0.4):.3f}\n"
    return Scene(text=_with_floor(text, y=-1.0), asset_dir=workdir)


def _light_plane_requests(scene, rng):
    """Origins in the plane of the horizontal light triangle, normals in that plane: a sample ray aims at a light point
    of the same y (exactly, for nine in ten samples), so it is axis-degenerate and walks the reference tree."""
    y = np.float32(scene.desc.lights[0].tri[1])
    n = 20_000
    pos = np.stack([rng.uniform(-9, 9, n), np.full(n, y), rng.uniform(-9, 9, n)], 1)
    nd = np.zeros((n, 3))
    nd[np.arange(n), rng.choice([0, 2], n)] = rng.choice([1.0, -1.0], n)
    return _req(pos, nd, *_keys(rng, n, 1, np.full(n, -1)))


def _axis_aligned_requests(scene, rng):
    """On the wall the light faces, around y = 0 where the light's corners lie too: shafts without a definite sign on y."""
    n = 20_000
    pos = np.stack([rng.uniform(-5.5, 5.5, n), rng.uniform(-0.05, 0.05, n), np.full(n, -2.0)], 1)
    pos[::4, 1] = 0.0
    nd = np.tile([[0.0, 0.0, 1.0]], (n, 1))
    return _req(pos, nd, *_keys(rng, n, 1, np.full(n, -1)))


AVATAR = ("imsize 40 30\neye 0 0 0\nviewdir 0 0 -1\nupdir 0 1 0\nhfov 60\nbkgcolor 0.1 0.1 0.1 1\nlight 0 5 -3 1 1 1 1\n"
          "shadow soft\nmtlcolor 1 1 1 1 1 1 1 1 1 0 1 1\nsphere 0 5 -3 0.5\nmtlcolor 0.8 0.4 0.2 1 1 1 0.3 0.6 0.2 10 1 1\n"
          "sphere 0 0 -4 1\nv -5 -1 0\nv 5 -1 0\nv 0 -1 -9\nf 1 2 3\n")

LIST_CASES = {
    "slab": (lambda wd: _slab_scene(wd), _slab_requests),
    "light_plane": (_light_plane_scene, _light_plane_requests),
    "axis_aligned": (lambda wd: Scene(text=AXIS_ALIGNED, asset_dir=wd), _axis_aligned_requests),
    "light_avatar": (lambda wd: Scene(text=AVATAR, asset_dir=wd),
                     lambda s, rng: scene_requests(s, ob.OracleScene(s), rng, 20_000)),
}
# (environment, traversal) -> which kernels answer: the lists with or without k_soft_filter, or k_shadow_soft
VARIANTS = [({}, TRAVERSAL_PRUNED), ({"WRT_LIST_POOL_CAP": "64"}, TRAVERSAL_PRUNED), ({"WRT_SOFT_FILTER": "0"}, TRAVERSAL_PRUNED),
            ({"WRT_SOFT_FILTER": "1"}, TRAVERSAL_PRUNED), ({"WRT_SOFT_FILTER": "2"}, TRAVERSAL_PRUNED),
            ({"WRT_SOFT_LISTS": "0"}, TRAVERSAL_PRUNED), ({}, TRAVERSAL_EXHAUSTIVE)]


@pytest.mark.parametrize("case", sorted(LIST_CASES))
def test_shadow_requests_soft_list_path_at_its_capacities(workdir, monkeypatch, case):
    """The same requests through every soft-shadow path: the lists (full pool, filter off / on the deep queues / on every
    queue), the per-ray kernel (lists off, exhaustive mode, a scene with a light-avatar primitive); the launch counts
    say which path answered."""
    make_scene, make_requests = LIST_CASES[case]
    scene = make_scene(workdir)
    orc = ob.OracleScene(scene)
    q = make_requests(scene, np.random.default_rng(len(case)))
    ref = oracle(orc, q)
    assert ((ref > 0) & (ref < 50)).mean() > 0.01 and len(np.unique(ref)) > 20, case
    avatar = scene.desc.n_prims > 0 and bool((np.ctypeslib.as_array(scene.desc.prim_flags, (scene.desc.n_prims,)) & 2).any())   # WRT_PRIM_LIGHT
    assert avatar == (case == "light_avatar")
    for env, traversal in VARIANTS:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        r = Renderer(scene)
        for k in env:
            monkeypatch.delenv(k)
        r.ctx.set_options(traversal=traversal)
        for queue, flags in RUNS:
            assert_bits(frame(r, q, queue, flags), ref, (case, env, traversal, queue, flags))
        r.ctx.enable_kernel_timing(True)
        for queue in (0, 1):
            assert_bits(frame(r, q, queue), ref, (case, env, traversal, queue, "timed"))
            got = r.ctx.kernel_launches()
            lists = not avatar and traversal == TRAVERSAL_PRUNED and env.get("WRT_SOFT_LISTS") != "0"
            filtered = lists and int(env.get("WRT_SOFT_FILTER", "2")) >= (2 if queue == 0 else 1)
            assert (got["soft_lists"], got["soft_filter"], got["shadow_soft"]) == (int(lists), int(filtered), 1), (case, env, queue, got)
        r.ctx.close()


# ---------------- directional lights ----------------

@pytest.mark.parametrize("k", [7, 8, 9, 30])
def test_shadow_requests_directional_rows(workdir, k):
    """Requests before a row of k translucent spheres, directional lights along the row (one with +0 and -0 components),
    the point's object on the ray (a sphere of the row), off it (the floor) or none: bit-exact through
    k_shadow_directional's culled walk (up to WRT_DIR_HITS = 8 hits) and its literal fall-back."""
    lights = ("light -1 -0.04 0.01 0 0.9 0.9 0.9\nlight -1 0 -0 0 0.5 0.5 0.5\nlight -1 -0 0.0001 0 0.4 0.4 0.4\n"
              "light 0 6 2 1 0.4 0.4 0.4\n")
    scene = _row_scene(workdir, k, list(np.linspace(0.1, 0.7, k)), lights)
    rng = np.random.default_rng(200 + k)
    n = 100_000
    x0 = -k / 2 - 1
    pos = np.stack([rng.uniform(x0 - 2, x0, n), rng.uniform(-0.3, 0.3, n), rng.uniform(-2.3, -1.7, n)], 1)
    pos[::5, 1:] = (0.0, -2.0)
    obj = rng.choice([-1, 0, k // 2, k - 1, k, k + 1], n)
    q = _req(pos, _unit(rng.normal(size=(n, 3))), *_keys(rng, n, scene.desc.n_lights, obj))
    q["obj"][:] = obj
    orc = ob.OracleScene(scene)
    ref = oracle(orc, q)
    d = ~_is_point(scene)[q["light"]]
    every = np.float32(1.0)
    for a in np.linspace(0.1, 0.7, k):
        every = every * (np.float32(1.0) - np.float32(f"{a:.4f}"))
    assert (ref[d] <= every * np.float32(1.0001)).mean() > 0.2
    r = Renderer(scene)
    check_runs(r, q, ref, f"row {k}", runs=((0, 0), (1, 0), (2, 0)))
    r.ctx.close()


# ---------------- queue shapes ----------------

@pytest.mark.parametrize("name", ["water_small", "water_soft", "directional", "many_lights"])
def test_shadow_requests_do_not_depend_on_the_batch(workdir, name):
    """Batches of 1, 31, 32, 33, 50, 4097 requests and the full batch, the same requests reversed and permuted: every
    request's answer is the oracle's, whatever its neighbours (chunk claiming, lane refill, filter blocks and the
    32-ray passes that span two requests)."""
    scene = SCENES[name][0](workdir)
    orc = ob.OracleScene(scene)
    rng = np.random.default_rng(99)
    q = scene_requests(scene, orc, rng, 30_000)
    ref = oracle(orc, q)
    r = Renderer(scene)
    n = len(ref)
    perm = rng.permutation(n)
    for traversal, queue in ((TRAVERSAL_PRUNED, 0), (TRAVERSAL_PRUNED, 1), (TRAVERSAL_EXHAUSTIVE, 2)):
        r.ctx.set_options(traversal=traversal)
        for size in (1, 31, 32, 33, 50, 4097, n):
            for start in (0, n - size):
                idx = np.arange(start, start + size)
                assert_bits(frame(r, q, queue, idx=idx), ref[idx], (name, traversal, queue, size, start))
        assert_bits(frame(r, q, queue, idx=np.arange(n)[::-1]), ref[::-1], (name, traversal, queue, "reversed"))
        assert_bits(frame(r, q, queue, SHAFT, idx=perm), ref[perm], (name, traversal, queue, "permuted"))
    r.ctx.close()
