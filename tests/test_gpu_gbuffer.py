"""The frame's per-pixel surface planes (wrt_render_gbuffer) against the CPU oracle, bit for bit, and the frame itself
unchanged by them.

The oracle side is composed of entries that already exist, in the device-math build (sphere uv): orc_primary_rays and
orc_trace_closest give the eye ray's record; orc_shading_surface (tests/shading_surface_oracle.c) the shading normal and Od the shader uses at it;
orc_shadow_requests, keyed as the frame keys level 0 (pixel y * W + x, path 1, the point's object, hit.pos and the shading
normal), the coefficient of each light (soft point lights: lit samples / 50 in float, as blinn_phong divides).  -1 is
expected exactly on unshaded pixels (misses, light avatars) and, in the pruned mode with the unlit-light culling on, on
lights 0..31 whose diffuse and specular factors both vanish (light_terms_vanish, recomputed here in float32)."""
import ctypes as C

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import IMG_SCENES, SOFT_SCENES, load_golden_scene
from test_gpu_float_frame import CROPS, forty_lights
from test_gpu_fuzz import random_scene
from test_gpu_parity import AXIS_ALIGNED, MANY_LIGHTS, light_bank
from test_oracle_shading_surface import scene_arrays, shaded_mask, shading_surface
from whittedstyle_raytracer_b200 import Renderer, Scene, cabi, fixtures
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED

pytestmark = pytest.mark.gpu

TRAVERSALS = (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE)
PLANES = ("hit", "normal", "albedo", "shadow")
F32 = np.float32


@pytest.fixture(scope="session", autouse=True)
def _devmath_oracle():
    import __graft_entry__ as g
    g.build_oracle(device_math=True)


def _normalized(v):
    """Vector.hpp:127-134 in float32, one rounding per operation as the kernels compute it."""
    mag = np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
    inv = np.where(mag > 0, F32(1) / np.where(mag > 0, mag, F32(1)), F32(1))
    return np.where((mag > 0)[:, None], v * inv[:, None], v)


def _dot(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2]


def terms_vanish(light, eye_org, pos, ndir, n_exp):
    """dev_shade.cuh light_terms_vanish: max(L.N, 0) == 0 and pow(max(H.N, 0), n) == 0."""
    with np.errstate(all="ignore"):
        p_eye = _normalized(eye_org - pos)
        if abs(light.pos[3] - 1.0) < 1e-5:
            ldir = _normalized(np.array(light.pos[:3], F32)[None, :] - pos)
        else:
            ldir = _normalized(np.tile(-np.array(light.pos[:3], F32), (len(pos), 1)))
        ndl = _dot(ldir, _normalized(ndir))
        mx = np.where(ndl < 0, F32(0), ndl)
        hn = _dot(_normalized(ldir + p_eye), ndir)
        mh = np.where(hn < 0, F32(0), hn)
        pw = np.where((mh == 0) & (n_exp > 0), F32(0),
                      np.power(mh.astype(np.float64), n_exp.astype(np.float64)).astype(F32))
    return (mx == 0) & (pw == 0)


def oracle_gbuffer(scene, x0=0, x1=None, y0=0, y1=None):
    """The oracle's planes of the pixel window [x0, x1) x [y0, y1), and the masks of shaded pixels and of lights whose
    terms vanish."""
    cam = scene.camera
    W = cam.width
    x1 = W if x1 is None else x1
    y1 = cam.height if y1 is None else y1
    h, w = y1 - y0, x1 - x0
    orc = ob.OracleScene(scene, device_math=True)
    o, d = orc.primary_rays()
    ys, xs = np.mgrid[y0:y1, x0:x1]
    pix = (ys * W + xs).ravel()
    hits = orc.trace_closest(o[pix], d[pix])
    nd, od = shading_surface(scene, hits, device_math=True)
    shaded = shaded_mask(scene, hits)
    _, _, n_exp = scene_arrays(scene)
    desc = scene.desc
    nl = desc.n_lights
    shadow = np.full((len(pix), nl), -1, F32)
    vanish = np.zeros((len(pix), nl), bool)
    sel = np.nonzero(shaded)[0]
    for li in range(nl):
        L = desc.lights[li]
        coeff = orc.shadow_requests(hits["pos"][sel], nd[sel], np.full(len(sel), li, np.int32), pix[sel].astype(np.uint32),
                                    np.ones(len(sel), np.uint32), hits["object"][sel])
        if abs(L.pos[3] - 1.0) < 1e-5 and desc.shadow_type != 0:
            coeff = coeff / F32(cabi.WRT_SOFT_SAMPLES)
        shadow[sel, li] = coeff
        vanish[sel, li] = terms_vanish(L, o[pix][sel], hits["pos"][sel], nd[sel], n_exp[hits["material"][sel]])
    return dict(hit=hits.reshape(h, w), normal=nd.reshape(h, w, 3), albedo=od.reshape(h, w, 3),
                shadow=shadow.reshape(h, w, nl), shaded=shaded.reshape(h, w), vanish=vanish.reshape(h, w, nl))


def assert_bits_equal(got, want, what):
    """float32 arrays equal bit for bit; NaN compares by class only."""
    gb, wb = got.view(np.uint32), want.view(np.uint32)
    same = (gb == wb) | (np.isnan(got) & np.isnan(want))
    if not same.all():
        bad = np.argwhere(~same)
        rows = [f"  at {tuple(int(v) for v in b)}: frame {got[tuple(b)]!r}, oracle {want[tuple(b)]!r}" for b in bad[:10]]
        raise AssertionError(f"{what}: {len(bad)} of {got.size} values differ\n" + "\n".join(rows))


def check_planes(got, want, what, culled):
    """got: the frame's planes (of the window); culled: the frame answered vanishing lights without a coefficient."""
    shaded = want["shaded"]
    g, wh = got["hit"], want["hit"]
    for f in ("hit", "object", "texture", "normalmap", "material", "prim"):
        assert np.array_equal(g[f], wh[f]), f"{what}: hit.{f}"
    for f in ("t", "pos", "ndir", "uv"):
        assert_bits_equal(np.ascontiguousarray(g[f]), np.ascontiguousarray(wh[f]), f"{what}: hit.{f}")
    for name in ("normal", "albedo"):
        assert_bits_equal(got[name][shaded], want[name][shaded], f"{what}: {name} on shaded pixels")
        assert not got[name][~shaded].view(np.uint32).any(), f"{what}: {name} is not +0 on unshaded pixels"
    nl = want["shadow"].shape[2]
    minus1 = np.broadcast_to(~shaded[..., None], want["shadow"].shape).copy()
    if culled:
        minus1 |= want["vanish"] & (np.arange(nl) < 32)
    sh = got["shadow"]
    assert np.array_equal(sh == F32(-1), minus1), (f"{what}: -1 on {int((sh == -1).sum())} entries, "
                                                  f"expected on {int(minus1.sum())} ({int((sh == -1)[~minus1].sum())} unexpected)")
    assert_bits_equal(sh[~minus1], want["shadow"][~minus1], f"{what}: shadow")


def check_scene(scene, what, want=None, traversals=TRAVERSALS):
    """Every plane equals the oracle's in each traversal mode, and the call's image is wrt_render's."""
    want = want or oracle_gbuffer(scene)
    r = Renderer(scene)
    try:
        for traversal in traversals:
            r.ctx.set_options(traversal=traversal)
            img = r.render().copy()
            got = r.render_gbuffer()
            assert np.array_equal(got["rgb"], img), f"{what}: image"
            check_planes(got, want, f"{what}, traversal {traversal}", culled=traversal == TRAVERSAL_PRUNED)
            if traversal == TRAVERSAL_EXHAUSTIVE:
                assert not (got["shadow"][want["shaded"]] == -1).any()
    finally:
        r.ctx.close()
    return want


# ---------------- scenes against the oracle ----------------

@pytest.mark.parametrize("name,kind", [(n, "img") for n in IMG_SCENES + ["config_800x600"]] + [(n, "soft") for n in SOFT_SCENES])
def test_gbuffer_fixture_scenes(workdir, name, kind):
    scene, _ = load_golden_scene(workdir, name, kind=kind)
    want = check_scene(scene, name)
    assert want["shaded"].any() and (~want["shaded"]).any()


LIGHT_SCENES = ([(f"bank_{n}_{'soft' if s else 'hard'}", lambda n=n, s=s: light_bank(n, soft=s)) for n in range(1, 6) for s in (False, True)]
                + [("many_lights", lambda: MANY_LIGHTS), ("axis_aligned", lambda: AXIS_ALIGNED)]
                + [(f"forty_lights_{'soft' if s else 'hard'}", lambda s=s: forty_lights(s)) for s in (False, True)])


@pytest.mark.parametrize("name,text", LIGHT_SCENES)
def test_gbuffer_light_scenes(workdir, name, text):
    scene = Scene(text=text(), asset_dir=workdir)
    want = check_scene(scene, name)
    if name.startswith("forty"):                       # lights past the 32 the frame's cull masks cover
        assert scene.desc.n_lights == 40 and want["vanish"][..., 32:].any() and want["vanish"][..., :32].any()


@pytest.mark.parametrize("seed", range(6))
def test_gbuffer_random_scenes(workdir, seed):
    text = random_scene(np.random.default_rng(1000 + seed))
    check_scene(Scene(text=text, asset_dir=workdir), f"random scene {seed}\n{text}")


@pytest.mark.parametrize("name", list(CROPS))
def test_gbuffer_4k_crops(workdir, name):
    """The GPU renders the whole 3840x2160 frame; the oracle computes the window's eye rays only."""
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name, bunny=fixtures.BENCH_CONFIGS[name].get("bunny", True))
    x0, y0 = CROPS[name]
    n = 256
    want = oracle_gbuffer(scene, x0, x0 + n, y0, y0 + n)
    assert want["shaded"].any()
    win = np.s_[y0:y0 + n, x0:x0 + n]
    r = Renderer(scene)
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal)
        got = r.render_gbuffer()
        check_planes({k: v[win] for k, v in got.items()}, want, f"{name} window, traversal {traversal}",
                     culled=traversal == TRAVERSAL_PRUNED)
    r.ctx.close()


def test_gbuffer_without_unlit_cull(workdir, monkeypatch):
    """WRT_UNLIT_CULL=0: every shaded pixel has every coefficient, in the pruned mode too."""
    monkeypatch.setenv("WRT_UNLIT_CULL", "0")
    for text in (forty_lights(False), light_bank(5, soft=True)):
        scene = Scene(text=text, asset_dir=workdir)
        want = oracle_gbuffer(scene)
        assert want["vanish"].any()
        r = Renderer(scene)
        for traversal in TRAVERSALS:
            r.ctx.set_options(traversal=traversal)
            got = r.render_gbuffer()
            check_planes(got, want, f"WRT_UNLIT_CULL=0, traversal {traversal}", culled=False)
            assert not (got["shadow"][want["shaded"]] == -1).any()
        r.ctx.close()


# ---------------- the frame is unchanged ----------------

def _subsets():
    import itertools
    return [c for k in range(len(PLANES) + 1) for c in itertools.combinations(PLANES, k)]


def test_gbuffer_is_the_plain_frame(workdir):
    """Same image and statistics as wrt_render for every subset of planes; the planes of a subset are those of the full
    call; launches grow by k_gbuffer_hit (hit) and k_gbuffer_surface (normal, albedo or shadow) per batch, and
    wrt_render's own count per frame stays what it was."""
    for name, kind in (("water_small", "img"), ("water_soft", "soft"), ("directional", "img")):
        scene, _ = load_golden_scene(workdir, name, kind=kind)
        r = Renderer(scene)
        n0 = r.ctx.launches
        img = r.render().copy()
        plain = r.ctx.launches - n0
        st = dict(r.last_stats)
        full = r.render_gbuffer()
        for planes in _subsets():
            n1 = r.ctx.launches
            got = r.render_gbuffer(planes=planes)
            extra = int("hit" in planes) + int(bool({"normal", "albedo", "shadow"} & set(planes)))
            assert r.ctx.launches - n1 == plain + extra, (name, planes)
            assert np.array_equal(got["rgb"], img), (name, planes)
            assert set(got) == {"rgb", *planes}
            for k in ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth", "shadow_rays_traced",
                      "shaft_culled_requests", "unlit_skipped_requests", "overflow_retries"):
                assert r.last_stats[k] == st[k], (name, planes, k)
            for p in planes:
                assert got[p].tobytes() == full[p].tobytes(), (name, planes, p)
        n2 = r.ctx.launches
        r.render()
        assert r.ctx.launches - n2 == plain, name
        r.ctx.close()


@pytest.mark.parametrize("name", ["spheres", "water_small", "bump"])
def test_gbuffer_tiles(workdir, name):
    """Rank r of N writes exactly its own pixels of every plane and leaves the rest of the caller's arrays as they were;
    the union over ranks equals the 1-rank planes (N = 3, 8)."""
    scene, _ = load_golden_scene(workdir, name)
    r = Renderer(scene)
    full = {k: v.copy() for k, v in r.render_gbuffer().items()}
    h, w = full["rgb"].shape[:2]

    def sentinel_out():
        out = {k: np.full_like(v, -7 if v.dtype != np.uint8 else 0) for k, v in full.items() if k != "hit"}
        out["hit"] = np.zeros_like(full["hit"])
        out["hit"]["prim"] = -7
        return out

    for world in (3, 8):
        merged = sentinel_out()
        owner = np.zeros((h, w), np.int32)
        for rank in range(world):
            r.ctx.set_tiles(rank=rank, world=world)
            mine = r.render_gbuffer(out=sentinel_out())
            written = mine["hit"]["prim"] != -7
            owner += written
            for k in PLANES:
                assert (mine[k][~written].view(np.uint8) == sentinel_out()[k][~written].view(np.uint8)).all(), (world, rank, k)
                merged[k][written] = mine[k][written]
            assert np.array_equal(mine["rgb"][written], full["rgb"][written])
        assert (owner == 1).all(), (world, int((owner == 0).sum()), int((owner > 1).sum()))
        for k in PLANES:
            assert merged[k].tobytes() == full[k].tobytes(), (name, world, k)
    r.ctx.set_tiles(rank=0, world=1)
    r.ctx.close()


@pytest.mark.parametrize("soft", [False, True])
def test_gbuffer_overflow(workdir, monkeypatch, soft):
    """A 200x150 bunny frame in batches of 8192 slots whose deep levels (queue_factor 0.02) overflow and are redone in
    halves: every batch exports, a redone batch over its first attempt, and the planes equal the single-batch ones."""
    name = f"gbuffer_overflow_{int(soft)}"
    fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(200, 150, soft=soft))
    scene = Scene.from_workdir(workdir, name)
    r = Renderer(scene)
    single = {}
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal)
        single[traversal] = {k: v.copy() for k, v in r.render_gbuffer().items()}
        assert r.last_stats["overflow_retries"] == 0
    r.ctx.close()
    monkeypatch.setenv("WRT_MAX_BATCH", "8192")
    r = Renderer(scene)
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal, queue_factor=0.02)
        got = r.render_gbuffer()
        assert r.last_stats["overflow_retries"] >= 1
        for k in ("rgb",) + PLANES:
            assert got[k].tobytes() == single[traversal][k].tobytes(), (traversal, k)
    r.ctx.close()


# ---------------- malformed input ----------------

def test_gbuffer_malformed_input(workdir):
    scene, _ = load_golden_scene(workdir, "water_small")
    r = Renderer(scene)
    lib = r.ctx.lib
    rgb = np.zeros((scene.camera.height, scene.camera.width, 3), np.uint8)
    gb = cabi.WrtGBuffer()
    st = cabi.WrtStats()
    assert lib.wrt_render_gbuffer(None, C.byref(gb), rgb.ctypes.data, C.byref(st)) != 0
    assert lib.wrt_render_gbuffer(r.ctx.h, None, rgb.ctypes.data, C.byref(st)) != 0
    assert b"null" in lib.wrt_last_error()
    with pytest.raises(ValueError):
        r.render_gbuffer(planes=("depth",))
    for k, bad in (("normal", np.zeros((scene.camera.height, scene.camera.width, 3), np.float64)),
                   ("shadow", np.zeros((scene.camera.height, scene.camera.width, 2), np.float32)),
                   ("albedo", np.zeros((scene.camera.width, scene.camera.height, 3), np.float32)),
                   ("hit", np.zeros((scene.camera.height, scene.camera.width * 2), cabi.HIT_DTYPE)[:, ::2])):
        with pytest.raises(ValueError):
            r.render_gbuffer(out={k: bad})
    r.ctx.close()
    from whittedstyle_raytracer_b200.renderer import Context
    c = Context()
    assert lib.wrt_render_gbuffer(c.h, C.byref(gb), rgb.ctypes.data, C.byref(st)) != 0     # no scene
    assert lib.wrt_upload_scene(c.h, scene.desc_ptr) == 0
    hits = np.zeros(rgb.shape[:2], cabi.HIT_DTYPE)
    gb.hit = hits.ctypes.data
    assert lib.wrt_render_gbuffer(c.h, C.byref(gb), rgb.ctypes.data, C.byref(st)) != 0     # no camera
    assert b"camera" in lib.wrt_last_error()
    c.close()
