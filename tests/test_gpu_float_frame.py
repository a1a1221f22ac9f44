"""The frame's unquantised colour (wrt_render_float: the level-0 colour k_combine_resolve quantises) against the CPU
oracle's, bit for bit.

The oracle here is its device-math build (oracle/liboracle_devmath.so): the same source, with powf, acosf and atan2f
evaluated the way the render core evaluates them (tests/test_oracle_device_math.py shows that this is the only
difference).  Every other operation is one IEEE rounding in the reference's order on both sides, so hit completion,
sphere uv, textures and normal maps, Fresnel, the child-ray directions and epsilon offsets, Blinn-Phong with
attenuation and depth cueing, and the bottom-up combine of k_surface_spawn, k_shade and k_combine_resolve must give
the oracle's float in every channel of every pixel.  The 8-bit image only sees an error that crosses a quantisation
step below 1.0.  NaN compares by class only (CPU and GPU payloads differ); +0 and -0 are distinct.

The same call's 8-bit image must be the reference quantiser int(255 * min(c, 1)), clamped to [0, 255], applied here
to the returned floats: values above 1, negative values and NaN (which the frame writes as 0) included."""
import numpy as np
import pytest

import oracle_bindings as ob
from conftest import IMG_SCENES, SOFT_SCENES, load_golden_scene
from test_gpu_fuzz import random_scene
from test_gpu_parity import AXIS_ALIGNED, EDGE_SCENES, MANY_LIGHTS, light_bank
from whittedstyle_raytracer_b200 import Renderer, Scene, fixtures
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED

pytestmark = pytest.mark.gpu

TRAVERSALS = (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE)


@pytest.fixture(scope="session", autouse=True)
def _devmath_oracle():
    import __graft_entry__ as g
    g.build_oracle(device_math=True)


def quantize(f):
    """Renderer.hpp:128-130 as the frame stores it: int(255 * std::min(c, 1.f)) in float, truncated, clamped to a
    byte.  std::min keeps a NaN colour; int(NaN) is 0 on the GPU and INT_MIN (clamped to 0) on x86-64."""
    m = np.where(f > np.float32(1), np.float32(1), f)
    q = np.float32(255) * m
    q = np.where(np.isnan(q), 0.0, np.trunc(q))
    return np.clip(q, 0, 255).astype(np.uint8)


def assert_bits_equal(got, want, what):
    gb, wb = got.view(np.uint32), want.view(np.uint32)
    same = (gb == wb) | (np.isnan(got) & np.isnan(want))
    if not same.all():
        bad = np.argwhere(~same)
        rows = [f"  pixel x={x} y={y} channel {k}: frame {got[y, x, k]!r} ({gb[y, x, k]:#010x}), "
                f"oracle {want[y, x, k]!r} ({wb[y, x, k]:#010x})" for y, x, k in bad[:10]]
        raise AssertionError(f"{what}: {len(bad)} of {got.size} float channels differ\n" + "\n".join(rows))


def oracle_float(scene, **kw):
    u8, fl, st = ob.OracleScene(scene, device_math=True).render(want_float=True, **kw)
    return fl, u8, st


def frame_float(r, traversal):
    r.ctx.set_options(traversal=traversal)
    fl, u8 = r.render_float()
    assert np.array_equal(u8, quantize(fl)), "the 8-bit frame is not int(255 * min(c, 1)) of its own float colour"
    return fl, u8, dict(r.last_stats)


def check_scene(scene, what, traversals=TRAVERSALS, want=None):
    """The frame's float colour equals the device-math oracle's bit for bit in each traversal mode, with the same ray
    counts; returns the float frame."""
    want_f, want_u8, ost = want or oracle_float(scene)
    r = Renderer(scene)
    try:
        for traversal in traversals:
            fl, u8, st = frame_float(r, traversal)
            assert_bits_equal(fl, want_f, f"{what}, traversal {traversal}")
            assert np.array_equal(u8, want_u8), what
            assert st["closest_rays"] == ost.closest_rays and st["shadow_rays"] == ost.shadow_rays, what
            assert st["rays_per_depth"] == [int(x) for x in ost.rays_per_depth], what
    finally:
        r.ctx.close()
    return fl


# ---------------- fixture scenes ----------------

@pytest.mark.parametrize("name,kind", [(n, "img") for n in IMG_SCENES + ["config_800x600"]] + [(n, "soft") for n in SOFT_SCENES])
def test_float_frame_fixture_scenes(workdir, name, kind):
    scene, _ = load_golden_scene(workdir, name, kind=kind)
    check_scene(scene, name)


def test_float_frame_is_the_plain_frame(workdir):
    """wrt_render_float renders the frame wrt_render renders, with the same launches (the float copy is a
    cudaMemcpyAsync, not a kernel) and the same statistics."""
    for name, kind in (("water_small", "img"), ("water_soft", "soft")):
        scene, _ = load_golden_scene(workdir, name, kind=kind)
        r = Renderer(scene)
        n0 = r.ctx.launches
        img = r.render().copy()
        n1 = r.ctx.launches
        st = dict(r.last_stats)
        fl, u8 = r.render_float()
        n2 = r.ctx.launches
        assert np.array_equal(u8, img), name
        assert n2 - n1 == n1 - n0, (name, n1 - n0, n2 - n1)
        for k in ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth", "shadow_rays_traced"):
            assert r.last_stats[k] == st[k], (name, k)
        r.ctx.close()


LIGHT_SCENES = ([(f"bank_{n}_{'soft' if s else 'hard'}", light_bank(n, soft=s)) for n in range(1, 6) for s in (False, True)]
                + [("many_lights", MANY_LIGHTS), ("axis_aligned", AXIS_ALIGNED)]
                + [(f"edge_{i}", text) for i, (text, _) in enumerate(EDGE_SCENES)])


@pytest.mark.parametrize("name,text", LIGHT_SCENES)
def test_float_frame_light_and_edge_scenes(workdir, name, text):
    check_scene(Scene(text=text, asset_dir=workdir), name)


def forty_lights(soft):
    """40 lights around two spheres (one glass) on a floor: point, attenuated (every 5th) and directional (every 7th),
    light k at azimuth k * pi / 32, so light 32 stands opposite light 0.  Past the 4-light kernel-parameter bank
    (WRT_INLINE_LIGHTS) and past the 32 lights whose culling k_surface_spawn records in its bit masks: on the far
    side of a sphere from light 0, light 0 is culled as unlit and light 32 is not."""
    w, h = (48, 32) if soft else (96, 64)
    lines = [f"imsize {w} {h}", "eye 0 1.5 7", "viewdir 0 -0.15 -1", "hfov 60", "updir 0 1 0", "bkgcolor 0.1 0.1 0.2 1.0"]
    if soft:
        lines.append("shadow soft")
    for k in range(40):
        a = k * np.pi / 32
        x, y, z = 7 * np.cos(a), 1.5 + (k % 4), 7 * np.sin(a) - 1
        c = 0.05 + 0.01 * (k % 3)
        if k % 7 == 4:
            lines.append(f"light {-x:.4f} {-y:.4f} {-z:.4f} 0 {c:.3f} {c:.3f} {c:.3f}")
        elif k % 5 == 3:
            lines.append(f"attlight {x:.4f} {y:.4f} {z:.4f} 1 {3 * c:.3f} {3 * c:.3f} {3 * c:.3f} 0.5 0.05 0.005")
        else:
            lines.append(f"light {x:.4f} {y:.4f} {z:.4f} 1 {c:.3f} {c:.3f} {c:.3f}")
    lines += ["mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.6 0.3 24 1 1.5", "sphere -1.3 0 -1 1.1",
              "mtlcolor 0.9 0.9 1.0 1 1 1 0.05 0.2 0.4 60 0.3 1.4", "sphere 1.3 0.1 0 1.0",
              "mtlcolor 0.4 0.7 0.4 1 1 1 0.2 0.7 0.1 10 1 1.0",
              "v -10 -1.1 8", "v 10 -1.1 8", "v 10 -1.1 -12", "v -10 -1.1 -12", "f 1 2 3", "f 1 3 4"]
    return "\n".join(lines) + "\n"


@pytest.mark.parametrize("soft", [False, True])
def test_float_frame_forty_lights(workdir, soft):
    scene = Scene(text=forty_lights(soft), asset_dir=workdir)
    assert scene.desc.n_lights == 40
    check_scene(scene, f"forty_lights soft={soft}")


@pytest.mark.parametrize("seed", range(24))
def test_float_frame_random_scenes(workdir, seed):
    """The 24 random scenes of tests/test_gpu_fuzz.py: glass, mirrors, textures and normal maps on spheres and
    triangles, depth cueing and parallel projection together."""
    text = random_scene(np.random.default_rng(1000 + seed))
    check_scene(Scene(text=text, asset_dir=workdir), f"random scene {seed}\n{text}")


# ---------------- 4K bench workloads: a contiguous window through the object ----------------

CROPS = {                      # (x0, y0) of a 256 x 256 window where the deep ray-tree levels do their work
    "bunny_shadow_4k": (1500, 1700), "gla_bunny_tex_4k": (1500, 1700), "water_bunny_tex_soft_4k": (1500, 1700),
    "f4_directional_4k": (1500, 1700), "f4_bump_4k": (1500, 1700), "f4_spheres_1k_4k": (1000, 900),
}


@pytest.mark.parametrize("name", list(CROPS))
def test_float_frame_4k_crops(workdir, name):
    """The GPU renders the whole 3840x2160 frame; the oracle renders the window with the full-size camera and RNG keys."""
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name, bunny=fixtures.BENCH_CONFIGS[name].get("bunny", True))
    x0, y0 = CROPS[name]
    n = 256
    want_f, want_u8, ost = oracle_float(scene, rows=(y0, y0 + n), cols=(x0, x0 + n))
    assert ost.closest_rays > 2 * n * n and ost.rays_per_depth[8] > 0, "the window is not where the deep levels work"
    win = np.s_[y0:y0 + n, x0:x0 + n]
    r = Renderer(scene)
    for traversal in TRAVERSALS:
        fl, u8, st = frame_float(r, traversal)         # (the sphere field overflows the automatic deep levels: redone)
        assert_bits_equal(fl[win], want_f[win], f"{name} window, traversal {traversal}")
        assert np.array_equal(u8[win], want_u8[win])
    r.ctx.close()


# ---------------- shading edges ----------------

def _camera(w, h, eye="0 0 6", viewdir="0 0 -1", hfov=50, bkg="0.2 0.3 0.4 1.0", parallel=False, soft=False):
    lines = [f"imsize {w} {h}", f"eye {eye}", f"viewdir {viewdir}", f"hfov {hfov}", "updir 0 1 0", f"bkgcolor {bkg}"]
    if parallel:
        lines.append("projection parallel")
    if soft:
        lines.append("shadow soft")
    return lines


_FLOOR = ["mtlcolor 0.5 0.55 0.5 1 1 1 0.3 0.7 0.1 10 1 1.0", "v -20 -1.5 10", "v 20 -1.5 10", "v 20 -1.5 -30",
          "v -20 -1.5 -30", "f 1 2 3", "f 1 3 4"]


def edge_scene(case, k):
    """Shading-edge scene `case`, variant k (0..5): the variant changes sizes, projection, shadow mode and materials
    around the same edge."""
    rng = np.random.default_rng(7919 * k + len(case))
    soft = k % 2 == 1
    f = lambda a, b: f"{rng.uniform(a, b):.3f}"        # noqa: E731
    if case == "pole":
        # a normal-mapped sphere on the axis of a 1-pixel camera (its ray is exactly -z): at the pole nDir.x = nDir.y = 0,
        # so change_normal_dir's tangent is 0/0 and the pixel is NaN.  ks = 0 and alpha = 1: no child rays of NaN.
        lines = _camera(1, 1, eye="0 0 6", hfov=[20, 40, 2, 60, 1, 10][k], parallel=k in (2, 3), soft=soft)
        lines += [f"light {f(-3, 3)} {f(2, 5)} 6 1 1 1 1", "mtlcolor 0.7 0.5 0.3 1 1 1 0.2 0.7 0 20 1 1",
                  "texture textures/harbor.ppm" if k % 3 == 0 else "", "bump textures/bumps.ppm", f"sphere 0 0 0 {1 + 0.3 * k}"]
    elif case == "seam":
        # textured (and bumped) spheres seen by a 1-row camera level with their centres: nDir.y = +-0 exactly, and on
        # the left half nDir.x < 0, so atan2 is +-pi and u sits on the seam (theta < 0 wraps by 2 pi)
        w, h = [(33, 1), (31, 1), (17, 1), (9, 1), (41, 1), (13, 1)][k]
        y = "-0" if k % 2 else "0"
        lines = _camera(w, h, eye=f"0 {y} 6", parallel=k in (1, 4), soft=soft, hfov=60)
        lines += [f"light 4 {f(2, 6)} 5 1 1 1 1", "mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.2 20 1 1", "texture textures/harbor.ppm"]
        if k >= 3:
            lines.append("bump textures/bumps.ppm")
        lines += [f"sphere 0 {y} 0 1.5", "mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.2 20 1 1", "texture textures/harbor.ppm",
                  f"sphere -2.5 {y} -1 0.8"]
    elif case == "glass":
        # eta below the ambient's (total internal reflection from outside), eta equal to it (F0 = 0), and ordinary glass
        amb = ["1.0", "1.5", "1.0", "1.33", "1.0", "2.0"][k]
        eta = ["0.6", "1.0", "1.0", "1.33", "0.9", "1.5"][k]
        lines = _camera(40 + k, 30, eye="0 0.5 6", bkg=f"0.2 0.3 0.4 {amb}", soft=soft)
        lines += [f"light 3 {f(4, 7)} 5 1 1 1 1", f"mtlcolor 0.9 0.95 1 1 1 1 0.05 0.2 {f(0.2, 0.6)} 60 {f(0.1, 0.5)} {eta}",
                  "sphere 0 0 0 1.4", f"mtlcolor 0.9 0.95 1 1 1 1 0.05 0.2 0.3 60 0.2 {eta}", "sphere 2 0.5 -2 0.9",
                  "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1", "sphere -1 -0.5 -4 1.2", *_FLOOR]
    elif case == "alpha":
        # alpha = 0 (fully transparent), alpha = 1, ks = 0 (no reflection child)
        alpha, ks = [("0", "0.4"), ("1", "0.4"), ("0", "0"), ("1", "0"), ("0.5", "0"), ("0", "1")][k]
        lines = _camera(37, 23, eye="0 0.5 6", soft=soft)
        lines += [f"light -3 {f(4, 7)} 5 1 1 1 1", "attlight 3 5 4 1 0.5 0.5 0.5 0.3 0.05 0.01",
                  f"mtlcolor 0.9 0.6 0.4 1 1 1 0.1 0.5 {ks} 40 {alpha} 1.3", "sphere 0 0 0 1.3",
                  f"mtlcolor 0.3 0.6 0.9 1 1 1 0.1 0.5 {ks} 40 {alpha} 1.6", "sphere 1.8 0 -2 1",
                  "mtlcolor 0.8 0.8 0.2 1 1 1 0.2 0.7 0.1 10 1 1", "sphere -1.2 0 -4 1.2"]
        lines += _FLOOR
    elif case == "mirrors":
        # two facing mirrors: paths bounce to level 8 and meet the depth cut; a light avatar seen in them at depth
        w, h = [(24, 16), (33, 7), (16, 24), (21, 21), (40, 8), (9, 31)][k]
        lines = _camera(w, h, eye="0 0 0", viewdir=f"{f(-0.3, 0.3)} {f(-0.2, 0.2)} -1", hfov=70, soft=soft)
        lines += ["light 0 2 -1 1 1 1 1", "mtlcolor 1 1 1 1 1 1 1 1 1 0 1 1", "sphere 0 2 -1 0.3",
                  f"mtlcolor 0.7 0.75 0.8 1 1 1 0.05 0.1 {f(0.7, 0.95)} 80 1 1",
                  "v -4 -3 -3", "v 4 -3 -3", "v 4 3 -3", "v -4 3 -3", "f 1 2 3", "f 1 3 4",
                  "v -4 -3 1", "v 4 -3 1", "v 4 3 1", "v -4 3 1", "f 5 7 6", "f 5 8 7",
                  f"mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 {f(0.3, 1)} 1.4", f"sphere {f(-1, 1)} -1 -1 0.6"]
    elif case == "depthcue":
        # depth cueing with shaded points nearer than distmin, farther than distmax and in between
        dmin, dmax = [(4, 12), (6, 9), (3.5, 16), (8, 8.5), (5, 15), (3.6, 7)][k]
        lines = _camera(44, 26, eye="0 1 8", viewdir="0 -0.2 -1", soft=soft, parallel=k == 4)
        lines += [f"light 2 {f(5, 8)} 6 1 1 1 1", f"depthcueing 0.3 0.3 0.35 {f(0.8, 1)} {f(0.1, 0.4)} {dmax} {dmin}",
                  "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 30 1 1", "sphere -1 0 4 0.8", "sphere 1 0 -2 1",
                  "mtlcolor 0.9 0.95 1 1 1 1 0.05 0.2 0.4 60 0.3 1.4", "sphere 0 0.5 -8 1.5"]
        lines += _FLOOR
    elif case == "attlight":
        # attenuation off (c1 < 0), c1 = 0, and an ordinary attenuated light beside a directional one
        c1 = ["-1", "0", "-0.5", "0", "0.5", "-2"][k]
        lines = _camera(29, 19, eye="0 1 7", viewdir="0 -0.1 -1", soft=soft, parallel=k == 3)
        lines += [f"attlight {f(-3, 3)} {f(3, 6)} 3 1 1 0.9 0.8 {c1} {f(0, 0.2)} {f(0, 0.02)}",
                  f"attlight -4 4 -2 1 0.5 0.5 0.6 {c1} 0.1 0",
                  "light 0.3 -1 -0.4 0 0.3 0.3 0.25", "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 30 1 1", "sphere 0 0 0 1.1",
                  "mtlcolor 0.9 0.95 1 1 1 1 0.05 0.2 0.4 60 0.3 1.4", "sphere 1.8 0 -1.5 0.8"]
        lines += _FLOOR
    elif case == "tiles":
        # parallel projection, a 1x1 image and widths / heights that are not multiples of the 8x4 tile
        w, h = [(1, 1), (7, 3), (9, 5), (13, 7), (17, 1), (1, 9)][k]
        lines = _camera(w, h, eye="0 1 6", viewdir="0.05 -0.1 -1", hfov=40, parallel=k % 3 != 0, soft=soft)
        lines += [f"light 3 {f(4, 7)} 5 1 1 1 1", "light -0.4 -1 -0.2 0 0.4 0.4 0.4",
                  f"mtlcolor 0.9 0.95 1 1 1 1 0.05 0.2 {f(0.2, 0.5)} 60 0.3 1.4", "sphere 0 0.5 0 1.2",
                  "mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.2 20 1 1", "texture textures/harbor.ppm", "sphere 1.5 0 -2 1"]
        lines += _FLOOR
    else:
        raise ValueError(case)
    return "\n".join(x for x in lines if x) + "\n"


EDGE_CASES = ["pole", "seam", "glass", "alpha", "mirrors", "depthcue", "attlight", "tiles"]


def edge_is_met(case, scene, want_f, ost):
    """The oracle's render really meets the edge the scene was built for."""
    if case == "pole":
        return bool(np.isnan(want_f).any())
    if case == "seam":
        o, d = ob.OracleScene(scene).primary_rays()
        hits = ob.OracleScene(scene).trace_closest(o, d)
        nd = hits["ndir"]
        return bool(((hits["texture"] >= 0) & (nd[:, 1] == 0) & (nd[:, 0] < 0)).any())
    if case == "mirrors":
        return ost.rays_per_depth[8] > 0
    if case == "glass":
        return ost.rays_per_depth[1] > 0
    if case == "depthcue":
        o, d = ob.OracleScene(scene).primary_rays()
        hits = ob.OracleScene(scene).trace_closest(o, d)
        dist = np.linalg.norm(hits["pos"][hits["hit"] != 0] - np.array(scene.desc.eye, np.float32), axis=1)
        return bool((dist <= scene.desc.distmin).any() and (dist >= scene.desc.distmax).any()
                    and ((dist > scene.desc.distmin) & (dist < scene.desc.distmax)).any())
    return True


@pytest.mark.parametrize("case", EDGE_CASES)
def test_float_frame_shading_edges(workdir, case):
    for k in range(6):
        text = edge_scene(case, k)
        scene = Scene(text=text, asset_dir=workdir)
        want = oracle_float(scene)
        assert edge_is_met(case, scene, want[0], want[2]), (case, k, text)
        check_scene(scene, f"{case} variant {k}\n{text}", want=want)


# ---------------- frame configurations (read at wrt_create: a fresh context each) ----------------

CONFIG_SCENES = ["water_small", "water_soft", "spheres", "forty_lights"]


def _config_scene(workdir, name):
    if name == "forty_lights":
        return Scene(text=forty_lights(False), asset_dir=workdir)
    return load_golden_scene(workdir, name, kind="soft" if name == "water_soft" else "img")[0]


@pytest.mark.parametrize("env", ["WRT_SHADE0_SEPARATE=0", "WRT_SHADE0_SEPARATE=1", "WRT_DEEP_SPLIT=1", "WRT_DEEP_SPLIT=5",
                                 "WRT_DEEP_SPLIT=8", "WRT_UNLIT_CULL=0", "WRT_SHAFT_CULL=0", "WRT_SOFT_LISTS=0", "WRT_HOST_BVH=1"])
def test_float_frame_configurations(workdir, monkeypatch, env):
    key, value = env.split("=")
    for name in CONFIG_SCENES:
        scene = _config_scene(workdir, name)
        want = oracle_float(scene)
        monkeypatch.setenv(key, value)
        check_scene(scene, f"{name} with {env}", want=want)
        monkeypatch.delenv(key)


@pytest.mark.parametrize("soft", [False, True])
def test_float_frame_overflow(workdir, monkeypatch, soft):
    """The float copy follows every batch and every re-render: a 200x150 bunny frame in 4 batches of 8192 slots whose
    deep levels (queue_factor 0.02) overflow and are redone in halves, and the same frame as one batch that overflows
    and is redone in finish_frame.  A redone batch's copy replaces the overflowed attempt's."""
    name = f"float_overflow_{int(soft)}"
    fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(200, 150, soft=soft))
    scene = Scene.from_workdir(workdir, name)
    want_f, want_u8, ost = oracle_float(scene)
    for max_batch in ("8192", None):
        if max_batch:
            monkeypatch.setenv("WRT_MAX_BATCH", max_batch)
        r = Renderer(scene)
        for traversal in TRAVERSALS:
            r.ctx.set_options(traversal=traversal, queue_factor=0.02)
            fl, u8 = r.render_float()
            st = r.last_stats
            assert st["overflow_retries"] >= 1, (max_batch, st)
            assert np.array_equal(u8, quantize(fl))
            assert_bits_equal(fl, want_f, f"overflow, max_batch {max_batch}, traversal {traversal}")
            assert st["closest_rays"] == ost.closest_rays and st["shadow_rays"] == ost.shadow_rays
        r.ctx.close()
        if max_batch:
            monkeypatch.delenv("WRT_MAX_BATCH")


@pytest.mark.parametrize("name", ["spheres", "water_small", "bump"])
def test_float_frame_tiles(workdir, name):
    """Rank r of N writes exactly its own pixels and leaves the rest of the caller's float buffer untouched; the union
    over ranks equals the 1-rank float frame bit for bit (N = 1, 3, 8)."""
    scene, _ = load_golden_scene(workdir, name)
    r = Renderer(scene)
    full, full_u8 = r.render_float()
    full, full_u8 = full.copy(), full_u8.copy()
    h, w = full.shape[:2]
    sentinel = np.float32(-1234.5)
    for world in (1, 3, 8):
        merged = np.full_like(full, sentinel)
        owner = np.zeros((h, w), np.int32)
        for rank in range(world):
            r.ctx.set_tiles(rank=rank, world=world)
            mine = np.full_like(full, sentinel)
            mine_u8 = np.zeros_like(full_u8)
            r.render_float(out_f=mine, out=mine_u8)
            written = (mine != sentinel).any(axis=2)
            owner += written
            merged[written] = mine[written]
            assert np.array_equal(mine_u8[written], full_u8[written])
        assert (owner == 1).all(), (world, int((owner == 0).sum()), int((owner > 1).sum()))
        assert_bits_equal(merged, full, f"{name}: {world} ranks")
    r.ctx.set_tiles(rank=0, world=1)
    r.ctx.close()
