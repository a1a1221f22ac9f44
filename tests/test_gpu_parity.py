"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the
same inputs, against the reference's golden vectors, and — at BASELINE.json's full
sizes — through size-independent properties.

Bars (DESIGN.md section "Parity"):
  * closest hit (flag, object, t, position, normal, triangle uv), soft / directional
    shadow queries: bit-exact;
  * hard-shadow coefficient: bit-exact (the reference tree's association rebuilt from path codes, csrc/cuda/shadow_assoc.h)
    (the reference multiplies the (1-alpha) factors in BVH-tree association);
  * sphere uv (acos/atan2): <= 2 ulp;
  * images: within 1 LSB per channel on >= 99.9 % of pixels vs the reference (north star),
    and >= 99.99 % bit-identical vs the oracle (only powf's last ulp differs);
  * soft shadows vs the true reference: PSNR >= 30 dB against the reference's mean image.
"""
import ctypes as C
import subprocess

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import GOLD, IMG_SCENES, RAY_SCENES, SOFT_SCENES, REPO, image_diff, load_golden_scene, psnr, ulp_diff
from whittedstyle_raytracer_b200 import MultiRenderer, Renderer, Scene, fixtures, read_ppm_p3
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED

pytestmark = pytest.mark.gpu


def gpu_render(scene, traversal=TRAVERSAL_PRUNED, **tiles):
    r = Renderer(scene)
    r.ctx.set_options(traversal=traversal)
    if tiles:
        r.ctx.set_tiles(**tiles)
    img = r.render()
    st = r.last_stats
    r.ctx.close()
    return img, st


@pytest.mark.parametrize("traversal", [TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE])
@pytest.mark.parametrize("name", IMG_SCENES)
def test_image_matches_oracle_and_reference(workdir, name, traversal):
    scene, g = load_golden_scene(workdir, name)
    img, st = gpu_render(scene, traversal)
    ref, ost = ob.OracleScene(scene).render()
    d = image_diff(img, ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["within1"] >= 0.999 * d["n"], ("vs oracle", d)
    d = image_diff(img, g["rgb"])
    assert d["within1"] >= 0.999 * d["n"], ("vs reference golden", d)
    assert st["closest_rays"] == ost.closest_rays == int(g["closest_rays"])
    assert st["shadow_rays"] == ost.shadow_rays == int(g["shadow_rays"])
    assert st["rays_per_depth"] == [int(x) for x in ost.rays_per_depth]


def test_config_txt_800x600_pixel_gate(workdir):
    """BASELINE.json configs[0] — the PR1 gate: +-1 LSB on >= 99.9 % of the reference's pixels."""
    scene, g = load_golden_scene(workdir, "config_800x600")
    img, st = gpu_render(scene)
    d = image_diff(img, g["rgb"])
    assert d["within1"] >= 0.999 * d["n"], d
    assert d["exact"] >= 0.999 * d["n"], d
    assert (st["closest_rays"], st["shadow_rays"]) == (952311, 817273)


@pytest.mark.parametrize("name", RAY_SCENES)
def test_strategy_queries_match_oracle_and_reference(workdir, name):
    scene, _ = load_golden_scene(workdir, name)
    g = np.load(GOLD / f"rays_{name}.npz")
    orc = ob.OracleScene(scene)
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        h = r.interStrategy.UpdateInter(g["orig"], g["dir"])
        for ref in (orc.trace_closest(g["orig"], g["dir"]), g["hits"]):
            for k in ("hit", "object", "texture", "normalmap"):
                assert np.array_equal(h[k], ref[k]), (k, traversal)
            for k in ("t", "pos", "ndir"):
                assert np.array_equal(h[k].view(np.int32), ref[k].view(np.int32)), (k, traversal)
            assert ulp_diff(h["uv"], ref["uv"]).max() <= 2
        soft = r.interStrategy.getSoftShadowSample(g["sh_pos"], g["sh_ndir"], g["sh_light"])
        assert np.array_equal(soft, g["sh_soft"])
    hard = r.interStrategy.getShadowCoeffi(g["sh_pos"], g["sh_ndir"], g["sh_light"])
    assert np.array_equal(hard, g["sh_hard"])          # the reference's own tree-association product, bit for bit
    dirc = r.interStrategy.getDirectionalShadowCoeffi(g["sh_pos"], g["sh_self"], g["sh_ldir"])
    assert np.array_equal(dirc, g["sh_dir"])
    r.ctx.close()


def test_million_random_rays_bit_exact(workdir):
    """1e6 rays (uniform, surface-leaving, axis-parallel) through the bunny BVH: both GPU
    traversals equal the oracle's exhaustive recursive traversal bit for bit."""
    scene, _ = load_golden_scene(workdir, "water_small")
    rng = np.random.default_rng(11)
    n = 1_000_000
    o = rng.uniform(-4, 4, (n, 3)).astype(np.float32)
    o[:, 1] -= 1.0
    o[:, 2] -= 3.0
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[:3000] = np.eye(3, dtype=np.float32)[rng.integers(0, 3, 3000)]
    orc = ob.OracleScene(scene)
    ref = orc.trace_closest(o, d)
    hp = ref["pos"][ref["hit"] == 1]
    k = len(hp)
    o[-k:] = hp + 5e-5 * d[-k:]                      # secondary-ray-like origins on the surface
    ref = orc.trace_closest(o, d)
    assert 0.05 < ref["hit"].mean() < 0.95
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        # the batch query (binary tree, one ray per thread) and the frame's own deep-level kernel (octant copies, 4-wide
        # nodes, deferred leaves, lane refill: wrt_trace_closest_wavefront)
        for query in (r.interStrategy.UpdateInter, r.interStrategy.UpdateInterWavefront):
            h = query(o, d)
            for f in ("hit", "object", "prim"):
                assert np.array_equal(h[f], ref[f]), (f, traversal, query.__name__)
            for f in ("t", "pos", "ndir"):
                assert np.array_equal(h[f].view(np.int32), ref[f].view(np.int32)), (f, traversal, query.__name__)
    # shadow queries from the same points
    m = ref["hit"] == 1
    pos, nd = ref["pos"][m][:200000], ref["ndir"][m][:200000]
    lp = np.tile(np.array([[-20, 70, 20]], np.float32), (len(pos), 1))
    lp[::3] = rng.uniform(-25, 25, (len(lp[::3]), 3)).astype(np.float32)
    assert np.array_equal(r.interStrategy.getSoftShadowSample(pos, nd, lp), orc.shadow_soft(pos, nd, lp))
    hard, href = r.interStrategy.getShadowCoeffi(pos, nd, lp), orc.shadow_hard(pos, nd, lp)
    assert np.array_equal(hard, href)
    r.ctx.close()


@pytest.mark.parametrize("case", ["glass_row", "glass_bunny"])
def test_hard_shadow_association_matches_the_reference_golden(workdir, case):
    """The same property against the UNMODIFIED reference's own coefficients (tests/golden/assoc_<case>.npz, made by
    tools/gen_assoc_golden.py; the oracle is pinned to the same files in tests/test_oracle_vs_reference.py): 20 000 shadow
    rays along a row of six glass spheres of different alphas / through the glass bunny, bit for bit in both traversal
    modes (BVHStrategy::ShadowHelper, BVHStrategy.hpp:24-48)."""
    g = np.load(GOLD / f"assoc_{case}.npz", allow_pickle=False)
    fixtures.write_config(workdir, f"assoc_{case}", str(g["config"]))
    scene = Scene.from_workdir(workdir, f"assoc_{case}", bunny=bool(g["bunny"]))
    ref = g["hard"]
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        got = r.interStrategy.getShadowCoeffi(g["pos"], g["ndir"], g["light"])
        assert np.array_equal(got, ref), (traversal, int((got != ref).sum()))
    r.ctx.close()


def test_hard_shadow_product_has_the_reference_association(workdir):
    """BVHStrategy::ShadowHelper multiplies the (1 - alpha) factors in the association of the reference's tree (`l * r`,
    BVHStrategy.hpp:43-47); a stack walk multiplies in visit order, which differs in the last bits from the third crossing
    on (csrc/cuda/shadow_assoc.h rebuilds the reference's association from the primitives' path codes).  Shadow rays along
    a row of six glass spheres of different alphas — up to six different factors != 1 on a ray — must give the oracle's
    (= the reference recursion's) coefficient bit for bit in both traversal modes, through the batch query and through a
    rendered frame; so must rays through the glass bunny (equal factors: 0.8^4 already depends on the association)."""
    alphas = [0.1, 0.25, 0.4, 0.55, 0.7, 0.85]
    text = fixtures._CAMERA.format(w=160, h=120) + "light 8 0.2 -2 1 1 1 1\n"
    for k, a in enumerate(alphas):
        text += f"mtlcolor 0.8 0.8 0.9 1 1 1 0.2 0.6 0.3 20 {a} 1.3\nsphere {-3 + k} 0 -2 0.42\n"
    text += "mtlcolor 0.7 0.7 0.7 1 1 1 0.2 0.8 0.0 10 1 1\nv -12 -0.6 6\nv 12 -0.6 6\nv 12 -0.6 -14\nv -12 -0.6 -14\nf 1 2 3\nf 1 3 4\n"
    fixtures.write_config(workdir, "glass_row", text)
    scene = Scene.from_workdir(workdir, "glass_row")
    rng = np.random.default_rng(5)
    n = 200_000
    pos = np.stack([rng.uniform(-6, 3.5, n), rng.uniform(-0.4, 0.4, n), rng.uniform(-2.4, -1.6, n)], 1).astype(np.float32)
    nd = rng.normal(size=(n, 3)).astype(np.float32)
    nd /= np.linalg.norm(nd, axis=1, keepdims=True)
    lp = np.stack([np.full(n, 8.0), rng.uniform(-0.4, 0.4, n), rng.uniform(-2.4, -1.6, n)], 1).astype(np.float32)
    orc = ob.OracleScene(scene)
    ref = orc.shadow_hard(pos, nd, lp)
    assert len(np.unique(ref)) > 30 and ((ref > 0) & (ref < 0.1)).mean() > 0.3       # many rays cross many spheres
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        got = r.interStrategy.getShadowCoeffi(pos, nd, lp)
        assert np.array_equal(got, ref), (traversal, int((got != ref).sum()), int(ulp_diff(got, ref).max()))
        img = r.render()
        oimg, ost = orc.render()
        d = image_diff(img, oimg)
        assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, (traversal, d)
        assert r.last_stats["shadow_rays"] == ost.shadow_rays
    r.ctx.close()
    # the glass bunny: shadow rays from behind it towards the light
    scene, _ = load_golden_scene(workdir, "water_small")
    orc = ob.OracleScene(scene)
    m = 100_000
    lp = np.tile(np.array([[-20, 70, 20]], np.float32), (m, 1))
    target = np.stack([rng.uniform(-1.2, 1.2, m), rng.uniform(-1.0, 1.2, m), rng.uniform(-3.2, -1.2, m)], 1)
    dirs = target - lp
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    pos = (target + dirs * rng.uniform(2.0, 6.0, (m, 1))).astype(np.float32)       # beyond the bunny, seen from the light
    nd = (-dirs).astype(np.float32)
    ref = orc.shadow_hard(pos, nd, lp)
    a4 = np.float32(0.8) * np.float32(0.8) * np.float32(0.8) * np.float32(0.8)
    assert ((ref > 0) & (ref <= a4)).mean() > 0.02                                  # rays with four and more crossings
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        got = r.interStrategy.getShadowCoeffi(pos, nd, lp)
        assert np.array_equal(got, ref), (traversal, int((got != ref).sum()))
    r.ctx.close()


def test_adversarial_rays_pruned_equals_exhaustive(workdir):
    """The pruned closest-hit walk skips boxes entered beyond t_best*(1+1e-3)+1e-3 (DESIGN.md section 4).  Rays built to
    stress that margin (ADVICE r1): aimed at points on and up to 2e-5 edge lengths OUTSIDE triangle edges and vertices
    (Triangle.hpp:41 accepts barycentrics down to -1e-5, so such hits lie outside the triangle and can lie outside its box),
    from grazing directions (down to 1e-4 rad off the triangle's plane), from origins on the plane itself, and
    through the 40-unit wall triangles whose slack is 4e-4 units.  Both traversals must equal the oracle's exhaustive
    recursive walk bit for bit."""
    scene, _ = load_golden_scene(workdir, "water_small")
    d = scene.desc
    geom = np.ctypeslib.as_array(d.prim_geom, shape=(d.n_prims, 12)).copy()
    rng = np.random.default_rng(23)
    n = 400_000
    prim = rng.integers(0, d.n_prims, n)
    big = np.argsort(-(np.linalg.norm(geom[:, 4:7], axis=1) + np.linalg.norm(geom[:, 8:11], axis=1)))[:4]
    prim[: n // 4] = big[rng.integers(0, len(big), n // 4)]       # a quarter of the rays at the largest triangles (the walls)
    v0, e1, e2 = geom[prim, 0:3], geom[prim, 4:7], geom[prim, 8:11]
    # barycentric targets: on edges / vertices, pushed outside by 0 .. 2e-5
    kind = rng.integers(0, 4, n)
    a = rng.random(n)
    eps = rng.choice([0.0, 5e-6, 9e-6, 1.1e-5, 2e-5], n) * rng.choice([1.0, -1.0], n)
    b1 = np.where(kind == 0, a, np.where(kind == 1, eps, np.where(kind == 2, a, rng.choice([0.0, 1.0], n))))
    b2 = np.where(kind == 0, eps, np.where(kind == 1, a, np.where(kind == 2, 1 - a + eps, rng.choice([0.0, 1.0], n) * 0 + eps)))
    target = v0 + b1[:, None] * e1 + b2[:, None] * e2
    nrm = np.cross(e1, e2)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    tang = e1 / np.maximum(np.linalg.norm(e1, axis=1, keepdims=True), 1e-30)
    phi = rng.random(n) * 2 * np.pi
    inplane = np.cos(phi)[:, None] * tang + np.sin(phi)[:, None] * np.cross(nrm, tang)
    graze = rng.choice([1e-4, 1e-3, 1e-2, 0.1, 1.0], n)               # elevation over the triangle's plane (rad)
    direction = np.cos(graze)[:, None] * inplane + np.sin(graze)[:, None] * nrm * rng.choice([1.0, -1.0], n)[:, None]
    dist = rng.choice([0.0, 1e-5, 1e-3, 0.5, 5.0, 30.0], n)          # 0: the origin lies on the target itself
    o = (target - dist[:, None] * direction).astype(np.float32)
    dd = direction.astype(np.float32)
    dd /= np.linalg.norm(dd, axis=1, keepdims=True)
    orc = ob.OracleScene(scene)
    ref = orc.trace_closest(o, dd)
    assert 0.2 < ref["hit"].mean() <= 1.0
    r = Renderer(scene)
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        r.ctx.set_options(traversal=traversal)
        for query in (r.interStrategy.UpdateInter, r.interStrategy.UpdateInterWavefront):
            h = query(o, dd)
            for f in ("hit", "object", "prim"):
                assert np.array_equal(h[f], ref[f]), (f, traversal, query.__name__, int((h[f] != ref[f]).sum()))
            for f in ("t", "pos", "ndir"):
                assert np.array_equal(h[f].view(np.int32), ref[f].view(np.int32)), (f, traversal, query.__name__)
    r.ctx.close()


@pytest.mark.parametrize("name", SOFT_SCENES)
def test_soft_shadows(workdir, name):
    """Same counter RNG on both sides: GPU == oracle bit for bit; both agree with the
    non-deterministic reference in the mean image (PSNR gate 30 dB)."""
    scene, g = load_golden_scene(workdir, name, kind="soft")
    img, st = gpu_render(scene)
    ref, ost = ob.OracleScene(scene).render()
    d = image_diff(img, ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
    assert psnr(img, g["mean_rgb"]) >= 30.0
    assert st["shadow_rays"] == ost.shadow_rays == int(g["shadow_rays"])
    img2, _ = gpu_render(scene, TRAVERSAL_EXHAUSTIVE)
    assert np.array_equal(img, img2)                 # deterministic, traversal-independent
    r = Renderer(scene)
    r.ctx.set_options(seed=1234)
    other = r.render()
    assert not np.array_equal(other, img) and psnr(other, g["mean_rgb"]) >= 30.0
    r.ctx.close()


@pytest.mark.parametrize("name,world,tile", [("water_small", 2, (32, 16)), ("spheres", 3, (8, 4)), ("smooth", 8, (64, 32))])
def test_tile_sharding_is_rank_count_invariant(workdir, name, world, tile):
    """N-rank interleaved tiles (each rank rendered on this one GPU in turn) reassemble
    into exactly the 1-rank image, via host buffers and via the packed device path +
    rank-0 scatter kernel that follows the NCCL gather."""
    import torch
    scene, _ = load_golden_scene(workdir, name)
    full, st_full = gpu_render(scene)
    h, w = full.shape[:2]
    merged = np.zeros_like(full)
    r = Renderer(scene)
    r.ctx.set_tiles(tile_w=tile[0], tile_h=tile[1], rank=0, world=world)
    counts = [r.ctx.tile_pixel_count(k, world) for k in range(world)]
    stride = max(counts) * 3
    gathered = torch.zeros(world * stride, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rays = 0
    for k in range(world):
        r.ctx.set_tiles(tile_w=tile[0], tile_h=tile[1], rank=k, world=world)
        r.render(out=merged)                          # only rank k's pixels are written
        part = gathered[k * stride:(k + 1) * stride]
        r.render_device(part.data_ptr())
        rays += r.finish_device()["rays"]
    assert np.array_equal(merged, full)
    assert rays == st_full["rays"]
    r.ctx.set_tiles(tile_w=tile[0], tile_h=tile[1], rank=0, world=world)
    image = torch.zeros(h * w * 3, dtype=torch.uint8, device="cuda")
    r.scatter_tiles(gathered.data_ptr(), world, stride, image.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(image.cpu().numpy().reshape(h, w, 3), full)
    r.ctx.close()


def test_queue_overflow_is_rerendered_not_dropped(workdir):
    """Eye inside a glass ball: every primary hit spawns a reflection and a transmission,
    so level 1 holds ~2x the primary rays.  With queue_factor 1 the level overflows; the
    frame must come out identical (re-rendered in halves), with the retry reported."""
    text = """imsize 160 96
eye 0 0 0
viewdir 0 0 -1
hfov 80
updir 0 1 0
bkgcolor 0.2 0.3 0.5 1.0
light 3 4 2 1 1 1 1
mtlcolor 0.9 0.9 1 1 1 1 0.1 0.2 0.4 50 0.1 1.5
sphere 0 0 0 2
mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 20 1 1
sphere 0 0 -6 1.5
sphere 4 1 -5 1.5
"""
    scene = Scene(text=text, asset_dir=workdir)
    ref, ost = ob.OracleScene(scene).render()
    r = Renderer(scene)
    r.ctx.set_options(queue_factor=4.0)
    img = r.render()
    assert r.last_stats["overflow_retries"] == 0
    assert r.last_stats["rays_per_depth"][1] > 1.5 * 160 * 96
    r.ctx.set_options(queue_factor=1.0)
    img2 = r.render()
    assert r.last_stats["overflow_retries"] >= 1
    assert np.array_equal(img, img2)
    assert r.last_stats["closest_rays"] == ost.closest_rays and r.last_stats["shadow_rays"] == ost.shadow_rays
    d = image_diff(img, ref)
    assert d["exact"] >= 0.9999 * d["n"], d
    r.ctx.close()


_BANK_LIGHTS = ["light 3 6 4 1 0.3 0.3 0.3", "light 0.3 -1 -0.4 0 0.3 0.3 0.25", "attlight 1 7 7 1 0.4 0.4 0.4 0.5 0.02 0.001",
                "light -4 5 3 1 0.3 0.2 0.2", "light -0.5 -1 0.3 0 0.2 0.3 0.2"]


def light_bank(n, soft):
    """The first n of a mix of point, attenuated and directional lights over two spheres (one glass) and a floor: the
    kernels keep WRT_INLINE_LIGHTS = 4 lights in their parameters and read the rest from global memory."""
    return ("imsize 96 64\neye 0 1 6\nviewdir 0 -0.1 -1\nhfov 60\nupdir 0 1 0\nbkgcolor 0.1 0.1 0.2 1.0\n"
            + ("shadow soft\n" if soft else "") + "\n".join(_BANK_LIGHTS[:n]) + "\n"
            + "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.6 0.3 24 1 1.5\nsphere -1.5 0 -1 1.2\n"
            + "mtlcolor 0.9 0.9 1.0 1 1 1 0.05 0.2 0.4 60 0.2 1.4\nsphere 1.4 0.2 0.5 1.0\n"
            + "mtlcolor 0.4 0.7 0.4 1 1 1 0.2 0.7 0.1 10 1 1.0\n"
            + "v -10 -1.2 8\nv 10 -1.2 8\nv 10 -1.2 -12\nv -10 -1.2 -12\nf 1 2 3\nf 1 3 4\n")


EDGE_SCENES = [
    ("imsize 7 5\neye 0 0 0\nviewdir 0 0 -1\nupdir 0 1 0\nhfov 60\nbkgcolor 0.5 0.25 1 1\n", "empty"),
    ("imsize 33 17\neye 0 0 0\nviewdir 0 0 -1\nupdir 0 1 0\nhfov 60\nbkgcolor 0.1 0.1 0.1 1\nlight 1 1 1 1 1 1 1\n"
     "mtlcolor 0.8 0.4 0.2 1 1 1 0.3 0.6 0.2 10 1 1\nsphere 0 0 -3 1\n", "one object (root is a leaf)"),
    ("imsize 1 1\neye 0 0 0\nviewdir 0 0 -1\nupdir 0 1 0\nhfov 60\nbkgcolor 0.1 0.1 0.1 1\nlight 1 1 1 1 1 1 1\nshadow soft\n"
     "mtlcolor 0.8 0.4 0.2 1 1 1 0.3 0.6 0.2 10 0.5 1.3\nsphere 0 0 -3 1\nsphere 0.5 0 -5 1\n", "two objects, 1x1 image, soft"),
    ("imsize 40 30\neye 0 0 0\nviewdir 0 0 -1\nupdir 0 1 0\nhfov 60\nbkgcolor 0.1 0.1 0.1 1\nlight 0 5 -3 1 1 1 1\nshadow soft\n"
     "mtlcolor 1 1 1 1 1 1 1 1 1 0 1 1\nsphere 0 5 -3 0.5\nmtlcolor 0.8 0.4 0.2 1 1 1 0.3 0.6 0.2 10 1 1\n"
     "sphere 0 0 -4 1\nv -5 -1 0\nv 5 -1 0\nv 0 -1 -9\nf 1 2 3\n", "light avatar + soft shadows (literal hasIntersection path)"),
    (light_bank(4, soft=False), "4 lights, point and directional: the whole kernel-parameter light bank"),
    (light_bank(5, soft=False), "5 lights: the 5th (directional) read from global memory"),
]


@pytest.mark.parametrize("text,expect", EDGE_SCENES)
def test_edge_scenes(workdir, text, expect):
    scene = Scene(text=text, asset_dir=workdir)
    ref, ost = ob.OracleScene(scene).render()
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        img, st = gpu_render(scene, traversal)
        d = image_diff(img, ref)
        assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, (expect, d)
        assert st["closest_rays"] == ost.closest_rays and st["shadow_rays"] == ost.shadow_rays, expect


def test_directional_light_on_bunny(workdir):
    """Directional shadows are a box-free O(N) loop in the reference (Renderer.hpp:381-400).  The GPU
    culls through the dilated tree and multiplies the accepted (1-alpha) factors in objList order:
    must equal the literal loop (oracle; GPU 'exhaustive' batch mode) bit for bit on the 4970-triangle
    bunny, including the translucent crossings."""
    text = fixtures.water_bunny_tex_config(160, 120).replace("light -20 70 20 1 1 1 1", "light -20 70 20 1 1 1 1\nlight 0.3 -1 -0.4 0 0.9 0.9 0.8")
    fixtures.write_config(workdir, "dirbunny", text)
    scene = Scene.from_workdir(workdir, "dirbunny")
    assert scene.desc.n_lights == 2
    ref, ost = ob.OracleScene(scene).render()
    img, st = gpu_render(scene)
    d = image_diff(img, ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
    assert st["shadow_rays"] == ost.shadow_rays
    # batch query: culled vs literal loop vs oracle on rays from the bunny's own surface
    orc = ob.OracleScene(scene)
    o, dd = orc.primary_rays()
    h = orc.trace_closest(o, dd)
    m = h["hit"] == 1
    pos, obj = h["pos"][m], h["object"][m]
    rng = np.random.default_rng(3)
    ldir = np.zeros((len(pos), 4), np.float32)
    ldir[:, :3] = rng.normal(size=(len(pos), 3))
    ldir[::5, 0] = 0.0                                  # some axis-degenerate directions
    ldir[::7, 1] = -0.0
    want = orc.shadow_directional(pos, obj, ldir)
    r = Renderer(scene)
    got = r.interStrategy.getDirectionalShadowCoeffi(pos, obj, ldir)
    r.ctx.set_options(traversal=TRAVERSAL_EXHAUSTIVE)
    literal = r.interStrategy.getDirectionalShadowCoeffi(pos, obj, ldir)
    r.ctx.close()
    assert np.array_equal(literal, want)
    assert np.array_equal(got, want)
    assert 0.02 < (want < 1).mean() < 0.98


def test_large_triangle_soup(workdir):
    """60 000 random triangles (12x the bunny): thread-parallel SAH build, deeper trees and stacks.
    GPU image == oracle (which walks the reference-topology tree exhaustively, ~250 box tests per ray)."""
    rng = np.random.default_rng(5)
    n = 60000
    c = rng.uniform(-8, 8, (n, 3))
    c[:, 2] -= 6
    lines = ["imsize 200 150", "eye 0 1 10", "viewdir 0 -0.1 -1", "hfov 60", "updir 0 1 0", "bkgcolor 0.2 0.3 0.5 1.0",
             "light 5 20 10 1 1 1 1", "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 0.6 1.3"]
    tri = c[:, None, :] + rng.uniform(-0.12, 0.12, (n, 3, 3))
    lines += ["v %.4f %.4f %.4f" % tuple(q) for q in tri.reshape(-1, 3)]
    lines += ["f %d %d %d" % (3 * i + 1, 3 * i + 2, 3 * i + 3) for i in range(n)]
    scene = Scene(text="\n".join(lines) + "\n", asset_dir=workdir)
    assert scene.n_prims == n
    ref, ost = ob.OracleScene(scene).render()
    for traversal in (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE):
        img, st = gpu_render(scene, traversal)
        d = image_diff(img, ref)
        assert d["exact"] >= 0.999 * d["n"] and d["within1"] >= 0.9999 * d["n"], (traversal, d)
        assert st["closest_rays"] == ost.closest_rays and st["shadow_rays"] == ost.shadow_rays


def test_render_is_deterministic_and_reusable(workdir):
    scene, _ = load_golden_scene(workdir, "water_small")
    r = Renderer(scene)
    a = r.render().copy()
    scene.set_imsize(97, 61)                         # not a multiple of the tile size
    r.ctx.set_camera(scene)
    small = r.render()
    ref, _ = ob.OracleScene(scene).render()
    assert image_diff(small, ref)["exact"] >= 0.9999 * 97 * 61
    scene.set_imsize(200, 150)
    r.ctx.set_camera(scene)
    assert np.array_equal(r.render(), a)
    assert r.ctx.launches > 0
    r.ctx.close()


def test_drop_in_executable(workdir):
    """`wrt <config>` in a cwd holding bunny.obj + textures writes the same P3 file the
    reference's executable would (here: the oracle's pixels through the same writer)."""
    exe = REPO / "whittedstyle_raytracer_b200" / "wrt"
    fixtures.write_config(workdir, "cli_scene", fixtures.bunny_shadow_config(120, 90))
    p = subprocess.run([str(exe), "cli_scene.txt"], cwd=workdir, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "Generating is done successfully!" in p.stdout and "Rendering Time consumed" in p.stdout
    got = read_ppm_p3(workdir / "cli_scene.ppm")
    scene = Scene.from_workdir(workdir, "cli_scene")
    ref, _ = ob.OracleScene(scene).render()
    assert image_diff(got, ref)["exact"] >= 0.9999 * 120 * 90
    text = (workdir / "cli_scene.ppm").read_text()
    assert text.startswith("P3\n120\n90\n255\n") and text.count("\n") == 4 + 120 * 90
    (workdir / "bad.txt").write_text("imsize 4 4\nfoo 1\n")
    p = subprocess.run([str(exe), "bad.txt"], cwd=workdir, capture_output=True, text=True)
    assert p.returncode == 255 and "ERROR: extraneous string in the input file" in p.stdout


def test_reference_renderer_with_cuda_strategy(workdir):
    """INTEGRATION.md level A: the reference's UNMODIFIED main.cpp / Renderer with
    integration/CudaStrategy.hpp plugged in at IIntersectStrategy (built by build() with
    WRT_REFERENCE_DIR set, through `make -C oracle ref_cuda`) — every UpdateInter / getShadowCoeffi call of the reference's own
    recursion runs on the GPU.  Its PPM must equal the stock reference executable's."""
    strat, stock = ob.REF_EXE.parent / "whitted_ref_cuda_strategy", ob.REF_EXE
    if not (strat.exists() and stock.exists()):
        pytest.skip("oracle/_ref executables not built (build() with WRT_REFERENCE_DIR set)")
    fixtures.write_config(workdir, "plug", fixtures.bunny_shadow_config(64, 48))
    out = {}
    for name, exe in (("stock", stock), ("cuda", strat)):
        p = subprocess.run([str(exe), "plug.txt"], cwd=workdir, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        out[name] = read_ppm_p3(workdir / "plug.ppm")
        (workdir / "plug.ppm").unlink()
    d = image_diff(out["cuda"], out["stock"])
    assert d["exact"] >= 0.999 * d["n"] and d["within1"] == d["n"], d


# ---------------- BASELINE.json full sizes: size-independent properties ----------------

FULL = [("bunny_shadow_4k", 17959375, 15256192), ("gla_bunny_tex_4k", 17959375, 14487729)]


@pytest.mark.parametrize("name,closest,shadow", FULL)
def test_4k_hard_shadow_configs(workdir, name, closest, shadow):
    """3840x2160: ray counts equal the reference's own (SURVEY.md section 3.3, measured with the
    instrumented reference); a 1/16 x 1/16 pixel sample equals the oracle; pruned == exhaustive;
    a 4-rank tile split reassembles into the same frame."""
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name)
    r = Renderer(scene)
    img = r.render().copy()
    assert (r.last_stats["closest_rays"], r.last_stats["shadow_rays"]) == (closest, shadow)
    sample, _ = ob.OracleScene(scene).render(stride=(16, 16))
    d = image_diff(img[::16, ::16], sample[::16, ::16])
    assert d["exact"] >= 0.9995 * d["n"] and d["within1"] >= 0.999 * d["n"], d
    r.ctx.set_options(traversal=TRAVERSAL_EXHAUSTIVE)
    assert np.array_equal(r.render(), img)
    r.ctx.set_options(traversal=TRAVERSAL_PRUNED)
    merged = np.zeros_like(img)
    for k in range(4):
        r.ctx.set_tiles(rank=k, world=4)
        r.render(out=merged)
    assert np.array_equal(merged, img)
    r.ctx.close()


def test_4k_soft_shadow_config(workdir):
    """water_bunny_tex + shadow soft at 3840x2160 (BASELINE.json's metric config): 742,345,825 rays
    like the reference; a strided pixel sample equals the oracle (same RNG keys at full size)."""
    name = "water_bunny_tex_soft_4k"
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name)
    r = Renderer(scene)
    img = r.render()
    assert (r.last_stats["closest_rays"], r.last_stats["shadow_rays"]) == (17959375, 724386450)
    sample, _ = ob.OracleScene(scene).render(stride=(48, 40))
    d = image_diff(img[::40, ::48], sample[::40, ::48])
    assert d["exact"] >= 0.999 * d["n"] and d["max"] <= 1, d
    r.ctx.close()


def test_4k_soft_contiguous_crop_through_the_bunny(workdir):
    """The same frame: a contiguous 256x256 window through the bunny's body (where the deep ray-tree levels, the
    candidate lists and the per-ray fall-backs all do their work) equals the oracle's render of that window with the
    full-size camera and RNG keys."""
    name = "water_bunny_tex_soft_4k"
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name)
    img, _ = gpu_render(scene)
    x0, y0, n = 1500, 1700, 256
    ref, ost = ob.OracleScene(scene).render(rows=(y0, y0 + n), cols=(x0, x0 + n))
    assert ost.closest_rays > 3 * n * n                      # the window really is on the glass bunny
    d = image_diff(img[y0:y0 + n, x0:x0 + n], ref[y0:y0 + n, x0:x0 + n])
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d


def test_8k_soft_shadow_config(workdir):
    """BASELINE.json configs[4]: glass bunny + shadow soft at 7680x4320, one 33 M-slot batch.  Against the oracle's full
    8K render (tests/golden/full_glass_bunny_soft_8k.npz, tools/gen_full_frame_golden.py: ~10 CPU-minutes, done once):
    ray counts per depth, every 16th pixel, per-band channel sums of the whole image; a 192x192 window through the bunny
    against the oracle run here; pruned == exhaustive; an 8-rank tile split reassembles into the 1-rank frame."""
    name = "glass_bunny_soft_8k"
    g = np.load(GOLD / f"full_{name}.npz")
    fixtures.write_config(workdir, name, str(g["config"]))
    scene = Scene.from_workdir(workdir, name, glass=True)
    r = Renderer(scene)
    img = r.render().copy()
    st = r.last_stats
    assert st["overflow_retries"] == 0
    assert (st["closest_rays"], st["shadow_rays"]) == (int(g["closest_rays"]), int(g["shadow_rays"])) == (74904376, 2961802900)
    assert st["rays_per_depth"] == [int(x) for x in g["rays_per_depth"]]
    k = int(g["sample_stride"])
    d = image_diff(img[::k, ::k], g["sample"])
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
    b = int(g["band_rows"])
    bands = img.reshape(img.shape[0] // b, b, img.shape[1], 3).astype(np.int64).sum(axis=(1, 2))
    assert np.abs(bands - g["band_sums"]).sum() <= 1e-4 * img.shape[0] * img.shape[1], "whole-frame band sums vs the oracle"
    x0, y0, n = 3100, 3500, 192
    ref, _ = ob.OracleScene(scene).render(rows=(y0, y0 + n), cols=(x0, x0 + n))
    d = image_diff(img[y0:y0 + n, x0:x0 + n], ref[y0:y0 + n, x0:x0 + n])
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
    merged = np.zeros_like(img)
    rays = 0
    for kk in range(8):
        r.ctx.set_tiles(rank=kk, world=8)
        r.render(out=merged)
        rays += r.last_stats["rays"]
    assert np.array_equal(merged, img) and rays == st["rays"]
    r.ctx.set_tiles(rank=0, world=1)
    r.ctx.set_options(traversal=TRAVERSAL_EXHAUSTIVE)
    assert np.array_equal(r.render(), img)
    r.ctx.close()


@pytest.mark.parametrize("soft", [False, True])
def test_multi_batch_frames_with_overflow(workdir, monkeypatch, soft):
    """The batch scheduler (frames larger than one batch; 8K frames used to need it, WRT_MAX_BATCH forces it here): a
    200x150 bunny frame cut into 4 batches of 8192 slots, with deep levels so small (queue_factor 0.02) that batches
    overflow and are re-rendered in halves — image, ray counts and per-depth counts equal the single-batch frame's.
    Then the automatic sizing: deep levels start at WRT_DEEP_FACTOR=0.01 of the batch, overflow, grow, same frame."""
    name = f"multibatch_{int(soft)}"
    fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(200, 150, soft=soft))
    scene = Scene.from_workdir(workdir, name)
    one, st_one = gpu_render(scene)
    assert st_one["overflow_retries"] == 0
    monkeypatch.setenv("WRT_MAX_BATCH", "8192")
    r = Renderer(scene)
    many = r.render().copy()
    st_many = dict(r.last_stats)
    r.ctx.set_options(queue_factor=0.02)
    tight = r.render().copy()
    st_tight = dict(r.last_stats)
    r.ctx.close()
    monkeypatch.setenv("WRT_DEEP_FACTOR", "0.01")
    monkeypatch.setenv("WRT_MAX_BATCH", "16384")
    r = Renderer(scene)
    auto = r.render().copy()
    st_auto = dict(r.last_stats)
    again = r.render().copy()                                  # the grown buffers are kept: no retry the second time
    st_again = dict(r.last_stats)
    r.ctx.close()
    monkeypatch.delenv("WRT_MAX_BATCH")
    monkeypatch.delenv("WRT_DEEP_FACTOR")
    assert st_many["overflow_retries"] == 0 and st_tight["overflow_retries"] >= 1
    for img, st in ((many, st_many), (tight, st_tight), (auto, st_auto), (again, st_again)):
        assert np.array_equal(img, one)
        for k in ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth", "shadow_rays_traced"):
            assert st[k] == st_one[k], k
    ref, ost = ob.OracleScene(scene).render()
    d = image_diff(one, ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d


def test_device_frame_overflow_is_rerendered_in_finish(workdir):
    """wrt_render_device / wrt_finish_device (the multi-GPU path): a rank whose frame overflows a queue re-renders it
    inside wrt_finish_device and reports the retry, so that the caller repeats the gather (parallel.py).  Three
    'ranks' rendered in turn on this GPU with deep levels fixed at 2 % of the batch."""
    import torch
    scene, _ = load_golden_scene(workdir, "water_small")
    full, st_full = gpu_render(scene)
    h, w = full.shape[:2]
    world = 3
    r = Renderer(scene)
    r.ctx.set_options(queue_factor=0.02)
    r.ctx.set_tiles(rank=0, world=world)
    stride = max(r.ctx.tile_pixel_count(k, world) for k in range(world)) * 3
    gathered = torch.zeros(world * stride, dtype=torch.uint8, device="cuda")
    rays, retries = 0, 0
    for k in range(world):
        r.ctx.set_tiles(rank=k, world=world)
        r.render_device(gathered[k * stride:(k + 1) * stride].data_ptr(), torch.cuda.current_stream().cuda_stream)
        st = r.finish_device()
        rays += st["rays"]
        retries += st["overflow_retries"]
    assert retries >= world and rays == st_full["rays"]
    r.ctx.set_tiles(rank=0, world=world)
    image = torch.zeros(h * w * 3, dtype=torch.uint8, device="cuda")
    r.scatter_tiles(gathered.data_ptr(), world, stride, image.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(image.cpu().numpy().reshape(h, w, 3), full)
    r.ctx.close()


def test_request_culling_changes_the_work_not_the_result(workdir, monkeypatch):
    """Shadow requests that cannot change the image are answered without tracing: soft-shadow requests
    whose whole shaft to the area light misses every leaf box (50 lit samples, shaft_cull.h) and lights
    whose diffuse and specular factors are exactly 0 at the point (dev_shade.cuh).  Same image, same ray
    counts (the reference traces those rays, so they are counted), and the oracle — which traces all of
    them — agrees.  Soft and hard shadows."""
    for soft in (True, False):
        name = f"cull_640_{int(soft)}"
        fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(640, 360, soft=soft))
        scene = Scene.from_workdir(workdir, name)
        on, st_on = gpu_render(scene)
        for k in ("WRT_SHAFT_CULL", "WRT_UNLIT_CULL", "WRT_SOFT_LISTS"):     # read by wrt_create; lists off too: an
            monkeypatch.setenv(k, "0")                                       # empty candidate list also answers "lit"
        off, st_off = gpu_render(scene)
        for k in ("WRT_SHAFT_CULL", "WRT_UNLIT_CULL", "WRT_SOFT_LISTS"):
            monkeypatch.delenv(k)
        assert np.array_equal(on, off)
        assert st_off["shaft_culled_requests"] == 0 and st_off["unlit_skipped_requests"] == 0
        assert st_off["shadow_rays_traced"] == st_off["shadow_rays"]
        assert st_on["unlit_skipped_requests"] > 0.02 * st_on["shadow_requests"]
        if soft:
            assert st_on["shaft_culled_requests"] > 0.25 * st_on["shadow_requests"]
        per = 50 if soft else 1
        assert st_on["shadow_rays_traced"] == st_on["shadow_rays"] - per * (st_on["shaft_culled_requests"] + st_on["unlit_skipped_requests"])
        for k in ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth"):
            assert st_on[k] == st_off[k], k
        ref, ost = ob.OracleScene(scene).render()
        d = image_diff(on, ref)
        assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
        assert st_on["shadow_rays"] == ost.shadow_rays


def test_candidate_list_pruning_changes_the_work_not_the_result(workdir, monkeypatch):
    """k_soft_filter drops from every candidate list the triangles no sample ray of the request can hit
    (shaft_cull.h wrt_pyramid_*): same image with the pruning off (0), on the deep queues (1, default) and on every
    queue (2); fewer rays traced (requests whose list empties need none) and the reference-equivalent counts unchanged."""
    name = "prune_640"
    fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(640, 360, soft=True))
    scene = Scene.from_workdir(workdir, name)
    out = {}
    for mode in ("0", "1", "2"):
        monkeypatch.setenv("WRT_SOFT_FILTER", mode)
        out[mode] = gpu_render(scene)
    monkeypatch.delenv("WRT_SOFT_FILTER")
    for mode in ("1", "2"):
        assert np.array_equal(out[mode][0], out["0"][0]), mode
        for k in ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth"):
            assert out[mode][1][k] == out["0"][1][k], (mode, k)
    assert out["1"][1]["shadow_rays_traced"] < out["0"][1]["shadow_rays_traced"]
    assert out["2"][1]["shadow_rays_traced"] <= out["1"][1]["shadow_rays_traced"]
    ref, ost = ob.OracleScene(scene).render()
    d = image_diff(out["1"][0], ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d


MANY_LIGHTS = """imsize 96 64
eye 0 1 6
viewdir 0 -0.1 -1
hfov 60
updir 0 1 0
bkgcolor 0.1 0.1 0.2 1.0
shadow soft
light 3 6 4 1 0.3 0.3 0.3
light -4 5 3 1 0.3 0.2 0.2
light 0 8 -2 1 0.2 0.3 0.2
light 6 2 6 1 0.2 0.2 0.3
light -6 3 -4 1 0.3 0.3 0.1
attlight 1 7 7 1 0.4 0.4 0.4 0.5 0.02 0.001
mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.6 0.3 24 1 1.5
sphere -1.5 0 -1 1.2
mtlcolor 0.9 0.9 1.0 1 1 1 0.05 0.2 0.4 60 0.2 1.4
sphere 1.4 0.2 0.5 1.0
mtlcolor 0.4 0.7 0.4 1 1 1 0.2 0.7 0.1 10 1 1.0
v -10 -1.2 8
v 10 -1.2 8
v 10 -1.2 -12
v -10 -1.2 -12
f 1 2 3
f 1 3 4
"""

AXIS_ALIGNED = """imsize 33 33
eye 0 0 3
viewdir 0 0 -1
hfov 70
updir 0 1 0
bkgcolor 0.1 0.1 0.2 1.0
shadow soft
light 0 0 5 1 1 1 1
mtlcolor 0.7 0.7 0.7 1 1 1 0.2 0.7 0.2 10 1 1.0
v -6 -6 -2
v 6 -6 -2
v 6 6 -2
v -6 6 -2
f 1 2 3
f 1 3 4
mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.6 0.3 24 1 1.0
sphere 0.3 0 0 0.5
sphere -1.2 0.4 -0.5 0.4
"""


@pytest.mark.parametrize("name,text", [("many_lights", MANY_LIGHTS), ("axis_aligned", AXIS_ALIGNED),
                                       ("bank_4", light_bank(4, soft=True)), ("bank_5", light_bank(5, soft=True))])
def test_soft_shadow_list_path_corner_cases(workdir, monkeypatch, name, text):
    """Soft shadows through the candidate-list kernels, bit-compared with the oracle (which traces all 50 samples of
    every request): six area lights (more than the kernel-parameter light bank holds, attenuation included); an odd
    image looking along -z at a wall from y = 0 with the light's corners at y = 0 too, so the middle rows' shafts have
    no definite sign on y (the shaft test drops the axis; rays of both signs share a list).  Exactly axis-degenerate
    samples are covered on the CPU (tests/test_shaft_cull.py) and take the same per-ray walk as the pool-full case
    forced here: with a 64-entry list pool almost every request overflows to that walk, same image."""
    scene = Scene(text=text, asset_dir=workdir)
    ref, ost = ob.OracleScene(scene).render()
    img, st = gpu_render(scene)
    d = image_diff(img, ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, d
    assert st["shadow_rays"] == ost.shadow_rays and st["closest_rays"] == ost.closest_rays
    assert st["shadow_rays_traced"] < st["shadow_rays"]
    monkeypatch.setenv("WRT_LIST_POOL_CAP", "64")
    small, st2 = gpu_render(scene)
    monkeypatch.delenv("WRT_LIST_POOL_CAP")
    assert np.array_equal(small, img) and st2["shadow_rays"] == st["shadow_rays"]
    monkeypatch.setenv("WRT_SOFT_LISTS", "0")
    plain, _ = gpu_render(scene)
    monkeypatch.delenv("WRT_SOFT_LISTS")
    assert np.array_equal(plain, img)


# ---------------- device BVH build, re-upload, multi-GPU contexts ----------------

@pytest.mark.parametrize("name", ["water_small", "spheres", "bump"])
def test_device_built_tree_equals_host_built_tree_in_every_result(workdir, monkeypatch, name):
    """The kernels walk a tree built on the device (PLOC, csrc/cuda/bvh_build.cuh).  Results do not depend on the
    topology (DESIGN.md section 4): with WRT_HOST_BVH=1 (the host's binned-SAH tree) image, ray counts and every strategy
    query are bit-identical."""
    scene, _ = load_golden_scene(workdir, name)
    g = np.load(GOLD / f"rays_{name}.npz")
    out = {}
    for host in ("0", "1"):
        monkeypatch.setenv("WRT_HOST_BVH", host)
        r = Renderer(scene)
        img = r.render().copy()
        h = r.interStrategy.UpdateInter(g["orig"], g["dir"])
        hard = r.interStrategy.getShadowCoeffi(g["sh_pos"], g["sh_ndir"], g["sh_light"])
        dirc = r.interStrategy.getDirectionalShadowCoeffi(g["sh_pos"], g["sh_self"], g["sh_ldir"])
        out[host] = (img, dict(r.last_stats), h, hard, dirc)
        r.ctx.close()
    monkeypatch.delenv("WRT_HOST_BVH")
    a, b = out["0"], out["1"]
    assert np.array_equal(a[0], b[0])
    for k in ("closest_rays", "shadow_rays", "rays_per_depth", "shadow_requests"):
        assert a[1][k] == b[1][k], k
    assert a[2].tobytes() == b[2].tobytes()
    assert np.array_equal(a[4], b[4])
    assert np.array_equal(a[3], b[3])                    # the hard-shadow product has the reference's association either way


def test_scene_reupload_switches_scenes_without_residue(workdir):
    """wrt_upload_scene on a live context: a larger scene, a smaller one, the first again — each frame equals the frame
    of a fresh context (device arrays are reused or regrown, the tree is rebuilt on the device every time)."""
    names = ["water_small", "spheres", "config_small", "water_small"]
    scenes = {n: load_golden_scene(workdir, n)[0] for n in set(names)}
    fresh = {n: gpu_render(sc)[0] for n, sc in scenes.items()}
    r = Renderer(scenes[names[0]])
    for n in names:
        r.ctx.upload_scene(scenes[n])
        r.scene = scenes[n]
        assert np.array_equal(r.render(), fresh[n]), n
    r.ctx.close()


def test_malformed_scene_descriptions_are_rejected(workdir):
    """Indices in a hand-filled WrtSceneDesc are validated at upload (ADVICE r1): material / leaf / child links."""
    import ctypes as C
    from whittedstyle_raytracer_b200 import cabi
    from whittedstyle_raytracer_b200.renderer import Context, CudaError
    scene, _ = load_golden_scene(workdir, "spheres")
    ctx = Context()
    d = cabi.WrtSceneDesc.from_buffer_copy(scene.desc)

    def upload_bad(field, idx, value, match):
        arr = getattr(scene.desc, field)
        n = scene.desc.n_nodes if field == "nodes" else scene.desc.n_prims
        copy = (arr._type_ * n)(*[arr[i] for i in range(n)])
        if field == "nodes":
            copy[idx].link = value
        else:
            copy[idx] = value
        bad = cabi.WrtSceneDesc.from_buffer_copy(d)
        setattr(bad, field, C.cast(copy, type(arr)))
        with pytest.raises(CudaError, match=match):
            ctx._check(ctx.lib.wrt_upload_scene(ctx.h, C.byref(bad)))

    upload_bad("prim_material", 3, 10_000, "material index")
    leaf = next(i for i in range(2, scene.desc.n_nodes) if scene.desc.nodes[i].link < 0)
    upload_bad("nodes", leaf, ~(scene.desc.n_prims + 5), "leaf link")
    inner = next(i for i in range(2, scene.desc.n_nodes) if scene.desc.nodes[i].link >= 0)
    upload_bad("nodes", inner, scene.desc.n_nodes + 7, "child link")
    ctx.upload_scene(scene)                              # and the context is still usable
    ctx.close()


@pytest.mark.parametrize("n_gpus", [1, 2, 4, 8])
def test_multi_gpu_contexts_in_one_process(workdir, monkeypatch, n_gpus):
    """wrt_multi_* (what `wrt --gpus N` uses): N contexts on N host threads, interleaved tiles, pixels stored straight
    into GPU 0's frame over NVLink — image and ray counts equal the single-GPU frame's; likewise through the
    copy + scatter path (WRT_MULTI_NO_PEER) and for soft shadows."""
    import torch
    if torch.cuda.device_count() < n_gpus:
        pytest.skip(f"needs {n_gpus} GPUs")
    for kind, name in (("img", "water_small"), ("soft", "water_soft")):
        scene, _ = load_golden_scene(workdir, name, kind=kind)
        full, st_full = gpu_render(scene)
        for no_peer in (False, True):
            if no_peer:
                monkeypatch.setenv("WRT_MULTI_NO_PEER", "1")
            m = MultiRenderer(scene, list(range(n_gpus)))
            assert m.uses_peer_stores == (not no_peer)
            img = m.render()
            st = m.last_stats
            again = m.render()
            m.close()
            if no_peer:
                monkeypatch.delenv("WRT_MULTI_NO_PEER")
            assert np.array_equal(img, full) and np.array_equal(again, full), (name, n_gpus, no_peer)
            for k in ("closest_rays", "shadow_rays", "rays_per_depth", "shadow_requests"):
                assert st[k] == st_full[k], k


def test_drop_in_executable_on_several_gpus(workdir):
    """`wrt --gpus N config.txt` writes byte for byte the PPM of the 1-GPU run."""
    import torch
    n = min(torch.cuda.device_count(), 8)
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    exe = REPO / "whittedstyle_raytracer_b200" / "wrt"
    fixtures.write_config(workdir, "cli_multi", fixtures.water_bunny_tex_config(320, 200, soft=True))
    out = []
    for args in ([], ["--gpus", str(n)]):
        p = subprocess.run([str(exe), "cli_multi.txt"] + args, cwd=workdir, capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
        out.append((workdir / "cli_multi.ppm").read_bytes())
        (workdir / "cli_multi.ppm").unlink()
    assert out[0] == out[1]
