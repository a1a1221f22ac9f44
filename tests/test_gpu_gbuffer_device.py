"""The frame's surface planes, float colour and 8-bit image delivered to device memory (wrt_render_gbuffer_device,
Renderer.render_gbuffer_device): byte for byte what the host forms return (render_gbuffer's planes, render_float's
colour, render's image), the planes also against the CPU oracle, and the frame itself unchanged by them.

The host forms are held to the oracle by tests/test_gpu_gbuffer.py and tests/test_gpu_float_frame.py; the oracle side
(oracle_gbuffer, check_planes) is that file's."""
import ctypes as C
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import IMG_SCENES, REPO, SOFT_SCENES, load_golden_scene
from test_gpu_float_frame import CROPS
from test_gpu_fuzz import random_scene
from test_gpu_gbuffer import LIGHT_SCENES, check_planes, oracle_gbuffer
from whittedstyle_raytracer_b200 import Renderer, Scene, cabi, fixtures
from whittedstyle_raytracer_b200.renderer import TRAVERSAL_EXHAUSTIVE, TRAVERSAL_PRUNED, Context, CudaError

pytestmark = pytest.mark.gpu

TRAVERSALS = (TRAVERSAL_PRUNED, TRAVERSAL_EXHAUSTIVE)
OUTPUTS = ("rgb", "rgb_f", "hit", "normal", "albedo", "shadow")
SURFACE = {"normal", "albedo", "shadow", "rgb_f"}       # the outputs k_gbuffer_surface writes
STAT_KEYS = ("closest_rays", "shadow_rays", "shadow_requests", "rays_per_depth", "shadow_rays_traced",
             "shaft_culled_requests", "unlit_skipped_requests", "overflow_retries")
SENTINEL = 0xA7                                         # byte every output is filled with before a tile frame


@pytest.fixture(scope="session", autouse=True)
def _devmath_oracle():
    import __graft_entry__ as g
    g.build_oracle(device_math=True)


def to_host(res):
    """The device outputs as numpy arrays in the host forms' layouts ("hit": (H, W) cabi.HIT_DTYPE)."""
    torch.cuda.synchronize()
    out = {}
    for k, t in res.items():
        a = t.cpu().numpy()
        out[k] = a.view(cabi.HIT_DTYPE)[..., 0] if k == "hit" else a
    return out


def host_frame(r):
    """What the host forms return for the same frame: render()'s image, render_float()'s colour, render_gbuffer()'s
    planes."""
    img = r.render().copy()
    rgb_f, _ = r.render_float()
    g = r.render_gbuffer()
    return dict(rgb=img, rgb_f=rgb_f, hit=g["hit"], normal=g["normal"], albedo=g["albedo"], shadow=g["shadow"])


def assert_same_bytes(got, want, what, keys=OUTPUTS):
    for k in keys:
        assert got[k].shape == want[k].shape, (what, k, got[k].shape, want[k].shape)
        assert got[k].tobytes() == want[k].tobytes(), f"{what}: {k} differs from the host form"


def check_scene(scene, what, oracle=False):
    """Every device output equals the host forms' in each traversal mode; with `oracle`, the planes pass check_planes."""
    want = oracle_gbuffer(scene) if oracle else None
    r = Renderer(scene)
    try:
        for traversal in TRAVERSALS:
            r.ctx.set_options(traversal=traversal)
            host = host_frame(r)
            got = to_host(r.render_gbuffer_device())
            assert_same_bytes(got, host, f"{what}, traversal {traversal}")
            if oracle:
                check_planes(got, want, f"{what}, traversal {traversal}", culled=traversal == TRAVERSAL_PRUNED)
    finally:
        r.ctx.close()


# ---------------- against the host forms and the oracle ----------------

@pytest.mark.parametrize("name,kind", [(n, "img") for n in IMG_SCENES + ["config_800x600"]] + [(n, "soft") for n in SOFT_SCENES])
def test_gbuffer_device_fixture_scenes(workdir, name, kind):
    scene, _ = load_golden_scene(workdir, name, kind=kind)
    check_scene(scene, name, oracle=True)


@pytest.mark.parametrize("name,text", LIGHT_SCENES)
def test_gbuffer_device_light_scenes(workdir, name, text):
    check_scene(Scene(text=text(), asset_dir=workdir), name)


@pytest.mark.parametrize("seed", range(6))
def test_gbuffer_device_random_scenes(workdir, seed):
    text = random_scene(np.random.default_rng(1000 + seed))
    check_scene(Scene(text=text, asset_dir=workdir), f"random scene {seed}\n{text}")


@pytest.mark.parametrize("name", list(CROPS))
def test_gbuffer_device_4k(workdir, name):
    """The whole 3840x2160 device frame equals the host forms'; its 256x256 window passes the oracle."""
    fixtures.write_config(workdir, name, fixtures.bench_config_text(name))
    scene = Scene.from_workdir(workdir, name, bunny=fixtures.BENCH_CONFIGS[name].get("bunny", True))
    x0, y0 = CROPS[name]
    n = 256
    want = oracle_gbuffer(scene, x0, x0 + n, y0, y0 + n)
    win = np.s_[y0:y0 + n, x0:x0 + n]
    r = Renderer(scene)
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal)
        host = host_frame(r)
        got = to_host(r.render_gbuffer_device())
        assert_same_bytes(got, host, f"{name}, traversal {traversal}")
        check_planes({k: v[win] for k, v in got.items()}, want, f"{name} window, traversal {traversal}",
                     culled=traversal == TRAVERSAL_PRUNED)
    r.ctx.close()


# ---------------- the frame is unchanged ----------------

def test_gbuffer_device_is_the_plain_frame(workdir):
    """For every non-empty subset of the six outputs: wrt_render's image and statistics, its launches plus k_gbuffer_hit
    (hit) and k_gbuffer_surface (any of normal, albedo, shadow, rgb_f), and the full call's values.  A render()
    afterwards keeps its launch count and leaves the previous call's tensors alone."""
    subsets = [c for k in range(1, len(OUTPUTS) + 1) for c in itertools.combinations(OUTPUTS, k)]
    for name, kind in (("water_small", "img"), ("water_soft", "soft"), ("directional", "img")):
        scene, _ = load_golden_scene(workdir, name, kind=kind)
        r = Renderer(scene)
        n0 = r.ctx.launches
        img = r.render().copy()
        plain = r.ctx.launches - n0
        st = dict(r.last_stats)
        full = to_host(r.render_gbuffer_device())
        assert np.array_equal(full["rgb"], img), name
        for planes in subsets:
            n1 = r.ctx.launches
            dev = r.render_gbuffer_device(planes=planes)
            extra = int("hit" in planes) + int(bool(SURFACE & set(planes)))
            assert r.ctx.launches - n1 == plain + extra, (name, planes)
            assert set(dev) == set(planes)
            for k in STAT_KEYS:
                assert r.last_stats[k] == st[k], (name, planes, k)
            got = to_host(dev)
            for p in planes:
                assert got[p].tobytes() == full[p].tobytes(), (name, planes, p)
        sums = {k: int(t.view(torch.uint8).to(torch.int64).sum()) for k, t in dev.items()}
        n2 = r.ctx.launches
        assert np.array_equal(r.render(), img), name
        assert r.ctx.launches - n2 == plain, name
        torch.cuda.synchronize()
        assert sums == {k: int(t.view(torch.uint8).to(torch.int64).sum()) for k, t in dev.items()}, name
        r.ctx.close()


# ---------------- tiles ----------------

def sentinel_out(r):
    """Every output of the frame as a new tensor filled with SENTINEL bytes."""
    cam, nl = r.scene.camera, r.scene.desc.n_lights
    h, w = cam.height, cam.width
    shapes = {"rgb": ((h, w, 3), torch.uint8), "rgb_f": ((h, w, 3), torch.float32), "hit": ((h, w, 15), torch.int32),
              "normal": ((h, w, 3), torch.float32), "albedo": ((h, w, 3), torch.float32), "shadow": ((h, w, nl), torch.float32)}
    out = {}
    for k, (shape, dtype) in shapes.items():
        t = torch.empty(shape, dtype=dtype, device="cuda")
        t.view(torch.uint8).fill_(SENTINEL)
        out[k] = t
    return out


@pytest.mark.parametrize("name", ["spheres", "water_small", "bump"])
def test_gbuffer_device_tiles(workdir, name):
    """Rank r of N (3, 8) writes exactly its own pixels of every output, each once, and leaves every other byte of the
    caller's tensors alone; the union over ranks equals the 1-rank frame."""
    scene, _ = load_golden_scene(workdir, name)
    r = Renderer(scene)
    full = to_host(r.render_gbuffer_device())
    h, w = full["rgb"].shape[:2]
    blank = to_host(sentinel_out(r))
    for world in (3, 8):
        owner = np.zeros((h, w), np.int32)
        merged = {k: v.copy() for k, v in blank.items()}
        for rank in range(world):
            r.ctx.set_tiles(rank=rank, world=world)
            mine = to_host(r.render_gbuffer_device(out=sentinel_out(r)))
            written = mine["hit"].view(np.uint8).reshape(h, w, 60)[..., :4] != SENTINEL
            written = written.any(axis=2)
            owner += written
            for k in OUTPUTS:
                assert mine[k][~written].tobytes() == blank[k][~written].tobytes(), (name, world, rank, k)
                assert mine[k][written].tobytes() == full[k][written].tobytes(), (name, world, rank, k)
                merged[k][written] = mine[k][written]
        assert (owner == 1).all(), (name, world, int((owner == 0).sum()), int((owner > 1).sum()))
        for k in OUTPUTS:
            assert merged[k].tobytes() == full[k].tobytes(), (name, world, k)
    r.ctx.set_tiles(rank=0, world=1)
    r.ctx.close()


# ---------------- overflow ----------------

def overflow_scene(workdir, soft):
    name = f"gbuffer_device_overflow_{int(soft)}"
    fixtures.write_config(workdir, name, fixtures.water_bunny_tex_config(200, 150, soft=soft))
    return Scene.from_workdir(workdir, name)


def single_batch_frames(scene):
    r = Renderer(scene)
    single = {}
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal)
        single[traversal] = to_host(r.render_gbuffer_device())
        assert r.last_stats["overflow_retries"] == 0
    r.ctx.close()
    return single


@pytest.mark.parametrize("soft", [False, True])
def test_gbuffer_device_overflow_multi_batch(workdir, monkeypatch, soft):
    """A 200x150 bunny frame in batches of 8192 slots whose deep levels (queue_factor 0.02) overflow and are redone in
    halves inside the call: every output equals the single-batch frame's."""
    scene = overflow_scene(workdir, soft)
    single = single_batch_frames(scene)
    monkeypatch.setenv("WRT_MAX_BATCH", "8192")
    r = Renderer(scene)
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal, queue_factor=0.02)
        got = to_host(r.render_gbuffer_device())
        assert r.last_stats["overflow_retries"] >= 1
        assert_same_bytes(got, single[traversal], f"multi-batch overflow, traversal {traversal}")
    r.ctx.close()


@pytest.mark.parametrize("soft", [False, True])
def test_gbuffer_device_overflow_in_finish(workdir, soft):
    """The same frame as one batch (queue_factor 0.02 only): wrt_render_gbuffer_device returns once it is enqueued, and
    wrt_finish_device finds the overflow, re-renders the frame into the same buffers and reports the retry."""
    scene = overflow_scene(workdir, soft)
    single = single_batch_frames(scene)
    r = Renderer(scene)
    lib = r.ctx.lib
    for traversal in TRAVERSALS:
        r.ctx.set_options(traversal=traversal, queue_factor=0.02)
        out = sentinel_out(r)
        gb = cabi.WrtGBuffer(hit=out["hit"].data_ptr(), normal=out["normal"].data_ptr(), albedo=out["albedo"].data_ptr(),
                             shadow=out["shadow"].data_ptr())
        stream = torch.cuda.current_stream().cuda_stream
        assert lib.wrt_render_gbuffer_device(r.ctx.h, C.byref(gb), out["rgb_f"].data_ptr(), out["rgb"].data_ptr(), stream) == 0
        st = cabi.WrtStats()
        assert lib.wrt_finish_device(r.ctx.h, C.byref(st)) == 0, lib.wrt_last_error()
        assert st.overflow_retries >= 1
        assert_same_bytes(to_host(out), single[traversal], f"overflow redone in finish, traversal {traversal}")
    r.ctx.close()


# ---------------- streams ----------------

def test_gbuffer_device_on_a_side_stream(workdir):
    """Outputs filled with a sentinel on a non-default stream, then rendered on it: the default stream's frame."""
    scene, _ = load_golden_scene(workdir, "water_soft", kind="soft")
    r = Renderer(scene)
    want = to_host(r.render_gbuffer_device())
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out = sentinel_out(r)
        res = r.render_gbuffer_device(out=out)
    assert all(res[k] is out[k] for k in OUTPUTS)
    assert_same_bytes(to_host(res), want, "side stream")
    r.ctx.close()


# ---------------- malformed input ----------------

def test_gbuffer_device_malformed_input(workdir):
    scene, _ = load_golden_scene(workdir, "water_small")
    r = Renderer(scene)
    lib = r.ctx.lib
    want = to_host(r.render_gbuffer_device())
    h, w = scene.camera.height, scene.camera.width
    rgb = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
    normal = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(ctx, gb, rgb_f, rgb_ptr):
        return lib.wrt_render_gbuffer_device(ctx, C.byref(gb) if gb is not None else None, rgb_f, rgb_ptr, stream)

    def refused(rc, words):
        assert rc != 0
        msg = lib.wrt_last_error()
        assert all(wd in msg for wd in words), msg
        assert np.array_equal(r.render(), want["rgb"])                 # the context still renders
        got = to_host(r.render_gbuffer_device())
        assert_same_bytes(got, want, "after a refused call")

    refused(call(None, cabi.WrtGBuffer(), None, rgb.data_ptr()), [b"null context"])
    refused(call(r.ctx.h, None, None, None), [b"NULL"])
    refused(call(r.ctx.h, cabi.WrtGBuffer(), None, None), [b"NULL"])
    host = np.zeros((h, w, 3), np.float32)
    refused(call(r.ctx.h, None, None, host.ctypes.data), [b"d_rgb", b"device memory"])
    refused(call(r.ctx.h, cabi.WrtGBuffer(normal=host.ctypes.data), None, rgb.data_ptr()), [b"d_planes->normal"])
    pinned = torch.zeros((h, w, 3), dtype=torch.float32, pin_memory=True)
    refused(call(r.ctx.h, cabi.WrtGBuffer(normal=normal.data_ptr()), pinned.data_ptr(), None), [b"d_rgb_f"])
    refused(call(r.ctx.h, cabi.WrtGBuffer(albedo=pinned.data_ptr()), None, None), [b"d_planes->albedo"])

    c = Context()
    refused(call(c.h, None, None, rgb.data_ptr()), [b"scene"])                         # no scene
    assert lib.wrt_upload_scene(c.h, scene.desc_ptr) == 0
    refused(call(c.h, cabi.WrtGBuffer(normal=normal.data_ptr()), None, rgb.data_ptr()), [b"camera"])   # no camera
    c.close()

    good = {"normal": normal}
    bad = {
        "a CPU tensor": {"rgb": torch.zeros((h, w, 3), dtype=torch.uint8)},
        "a numpy array": {"rgb": np.zeros((h, w, 3), np.uint8)},
        "the wrong dtype": {"normal": torch.zeros((h, w, 3), dtype=torch.float64, device="cuda")},
        "the wrong shape": {"shadow": torch.zeros((h, w, scene.desc.n_lights + 1), dtype=torch.float32, device="cuda")},
        "the wrong device": {"albedo": torch.zeros((h, w, 3), dtype=torch.float32, device="meta")},
        "a non-contiguous tensor": {"hit": torch.zeros((h, 2 * w, 15), dtype=torch.int32, device="cuda")[:, ::2]},
        "transposed pixels": {"rgb_f": torch.zeros((w, h, 3), dtype=torch.float32, device="cuda")},
    }
    for what, out in bad.items():
        with pytest.raises(ValueError):
            r.render_gbuffer_device(out={**good, **out})
    with pytest.raises(ValueError):
        r.render_gbuffer_device(planes=("depth",))
    with pytest.raises(ValueError):
        r.render_gbuffer_device(planes=())
    assert_same_bytes(to_host(r.render_gbuffer_device()), want, "after the ValueErrors")
    r.ctx.close()


def test_gbuffer_device_without_lights(workdir):
    """A scene without lights has no shadow plane: requesting it alone is an error, beside other outputs it is ignored."""
    text = "\n".join(["imsize 40 30", "eye 0 0 5", "viewdir 0 0 -1", "hfov 45", "updir 0 1 0", "bkgcolor 0.1 0.1 0.2 1.0",
                      "mtlcolor 0.8 0.2 0.2 1 1 1 0.2 0.6 0.2 10 1 1", "sphere 0 0 0 1"])
    scene = Scene(text=text, asset_dir=workdir)
    assert scene.desc.n_lights == 0
    r = Renderer(scene)
    host = host_frame(r)
    got = to_host(r.render_gbuffer_device())
    assert got["shadow"].shape == (30, 40, 0)
    assert_same_bytes(got, host, "no lights")
    with pytest.raises(CudaError):
        r.render_gbuffer_device(planes=("shadow",))
    r.ctx.close()


# ---------------- bounds-checking build ----------------

def test_device_planes_under_the_bounds_checking_build():
    """The tile and overflow cases above, against libwrt_cuda_debug.so (-DWRT_DEBUG_BOUNDS: every row-major store of the
    two plane kernels is checked against W x H), in a subprocess: the library is chosen at load time."""
    lib = REPO / "whittedstyle_raytracer_b200" / "libwrt_cuda_debug.so"
    assert lib.exists(), "libwrt_cuda_debug.so is not built (__graft_entry__.build_cuda_debug)"
    env = dict(os.environ, WRT_CUDA_LIB=str(lib))
    p = subprocess.run([sys.executable, "-m", "pytest", __file__, "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "test_gbuffer_device_tiles or test_gbuffer_device_overflow"],
                       cwd=REPO, env=env, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert " passed" in p.stdout and "WRT_DEBUG_BOUNDS" not in p.stdout
