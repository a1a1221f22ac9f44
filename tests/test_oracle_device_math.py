"""The device-math build of the CPU oracle (oracle/liboracle_devmath.so, whitted_oracle.c with -DORC_DEVICE_MATH) against
the default build and the reference's goldens.  The variant evaluates powf, acosf and atan2f as the render core does
(dev_math.cuh, dev_shade.cuh complete_hit) and changes nothing else, so it must still meet the reference bars, render
the default oracle's 8-bit image but for the rare pixel where glibc's float functions differ in the last ulp, and trace
exactly the same rays.  tests/test_gpu_float_frame.py holds the frame's float colour to this build bit for bit."""
import numpy as np
import pytest

import oracle_bindings as ob
from conftest import IMG_SCENES, SOFT_SCENES, image_diff, load_golden_scene, psnr


@pytest.fixture(scope="session", autouse=True)
def _devmath_oracle():
    import __graft_entry__ as g
    g.build_oracle(device_math=True)


def float_difference(a, b):
    """Channels whose float32 bits differ (NaN against NaN counts as equal) and the largest absolute difference."""
    nan = np.isnan(a) & np.isnan(b)
    diff = (a.view(np.uint32) != b.view(np.uint32)) & ~nan
    big = float(np.abs(a[diff].astype(np.float64) - b[diff].astype(np.float64)).max()) if diff.any() else 0.0
    return int(diff.sum()), big


def render_both(scene):
    u8, fl, st = ob.OracleScene(scene).render(want_float=True)
    u8d, fld, std = ob.OracleScene(scene, device_math=True).render(want_float=True)
    return (u8, fl, st), (u8d, fld, std)


def assert_same_rays(st, std):
    assert (std.closest_rays, std.shadow_rays) == (st.closest_rays, st.shadow_rays)
    assert list(std.rays_per_depth) == list(st.rays_per_depth)
    assert (std.box_tests, std.prim_tests) == (st.box_tests, st.prim_tests)


@pytest.mark.parametrize("name", IMG_SCENES)
def test_device_math_oracle_meets_the_reference_golden(workdir, name):
    scene, g = load_golden_scene(workdir, name)
    (u8, fl, st), (u8d, fld, std) = render_both(scene)
    d = image_diff(u8d, g["rgb"])
    assert d["within1"] >= 0.999 * d["n"], ("vs reference golden", d)
    d = image_diff(u8d, u8)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, ("vs default oracle", d)
    assert_same_rays(st, std)
    assert std.closest_rays == int(g["closest_rays"]) and std.shadow_rays == int(g["shadow_rays"])
    n, big = float_difference(fld, fl)
    print(f"{name}: {n} of {fl.size} float channels differ from the default oracle, largest by {big:.3g}")
    # a last-ulp change of one libm result moves a colour by far less than one 8-bit step
    assert big < 1e-3, (n, big)


@pytest.mark.parametrize("name", SOFT_SCENES)
def test_device_math_oracle_soft_scenes(workdir, name):
    scene, g = load_golden_scene(workdir, name, kind="soft")
    (u8, fl, st), (u8d, fld, std) = render_both(scene)
    assert psnr(u8d, g["mean_rgb"]) >= 30.0
    d = image_diff(u8d, u8)
    assert d["exact"] >= 0.9999 * d["n"] and d["max"] <= 1, ("vs default oracle", d)
    assert_same_rays(st, std)
    assert std.closest_rays == int(g["closest_rays"]) and std.shadow_rays == int(g["shadow_rays"])
    n, big = float_difference(fld, fl)
    print(f"{name}: {n} of {fl.size} float channels differ from the default oracle, largest by {big:.3g}")
    assert big < 1e-3, (n, big)


def test_device_math_differs_only_in_the_three_functions(workdir):
    """A scene where the variant's three functions cannot change a colour: no textured sphere, every specular exponent
    is 2 (x*x in both builds), and ks = 0, alpha = 1 everywhere, so Fresnel's pow(x, 5), evaluated at every hit,
    multiplies only zero children.  The two builds must render identical floats."""
    text = ("imsize 48 32\neye 0 1 6\nviewdir 0 -0.1 -1\nhfov 60\nupdir 0 1 0\nbkgcolor 0.1 0.1 0.2 1.0\n"
            "light 3 6 4 1 0.7 0.7 0.7\nattlight 1 7 7 1 0.4 0.4 0.4 0.5 0.02 0.001\n"
            "mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.6 0 2 1 1.5\nsphere -1.5 0 -1 1.2\n"
            "mtlcolor 0.4 0.7 0.4 1 1 1 0.2 0.7 0 2 1 1.0\n"
            "v -10 -1.2 8\nv 10 -1.2 8\nv 10 -1.2 -12\nv -10 -1.2 -12\nf 1 2 3\nf 1 3 4\n")
    from whittedstyle_raytracer_b200 import Scene
    scene = Scene(text=text, asset_dir=workdir)
    (u8, fl, st), (u8d, fld, std) = render_both(scene)
    assert np.array_equal(fl.view(np.uint32), fld.view(np.uint32))
    assert np.array_equal(u8, u8d)
    assert_same_rays(st, std)
