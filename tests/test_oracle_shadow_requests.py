"""The oracle's per-request shadow answer (orc_shadow_requests), which the frame's shadow kernels are held to request by
request (tests/test_gpu_shadow_requests.py), against the oracle's per-ray queries it is built from: the soft-shadow sum is
50 x the mean of the 50 visibility samples at the light points include/wrt_rng.h draws; hard and directional requests are
the plain queries.  The frame oracle's soft-shadow term divides the same sum (the image goldens pin it)."""
import ctypes as C

import numpy as np

import oracle_bindings as ob
from conftest import load_golden_scene


def _requests(scene, orc, rng, n):
    cam = scene.camera
    o, d = orc.primary_rays()
    pick = rng.integers(0, len(o), n)
    h = orc.trace_closest(o[pick], d[pick])
    h = h[h["hit"] == 1]
    nd = h["ndir"].copy()
    nd[1::2] *= -1.0                                           # flipped normals too
    m = len(h)
    pixel = rng.integers(0, cam.width * cam.height, m).astype(np.uint32)
    pixel[:2] = (0, 0xFFFFFFFF)
    return h["pos"], nd, h["object"], pixel, rng.integers(1, 512, m).astype(np.uint32)


def test_soft_request_is_the_sum_of_its_samples(workdir):
    scene, _ = load_golden_scene(workdir, "water_soft", kind="soft")
    orc = ob.OracleScene(scene)
    rng = np.random.default_rng(50)
    pos, nd, obj, pixel, path = _requests(scene, orc, rng, 3000)
    n = len(pos)
    assert n > 2000
    nl = scene.desc.n_lights
    light = rng.integers(0, nl, n).astype(np.int32)
    got = orc.shadow_requests(pos, nd, light, pixel, path, obj)
    tri = np.array([list(scene.desc.lights[i].tri) for i in range(nl)], np.float32).reshape(nl, 3, 3)
    uv = (C.c_float * 2)()
    lp = np.zeros((n, 50, 3), np.float32)
    for i in range(n):
        t = tri[light[i]]
        for k in range(50):
            orc.lib.orc_light_sample_uv(0x5EED, int(pixel[i]), int(path[i]), int(light[i]), k, uv)
            u, v = np.float32(uv[0]), np.float32(uv[1])
            lp[i, k] = t[0] * (np.float32(1) - u - v) + t[1] * u + t[2] * v        # randomSampleTriangle, one rounding per op
    samples = orc.shadow_soft(np.repeat(pos, 50, 0), np.repeat(nd, 50, 0), lp.reshape(-1, 3)).reshape(n, 50)
    assert np.array_equal(got, (50.0 * samples.astype(np.float64).mean(axis=1)).astype(np.float32))
    assert 0.05 < (got < 50).mean() < 0.95 and (got > 0).mean() > 0.05            # shadowed, penumbra and lit requests


def test_hard_and_directional_requests_are_the_plain_queries(workdir):
    scene, _ = load_golden_scene(workdir, "directional")
    orc = ob.OracleScene(scene)
    rng = np.random.default_rng(51)
    pos, nd, obj, pixel, path = _requests(scene, orc, rng, 20000)
    d = scene.desc
    lights = [d.lights[i] for i in range(d.n_lights)]
    point = [abs(L.pos[3] - 1.0) < 1e-5 for L in lights]
    assert any(point) and not all(point)
    for li, L in enumerate(lights):
        light = np.full(len(pos), li, np.int32)
        got = orc.shadow_requests(pos, nd, light, pixel, path, obj)
        if point[li]:
            want = orc.shadow_hard(pos, nd, np.tile(np.array(L.pos[:3], np.float32), (len(pos), 1)))
        else:
            want = orc.shadow_directional(pos, obj, np.tile(np.array(L.pos[:4], np.float32), (len(pos), 1)))
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), li
        assert 0.02 < (got < 1).mean() < 0.98, li
