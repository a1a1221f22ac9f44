"""`bench.py --dump-outputs DIR`: the last timed step's frame and ray counts as .npy files, within 64 MiB, the same
pixel sample on every run; on the GPU, the dumped frame is the frame the renderer and the oracle compute."""
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle_bindings as ob
from conftest import REPO, image_diff


def test_large_frame_is_dumped_as_a_fixed_sample_within_budget(tmp_path):
    h, w = 2160, 3840
    img = (np.arange(h * w * 3, dtype=np.int64) % 251).astype(np.uint8).reshape(h, w, 3)
    counts = {"closest_rays": 17959375, "shadow_rays": 724386450, "shadow_requests": 14487729, "rays_per_depth": [8294400, 1332338]}
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, img, counts)
    total = sum(f.stat().st_size for f in (tmp_path / "a").iterdir())
    assert total <= bench.DUMP_BUDGET_BYTES
    sample, idx = np.load(tmp_path / "a" / "image.npy"), np.load(tmp_path / "a" / "image_pixel_index.npy")
    assert sample.dtype == np.float32 and sample.shape == (bench.DUMP_SAMPLE_PIXELS, 3)
    assert idx.dtype == np.float64 and len(np.unique(idx)) == len(idx)
    assert np.array_equal(sample, img.reshape(-1, 3)[idx.astype(np.int64)].astype(np.float32))
    for f in (tmp_path / "a").iterdir():
        assert np.array_equal(np.load(f), np.load(tmp_path / "b" / f.name)), f.name
    assert np.load(tmp_path / "a" / "shadow_rays.npy") == 724386450.0
    assert np.load(tmp_path / "a" / "rays_per_depth.npy").dtype == np.float64


def test_small_frame_is_dumped_whole(tmp_path):
    img = np.random.default_rng(1).integers(0, 256, (600, 800, 3)).astype(np.uint8)
    bench.dump_outputs(tmp_path, img, {"closest_rays": 1})
    got = np.load(tmp_path / "image.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img.astype(np.float32))
    assert not (tmp_path / "image_pixel_index.npy").exists()


@pytest.mark.gpu
def test_bench_dumps_the_frame_it_timed(workdir, tmp_path):
    from whittedstyle_raytracer_b200 import Scene, fixtures
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, str(REPO / "bench.py"), "--workload", "config", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    img = np.load(out / "image.npy")
    assert img.shape == (600, 800, 3) and img.dtype == np.float32
    fixtures.write_config(workdir, "dump_config", fixtures.bench_config_text("config"))
    scene = Scene.from_workdir(workdir, "dump_config")
    ref, st = ob.OracleScene(scene).render()
    d = image_diff(img.astype(np.uint8), ref)
    assert d["exact"] >= 0.9999 * d["n"] and d["within1"] >= 0.999 * d["n"], d
    assert float(np.load(out / "closest_rays.npy")) == st.closest_rays
    assert float(np.load(out / "shadow_rays.npy")) == st.shadow_rays
    assert np.array_equal(np.load(out / "rays_per_depth.npy"), np.asarray(st.rays_per_depth, np.float64))
