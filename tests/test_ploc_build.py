"""The device BVH build (csrc/cuda/ploc_bvh.h + bvh_build.cuh) on the CPU: tests/ploc_check.cpp compiles the SAME per-item
steps the kernels run, emulates the passes in barrier order and checks the resulting tree — every primitive in exactly one
leaf, leaf boxes == the reference's per-primitive boxes, every inner box (and dilated box) the exact union of its
children, sibling pairs adjacent, 2n records, depth, and a surface-area cost close to the host's binned-SAH build
(the tree only has to be valid for parity — DESIGN.md section 4 — but its cost is what the traversal kernels pay).
The GPU tests then run every parity case on the tree the kernels really build.

Fans, slivers and nested sizes (fixtures.DEEP_TREE_GEOMETRY) make PLOC build trees far deeper than log2 n.  The traversal
stack has 90 rows (wrt_upload_scene); a scene whose PLOC tree needs more is given the host's binned-SAH tree instead,
which must then fit (tests/test_gpu_capacity_edges.py renders these scenes on the GPU)."""
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import REPO
from whittedstyle_raytracer_b200 import fixtures

PKG = REPO / "whittedstyle_raytracer_b200"


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = tmp_path_factory.mktemp("ploc") / "ploc_check"
    cuda_inc = next((p for p in (Path("/usr/local/cuda/include"), Path("/usr/local/cuda/targets/x86_64-linux/include"))
                     if (p / "vector_types.h").exists()), None)
    if cuda_inc is None:
        pytest.skip("CUDA headers (vector_types.h) not found")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", f"-I{cuda_inc}",
                    str(REPO / "tests" / "ploc_check.cpp"), "-o", str(exe), f"-L{PKG}", "-lwrt_host",
                    f"-Wl,-rpath,{PKG}", "-pthread"], check=True)
    return exe


def _soup(n, seed):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-8, 8, (n, 3))
    lines = ["imsize 8 8", "eye 0 1 10", "viewdir 0 -0.1 -1", "hfov 60", "updir 0 1 0", "bkgcolor 0.2 0.3 0.5 1.0",
             "light 5 20 10 1 1 1 1", "mtlcolor 0.7 0.6 0.5 1 1 1 0.2 0.7 0.3 20 1 1"]
    tri = c[:, None, :] + rng.uniform(-0.12, 0.12, (n, 3, 3))
    lines += ["v %.4f %.4f %.4f" % tuple(q) for q in tri.reshape(-1, 3)]
    lines += ["f %d %d %d" % (3 * i + 1, 3 * i + 2, 3 * i + 3) for i in range(n)]
    return "\n".join(lines) + "\n"


_HEAD = "imsize 4 4\neye 0 0 5\nviewdir 0 0 -1\nhfov 60\nupdir 0 1 0\nbkgcolor 0 0 0 1\nmtlcolor 1 1 1 1 1 1 0.2 0.7 0.3 20 1 1\n"

STACK_ROWS_MAX = 90


def stack_rows(ref_depth, walked_depth):
    """Traversal-stack rows wrt_upload_scene reserves: one push per level of the binary walks (reference tree and walked
    tree), up to three per two levels in the 4-wide walks, plus two."""
    return max(ref_depth, walked_depth, 3 * ((walked_depth + 1) // 2)) + 2


CASES = {
    # name: (config text, with bunny, max cost ratio vs the host's binned SAH, PLOC tree fits the stack)
    "bunny": (lambda: fixtures.water_bunny_tex_config(8, 8), True, 1.05, True),
    "spheres_1k": (lambda: fixtures.f4_spheres_config(8, 8), False, 1.30, True),
    "soup_20k": (lambda: _soup(20000, 3), False, 1.30, True),
    "identical_boxes": (lambda: _HEAD + "sphere 0 0 0 1\n" * 37, False, 2.0, True),
    "two": (lambda: _HEAD + "sphere 0 0 0 1\nsphere 3 0 0 1\n", False, 1.01, True),
    "one": (lambda: _HEAD + "sphere 0 0 0 1\n", False, 1.01, True),
    # deep PLOC trees (PLOC depth 45, 68, 70, 105, 114, 29 — the host's SAH tree stays at 10 .. 34 levels)
    "fan_1000": (lambda: _HEAD + fixtures.fan_geometry(1000), False, 1.05, True),
    "fan_2000": (lambda: _HEAD + fixtures.fan_geometry(2000), False, 1.05, False),
    "cylinder_2000": (lambda: _HEAD + fixtures.cylinder_geometry(2000), False, 1.05, False),
    "slivers_4000": (lambda: _HEAD + fixtures.sliver_geometry(4000), False, 1.05, False),
    "mixed_radii_5000": (lambda: _HEAD + fixtures.mixed_radius_spheres(5000, 1), False, 1.05, False),
    "chain_30": (lambda: _HEAD + fixtures.sphere_chain(30), False, 1.05, True),
}
DEEP = {"fan_1000", "fan_2000", "cylinder_2000", "slivers_4000", "mixed_radii_5000", "chain_30"}


@pytest.mark.parametrize("name", sorted(CASES))
def test_ploc_tree_is_a_valid_tree_over_the_reference_boxes(checker, tmp_path, name):
    text, bunny, max_ratio, fits = CASES[name]
    fixtures.ensure_assets(tmp_path)
    fixtures.write_config(tmp_path, name, text())
    p = subprocess.run([str(checker), str(tmp_path / f"{name}.txt"), str(tmp_path / "bunny.obj") if bunny else "", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    r = json.loads(p.stdout.strip().splitlines()[-1])
    assert "error" not in r, r
    assert r["records"] == max(2 * r["n"], 2) == r["ref_nodes"]
    assert r["missing"] == 0 and r["bad_union"] == 0 and r["bad_leaf_box"] == 0
    assert r["bad_dilated_union"] == 0 and r["dilated_leaf_diff"] == 0
    assert r["depth"] == r["depth_seen"]
    # which tree the kernels walk: PLOC's when it fits the stack, else the host's SAH tree, which always must
    assert (stack_rows(r["ref_depth"], r["depth"]) <= STACK_ROWS_MAX) == fits, r
    assert stack_rows(r["ref_depth"], r["host_depth"]) <= STACK_ROWS_MAX, r
    # a pass merges at least one pair, so n - 1 passes always suffice; on balanced inputs every pass merges a large share
    # of the clusters, but on fans a pass merges only the few mutual nearest neighbours among near-identical boxes
    # (~n/10 passes)
    assert r["passes"] <= max(r["n"] - 1, 0)
    if name not in DEEP:
        assert r["passes"] <= 4 * max(1, int(np.ceil(np.log2(max(r["n"], 2))))) + 8
    assert r["cost"] <= max_ratio * r["host_sah_cost"] + 1e-6, r
