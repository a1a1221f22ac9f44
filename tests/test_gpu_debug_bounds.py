"""The bounds-checking build of the render core (libwrt_cuda_debug.so, -DWRT_DEBUG_BOUNDS): every ray-queue, request-queue,
candidate-pool, node, coefficient and traversal-stack index is checked inside the kernels and a violation fails the
frame with the source line.  compute-sanitizer is not available on the GPU pool, so this build is how the capacity
arguments in kernels.cuh are checked: the 24 random scenes, the multi-batch / overflow / pool-full cases, the edge
scenes, the capacity-edge scenes (deep trees, stack budget, shadow crossings, list cap), the frame's shadow kernels on
given requests (tests/test_gpu_shadow_requests.py) and the float-frame shading edges, overflow and tile cases
(tests/test_gpu_float_frame.py) all run under it, in a
subprocess (the library is chosen at load time through WRT_CUDA_LIB)."""
import os
import subprocess
import sys

import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu


def test_fuzz_and_overflow_cases_under_the_bounds_checking_build():
    lib = REPO / "whittedstyle_raytracer_b200" / "libwrt_cuda_debug.so"
    assert lib.exists(), "libwrt_cuda_debug.so is not built (__graft_entry__.build_cuda_debug)"
    env = dict(os.environ, WRT_CUDA_LIB=str(lib))
    sel = ("test_random_scene or test_multi_batch_frames_with_overflow or test_queue_overflow_is_rerendered or "
           "test_edge_scenes or test_soft_shadow_list_path_corner_cases or test_device_frame_overflow or "
           "test_image_matches_oracle_and_reference or test_deep_tree or test_fan_walked_at_the_stack_budget or "
           "test_hard_shadow_crossings or test_directional_crossings or test_soft_shadow_shafts_past_the_list_cap or "
           "test_shadow_requests or test_float_frame_shading_edges or test_float_frame_overflow or test_float_frame_tiles or "
           "test_float_frame_forty_lights")
    p = subprocess.run([sys.executable, "-m", "pytest", str(REPO / "tests" / "test_gpu_fuzz.py"),
                        str(REPO / "tests" / "test_gpu_parity.py"), str(REPO / "tests" / "test_gpu_capacity_edges.py"),
                        str(REPO / "tests" / "test_gpu_shadow_requests.py"), str(REPO / "tests" / "test_gpu_float_frame.py"),
                        "-m", "gpu", "-x", "-q", "-k", sel, "-p", "no:cacheprovider"],
                       cwd=REPO, env=env, capture_output=True, text=True, timeout=2700)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert " passed" in p.stdout and "WRT_DEBUG_BOUNDS" not in p.stdout


def test_the_debug_build_reports_a_violation(workdir, tmp_path):
    """The check itself works: with a traversal stack one row too short for the tree (WRT_DEBUG_STACK_ROWS) the
    bounds-checking build fails the frame instead of corrupting shared memory."""
    lib = REPO / "whittedstyle_raytracer_b200" / "libwrt_cuda_debug.so"
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from conftest import load_golden_scene\n"
        "from pathlib import Path\n"
        "from whittedstyle_raytracer_b200 import Renderer, fixtures\n"
        "from whittedstyle_raytracer_b200.renderer import CudaError\n"
        "wd = Path(%r); fixtures.ensure_assets(wd)\n"
        "scene, _ = load_golden_scene(wd, 'water_small')\n"
        "r = Renderer(scene)\n"
        "try:\n"
        "    r.render(); print('NO ERROR')\n"
        "except CudaError as e:\n"
        "    print('CAUGHT', e)\n" % (str(REPO), str(REPO / "tests"), str(tmp_path)))
    env = dict(os.environ, WRT_CUDA_LIB=str(lib), WRT_DEBUG_STACK_ROWS="3")
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert "CAUGHT" in p.stdout and "WRT_DEBUG_BOUNDS" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]
