"""Cost of the exported planes: wrt_render against wrt_render_float, and against wrt_render_gbuffer with every plane and
with `hit` only, on the 4K workloads; and on the device, wrt_render_gbuffer_device with all six outputs (8-bit and float
colour, hit, normal, albedo, shadow) against wrt_render_device into a tile buffer.  The six calls alternate round by
round.  Host wall time of the call until its results are final (output arrays and tensors allocated once and reused,
so no first-touch page faults are timed; the device calls include wrt_finish_device) and the frame's device time
(gpu_ms: first kernel to the last batch's copies or plane stores).  Prints one JSON object with the card's name and
power limit.
Usage: gpu_gbuffer_time.py [--rounds N] [--out FILE] [workload ...]"""
import argparse
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
from whittedstyle_raytracer_b200 import Renderer, Scene, fixtures  # noqa: E402

WORKLOADS = ["bunny_shadow_4k", "gla_bunny_tex_4k", "water_bunny_tex_soft_4k", "f4_directional_4k", "f4_bump_4k",
             "f4_spheres_1k_4k"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    ap.add_argument("workloads", nargs="*", default=WORKLOADS)
    a = ap.parse_args()
    wd = Path(tempfile.mkdtemp(prefix="wrt_gbuffer_time_"))
    fixtures.ensure_assets(wd)
    result = {"card": card(), "rounds": a.rounds, "workloads": {}}
    for name in a.workloads:
        fixtures.write_config(wd, name, fixtures.bench_config_text(name))
        scene = Scene.from_workdir(wd, name, bunny=fixtures.BENCH_CONFIGS[name].get("bunny", True))
        r = Renderer(scene)
        full = r.render_gbuffer()                       # allocates the output arrays once (and warms every mode)
        hit_only = {"rgb": full["rgb"], "hit": full["hit"]}
        rgb_f = np.zeros(full["rgb"].shape, np.float32)
        dev_out = r.render_gbuffer_device()             # preallocated tensors of all six outputs
        tiles = torch.zeros(r.ctx.tile_pixel_count(0, 1) * 3, dtype=torch.uint8, device="cuda")

        def render_device():
            r.render_device(tiles.data_ptr(), torch.cuda.current_stream().cuda_stream)
            r.finish_device()
        calls = {"render": lambda: r.render(out=full["rgb"]),
                 "render_float": lambda: r.render_float(out_f=rgb_f, out=full["rgb"]),
                 "gbuffer_all": lambda: r.render_gbuffer(out=full),
                 "gbuffer_hit": lambda: r.render_gbuffer(planes=("hit",), out=hit_only),
                 "gbuffer_device_all": lambda: r.render_gbuffer_device(out=dev_out),
                 "render_device": render_device}
        for f in calls.values():
            f()
        wall = {k: [] for k in calls}
        dev = {k: [] for k in calls}
        for _ in range(a.rounds):
            for k, f in calls.items():
                t0 = time.perf_counter()
                f()
                wall[k].append(1e3 * (time.perf_counter() - t0))
                dev[k].append(r.last_stats["gpu_ms"])
        n_lights = scene.desc.n_lights
        px = scene.camera.width * scene.camera.height
        row = {"pixels": px, "n_lights": n_lights, "plane_bytes": px * (60 + 24 + 4 * n_lights)}
        for k in calls:
            row[k] = {"wall_ms_median": round(statistics.median(wall[k]), 3), "wall_ms_min": round(min(wall[k]), 3),
                      "gpu_ms_median": round(statistics.median(dev[k]), 3)}
        result["workloads"][name] = row
        print(name, json.dumps(row), flush=True)
        r.ctx.close()
    print(json.dumps(result))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
