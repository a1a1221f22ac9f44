"""Development aid: one rank's share of the metric frame (rank 0 of WORLD) and the whole frame under different launch
knobs (environment variables read by wrt_create).  Usage: gpu_share_sweep.py [workload] [world ...]

Every configuration gets its own context; prints min-of-8 frame time per (world, knob set) and, for the knob sets marked
with '*', the serialised per-family times."""
import os
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
from whittedstyle_raytracer_b200 import Scene, Renderer, fixtures  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "water_bunny_tex_soft_4k"
worlds = [int(a) for a in sys.argv[2:]] or [8, 1]
wd = Path("/tmp/wrt_perf")
fixtures.ensure_assets(wd)
fixtures.write_config(wd, name, fixtures.bench_config_text(name))
scene = Scene.from_workdir(wd, name)

KNOBS = [
    ("*default", {}),
    ("deep_split=4", {"WRT_DEEP_SPLIT": "4"}),
    ("deep_split=6", {"WRT_DEEP_SPLIT": "6"}),
    ("deep_split=7", {"WRT_DEEP_SPLIT": "7"}),
    ("deep_split=8", {"WRT_DEEP_SPLIT": "8"}),
    ("shade0_separate=0", {"WRT_SHADE0_SEPARATE": "0"}),
    ("default (again)", {}),
]
if os.environ.get("SWEEP_KNOBS"):             # "label:K=V,K=V;label2:..." replaces the table above
    KNOBS = []
    for item in os.environ["SWEEP_KNOBS"].split(";"):
        label, _, kvs = item.partition(":")
        KNOBS.append((label, dict(kv.split("=") for kv in kvs.split(",") if kv)))
ALL = sorted({k for _, kv in KNOBS for k in kv})

for label, kv in KNOBS:
    for k in ALL:
        os.environ.pop(k, None)
    os.environ.update(kv)
    r = Renderer(scene)
    line = [f"{label:28s}"]
    for world in worlds:
        r.ctx.set_tiles(8, 4, 0, world)
        ts = []
        for it in range(9):
            r.render()
            ts.append(r.last_stats["gpu_ms"])
        line.append(f"world {world}: {min(ts[1:]):7.3f} ms")
    print("  ".join(line), flush=True)
    if label.startswith("*"):
        r.ctx.enable_kernel_timing(True)
        for world in worlds:
            r.ctx.set_tiles(8, 4, 0, world)
            for it in range(3):
                r.render()
            print(f"    world {world} serialised {r.last_stats['gpu_ms']:.3f} ms",
                  {k: round(v, 3) for k, v in r.ctx.kernel_times().items() if v > 0}, flush=True)
    r.ctx.close()
    del r
