#!/usr/bin/env python
"""bench.py — Mrays/s (all ray types) and ms/frame of the Whitted hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A step = one frame of the workload (default: BASELINE.json configs[3], out/water_bunny_tex.txt
+ `shadow soft` at 3840x2160 — the configuration the north-star metric is quoted on).
N > 1 (launched by torchrun, one rank per GPU): the same frame strong-scaled over interleaved
tiles, gathered to rank 0 with one NCCL gather; time = max over ranks.
Prints ONE JSON line (rank 0).  `value` = rays of the whole frame / device time with the scene
resident in HBM; `e2e` = the same through the host-buffer C-ABI call (scene H2D upload +
render + image D2H inside the timed region).  `--impl reference` times the UNMODIFIED
reference (oracle/_ref, single-threaded by construction) on a bounded pixel sample of the
same frame; beside its value the line carries `all_cores`: the same sample traced by one
independent reference process per host core (what the whole host could do; not the reference's mode).
`--dump-outputs DIR` writes the frame and ray counts of the last timed step as .npy files (dump_outputs): the inputs
are the same from run to run, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

METRIC = "Mrays/s (all ray types), out/water_bunny_tex.txt + shadow soft @ 3840x2160"
UNIT = "Mrays/s"
DEFAULT_WORKLOAD = "water_bunny_tex_soft_4k"
WORKLOAD_DESC = {
    "config": "config.txt (== bunny_shadow.txt) @ 800x600, hard shadows (BASELINE.json configs[0])",
    "bunny_shadow_4k": "bunny_shadow.txt @ 3840x2160, hard shadows (BASELINE.json configs[1])",
    "gla_bunny_tex_4k": "gla_bunny_tex.txt @ 3840x2160, hard shadows + Fresnel recursion (BASELINE.json configs[2])",
    "water_bunny_tex_soft_4k": "out/water_bunny_tex.txt + shadow soft @ 3840x2160 (BASELINE.json configs[3])",
    "glass_bunny_soft_8k": "glass-bunny + shadow soft @ 7680x4320 (BASELINE.json configs[4])",
    "f4_directional_4k": "water_bunny_tex + a directional light @ 3840x2160, hard shadows (SURVEY section 8 f4)",
    "f4_bump_4k": "water_bunny_tex with a normal-mapped wall @ 3840x2160, hard shadows (SURVEY section 8 f4)",
    "f4_spheres_1k_4k": "1024 spheres over a floor, 2 lights, no bunny @ 3840x2160, hard shadows (SURVEY section 8 f4)",
}
PER_CONFIG = ["config", "bunny_shadow_4k", "gla_bunny_tex_4k", "glass_bunny_soft_8k", "f4_directional_4k", "f4_bump_4k",
              "f4_spheres_1k_4k"]
# Reference traversal work per ray (BASELINE.md section 2): box tests, triangle tests -> FLOPs at 21 / 61 per test
ALGO_TESTS = {"config": (75.1, 4.11), "bunny_shadow_4k": (77.5, 4.28), "gla_bunny_tex_4k": (69.5, 4.30),
              "water_bunny_tex_soft_4k": (48.6, 2.86), "glass_bunny_soft_8k": (48.6, 2.86),
              # f4 workloads: not in SURVEY's table; the bunny scenes reuse gla_bunny_tex's counts, the sphere field is
              # counted by the oracle (median-split tree over 1026 objects)
              "f4_directional_4k": (69.5, 4.30), "f4_bump_4k": (69.5, 4.30), "f4_spheres_1k_4k": (40.0, 3.0)}
# Algorithmic HBM bytes per unit of each traversal kernel (DESIGN.md section 6): what one launch must move
# at minimum.  (SURVEY.md section 8d's 112 B/ray is the whole pipeline's queue traffic per closest-hit ray.)
ALGO_BYTES = {
    "trace_closest": 48.0,                 # ray 2 x float4 read + hit float4 written, per ray
    "shadow_hard": 36.0,                   # request 32 B read + coefficient 4 B written, per ray
    # one 32 B request + 8 B list reference + 4 B coefficient serve 50 sample rays, which also read the request's
    # candidate list once (written once by k_soft_lists): ~25 members x 4 B x (write + read) per request
    "shadow_soft": (44.0 + 8.0 * 25.0) / 50.0,
    "soft_lists": 32.0 + 8.0 + 4.0 * 25.0, # per request: request read, reference + list written
    "shadow_directional": 36.0,
}


# --dump-outputs: at most this many bytes of .npy data; a larger frame is dumped as a fixed, seeded pixel sample
DUMP_BUDGET_BYTES = 64 << 20
DUMP_SAMPLE_PIXELS = 1 << 21
DUMP_SEED = 0
DUMP_COUNTS = ("closest_rays", "shadow_rays", "shadow_requests")     # + rays_per_depth


def flops_per_ray(workload):
    b, t = ALGO_TESTS[workload]
    return 21.0 * b + 61.0 * t


def peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


class quiet_stdout:
    """The reference prints progress to stdout; keep bench.py's stdout to the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def prepare_scene(workload, workdir):
    from whittedstyle_raytracer_b200 import Scene, fixtures
    fixtures.ensure_assets(workdir)
    fixtures.write_config(workdir, workload, fixtures.bench_config_text(workload))
    glass = bool(fixtures.BENCH_CONFIGS[workload].get("glass"))
    bunny = bool(fixtures.BENCH_CONFIGS[workload].get("bunny", True))
    return Scene.from_workdir(workdir, workload, bunny=bunny, glass=glass), glass


# --------------------------------------------------------------------------------------
# reference arm: the unmodified reference on the host cores
# --------------------------------------------------------------------------------------
def cpu_reference_sample(scene, workdir, workload, glass, target_seconds):
    """Traces a strided pixel sample of the workload's frame with the reference's own traceRay
    (oracle/_ref/libwhitted_ref.so, 1 thread — the reference has no threading), or with the
    oracle port (all cores) when the reference library did not travel.  Returns a dict."""
    sys.path.insert(0, str(REPO / "tests"))
    import numpy as np
    import oracle_bindings as ob
    w, h = scene.width, scene.height
    soft = scene.desc.shadow_type != 0
    rays_per_px = 90.0 if soft else 4.0
    ref_rate = 1.5e6 if soft else 0.7e6                      # measured rate of the reference on the GPU box host (rays/s)
    if ob.have_reference():
        want_px = max(256.0, target_seconds * ref_rate / rays_per_px)
        stride = max(1, int(round((w * h / want_px) ** 0.5)))
        with quiet_stdout():
            from whittedstyle_raytracer_b200 import fixtures
            ref = ob.ReferenceScene(workdir, workload, glass=glass, bunny=bool(fixtures.BENCH_CONFIGS[workload].get("bunny", True)))
            o, d = ob.OracleScene(scene).primary_rays()
            o = o.reshape(h, w, 3)[::stride, ::stride].reshape(-1, 3)
            d = d.reshape(h, w, 3)[::stride, ::stride].reshape(-1, 3)
            ref.counters(reset=True)
            _, secs = ref.trace_pixels(o, d)
            closest, shadow = ref.counters(reset=True)
        rays = closest + shadow
        return dict(value=rays / secs / 1e6, unit=UNIT, cores=1, kind="reference", seconds=secs, rays=rays,
                    sample=f"every {stride}th pixel in x and y of the {w}x{h} frame ({len(o)} primary rays, {rays} rays) "
                           f"through the unmodified reference's traceRay, 1 thread (the reference is single-threaded)")
    cores = os.cpu_count() or 1
    want_px = max(256.0, target_seconds * ref_rate * cores * 0.5 / rays_per_px)
    stride = max(1, int(round((w * h / want_px) ** 0.5)))
    t0 = time.time()
    _, st = ob.OracleScene(scene).render(stride=(stride, stride))
    secs = time.time() - t0
    rays = st.closest_rays + st.shadow_rays
    return dict(value=rays / secs / 1e6, unit=UNIT, cores=cores, kind="port", seconds=secs, rays=rays,
                sample=f"every {stride}th pixel in x and y of the {w}x{h} frame ({rays} rays) through the oracle port "
                       f"(oracle/whitted_oracle.c, OpenMP, {cores} threads); oracle/_ref was not available")


def _reference_worker(job):
    """One of P independent processes of the all-cores figure: loads the unmodified reference, traces its interleaved
    share of the pixel sample, returns (rays, seconds of its trace_pixels call)."""
    workdir, workload, glass, bunny, rays_file, part, parts = job
    sys.path.insert(0, str(REPO / "tests"))
    import numpy as np
    import oracle_bindings as ob
    od = np.load(rays_file, mmap_mode="r")                  # (o, d) pairs, shared through the page cache
    o, d = np.array(od[part::parts, 0]), np.array(od[part::parts, 1])
    with quiet_stdout():
        ref = ob.ReferenceScene(workdir, workload, glass=glass, bunny=bunny)
        ref.counters(reset=True)
        _, secs = ref.trace_pixels(o, d)
        closest, shadow = ref.counters(reset=True)
    return closest + shadow, float(secs)


def cpu_reference_all_cores(scene, workdir, workload, glass, target_seconds, procs=None):
    """The host's whole-socket figure beside the 1-thread one: P independent processes of the unmodified reference, each
    tracing an interleaved share of a (P times larger) pixel sample.  NOT how the reference runs — it has no threading
    (Renderer.hpp:104-131 is one serial loop) — so it is reported beside the arm's value, never as it.  None when the
    reference library did not travel."""
    sys.path.insert(0, str(REPO / "tests"))
    import multiprocessing as mp
    import numpy as np
    import oracle_bindings as ob
    if not ob.have_reference():
        return None
    from whittedstyle_raytracer_b200 import fixtures
    procs = procs or max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    procs = min(procs, 64)                                  # bounded: process start + scene load per worker, memory
    w, h = scene.width, scene.height
    soft = scene.desc.shadow_type != 0
    rays_per_px = 90.0 if soft else 4.0
    ref_rate = 1.5e6 if soft else 0.7e6
    want_px = min(float(w * h), 2.1e6, max(256.0 * procs, target_seconds * ref_rate * procs / rays_per_px))
    stride = max(1, int(round((w * h / want_px) ** 0.5)))
    o, d = ob.OracleScene(scene).primary_rays()
    o = o.reshape(h, w, 3)[::stride, ::stride].reshape(-1, 3)
    d = d.reshape(h, w, 3)[::stride, ::stride].reshape(-1, 3)
    # (neighbouring sample pixels go to different processes: the bunny's pixels, where the rays are, spread evenly)
    rays_file = str(Path(workdir) / "all_cores_rays.npy")
    np.save(rays_file, np.stack([o, d], axis=1).astype(np.float32))
    bunny = bool(fixtures.BENCH_CONFIGS[workload].get("bunny", True))
    jobs = [(str(workdir), workload, glass, bunny, rays_file, k, procs) for k in range(procs)]
    t0 = time.time()
    with mp.get_context("spawn").Pool(procs) as pool:
        res = pool.map_async(_reference_worker, jobs).get(timeout=60.0 + 10.0 * target_seconds)   # (a dead worker must not hang the arm)
    wall = time.time() - t0
    rays = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return dict(value=rays / slowest / 1e6, unit=UNIT, cores=procs, kind="reference x P processes", rays=rays,
                seconds=slowest, wall_seconds_with_process_start_and_scene_load=wall,
                sample=f"every {stride}th pixel in x and y of the {w}x{h} frame ({len(o)} primary rays, {rays} rays), "
                       f"interleaved over {procs} independent processes of the unmodified reference; rate = all rays / the "
                       f"slowest process's trace time.  Not the reference's own mode of operation (it is single-threaded)")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    workdir = Path(tempfile.mkdtemp(prefix="wrt_bench_ref_"))
    scene, glass = prepare_scene(args.workload, workdir)
    total = args.steps + args.warmup
    per_step = min(10.0, max(1.0, 150.0 / max(1, total)))      # the whole arm stays within ~2.5 minutes
    if args.ref_step_seconds is not None:
        per_step = args.ref_step_seconds
    vals, last = [], None
    for i in range(total):
        last = cpu_reference_sample(scene, workdir, args.workload, glass, per_step)
        if i >= args.warmup:
            vals.append(last)
    rays = sum(v["rays"] for v in vals)
    secs = sum(v["seconds"] for v in vals)
    value = rays / secs / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / max(1, len(vals)) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC[args.workload], "step": "bounded pixel sample of the frame: " + last["sample"]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_all_cores:
        try:
            line["all_cores"] = cpu_reference_all_cores(scene, workdir, args.workload, glass, min(8.0, per_step))
        except Exception as e:                                   # the arm's own number must not depend on it
            line["all_cores"] = {"unavailable": f"{type(e).__name__}: {e}"}
    emit(line)
    return 0


# --------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------
KERNEL_NAMES = {"shadow_soft": "k_soft_list_rays", "soft_lists": "k_soft_lists", "trace_closest": "k_trace_closest",
                "shadow_hard": "k_shadow_hard", "surface": "k_surface_spawn", "shadow_directional": "k_shadow_directional",
                "shade": "k_shade", "combine": "k_combine_resolve", "soft_filter": "k_soft_filter"}


def dump_outputs(out_dir, image, counts):
    """--dump-outputs: what the timed path returned in its last step, as .npy files in `out_dir`.  image.npy is the
    (H, W, 3) frame as float32 or, when that would exceed half of DUMP_BUDGET_BYTES, the pixels at DUMP_SAMPLE_PIXELS
    fixed, seeded positions ((N, 3) float32, positions y * W + x in image_pixel_index.npy); every entry of `counts`
    (the frame's ray counts) goes to <name>.npy as float64."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    h, w, _ = image.shape
    if h * w * 3 * 4 > DUMP_BUDGET_BYTES // 2:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, DUMP_SAMPLE_PIXELS, replace=False))
        np.save(out / "image.npy", image.reshape(-1, 3)[idx].astype(np.float32))
        np.save(out / "image_pixel_index.npy", idx.astype(np.float64))
    else:
        np.save(out / "image.npy", image.astype(np.float32))
    for name, v in counts.items():
        np.save(out / f"{name}.npy", np.asarray(v, dtype=np.float64))


def measure_workload(workload, steps, warmup, dist_env, cpu_seconds, want_clocks, dump_dir=None):
    """Benchmarks one workload on this rank (all ranks call it together).  Returns the JSON-line dict on rank 0.
    With `dump_dir`, rank 0 also writes the frame and ray counts of the last timed step there (dump_outputs)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from whittedstyle_raytracer_b200 import cabi
    from whittedstyle_raytracer_b200.parallel import DistributedRenderer

    world, rank, local = dist_env

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    workdir = Path(tempfile.mkdtemp(prefix=f"wrt_bench_{rank}_"))
    scene, glass = prepare_scene(workload, workdir)
    tile = tuple(int(x) for x in os.environ.get("WRT_TILE", "8x4").split("x"))
    dr = DistributedRenderer(scene, rank, world, local, tile=tile)
    ctx = dr.renderer.ctx
    w, h = scene.width, scene.height
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2

    def l2_flush():
        flush.fill_(rank + 1)

    sampler = ClockSampler(local) if (rank == 0 and want_clocks) else None      # started early: nvidia-smi needs ~1 s to emit
    # ---- warm-up ----
    for _ in range(max(warmup, 3)):
        dr.frame()
        stats = dr.finish()
    barrier()
    keys = ["rays", "closest_rays", "shadow_rays", "shaft_culled_requests", "unlit_skipped_requests", "shadow_rays_traced"]
    rays_t = torch.tensor([stats[k] for k in keys], dtype=torch.int64, device="cuda")
    per_rank_rays = torch.zeros(world, dtype=torch.int64, device="cuda")
    per_rank_rays[rank] = stats["closest_rays"] + stats["shadow_rays_traced"]
    if world > 1:
        dist.all_reduce(rays_t)
        dist.all_reduce(per_rank_rays)
    rays_frame, closest_frame, shadow_frame, culled_frame, unlit_frame, shadow_traced_frame = (int(x) for x in rays_t.tolist())
    traced_frame = closest_frame + shadow_traced_frame
    # Shadow requests that provably cannot change the image are answered without tracing (DESIGN.md section 4b).
    # `value` counts only the rays the kernels really trace; the reference's own count for the same image (it traces
    # all of them, SURVEY.md section 8d) is reported beside it as `reference_equivalent`.

    # ---- timed: device-resident scene, CUDA events on the launching (current) stream ----
    launches0 = ctx.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(steps)]
    barrier()
    t_wall0 = time.time()
    for k in range(steps):
        l2_flush()
        if world > 1:
            dist.barrier()
        dr.render_done = ev[k][2]
        ev[k][0].record()
        dr.frame()
        ev[k][1].record()
        last = dr.finish()
    dr.render_done = None
    barrier()
    t_wall1 = time.time()
    dump = None
    if dump_dir is not None:                    # the last timed step's frame and counts, before later passes overwrite them
        cnt = torch.tensor([last[k] for k in DUMP_COUNTS] + last["rays_per_depth"], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(cnt)
        cnt = cnt.tolist()
        if rank == 0:
            counts = dict(zip(DUMP_COUNTS, cnt))
            counts["rays_per_depth"] = cnt[len(DUMP_COUNTS):]
            dump = (dr.image.cpu().numpy(), counts)
    launches = ctx.launches - launches0
    ms_local = sum(a.elapsed_time(b) for a, b, _ in ev)
    render_local = sum(a.elapsed_time(c) for a, _, c in ev) / steps      # this rank's tiles only, no gather
    rr = torch.zeros(world, dtype=torch.float64, device="cuda")
    rr[rank] = render_local
    if world > 1:
        dist.all_reduce(rr)
    per_rank_render_ms = [round(float(x), 4) for x in rr.tolist()]
    ms_t = torch.tensor([ms_local], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms_t.item()) / steps
    value = traced_frame / (ms_per_step * 1e-3) / 1e6
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None

    # ---- per-kernel times of one frame (events around every launch, launches serialised; separate, untimed pass) ----
    ctx.enable_kernel_timing(True)
    fam_ms, fam_launches, fam_n = {}, {}, 3
    for _ in range(fam_n):
        l2_flush()
        dr.frame()
        dr.finish()
        for k2, v in ctx.kernel_times().items():
            fam_ms[k2] = fam_ms.get(k2, 0.0) + v / fam_n
        fam_launches = ctx.kernel_launches()
    ctx.enable_kernel_timing(False)
    barrier()

    # ---- e2e: host buffers through the C ABI; scene H2D + render + image D2H every step ----
    lib = cabi.load_cuda()
    host_img = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory()
    st = cabi.WrtStats()
    import ctypes as C
    d2h = 0

    def e2e_step():
        nonlocal d2h
        ctx._check(lib.wrt_upload_scene(ctx.h, scene.desc_ptr))
        ctx._check(lib.wrt_set_camera(ctx.h, scene.camera_ptr))
        if world == 1:
            ctx._check(lib.wrt_render(ctx.h, host_img.data_ptr(), C.byref(st)))
            d2h = h * w * 3
        else:
            img = dr.frame()
            dr.finish()
            if rank == 0:
                host_img.copy_(img, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                d2h = h * w * 3
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
        if world > 1:
            dist.barrier()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms_per_step = float(e2e_t.item()) / steps * 1e3
    e2e_value = traced_frame / (e2e_ms_per_step * 1e-3) / 1e6
    checksum = int(host_img.numpy().astype(np.uint64).sum()) if rank == 0 else 0

    # ---- roofline of the dominant kernel family ----
    hbm_peak, peak_src = peaks()
    dom = max(fam_ms, key=fam_ms.get)
    dom_share = fam_ms[dom] / max(1e-9, sum(fam_ms.values()))
    # units the dominant family processes in one frame on this rank
    if dom in ("shadow_soft", "shadow_hard", "shadow_directional"):
        dom_units = stats["shadow_rays_traced"]                  # rays the kernel really traces
    elif dom == "soft_lists":
        dom_units = stats["shadow_rays_traced"] // 50            # requests
    elif dom in ("trace_closest", "surface"):
        dom_units = stats["closest_rays"]
    else:
        dom_units = stats["closest_rays"] + stats["shadow_rays_traced"]
    dom_launches = max(1, int(fam_launches.get(dom, 1)))        # counted by the library during the run
    dom_s = fam_ms[dom] * 1e-3
    fma_tf, muladd_tf = ctx.measure_fp32_peak()
    fpr = flops_per_ray(workload)
    bpu = ALGO_BYTES.get(dom, 112.0)
    kname = KERNEL_NAMES.get(dom, f"k_{dom}")
    executed = profile_executed(kname)
    roofline = {
        "kernel": kname, "share_of_step": dom_share, "launches_per_step": dom_launches,
        "avg_launch_ms": fam_ms[dom] / dom_launches, "units_per_step": dom_units,
        "bound": "hbm", "achieved": dom_units * bpu / dom_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
        "frac": dom_units * bpu / dom_s / 1e9 / hbm_peak, "peak_source": peak_src,
        "algorithmic_bytes_per_unit": bpu, "algorithmic_bytes_per_launch": dom_units * bpu / dom_launches,
        "traffic": profile_traffic(kname),
        "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu "
                          "capture of this command (cannot be measured outside a profiler)",
        "binding_bound": "NOT hbm and not tensor: the L1 data pipe of a divergent per-lane walk (every lane fetches its own "
                         "128-byte node: l1tex__data_pipe_lsu_wavefronts at 87 % of peak on a deep level, profiles/NOTES.md) and "
                         "instruction issue at half-empty warps; `bound` says hbm only because the schema offers hbm|tensor — "
                         "`fp32.executed` (ncu counters of the work the kernel really executes) and `lane_issue_frac` say how "
                         "close to the SIMT roof it runs",
        # FP32, three views: (1) executed — from the committed ncu counters of this kernel (profiles/r02_exec_metrics.json):
        # FADD+FMUL+2*FFMA thread-instructions / its duration, and lane-issue utilisation = IPC/4 x active lanes/32;
        # (2) algorithmic — the reference's own traversal counts per ray (SURVEY.md section 8d) x the rays this kernel
        # traces, live time; (3) the measured FP32 peaks of this GPU.
        "fp32": {"executed": executed,
                 "algorithmic_flops_per_ray": fpr, "algorithmic_tflops": dom_units * fpr / dom_s / 1e12,
                 "peak_tflops_fma_measured": fma_tf, "peak_tflops_fmul_fadd_measured": muladd_tf,
                 "algorithmic_frac_of_fma_peak": dom_units * fpr / dom_s / 1e12 / max(fma_tf, 1e-9),
                 "algorithmic_frac_of_fmul_fadd_peak": dom_units * fpr / dom_s / 1e12 / max(muladd_tf, 1e-9)},
    }

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and cpu_seconds > 0:
        c = cpu_reference_sample(scene, workdir, workload, glass, cpu_seconds)
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cpu["seconds"] = c["seconds"]
        # time to the same image: the reference traces rays_frame rays for this frame
        cpu["frame_seconds_extrapolated"] = rays_frame / (c["value"] * 1e6)

    line = None
    if rank == 0:
        line = {
            "metric": METRIC if workload == DEFAULT_WORKLOAD else f"Mrays/s (all ray types), {WORKLOAD_DESC[workload]}",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "value_definition": "rays the kernels traced (closest-hit + shadow) / device time; the same frame costs the reference "
                                "`reference_equivalent.rays_per_frame` rays (it also traces the shadow rays whose result provably "
                                "cannot change the image, DESIGN.md section 4b)",
            "reference_equivalent": {"rays_per_frame": rays_frame, "mrays_per_s": rays_frame / (ms_per_step * 1e-3) / 1e6,
                                     "e2e_mrays_per_s": rays_frame / (e2e_ms_per_step * 1e-3) / 1e6},
            "config": {"workload": WORKLOAD_DESC[workload], "width": w, "height": h, "rays_traced_per_frame": traced_frame,
                       "closest_hit_rays": closest_frame, "shadow_rays_reference": shadow_frame,
                       "shadow_rays_traced": shadow_traced_frame,
                       "request_culling": {"shaft_empty_requests": culled_frame, "unlit_light_requests": unlit_frame,
                                           "note": "shadow requests answered without tracing: whole shaft to the area light "
                                                   "misses every leaf box (=50 lit samples) / light's diffuse+specular factors "
                                                   "exactly 0 (coefficient unused); bit-identical image; WRT_SHAFT_CULL=0 "
                                                   "WRT_UNLIT_CULL=0 disable"},
                       "parallelism": f"tiles{tile[0]}x{tile[1]}-interleaved x{world}" + ("+nccl-gather" if world > 1 else ""),
                       "traversal": "pruned", "l2": "flushed between timed steps (256 MiB write)",
                       "scene_bytes": scene.upload_bytes, "image_checksum": checksum},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms_per_step,
                    "h2d_bytes_per_step": int(scene.upload_bytes), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "launches_per_frame": int(launches) // steps,
            "kernel_ms_per_step": fam_ms,
            "kernel_launches_per_step": fam_launches,
            "per_rank_render_ms": per_rank_render_ms,
            "per_rank_rays_traced": [int(x) for x in per_rank_rays.tolist()],
            "roofline": roofline,
            "cpu_baseline": cpu,
            # `value` counts traced rays, so every shadow ray answered exactly without tracing LOWERS it while the frame gets
            # faster; the like-for-like comparison with the reference is the time to the same (bit-identical) image
            "time_to_image": None if cpu is None else {
                "frame_ms_device": ms_per_step, "frame_ms_e2e": e2e_ms_per_step,
                "reference_frame_s": cpu["frame_seconds_extrapolated"],
                "speedup_device": cpu["frame_seconds_extrapolated"] / (ms_per_step * 1e-3),
                "speedup_e2e": cpu["frame_seconds_extrapolated"] / (e2e_ms_per_step * 1e-3),
                "note": "reference_frame_s = the frame's reference ray count / the reference's measured rays per second "
                        "(cpu_baseline, 1 thread: the reference is single-threaded)"},
            "clocks": clocks,
        }
    barrier()
    dr.close()
    del flush
    torch.cuda.empty_cache()
    if dump is not None:
        dump_outputs(dump_dir, *dump)
    return line


def run_cuda_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with --nproc-per-node {args.gpus} (one rank per GPU)")
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    env = (world, rank, local)
    cpu_s = 0.0 if args.no_cpu_baseline else args.cpu_seconds
    line = measure_workload(args.workload, args.steps, args.warmup, env, cpu_s, True, args.dump_outputs)
    # The other BASELINE.json configs and the section-8 f4 workloads ride along in the same line (N = 1 only, fewer
    # steps, a smaller CPU sample each) so that the driver's record carries all of them.
    if world == 1 and args.workload == DEFAULT_WORKLOAD and not args.no_per_config:
        per = {}
        keep = ("metric", "value", "unit", "ms_per_step", "steps", "reference_equivalent", "e2e", "launches_per_frame",
                "kernel_ms_per_step", "kernel_launches_per_step", "cpu_baseline")
        for name in PER_CONFIG:
            try:
                r = measure_workload(name, min(args.steps, 5), 3, env, 0.0 if args.no_cpu_baseline else args.per_config_cpu_seconds, False)
                per[name] = {k: r[k] for k in keep}
                per[name]["rays_traced_per_frame"] = r["config"]["rays_traced_per_frame"]
                per[name]["image_checksum"] = r["config"]["image_checksum"]
                per[name]["dominant_kernel"] = {k: r["roofline"][k] for k in ("kernel", "share_of_step", "avg_launch_ms", "launches_per_step")}
            except Exception as e:                                  # a failing side workload must not lose the headline
                per[name] = {"error": f"{type(e).__name__}: {e}"}
        line["per_config"] = per
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def profile_executed(kernel):
    """Executed-work counters of `kernel` from the committed ncu capture (tools/summarize_ncu.py --exec):
    smsp__sass_thread_inst_executed_op_{fadd,fmul,ffma}_pred_on.sum, smsp__inst_executed.sum,
    smsp__thread_inst_executed.sum, IPC and duration -> executed TFLOP/s and lane-issue utilisation."""
    p = REPO / "profiles" / "r02_exec_metrics.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            e = d.get("kernels", {}).get(kernel)
            if e is not None:
                e = dict(e)
                e["source"] = f"profiles/r02_exec_metrics.json ({d.get('command', 'ncu')})"
            return e
        except (ValueError, OSError):
            return None
    return None


def profile_traffic(family):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/*.json written by tools/summarize_ncu.py), or None."""
    p = REPO / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(family)
        except (ValueError, OSError):
            return None
    return None


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else any library prints to fd 1
    (NCCL's version banner, the reference's progress text) was rerouted to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOAD_DESC))
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="size of the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true", help="skip the other configs' short runs (per_config)")
    ap.add_argument("--no-all-cores", action="store_true",
                    help="reference arm: skip the extra figure from P independent reference processes (all_cores)")
    ap.add_argument("--per-config-cpu-seconds", type=float, default=4.0)
    ap.add_argument("--ref-step-seconds", type=float, default=None,
                    help="--impl reference: CPU seconds per step's pixel sample (default: 150 s / (steps + warmup), 1..10 s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of --workload, write its last step's frame and ray counts to "
                         "DIR/<name>.npy (float32 / float64, at most 64 MiB: a larger frame as a fixed, seeded pixel "
                         "sample); the per_config runs that follow the default workload are not dumped")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    if args.dump_outputs is not None and args.impl == "reference":
        raise SystemExit("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_cuda_arm(args)


if __name__ == "__main__":
    sys.exit(main())
