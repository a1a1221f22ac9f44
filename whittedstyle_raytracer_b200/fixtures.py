"""Deterministic scene fixtures: benchmark configs, synthetic coverage configs,
stand-in textures and the bunny mesh.

Why this exists (SURVEY.md section 0.1): the reference's texture blobs
(`textures/harbor.ppm` ...) are missing from the mount, no shipped config holds a
sphere / `shadow soft` / `bump` / `attlight` / `depthcueing`, and the 4K/8K
benchmark configs are derived from the shipped ones by rewriting `imsize`.
Both the CPU oracle and the CUDA path read the files this module writes, so
they always see identical inputs.

The scene *data* of the four shipped configs (config.txt == bunny_shadow.txt,
gla_bunny_tex.txt == out/water_bunny_tex.txt) is restated here token for token
(the grammar is whitespace-insensitive).  The Stanford bunny mesh the
reference's driver loads from `bunny.obj` (src/main.cpp:46) is kept as float32
positions + faces in assets/bunny_mesh.npz and written back as an OBJ whose
numbers round-trip through std::stof to exactly the same floats.
"""
from __future__ import annotations

import os
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
ASSETS = REPO / "assets"

_CAMERA = """imsize {w} {h}
eye 0 1 3
viewdir 0 0 -1
hfov 90
updir 0 1 0
bkgcolor 0.356 0.698 0.976 1.0
"""

_WALL_VERTS = """v -20 -20 -20
v 20 20 -20
v -20 20 -20
v 20 -20 -20
"""

_VT = """vt 0 1
vt 1 0
vt 0 0
vt 1 1
"""


def bunny_shadow_config(w: int = 800, h: int = 600, soft: bool = False) -> str:
    """config.txt / bunny_shadow.txt: floor + textured back wall (+ bunny from main())."""
    return (
        _CAMERA.format(w=w, h=h)
        + "\nlight -10 8 10 1 1 1 1\n"
        + ("shadow soft\n" if soft else "")
        + "\n" + _WALL_VERTS
        + "\nv -20 -7 2\nv 20 -7 -20\nv -20 -7 -20\nv 20 -7 2\n\n"
        + _VT
        + "\nmtlcolor 0.5 0.5 0.5 0.33 0.66 0.99 0.4 0.8 0 64 1 0.2\n"
        + "f 5 6 7\nf 5 8 6\n\n"
        + "texture textures/harbor.ppm\nf 1/1 2/2 3/3\nf 1/1 4/4 2/2\n"
    )


def water_bunny_tex_config(w: int = 800, h: int = 600, soft: bool = False) -> str:
    """gla_bunny_tex.txt / out/water_bunny_tex.txt: textured back wall (+ bunny from main())."""
    return (
        _CAMERA.format(w=w, h=h)
        + "\nlight -20 70 20 1 1 1 1\n"
        + ("shadow soft\n" if soft else "")
        + "\n" + _WALL_VERTS + "\n" + _VT
        + "\nmtlcolor 0.529 0.807 0.921 0.33 0.66 0.99 0.4 0.8 0 64 1 0.2\n"
        + "texture textures/harbor.ppm\nf 1/1 2/2 3/3\nf 1/1 4/4 2/2"
    )


# ---- synthetic coverage configs (features no shipped config exercises) ----

def spheres_config(w: int = 320, h: int = 240) -> str:
    """Spheres, attenuated light, depth cueing, textured sphere, light avatar, glass + mirror."""
    return f"""imsize {w} {h}
eye 0 2 8
viewdir 0 -0.15 -1
hfov 60
updir 0 1 0
bkgcolor 0.1 0.15 0.3 1.0
attlight 4 9 6 1 1 1 1 0.4 0.02 0.001
light -6 5 4 1 0.5 0.4 0.3
depthcueing 0.2 0.2 0.25 1.0 0.3 30 6
mtlcolor 0.8 0.2 0.2 1 1 1 0.2 0.7 0.4 32 1 1.5
sphere -2.5 0 -2 1.5
mtlcolor 0.9 0.9 1.0 1 1 1 0.05 0.1 0.3 80 0.15 1.5
sphere 1.2 0.3 0.5 1.3
mtlcolor 0.2 0.8 0.3 1 1 1 0.2 0.6 0.0 16 1 1.0
sphere 3.5 -0.5 -3 1.0
mtlcolor 1 1 1 1 1 1 1 1 1 0 1 1
sphere 4 9 6 0.3
mtlcolor 0.5 0.5 0.5 0.3 0.3 0.3 0.2 0.8 0.2 20 1 1.0
texture textures/harbor.ppm
sphere -0.5 3.2 -4 1.6
mtlcolor 0.6 0.6 0.6 1 1 1 0.3 0.7 0.1 10 1 1.0
v -12 -1.5 6
v 12 -1.5 6
v 12 -1.5 -14
v -12 -1.5 -14
f 1 2 3
f 1 3 4
"""


def parallel_config(w: int = 240, h: int = 180) -> str:
    return f"""imsize {w} {h}
eye 0 1 6
viewdir 0.1 -0.2 -1
hfov 70
updir 0 1 0
bkgcolor 0.3 0.3 0.35 1.0
projection parallel
light 5 8 8 1 1 1 1
mtlcolor 0.7 0.3 0.2 1 1 1 0.2 0.7 0.3 40 1 1.0
sphere -1 0.5 -1 1.2
mtlcolor 0.2 0.4 0.8 1 1 1 0.2 0.7 0.5 60 1 1.0
sphere 1.5 0.2 0 0.9
mtlcolor 0.5 0.6 0.5 1 1 1 0.3 0.6 0 8 1 1.0
v -6 -1 4
v 6 -1 4
v 6 -1 -8
v -6 -1 -8
f 1 2 3
f 1 3 4
"""


def bump_config(w: int = 240, h: int = 180) -> str:
    """Normal maps on a textured triangle pair and on a sphere (`bump` is one-shot)."""
    return f"""imsize {w} {h}
eye 0 1 7
viewdir 0 -0.1 -1
hfov 60
updir 0 1 0
bkgcolor 0.2 0.25 0.3 1.0
light 3 7 8 1 1 1 1
v -6 -2 -6
v 6 -2 -6
v 6 6 -6
v -6 6 -6
vt 0 1
vt 1 1
vt 1 0
vt 0 0
mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.3 30 1 1.0
texture textures/harbor.ppm
bump textures/bumps.ppm
f 1/1 2/2 3/3
bump textures/bumps.ppm
f 1/1 3/3 4/4
bump textures/bumps.ppm
sphere 0 0.5 -1 1.7
mtlcolor 0.4 0.7 0.4 1 1 1 0.2 0.7 0.2 20 1 1.0
bump textures/bumps.ppm
sphere -3 0 0 1.0
"""


def directional_config(w: int = 200, h: int = 150) -> str:
    """Directional light (w = 0): O(N) shadow loop that bypasses the BVH."""
    return f"""imsize {w} {h}
eye 0 2 9
viewdir 0 -0.2 -1
hfov 55
updir 0 1 0
bkgcolor 0.4 0.5 0.7 1.0
light -1 -2 -1.5 0 1 0.95 0.9
light 6 6 6 1 0.3 0.3 0.4
mtlcolor 0.8 0.5 0.2 1 1 1 0.2 0.7 0.3 25 1 1.0
sphere -1.5 0 0 1.4
mtlcolor 0.7 0.9 1.0 1 1 1 0.1 0.2 0.3 70 0.3 1.4
sphere 1.8 0.2 1 1.1
mtlcolor 0.5 0.5 0.55 1 1 1 0.3 0.7 0 10 1 1.0
v -10 -1.4 8
v 10 -1.4 8
v 10 -1.4 -10
v -10 -1.4 -10
f 1 2 3
f 1 3 4
"""


def smooth_config(w: int = 200, h: int = 150) -> str:
    """`vn` normals with the a//n and a/t/n face forms; a mirror quad; glass pyramid."""
    return f"""imsize {w} {h}
eye 0 1.5 7
viewdir 0 -0.15 -1
hfov 60
updir 0 1 0
bkgcolor 0.25 0.3 0.45 1.0
light 4 8 6 1 1 1 1
v -5 -1 5
v 5 -1 5
v 5 -1 -7
v -5 -1 -7
v -1.5 -1 0
v 1.5 -1 0
v 0 -1 -2.5
v 0 2 -1
v -5 -1 -7
v 5 -1 -7
v 5 6 -7
v -5 6 -7
vn 0 1 0
vn -0.7 0.5 0.5
vn 0.7 0.5 0.5
vn 0 0.5 -1
vn 0 1 0.2
vn 0 0 1
vt 0 0
vt 1 0
vt 1 1
vt 0 1
mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.7 0.2 20 1 1.0
f 1//1 2//1 3//1
f 1//1 3//1 4//1
mtlcolor 0.85 0.95 1.0 1 1 1 0.05 0.15 0.25 60 0.25 1.45
f 5//2 6//3 8//5
f 6//3 7//4 8//5
f 7//4 5//2 8//5
mtlcolor 0.9 0.9 0.9 1 1 1 0.1 0.3 0.8 100 1 1.0
texture textures/harbor.ppm
f 9/1/6 10/2/6 11/3/6
f 9/1/6 11/3/6 12/4/6
"""


COVERAGE_CONFIGS = {
    "spheres": spheres_config,
    "parallel": parallel_config,
    "bump": bump_config,
    "directional": directional_config,
    "smooth": smooth_config,
}


def _write_p3(path: Path, rgb: np.ndarray) -> None:
    h, w, _ = rgb.shape
    body = "\n".join(" ".join(map(str, px)) for px in rgb.reshape(-1, 3).tolist())
    path.write_text(f"P3\n{w} {h}\n255\n{body}\n")


def harbor_texture(w: int = 512, h: int = 256) -> np.ndarray:
    """Stand-in for the missing textures/harbor.ppm (same generator as SURVEY.md section 8d)."""
    i = np.arange(w)[None, :]
    j = np.arange(h)[:, None]
    r = np.broadcast_to(i * 255 // (w - 1), (h, w))
    g = np.broadcast_to(j * 255 // (h - 1), (h, w))
    b = ((i // 32 + j // 32) % 2) * 200 + 25
    return np.stack([r, g, b], axis=-1).astype(np.int64)


def bumps_texture(w: int = 64, h: int = 64) -> np.ndarray:
    """Tangent-space normal map: a grid of smooth bumps, encoded (n+1)/2*255."""
    x = (np.arange(w)[None, :] + 0.5) / w * 4 * np.pi
    y = (np.arange(h)[:, None] + 0.5) / h * 4 * np.pi
    nx = 0.45 * np.cos(x) * np.ones_like(y)
    ny = 0.45 * np.cos(y) * np.ones_like(x)
    nz = np.sqrt(np.clip(1 - nx * nx - ny * ny, 0, 1))
    n = np.stack([nx, ny, nz], axis=-1)
    return np.clip(np.floor((n + 1) * 0.5 * 255 + 0.5), 0, 255).astype(np.int64)


def write_bunny_obj(path: Path) -> None:
    m = np.load(ASSETS / "bunny_mesh.npz")
    pos, faces = m["positions"], m["faces"]
    with open(path, "w") as f:
        f.write("# Stanford bunny, 2503 vertices / 4968 faces (float32, %.9g round-trips through stof)\n")
        for p in pos:
            f.write("v %.9g %.9g %.9g\n" % (p[0], p[1], p[2]))
        for t in faces:
            f.write("f %d %d %d\n" % (t[0], t[1], t[2]))


def ensure_assets(workdir: os.PathLike | str) -> Path:
    """Creates `workdir` with textures/harbor.ppm, textures/bumps.ppm and bunny.obj
    (idempotent) — the cwd layout the reference executable expects."""
    wd = Path(workdir)
    (wd / "textures").mkdir(parents=True, exist_ok=True)
    if not (wd / "textures" / "harbor.ppm").exists():
        _write_p3(wd / "textures" / "harbor.ppm", harbor_texture())
    if not (wd / "textures" / "bumps.ppm").exists():
        _write_p3(wd / "textures" / "bumps.ppm", bumps_texture())
    if not (wd / "bunny.obj").exists():
        write_bunny_obj(wd / "bunny.obj")
    return wd


def write_config(workdir: os.PathLike | str, name: str, text: str) -> Path:
    p = Path(workdir) / f"{name}.txt"
    p.write_text(text)
    return p


# ---- SURVEY.md section 8 f4: the rarely used branches "at speed" (4K bench workloads) ----

def f4_directional_config(w: int = 3840, h: int = 2160, soft: bool = False) -> str:
    """The textured-wall bunny scene lit by a point light AND a directional light (w = 0): every shaded hit runs the
    box-free directional shadow loop of Renderer.hpp:381-400 over 4970 objects."""
    return water_bunny_tex_config(w, h, soft).replace("light -20 70 20 1 1 1 1",
                                                      "light -20 70 20 1 1 1 1\nlight 0.3 -1 -0.4 0 0.9 0.9 0.8")


def f4_bump_config(w: int = 3840, h: int = 2160, soft: bool = False) -> str:
    """The same scene with a normal map on both wall triangles (changeNormalDir, Renderer.hpp:417-474, on ~90 % of
    the primary hits; `bump` is one-shot, so it is repeated per face)."""
    t = water_bunny_tex_config(w, h, soft)
    return t.replace("texture textures/harbor.ppm\nf 1/1 2/2 3/3\nf 1/1 4/4 2/2",
                     "texture textures/harbor.ppm\nbump textures/bumps.ppm\nf 1/1 2/2 3/3\nbump textures/bumps.ppm\nf 1/1 4/4 2/2")


def f4_spheres_config(w: int = 3840, h: int = 2160, soft: bool = False) -> str:
    """1024 spheres (Sphere::intersect, Sphere.hpp:25-120, with its double-precision `C`) over a floor: a quarter
    glass, a quarter mirror-ish, a quarter textured; one plain and one attenuated point light; no bunny."""
    rng = np.random.default_rng(1024)
    lines = [f"imsize {w} {h}", "eye 0 6 16", "viewdir 0 -0.35 -1", "hfov 60", "updir 0 1 0", "bkgcolor 0.25 0.35 0.55 1.0",
             "light 12 30 14 1 0.8 0.8 0.8", "attlight -10 14 6 1 0.6 0.6 0.5 0.6 0.01 0.0005"]
    if soft:
        lines.append("shadow soft")
    mats = ["mtlcolor 0.8 0.3 0.2 1 1 1 0.2 0.7 0.3 32 1 1.0",
            "mtlcolor 0.9 0.95 1.0 1 1 1 0.05 0.2 0.4 60 0.25 1.45",
            "mtlcolor 0.7 0.7 0.75 1 1 1 0.1 0.4 0.7 80 1 1.0",
            "mtlcolor 0.6 0.6 0.6 1 1 1 0.2 0.8 0.2 20 1 1.0\ntexture textures/harbor.ppm"]
    k = 0
    for gy in range(32):
        for gx in range(32):
            if k % 256 == 0:
                lines.append(mats[k // 256])
            r = 0.22 + 0.16 * rng.random()
            x = (gx - 15.5) * 0.95 + 0.25 * (rng.random() - 0.5)
            z = -(gy * 0.95) + 4 + 0.25 * (rng.random() - 0.5)
            y = r - 1.0 + (1.2 * rng.random() if rng.random() < 0.3 else 0.0)
            lines.append("sphere %.4f %.4f %.4f %.4f" % (x, y, z, r))
            k += 1
    lines += ["mtlcolor 0.5 0.55 0.5 1 1 1 0.3 0.7 0.1 10 1 1.0", "v -40 -1 20", "v 40 -1 20", "v 40 -1 -60", "v -40 -1 -60",
              "f 1 2 3", "f 1 3 4"]
    return "\n".join(lines) + "\n"


# ---- geometry whose device-built (PLOC) tree is very deep: fans, slivers, nested sizes ----
# Body lines only (v / f / sphere, no header, no mtlcolor); face indices start at vertex 1, so a body must come before
# any other vertex of the config.  Numbers are fixed-point (%.6f): the config grammar rejects exponent notation.

def _ring(n: int, y: float) -> list[str]:
    return ["v %.6f %.6f %.6f" % (np.cos(2 * np.pi * i / n), y, np.sin(2 * np.pi * i / n)) for i in range(n)]


def fan_geometry(n: int) -> str:
    """A flat unit disc in y = 0 cut into n triangles that all share the centre vertex (0, 0, 0)."""
    lines = ["v 0.000000 0.000000 0.000000"] + _ring(n, 0.0)
    lines += ["f 1 %d %d" % (2 + i, 2 + (i + 1) % n) for i in range(n)]
    return "\n".join(lines) + "\n"


def cylinder_geometry(n: int) -> str:
    """Radius 1, y from 0 to 2: n side quads (two triangles each) and a fan cap around each end's centre; 4n triangles."""
    lines = ["v 0.000000 0.000000 0.000000", "v 0.000000 2.000000 0.000000"] + _ring(n, 0.0) + _ring(n, 2.0)
    lo = lambda i: 3 + i % n                           # noqa: E731
    hi = lambda i: 3 + n + i % n                       # noqa: E731
    for i in range(n):
        lines += ["f 1 %d %d" % (lo(i), lo(i + 1)), "f 2 %d %d" % (hi(i + 1), hi(i)),
                  "f %d %d %d" % (lo(i), hi(i), hi(i + 1)), "f %d %d %d" % (lo(i), hi(i + 1), lo(i + 1))]
    return "\n".join(lines) + "\n"


def sliver_geometry(n: int = 4000) -> str:
    """n thin triangles in z = 0 sharing the vertex (0, 0, 0), each 0.001 rad wide, spread around the full circle."""
    lines = ["v 0.000000 0.000000 0.000000"]
    for i in range(n):
        a = 2 * np.pi * i / n
        lines += ["v %.6f %.6f 0.000000" % (np.cos(a), np.sin(a)), "v %.6f %.6f 0.000000" % (np.cos(a + 0.001), np.sin(a + 0.001))]
    lines += ["f 1 %d %d" % (2 + 2 * i, 3 + 2 * i) for i in range(n)]
    return "\n".join(lines) + "\n"


def mixed_radius_spheres(n: int = 5000, seed: int = 1) -> str:
    """n spheres centred on the x axis in [-1, 1] with radii 10^U(-3, 2): tiny spheres nested inside huge ones."""
    import random
    rnd = random.Random(seed)
    lines = []
    for _ in range(n):
        x = rnd.uniform(-1, 1)
        lines.append("sphere %.6f 0 0 %.6f" % (x, 10 ** rnd.uniform(-3, 2)))
    return "\n".join(lines) + "\n"


def sphere_chain(n: int = 30) -> str:
    """Sphere k at (1.5^k, 0, 0) with radius 0.4 * 1.5^k: every sphere is larger than all the ones before it together."""
    return "".join("sphere %.6f 0 0 %.6f\n" % (1.5 ** k, 0.4 * 1.5 ** k) for k in range(n))


DEEP_TREE_GEOMETRY = {
    "fan_1000": lambda: fan_geometry(1000),
    "fan_2000": lambda: fan_geometry(2000),
    "cylinder_2000": lambda: cylinder_geometry(2000),
    "slivers_4000": lambda: sliver_geometry(4000),
    "mixed_radii_5000": lambda: mixed_radius_spheres(5000, 1),
    "chain_30": lambda: sphere_chain(30),
}


# BASELINE.json `configs`, in order.  (name, config text builder kwargs, uses bunny, soft)
BENCH_CONFIGS = {
    "config": dict(builder=bunny_shadow_config, w=800, h=600, soft=False),
    "bunny_shadow_4k": dict(builder=bunny_shadow_config, w=3840, h=2160, soft=False),
    "gla_bunny_tex_4k": dict(builder=water_bunny_tex_config, w=3840, h=2160, soft=False),
    "water_bunny_tex_soft_4k": dict(builder=water_bunny_tex_config, w=3840, h=2160, soft=True),
    "glass_bunny_soft_8k": dict(builder=water_bunny_tex_config, w=7680, h=4320, soft=True, glass=True),
    # SURVEY.md section 8 f4 (not BASELINE configs): directional light / normal maps / spheres at 4K
    "f4_directional_4k": dict(builder=f4_directional_config, w=3840, h=2160, soft=False),
    "f4_bump_4k": dict(builder=f4_bump_config, w=3840, h=2160, soft=False),
    "f4_spheres_1k_4k": dict(builder=f4_spheres_config, w=3840, h=2160, soft=False, bunny=False),
}


def bench_config_text(name: str, w: int | None = None, h: int | None = None) -> str:
    c = BENCH_CONFIGS[name]
    return c["builder"](w or c["w"], h or c["h"], c["soft"])
