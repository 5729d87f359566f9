#!/usr/bin/env python
"""Writes scene description files for rays1_b200 --scene-file (SURVEY.md 8f rank 3: sphere-count sweeps without a
recompile).  `--preset large` reproduces create_large_scene() (src/latest/rayweek1.cpp:654-719 of the reference) through
the file format; `--grid W H` builds the same recipe on a W x H grid (66 x 62 = the synthetic 4096-sphere scene).
`--cloud N [--seed S]` scatters N overlapping spheres of radii 0.02 .. 2 through a cube above a ground sphere: unlike the flat
grids, a hard case for a bounding volume hierarchy.

  python tools/make_scene.py --grid 30 16 --out large.r1scene
  ./rays1bench_b200/rays1_b200 --scene-file large.r1scene --spp 64
"""
import argparse
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def fma32(a, b, c):
    """float32 fma: the product of two float32 values is exact in float64, one rounding at the end"""
    return np.float32(np.float64(np.float32(a)) * np.float64(np.float32(b)) + np.float64(np.float32(c)))


def grid_scene(gw, gh, ior_mod, lookfrom, focus):
    """The reference's large-scene recipe; colours from glibc srand(111)/rand() like the C++ builders."""
    libc = ctypes.CDLL(None)
    libc.srand(111)
    f = np.float32
    spheres = []
    for y in range(gh):
        for x in range(gw):
            px, py, pz = f(x - gw // 2) * f(1.1), f(0), f(y - gh // 2) * f(1.1)
            # the constant expressions as the reference's fast-math build evaluates them (rays1_host.cpp:grid_scene)
            r, g, b = (f(libc.rand() & 0xff) * (f(1.0) / f(255.0)) for _ in range(3))
            i = x + y * gw
            if i % 20 == 0:
                k = i % ior_mod if ior_mod else i
                spheres.append((px, py, pz, f(0.45), 2, 1, 1, 1, fma32(k, 0.05, 1.2)))
            elif i % 10 == 0:
                spheres.append((px, py + f(0.1), pz, f(0.45), 1, r, g, b, fma32(f(0.5) * f(y), f(1.0) / f(gh), 0.01)))
            else:
                spheres.append((px, py, pz, f(0.45), 0, r, g, b, 0))
    spheres.append((0, f(-1000.5), 0, 1000, 0, 0.5, 0.5, 0.5, 0))
    spheres.append((5, 3, 0, 2, 1, 0.5, 0.5, 0.8, 0.65))
    spheres.append((0, 3, 0, 2, 2, 1, 1, 1, 1.5))
    spheres.append((-5, 3, 0, 2, 1, 0.8, 0.2, 0.2, 0.05))
    camera = (*lookfrom, 0, 0, 0, 60, 0.1, focus)
    return camera, spheres


def cloud_scene(n, seed=1):
    """n spheres, centres uniform in a cube of side 2 n^(1/3) (at least 4) above the ground, radii log-uniform in [0.02, 2]
    (about 30 % of the cube's volume summed over the spheres: heavy overlap), 70 % Lambertian, 20 % metal, 10 % glass; then the
    ground sphere (radius 10 000) and a camera outside the cube looking at its centre."""
    rng = np.random.default_rng(seed)
    f = np.float32
    half = max(2.0, float(n) ** (1.0 / 3.0))
    c = rng.uniform(-half, half, (n, 3))
    c[:, 1] += half + 0.5
    r = np.exp(rng.uniform(np.log(0.02), np.log(2.0), n))
    kind = rng.choice([0, 1, 2], n, p=[0.7, 0.2, 0.1])
    col = rng.uniform(0.1, 0.9, (n, 3))
    fuzz = rng.uniform(0.0, 0.5, n)
    spheres = []
    for i in range(n):
        x, y, z = (f(v) for v in c[i])
        if kind[i] == 0:
            spheres.append((x, y, z, f(r[i]), 0, *(f(v) for v in col[i]), 0))
        elif kind[i] == 1:
            spheres.append((x, y, z, f(r[i]), 1, *(f(v) for v in col[i]), f(fuzz[i])))
        else:
            spheres.append((x, y, z, f(r[i]), 2, 1, 1, 1, f(1.5)))
    spheres.append((0, f(-10000), 0, 10000, 0, 0.5, 0.5, 0.5, 0))
    camera = (0, 1.6 * half + 1, 3.2 * half + 3, 0, half, 0, 50, 0.02, float(np.hypot(0.6 * half + 1, 3.2 * half + 3)))
    return camera, spheres


def main():
    import rays1bench_b200 as r1
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", choices=["large", "synth4096"])
    ap.add_argument("--grid", type=int, nargs=2, metavar=("W", "H"))
    ap.add_argument("--cloud", type=int, metavar="N")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if args.cloud:
        cam, sph = cloud_scene(args.cloud, args.seed)
    elif args.preset == "large" or (not args.preset and not args.grid):
        cam, sph = grid_scene(30, 16, 0, (3, 8, 15), 10.0)
    elif args.preset == "synth4096":
        cam, sph = grid_scene(66, 62, 480, (6, 16, 30), 20.0)
    else:
        gw, gh = args.grid
        scale = max(gw / 30.0, gh / 16.0)
        cam, sph = grid_scene(gw, gh, 480, (3 * scale, 8 * scale, 15 * scale), 10.0 * scale)
    r1.write_scene_file(args.out, cam, sph)
    print("%s: %d spheres" % (args.out, len(sph)))


if __name__ == "__main__":
    main()
