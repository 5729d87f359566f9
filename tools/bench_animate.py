#!/usr/bin/env python
"""Measures animated scenes on one GPU: spheres moved on the device with a refitted BVH (r1_scene_move_spheres), the camera moved
(r1_scene_move_camera) and the spheres recoloured (r1_scene_set_materials) on the device, against a device rebuild of the tree,
against re-committing the scene every frame, and against the host path of a new scene per frame.

Scenes: `make_scene.py --cloud 100000`, `--grid 316 316` and `--cloud 1000000`.  Each runs `--frames` frames of seeded linear
motion: every sphere of radius < 100 (not the ground) moves along a fixed random velocity, scaled so that by the last frame it has
travelled `--travel` times the scene's extent -- far enough to tangle a tree whose topology was built for frame 0.  The camera
orbits the scene's look-at point, `--orbit` degrees per frame, and every moving Lambertian or metal sphere is coloured by its speed,
with a hue that turns each frame.  Positions, camera constants (r1_camera_constants) and colours are computed in numpy and uploaded
to the GPU before the timed region.  Per frame:
  - refit: move + refit on a scene that keeps its frame-0 tree; device ms (CUDA events of the call) and host wall time;
  - camera: move_camera on that scene, wall time (no device work: the constants reach the next launch by value);
  - materials: set_materials of every sphere's albedo on that scene, device ms and wall time;
  - rebuild: move + r1_scene_build_bvh(DEVICE) on a second copy (which also gets the camera and the colours); device ms and wall
    time of both calls;
  - re-commit: what a new camera needs without move_camera -- r1_scene_set_camera_raw + r1_scene_commit (which restores the
    committed positions and drops the tree) + move every sphere again + r1_scene_build_bvh(DEVICE), on a third copy; wall time.
    Materials have no such path: only a new scene changes them;
  - host path: r1_scene_commit + r1_scene_build_bvh(HOST) (host build and upload) of a new scene of the frame's values, wall time
    (creating that scene from its file is reported apart, as `host_scene_create_s`);
  - BVH Mrays/s at `--size` with the refit tree and with the rebuilt tree, alternated `--runs` times with L2 overwritten (256 MiB)
    before every render.
The refit and rebuilt images must be byte-equal (and ray counts equal), and both must equal the image of the freshly committed scene
of the frame's positions, camera and colours, on every frame.  The card's name, power limit and SM clocks come from
`nvidia-smi --query-gpu` (read-only) in the same call.  The JSON goes to stdout and, with --out, to a file, only after a complete
run.  There is no CPU path.

    python tools/bench_animate.py [--frames 6] [--runs 3] [--size 640 360 32] [--out profiles/r05_bench_animate.json]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_tensor_stream import ClockSampler, gpu_info  # noqa: E402

SCENES = {"cloud1e5": ("cloud", 100000), "grid1e5": ("grid", (316, 316)), "cloud1e6": ("cloud", 1000000)}
ASPECT = np.float32(1280) / np.float32(720)   # the aspect of scene-file cameras at r1_host_configure's default image size


def scene_spheres(name):
    import make_scene
    kind, arg = SCENES[name]
    if kind == "cloud":
        return make_scene.cloud_scene(arg)
    gw, gh = arg
    scale = max(gw / 30.0, gh / 16.0)
    return make_scene.grid_scene(gw, gh, 480, (3 * scale, 8 * scale, 15 * scale), 10.0 * scale)


def positions(soa, frames, travel, seed):
    """[frames, n, 3] float32 centres: frame 0 = the scene, then linear motion of every sphere of radius < 100"""
    c0 = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1).astype(np.float64)
    moving = soa["inv_radius"] > 0.01
    extent = float((c0[moving].max(0) - c0[moving].min(0)).max())
    v = np.random.default_rng(seed).normal(size=c0.shape) * moving[:, None]
    v *= travel * extent / max(frames - 1, 1) / np.sqrt(3.0)
    return np.stack([c0 + k * v for k in range(frames)]).astype(np.float32)


def cameras(cam, frames, orbit_deg):
    """per frame, a scene-file camera statement (from xyz, at xyz, vfov, aperture, focus) of float32 values: `cam` turned about the
    vertical through its look-at point by orbit_deg per frame"""
    frm, at = np.array(cam[0:3], np.float64), np.array(cam[3:6], np.float64)
    d = frm - at
    out = []
    for k in range(frames):
        a = np.radians(orbit_deg * k)
        turned = at + (d[0] * np.cos(a) + d[2] * np.sin(a), d[1], d[2] * np.cos(a) - d[0] * np.sin(a))
        out.append(tuple(float(np.float32(v)) for v in tuple(turned) + tuple(cam[3:])))
    return out


def colours(soa, pos):
    """[frames, n, 3] float32 albedos: every moving Lambertian or metal sphere coloured by its speed, the hue turning each frame;
    the other spheres keep theirs (a scene file gives dielectrics no albedo)"""
    frames = len(pos)
    speed = np.linalg.norm(pos[-1].astype(np.float64) - pos[0], axis=1)
    u = speed / max(float(speed.max()), 1e-30)
    recolour = (soa["inv_radius"] > 0.01) & np.isin(soa["kind"], (0, 1))
    out = np.repeat(soa["albedo"][None], frames, 0)
    for k in range(frames):
        hue = (u + 0.15 * k)[:, None] + np.array([0.0, 1.0 / 3.0, 2.0 / 3.0])
        out[k][recolour] = (0.5 + 0.4 * np.cos(2 * np.pi * hue))[recolour]
    return out.astype(np.float32)


def render(r1, s, flush, torch, size):
    flush.zero_()
    torch.cuda.synchronize()
    return s.render(*size, variant=r1.VARIANT_MEGAKERNEL_BVH)


def run_scene(r1, torch, name, flush, args, tmp):
    cam, sph = scene_spheres(name)
    path = os.path.join(tmp, name + ".r1scene")
    r1.write_scene_file(path, cam, sph)
    refit_s, rebuild_s, recommit_s = (r1.create_scene_from_file(path) for _ in range(3))
    soa = refit_s.soa()
    n = len(soa["cx"])
    pos = positions(soa, args.frames, args.travel, args.seed)
    alb = colours(soa, pos)
    cams = cameras(cam, args.frames, args.orbit)
    cam22 = [r1.camera_constants(c[0:3], c[3:6], (0, 1, 0), c[6], ASPECT, c[7], c[8]) for c in cams]
    size = tuple(args.size)
    entry = {"spheres": n, "frames": []}
    try:
        for s in (refit_s, rebuild_s, recommit_s):
            s.build_bvh(r1.BVH_BUILD_DEVICE)
            s.set_materials(albedo=torch.from_numpy(soa["albedo"]).cuda(0))     # warm-up: the scene's own colours
            render(r1, s, flush, torch, (96, 54, 4))                         # warm-up
        for k in range(args.frames):
            d_pos = torch.from_numpy(pos[k]).cuda(0)
            d_alb = torch.from_numpy(alb[k]).cuda(0)
            torch.cuda.synchronize()
            fr = {"frame": k}
            t0 = time.perf_counter()
            fr["refit_device_ms"] = refit_s.move_spheres(d_pos)
            fr["refit_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            t0 = time.perf_counter()
            refit_s.move_camera(cam22[k])
            fr["camera_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            t0 = time.perf_counter()
            fr["materials_device_ms"] = refit_s.set_materials(albedo=d_alb)
            fr["materials_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            t0 = time.perf_counter()
            ms_move = rebuild_s.move_spheres(d_pos)
            ms_build = rebuild_s.build_bvh(r1.BVH_BUILD_DEVICE)
            fr["rebuild_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            fr["rebuild_device_ms"] = ms_move + ms_build
            rebuild_s.move_camera(cam22[k])
            rebuild_s.set_materials(albedo=d_alb)
            # a new camera without move_camera: install it on the host and re-commit, then move and rebuild again
            t0 = time.perf_counter()
            recommit_s.set_camera_raw(cam22[k], 0)
            recommit_s.move_spheres(d_pos)
            recommit_s.build_bvh(r1.BVH_BUILD_DEVICE)
            fr["recommit_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            # the host path: a new scene of this frame's values, committed, with the host tree built and uploaded
            fpath = os.path.join(tmp, "%s_frame.r1scene" % name)
            r1.write_scene_file(fpath, cams[k], [tuple(pos[k][i]) + tuple(sp[3:5]) + tuple(alb[k][i]) + (sp[8],) for i, sp in enumerate(sph)])
            t0 = time.perf_counter()
            fresh = r1.create_scene_from_file(fpath, commit=False)
            fr["host_scene_create_s"] = time.perf_counter() - t0
            try:
                t0 = time.perf_counter()
                r1._check(r1.lib.r1_scene_commit(fresh.handle, 0), "r1_scene_commit")
                fresh.build_bvh(r1.BVH_BUILD_HOST)
                fr["host_path_s"] = time.perf_counter() - t0
                runs = {"refit": [], "rebuilt": []}
                images = {}
                for _ in range(args.runs):
                    for label, s in (("refit", refit_s), ("rebuilt", rebuild_s)):
                        rgb, res = render(r1, s, flush, torch, size)
                        runs[label].append({"mrays_per_s": res.num_rays / (res.kernel_ms * 1e-3) / 1e6, "kernel_ms": res.kernel_ms})
                        images.setdefault(label, (rgb, res.num_rays))
                fr["median_mrays_per_s"] = {b: float(np.median([r["mrays_per_s"] for r in rs])) for b, rs in runs.items()}
                fr["runs"] = runs
                (a, ra), (b, rb) = images["refit"], images["rebuilt"]
                fr["refit_equals_rebuilt"] = bool(np.array_equal(a, b) and ra == rb)
                c, rc = render(r1, fresh, flush, torch, size)
                fr["equals_fresh_commit"] = bool(np.array_equal(a, c) and ra == rc.num_rays)
            finally:
                fresh.close()
            entry["frames"].append(fr)
            print("%-9s frame %d: move+refit %.3f ms (wall %.3f), camera wall %.3f ms, materials %.3f ms (wall %.3f), move+rebuild %.3f ms "
                  "(wall %.3f), re-commit %.3f ms wall, host path %.3f s; Mrays/s refit %.0f, rebuilt %.0f; equal %s, fresh %s"
                  % (name, k, fr["refit_device_ms"], fr["refit_wall_ms"], fr["camera_wall_ms"], fr["materials_device_ms"], fr["materials_wall_ms"],
                     fr["rebuild_device_ms"], fr["rebuild_wall_ms"], fr["recommit_wall_ms"], fr["host_path_s"], fr["median_mrays_per_s"]["refit"],
                     fr["median_mrays_per_s"]["rebuilt"], fr["refit_equals_rebuilt"], fr["equals_fresh_commit"]), file=sys.stderr, flush=True)
            if not fr["refit_equals_rebuilt"] or not fr["equals_fresh_commit"]:
                raise SystemExit("%s frame %d: images differ" % (name, k))
    finally:
        refit_s.close()
        rebuild_s.close()
        recommit_s.close()
    return entry


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--travel", type=float, default=0.05, help="distance a moving sphere covers by the last frame, in scene extents")
    ap.add_argument("--orbit", type=float, default=3.0, help="degrees the camera turns about the scene per frame")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--size", type=int, nargs=3, default=(640, 360, 32), metavar=("W", "H", "SPP"))
    ap.add_argument("--scenes", nargs="+", default=list(SCENES), choices=list(SCENES))
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()
    if args.frames < 2:
        ap.error("--frames must be at least 2")

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement has no CPU path")
    import rays1bench_b200 as r1
    if r1.device_count() < 1:
        raise SystemExit("no CUDA device visible to the library")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    result = {"gpu": gpu_info(), "size": list(args.size), "frames": args.frames, "runs": args.runs, "travel": args.travel, "orbit_deg": args.orbit, "scenes": {}}
    with tempfile.TemporaryDirectory() as tmp, ClockSampler() as clocks:
        for name in args.scenes:
            result["scenes"][name] = run_scene(r1, torch, name, flush, args, tmp)
    result["sm_clock_samples_mhz"] = {"min": min(clocks.samples, default=0.0), "median": float(np.median(clocks.samples)) if clocks.samples else 0.0,
                                      "max": max(clocks.samples, default=0.0)}
    text = json.dumps(result)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
