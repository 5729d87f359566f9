#!/usr/bin/env python
"""Measures batches of views (r1_render_views_device) against the same views rendered one by one (r1_scene_move_camera +
r1_render_device per view) on one GPU.

Scenes: large (485 spheres: the tensor-core filter, tc3, by default), synth4096 (4096 spheres: PACKED by default) and a
`make_scene.py --cloud 100000` cloud on the BVH variant (built on the device).  Sizes: 64x64x16, 128x128x64 and 256x256x64, the
small images a multi-view caller renders, and 1280x720x250 as the control, where a render is long enough that its fixed costs do
not show.  K = 1, 8, 64 and 256 views (the control: 1 and 8 only, and not on the cloud, where one such view takes seconds), orbit
cameras around the scene's look-at point, seed v for view v.

Per (scene, size, K) both arms run on one stream into caller-owned device buffers, with CUDA events around the whole sequence:
  - single: K x (move_camera + render_device), one image buffer per view;
  - batch: one render_views_device into K images.
The arms alternate, `--runs` times each after one warm-up of each; the smallest time of each arm is reported, with the spread.  The
images and ray counts of both arms must be equal in every run, or the script fails.  Mrays/s = the views' rays over the sequence
time; ms per view = the sequence time over K.  The card's name, power limit and SM clocks come from `nvidia-smi --query-gpu`
(read-only) in the same call.  The JSON goes to stdout and, with --out, to a file, only after a complete run.  There is no CPU path.

    python tools/bench_views.py [--runs 3] [--out profiles/r06_bench_views.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_tensor_stream import gpu_info  # noqa: E402

SIZES = ((64, 64, 16), (128, 128, 64), (256, 256, 64), (1280, 720, 250))
KS = (1, 8, 64, 256)
CONTROL_KS = (1, 8)
F = np.float32


def make_scenes(r1):
    import make_scene
    r1.configure(width=1280, height=720, spp=250, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    out = {"large": (r1.create_scene("large"), r1.VARIANT_MEGAKERNEL, np.array((0, 0, 0), F), 14.0),
           "synth4096": (r1.create_scene("synth4096"), r1.VARIANT_MEGAKERNEL, None, None)}
    cam, sph = make_scene.cloud_scene(100000)
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), "bench_views_cloud.r1scene")
    r1.write_scene_file(path, cam, sph)
    cloud = r1.create_scene_from_file(path)
    os.unlink(path)
    cloud.build_bvh(r1.BVH_BUILD_DEVICE)
    out["cloud1e5"] = (cloud, r1.VARIANT_MEGAKERNEL_BVH, None, None)
    return out


def orbit_cams(r1, scene, k, target, dist):
    """k cameras on a quarter circle around `target` (default: the point `dist` ahead of the scene's camera, `dist` defaulting to
    the camera's distance from the world origin), at the height and distance of the scene's own camera"""
    c = scene.camera()
    origin, w = c[0:3].astype(np.float64), c[18:21].astype(np.float64)
    if dist is None:
        dist = float(np.linalg.norm(origin))
    if target is None:
        target = origin - dist * w
    rel = origin - target
    radius, height = float(np.hypot(rel[0], rel[2])), float(rel[1])
    a0 = float(np.arctan2(rel[0], rel[2]))
    out = []
    for v in range(k):
        a = a0 + 0.5 * np.pi * v / k
        frm = np.array([target[0] + radius * np.sin(a), target[1] + height, target[2] + radius * np.cos(a)], F)
        out.append(r1.camera_constants(frm, np.asarray(target, F), (0, 1, 0), 60.0, F(1280) / F(720), 0.1, float(np.linalg.norm(rel))))
    return np.stack(out)


def measure(r1, torch, scene, variant, cams, w, h, spp, runs):
    k = len(cams)
    npix = w * h
    seeds = np.arange(k, dtype=np.uint32)
    home = scene.camera()
    st = torch.cuda.Stream(0)
    single_rgb = torch.zeros((k, npix * 3), dtype=torch.uint8, device="cuda:0")
    single_rays = torch.zeros(k, dtype=torch.int64, device="cuda:0")
    batch_rgb = torch.zeros(k * npix * 3, dtype=torch.uint8, device="cuda:0")
    batch_rays = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    kw = dict(width=w, height=h, spp=spp, variant=variant)

    def single():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            for v in range(k):
                scene.move_camera(cams[v])
                scene.render_device(single_rgb[v].data_ptr(), single_rays[v:v + 1].data_ptr(), st.cuda_stream, seed=int(seeds[v]), **kw)
            e1.record(st)
        e1.synchronize()
        scene.move_camera(home)
        return e0.elapsed_time(e1)

    def batch():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            scene.render_views_device(cams, batch_rgb.data_ptr(), batch_rays.data_ptr(), seeds=seeds, stream_ptr=st.cuda_stream, **kw)
            e1.record(st)
        e1.synchronize()
        return e0.elapsed_time(e1)

    def check():
        if not torch.equal(single_rgb.reshape(-1), batch_rgb) or int(single_rays.sum().item()) != int(batch_rays.item()):
            raise SystemExit("images or ray counts of the two arms differ: %dx%dx%d K=%d" % (w, h, spp, k))

    single(), batch()                                                     # warm-up
    check()
    t_single, t_batch = [], []
    for _ in range(runs):
        t_single.append(single())
        t_batch.append(batch())
        check()
    rays = int(batch_rays.item())
    best_s, best_b = min(t_single), min(t_batch)
    return {"width": w, "height": h, "spp": spp, "views": k, "rays": rays,
            "single_ms": [round(t, 4) for t in t_single], "batch_ms": [round(t, 4) for t in t_batch],
            "single_mrays_s": round(rays / best_s / 1e3, 1), "batch_mrays_s": round(rays / best_b / 1e3, 1),
            "single_ms_per_view": round(best_s / k, 4), "batch_ms_per_view": round(best_b / k, 4),
            "speedup": round(best_s / best_b, 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--scenes", nargs="+", default=["large", "synth4096", "cloud1e5"])
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()
    import torch
    import rays1bench_b200 as r1
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark has no CPU path")
    info = gpu_info()
    scenes = make_scenes(r1)
    rows = []
    for name in args.scenes:
        scene, variant, target, dist = scenes[name]
        kernel = r1.lib.r1_kernel_name(scene.handle, variant).decode()
        for w, h, spp in SIZES:
            control = (w, h) == (1280, 720)
            if control and variant == r1.VARIANT_MEGAKERNEL_BVH:
                continue
            for k in (CONTROL_KS if control else KS):
                row = measure(r1, torch, scene, variant, orbit_cams(r1, scene, k, target, dist), w, h, spp, args.runs)
                row.update(scene=name, kernel=kernel)
                rows.append(row)
                print("%-9s %-15s %4dx%-4dx%-3d K=%-3d single %8.3f ms/view %9.1f Mrays/s | batch %8.3f ms/view %9.1f Mrays/s | x%.2f"
                      % (name, kernel, w, h, spp, k, row["single_ms_per_view"], row["single_mrays_s"], row["batch_ms_per_view"],
                         row["batch_mrays_s"], row["speedup"]), file=sys.stderr)
    info_after = gpu_info()
    result = {"gpu": info, "gpu_after": info_after, "runs": args.runs, "rows": rows}
    text = json.dumps(result)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
