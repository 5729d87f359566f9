#!/usr/bin/env python
"""Measures the BVH variant (R1_VARIANT_MEGAKERNEL_BVH, r1::megakernel_pool<kScanBvh>) against the brute-force scans PACKED (the FFMA2
kernel), TENSOR_STREAM (r1::megakernel_tcs) and TENSOR (tc3, where the scene fits its shared-memory operand) in one process on one
GPU.

Per scene the variants run alternated, `--runs` times each, with L2 overwritten (256 MiB) before every render.  Every run reports
Mrays/s over the device time of the render (kernel_ms: CUDA events around trace kernel + resolve; the BVH's first-use upload
happens before them and is not in it), trace_ms, and whether the image is byte-equal to PACKED's with the same ray count.  Scenes
above `--full-limit` spheres compare the variants at `--mid-size` (above `--mid-limit`: `--small-size`), where the brute-force
scans finish in seconds, and time BVH alone at the full size as well.  Per scene
also: the host build time of the BVH (r1_bvh_export on a fresh copy of the scene), its node and leaf-record counts, bytes and
depth.  On `--config-scenes` every BVH thread count and two scheduling settings run too.  The card's name, power limit and SM
clocks come from `nvidia-smi --query-gpu` (read-only) in the same call; the SM clock is sampled every 100 ms while renders run.

    python tools/bench_bvh.py [--runs 3] [--size 1280 720 250] [--out profiles/r03_bench_bvh.json]

There is no CPU path: without a CUDA device the script fails.
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

# scenes of tools/make_scene.py: grid (w, h) or cloud n
GRIDS = {"grid8016": (90, 89), "grid1e5": (316, 316), "grid1e6": (1000, 1000)}
CLOUDS = {"cloud1e5": 100000, "cloud1e6": 1000000}
# (label, threads, R1_SCHED) of the BVH kernel on the config scenes; the first is the default
BVH_CONFIGS = (("bvh", 0, None), ("bvh_t512", 512, None), ("bvh_t768", 768, None), ("bvh_sched8", 0, "8,16"), ("bvh_sched1", 0, "1,1"))


def make(r1, name, directory):
    import make_scene
    if name in GRIDS:
        gw, gh = GRIDS[name]
        scale = max(gw / 30.0, gh / 16.0)
        cam, sph = make_scene.grid_scene(gw, gh, 480, (3 * scale, 8 * scale, 15 * scale), 10.0 * scale)
    elif name in CLOUDS:
        cam, sph = make_scene.cloud_scene(CLOUDS[name])
    else:
        return r1.create_scene(name), None
    path = os.path.join(directory, name + ".r1scene")
    r1.write_scene_file(path, cam, sph)
    return r1.create_scene_from_file(path), path


def bvh_stats(r1, name, path):
    """host build time of a fresh copy of the scene (commit=False: no device), and the tree's size"""
    s = r1.create_scene(name, commit=False) if path is None else r1.create_scene_from_file(path, commit=False)
    t0 = time.perf_counter()
    nodes, leaves, depth = s.bvh()
    dt = time.perf_counter() - t0
    s.close()
    return {"host_build_s": dt, "nodes": len(nodes), "leaf_records": len(leaves), "bytes": int(nodes.nbytes + leaves.nbytes), "depth": depth}


def render(r1, s, flush, torch, size, v, threads, sched):
    if sched:
        os.environ["R1_SCHED"] = sched
    flush.zero_()
    torch.cuda.synchronize()
    try:
        return s.render(*size, variant=v, threads=threads)
    finally:
        os.environ.pop("R1_SCHED", None)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--size", type=int, nargs=3, default=(1280, 720, 250), metavar=("W", "H", "SPP"))
    ap.add_argument("--full-limit", type=int, default=20000, help="scenes with more spheres compare at --mid-size")
    ap.add_argument("--mid-size", type=int, nargs=3, default=(640, 360, 32), metavar=("W", "H", "SPP"))
    ap.add_argument("--mid-limit", type=int, default=200000, help="scenes with more spheres compare at --small-size")
    ap.add_argument("--small-size", type=int, nargs=3, default=(320, 180, 8), metavar=("W", "H", "SPP"))
    ap.add_argument("--scenes", nargs="+", default=["small", "medium", "large", "synth4096", "grid8016", "grid1e5", "cloud1e5", "grid1e6", "cloud1e6"])
    ap.add_argument("--config-scenes", nargs="*", default=["large", "cloud1e5"])
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement has no CPU path")
    import rays1bench_b200 as r1
    if r1.device_count() < 1:
        raise SystemExit("no CUDA device visible to the library")
    full = tuple(args.size)
    r1.configure(width=full[0], height=full[1], spp=full[2], max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    result = {"gpu": gpu_info(), "size": list(full), "runs": args.runs, "scenes": {}}
    with tempfile.TemporaryDirectory() as tmp, ClockSampler() as clocks:
        for name in args.scenes:
            s, path = make(r1, name, tmp)
            n = s.count()
            n32 = (n + 31) // 32 * 32
            entry = {"spheres": n, "real_spheres": int((s.soa()["inv_radius"] > 0).sum()), "bvh": bvh_stats(r1, name, path)}
            size = full if n <= args.full_limit else tuple(args.mid_size) if n <= args.mid_limit else tuple(args.small_size)
            entry["compare_size"] = list(size)
            runs = [("packed", r1.VARIANT_MEGAKERNEL_PACKED, 0, None), ("tensor_stream", r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, 0, None)]
            if n32 <= 768:
                runs.append(("tensor", r1.VARIANT_MEGAKERNEL_TENSOR, 0, None))
            for label, threads, sched in (BVH_CONFIGS if name in args.config_scenes else BVH_CONFIGS[:1]):
                runs.append((label, r1.VARIANT_MEGAKERNEL_BVH, threads, sched))
            t0 = time.perf_counter()
            s.render(96, 54, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)        # first use: host build + upload (elapsed_seconds includes it)
            entry["bvh_first_render_s"] = time.perf_counter() - t0
            for label, v, threads, sched in runs:                         # warm-up: module load, first launch of every kernel
                render(r1, s, flush, torch, (96, 54, 4), v, threads, sched)
            entry["runs"] = {label: [] for label, _, _, _ in runs}
            kernels = {}
            for rep in range(args.runs):
                base = None
                for label, v, threads, sched in runs:
                    rgb, res = render(r1, s, flush, torch, size, v, threads, sched)
                    if base is None:
                        base = (rgb, res.num_rays)
                    entry["runs"][label].append({"mrays_per_s": res.num_rays / (res.kernel_ms * 1e-3) / 1e6, "kernel_ms": res.kernel_ms,
                                                 "trace_ms": res.trace_ms, "num_rays": int(res.num_rays),
                                                 "image_equal_to_packed": bool(np.array_equal(rgb, base[0])),
                                                 "rays_equal_to_packed": int(res.num_rays) == int(base[1])})
                    kernels[label] = r1.lib.r1_kernel_name(s.handle, v).decode()
            entry["kernels"] = kernels
            entry["median_mrays_per_s"] = {k: float(np.median([r["mrays_per_s"] for r in rs])) for k, rs in entry["runs"].items()}
            entry["all_images_equal"] = all(r["image_equal_to_packed"] and r["rays_equal_to_packed"] for rs in entry["runs"].values() for r in rs)
            if size != full:                                              # BVH alone at the full size
                fr = [render(r1, s, flush, torch, full, r1.VARIANT_MEGAKERNEL_BVH, 0, None)[1] for _ in range(args.runs)]
                entry["bvh_full_size"] = {"mrays_per_s": [r.num_rays / (r.kernel_ms * 1e-3) / 1e6 for r in fr], "kernel_ms": [r.kernel_ms for r in fr],
                                          "num_rays": [int(r.num_rays) for r in fr]}
                entry["bvh_full_size"]["median_mrays_per_s"] = float(np.median(entry["bvh_full_size"]["mrays_per_s"]))
            result["scenes"][name] = entry
            s.close()
            print("%-10s %7d spheres at %s: %s  images equal: %s%s" % (
                name, n, "x".join(map(str, size)), "  ".join("%s %.0f" % kv for kv in entry["median_mrays_per_s"].items()), entry["all_images_equal"],
                "  bvh full size %.0f" % entry["bvh_full_size"]["median_mrays_per_s"] if "bvh_full_size" in entry else ""), file=sys.stderr, flush=True)
    result["sm_clock_mhz_during"] = {"min": min(clocks.samples), "median": float(np.median(clocks.samples)), "max": max(clocks.samples),
                                     "samples": len(clocks.samples)} if clocks.samples else None
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)
    if not all(e["all_images_equal"] for e in result["scenes"].values()):
        raise SystemExit("an image or a ray count differs from PACKED")


if __name__ == "__main__":
    main()
