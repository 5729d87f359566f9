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

With `--builders host device` the script compares the two trees of r1_scene_build_bvh instead of the variants.  Per scene: the
host build time (as above); the device build time, median over `--builds` builds after one warm-up, as CUDA events around the
device work and as host wall time of the call; node count, depth and SAH cost of each tree (from the exports; cost = 1 + sum over
child slots of area(slot box) / area(root box) x (1 for an inner node, the sphere count for a leaf)); and BVH Mrays/s with each
tree at `--builder-size`, alternated `--runs` times with L2 overwritten before every render, images and ray counts compared.

    python tools/bench_bvh.py [--runs 3] [--size 1280 720 250] [--out profiles/r03_bench_bvh.json]
    python tools/bench_bvh.py --builders host device [--builds 7] [--builder-size 640 360 32] [--out profiles/r04_bench_bvh_build.json]

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


def sah_cost(nodes):
    """1 + sum over used child slots of area / root area x (1 inner, count leaf); boxes as exported"""
    lo = np.stack([nodes["lo0"], nodes["lo1"]], 1).astype(np.float64)
    hi = np.stack([nodes["hi0"], nodes["hi1"]], 1).astype(np.float64)
    ch = nodes["child"]
    used = ch != -1
    e = hi - lo
    area = e[..., 0] * e[..., 1] + e[..., 1] * e[..., 2] + e[..., 2] * e[..., 0]
    if not used[0].any():
        return 0.0
    rl, rh = lo[0][used[0]].min(0), hi[0][used[0]].max(0)
    re = rh - rl
    root_area = re[0] * re[1] + re[1] * re[2] + re[2] * re[0]
    weight = np.where(ch >= 0, 1.0, (~ch) & 7)
    return float(1.0 + (area * weight)[used].sum() / root_area)


def tree_stats(nodes, leaves, depth):
    return {"nodes": len(nodes), "leaf_records": len(leaves), "depth": depth, "sah_cost": sah_cost(nodes)}


def compare_builders(r1, s, name, path, flush, torch, args):
    """host and device trees of one scene: build times, tree statistics, BVH render rates with each (alternated)"""
    entry = {"spheres": s.count(), "host": bvh_stats(r1, name, path)}
    host_nodes, host_leaves, host_depth = s.bvh()
    entry["host"].update(tree_stats(host_nodes, host_leaves, host_depth))
    entry["host"]["upload_ms"] = s.build_bvh(r1.BVH_BUILD_HOST)
    s.build_bvh(r1.BVH_BUILD_DEVICE)                                      # warm-up: module load, the sort's first launch
    dev_ms, wall_s = [], []
    for _ in range(args.builds):
        t0 = time.perf_counter()
        dev_ms.append(s.build_bvh(r1.BVH_BUILD_DEVICE))
        wall_s.append(time.perf_counter() - t0)
    dn, dl, dd = s.bvh_on_device()
    entry["device"] = dict(tree_stats(dn, dl, dd), build_ms=dev_ms, build_ms_median=float(np.median(dev_ms)), wall_s=wall_s,
                           wall_s_median=float(np.median(wall_s)))
    size = tuple(args.builder_size)
    entry["render_size"] = list(size)
    runs = {"host": [], "device": []}
    images = {}
    for builder in ("host", "device"):                                    # warm-up of each tree
        s.build_bvh(r1.BVH_BUILD_HOST if builder == "host" else r1.BVH_BUILD_DEVICE)
        render(r1, s, flush, torch, (96, 54, 4), r1.VARIANT_MEGAKERNEL_BVH, 0, None)
    for _ in range(args.runs):
        for builder in ("host", "device"):
            s.build_bvh(r1.BVH_BUILD_HOST if builder == "host" else r1.BVH_BUILD_DEVICE)
            rgb, res = render(r1, s, flush, torch, size, r1.VARIANT_MEGAKERNEL_BVH, 0, None)
            images.setdefault(builder, (rgb, int(res.num_rays)))
            runs[builder].append({"mrays_per_s": res.num_rays / (res.kernel_ms * 1e-3) / 1e6, "kernel_ms": res.kernel_ms,
                                  "num_rays": int(res.num_rays), "image_equal": bool(np.array_equal(rgb, images["host"][0])),
                                  "rays_equal": int(res.num_rays) == images["host"][1]})
    entry["runs"] = runs
    entry["median_mrays_per_s"] = {b: float(np.median([r["mrays_per_s"] for r in rs])) for b, rs in runs.items()}
    entry["all_images_equal"] = all(r["image_equal"] and r["rays_equal"] for rs in runs.values() for r in rs)
    return entry


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
    ap.add_argument("--builders", nargs="*", choices=("host", "device"), help="compare the host and device trees instead of the variants")
    ap.add_argument("--builds", type=int, default=7, help="timed device builds per scene (after one warm-up)")
    ap.add_argument("--builder-size", type=int, nargs=3, default=(640, 360, 32), metavar=("W", "H", "SPP"))
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()
    if args.builders is not None and sorted(args.builders) != ["device", "host"]:
        ap.error("--builders compares both trees: pass `--builders host device`")
    if args.builders and "--scenes" not in sys.argv:
        args.scenes = ["large", "synth4096", "grid8016", "grid1e5", "cloud1e5", "grid1e6", "cloud1e6"]

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
            if args.builders:
                entry = result["scenes"][name] = compare_builders(r1, s, name, path, flush, torch, args)
                s.close()
                print("%-10s %7d spheres: host build %.3f s, device build %.2f ms (wall %.2f ms); nodes %d / %d, depth %d / %d, SAH %.1f / %.1f; "
                      "Mrays/s host tree %.0f, device tree %.0f; images equal: %s" % (
                          name, entry["spheres"], entry["host"]["host_build_s"], entry["device"]["build_ms_median"], 1e3 * entry["device"]["wall_s_median"],
                          entry["host"]["nodes"], entry["device"]["nodes"], entry["host"]["depth"], entry["device"]["depth"], entry["host"]["sah_cost"],
                          entry["device"]["sah_cost"], entry["median_mrays_per_s"]["host"], entry["median_mrays_per_s"]["device"], entry["all_images_equal"]),
                      file=sys.stderr, flush=True)
                continue
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
