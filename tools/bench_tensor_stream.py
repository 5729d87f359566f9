#!/usr/bin/env python
"""Measures the streamed tensor-core variant (R1_VARIANT_MEGAKERNEL_TENSOR_STREAM, r1::megakernel_tcs) against PACKED (the FFMA2
kernel) and TENSOR (tc3, where the scene fits its shared-memory operand) in one process on one GPU.

Per scene the variants run alternated, `--runs` times each, with L2 overwritten (256 MiB) before every render.  Every run
reports Mrays/s over the device time of the render (kernel_ms: CUDA events around trace kernel + resolve), trace_ms, whether
the image is byte-equal to PACKED's and the ray counts are equal, the algorithmic FP32 work (16 flops per ray-sphere test x real
spheres + 70 per ray, as bench.py) against the nominal FP32 FMA peak (SMs x 128 lanes x 2 x clocks.max.sm), and for the
streamed kernel the L2 -> SM bytes its operand ring moves.  The kernel does not count its fills; the figure is a LOWER BOUND
from the ray count: the ring refills one stage per chunk a CTA's groups scan together and a group's scan traces at most 128
rays, so fills >= rays / (128 x groups) x nchunks, and each fill moves the chunk's operand rows (128 B per sphere) and exact
records (16 B per sphere): l2_to_sm_bytes_min = rays / (128 x groups) x (n32 x 128 + n_pad x 16).  Scans with idle lanes
(the end of a render, paths that ended) make the true count higher.  The card's name, power limit and SM clocks come from
`nvidia-smi --query-gpu` (read-only) in the same call; the SM clock is sampled every 100 ms while the renders run.

    python tools/bench_tensor_stream.py [--runs 3] [--size 1280 720 250] [--out result.json]

There is no CPU path: without a CUDA device the script fails.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# grid scenes of tools/make_scene.py: (grid w, grid h) -> spheres after the loader's padding to 8
GRIDS = {"grid1000": (32, 31), "grid2000": (45, 44), "grid8000": (90, 89)}
# threads of the streamed kernel (128 per ray group): 0 = the default, 4 groups
TCS_CONFIGS = (0, 384, 256, 128)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True,
                         check=True).stdout.strip()
    name, power, sm, sm_max = [v.strip() for v in out.split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_clock_mhz": float(sm), "sm_clock_max_mhz": float(sm_max)}


class ClockSampler:
    """clocks.sm every 100 ms from a read-only nvidia-smi loop, for the duration of the measurement"""

    def __enter__(self):
        self.proc = subprocess.Popen(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-lms", "100"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        return self

    def __exit__(self, *exc):
        self.proc.terminate()
        out, _ = self.proc.communicate(timeout=10)
        self.samples = [float(v) for v in out.split() if v.replace(".", "", 1).isdigit()]
        return False


def make(r1, name, directory):
    if name not in GRIDS:
        return r1.create_scene(name)
    import make_scene
    gw, gh = GRIDS[name]
    scale = max(gw / 30.0, gh / 16.0)
    cam, sph = make_scene.grid_scene(gw, gh, 480, (3 * scale, 8 * scale, 15 * scale), 10.0 * scale)
    path = os.path.join(directory, name + ".r1scene")
    r1.write_scene_file(path, cam, sph)
    return r1.create_scene_from_file(path)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--size", type=int, nargs=3, default=(1280, 720, 250), metavar=("W", "H", "SPP"))
    ap.add_argument("--scenes", nargs="+", default=["synth4096", "large", "grid1000", "grid2000", "grid8000"])
    ap.add_argument("--config-scene", default="synth4096", help="scene on which every streamed configuration runs (the others run the default)")
    ap.add_argument("--out", help="also write the JSON result here")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement has no CPU path")
    import rays1bench_b200 as r1
    if r1.device_count() < 1:
        raise SystemExit("no CUDA device visible to the library")
    W, H, SPP = args.size
    r1.configure(width=W, height=H, spp=SPP, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    props = torch.cuda.get_device_properties(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    info_before = gpu_info()
    peak = props.multi_processor_count * 128 * 2 * info_before["sm_clock_max_mhz"] * 1e6
    result = {"gpu": info_before, "size": [W, H, SPP], "runs": args.runs, "fp32_peak_tflops_nominal": peak / 1e12, "scenes": {}}
    with tempfile.TemporaryDirectory() as tmp, ClockSampler() as clocks:
        for name in args.scenes:
            s = make(r1, name, tmp)
            soa = s.soa()
            n = s.count()
            n_real = int((soa["inv_radius"] > 0).sum())
            n32, n_pad = (n + 31) // 32 * 32, (n + 15) // 16 * 16
            runs = [("packed", r1.VARIANT_MEGAKERNEL_PACKED, 0)]
            if n32 <= 768:
                runs.append(("tensor", r1.VARIANT_MEGAKERNEL_TENSOR, 0))
            for threads in (TCS_CONFIGS if name == args.config_scene else TCS_CONFIGS[:1]):
                label = "tensor_stream" + ("" if not threads else "_g%d" % (threads // 128))
                runs.append((label, r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, threads))
            for label, v, threads in runs:                            # warm-up: module load, first launch of every kernel
                s.render(96, 54, 4, variant=v, threads=threads)
            entry = {"spheres": n, "real_spheres": n_real, "n32": n32, "kernels": {}, "runs": {label: [] for label, _, _ in runs}}
            for rep in range(args.runs):
                base = None
                for label, v, threads in runs:
                    flush.zero_()
                    torch.cuda.synchronize()
                    rgb, res = s.render(W, H, SPP, variant=v, threads=threads)
                    if base is None:
                        base = (rgb, res.num_rays)
                    flops = float(res.num_rays) * (16.0 * n_real + 70.0)
                    run = {"mrays_per_s": res.num_rays / (res.kernel_ms * 1e-3) / 1e6, "kernel_ms": res.kernel_ms, "trace_ms": res.trace_ms,
                           "num_rays": int(res.num_rays), "image_equal_to_packed": bool(np.array_equal(rgb, base[0])),
                           "rays_equal_to_packed": int(res.num_rays) == int(base[1]),
                           "fp32_roofline_frac": flops / (res.kernel_ms * 1e-3) / peak}
                    if v == r1.VARIANT_MEGAKERNEL_TENSOR_STREAM:
                        groups = threads // 128 if threads else 4
                        fills = res.num_rays / (128.0 * groups) * ((n32 + 127) // 128)
                        run["fills_min"] = fills
                        run["l2_to_sm_bytes_min"] = res.num_rays / (128.0 * groups) * (n32 * 128 + n_pad * 16)
                        run["l2_to_sm_gb_per_s_per_sm_min"] = run["l2_to_sm_bytes_min"] / (res.trace_ms * 1e-3) / props.multi_processor_count / 1e9
                    entry["runs"][label].append(run)
                    entry["kernels"][label] = r1.lib.r1_kernel_name(s.handle, v).decode()
            entry["median_mrays_per_s"] = {k: float(np.median([r["mrays_per_s"] for r in rs])) for k, rs in entry["runs"].items()}
            entry["all_images_equal"] = all(r["image_equal_to_packed"] and r["rays_equal_to_packed"] for rs in entry["runs"].values() for r in rs)
            result["scenes"][name] = entry
            s.close()
            print("%-10s %s  images equal: %s" % (name, "  ".join("%s %.0f" % kv for kv in entry["median_mrays_per_s"].items()), entry["all_images_equal"]),
                  file=sys.stderr, flush=True)
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
