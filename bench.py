#!/usr/bin/env python
"""bench.py -- Mrays/s of the Rays1 trace loop on N B200s (BASELINE.json: "Mrays/s (large scene) at 1/2/4/8 B200;
% of FP32 FMA peak; vs host CPU").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload large|medium|small|large4k|synth4096]
                  [--variant mega|wavefront|scalar] [--impl reference] [--dump-outputs DIR]
  N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one full render of the workload (every pixel x sample through generate -> scan -> shade -> resolve, and for
N > 1 the framebuffer gather + ray-counter reduce).  `value` times the steps on the device (CUDA events on the launching
stream, inputs resident in HBM, max over ranks); `e2e` times the reference-facing call -- create_large_scene() +
benchmark(scene, pixels, ...) -- with HOST buffers (scene upload and framebuffer download inside).  `roofline` is the
FP32-FMA roofline of the trace kernel (this path is compute-bound: <= 128 KB of sphere data lives in shared memory);
`cpu_baseline` is the reference's own src/latest code (oracle/_ref, its TileRenderScheduler on all host threads) on a
bounded sample.  One JSON line on stdout, printed by rank 0.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark writes nothing into the tree it runs from (which may be read-only): no bytecode caches for the modules it
# imports beyond what build() imported (rays1bench_b200/dist.py, tests/cpu_checkers.py)
sys.dont_write_bytecode = True

WORKLOADS = {
    # name: (scene, width, height, spp, max_bounces)  -- BASELINE.json configs
    "small": ("small", 1280, 720, 250, 50),        # config 1
    "medium": ("medium", 1280, 720, 250, 50),      # config 2
    "large": ("large", 1280, 720, 250, 50),        # config 3 (the metric's configuration)
    "large4k": ("large", 3840, 2160, 1024, 50),    # config 4
    "synth4096": ("synth4096", 1280, 720, 250, 50) # config 5
}
METRIC = "Mrays/s (large scene)"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the `ncu --set full` captures
# summarised under profiles/; keyed "<workload>/<variant>" in profiles/ncu_traffic.json (null where nothing was captured)
def ncu_traffic(workload, variant):
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        return None, None
    e = table.get("%s/%s" % (workload, variant))
    return (e["dram_bytes_per_launch"], e.get("source")) if e else (None, None)


NOMINAL_SM_MHZ = 1965.0
# BASELINE.md section 1: the reference's own published figure for this metric and configuration (step13, large scene,
# 1280x720, 250 spp) -- 59.362 Mrays/s on an i9-9900K 8c/16t, README.md:52 of the reference.  CPU hardware, quoted as published.
PUBLISHED_MRAYS = {"large": 59.362, "medium": 215.403, "small": 321.238}


def metric_name(workload):
    """BASELINE.json's metric is quoted on the large scene; other workloads say which scene they measured."""
    scene = WORKLOADS[workload][0]
    return METRIC if scene == "large" else "Mrays/s (%s scene)" % scene


def workload_label(name):
    scene, w, h, spp, mb = WORKLOADS[name]
    return "%s scene %dx%d %d spp depth %d" % (scene, w, h, spp, mb)


DUMP_BUDGET = 64_000_000   # bytes --dump-outputs may write in all
NPY_HEADER = 128           # bytes numpy writes in front of each of the (at most three) arrays below


def dump_outputs(out_dir, image, num_rays):
    """--dump-outputs: what the timed path handed its caller in its last step, so that two builds can be compared output for
    output.  image.npy = the RGB8 framebuffer [H, W, 3] (row 0 = bottom) as float32, num_rays.npy = the ray count as float64.
    An image that does not fit the budget (the 3840x2160 workload) is replaced by a fixed, seeded sample of its pixels [n, 3]
    that fills it; their flat indices y * W + x go to image_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    rays = np.array([num_rays], np.float64)
    img = image.astype(np.float32)
    room = DUMP_BUDGET - 3 * NPY_HEADER - rays.nbytes       # for image.npy and, when sampled, image_index.npy
    if img.nbytes > room:
        h, w = img.shape[:2]
        n = room // (3 * 4 + 8)                              # per kept pixel: three float32 values + one float64 index
        idx = np.sort(np.random.default_rng(0).choice(h * w, n, replace=False))
        np.save(os.path.join(out_dir, "image_index.npy"), idx.astype(np.float64))
        img = img.reshape(-1, 3)[idx]
    np.save(os.path.join(out_dir, "image.npy"), img)
    np.save(os.path.join(out_dir, "num_rays.npy"), rays)


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        self.mark = 0

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        t1 = time.time()
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        rows = [r for t, r in self.rows if self.t0 <= t <= t1 + 0.2 and len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in rows)
        reasons = set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in rows:
            for k, nm in enumerate(names):
                if r[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": sorted(reasons), "samples": len(rows),
                "power_w_max": max(float(r[2]) for r in rows)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def reference_step(ref, scene, w, h, spp):
    _, rays, el = ref.render(scene, w, h, spp)  # the reference's own TileRenderScheduler on hardware_concurrency() threads
    return rays, el


_NATIVE = None


def native_build_usable():
    global _NATIVE
    if _NATIVE is None:
        _NATIVE = _native_build_usable()
    return _NATIVE


def _native_build_usable():
    """oracle/_ref/*_native* were built with the reference's exact line (bench.py:175: -flto -march=native) on the build
    container's CPU; they may only run on a host that has every instruction-set flag that CPU had."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    try:
        need = set(open(os.path.join(ref_dir, "native_cpu_flags.txt")).read().split())
        have = set()
        for line in open("/proc/cpuinfo"):
            if line.startswith("flags"):
                have = set(line.split(":", 1)[1].split())
                break
        isa = {f for f in need if f.startswith(("avx", "sse", "ssse", "fma", "bmi", "adx", "aes", "pclmul", "sha", "vaes", "vpclmul", "gfni", "amx",
                                                "movdir", "cldemote", "clwb", "clflushopt", "rdseed", "rdrand", "xsave", "fsgsbase", "f16c", "popcnt",
                                                "lzcnt", "abm", "movbe", "serialize", "waitpkg", "pku", "rdpid", "enqcmd", "uintr", "ptwrite", "tsxldtrk"))}
        march = open(os.path.join(ref_dir, "native_march.txt")).read().strip()
        ok = isa <= have and os.path.exists(os.path.join(ref_dir, "libref_rays1_native.so"))
        if ok:  # belt and braces: an illegal instruction must kill a throw-away process, not this one
            probe = ("import sys; sys.path.insert(0, %r); from cpu_checkers import RefLib; r = RefLib(native=True); "
                     "s = r.scene_create('small'); r.render(s, 64, 36, 1)" % os.path.join(ROOT, "tests"))
            ok = subprocess.run([sys.executable, "-c", probe], capture_output=True, timeout=120).returncode == 0
        return ok, march
    except (OSError, subprocess.SubprocessError):
        return False, None


def reference_executable(budget_runs=3):
    """BASELINE.md section 3: the UNMODIFIED reference executable, `-n 3`, at its compiled-in workload (1280x720x250, small +
    medium + large), threads = hardware_concurrency(); mean (what log_results writes, common.h:47-60) and best per scene."""
    import re
    import tempfile
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    usable, march = native_build_usable()
    exe = os.path.join(ref_dir, "rays1_latest_native") if usable and os.path.exists(os.path.join(ref_dir, "rays1_latest_native")) else \
        os.path.join(ref_dir, "rays1_latest")
    if not os.path.exists(exe):
        return None
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.time()
        txt = subprocess.run([exe, "-n", str(budget_runs)], cwd=tmp, capture_output=True, text=True, timeout=900).stdout
        wall = time.time() - t0
    out, cur, threads = {}, None, None
    for line in txt.splitlines():
        if line.strip() in ("small", "medium", "large"):
            cur = line.strip()
        m = re.match(r"mrays/s:\s+([0-9.]+)", line)
        if m and cur:
            out.setdefault(cur, []).append(float(m.group(1)))
        m = re.match(r"threads:\s+(\S+)", line)
        if m:
            threads = m.group(1)
    return {"exe": os.path.basename(exe), "runs": budget_runs, "threads": threads, "wall_s": wall,
            "build": "g++ 13.3 -pthread -ffast-math -O3 -g -fno-rtti -fno-exceptions -std=c++17 -flto -march=%s -m64 -DNDEBUG (bench.py:175 of the reference%s), "
                     "built in the build container" % ((march, ", native = the container's CPU") if exe.endswith("_native") else ("x86-64-v3", "; no -flto")),
            "mrays_per_s": {k: {"mean": sum(v) / len(v), "best": max(v)} for k, v in out.items()}}


def cpu_reference(workload, budget_s, steps, warmup):
    """Times the reference's CPU implementation on a bounded sample of the workload: oracle/_ref = the unmodified src/latest
    compiled in place (the MAX_SPHERES = 4096 build of the same sources for the 4096-sphere scene, which the reference cannot
    hold otherwise), its own TileRenderScheduler on hardware_concurrency() threads.  The oracle port only where no reference
    build is present.  Returns per-step results."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cpu_checkers import Oracle, RefLib
    scene_name, w, h, spp, mb = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    build = None
    if RefLib.available(4096 if scene_name == "synth4096" else 1024) and w * 9 == h * 16:
        usable, march = native_build_usable()
        if scene_name == "synth4096":
            ref = RefLib(4096)
            build = "-ffast-math -O3 -march=x86-64-v3, MAX_SPHERES = 4096 (rayweek1.cpp:174 patched in a temporary copy), built in the build container"
        elif usable:
            ref = RefLib(native=True)
            build = "bench.py:175 of the reference verbatim: -ffast-math -O3 -flto -march=native (= %s, the build container's CPU)" % march
        else:
            ref = RefLib()
            build = "-ffast-math -O3 -march=x86-64-v3 (this host lacks ISA flags of the native build), built in the build container"
        kind, scene = "reference", ref.scene_create(scene_name)
        cores = ref.hardware_concurrency()
        run = lambda s: reference_step(ref, scene, w, h, s)  # noqa: E731
    else:
        orc = Oracle()
        kind, scene = "port", orc.scene_create(scene_name, w, h)
        build = "oracle/rays1_oracle.c (plain C restatement), -O2"
        def run(s):  # noqa: E306
            _, rays, el = orc.render(scene, w, h, s, mb, threads=cores)
            return rays, el
    rays, el = run(1)  # calibration: one sample per pixel
    sample_spp = int(max(1, min(spp, budget_s / max(el, 1e-3))))
    results = [run(sample_spp) for _ in range(warmup + steps)][warmup:]
    tot_rays, tot_s = sum(r for r, _ in results), sum(e for _, e in results)
    return dict(kind=kind, cores=cores, build=build, threads="%d/%d" % (cores, os.cpu_count() or cores),
                sample="%s scene %dx%d at %d spp (%d of %d spp; Mrays/s does not depend on spp)" %
                (scene_name, w, h, sample_spp, sample_spp, spp), value=tot_rays / tot_s / 1e6, ms_per_step=1e3 * tot_s / len(results),
                rays_per_sample=tot_rays / (len(results) * w * h * sample_spp))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="large", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="mega", choices=["mega", "wavefront", "scalar", "coop", "deferred", "dual", "tensor", "packed"])
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work per reference step / baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-exe", action="store_true", help="skip the `rays1_latest -n 3` run of the unmodified reference executable")
    ap.add_argument("--threads", type=int, default=0, help="threads per persistent CTA (512/768/1024; 0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's image and ray count to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 path computed (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != max(args.gpus, 1) and world > 1:
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))
    scene_name, W, H, SPP, MB = WORKLOADS[args.workload]
    config = {"workload": workload_label(args.workload), "scene": scene_name, "width": W, "height": H, "spp": SPP, "max_bounces": MB,
              "partition": "interleaved row tiles of 1 row, row k -> rank k %% %d" % world, "variant": args.variant,
              "scheduling": "lane fetch (R1_POOL=0)" if os.environ.get("R1_POOL") == "0" else "warp sample pool",
              "l2": "flushed between timed steps (256 MiB write); the kernel's inputs (<= 128 KB of spheres) are staged to shared memory"}

    # -------------------------------------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = args.steps, max(args.warmup, 1)
        # bounded sample per step, and the whole run (warm-up + steps) within about 2.5 minutes of CPU time
        r = cpu_reference(args.workload, min(args.cpu_budget, 150.0 / (steps + warmup)), steps, warmup)
        line = {"impl": "reference", "metric": metric_name(args.workload), "value": r["value"], "unit": "Mrays/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": r["value"] / PUBLISHED_MRAYS[args.workload] if args.workload in PUBLISHED_MRAYS else None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "Mrays/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                                 "build": r["build"], "threads": r["threads"]},
                "e2e": {"value": r["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "rays_per_sample": r["rays_per_sample"]}
        print(json.dumps(line))
        return

    # -------------------------------------------------------------------------------------------- B200 arm
    # NCCL's INFO log (communicator ranks, transports, NVLS) stays ON: it is the evidence that N ranks really formed one
    # communicator.  The image presets NCCL_DEBUG=VERSION (banner only), so anything quieter than INFO is raised to INFO; the log
    # goes where NCCL sends it by default (stdout, like the version banner) -- the JSON line is still one line of its own,
    # printed after every rank has gone quiet at a barrier.  R1_NCCL_DEBUG overrides.
    if os.environ.get("R1_NCCL_DEBUG"):
        os.environ["NCCL_DEBUG"] = os.environ["R1_NCCL_DEBUG"]
    elif os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = "INFO"
    import torch
    import torch.distributed as dist

    import rays1bench_b200 as r1
    from rays1bench_b200 import dist as r1d

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU implementation (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")  # host-side rendezvous for the in-process leg (no kernel spinning on the GPUs)
    variant = r1.VARIANTS[args.variant]
    row_tile = r1.DEFAULT_ROW_TILE
    r1.configure(width=W, height=H, spp=SPP, max_bounces=MB, variant=variant, n_gpus=1, seed=0, quiet=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # resident inputs + output buffers (value arm): scene committed once, torch owns the output tensors
    # the host builders commit to devices 0..n-1 of ONE process; under torchrun each rank commits to its own GPU
    scene = r1.create_scene(scene_name, commit=False)
    r1._check(r1.lib.r1_scene_commit(scene.handle, local_rank), "r1_scene_commit")
    n_real = r1.REAL_SPHERES[scene_name]
    n_pad = (scene.count() + 15) // 16 * 16
    n32 = (scene.count() + 31) // 32 * 32
    kernel = "r1::" + r1.lib.r1_kernel_name(scene.handle, variant).decode()   # what the variant resolves to for this scene
    if args.threads and args.variant == "mega":
        kernel = "r1::megakernel_pool"                                          # explicit tuning knobs address the packed kernel
    traffic_key = "tensor" if "megakernel_tc" in kernel else ("mega" if args.variant == "packed" else args.variant)

    my_rows = r1.local_rows(H, row_tile, rank, world)
    max_rows = r1d.max_local_rows(H, row_tile, world)
    d_rgb = torch.zeros((max_rows, W, 3), dtype=torch.uint8, device=dev)
    d_rays = torch.zeros(1, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    kw = dict(width=W, height=H, spp=SPP, max_bounces=MB, variant=variant, seed=0, rank=rank, world=world, row_tile=row_tile, device=local_rank, threads=args.threads)

    def step():
        """one pass of the hot path; returns (#kernels of ours launched, final image tensor on rank 0)"""
        res = scene.render_device(d_rgb.data_ptr(), d_rays.data_ptr(), stream.cuda_stream, **kw)
        launches = res.launches
        img = d_rgb
        if world > 1:
            gathered = r1d.gather_framebuffer(d_rgb, H, row_tile, rank, world)
            r1d.reduce_ray_count(d_rays, world)
            if rank == 0:
                img = r1d.deinterleave(gathered, W, H, row_tile, world)
                launches += 1
        return launches, img

    total_ms, trace_ms, total_rays, launches = 0.0, 0.0, 0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = None
    for it in range(args.warmup + args.steps):
        timed = it >= args.warmup
        if it == args.warmup:
            sampler = ClockSampler(local_rank) if rank == 0 else None
            if sampler:
                sampler.begin()
        flush.zero_()  # L2 flush between iterations (outside the timed events)
        barrier()
        e0.record(stream)
        n_l, img = step()
        e1.record(stream)
        barrier()
        if timed:
            total_ms += e0.elapsed_time(e1)
            waited = scene.render_wait(local_rank)
            trace_ms += waited.trace_ms
            n_l = waited.launches + (1 if (world > 1 and rank == 0) else 0)  # trace kernel(s) + resolve (+ de-interleave); the
            #                                                                 wavefront's loop iterations are counted on the device
            total_rays += int(d_rays.item()) if rank == 0 else 0  # for N > 1 the reduced total lives on rank 0
            launches += n_l
    clocks = sampler.end() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, img[:H].cpu().numpy(), int(d_rays.item()))
    ms_value = allmax(total_ms)        # max over ranks of the summed per-step device times
    ms_trace = allmax(trace_ms)

    # ---- e2e: the reference-facing call with HOST buffers, every step = scene upload + render + download
    pixels_t = torch.zeros((H, W, 3), dtype=torch.uint8).pin_memory()
    pixels = pixels_t.numpy()
    h2d = n_pad * (32 + 32)   # scan + exact + 32-byte shading record per sphere
    d2h = W * H * 3 + 8
    e2e_s, e2e_rays = 0.0, 0
    for it in range(args.warmup + args.steps):
        barrier()
        t0 = time.perf_counter()
        if world == 1:
            sc = r1.create_scene(scene_name)                   # builders emit the device buffers (H2D)
            res = r1.benchmark(sc, pixels, False, scene_name)  # render + D2H into the caller's pixels; consumes the scene
            rays_step = res.num_rays
        else:
            sc = r1.create_scene(scene_name, commit=False)
            r1._check(r1.lib.r1_scene_commit(sc.handle, local_rank), "r1_scene_commit")  # H2D on this rank's GPU
            sc.render_device(d_rgb.data_ptr(), d_rays.data_ptr(), stream.cuda_stream, **kw)
            gathered = r1d.gather_framebuffer(d_rgb, H, row_tile, rank, world)
            r1d.reduce_ray_count(d_rays, world)
            rays_step = 0
            if rank == 0:
                img = r1d.deinterleave(gathered, W, H, row_tile, world)
                pixels_t.copy_(img, non_blocking=True)         # D2H of the RGB8 image into pinned host memory
                rays_step = int(d_rays.cpu().item())
            torch.cuda.synchronize()
            sc.close()
        dt = time.perf_counter() - t0
        dt = allmax(dt)
        if it >= args.warmup:
            e2e_s += dt
            e2e_rays += rays_step

    # ---- e2e_inprocess (N > 1): the DROP-IN surface at N GPUs -- ONE process, configure(n_gpus=N) + create_<scene>_scene() +
    # benchmark(scene, pixels, ...), i.e. rays1_host.cpp's MultiGpu path (ncclCommInitAll, grouped send/recv, ncclReduce) that
    # replaces TileRenderScheduler::run.  Rank 0 drives all N devices while the other ranks wait on the HOST (gloo), their GPUs idle.
    inproc = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
        if rank == 0:
            torchrun_img = pixels.copy()
            torchrun_rays = e2e_rays // max(args.steps, 1)
            try:
                r1.configure(width=W, height=H, spp=SPP, max_bounces=MB, variant=variant, n_gpus=world, seed=0, quiet=True)
                ip_s, ip_rays, ip_kms = 0.0, 0, 0.0
                for it in range(args.warmup + args.steps):
                    t0 = time.perf_counter()
                    sc = r1.create_scene(scene_name)                    # replicas on devices 0..N-1 (H2D)
                    res = r1.benchmark(sc, pixels, False, scene_name)   # trace on N devices, gather, reduce, D2H
                    dt = time.perf_counter() - t0
                    if it >= args.warmup:
                        ip_s += dt; ip_rays += res.num_rays; ip_kms += res.kernel_ms
                inproc = {"value": ip_rays / ip_s / 1e6, "unit": "Mrays/s", "ms_per_step": 1e3 * ip_s / args.steps,
                          "kernel_ms_per_step": ip_kms / args.steps, "api": "one process: configure(n_gpus=%d) + create_%s_scene() + benchmark()" % (world, scene_name),
                          "image_equal_to_torchrun_path": bool(np.array_equal(pixels, torchrun_img)), "rays_equal": int(ip_rays // args.steps) == int(torchrun_rays)}
            except r1.Rays1Error as e:
                inproc = {"error": str(e)}
            finally:
                r1.configure(n_gpus=1)
        dist.barrier(group=cpu_group)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (FP32 FMA pipe)
    f_ray = r1.flops_per_ray(n_real)
    peak_scalar, mhz_est = r1.fma_peak(local_rank, packed=False)
    peak_packed, _ = r1.fma_peak(local_rank, packed=True)
    peak_meas = max(peak_scalar, peak_packed)
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    peak_nominal = sm_count * 128 * 2 * NOMINAL_SM_MHZ * 1e6 / 1e12
    achieved = total_rays * f_ray / (ms_trace * 1e-3) / 1e12 / world  # per GPU
    hbm_bytes = W * H * (32 * 2 + 3) + n_pad * 32 * sm_count   # fixed-point accumulators zeroed + written back, RGB8 out, staging
    roofline = {"bound": "fp32_fma", "kernel": kernel, "achieved": achieved,
                "peak": peak_meas, "unit": "TFLOP/s", "frac": achieved / peak_meas,
                "peak_source": "FFMA/FFMA2 chain microbenchmark on this GPU (r1_fma_peak), per GPU; scalar %.1f / packed %.1f TFLOP/s (SM clock during the run: see clocks)" %
                               (peak_scalar, peak_packed),
                "peak_nominal": peak_nominal, "frac_nominal": achieved / peak_nominal,
                "flops_per_ray": f_ray, "flops_model": "16 per ray-sphere test (FMA=2) x %d real spheres + 70 shading (SURVEY.md 8d)" % n_real,
                "traffic": ncu_traffic(args.workload, traffic_key)[0] if world == 1 else None,
                "traffic_source": ncu_traffic(args.workload, traffic_key)[1] if world == 1 else None,
                "traffic_note": "DRAM bytes per launch of the dominant kernel (ncu --set full, profiles/ncu_traffic.json); algorithmic FLOPs are "
                                "the REFERENCE's 16 per test, the filter executes 8 FMA-pipe instructions per test plus an exact re-test of "
                                "the 0.4 % candidates",
                "hbm": {"algorithmic_bytes_per_step": hbm_bytes, "achieved_gbs": hbm_bytes * args.steps / (ms_trace * 1e-3) / 1e9,
                        "note": "pixel accumulators (32 B, L2 atomics) + RGB8 out + sphere staging per CTA: HBM is idle on this path"}}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        roofline["hbm"]["peak_gbs"] = peaks.get("hbm_gbs")
    except (OSError, ValueError):
        pass
    if "megakernel_tc" in kernel:
        # The filter of this kernel runs on the tensor cores: 128 rays x n32 spheres x K = 32 split-TF32 MACs per scan, one 4-byte
        # filter value per test read back from TMEM.  The FP32 roofline above keeps the ALGORITHMIC flops (the reference's 16 per
        # test) against the FP32 FMA peak -- a fraction above 1 says the work left the FP32 pipe; the two hardware bounds of the
        # filter as built are below.
        tests = total_rays * n32 / world                                      # per GPU, padded columns included
        tf32_exec = tests * 2 * 32 / (ms_trace * 1e-3) / 1e12
        bf16_peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
        tf32_peak = (bf16_peak / 2.0) if bf16_peak else 1125.0
        tmem_peak = r1.tmem_read_peak(local_rank, 16) * sm_count               # bytes/s, measured live (16 warps per SM)
        tmem_bps = tests * 4 / (ms_trace * 1e-3)
        roofline["note"] = ("frac > 1 is not an error: the filter (8 of the reference's 10 FMA-pipe instructions per test) runs as a split-TF32 "
                            "GEMM on the tensor cores; see `tensor` and `tmem_read` for the hardware bounds of this kernel")
        roofline["limiter"] = ("latency: no unit saturated (ncu of the large scene: issue slots 61 %, ALU pipe 59 %, tensor pipe 50 %, TMEM reads "
                               "31 %; 26 % of the stall samples wait for an accumulator chunk) -- profiles/r02_ncu_megakernel_tc3.md")
        roofline["tensor"] = {"executed": tf32_exec, "peak": tf32_peak, "unit": "TFLOP/s", "frac": tf32_exec / tf32_peak,
                              "peak_source": "MEASURED_PEAKS.json sustained dense bf16 / 2" if bf16_peak else "nominal dense TF32 (half of 2.25 PFLOP/s bf16)",
                              "flops_model": "2 x K = 32 (11 lifted features x {hi hi, lo hi, hi lo}) per ray-sphere test, %d columns per ray" % n32}
        roofline["tmem_read"] = {"achieved": tmem_bps / 1e12, "peak": tmem_peak / 1e12, "unit": "TB/s", "frac": tmem_bps / tmem_peak,
                                 "peak_source": "tcgen05.ld 32x32b.x32 microbenchmark on this GPU (r1_tmem_read_peak, 16 warps per SM)",
                                 "bytes_model": "4 bytes per ray-sphere test (one FP32 accumulator column)"}

    line = {"metric": metric_name(args.workload), "value": total_rays / (ms_value * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": (total_rays / (ms_value * 1e-3) / 1e6) / PUBLISHED_MRAYS[args.workload] if args.workload in PUBLISHED_MRAYS else None,
            "baseline_note": "published by the reference for this scene at 1280x720x250 on an i9-9900K (BASELINE.md section 1); no GPU number is published",
            "dtype": "f32", "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": e2e_rays / e2e_s / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / args.steps,
                    "api": "create_%s_scene() + benchmark(scene, pixels, write_tga=False, name)" % scene_name if world == 1 else
                           "per rank: scene commit + r1_render_device; NCCL gather + reduce; rank 0 de-interleave + D2H"},
            "gpu_launches": launches, "roofline": roofline,
            "kernel_only": {"trace_ms_per_step": ms_trace / args.steps, "mrays_per_s": total_rays / (ms_trace * 1e-3) / 1e6},
            "rays_per_step": total_rays // args.steps, "rays_per_sample": total_rays / (args.steps * W * H * SPP)}
    if inproc is not None:
        line["e2e_inprocess"] = inproc
    if world > 1:
        line["nccl"] = {"nranks": world, "debug": os.environ.get("NCCL_DEBUG"), "debug_file": os.environ.get("NCCL_DEBUG_FILE")}
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(args.workload, args.cpu_budget, 1, 0)
        line["cpu_baseline"] = {"value": r["value"], "unit": "Mrays/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                                "build": r["build"], "threads": r["threads"]}
        if scene_name in ("small", "medium", "large") and (W, H, SPP) == (1280, 720, 250) and not args.no_reference_exe:
            exe = reference_executable(3)   # BASELINE.md section 3: the unmodified executable, -n 3, mean and best
            if exe:
                line["cpu_baseline"]["executable_n3"] = exe
    sys.stdout.flush()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
