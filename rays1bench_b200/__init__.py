"""rays1bench_b200 -- B200-native trace loop of the Rays1 benchmark behind the reference's own surface.

This module is the thin Python view of ``librays1_b200.so`` (C ABI: ``include/rays1_b200.h``).  It mirrors the
reference's host interface for the path -- ``create_small_scene() / create_medium_scene() / create_large_scene()`` and
``benchmark(scene, pixels, write_tga, scene_name)`` (``src/latest/rayweek1.cpp:552, 582, 654, 845`` of the reference)
-- plus the device-facing entry points the parity tests call.  All compute runs in the CUDA library: there is no
Python or CPU implementation of the path here, and importing fails loudly when the library has not been built.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("R1_LIBRARY") or os.path.join(_HERE, "librays1_b200.so")   # R1_LIBRARY: an alternative build, for A/B runs
EXE_PATH = os.path.join(_HERE, "rays1_b200")

VARIANT_MEGAKERNEL, VARIANT_WAVEFRONT, VARIANT_MEGAKERNEL_SCALAR, VARIANT_MEGAKERNEL_COOP, VARIANT_MEGAKERNEL_DEFERRED, VARIANT_MEGAKERNEL_DUAL, VARIANT_MEGAKERNEL_TENSOR, VARIANT_MEGAKERNEL_PACKED = 0, 1, 2, 3, 4, 5, 6, 7
VARIANT_MEGAKERNEL_TENSOR_STREAM = 9   # 8 stays unassigned (include/rays1_b200.h)
VARIANTS = {"mega": VARIANT_MEGAKERNEL, "wavefront": VARIANT_WAVEFRONT, "scalar": VARIANT_MEGAKERNEL_SCALAR, "coop": VARIANT_MEGAKERNEL_COOP,
            "deferred": VARIANT_MEGAKERNEL_DEFERRED, "dual": VARIANT_MEGAKERNEL_DUAL, "tensor": VARIANT_MEGAKERNEL_TENSOR, "packed": VARIANT_MEGAKERNEL_PACKED,
            "tensor_stream": VARIANT_MEGAKERNEL_TENSOR_STREAM}
MAT_NONE, MAT_LAMBERT, MAT_METAL, MAT_DIELECTRIC = -1, 0, 1, 2

# the reference's compile-time workload (src/common/common.h:18-25)
SCREEN_W, SCREEN_H, NUM_SAMPLES_PER_PIXEL, MAX_BOUNCES = 1280, 720, 250, 50
DEFAULT_ROW_TILE = 1  # rows per interleaved tile of the multi-GPU partition (library default)


class Rays1Error(RuntimeError):
    pass


class Result(C.Structure):
    """r1_result (replaces RESULT, src/common/common.h:36-45)."""
    _fields_ = [("elapsed_seconds", C.c_double), ("kernel_ms", C.c_double), ("trace_ms", C.c_double),
                ("num_rays", C.c_uint64), ("num_samples", C.c_uint64), ("launches", C.c_uint32), ("n_units", C.c_uint32)]

    def get_mrays_per_sec(self):
        return self.num_rays / self.elapsed_seconds / 1e6 if self.elapsed_seconds else 0.0


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("max_bounces", C.c_int32),
                ("variant", C.c_int32), ("seed", C.c_uint32), ("rank", C.c_int32), ("world", C.c_int32),
                ("row_tile", C.c_int32), ("blocks_per_sm", C.c_int32), ("threads", C.c_int32), ("device", C.c_int32)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: build it with `python -m rays1bench_b200.build` (nvcc, sm_100a). "
                          "There is no CPU fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
    i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
    u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
    u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
    u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    sig = {
        "r1_abi_version": (ci, []),
        "r1_last_error": (C.c_char_p, []),
        "r1_device_count": (ci, []),
        "r1_scene_create": (vp, [C.c_uint32]),
        "r1_scene_destroy": (None, [vp]),
        "r1_scene_set_camera": (ci, [vp, f32p, f32p, f32p, cf, cf, cf, cf]),
        "r1_scene_set_camera_raw": (ci, [vp, f32p]),
        "r1_scene_add_sphere": (ci, [vp, cf, cf, cf, cf, ci, cf, cf, cf, cf]),
        "r1_scene_pad": (ci, [vp, C.c_uint32]),
        "r1_scene_count": (C.c_uint32, [vp]),
        "r1_scene_get_soa": (ci, [vp, f32p, f32p, f32p, f32p, f32p, i32p, f32p, f32p]),
        "r1_scene_get_camera": (ci, [vp, f32p]),
        "r1_scene_commit": (ci, [vp, ci]),
        "r1_render": (ci, [vp, C.POINTER(RenderParams), u8p, C.POINTER(Result)]),
        "r1_render_device": (ci, [vp, C.POINTER(RenderParams), vp, vp, vp, C.POINTER(Result)]),
        "r1_render_wait": (ci, [vp, ci, C.POINTER(Result)]),
        "r1_wavefront_graph_builds": (ci, [ci]),
        "r1_local_rows": (C.c_int64, [ci, ci, ci, ci]),
        "r1_local_pixels": (C.c_int64, [ci, ci, ci, ci, ci]),
        "r1_global_row": (ci, [ci, ci, ci, ci]),
        "r1_deinterleave_rows": (ci, [ci, vp, C.c_uint64, vp, ci, ci, ci, ci, vp]),
        "r1_trace_rays": (ci, [vp, ci, f32p, f32p, cf, cf, ci, i32p, f32p, f32p, f32p]),
        "r1_filter_probe": (ci, [vp, ci, f32p, f32p, ci, f32p]),
        "r1_tensor_operand": (ci, [vp, u8p, C.c_uint64, C.POINTER(C.c_uint32)]),
        "r1_scatter": (ci, [vp, ci, f32p, f32p, f32p, i32p, f32p, f32p, i32p, f32p, f32p]),
        "r1_get_ray": (ci, [vp, ci, f32p, f32p, f32p, f32p, f32p]),
        "r1_replay_pixels": (ci, [vp, ci, i32p, ci, ci, ci, ci, u32p, u32p, f32p, u32p]),
        "r1_rng_draws": (ci, [C.c_uint32, C.c_uint32, C.c_uint32, ci, u32p]),
        "r1_sample_points": (ci, [ci, u32p, u32p, C.c_uint32, ci, f32p]),
        "r1_render_sums": (ci, [vp, C.POINTER(RenderParams), u64p, u8p, C.POINTER(Result)]),
        "r1_fma_peak": (ci, [ci, ci, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "r1_tmem_read_peak": (ci, [ci, ci, C.POINTER(C.c_double)]),
        "r1_kernel_name": (C.c_char_p, [vp, ci]),
        "r1_host_configure": (ci, [ci, ci, ci, ci, ci, ci, C.c_uint32]),
        "r1_host_set_quiet": (ci, [ci]),
        "r1_host_create_scene": (vp, [C.c_char_p, ci]),
        "r1_host_create_scene_from_file": (vp, [C.c_char_p, ci]),
        "r1_host_scene_handle": (vp, [vp]),
        "r1_host_benchmark": (ci, [vp, u8p, C.c_uint64, ci, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
        "r1_host_destroy_scene": (None, [vp]),
        "r1_host_write_tga": (ci, [C.c_char_p, ci, ci, u8p, C.c_uint64]),
        "r1_host_log_results": (ci, [C.c_char_p, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), ci]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what include/rays1_b200.h declares
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTED = _load()


def _check(rc, what):
    if rc < 0:
        raise Rays1Error("%s failed (%d): %s" % (what, rc, lib.r1_last_error().decode(errors="replace")))
    return rc


def device_count():
    return _check(lib.r1_device_count(), "r1_device_count")


# ------------------------------------------------------------------------------------------------ reference surface

class Scene:
    """Host scene handle (``Scene*`` of the reference, rayweek1.cpp:539-549).  ``benchmark`` consumes it."""

    def __init__(self, ptr, name):
        if not ptr:
            raise Rays1Error("scene %r could not be created: %s" % (name, lib.r1_last_error().decode(errors="replace")))
        self._ptr = ptr
        self.name = name

    @property
    def handle(self):
        if not self._ptr:
            raise Rays1Error("scene %r was already consumed by benchmark()" % self.name)
        return lib.r1_host_scene_handle(self._ptr)

    def close(self):
        if self._ptr:
            lib.r1_host_destroy_scene(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- inspection (parity tests)
    def count(self):
        return int(lib.r1_scene_count(self.handle))

    def soa(self):
        n = self.count()
        f = np.float32
        out = dict(cx=np.zeros(n, f), cy=np.zeros(n, f), cz=np.zeros(n, f), radius_sq=np.zeros(n, f), inv_radius=np.zeros(n, f),
                   kind=np.zeros(n, np.int32), albedo=np.zeros((n, 3), f), param=np.zeros(n, f))
        _check(lib.r1_scene_get_soa(self.handle, out["cx"], out["cy"], out["cz"], out["radius_sq"], out["inv_radius"], out["kind"],
                                    out["albedo"], out["param"]), "r1_scene_get_soa")
        return out

    def camera(self):
        out = np.zeros(22, np.float32)
        _check(lib.r1_scene_get_camera(self.handle, out), "r1_scene_get_camera")
        return out

    def set_camera_raw(self, cam22, device=None):
        """install the 22 camera constants as given (e.g. the reference's recorded ones) and re-commit the scene"""
        _check(lib.r1_scene_set_camera_raw(self.handle, np.ascontiguousarray(cam22, np.float32)), "r1_scene_set_camera_raw")
        if device is not None:
            _check(lib.r1_scene_commit(self.handle, device), "r1_scene_commit")

    # -- device entry points
    def render(self, width=SCREEN_W, height=SCREEN_H, spp=NUM_SAMPLES_PER_PIXEL, max_bounces=MAX_BOUNCES, variant=VARIANT_MEGAKERNEL,
               seed=0, rank=0, world=1, row_tile=DEFAULT_ROW_TILE, device=-1, blocks_per_sm=0, threads=0):
        """r1_render: host buffer out.  Returns (rgb[local_rows, width, 3] uint8 with row 0 = bottom, Result)."""
        p = RenderParams(width, height, spp, max_bounces, variant, seed, rank, world, row_tile, blocks_per_sm, threads, device)
        rows = int(lib.r1_local_rows(height, row_tile, rank, world))
        rgb = np.zeros((rows, width, 3), np.uint8)
        res = Result()
        buf = rgb if rgb.size else np.zeros(16, np.uint8)
        _check(lib.r1_render(self.handle, C.byref(p), buf, C.byref(res)), "r1_render")
        return rgb, res

    def render_sums(self, width=SCREEN_W, height=SCREEN_H, spp=NUM_SAMPLES_PER_PIXEL, max_bounces=MAX_BOUNCES, variant=VARIANT_MEGAKERNEL,
                    seed=0, rank=0, world=1, row_tile=DEFAULT_ROW_TILE, device=-1, blocks_per_sm=0, threads=0):
        """r1_render_sums: render() plus the fixed-point pixel sums the bytes were resolved from.
        Returns (rgb[local_rows, width, 3] uint8, sums[local_rows, width, 3] uint64 in units of 2^-24, Result)."""
        p = RenderParams(width, height, spp, max_bounces, variant, seed, rank, world, row_tile, blocks_per_sm, threads, device)
        rows = int(lib.r1_local_rows(height, row_tile, rank, world))
        rgb = np.zeros((rows, width, 3), np.uint8)
        sums = np.zeros((rows, width, 3), np.uint64)
        res = Result()
        _check(lib.r1_render_sums(self.handle, C.byref(p), sums.reshape(-1) if sums.size else np.zeros(1, np.uint64),
                                  rgb if rgb.size else np.zeros(16, np.uint8), C.byref(res)), "r1_render_sums")
        return rgb, sums, res

    def render_device(self, d_rgb_ptr, d_num_rays_ptr, stream_ptr=None, **kw):
        """r1_render_device: asynchronous, device pointers (e.g. torch tensors' data_ptr())."""
        p = RenderParams(kw.get("width", SCREEN_W), kw.get("height", SCREEN_H), kw.get("spp", NUM_SAMPLES_PER_PIXEL),
                         kw.get("max_bounces", MAX_BOUNCES), kw.get("variant", VARIANT_MEGAKERNEL), kw.get("seed", 0), kw.get("rank", 0),
                         kw.get("world", 1), kw.get("row_tile", DEFAULT_ROW_TILE), kw.get("blocks_per_sm", 0), kw.get("threads", 0), kw.get("device", -1))
        res = Result()
        _check(lib.r1_render_device(self.handle, C.byref(p), C.c_void_p(d_rgb_ptr), C.c_void_p(d_num_rays_ptr),
                                    C.c_void_p(stream_ptr or 0), C.byref(res)), "r1_render_device")
        return res

    def render_wait(self, device=-1):
        res = Result()
        _check(lib.r1_render_wait(self.handle, device, C.byref(res)), "r1_render_wait")
        return res

    def trace_rays(self, org, dir_, t_min=0.001, t_max=float(np.finfo(np.float32).max), variant=VARIANT_MEGAKERNEL):
        org = np.ascontiguousarray(org, np.float32).reshape(-1, 3)
        dir_ = np.ascontiguousarray(dir_, np.float32).reshape(-1, 3)
        n = org.shape[0]
        idx = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        p = np.zeros((n, 3), np.float32)
        nrm = np.zeros((n, 3), np.float32)
        _check(lib.r1_trace_rays(self.handle, n, org, dir_, t_min, t_max, variant, idx, t, p, nrm), "r1_trace_rays")
        return idx, t, p, nrm

    def tensor_operand(self):
        """r1_tensor_operand (host only): the sphere operand of the tensor-core filter as float32 [n32, 32] = {hi | hi | lo} words
        of the 11 lifted features, un-tiled from the tcgen05 core-matrix layout."""
        n32 = C.c_uint32(0)
        n = (self.count() + 31) // 32 * 32
        raw = np.zeros(max(n, 32) * 128, np.uint8)
        _check(lib.r1_tensor_operand(self.handle, raw, raw.size, C.byref(n32)), "r1_tensor_operand")
        r, k = np.meshgrid(np.arange(n32.value), np.arange(32), indexing="ij")
        off = (r // 8) * 1024 + (k // 4) * 128 + (r % 8) * 16 + (k % 4) * 4
        return raw.view(np.float32)[off // 4]

    def filter_probe(self, org, dir_, n_spheres, layout=0):
        """r1_filter_probe: values of the tensor-core filter, shape (rays, n32); sign bit clear = sphere flagged."""
        org = np.ascontiguousarray(org, np.float32).reshape(-1, 3)
        dir_ = np.ascontiguousarray(dir_, np.float32).reshape(-1, 3)
        n, n32 = org.shape[0], (n_spheres + 31) // 32 * 32
        e = np.zeros((n, n32), np.float32)
        _check(lib.r1_filter_probe(self.handle, n, org, dir_, layout, e.reshape(-1)), "r1_filter_probe")
        return e

    def scatter(self, dir_in, p, normal, index, rand_sphere, rand_u):
        c = lambda a, dt=np.float32: np.ascontiguousarray(a, dt)  # noqa: E731
        n = len(index)
        ok = np.zeros(n, np.int32)
        atten = np.zeros((n, 3), np.float32)
        dout = np.zeros((n, 3), np.float32)
        _check(lib.r1_scatter(self.handle, n, c(dir_in), c(p), c(normal), c(index, np.int32), c(rand_sphere), c(rand_u), ok, atten, dout),
               "r1_scatter")
        return ok, atten, dout

    def replay_pixels(self, xy, width, height, spp, state, state4, max_bounces=MAX_BOUNCES):
        """r1_replay_pixels: per-pixel radiance sums driven by the reference's xorshift streams from recorded states."""
        n = len(xy)
        col = np.zeros((n, 3), np.float32)
        rays = np.zeros(n, np.uint32)
        _check(lib.r1_replay_pixels(self.handle, n, np.ascontiguousarray(xy, np.int32).reshape(-1), width, height, spp, max_bounces,
                                    np.ascontiguousarray(state, np.uint32), np.ascontiguousarray(state4, np.uint32).reshape(-1),
                                    col.reshape(-1), rays), "r1_replay_pixels")
        return col, rays

    def get_ray(self, su, tv, disk):
        n = len(su)
        org = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        _check(lib.r1_get_ray(self.handle, n, np.ascontiguousarray(su, np.float32), np.ascontiguousarray(tv, np.float32),
                              np.ascontiguousarray(disk, np.float32), org, d), "r1_get_ray")
        return org, d


_configured = {"width": SCREEN_W, "height": SCREEN_H}


def configure(width=0, height=0, spp=0, max_bounces=0, variant=-1, n_gpus=0, seed=0, quiet=None):
    """Runtime stand-in for the reference's compile-time macros (common.h:3-31).  Affects scenes created afterwards
    (camera aspect, GPU replicas) and benchmark()."""
    _check(lib.r1_host_configure(width, height, spp, max_bounces, variant, n_gpus, seed), "r1_host_configure")
    if width > 0:
        _configured["width"] = width
    if height > 0:
        _configured["height"] = height
    if quiet is not None:
        lib.r1_host_set_quiet(1 if quiet else 0)


def create_scene(name, commit=True):
    """commit=False builds the host SoA only (no GPU needed); such a scene cannot render."""
    return Scene(lib.r1_host_create_scene(name.encode(), 1 if commit else 0), name)


def create_scene_from_file(path, commit=True):
    """Scene from a text description (see include/rays1_b200.h: camera / sphere statements)."""
    return Scene(lib.r1_host_create_scene_from_file(os.fsencode(path), 1 if commit else 0), os.path.basename(path))


def write_scene_file(path, camera_args, spheres):
    """camera_args = (from xyz, at xyz, vfov, aperture, focus); spheres = iterable of (cx, cy, cz, radius, kind, r, g, b, param)."""
    names = {MAT_LAMBERT: "lambert", MAT_METAL: "metal", MAT_DIELECTRIC: "dielectric", MAT_NONE: "none"}
    with open(path, "w") as f:
        f.write("camera " + " ".join("%.9g" % v for v in camera_args) + "\n")
        for cx, cy, cz, radius, kind, r, g, b, param in spheres:
            f.write("sphere %.9g %.9g %.9g %.9g %s" % (cx, cy, cz, radius, names[int(kind)]))
            if kind == MAT_LAMBERT:
                f.write(" %.9g %.9g %.9g" % (r, g, b))
            elif kind == MAT_METAL:
                f.write(" %.9g %.9g %.9g %.9g" % (r, g, b, param))
            elif kind == MAT_DIELECTRIC:
                f.write(" %.9g" % param)
            f.write("\n")


def create_small_scene():
    """rayweek1.cpp:552-579"""
    return create_scene("small")


def create_medium_scene():
    """rayweek1.cpp:582-651"""
    return create_scene("medium")


def create_large_scene():
    """rayweek1.cpp:654-719"""
    return create_scene("large")


def create_synth4096_scene():
    """SURVEY.md 8d config 5 (not in the reference): 66 x 62 grid + 4 = 4096 spheres."""
    return create_scene("synth4096")


def benchmark(scene, pixels, write_tga, scene_name):
    """benchmark(scene, pixels, write_tga, scene_name) of the reference (rayweek1.cpp:845-927): renders into the
    caller-owned ``pixels`` (uint8[H, W, 3], row 0 = bottom), prints the report block, CONSUMES the scene, optionally writes
    out_<scene_name>.tga (which swaps R and B in ``pixels`` in place).  Returns a Result (elapsed_seconds, num_rays)."""
    if pixels.dtype != np.uint8 or not pixels.flags["C_CONTIGUOUS"]:
        raise ValueError("pixels must be a C-contiguous uint8 array")
    need = _configured["width"] * _configured["height"] * 3
    if pixels.size != need:
        raise ValueError("pixels has %d bytes, the configured %dx%d image needs %d (call configure() first)" %
                         (pixels.size, _configured["width"], _configured["height"], need))
    el, rays, kms = C.c_double(0), C.c_uint64(0), C.c_double(0)
    ptr, scene._ptr = scene._ptr, None  # ownership moves to benchmark() (delete scene, rayweek1.cpp:905)
    if not ptr:
        raise Rays1Error("scene %r was already consumed" % scene.name)
    _check(lib.r1_host_benchmark(ptr, pixels.reshape(-1), pixels.size, 1 if write_tga else 0, scene_name.encode(), C.byref(el), C.byref(rays),
                                 C.byref(kms)), "benchmark")
    res = Result()
    res.elapsed_seconds, res.num_rays, res.kernel_ms = el.value, rays.value, kms.value
    return res


def tga_write_rgb24(filename, width, height, pixels):
    """tga_write_rgb24 (common.h:86-122).  !!! swaps R and B in ``pixels`` in place, like the reference."""
    if pixels.dtype != np.uint8 or not pixels.flags["C_CONTIGUOUS"] or pixels.size < width * height * 3:
        raise ValueError("pixels must be a C-contiguous uint8 array of at least width * height * 3 bytes")
    _check(lib.r1_host_write_tga(filename.encode(), width, height, pixels.reshape(-1), pixels.size), "tga_write_rgb24")


def log_results(version, scene, results):
    """log_results (common.h:47-77) -> out_<scene>.txt in the current directory."""
    n = len(results)
    el = (C.c_double * n)(*[r.elapsed_seconds for r in results])
    rays = (C.c_uint64 * n)(*[r.num_rays for r in results])
    _check(lib.r1_host_log_results(version.encode(), scene.encode(), el, rays, n), "log_results")


def rng_draws(pixel, sample, seed, n):
    out = np.zeros(n, np.uint32)
    _check(lib.r1_rng_draws(pixel, sample, seed, n, out), "r1_rng_draws")
    return out


def sample_points(pixel, sample, seed, bounces):
    """r1_sample_points: the random points a render draws for the (global pixel, sample) keys -> float32 [n, 2 + 4 bounces]:
    lens-disk (x, y), then (ru, ball x, y, z) per depth."""
    pixel = np.ascontiguousarray(pixel, np.uint32).reshape(-1)
    sample = np.ascontiguousarray(sample, np.uint32).reshape(-1)
    if pixel.shape != sample.shape:
        raise ValueError("pixel and sample keys differ in length")
    out = np.zeros((len(pixel), 2 + 4 * max(bounces, 0)), np.float32)   # bounces < 0: the library refuses it
    _check(lib.r1_sample_points(len(pixel), pixel, sample, seed, bounces, out.reshape(-1) if out.size else np.zeros(1, np.float32)),
           "r1_sample_points")
    return out


def fma_peak(device=0, packed=False):
    """FP32 FMA throughput microbenchmark -> (TFLOP/s, estimated SM MHz)."""
    tf, mhz = C.c_double(0), C.c_double(0)
    _check(lib.r1_fma_peak(device, 1 if packed else 0, C.byref(tf), C.byref(mhz)), "r1_fma_peak")
    return tf.value, mhz.value


def tmem_read_peak(device=0, warps=16):
    """TMEM read throughput microbenchmark -> bytes per second per SM."""
    v = C.c_double(0)
    _check(lib.r1_tmem_read_peak(device, warps, C.byref(v)), "r1_tmem_read_peak")
    return v.value


def local_rows(height, row_tile, rank, world):
    return int(lib.r1_local_rows(height, row_tile, rank, world))


def global_row(local_row, row_tile, rank, world):
    return int(lib.r1_global_row(local_row, row_tile, rank, world))


def assemble_rows(parts, height, row_tile=DEFAULT_ROW_TILE):
    """Host-side de-interleave of per-rank row blocks (used by tests; the product path does this on the GPU)."""
    world = len(parts)
    width = parts[0].shape[1]
    out = np.zeros((height, width, 3), np.uint8)
    for r, part in enumerate(parts):
        for lr in range(part.shape[0]):
            out[global_row(lr, row_tile, r, world)] = part[lr]
    return out


# FLOPs per ray for the roofline (SURVEY.md 8d / BASELINE.md 4): 16 per ray-sphere test (FMA = 2) x real spheres + 70 shading
def flops_per_ray(n_real_spheres):
    return 16 * n_real_spheres + 70


REAL_SPHERES = {"small": 5, "medium": 46, "large": 484, "synth4096": 4096}
