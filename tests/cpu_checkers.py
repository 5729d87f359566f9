"""ctypes bindings for the two CPU checkers (test infrastructure only).

* ``Oracle``  -- oracle/librays1_oracle.so, the plain-C restatement (always available; built by oracle/Makefile).
* ``RefLib``  -- oracle/_ref/libref_rays1.so, C entry points around the UNMODIFIED reference sources
  (/root/reference/src/latest compiled where it lies).  Present wherever oracle/_ref/ was built or shipped.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "librays1_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_rays1.so")
REF4096_SO = os.path.join(ROOT, "oracle", "_ref", "libref_rays1_4096.so")  # MAX_SPHERES patched to 4096 (oracle/Makefile)
REF_NATIVE_SO = os.path.join(ROOT, "oracle", "_ref", "libref_rays1_native.so")  # timing build: the reference's exact flags (-flto -march=native)
REF_EXE = os.path.join(ROOT, "oracle", "_ref", "rays1_latest")

_f = np.float32
_fp = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_up = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_bp = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


def build_oracle():
    """(Re)build the checkers with oracle/Makefile (gcc only; the _ref targets are skipped without /root/reference)."""
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s"], check=True)


class _Checker:
    """Common surface of the oracle and the reference harness (same entry points, different prefix)."""

    def __init__(self, path, prefix, has_size_args):
        self.lib = C.CDLL(path)
        self.prefix = prefix
        self._has_size_args = has_size_args
        g = lambda name: getattr(self.lib, prefix + name)  # noqa: E731
        g("scene_create").restype = C.c_void_p
        g("scene_create").argtypes = [C.c_char_p, C.c_int, C.c_int] if has_size_args else [C.c_char_p]
        g("scene_destroy").argtypes = [C.c_void_p]
        g("scene_count").restype = C.c_uint32
        g("scene_count").argtypes = [C.c_void_p]
        g("scene_get_soa").argtypes = [C.c_void_p, _fp, _fp, _fp, _fp, _fp, _ip, _fp, _fp]
        g("scene_get_camera").argtypes = [C.c_void_p, _fp]
        g("hit").argtypes = [C.c_void_p, C.c_int, _fp, _fp, C.c_float, C.c_float, _ip, _fp, _fp, _fp]
        for n in ("xorshift32",):
            g(n).restype = C.c_uint32
            g(n).argtypes = [_up]
        for n in ("myrand01", "myrand02"):
            g(n).restype = C.c_float
            g(n).argtypes = [_up]
        g("myrand01_x4").argtypes = [_up, _fp]
        g("random_in_unit_sphere").argtypes = [_up, _fp]
        g("random_in_unit_disk").argtypes = [_up, _fp]
        self._g = g

    # -- scenes
    def scene_create(self, name, w=1280, h=720):
        if self._has_size_args:
            s = self._g("scene_create")(name.encode(), w, h)
        else:
            assert w * 9 == h * 16, "the reference hard-codes a 16:9 aspect (SCREEN_W/SCREEN_H, common.h:19-20)"
            s = self._g("scene_create")(name.encode())
        if not s:
            raise ValueError("unknown scene %r" % name)
        return s

    def scene_destroy(self, s):
        self._g("scene_destroy")(s)

    def scene_count(self, s):
        return int(self._g("scene_count")(s))

    def scene_soa(self, s):
        n = self.scene_count(s)
        out = dict(cx=np.zeros(n, _f), cy=np.zeros(n, _f), cz=np.zeros(n, _f), radius_sq=np.zeros(n, _f),
                   inv_radius=np.zeros(n, _f), kind=np.zeros(n, np.int32), albedo=np.zeros((n, 3), _f),
                   param=np.zeros(n, _f))
        self._g("scene_get_soa")(s, out["cx"], out["cy"], out["cz"], out["radius_sq"], out["inv_radius"],
                                 out["kind"], out["albedo"], out["param"])
        return out

    def scene_camera(self, s):
        out = np.zeros(22, _f)
        self._g("scene_get_camera")(s, out)
        return out

    # -- hit
    def hit(self, s, org, dir_, t_min=0.001, t_max=np.finfo(np.float32).max):
        org = np.ascontiguousarray(org, _f)
        dir_ = np.ascontiguousarray(dir_, _f)
        n = org.shape[0]
        idx = np.zeros(n, np.int32)
        t = np.zeros(n, _f)
        p = np.zeros((n, 3), _f)
        nrm = np.zeros((n, 3), _f)
        self._g("hit")(s, n, org, dir_, t_min, t_max, idx, t, p, nrm)
        return idx, t, p, nrm

    # -- rng
    def xorshift32(self, state):
        st = np.array([state], np.uint32)
        v = self._g("xorshift32")(st)
        return int(v), int(st[0])

    def myrand01(self, state):
        st = np.array([state], np.uint32)
        return float(self._g("myrand01")(st)), int(st[0])

    def myrand02(self, state):
        st = np.array([state], np.uint32)
        return float(self._g("myrand02")(st)), int(st[0])

    def myrand01_x4(self, state4):
        st = np.array(state4, np.uint32)
        out = np.zeros(4, _f)
        self._g("myrand01_x4")(st, out)
        return out, st

    def random_in_unit_sphere(self, state4):
        st = np.array(state4, np.uint32)
        out = np.zeros(3, _f)
        self._g("random_in_unit_sphere")(st, out)
        return out, st

    def random_in_unit_disk(self, state):
        st = np.array([state], np.uint32)
        out = np.zeros(2, _f)
        self._g("random_in_unit_disk")(st, out)
        return out, int(st[0])


class Oracle(_Checker):
    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        super().__init__(ORACLE_SO, "orc_", True)
        L = self.lib
        L.orc_scatter.argtypes = [C.c_void_p, C.c_int, _fp, _fp, _fp, _ip, _fp, _fp, _ip, _fp, _fp]
        L.orc_get_ray.argtypes = [C.c_void_p, C.c_int, _fp, _fp, _fp, _fp, _fp]
        L.orc_replay_pixels.argtypes = [C.c_void_p, C.c_int, _ip, C.c_int, C.c_int, C.c_int, C.c_int, _up, _up, _fp, _up]
        L.orc_scene_set_camera.argtypes = [C.c_void_p, _fp]
        L.orc_rsqrt12.restype = C.c_float
        L.orc_rsqrt12.argtypes = [C.c_float]
        L.orc_hw_rsqrtss.restype = C.c_float
        L.orc_hw_rsqrtss.argtypes = [C.c_float]
        L.orc_render.restype = C.c_uint64
        L.orc_render.argtypes = [C.c_void_p, _bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.orc_scene_create_from_soa.restype = C.c_void_p
        L.orc_scene_create_from_soa.argtypes = [C.c_int, _fp, _fp, _fp, _fp, _fp, _ip, _fp, _fp]
        L.orc_keyed_draw.restype = C.c_uint32
        L.orc_keyed_draw.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.orc_quantise_radiance.restype = C.c_uint32
        L.orc_quantise_radiance.argtypes = [C.c_float]
        L.orc_resolve.restype = C.c_uint8
        L.orc_resolve.argtypes = [C.c_uint64, C.c_int]
        L.orc_local_rows.restype = C.c_int
        L.orc_local_rows.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_render_keyed.restype = C.c_int64
        L.orc_render_keyed.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       _u64p, _bp, C.POINTER(C.c_uint64)]

    # -- the device integrator (counter-based generator, forward throughput, fixed-point sums)
    def keyed_draw(self, pixel, sample, seed, i):
        return int(self.lib.orc_keyed_draw(pixel, sample, seed, i))

    def quantise_radiance(self, c):
        return int(self.lib.orc_quantise_radiance(c))

    def resolve(self, total, spp):
        return int(self.lib.orc_resolve(total, spp))

    def local_rows(self, height, row_tile, rank, world):
        return int(self.lib.orc_local_rows(height, row_tile, rank, world))

    def render_keyed(self, s, w, h, spp, max_bounces, seed=0, rank=0, world=1, row_tile=1, points=None):
        """The rank's rows as the GPU renderer computes them -> (sums[rows, w, 3] uint64, rgb[rows, w, 3] uint8, num_rays).
        points: r1.sample_points() of the rank's (pixel, sample) keys in local pixel order (bit-exact), or None (libm)."""
        rows = self.local_rows(h, row_tile, rank, world)
        sums = np.zeros((rows, w, 3), np.uint64)
        rgb = np.zeros((rows, w, 3), np.uint8)
        rays = C.c_uint64(0)
        if points is not None:
            points = np.ascontiguousarray(points, _f)
            assert points.size == rows * w * spp * (2 + 4 * max_bounces), "points table does not match the rank's samples"
        n = self.lib.orc_render_keyed(s, w, h, spp, max_bounces, seed, rank, world, row_tile,
                                      None if points is None else points.ctypes.data, sums.reshape(-1) if sums.size else np.zeros(1, np.uint64),
                                      rgb.reshape(-1) if rgb.size else np.zeros(1, np.uint8), C.byref(rays))
        assert n == rows * w
        return sums, rgb, int(rays.value)

    def scene_create_from_soa(self, soa):
        """a scene holding the spheres of ``soa`` (the dict of Scene.soa() / scene_soa()) as given, for hit() on any scene;
        destroy it with scene_destroy"""
        c = lambda k, dt=_f: np.ascontiguousarray(soa[k], dt)  # noqa: E731
        s = self.lib.orc_scene_create_from_soa(len(soa["cx"]), c("cx"), c("cy"), c("cz"), c("radius_sq"), c("inv_radius"), c("kind", np.int32),
                                               c("albedo"), c("param"))
        if not s:
            raise ValueError("orc_scene_create_from_soa failed")
        return s

    def scene_set_camera(self, s, cam22):
        self.lib.orc_scene_set_camera(s, np.ascontiguousarray(cam22, _f))

    def scatter(self, s, dir_in, p, normal, index, rand_sphere, rand_u):
        n = len(index)
        ok = np.zeros(n, np.int32)
        atten = np.zeros((n, 3), _f)
        dout = np.zeros((n, 3), _f)
        self.lib.orc_scatter(s, n, np.ascontiguousarray(dir_in, _f), np.ascontiguousarray(p, _f),
                             np.ascontiguousarray(normal, _f), np.ascontiguousarray(index, np.int32),
                             np.ascontiguousarray(rand_sphere, _f), np.ascontiguousarray(rand_u, _f), ok, atten, dout)
        return ok, atten, dout

    def get_ray(self, s, su, tv, disk):
        n = len(su)
        org = np.zeros((n, 3), _f)
        d = np.zeros((n, 3), _f)
        self.lib.orc_get_ray(s, n, np.ascontiguousarray(su, _f), np.ascontiguousarray(tv, _f),
                             np.ascontiguousarray(disk, _f), org, d)
        return org, d

    def replay_pixels(self, s, xy, w, h, spp, state, state4, max_bounces=50):
        n = len(xy)
        col = np.zeros((n, 3), _f)
        rays = np.zeros(n, np.uint32)
        self.lib.orc_replay_pixels(s, n, np.ascontiguousarray(xy, np.int32), w, h, spp, max_bounces, np.ascontiguousarray(state, np.uint32),
                                   np.ascontiguousarray(state4, np.uint32), col, rays)
        return col, rays

    def render(self, s, w, h, spp, max_bounces=50, threads=0):
        """threads <= 0: the reference's single-thread branch (deterministic seeds, rayweek1.cpp:880-881)."""
        rgb = np.zeros((h, w, 3), np.uint8)
        el = C.c_double(0)
        rays = self.lib.orc_render(s, rgb, w, h, spp, max_bounces, threads, C.byref(el))
        return rgb, int(rays), el.value


class RefLib(_Checker):
    """max_spheres=4096 selects the build whose Hitable::hit holds 4096 spheres (the one-line MAX_SPHERES patch of
    rayweek1.cpp:174, SURVEY.md section 7 step 1); it also knows the "synth4096" scene (BASELINE.json config 5)."""

    @staticmethod
    def available(max_spheres=1024):
        return os.path.exists(REF4096_SO if max_spheres > 1024 else REF_SO)

    def __init__(self, max_spheres=1024, native=False):
        super().__init__(REF4096_SO if max_spheres > 1024 else (REF_NATIVE_SO if native else REF_SO), "ref_", False)
        L = self.lib
        assert L.ref_max_spheres() >= max_spheres
        L.ref_record_paths.restype = C.c_int
        L.ref_record_paths.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint32, _fp, _fp, _ip, _ip, _fp, _fp,
                                       _fp, _fp, _fp, _ip, _fp, _fp, _fp, _fp, _fp]
        L.ref_get_ray.argtypes = [C.c_void_p, C.c_int, _fp, _fp, C.c_uint32, _fp, _fp, _fp]
        L.ref_hit_scatter.argtypes = [C.c_void_p, C.c_int, _fp, _fp, C.c_uint32, _ip, _fp, _fp, _fp, _fp, _fp, _ip, _fp, _fp]
        L.ref_render.restype = C.c_uint64
        L.ref_render.argtypes = [C.c_void_p, _bp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.ref_hardware_concurrency.restype = C.c_int
        L.ref_replay_pixels.argtypes = [C.c_void_p, C.c_int, _ip, C.c_int, C.c_int, C.c_int, C.c_uint32, _up, _up, _fp, _up]

    def record_paths(self, s, n, w=1280, h=720, seed=1):
        a = dict(org=np.zeros((n, 3), _f), dir=np.zeros((n, 3), _f), depth=np.zeros(n, np.int32),
                 index=np.zeros(n, np.int32), t=np.zeros(n, _f), p=np.zeros((n, 3), _f), normal=np.zeros((n, 3), _f),
                 rand_sphere=np.zeros((n, 3), _f), rand_u=np.zeros(n, _f), scat_ok=np.zeros(n, np.int32),
                 atten=np.zeros((n, 3), _f), scat_dir=np.zeros((n, 3), _f), cam_su=np.zeros(n, _f),
                 cam_tv=np.zeros(n, _f), cam_disk=np.zeros((n, 2), _f))
        got = self.lib.ref_record_paths(s, n, w, h, seed, a["org"], a["dir"], a["depth"], a["index"], a["t"], a["p"],
                                        a["normal"], a["rand_sphere"], a["rand_u"], a["scat_ok"], a["atten"],
                                        a["scat_dir"], a["cam_su"], a["cam_tv"], a["cam_disk"])
        return {k: v[:got] for k, v in a.items()}

    def hit_scatter(self, s, org, dir_, seed=9):
        """Hitable::hit + Material::scatter for given rays; returns the record ref_record_paths writes per segment."""
        org = np.ascontiguousarray(org, _f)
        dir_ = np.ascontiguousarray(dir_, _f)
        n = org.shape[0]
        a = dict(org=org, dir=dir_, index=np.zeros(n, np.int32), t=np.zeros(n, _f), p=np.zeros((n, 3), _f), normal=np.zeros((n, 3), _f),
                 rand_sphere=np.zeros((n, 3), _f), rand_u=np.zeros(n, _f), scat_ok=np.zeros(n, np.int32), atten=np.zeros((n, 3), _f),
                 scat_dir=np.zeros((n, 3), _f))
        self.lib.ref_hit_scatter(s, n, org, dir_, seed, a["index"], a["t"], a["p"], a["normal"], a["rand_sphere"], a["rand_u"],
                                 a["scat_ok"], a["atten"], a["scat_dir"])
        return a

    def get_ray(self, s, su, tv, seed=10001):
        n = len(su)
        disk = np.zeros((n, 2), _f)
        org = np.zeros((n, 3), _f)
        d = np.zeros((n, 3), _f)
        self.lib.ref_get_ray(s, n, np.ascontiguousarray(su, _f), np.ascontiguousarray(tv, _f), seed, disk, org, d)
        return disk, org, d

    def replay_pixels(self, s, xy, w, h, spp, seed=5):
        """-> (state[n], state4[n,4] before each pixel, float colour sum[n,3], rays[n])"""
        n = len(xy)
        state = np.zeros(n, np.uint32)
        state4 = np.zeros((n, 4), np.uint32)
        col = np.zeros((n, 3), _f)
        rays = np.zeros(n, np.uint32)
        self.lib.ref_replay_pixels(s, n, np.ascontiguousarray(xy, np.int32), w, h, spp, seed, state, state4, col, rays)
        return state, state4, col, rays

    def render(self, s, w, h, spp, threads=0):
        """threads <= 0: std::thread::hardware_concurrency(), as benchmark() does (rayweek1.cpp:869)."""
        rgb = np.zeros((h, w, 3), np.uint8)
        el = C.c_double(0)
        rays = self.lib.ref_render(s, rgb, w, h, spp, threads, C.byref(el))
        return rgb, int(rays), el.value

    def hardware_concurrency(self):
        return int(self.lib.ref_hardware_concurrency())
