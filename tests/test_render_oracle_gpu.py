"""Whole renders, bit for bit, against the oracle's restatement of the device integrator (orc_render_keyed).

Every variant shares the code that turns hits and scatters into pixels: the primary ray's RNG key and jitter, the draw indices of
each bounce, the forward throughput product, the depth cap, the fixed-point quantiser, the 64-bit pixel sums, the resolve, the
work decomposition (rank rows, row tiles, units of several samples above 256 spp) and the ray counter.  Comparing variants with
each other cannot see a fault there, and the statistical gates against the reference cannot see a last-bit rounding fault, a
shifted draw index or permuted keys.  Here each render's fixed-point sums (r1_render_sums), then its bytes, then its ray count
must equal the oracle's exactly.  The oracle takes the lens-disk and unit-ball samples, the one part of a sample a CPU cannot
reproduce (SFU approximations), from r1_sample_points; everything else -- the generator included -- it computes itself."""
import contextlib

import numpy as np
import pytest

from test_gpu_parity import scenes  # noqa: F401  (module fixture: the four built-in scenes)
from test_render_oracle_cpu import KEYS, SEEDS, keyed_draws, rand01, rand02
from test_scan_edges_gpu import FLT_MAX, RawScene, _f, edge_scenes  # noqa: F401
from test_tensor_stream_gpu import big_scenes  # noqa: F401

pytestmark = pytest.mark.gpu

MB = 50                                   # the reference's MAX_BOUNCES
POINTS_BUDGET = 64 << 20                  # bytes of injected points per oracle call; larger cases are split by rows
SIZES = ((1, 1, 1), (7, 3, 5), (33, 7, 3), (96, 54, 8))
FRAME = (96, 54, 8)


# ---- helpers ----------------------------------------------------------------------------------------------------------------

@contextlib.contextmanager
def environment(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        yield
    finally:
        for k in env:
            monkeypatch.delenv(k, raising=False)


def global_rows(oracle, h, rank, world, row_tile):
    return [((lr // row_tile) * world + rank) * row_tile + lr % row_tile for lr in range(oracle.local_rows(h, row_tile, rank, world))]


def sample_keys(ys, w, spp):
    """(global pixel, sample) of every sample of rows ys, in the oracle's order: local pixel, then sample"""
    pix = (np.asarray(ys, np.int64)[:, None] * w + np.arange(w)[None, :]).reshape(-1)
    return np.repeat(pix, spp).astype(np.uint32), np.tile(np.arange(spp), len(pix)).astype(np.uint32)


class Expected:
    """The oracle's renders of the GPU scenes, cached per (scene, image, partition): every variant is compared with one oracle
    render.  The oracle scene is built from the GPU scene's own SoA and camera constants."""

    def __init__(self, r1, oracle):
        self.r1, self.oracle, self.scenes, self.renders = r1, oracle, {}, {}

    def scene(self, s):
        key = s.handle
        if key not in self.scenes:
            so = self.oracle.scene_create_from_soa(s.soa())
            self.oracle.scene_set_camera(so, s.camera())
            self.scenes[key] = so
        return self.scenes[key]

    def render(self, s, w, h, spp, mb, seed, rank, world, row_tile):
        key = (s.handle, w, h, spp, mb, seed, rank, world, row_tile)
        if key not in self.renders:
            self.renders[key] = self._render(self.scene(s), w, h, spp, mb, seed, rank, world, row_tile)
        return self.renders[key]

    def _render(self, so, w, h, spp, mb, seed, rank, world, row_tile):
        ys = global_rows(self.oracle, h, rank, world, row_tile)
        row_bytes = w * spp * (2 + 4 * mb) * 4
        parts = max(1, -(-len(ys) * row_bytes // POINTS_BUDGET))
        if parts == 1:
            pts = self.r1.sample_points(*sample_keys(ys, w, spp), seed, mb)
            return self.oracle.render_keyed(so, w, h, spp, mb, seed, rank, world, row_tile, pts)
        # split by rows: rows y = r (mod parts) of a whole image are rank r of `parts` with single-row tiles
        assert world == 1, "only whole images are split"
        sums, rgb, rays = np.zeros((h, w, 3), np.uint64), np.zeros((h, w, 3), np.uint8), 0
        for r in range(parts):
            sub = global_rows(self.oracle, h, r, parts, 1)
            pts = self.r1.sample_points(*sample_keys(sub, w, spp), seed, mb)
            s_, c_, n_ = self.oracle.render_keyed(so, w, h, spp, mb, seed, r, parts, 1, pts)
            sums[sub], rgb[sub], rays = s_, c_, rays + n_
        return sums, rgb, rays

    def close(self):
        for so in self.scenes.values():
            self.oracle.scene_destroy(so)


@pytest.fixture(scope="module")
def expected(r1, oracle):
    e = Expected(r1, oracle)
    yield e
    e.close()


def first_difference(got, want, ys):
    bad = np.argwhere((got != want).reshape(len(ys), -1, 3).any(axis=2))
    lr, x = bad[0]
    return len(bad), int(x), int(ys[lr]), lr


def assert_matches(expected, s, got_sums, got_rgb, got_rays, w, h, spp, mb=MB, seed=0, rank=0, world=1, row_tile=1, what=""):
    """sums, then bytes, then the ray count; a failure names the first differing pixel by its global (x, y)"""
    want_sums, want_rgb, want_rays = expected.render(s, w, h, spp, mb, seed, rank, world, row_tile)
    ys = global_rows(expected.oracle, h, rank, world, row_tile)
    case = "%s %dx%dx%d bounces %d seed %d rank %d/%d tile %d" % (what, w, h, spp, mb, seed, rank, world, row_tile)
    assert got_sums.shape == want_sums.shape and got_rgb.shape == want_rgb.shape, case
    if not np.array_equal(got_sums, want_sums):
        n, x, y, lr = first_difference(got_sums, want_sums, ys)
        raise AssertionError("%s: fixed-point sums differ at %d pixels; first at (x %d, y %d): GPU %s, oracle %s; rays GPU %d, oracle %d"
                             % (case, n, x, y, got_sums[lr, x].tolist(), want_sums[lr, x].tolist(), got_rays, want_rays))
    if not np.array_equal(got_rgb, want_rgb):
        n, x, y, lr = first_difference(got_rgb, want_rgb, ys)
        raise AssertionError("%s: bytes differ at %d pixels (sums agree); first at (x %d, y %d): GPU %s, oracle %s, sums %s"
                             % (case, n, x, y, got_rgb[lr, x].tolist(), want_rgb[lr, x].tolist(), want_sums[lr, x].tolist()))
    assert got_rays == want_rays, "%s: %d rays, oracle %d (sums and bytes agree)" % (case, got_rays, want_rays)


def check(r1, expected, monkeypatch, s, w, h, spp, mb=MB, seed=0, rank=0, world=1, row_tile=1, variant=0, threads=0, blocks_per_sm=0,
          env=None, what=""):
    with environment(monkeypatch, env or {}):
        rgb, sums, res = s.render_sums(w, h, spp, mb, variant, seed, rank, world, row_tile, threads=threads, blocks_per_sm=blocks_per_sm)
    assert_matches(expected, s, sums, rgb, res.num_rays, w, h, spp, mb, seed, rank, world, row_tile,
                   what="%s (variant %d, threads %d, blocks/SM %d, %s)" % (what, variant, threads, blocks_per_sm, env or {}))
    return rgb, sums, res


# ---- the generator and the injected points ---------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", SEEDS)
def test_generator_matches_the_oracle(r1, oracle, seed):
    idx = np.arange(160, dtype=np.uint32)
    for pixel, sample in KEYS:
        got = r1.rng_draws(pixel, sample, seed, len(idx))
        assert np.array_equal(got, keyed_draws(pixel, sample, seed, idx)), (pixel, sample, seed)
        assert [oracle.keyed_draw(pixel, sample, seed, i) for i in (0, 3, 155)] == got[[0, 3, 155]].tolist()


@pytest.mark.parametrize("seed", SEEDS)
def test_sample_points(r1, seed):
    """ru is the CPU's rand01 bit for bit; the disk and ball points are the libm formulas within 1e-5 and lie in the unit disk /
    ball"""
    bounces = 6
    rng = np.random.default_rng(seed & 0xFFFF)
    pixel = np.concatenate([[k[0] for k in KEYS], rng.integers(0, 1 << 32, 3000)]).astype(np.uint32)
    sample = np.concatenate([[k[1] for k in KEYS], rng.integers(0, 1 << 20, 3000)]).astype(np.uint32)
    pts = r1.sample_points(pixel, sample, seed, bounces)
    assert pts.shape == (len(pixel), 2 + 4 * bounces)
    idx = np.arange(4 + 3 * bounces, dtype=np.uint32)
    draws = np.stack([keyed_draws(int(p), int(s), seed, idx) for p, s in zip(pixel, sample)])
    r, a = np.sqrt(rand01(draws[:, 2]).astype(np.float64)), rand02(draws[:, 3]).astype(np.float64) * np.pi
    disk = np.stack([r * np.cos(a), r * np.sin(a)], axis=1)
    assert np.abs(pts[:, :2] - disk).max() < 1e-5
    assert (np.hypot(pts[:, 0].astype(np.float64), pts[:, 1]) <= 1 + 1e-5).all()
    for d in range(bounces):
        i = 4 + 3 * d
        q = pts[:, 2 + 4 * d: 6 + 4 * d]
        ru = rand01(draws[:, i])
        assert np.array_equal(q[:, 0].view(np.uint32), ru.view(np.uint32)), "depth %d: ru is not rand01(4 + 3 d)" % d
        z = (np.float32(1) - rand02(draws[:, i + 1])).astype(np.float64)
        az = rand02(draws[:, i + 2]).astype(np.float64) * np.pi
        rad = np.cbrt(ru.astype(np.float64))
        rho = rad * np.sqrt(np.maximum(0.0, 1 - z * z))
        ball = np.stack([rho * np.cos(az), rho * np.sin(az), rad * z], axis=1)
        assert np.abs(q[:, 1:] - ball).max() < 1e-5, d
        assert (np.linalg.norm(q[:, 1:].astype(np.float64), axis=1) <= 1 + 1e-5).all()


# ---- the default variant ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ("small", "medium", "large", "synth4096"))
def test_default_variant(r1, expected, scenes, monkeypatch, name):  # noqa: F811
    """every built-in scene at 1x1x1, 7x3x5, 33x7x3 and a frame (synth4096: 48x27x4, the CPU scan is the slow part)"""
    for w, h, spp in SIZES[:3] + (((48, 27, 4),) if name == "synth4096" else (FRAME,)):
        rgb, _, _ = check(r1, expected, monkeypatch, scenes[name], w, h, spp, what=name)
    assert rgb.any()


def test_resolve_on_a_full_frame(r1, expected, scenes, monkeypatch):  # noqa: F811
    """the resolve (mean, correctly rounded square root, x 255.99, truncation) can only go wrong in a byte where sqrt(mean) x
    255.99 lies within an ulp or so of an integer -- about one value in 10^5, so the small frames above rarely see it.  A
    1280x720 frame at 1 spp resolves 2.8 million distinct sums"""
    rgb, _, _ = check(r1, expected, monkeypatch, scenes["medium"], 1280, 720, 1, mb=2, what="medium full frame")
    assert len(np.unique(rgb)) > 200


@pytest.mark.parametrize("mb", (0, 1, 2))
def test_medium_at_low_depth_caps(r1, expected, scenes, monkeypatch, mb):  # noqa: F811
    check(r1, expected, monkeypatch, scenes["medium"], *FRAME, mb=mb, what="medium")


@pytest.mark.parametrize("seed", (1, 0xFFFFFFFF))
def test_large_at_other_seeds(r1, expected, scenes, monkeypatch, seed):  # noqa: F811
    _, sums, _ = check(r1, expected, monkeypatch, scenes["large"], *FRAME, seed=seed, what="large")
    _, base, _ = scenes["large"].render_sums(*FRAME, MB, 0, 0)
    assert not np.array_equal(sums, base), "the seed must change the render"


# ---- every variant and knob ---------------------------------------------------------------------------------------------------

def variant_runs(r1):
    """name -> (variant, threads, blocks_per_sm, environment)"""
    V = r1
    runs = {"scalar": (V.VARIANT_MEGAKERNEL_SCALAR, 0, 0, {}), "coop": (V.VARIANT_MEGAKERNEL_COOP, 0, 0, {}),
            "deferred": (V.VARIANT_MEGAKERNEL_DEFERRED, 0, 0, {}), "dual768": (V.VARIANT_MEGAKERNEL_DUAL, 768, 0, {}),
            "dual512": (V.VARIANT_MEGAKERNEL_DUAL, 512, 0, {}), "packed": (V.VARIANT_MEGAKERNEL_PACKED, 0, 0, {}),
            "tensor": (V.VARIANT_MEGAKERNEL_TENSOR, 0, 0, {}), "wavefront": (V.VARIANT_WAVEFRONT, 0, 0, {}),
            "pool0": (V.VARIANT_MEGAKERNEL, 0, 0, {"R1_POOL": "0"}), "pool0_coop": (V.VARIANT_MEGAKERNEL_COOP, 0, 0, {"R1_POOL": "0"}),
            "unstaged": (V.VARIANT_MEGAKERNEL, 0, 0, {"R1_FORCE_UNSTAGED": "1"}),
            "unstaged_deferred": (V.VARIANT_MEGAKERNEL_DEFERRED, 0, 0, {"R1_FORCE_UNSTAGED": "1"}),
            "threads512": (V.VARIANT_MEGAKERNEL, 512, 0, {}), "threads768": (V.VARIANT_MEGAKERNEL, 768, 0, {}),
            "blocks2": (V.VARIANT_MEGAKERNEL, 0, 2, {})}
    for g in (1, 2, 3, 4):
        runs["stream%dg" % g] = (V.VARIANT_MEGAKERNEL_TENSOR_STREAM, 128 * g, 0, {})
    for st in (2, 3, 4):
        runs["stream_stages%d" % st] = (V.VARIANT_MEGAKERNEL_TENSOR_STREAM, 512, 0, {"R1_TCS_STAGES": str(st)})
    for g in (4, 5, 6, 7):
        runs["tc3_%dg" % g] = (V.VARIANT_MEGAKERNEL_TENSOR, 0, 0, {"R1_TC3": str(g)})
    return runs


import rays1bench_b200 as _r1mod  # noqa: E402
RUNS = variant_runs(_r1mod)


@pytest.mark.parametrize("run", sorted(RUNS))
@pytest.mark.parametrize("name", ("large", "medium"))
def test_every_variant_and_knob(r1, expected, scenes, monkeypatch, name, run):  # noqa: F811
    v, threads, bps, env = RUNS[run]
    check(r1, expected, monkeypatch, scenes[name], *FRAME, variant=v, threads=threads, blocks_per_sm=bps, env=env, what="%s %s" % (name, run))


# ---- more than 256 samples per pixel --------------------------------------------------------------------------------------------

SPP_VARIANTS = {"default": (0, 0, {}), "packed": (7, 0, {}), "pool0": (0, 0, {"R1_POOL": "0"}), "wavefront": (1, 0, {}), "stream": (9, 0, {})}


@pytest.mark.parametrize("spp", (257, 514, 1000))
@pytest.mark.parametrize("name", ("small", "medium", "large"))
def test_more_than_256_samples_per_pixel(r1, expected, scenes, monkeypatch, name, spp):  # noqa: F811
    """units of ceil(spp / 256) samples (514: a one-sample last unit) on a 5x3 image"""
    for run, (v, threads, env) in SPP_VARIANTS.items():
        check(r1, expected, monkeypatch, scenes[name], 5, 3, spp, variant=v, threads=threads, env=env, what="%s %s" % (name, run))


@pytest.mark.parametrize("spp", (257, 514, 1000))
@pytest.mark.parametrize("name", ("small", "medium", "large"))
def test_lane_fetch_continues_a_pixel_across_units(r1, expected, scenes, monkeypatch, name, spp):  # noqa: F811
    """R1_POOL=0: a lane takes k = min(kmax, left / (lanes x div)) units per fetch and continues a pixel from one unit to the next
    (r1::megakernel, `s_end = min(s + samples_per_unit, spp)`).  k >= 2 needs more than 2 x lanes x div units: 512 threads on every
    SM, div = 1 (R1_SCHED; the large scene's default kmax is 1) and a 40x32 image (>= 154 000 units at 257 spp)"""
    if name == "large" and spp == 1000:
        pytest.skip("1000 = 4 x 250 has no short last unit; covered on small and medium")
    env = {"R1_POOL": "0", "R1_SCHED": "8,1" if name == "large" else "64,1"}
    check(r1, expected, monkeypatch, scenes[name], 40, 32, spp, variant=r1.VARIANT_MEGAKERNEL_PACKED, threads=512, env=env,
          what="%s lane fetch" % name)


# ---- partitions -----------------------------------------------------------------------------------------------------------------

PART_VARIANTS = {"default": 0, "wavefront": 1, "stream": 9}


@pytest.mark.parametrize("run", sorted(PART_VARIANTS))
def test_rank_shares(r1, expected, scenes, monkeypatch, run):  # noqa: F811
    """rank 1 of 3, rank 2 of 3 with 8-row tiles, and a rank without rows each equal the oracle's rows; the ray counts of all
    ranks add up to the whole image's"""
    s, v = scenes["large"], PART_VARIANTS[run]
    w, h, spp = FRAME
    _, _, whole = check(r1, expected, monkeypatch, s, w, h, spp, variant=v, what=run)
    for row_tile in (1, 8):
        total = 0
        for rank in range(3):
            _, _, res = check(r1, expected, monkeypatch, s, w, h, spp, rank=rank, world=3, row_tile=row_tile, variant=v, what=run)
            total += res.num_rays
        assert total == whole.num_rays, (run, row_tile)
    rgb, sums, res = check(r1, expected, monkeypatch, s, w, 10, spp, rank=2, world=3, row_tile=8, variant=v, what=run + " no rows")
    assert rgb.shape[0] == 0 and sums.shape[0] == 0 and res.num_rays == 0


# ---- scenes with edge paths --------------------------------------------------------------------------------------------------

def edge_runs(r1, n):
    runs = [(0, 0, {}), (r1.VARIANT_MEGAKERNEL_PACKED, 0, {}), (r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, 0, {}), (r1.VARIANT_WAVEFRONT, 0, {}),
            (r1.VARIANT_MEGAKERNEL_COOP, 0, {"R1_POOL": "0"})]
    if (n + 31) // 32 * 32 <= 768:
        runs.append((r1.VARIANT_MEGAKERNEL_TENSOR, 0, {}))
    return runs


def test_ties_shade_with_the_lower_index(r1, expected, edge_scenes, monkeypatch):  # noqa: F811
    """exact duplicates with different materials (red Lambertian below, green metal above): every variant shades with the lower
    index, so the frame is the oracle's"""
    s = edge_scenes["ties"]
    for v, threads, env in edge_runs(r1, 200):
        rgb, _, _ = check(r1, expected, monkeypatch, s, 64, 36, 4, variant=v, threads=threads, env=env, what="ties")
    assert rgb.any()


def test_candidate_flood(r1, expected, edge_scenes, monkeypatch):  # noqa: F811
    """96 radius-5 spheres around the unit cube, seen from outside: every ray through the cluster flags nearly every sphere"""
    s = edge_scenes["flood96"]
    for v, threads, env in edge_runs(r1, 96):
        rgb, _, _ = check(r1, expected, monkeypatch, s, 48, 27, 4, variant=v, threads=threads, env=env, what="flood96")
    assert rgb.any()


@pytest.fixture(scope="module")
def inside_flood(r1):
    """24 Lambertian spheres of radius 5 +- 0.05 centred in the unit cube, the camera at the origin inside all of them: every
    path starts inside every sphere and crosses 24 surfaces on its way out"""
    rng = np.random.default_rng(2024)
    spheres = [_f(*rng.uniform(-0.5, 0.5, 3), 5.0 + rng.uniform(-0.05, 0.05)) + (r1.MAT_LAMBERT,) + _f(*rng.uniform(0.75, 0.95, 3), 0)
               for _ in range(24)]
    s = RawScene(_f(0, 0, 0, 0, 0, -1, 70, 0.0, 1), spheres)
    yield s
    s.close()


@pytest.mark.parametrize("mb", (4, MB))
def test_paths_start_inside_spheres_and_reach_the_depth_cap(r1, expected, inside_flood, monkeypatch, mb):
    """at 4 bounces every path reaches the cap: exactly 5 rays per sample and a black frame; at 50 every path gets out"""
    w, h, spp = 48, 27, 4
    for v, threads, env in edge_runs(r1, 24):
        rgb, sums, res = check(r1, expected, monkeypatch, inside_flood, w, h, spp, mb=mb, variant=v, threads=threads, env=env, what="inside flood")
    if mb == 4:
        assert res.num_rays == 5 * w * h * spp and not sums.any()
    else:
        assert (sums > 0).all()


def test_8016_sphere_grid(r1, expected, big_scenes, monkeypatch):  # noqa: F811
    """beyond the staging limit: the default (the packed scan from global memory) and the streamed tensor-core filter"""
    s = big_scenes[8016]
    assert r1.lib.r1_kernel_name(s.handle, 0).decode() == "megakernel_pool"
    for v, threads, env in ((0, 0, {}), (r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, 0, {}), (r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, 256, {}),
                            (r1.VARIANT_MEGAKERNEL_PACKED, 0, {"R1_POOL": "0"})):
        check(r1, expected, monkeypatch, s, 48, 27, 2, variant=v, threads=threads, env=env, what="grid8016")


@pytest.fixture(scope="module")
def fuzz_scene(r1):
    """a fuzz-1 metal sphere filling most of the view over a Lambertian ground: many of its scatters point into the surface
    and end the path black (Metal::scatter returns false)"""
    cam = _f(0, 1, 4, 0, 0.6, 0, 50, 0.05, 4)
    spheres = [_f(0, 0.6, 0, 1.2) + (r1.MAT_METAL,) + _f(0.9, 0.8, 0.7, 1.0), _f(0, -1000, 0, 1000) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0),
               _f(1.8, 0.4, 0.5, 0.4) + (r1.MAT_DIELECTRIC,) + _f(0, 0, 0, 1.5)]
    s = RawScene(cam, spheres)
    yield s
    s.close()


def test_fuzz_1_metal_ends_paths(r1, oracle, expected, fuzz_scene, monkeypatch):
    s = fuzz_scene
    # on the CPU: a fuzz-1 reflection off this sphere often points into it, so scatter returns false
    so = expected.scene(s)
    rng = np.random.default_rng(12)
    n = 2000
    nrm = rng.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    p = np.array([0, 0.6, 0]) + 1.2 * nrm
    din = rng.normal(size=(n, 3))                           # incoming directions uniform over the hemisphere facing the surface
    din /= np.linalg.norm(din, axis=1, keepdims=True)
    din *= -np.sign((din * nrm).sum(axis=1))[:, None]
    ball = rng.normal(size=(n, 3))
    ball *= (rng.uniform(size=(n, 1)) ** (1 / 3)) / np.linalg.norm(ball, axis=1, keepdims=True)
    ok, _, _ = oracle.scatter(so, din.astype(np.float32), p.astype(np.float32), nrm.astype(np.float32), np.zeros(n, np.int32),
                              ball.astype(np.float32), np.zeros(n, np.float32))
    assert 0.05 < 1 - ok.mean() < 0.95
    for v, threads, env in edge_runs(r1, 3):
        rgb, _, _ = check(r1, expected, monkeypatch, s, 64, 36, 8, variant=v, threads=threads, env=env, what="fuzz-1 metal")
    assert rgb.any()


# ---- other surfaces -------------------------------------------------------------------------------------------------------------

def test_render_device_into_torch_buffers(r1, expected, scenes):  # noqa: F811
    torch = pytest.importorskip("torch")
    s = scenes["large"]
    w, h, spp = FRAME
    for rank, world in ((0, 1), (1, 3)):
        n = r1.local_rows(h, 1, rank, world) * w
        d_rgb = torch.zeros(n * 3, dtype=torch.uint8, device="cuda")
        d_rays = torch.full((1,), 12345, dtype=torch.int64, device="cuda")
        stream = torch.cuda.Stream()
        s.render_device(d_rgb.data_ptr(), d_rays.data_ptr(), stream.cuda_stream, width=w, height=h, spp=spp, max_bounces=MB, rank=rank,
                        world=world)
        s.render_wait()
        stream.synchronize()
        want_sums, want_rgb, want_rays = expected.render(s, w, h, spp, MB, 0, rank, world, 1)
        assert np.array_equal(d_rgb.cpu().numpy().reshape(want_rgb.shape), want_rgb), (rank, world)
        assert int(d_rays.item()) == want_rays, (rank, world)


def test_benchmark_after_configure(r1, oracle):
    """the reference-shaped surface: configure() then benchmark() on a fresh scene renders the oracle's frame and ray count"""
    w, h, spp, seed = 64, 36, 4, 5
    own = Expected(r1, oracle)                 # benchmark() frees the scene: its oracle render is not kept past this test
    try:
        r1.configure(width=w, height=h, spp=spp, max_bounces=MB, variant=0, n_gpus=1, seed=seed, quiet=True)
        scene = r1.create_large_scene()
        _, want_rgb, want_rays = own.render(scene, w, h, spp, MB, seed, 0, 1, 1)
        pixels = np.zeros((h, w, 3), np.uint8)
        out = r1.benchmark(scene, pixels, False, "large")
        assert np.array_equal(pixels, want_rgb) and out.num_rays == want_rays
    finally:
        own.close()
        r1.configure(width=1280, height=720, spp=250, max_bounces=MB, variant=0, n_gpus=1, seed=0, quiet=True)
