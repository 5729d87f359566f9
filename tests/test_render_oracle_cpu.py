"""CPU checks of the oracle's restatement of the device integrator (orc_render_keyed and its parts), which
tests/test_render_oracle_gpu.py compares whole renders with: the counter-based generator against a numpy restatement of its
specification, the fixed-point quantiser and the resolve at their edge values, and the integrator itself -- ray counting at
max_bounces 0, the rank partition, and rays per sample against the reference's own measurement."""
import numpy as np
import pytest

F32 = np.float32
M32, M64 = (1 << 32) - 1, (1 << 64) - 1
KEYS = ((0, 0), (M32, (1 << 20) - 1)) + tuple(tuple(int(v) for v in k) for k in np.random.default_rng(31).integers(0, 1 << 32, (8, 2)))
SEEDS = (0, 1, 0xFFFFFFFF)


# ---- numpy restatement of the generator (r1_device.cuh, "RNG") ----------------------------------------------------------------

def mix64(z):
    z = int(z) & M64
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M64
    return z ^ (z >> 31)


def keyed_draws(pixel, sample, seed, idx):
    """draws idx (uint32 array) of stream (pixel, sample) under the global seed, in numpy uint64 arithmetic"""
    z = mix64(((pixel << 32) | sample) ^ mix64(0x9E3779B97F4A7C15 * (seed + 1)))
    k0, k1 = np.uint64(z & M32), np.uint64(z >> 32)
    m = np.uint64(M32)
    x = (k0 + np.uint64(0x9E3779B9) * np.asarray(idx, np.uint64)) & m
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x21f0aaad)) & m
    x ^= k1
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x735a2d97)) & m
    x ^= x >> np.uint64(15)
    return x.astype(np.uint32)


def rand01(draws):
    return (np.asarray(draws, np.uint32) >> 8).astype(F32) * F32(2.0 ** -24)


def rand02(draws):
    return (np.asarray(draws, np.uint32) >> 8).astype(F32) * F32(2.0 ** -23)


# ---- numpy restatement of the quantiser and the resolve -------------------------------------------------------------------

def quantise(c):
    """cvt.rni.sat.u32.f32 of c * 2^24"""
    x = F32(c) * F32(2.0 ** 24)
    if np.isnan(x) or x <= 0:
        return 0
    if x >= F32(M32):
        return M32
    return int(np.rint(x))


def u64_to_f32(n):
    """round to nearest even of an integer to 24 significant bits (no double rounding through float64)"""
    if n.bit_length() <= 24:
        return F32(n)
    shift = n.bit_length() - 24
    q, r = divmod(n, 1 << shift)
    half = 1 << (shift - 1)
    if r > half or (r == half and q & 1):
        q += 1
    return F32(q * 2.0 ** shift)


def resolve(total, spp):
    mean = (u64_to_f32(total) * F32(2.0 ** -24)) * F32(F32(1.0) / F32(spp))
    return int(F32(np.sqrt(mean)) * F32(255.99)) & 0xFF


# ---- generator ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", SEEDS)
def test_keyed_draws_match_the_specification(oracle, seed):
    idx = np.arange(160, dtype=np.uint32)        # primary draws 0..3 and the scatter draws of 52 bounces
    for pixel, sample in KEYS:
        want = keyed_draws(pixel, sample, seed, idx)
        got = np.array([oracle.keyed_draw(pixel, sample, seed, int(i)) for i in idx], np.uint32)
        assert np.array_equal(got, want), (pixel, sample, seed)
    # the key words differ between neighbouring pixels, samples and seeds
    firsts = {int(keyed_draws(p, s, sd, [0])[0]) for p in (0, 1, 2) for s in (0, 1, 2) for sd in SEEDS}
    assert len(firsts) == 27


def test_uniforms_have_24_bits():
    d = np.array([0, 255, 256, 0xFFFFFFFF, 0x80000000], np.uint32)
    assert rand01(d).tolist() == [0.0, 0.0, 2.0 ** -24, 1 - 2.0 ** -24, 0.5]
    assert rand02(d).tolist() == [0.0, 0.0, 2.0 ** -23, 2 - 2.0 ** -23, 1.0]


# ---- fixed point ----------------------------------------------------------------------------------------------------------

QUANTISE_EDGES = (0.0, -0.0, 1.0, 0.5, 2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -25, 5 * 2.0 ** -25, 7 * 2.0 ** -25,      # ties 0.5 .. 3.5
                  (2 ** 22 + 0.5) * 2.0 ** -24, (2 ** 22 + 1.5) * 2.0 ** -24, (2 ** 23 - 0.5) * 2.0 ** -24,          # the largest ties
                  float(np.nextafter(F32(2.0 ** -25), F32(1))), float(np.nextafter(F32(2.0 ** -25), F32(0))),
                  float("nan"), -float("nan"), -1.0, -1e-30, -float("inf"), float("inf"), 255.99, 300.0, 256.0,
                  float(np.nextafter(F32(256), F32(0))), 1e-45, 0.7000000476837158)


def test_quantise_edges(oracle):
    for c in QUANTISE_EDGES:
        assert oracle.quantise_radiance(c) == quantise(c), c
    assert [quantise(c) for c in (2.0 ** -25, 3 * 2.0 ** -25, 5 * 2.0 ** -25, 7 * 2.0 ** -25)] == [0, 2, 2, 4]   # half to even
    assert quantise(float("nan")) == 0 and quantise(-1.0) == 0 and quantise(300.0) == M32
    assert quantise(float(np.nextafter(F32(256), F32(0)))) == 2 ** 32 - 256


RESOLVE_EDGES = (0, 1, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 3 * 2 ** 23, 2 ** 32 - 1, 2 ** 52 - 1, 2 ** 52, 2 ** 52 + 2 ** 28,
                 2 ** 52 + 3 * 2 ** 28, 2 ** 52 + 2 ** 28 + 1, 2 ** 52 + 2 ** 29, 2 ** 60 + 2 ** 36, M64)


@pytest.mark.parametrize("spp", (1, 3, 8, 250, 257, 1000, 1 << 20))
def test_resolve_edges(oracle, spp):
    for total in RESOLVE_EDGES + (spp * (2 ** 24), spp * M32, spp * (2 ** 24) // 4, spp * 9437184):
        assert oracle.resolve(total, spp) == resolve(total, spp), (total, spp)
    assert resolve(spp * 2 ** 24, spp) == 255 and resolve(0, spp) == 0
    # ties of the uint64 -> float conversion: to even, never through a double rounding
    assert u64_to_f32(2 ** 52 + 2 ** 28) == F32(2.0 ** 52) and u64_to_f32(2 ** 52 + 3 * 2 ** 28) == F32(2.0 ** 52 + 2 ** 30)


# ---- the integrator without injected points ----------------------------------------------------------------------------------

def scene_of(oracle, name, w, h):
    return oracle.scene_create(name, w, h)


def test_zero_bounces_trace_one_ray_per_sample(oracle):
    """max_bounces = 0: every sample traces its primary ray only; a pixel is black exactly when all of its primary rays hit"""
    w, h, spp, seed = 32, 18, 4, 7
    so = scene_of(oracle, "small", w, h)
    sums, rgb, rays = oracle.render_keyed(so, w, h, spp, 0, seed)
    assert rays == w * h * spp
    # the primary rays restated here: jitter from draws 0 / 1, the lens disk from draws 2 / 3 in double precision
    cam_u, cam_v, disk, xy = [], [], [], []
    for y in range(h):
        for x in range(w):
            for s in range(spp):
                d = keyed_draws(y * w + x, s, seed, np.arange(4, dtype=np.uint32))
                u01 = rand01(d)
                cam_u.append((u01[0] + F32(x)) * (F32(1) / F32(w)))
                cam_v.append((u01[1] + F32(y)) * (F32(1) / F32(h)))
                r, a = np.sqrt(np.float64(u01[2])), np.float64(rand02(d[3:])[0]) * np.pi
                disk.append((r * np.cos(a), r * np.sin(a)))
    org, dirs = oracle.get_ray(so, np.array(cam_u, F32), np.array(cam_v, F32), np.array(disk, F32))
    idx = oracle.hit(so, org, dirs)[0].reshape(h, w, spp)
    all_hit = (idx >= 0).all(axis=2)
    assert all_hit.any() and not all_hit.all()
    black = (sums == 0).all(axis=2)
    assert np.array_equal(black, all_hit)
    assert not rgb[all_hit].any() and (rgb[~all_hit].max(axis=1) > 0).all()
    oracle.scene_destroy(so)


@pytest.mark.parametrize("row_tile", (1, 8))
def test_rank_shares_assemble_to_the_whole_image(oracle, row_tile):
    """3 ranks (with row_tile 8 on 10 rows, rank 2 owns none): their rows, in ascending global order, are the whole image's"""
    w, h, spp, mb, seed = 24, 10, 4, 50, 3
    so = scene_of(oracle, "medium", 64, 36)
    whole_sums, whole_rgb, whole_rays = oracle.render_keyed(so, w, h, spp, mb, seed)
    rays, rows = 0, []
    sums_at, rgb_at = np.zeros_like(whole_sums), np.zeros_like(whole_rgb)
    for rank in range(3):
        s, c, n = oracle.render_keyed(so, w, h, spp, mb, seed, rank=rank, world=3, row_tile=row_tile)
        ys = [((lr // row_tile) * 3 + rank) * row_tile + lr % row_tile for lr in range(s.shape[0])]
        assert ys == sorted(ys) and all(y < h for y in ys)
        sums_at[ys], rgb_at[ys] = s, c
        rows += ys
        rays += n
        if row_tile == 8 and rank == 2:
            assert s.shape[0] == 0 and n == 0
    assert sorted(rows) == list(range(h))
    assert np.array_equal(sums_at, whole_sums) and np.array_equal(rgb_at, whole_rgb) and rays == whole_rays
    assert whole_rgb.any()
    oracle.scene_destroy(so)


@pytest.mark.parametrize("name", ("small", "medium", "large"))
def test_rays_per_sample_match_the_reference(oracle, ref_stats, name):
    """an independent pin of the restated integrator to the reference: rays per sample at 320x180x8 within 0.5 % of what the
    reference's own render measured (320x180 at 16384 spp)"""
    w, h, spp = 320, 180, 8
    so = scene_of(oracle, name, w, h)
    _, rgb, rays = oracle.render_keyed(so, w, h, spp, 50, 0)
    want = ref_stats["render"][name]["rays_per_sample"]
    got = rays / (w * h * spp)
    assert abs(got / want - 1) < 0.005, (name, got, want)
    assert rgb.any()
    oracle.scene_destroy(so)
