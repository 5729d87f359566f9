"""The float64 expectation of tests/estimator_reference.py, checked where no GPU is needed: its closed forms against scipy, the
model against the oracle's libm mode (orc_render_keyed without injected points) on every case, and the draws a path consumes
together against independence (2-D chi^2 on their top bits).  tests/test_estimator_gpu.py then holds the renderer to the same
model."""
import numpy as np
import pytest

import estimator_reference as er
from test_render_oracle_cpu import M32, M64, keyed_draws
from test_scan_edges_gpu import RawScene, _f

FRAME = (8, 6)
SPP = 1 << 16


def spheres_of(spec):
    return [_f(*c[:4]) + (c[4],) + _f(*c[5:]) for c in spec]


# ---- closed forms ---------------------------------------------------------------------------------------------------------------

def _ball_expectation(g):
    """E[g(rho, c)] for u = rho (.., c) uniform in the unit ball: density 3 rho^2 in rho, c uniform in [-1, 1]"""
    from scipy.integrate import dblquad
    return dblquad(lambda c, rho: 1.5 * rho * rho * g(rho, c), 0, 1, -1, 1, epsabs=1e-14, epsrel=1e-13)[0]


def test_lambertian_closed_forms_against_scipy():
    """unit(n + u): E[cos] = 4/5 and E[cos^2] = 2/3, so E[w_y^2] = 2/3 n_y^2 + 1/6 (1 - n_y^2)"""
    cos = lambda rho, c: (1 + rho * c) / np.sqrt(1 + 2 * rho * c + rho * rho)  # noqa: E731
    assert abs(_ball_expectation(cos) - er.KAPPA_LAMBERT) < 1e-13
    assert abs(_ball_expectation(lambda rho, c: cos(rho, c) ** 2) - er.COS2_LAMBERT) < 1e-13
    # the model's 2-D quadrature at fuzz 1 is the Lambertian law: it converges towards the closed forms
    k, lam = er.fuzz_moments(1.0, 400)
    assert abs(k - 0.8) < 1e-6 and abs(lam - 2 / 3) < 1e-6


@pytest.mark.parametrize("f", (0.1, 0.3, 0.6))
def test_fuzz_moments_against_scipy(f):
    n2 = lambda rho, c: 1 + 2 * f * rho * c + (f * rho) ** 2  # noqa: E731
    k, lam = er.fuzz_moments(f)
    assert abs(k - _ball_expectation(lambda rho, c: (1 + f * rho * c) / np.sqrt(n2(rho, c)))) < 1e-13
    assert abs(lam - _ball_expectation(lambda rho, c: (1 + f * rho * c) ** 2 / n2(rho, c))) < 1e-13


# ---- the model against the oracle's libm mode ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def libm_renders(oracle):
    """case -> (model, sums, rays) of an 8x6 frame at 2^16 spp"""
    out = {}
    w, h = FRAME
    for name, (cam, spec, mb) in er.CASES.items():
        s = RawScene(_f(*cam), spheres_of(spec), commit=False)
        soa, cam22 = s.soa(), s.camera()
        s.close()
        so = oracle.scene_create_from_soa(soa)
        oracle.scene_set_camera(so, cam22)
        sums, _, rays = oracle.render_keyed(so, w, h, SPP, mb, 0)
        oracle.scene_destroy(so)
        out[name] = (er.expectation(cam22, soa, w, h, mb), sums, rays)
    return out


@pytest.mark.parametrize("name", sorted(er.CASES))
def test_model_matches_the_oracle_libm_mode(libm_renders, name):
    model, sums, rays = libm_renders[name]
    st = er.converge_stats(model, sums, rays, SPP, name, deterministic_rays=er.CASES[name][1][0][4] != er.MAT_DIELECTRIC)
    print("libm %-12s %s" % (name, st))


def test_the_cases_reach_what_they_are_for(libm_renders):
    """the sky's d_y varies strongly; the wide lens matters; the cap carries mass at ior 24.2"""
    pin, lens = libm_renders["sky_pinhole"][0], libm_renders["sky_lens"][0]
    assert np.ptp(pin["mean"][..., 0]) > 0.2 and np.ptp(lens["mean"][..., 0]) > 0.1
    mb1 = libm_renders["ior24_mb1"][0]
    assert 0.1 < 1 - mb1["mean"][..., 2].mean() < 0.2, "at one bounce the refracted share of the paths ends black"
    glass = libm_renders["glass"][0]
    assert 2.9 < glass["rays"].mean() < 3.1


# ---- the draws a path consumes together ----------------------------------------------------------------------------------------

def mix64(z):
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    return z ^ (z >> np.uint64(31))


def stream_keys(pixel, sample, seed):
    """vectorised (k0, k1) of streams (pixel, sample) under the global seed"""
    with np.errstate(over="ignore"):
        mix = mix64(np.uint64((0x9E3779B97F4A7C15 * (seed + 1)) & M64))
        z = mix64(((np.asarray(pixel, np.uint64) << np.uint64(32)) | np.asarray(sample, np.uint64)) ^ mix)
    return z & np.uint64(M32), z >> np.uint64(32)


def draws(k0, k1, i):
    m = np.uint64(M32)
    x = (k0 + np.uint64((0x9E3779B9 * i) & M32)) & m
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x21f0aaad)) & m
    x ^= k1
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x735a2d97)) & m
    x ^= x >> np.uint64(15)
    return x.astype(np.uint32)


def test_vectorised_generator_matches_the_specification():
    rng = np.random.default_rng(5)
    pixel, sample = rng.integers(0, 1 << 32, 64, dtype=np.uint64), rng.integers(0, 1 << 32, 64, dtype=np.uint64)
    for seed in (0, 1, 0xFFFFFFFF):
        k0, k1 = stream_keys(pixel, sample, seed)
        got = np.stack([draws(k0, k1, i) for i in range(160)], axis=1)
        want = np.stack([keyed_draws(int(p), int(s), seed, np.arange(160, dtype=np.uint32)) for p, s in zip(pixel, sample)])
        assert np.array_equal(got, want), seed


BITS = 4                                          # top bits of each draw: 16 x 16 cells
KEY_SIDE = 1 << 12                                # pixels 0 .. 4095 x samples 0 .. 4095: 2^24 streams
# (what, (pixel offset, sample offset, draw) of the first, of the second): draws 0 / 1 jitter, 2 / 3 lens, 4 + 3 d .. 6 + 3 d the
# scatter of depth d (ru, ball z, ball azimuth)
PAIRS = (("jitter x / y", (0, 0, 0), (0, 0, 1)), ("lens radius / angle", (0, 0, 2), (0, 0, 3)),
         ("jitter x / lens radius", (0, 0, 0), (0, 0, 2)), ("jitter y / lens angle", (0, 0, 1), (0, 0, 3)),
         ("depth 0 ru / z", (0, 0, 4), (0, 0, 5)), ("depth 0 z / azimuth", (0, 0, 5), (0, 0, 6)),
         ("depth 5 ru / azimuth", (0, 0, 19), (0, 0, 21)), ("depth 0 / 1 ru", (0, 0, 4), (0, 0, 7)),
         ("depth 0 azimuth / 1 ru", (0, 0, 6), (0, 0, 7)), ("adjacent samples, draw 0", (0, 0, 0), (0, 1, 0)),
         ("adjacent samples, draw 4", (0, 0, 4), (0, 1, 4)), ("adjacent pixels, draw 0", (0, 0, 0), (1, 0, 0)),
         ("adjacent pixels, draw 2", (0, 0, 2), (1, 0, 2)))


@pytest.fixture(scope="module")
def battery_keys():
    p, s = np.meshgrid(np.arange(KEY_SIDE, dtype=np.uint64), np.arange(KEY_SIDE, dtype=np.uint64), indexing="ij")
    p, s = p.ravel(), s.ravel()
    return {(dp, ds): stream_keys(p + np.uint64(dp), s + np.uint64(ds), 0) for dp, ds in ((0, 0), (0, 1), (1, 0))}


@pytest.mark.parametrize("pair", [p[0] for p in PAIRS])
def test_draws_consumed_together_are_independent(battery_keys, pair):
    _, (p0, s0, i0), (p1, s1, i1) = next(p for p in PAIRS if p[0] == pair)
    a = draws(*battery_keys[(p0, s0)], i0) >> np.uint32(32 - BITS)
    b = draws(*battery_keys[(p1, s1)], i1) >> np.uint32(32 - BITS)
    counts = np.bincount((a.astype(np.int64) << BITS) | b, minlength=1 << (2 * BITS))
    want = len(a) / counts.size
    chi2 = float(((counts - want) ** 2 / want).sum())
    dof = counts.size - 1
    z = (chi2 - dof) / np.sqrt(2 * dof)
    print("battery %-26s chi2 %.1f / %d  z %.2f" % (pair, chi2, dof, z))
    assert abs(z) < 4, (pair, chi2, z)
