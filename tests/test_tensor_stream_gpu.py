"""The streamed tensor-core filter (R1_VARIANT_MEGAKERNEL_TENSOR_STREAM, r1::megakernel_tcs and r1::trace_rays_tcs_kernel) at
every scene size.

The kernel scans the sphere operand in 128-sphere chunks like megakernel_tc3, but the chunks stream through a ring of
shared-memory stages shared by the CTA's ray groups, so no scene is too large for it.  Ray-level cases go through
trace_rays(variant=tensor_stream), whose kernel fills its stages with the render kernel's device function (tcs_fill): the
addressing of chunk c, the short last chunk, and the exact records that exist (n_pad is padded to 16, n32 to 32).  They are
compared bit for bit (index, t, p, normal) with the oracle's Hitable::hit or with the reference's recorded vectors.  The ring's
multi-group release protocol, and the exit of groups that run out of work, are covered by renders compared byte for byte with
PACKED, with the same ray count, for every supported ray-group count and ring depth, on images small enough to leave CTAs and
groups without work."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_parity import bits, scenes  # noqa: F401  (module fixture: the four built-in scenes)
from test_scan_edges_gpu import (BOUNDARY_SCENES, FLOODS, FLT_MAX, SWEEP, T_BOUND, RawScene, _f, aimed_rays, boundary_queries,  # noqa: F401
                                 boundary_rays, check_against_oracle, edge_scenes, pair_centre, scene_rays)

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene  # noqa: E402

STREAM = ("tensor_stream",)
ALL = ("small", "medium", "large", "synth4096")
# threads of every configuration the render kernel has: 1 .. 4 ray groups (0: the default, 4), each with the 6-stage ring
CONFIGS = (0, 128, 256, 384)
# (width, height, spp, rank, world): a frame, images with fewer samples than one CTA (or one group) has lanes, and a rank
RENDER_CASES = ((96, 54, 8, 0, 1), (7, 3, 5, 0, 1), (1, 1, 3, 0, 1), (96, 54, 8, 1, 3))
# sweep scenes above 768 spheres: n32 mod 128 = 32, 64, 96 and 0
ABOVE_768 = ("n790", "n830", "n860", "n1000")
# exact duplicates across streamed chunk boundaries of a 2 100-sphere scene (17 chunks, the last one 64 columns), incl. the last two
BIG_TIE_COUNT = 2100
BIG_TIE_PAIRS = ((127, 128), (255, 256), (1023, 1024), (2047, 2048), (2098, 2099))


def trace(r1, s, org, d, t_min=0.001, t_max=FLT_MAX):
    return s.trace_rays(org, d, t_min, t_max, variant=r1.VARIANT_MEGAKERNEL_TENSOR_STREAM)


def assert_same(got, want, what):
    bad = np.where(got[0] != want[0])[0]
    assert len(bad) == 0, "%s: %d rays differ, e.g. ray %d: index %d, want %d" % (what, len(bad), bad[0], got[0][bad[0]], want[0][bad[0]])
    for name, a, b in zip(("t", "p", "normal"), got[1:], want[1:]):
        assert np.array_equal(bits(a), bits(b)), "%s: %s differs" % (what, name)


def render_like_packed(r1, s, cases, configs, what):
    for w, h, spp, rank, world in cases:
        base, r0 = s.render(w, h, spp, rank=rank, world=world, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        for threads in configs:
            rgb, res = s.render(w, h, spp, rank=rank, world=world, variant=r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, threads=threads)
            assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays, (what, (w, h, spp, rank, world), threads)


def grid(r1, directory, gw, gh, lookfrom, focus):
    cam, sph = make_scene.grid_scene(gw, gh, 480, lookfrom, focus)
    path = str(directory / ("grid%dx%d.r1scene" % (gw, gh)))
    r1.write_scene_file(path, cam, sph)
    return r1.create_scene_from_file(path)


@pytest.fixture(scope="module")
def big_scenes(r1, tmp_path_factory):
    """beyond the 4096-sphere staging limit: the 5 048-sphere scene of test_scene_above_staging_limit and 8 016 spheres"""
    d = tmp_path_factory.mktemp("big")
    out = {5048: grid(r1, d, 72, 70, (7, 18, 34), 22.0), 8016: grid(r1, d, 90, 89, (9, 22, 42), 27.0)}
    yield out
    for s in out.values():
        s.close()


def grid_rays(soa, n=3000, seed=606):
    """rays from around the grid in every direction and rays grazing random spheres from 5 .. 20 000 units"""
    rng = np.random.default_rng(seed)
    span = float(np.abs(soa["cx"][soa["inv_radius"] > 0.01]).max())
    org = rng.normal(size=(n, 3)) * [0.5 * span, 2, 0.5 * span] + [0, 2, 0]
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    return np.concatenate([org, o2]).astype(np.float32), np.concatenate([d, d2]).astype(np.float32)


# ---- ray level ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALL)
def test_reference_golden_rays(r1, scenes, golden_rays, name):  # noqa: F811
    """the reference's recorded hit() vectors: the same records as PACKED, bit for bit, and the recorded index, t and normal"""
    g = golden_rays[name]
    org = np.concatenate([g["seg_org"], g["edge_org"]])
    d = np.concatenate([g["seg_dir"], g["edge_dir"]])
    got = trace(r1, scenes[name], org, d)
    assert_same(got, scenes[name].trace_rays(org, d, variant=r1.VARIANT_MEGAKERNEL_PACKED), name)
    want_idx = np.concatenate([g["seg_index"], g["edge_index"]])
    assert np.array_equal(got[0], want_idx)
    m = want_idx >= 0
    assert m.sum() > 1000
    assert np.array_equal(bits(got[1][m]), bits(np.concatenate([g["seg_t"], g["edge_t"]])[m]))
    assert np.array_equal(bits(got[3][m]), bits(np.concatenate([g["seg_normal"], g["edge_normal"]])[m]))


@pytest.mark.parametrize("name", ("large", "synth4096"))
def test_dielectric_exit_golden_rays(r1, scenes, golden_rays, name):  # noqa: F811
    """rays leaving the ior >= 5 dielectric spheres from inside: the recorded hit records bit for bit"""
    g = golden_rays[name]
    idx, t, p, n = trace(r1, scenes[name], g["diel_org"], g["diel_dir"])
    assert np.array_equal(idx, g["diel_index"]) and len(idx) >= 200
    assert np.array_equal(bits(t), bits(g["diel_t"])) and np.array_equal(bits(p), bits(g["diel_p"])) and np.array_equal(bits(n), bits(g["diel_normal"]))


@pytest.mark.parametrize("name", ("large", "synth4096"))
def test_fresh_far_and_grazing_rays_match_oracle(r1, scenes, oracle, name):  # noqa: F811
    """rays around the scene and rays grazing spheres (+-2 % of the radius) from 5 .. 20 000 units: the filter stays
    conservative at 4 096 columns; whole range and a t window"""
    soa = scenes[name].soa()
    rng = np.random.default_rng(4321)
    n = 4000
    o1 = (rng.normal(size=(n, 3)) * [8, 2, 8] + [0, 2, 0]).astype(np.float32)
    d1 = rng.normal(size=(n, 3))
    d1 /= np.linalg.norm(d1, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    org, d = np.concatenate([o1, o2]).astype(np.float32), np.concatenate([d1, d2]).astype(np.float32)
    so = oracle.scene_create(name)
    try:
        for t_min, t_max in ((0.001, FLT_MAX), (0.5, 6.0)):
            want = oracle.hit(so, org, d, t_min, t_max)
            assert (want[0] >= 0).sum() > 1500
            assert_same(trace(r1, scenes[name], org, d, t_min, t_max), want, "%s [%g, %g]" % (name, t_min, t_max))
    finally:
        oracle.scene_destroy(so)


def check_scene(r1, oracle, s, name, windows):
    soa = s.soa()
    org, d = scene_rays(name, soa)
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in windows:
            want = oracle.hit(so, org, d, t_min, t_max)
            check_against_oracle(r1, s, want, org, d, t_min, t_max, STREAM, "%s [%g, %g]" % (name, t_min, t_max))
    finally:
        oracle.scene_destroy(so)


@pytest.mark.parametrize("n", SWEEP)
def test_sphere_count_sweep_matches_oracle(r1, oracle, edge_scenes, n):
    """every last-chunk shape (n32 = 32 .. 160 and 1 024), and the unpadded counts 1, 5, 13, 31 and 33"""
    check_scene(r1, oracle, edge_scenes["n%d" % n], "n%d" % n, ((0.001, FLT_MAX), (0.5, 40.0)))


@pytest.mark.parametrize("n", FLOODS)
def test_candidate_floods_match_oracle(r1, oracle, edge_scenes, n):
    """every ray flags (nearly) every sphere, up to 4 096 of them"""
    check_scene(r1, oracle, edge_scenes["flood%d" % n], "flood%d" % n, ((0.001, FLT_MAX), (6.0, 40.0)))


def test_ties_go_to_the_lower_index(r1, oracle, edge_scenes):
    check_scene(r1, oracle, edge_scenes["ties"], "ties", ((0.001, FLT_MAX), (T_BOUND, FLT_MAX), (4.0, 30.0)))


def big_tie_scene():
    """BIG_TIE_COUNT spheres through the raw ABI (no padding: the last pair is the last two spheres): the BIG_TIE_PAIRS as exact
    duplicates (lower: red Lambertian, higher: green metal) in a row, small filler spheres far below"""
    rng = np.random.default_rng(2048)
    red, green = (0,) + _f(0.9, 0.1, 0.1, 0), (1,) + _f(0.1, 0.9, 0.1, 0.0)
    sph = [None] * BIG_TIE_COUNT
    for k, (lo, hi) in enumerate(BIG_TIE_PAIRS):
        sph[lo] = _f(*pair_centre(k), 1.0) + red
        sph[hi] = _f(*pair_centre(k), 1.0) + green
    for i in range(BIG_TIE_COUNT):
        if sph[i] is None:
            x, z = rng.integers(-60, 61, 2)
            sph[i] = _f(x, -30, z, 0.25) + (0,) + _f(*rng.uniform(0.1, 0.9, 3), 0)
    return RawScene(_f(0, 14, 24, 0, 1, 0, 55, 0.0, 24), sph)


def test_ties_across_streamed_chunk_boundaries(r1, oracle):
    """exact duplicates at (127, 128), (255, 256), (1023, 1024), (2047, 2048) and the last two spheres: the lower index wins,
    whether the two sit in one chunk or in chunks that pass through different stages"""
    s = big_tie_scene()
    try:
        assert s.count() == BIG_TIE_COUNT
        soa = s.soa()
        rng = np.random.default_rng(17)
        lows = np.repeat([lo for lo, _ in BIG_TIE_PAIRS], 200)
        org, d = aimed_rays(soa, lows, rng, rng.uniform(5.0, 200.0, len(lows)))
        tan_o, tan_d = [], []                                    # tangent rays: discr = +0, root t = L for both duplicates
        for k in range(len(BIG_TIE_PAIRS)):
            c = np.array(pair_centre(k))
            for L in (3.0, 5.0, 7.0):
                tan_o += [c + (1, 0, -L), c + (0, 1, -L)]
                tan_d += [(0, 0, 1), (0, 0, 1)]
        org = np.concatenate([org, tan_o]).astype(np.float32)
        d = np.concatenate([d, tan_d]).astype(np.float32)
        so = oracle.scene_create_from_soa(soa)
        try:
            for t_min in (0.001, T_BOUND):
                want = oracle.hit(so, org, d, t_min)
                for lo, hi in BIG_TIE_PAIRS:
                    assert (want[0] == lo).sum() > 50 and not (want[0] == hi).any()
                check_against_oracle(r1, s, want, org, d, t_min, FLT_MAX, STREAM, "big ties, t_min %g" % t_min)
        finally:
            oracle.scene_destroy(so)
    finally:
        s.close()


@pytest.mark.parametrize("name", BOUNDARY_SCENES)
@pytest.mark.parametrize("t_min", (0.001, T_BOUND), ids=("tmin_0.001", "tmin_2^-24"))
def test_root_boundaries_match_oracle(r1, oracle, edge_scenes, name, t_min):
    """per hit ray, t_max = t / t + ulp and t_min = t / t - ulp"""
    s = edge_scenes[name]
    soa = s.soa()
    so = oracle.scene_create_from_soa(soa)
    try:
        org, d, t = boundary_rays(name, soa, so, oracle, t_min)
        assert len(org) >= 40
        for k in range(len(org)):
            for lo, hi in boundary_queries(t_min, t[k]):
                want = oracle.hit(so, org[k:k + 1], d[k:k + 1], lo, hi)
                check_against_oracle(r1, s, want, org[k:k + 1], d[k:k + 1], lo, hi, STREAM, "%s ray %d [%r, %r]" % (name, k, lo, hi))
    finally:
        oracle.scene_destroy(so)


@pytest.mark.parametrize("count", (5048, 8016))
def test_scenes_beyond_staging_match_oracle(r1, oracle, big_scenes, count):
    """above 4 096 spheres only the streamed filter's ray kernel answers; every other variant refuses"""
    s = big_scenes[count]
    assert s.count() == count
    soa = s.soa()
    org, d = grid_rays(soa)
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in ((0.001, FLT_MAX), (0.5, 6.0)):
            want = oracle.hit(so, org, d, t_min, t_max)
            assert (want[0] >= 0).sum() > 1500 and (want[0] >= 4096).sum() > 100
            assert_same(trace(r1, s, org, d, t_min, t_max), want, "%d spheres [%g, %g]" % (count, t_min, t_max))
    finally:
        oracle.scene_destroy(so)
    for v in ("mega", "packed", "scalar", "coop", "deferred"):
        with pytest.raises(r1.Rays1Error, match=r"\(-4\).*stages at most"):
            s.trace_rays(org[:1], d[:1], variant=r1.VARIANTS[v])
    with pytest.raises(r1.Rays1Error, match=r"\(-4\).*768"):
        s.trace_rays(org[:1], d[:1], variant=r1.VARIANT_MEGAKERNEL_TENSOR)


# ---- renders ----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALL)
def test_builtin_scenes_render_like_packed(r1, scenes, name):  # noqa: F811
    render_like_packed(r1, scenes[name], RENDER_CASES, CONFIGS, name)


@pytest.mark.parametrize("name", ABOVE_768 + ("flood4096",))
def test_scenes_above_768_spheres_render_like_packed(r1, edge_scenes, name):
    s = edge_scenes[name]
    n32 = (s.count() + 31) // 32 * 32
    assert n32 > 768
    cases = RENDER_CASES if not name.startswith("flood") else ((48, 27, 4, 0, 1), (7, 3, 5, 0, 1))
    render_like_packed(r1, s, cases, CONFIGS, name)


def test_above_768_sweep_covers_every_last_chunk(edge_scenes):
    assert sorted((edge_scenes[n].count() + 31) // 32 * 32 % 128 for n in ABOVE_768) == [0, 32, 64, 96]


@pytest.mark.parametrize("count", (5048, 8016))
def test_scenes_beyond_staging_render_like_packed(r1, big_scenes, count):
    render_like_packed(r1, big_scenes[count], RENDER_CASES[:2] + RENDER_CASES[3:], (0, 128), count)


def test_full_size_synth4096_renders_like_packed(r1, scenes):  # noqa: F811
    s = scenes["synth4096"]
    base, r0 = s.render(1280, 720, 250, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    rgb, res = s.render(1280, 720, 250, variant=r1.VARIANT_MEGAKERNEL_TENSOR_STREAM)
    assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
    print("synth4096 1280x720x250: packed %.1f ms, tensor_stream %.1f ms (trace)" % (r0.trace_ms, res.trace_ms))


def test_unsupported_configurations_are_refused(r1, scenes):  # noqa: F811
    s = scenes["large"]
    for threads in (640, 1024):
        with pytest.raises(r1.Rays1Error, match=r"\(-1\).*tensor-stream"):
            s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_TENSOR_STREAM, threads=threads)
    base, r0 = s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    rgb, res = s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_TENSOR_STREAM)   # no sticky error
    assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays


# ---- names and the executable -------------------------------------------------------------------------------------------------

def test_kernel_name(r1, scenes, big_scenes):  # noqa: F811
    for s in list(scenes.values()) + list(big_scenes.values()):
        assert r1.lib.r1_kernel_name(s.handle, r1.VARIANT_MEGAKERNEL_TENSOR_STREAM).decode() == "megakernel_tcs"


def test_executable_variant_flag(r1, tmp_path):
    common = ["-w", "--scene", "synth4096", "--spp", "4", "--width", "320", "--height", "180"]
    out = {}
    for v in ("packed", "tensor-stream"):
        d = tmp_path / v
        d.mkdir()
        run = subprocess.run([r1.EXE_PATH, "--variant", v] + common, cwd=d, capture_output=True, text=True, timeout=300)
        assert run.returncode == 0, run.stderr
        out[v] = (open(d / "out_synth4096.tga", "rb").read(), open(d / "out_synth4096.txt").read().split("|")[2])
    assert out["packed"] == out["tensor-stream"]
