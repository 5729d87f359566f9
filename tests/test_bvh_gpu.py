"""The BVH variant (R1_VARIANT_MEGAKERNEL_BVH: r1::megakernel_pool<kScanBvh> and r1::trace_rays_bvh_kernel) against the brute-force
scan.

Ray-level cases go through trace_rays(variant=bvh), whose kernel runs the render kernel's traversal (bvh_trace), and are compared
bit for bit (index, t, p, normal) with the oracle's Hitable::hit or the reference's recorded vectors: the built-in scenes, the
sweep, flood, tie and root-boundary fixtures of test_scan_edges_gpu, the 5 048- and 8 016-sphere grids and a 100 000-sphere
cloud.  Renders are compared byte for byte with PACKED, with the same ray count, for every thread count the variant builds."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_parity import bits, scenes  # noqa: F401  (module fixture: the four built-in scenes)
from test_scan_edges_gpu import (BOUNDARY_SCENES, FLOODS, FLT_MAX, RENDER_SCENES, SWEEP, T_BOUND, aimed_rays,  # noqa: F401
                                 boundary_queries, boundary_rays, check_against_oracle, edge_scenes, scene_rays)
from test_render_oracle_gpu import check, expected  # noqa: F401
from test_tensor_stream_gpu import assert_same, big_scenes, grid_rays  # noqa: F401

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene  # noqa: E402

BVH = ("bvh",)
ALL = ("small", "medium", "large", "synth4096")
THREADS = (0, 512, 768, 1024)
RENDER_CASES = ((96, 54, 8, 0, 1), (7, 3, 5, 0, 1), (1, 1, 3, 0, 1), (96, 54, 8, 1, 3))


def trace(r1, s, org, d, t_min=0.001, t_max=FLT_MAX):
    return s.trace_rays(org, d, t_min, t_max, variant=r1.VARIANT_MEGAKERNEL_BVH)


def render_like_packed(r1, s, cases, threads, what):
    for w, h, spp, rank, world in cases:
        base, r0 = s.render(w, h, spp, rank=rank, world=world, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        for th in threads:
            rgb, res = s.render(w, h, spp, rank=rank, world=world, variant=r1.VARIANT_MEGAKERNEL_BVH, threads=th)
            assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays, (what, (w, h, spp, rank, world), th)


@pytest.fixture(scope="module")
def cloud(r1, tmp_path_factory):
    cam, sph = make_scene.cloud_scene(100000, seed=5)
    path = str(tmp_path_factory.mktemp("cloud") / "cloud.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path)
    yield s
    s.close()


# ---- ray level ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALL)
def test_reference_golden_rays(r1, scenes, golden_rays, name):  # noqa: F811
    g = golden_rays[name]
    org = np.concatenate([g["seg_org"], g["edge_org"]])
    d = np.concatenate([g["seg_dir"], g["edge_dir"]])
    got = trace(r1, scenes[name], org, d)
    assert_same(got, scenes[name].trace_rays(org, d, variant=r1.VARIANT_MEGAKERNEL_PACKED), name)
    want_idx = np.concatenate([g["seg_index"], g["edge_index"]])
    assert np.array_equal(got[0], want_idx)
    m = want_idx >= 0
    assert np.array_equal(bits(got[1][m]), bits(np.concatenate([g["seg_t"], g["edge_t"]])[m]))
    assert np.array_equal(bits(got[3][m]), bits(np.concatenate([g["seg_normal"], g["edge_normal"]])[m]))


@pytest.mark.parametrize("name", ("large", "synth4096"))
def test_dielectric_exit_golden_rays(r1, scenes, golden_rays, name):  # noqa: F811
    g = golden_rays[name]
    idx, t, p, n = trace(r1, scenes[name], g["diel_org"], g["diel_dir"])
    assert np.array_equal(idx, g["diel_index"]) and len(idx) >= 200
    assert np.array_equal(bits(t), bits(g["diel_t"])) and np.array_equal(bits(p), bits(g["diel_p"])) and np.array_equal(bits(n), bits(g["diel_normal"]))


@pytest.mark.parametrize("name", ALL)
def test_fresh_far_and_grazing_rays_match_oracle(r1, scenes, oracle, name):  # noqa: F811
    soa = scenes[name].soa()
    rng = np.random.default_rng(4321)
    n = 4000
    o1 = (rng.normal(size=(n, 3)) * [8, 2, 8] + [0, 2, 0]).astype(np.float32)
    d1 = rng.normal(size=(n, 3))
    d1 /= np.linalg.norm(d1, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    d3 = np.zeros((300, 3))
    d3[np.arange(300), rng.integers(0, 3, 300)] = rng.choice([-1.0, 1.0], 300)   # axis-aligned: +-0 components
    o3 = o1[:300]
    org = np.concatenate([o1, o2, o3]).astype(np.float32)
    d = np.concatenate([d1, d2, d3]).astype(np.float32)
    so = oracle.scene_create(name)
    try:
        for t_min, t_max in ((0.001, FLT_MAX), (0.5, 6.0), (T_BOUND, FLT_MAX)):
            want = oracle.hit(so, org, d, t_min, t_max)
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
            check_against_oracle(r1, s, want, org, d, t_min, t_max, BVH, "%s [%g, %g]" % (name, t_min, t_max))
    finally:
        oracle.scene_destroy(so)


@pytest.mark.parametrize("n", SWEEP)
def test_sphere_count_sweep_matches_oracle(r1, oracle, edge_scenes, n):
    check_scene(r1, oracle, edge_scenes["n%d" % n], "n%d" % n, ((0.001, FLT_MAX), (0.5, 40.0)))


@pytest.mark.parametrize("n", FLOODS)
def test_candidate_floods_match_oracle(r1, oracle, edge_scenes, n):
    check_scene(r1, oracle, edge_scenes["flood%d" % n], "flood%d" % n, ((0.001, FLT_MAX), (6.0, 40.0)))


def test_ties_go_to_the_lower_index(r1, oracle, edge_scenes):
    check_scene(r1, oracle, edge_scenes["ties"], "ties", ((0.001, FLT_MAX), (T_BOUND, FLT_MAX), (4.0, 30.0)))


@pytest.mark.parametrize("name", BOUNDARY_SCENES)
@pytest.mark.parametrize("t_min", (0.001, T_BOUND), ids=("tmin_0.001", "tmin_2^-24"))
def test_root_boundaries_match_oracle(r1, oracle, edge_scenes, name, t_min):
    s = edge_scenes[name]
    soa = s.soa()
    so = oracle.scene_create_from_soa(soa)
    try:
        org, d, t = boundary_rays(name, soa, so, oracle, t_min)
        assert len(org) >= 40
        for k in range(len(org)):
            for lo, hi in boundary_queries(t_min, t[k]):
                want = oracle.hit(so, org[k:k + 1], d[k:k + 1], lo, hi)
                check_against_oracle(r1, s, want, org[k:k + 1], d[k:k + 1], lo, hi, BVH, "%s ray %d [%r, %r]" % (name, k, lo, hi))
    finally:
        oracle.scene_destroy(so)


@pytest.mark.parametrize("count", (5048, 8016))
def test_scenes_beyond_staging_match_oracle(r1, oracle, big_scenes, count):  # noqa: F811
    s = big_scenes[count]
    soa = s.soa()
    org, d = grid_rays(soa)
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in ((0.001, FLT_MAX), (0.5, 6.0)):
            want = oracle.hit(so, org, d, t_min, t_max)
            assert (want[0] >= 4096).sum() > 100
            assert_same(trace(r1, s, org, d, t_min, t_max), want, "%d spheres [%g, %g]" % (count, t_min, t_max))
    finally:
        oracle.scene_destroy(so)


def test_cloud_matches_oracle(r1, oracle, cloud):
    """100 000 overlapping spheres: rays around and through the cloud, rays grazing spheres from 5 .. 20 000 units"""
    soa = cloud.soa()
    rng = np.random.default_rng(31)
    n = 2000
    span = float(np.abs(soa["cx"][:-8]).max())
    o1 = (rng.uniform(-1.2 * span, 1.2 * span, (n, 3)) + [0, span, 0]).astype(np.float32)
    d1 = rng.normal(size=(n, 3))
    d1 /= np.linalg.norm(d1, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    org, d = np.concatenate([o1, o2]).astype(np.float32), np.concatenate([d1, d2]).astype(np.float32)
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in ((0.001, FLT_MAX), (0.5, 40.0)):
            want = oracle.hit(so, org, d, t_min, t_max)
            assert (want[0] >= 0).sum() > 1500
            assert_same(trace(r1, cloud, org, d, t_min, t_max), want, "cloud [%g, %g]" % (t_min, t_max))
    finally:
        oracle.scene_destroy(so)


# ---- renders ----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALL)
def test_builtin_scenes_render_like_packed(r1, scenes, name):  # noqa: F811
    render_like_packed(r1, scenes[name], RENDER_CASES, THREADS, name)


@pytest.mark.parametrize("name", RENDER_SCENES)
def test_edge_scenes_render_like_packed(r1, edge_scenes, name):
    cases = ((48, 27, 4, 0, 1), (7, 3, 5, 0, 1), (48, 27, 4, 1, 3))
    render_like_packed(r1, edge_scenes[name], cases, (0, 1024), name)


@pytest.mark.parametrize("count", (5048, 8016))
def test_scenes_beyond_staging_render_like_packed(r1, big_scenes, count):  # noqa: F811
    render_like_packed(r1, big_scenes[count], RENDER_CASES[:2] + RENDER_CASES[3:], (0,), count)


def test_full_size_synth4096_renders_like_packed(r1, scenes):  # noqa: F811
    s = scenes["synth4096"]
    base, r0 = s.render(1280, 720, 250, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    rgb, res = s.render(1280, 720, 250, variant=r1.VARIANT_MEGAKERNEL_BVH)
    assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
    print("synth4096 1280x720x250: packed %.1f ms, bvh %.1f ms (trace)" % (r0.trace_ms, res.trace_ms))


def test_render_sums_match_the_oracle(r1, expected, monkeypatch, scenes):  # noqa: F811
    """the fixed-point pixel sums, bytes and ray count of a BVH render equal the CPU restatement of the integrator (render_keyed)"""
    check(r1, expected, monkeypatch, scenes["large"], 40, 24, 3, variant=r1.VARIANT_MEGAKERNEL_BVH, what="large")
    check(r1, expected, monkeypatch, scenes["medium"], 24, 14, 2, rank=1, world=3, variant=r1.VARIANT_MEGAKERNEL_BVH, threads=1024, what="medium")


def test_multi_gpu_in_process_equals_one_gpu(r1, tmp_path):
    if r1.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = {}
    for n in (1, 2):
        r1.configure(width=96, height=54, spp=8, max_bounces=50, variant=r1.VARIANT_MEGAKERNEL_BVH, n_gpus=n, seed=0, quiet=True)
        s = r1.create_scene("large")
        pix = np.zeros((54, 96, 3), np.uint8)
        res = r1.benchmark(s, pix, False, "large")
        out[n] = (pix.copy(), res.num_rays)
    r1.configure(width=1280, height=720, spp=250, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    assert np.array_equal(out[1][0], out[2][0]) and out[1][1] == out[2][1]


# ---- names, first-use upload, refusals, the executable ---------------------------------------------------------------------

def test_kernel_name_and_first_use_upload(r1, tmp_path):
    s = r1.create_scene("large")
    assert r1.lib.r1_kernel_name(s.handle, r1.VARIANT_MEGAKERNEL_BVH).decode() == "megakernel_bvh"
    first, r0 = s.render(64, 36, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)      # builds and uploads the tree
    again, r1_ = s.render(64, 36, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)
    assert np.array_equal(first, again) and r0.num_rays == r1_.num_rays
    s.close()


def test_changed_spheres_need_a_new_commit(r1):
    from test_scan_edges_gpu import RawScene, _f
    sph = [_f(0, 0, 0, 1) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), _f(0, -1001, 0, 1000) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0)]
    s = RawScene(_f(0, 1, 10, 0, 0, 0, 40, 0, 10), sph)
    try:
        r1._check(r1.lib.r1_scene_add_sphere(s.handle, 2, 0, 0, 1, r1.MAT_METAL, 0.5, 0.5, 0.5, 0), "add")
        with pytest.raises(r1.Rays1Error, match=r"\(-2\).*commit it again"):
            s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_BVH)
        r1._check(r1.lib.r1_scene_commit(s.handle, 0), "commit")
        base, r0 = s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        rgb, res = s.render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_BVH)
        assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
    finally:
        s.close()


def test_unsupported_thread_counts_are_refused(r1, scenes):  # noqa: F811
    with pytest.raises(r1.Rays1Error, match=r"\(-1\).*bvh"):
        scenes["large"].render(16, 9, 2, variant=r1.VARIANT_MEGAKERNEL_BVH, threads=640)


def test_executable_variant_flag(r1, tmp_path):
    common = ["-w", "--scene", "synth4096", "--spp", "4", "--width", "320", "--height", "180"]
    out = {}
    for v in ("packed", "bvh"):
        d = tmp_path / v
        d.mkdir()
        run = subprocess.run([r1.EXE_PATH, "--variant", v] + common, cwd=d, capture_output=True, text=True, timeout=300)
        assert run.returncode == 0, run.stderr
        out[v] = (open(d / "out_synth4096.tga", "rb").read(), open(d / "out_synth4096.txt").read().split("|")[2])
    assert out["packed"] == out["bvh"]
