"""The device BVH builder (r1_scene_build_bvh with R1_BVH_BUILD_DEVICE, r1_bvh_device.cu) on the GPU.

The tree the device builds equals the CPU restatement (tests/lbvh_restatement.py) byte for byte, on every scene below; a HOST
build puts the host tree there unchanged.  This module owns its scenes and gives every one of them the device tree before its
first test, so the ray-level and render cases of test_bvh_gpu, imported here, run the traversal over the device tree; after every
test each scene must still hold it.  Also: the 10^6-sphere cloud, refusals, and what a re-commit does to a device's tree."""
import os
import sys

import numpy as np
import pytest

import lbvh_restatement as lbvh
from conftest import ROOT
from test_bvh_cpu import EDGE, check_structure
from test_bvh_device_cpu import CAM, MAX_DEPTH, SPECIAL, special_spheres
from test_bvh_gpu import (ALL, cloud, render_like_packed, trace, RENDER_CASES, THREADS,  # noqa: F401
                          test_builtin_scenes_render_like_packed, test_candidate_floods_match_oracle, test_cloud_matches_oracle,
                          test_dielectric_exit_golden_rays, test_edge_scenes_render_like_packed, test_fresh_far_and_grazing_rays_match_oracle,
                          test_full_size_synth4096_renders_like_packed, test_reference_golden_rays, test_render_sums_match_the_oracle,
                          test_root_boundaries_match_oracle, test_scenes_beyond_staging_match_oracle,
                          test_scenes_beyond_staging_render_like_packed, test_sphere_count_sweep_matches_oracle, test_ties_go_to_the_lower_index)
from test_gpu_parity import scenes  # noqa: F401
from test_render_oracle_gpu import expected  # noqa: F401
from test_scan_edges_gpu import FLT_MAX, RawScene, _f, edge_scenes  # noqa: F401
from test_tensor_stream_gpu import assert_same, big_scenes  # noqa: F401

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene  # noqa: E402

TREE_SCENES = ALL + EDGE + ("grid5048", "grid8016", "cloud") + SPECIAL


@pytest.fixture(scope="module")
def special_scenes(r1):
    out = {name: RawScene(CAM, special_spheres(r1, name)) for name in SPECIAL}
    yield out
    for s in out.values():
        s.close()


def tree_bytes(tree):
    nodes, leaves, depth = tree
    return nodes.tobytes(), leaves.tobytes(), depth


@pytest.fixture(scope="module")
def device_trees(r1, scenes, edge_scenes, big_scenes, cloud, special_scenes):  # noqa: F811
    """name -> (scene, restated tree, device build time in ms): every scene of the module, holding its device tree"""
    by_name = dict(scenes)
    by_name.update({name: edge_scenes[name] for name in EDGE})
    by_name.update({"grid5048": big_scenes[5048], "grid8016": big_scenes[8016], "cloud": cloud})
    by_name.update(special_scenes)
    out = {}
    for name, s in by_name.items():
        ms = s.build_bvh(r1.BVH_BUILD_DEVICE)
        out[name] = (s, tree_bytes(lbvh.build(s.soa())), ms)
    return out


@pytest.fixture(autouse=True)
def still_on_the_device_tree(request):
    """after every test that uses the module's scenes: each still holds its device tree"""
    yield
    if "device_trees" in request.fixturenames or any(f in request.fixturenames for f in ("scenes", "edge_scenes", "big_scenes", "cloud")):
        for name, (s, want, _) in request.getfixturevalue("device_trees").items():
            assert tree_bytes(s.bvh_on_device()) == want, "%s no longer holds its device tree" % name


@pytest.fixture(autouse=True)
def _trees_first(request):
    """the module's scenes get their device trees before any test touches them"""
    if any(f in request.fixturenames for f in ("scenes", "edge_scenes", "big_scenes", "cloud")):
        request.getfixturevalue("device_trees")


# ---- the tree ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", TREE_SCENES)
def test_device_tree_equals_the_restatement(device_trees, name):
    s, want, ms = device_trees[name]
    got = s.bvh_on_device()
    assert got[2] == want[2] and got[2] <= MAX_DEPTH
    assert got[0].tobytes() == want[0], "%s: nodes differ from the restatement" % name
    assert got[1].tobytes() == want[1], "%s: leaf records differ from the restatement" % name
    check_structure(s, *got)
    assert ms > 0


@pytest.mark.parametrize("name", ("large", "cloud", "coincident_radii", "real0", "real5"))
def test_two_builds_give_the_same_bytes(r1, device_trees, name):
    s, want, _ = device_trees[name]
    s.build_bvh(r1.BVH_BUILD_DEVICE)
    assert tree_bytes(s.bvh_on_device()) == want


def test_every_device_builds_the_same_tree(r1, tmp_path):
    n = r1.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    cam, sph = make_scene.cloud_scene(20000, seed=9)
    path = str(tmp_path / "cloud.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path, commit=False)
    try:
        want = tree_bytes(lbvh.build(s.soa()))
        for dev in range(n):
            r1._check(r1.lib.r1_scene_commit(s.handle, dev), "commit")
            s.build_bvh(r1.BVH_BUILD_DEVICE, device=dev)
            assert tree_bytes(s.bvh_on_device(device=dev)) == want, "device %d" % dev
    finally:
        s.close()


def test_non_finite_spheres_are_refused(r1):
    for bad in (_f(np.nan, 0, 0, 1), _f(0, np.inf, 0, 1), _f(0, 0, 0, 1e20)):   # 1e20: radius_sq overflows to inf
        sph = [_f(0, 0, 0, 1) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), bad + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0)]
        s = RawScene(CAM, sph)
        try:
            with pytest.raises(r1.Rays1Error, match=r"\(-1\).*non-finite"):
                s.build_bvh(r1.BVH_BUILD_DEVICE)
            with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):          # the failed build left the device without a tree
                s.bvh_on_device()
        finally:
            s.close()


def test_host_build_puts_the_host_tree_on_the_device(r1):
    for name in ("large", "synth4096"):
        s = r1.create_scene(name)
        try:
            with pytest.raises(r1.Rays1Error, match=r"\(-2\).*holds no bvh"):
                s.bvh_on_device()
            assert s.build_bvh(r1.BVH_BUILD_HOST) >= 0
            assert tree_bytes(s.bvh_on_device()) == tree_bytes(s.bvh())
        finally:
            s.close()


# ---- 10^6 spheres ----------------------------------------------------------------------------------------------------------

def test_million_sphere_cloud(r1, oracle, tmp_path):
    cam, sph = make_scene.cloud_scene(1000000)
    path = str(tmp_path / "cloud1e6.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path)
    try:
        ms = s.build_bvh(r1.BVH_BUILD_DEVICE)
        nodes, leaves, depth = s.bvh_on_device()
        assert depth <= MAX_DEPTH and len(leaves) == s.count() - 7
        check_structure(s, nodes, leaves, depth)
        dev_rgb, dev_res = s.render(320, 180, 8, variant=r1.VARIANT_MEGAKERNEL_BVH)
        # 2 000 rays through and around the cloud against the oracle
        soa = s.soa()
        rng = np.random.default_rng(41)
        span = float(np.abs(soa["cx"][:-8]).max())
        o = (rng.uniform(-1.2 * span, 1.2 * span, (2000, 3)) + [0, span, 0]).astype(np.float32)
        d = rng.normal(size=(2000, 3))
        d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
        so = oracle.scene_create_from_soa(soa)
        try:
            want = oracle.hit(so, o, d, 0.001, FLT_MAX)
        finally:
            oracle.scene_destroy(so)
        assert (want[0] >= 0).sum() > 1000
        assert_same(trace(r1, s, o, d), want, "cloud 10^6")
        host_ms = s.build_bvh(r1.BVH_BUILD_HOST)
        host_rgb, host_res = s.render(320, 180, 8, variant=r1.VARIANT_MEGAKERNEL_BVH)
        assert np.array_equal(dev_rgb, host_rgb) and dev_res.num_rays == host_res.num_rays
        print("cloud 10^6: device build %.2f ms (depth %d, %d nodes), host tree upload %.2f ms" % (ms, depth, len(nodes), host_ms))
    finally:
        s.close()


# ---- lifecycle -------------------------------------------------------------------------------------------------------------

def test_a_recommit_returns_to_the_first_use_host_tree(r1):
    s = r1.create_scene("medium")
    try:
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        dev = tree_bytes(s.bvh_on_device())
        assert dev == tree_bytes(lbvh.build(s.soa()))
        s.build_bvh(r1.BVH_BUILD_HOST)
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(s.bvh())
        r1._check(r1.lib.r1_scene_commit(s.handle, 0), "commit")
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            s.bvh_on_device()
        base, r0 = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        rgb, res = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)     # first use: the host tree
        assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(s.bvh()) and tree_bytes(s.bvh()) != dev
    finally:
        s.close()


def test_spheres_added_after_the_commit_refuse_the_build(r1):
    sph = [_f(0, 0, 0, 1) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), _f(0, -1001, 0, 1000) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0)]
    s = RawScene(CAM, sph)
    try:
        r1._check(r1.lib.r1_scene_add_sphere(s.handle, 2, 0, 0, 1, r1.MAT_METAL, 0.5, 0.5, 0.5, 0), "add")
        for builder in (r1.BVH_BUILD_HOST, r1.BVH_BUILD_DEVICE):
            with pytest.raises(r1.Rays1Error, match=r"\(-2\).*commit it again"):
                s.build_bvh(builder)
    finally:
        s.close()
