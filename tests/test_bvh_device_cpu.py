"""CPU checks of the device BVH builder (r1_scene_build_bvh with R1_BVH_BUILD_DEVICE, DESIGN.md section 4.9) through its
restatement, tests/lbvh_restatement.py.  The restated tree must have the structure DESIGN.md section 4.8 requires of any BVH the
traversal runs (test_bvh_cpu.check_structure) with depth <= 62, and the kernel's box test must pass the winning sphere's leaf and
every ancestor for the oracle's Hitable::hit (test_bvh_cpu.check_conservative).  The device's tree is compared with the
restatement byte for byte on the GPU by tests/test_bvh_device_gpu.py.  Also: header, Python and library agree on the new names,
and the entry points refuse bad arguments and uncommitted scenes without a device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import lbvh_restatement as lbvh
from conftest import ROOT
from test_bvh_cpu import BUILTIN, EDGE, all_rays, check_conservative, check_structure, cloud, host_scenes  # noqa: F401
from test_scan_edges_gpu import FLT_MAX, T_BOUND, RawScene, _f

MAX_DEPTH = 62
CAM = _f(0, 1, 20, 0, 0, 0, 40, 0, 20)


def _sphere(r1, x, y, z, radius, kind=None):
    kind = r1.MAT_LAMBERT if kind is None else kind
    return _f(x, y, z, radius) + (kind,) + _f(0.5, 0.5, 0.5, 0)


def special_spheres(r1, name):
    """sphere lists of the scenes the builder's special cases need (raw ABI, no padding)"""
    never = [_sphere(r1, 3, 0, 0, 0, r1.MAT_NONE), _sphere(r1, 6, 0, 0, -2)]               # inv_radius == 0: not in the tree
    if name.startswith("real"):                                                             # real0 .. real5: the root's leaf cases
        k = int(name[4:])
        sph = [_sphere(r1, 2.5 * j, 0.5 * (j % 2), -j, 0.5 + 0.1 * j) for j in range(k)]
        return never[:1] + sph + never[1:]
    if name == "coincident_equal":                                                          # 1 000 spheres at one point
        return [_sphere(r1, 1, 2, 3, 0.5) for _ in range(1000)]
    if name == "coincident_radii":
        return [_sphere(r1, 1, 2, 3, r) for r in np.linspace(0.1, 2.0, 1000)]
    if name == "morton_exhausted":
        # centres at 2^-k along x and one far sphere: every small centre quantises to q = 0, so their keys differ in the index
        # bits alone and the tree below them is built from those
        return [_sphere(r1, 2.0 ** -k, 0, 0, 2.0 ** -k / 4) for k in range(48)] + [_sphere(r1, 4096, 0, 0, 1)]
    raise KeyError(name)


SPECIAL = ("real0", "real1", "real4", "real5", "coincident_equal", "coincident_radii", "morton_exhausted")


class Restated:
    """a scene whose bvh() is the restatement's tree (for check_structure and check_conservative)"""

    def __init__(self, s):
        self.s = s
        self.tree = lbvh.build(s.soa())

    def soa(self):
        return self.s.soa()

    def bvh(self):
        return self.tree


@pytest.fixture(scope="module")
def special_scenes(r1):
    out = {name: RawScene(CAM, special_spheres(r1, name), commit=False) for name in SPECIAL}
    yield out
    for s in out.values():
        s.close()


def check_restated(s):
    nodes, leaves, depth = lbvh.build(s.soa())
    check_structure(s, nodes, leaves, depth)
    assert depth <= MAX_DEPTH
    return nodes, leaves, depth


# ---- structure -------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", BUILTIN + EDGE)
def test_restated_structure(host_scenes, name):  # noqa: F811
    check_restated(host_scenes[name])


def test_restated_structure_of_a_cloud(cloud):  # noqa: F811
    nodes, leaves, depth = check_restated(cloud)
    assert len(leaves) == cloud.count() - 7


@pytest.mark.parametrize("name", SPECIAL)
def test_restated_structure_of_special_scenes(special_scenes, name):
    s = special_scenes[name]
    nodes, leaves, depth = check_restated(s)
    real = int((s.soa()["inv_radius"] != 0).sum())
    assert len(leaves) == real
    if real <= 4:
        # one node, a leaf of every real sphere in slot 0 and nothing in slot 1: the host builder's root, byte for byte
        assert len(nodes) == 1 and depth == 1
        hn, hl, hd = s.bvh()
        assert nodes.tobytes() == hn.tobytes() and leaves.tobytes() == hl.tobytes() and depth == hd
    else:
        assert (nodes["child"][0] != -1).all()                              # the root splits: both slots are used
    if name.startswith("coincident"):
        assert depth <= 9                                                   # identical Morton codes: the index bits halve the range


def test_leaf_records_follow_the_sorted_keys(special_scenes):
    """leaf `first` ascends in preorder and the records, read leaf by leaf, are the sorted keys' spheres"""
    s = special_scenes["morton_exhausted"]
    soa = s.soa()
    real = np.nonzero(soa["inv_radius"] != 0)[0]
    keys = lbvh.sorted_keys(soa, real)
    nodes, leaves, _ = lbvh.build(soa)
    assert (keys >> np.uint64(32) == 0).sum() == len(real) - 1               # every small centre has Morton code 0
    ids = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
    ch = nodes["child"]
    first, count = (~ch[ch < -1]) >> 3, (~ch[ch < -1]) & 7
    for f, c in zip(first, count):
        assert np.array_equal(leaves["index"][f:f + c], np.sort(ids[f:f + c]))


def test_morton_quantisation_follows_the_specification(r1):
    """q = min(1023, floor((c - lo) / ext * 1024)), bits interleaved x -> 3b + 2, y -> 3b + 1, z -> 3b"""
    soa = {"cx": np.array([0, 1, 0.5, 0.25], np.float32), "cy": np.array([0, 0, 1, 0], np.float32),
           "cz": np.array([0, 0, 0, 1], np.float32)}
    keys = lbvh.sorted_keys(soa, np.arange(4))
    got = {int(k & np.uint64(0xFFFFFFFF)): int(k >> np.uint64(32)) for k in keys}
    assert got[0] == 0
    assert got[1] == int(lbvh.spread3(np.array([1023], np.uint64))[0]) << 2           # q_x = 1023 (clamped from 1024)
    assert got[2] == (int(lbvh.spread3(np.array([512], np.uint64))[0]) << 2) | (int(lbvh.spread3(np.array([1023], np.uint64))[0]) << 1)
    assert got[3] == (int(lbvh.spread3(np.array([256], np.uint64))[0]) << 2) | int(lbvh.spread3(np.array([1023], np.uint64))[0])


# ---- conservativeness of the box test on the restated trees ------------------------------------------------------------------

@pytest.mark.parametrize("name", EDGE + BUILTIN)
def test_box_test_passes_the_winners_path_in_the_restated_tree(oracle, host_scenes, name):  # noqa: F811
    s = Restated(host_scenes[name])
    soa = s.soa()
    org, d = all_rays(name if name in EDGE else "n%d" % 200, soa)
    n = check_conservative(s, oracle, org, d, ((0.001, FLT_MAX), (0.5, 40.0), (T_BOUND, FLT_MAX)), name)
    assert n > 500


def test_box_test_on_the_restated_tree_of_a_cloud(oracle, cloud):  # noqa: F811
    from test_scan_edges_gpu import aimed_rays
    from test_bvh_cpu import surface_rays, zero_component_rays
    s = Restated(cloud)
    soa = s.soa()
    rng = np.random.default_rng(78)
    n = 3000
    span = float(np.abs(soa["cx"][:-8]).max())
    o1 = (rng.uniform(-1.2 * span, 1.2 * span, (n, 3)) + [0, span, 0]).astype(np.float32)
    d1 = rng.normal(size=(n, 3))
    d1 = (d1 / np.linalg.norm(d1, axis=1, keepdims=True)).astype(np.float32)
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    o3, d3 = zero_component_rays(soa, rng)
    o4, d4 = surface_rays(soa, rng)
    org = np.concatenate([o1, o2, o3, o4]).astype(np.float32)
    d = np.concatenate([d1, d2, d3, d4]).astype(np.float32)
    assert check_conservative(s, oracle, org, d, ((0.001, FLT_MAX), (0.5, 40.0)), "cloud") > 4000


# ---- interface -------------------------------------------------------------------------------------------------------------

def test_header_python_and_library_agree_on_the_builders(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    values = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(R1_BVH_BUILD_\w+)\s*=\s*(\d+)", header)}
    assert values == {"R1_BVH_BUILD_HOST": 0, "R1_BVH_BUILD_DEVICE": 1}
    assert (r1.BVH_BUILD_HOST, r1.BVH_BUILD_DEVICE) == (0, 1)
    for fn in ("r1_scene_build_bvh", "r1_bvh_export_device"):
        assert "int %s(" % fn in header and fn in r1.EXPORTED


def test_build_and_export_refuse_bad_arguments_and_uncommitted_scenes(r1):
    lib = r1.lib
    ms = C.c_double(0)
    nn = C.c_uint32(0)
    assert lib.r1_scene_build_bvh(None, -1, r1.BVH_BUILD_DEVICE, C.byref(ms)) == -1
    assert lib.r1_bvh_export_device(None, -1, None, 0, None, 0, C.byref(nn), None, None) == -1
    sc = lib.r1_scene_create(4)
    try:
        assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0) == 0
        for bad in (2, -1, 99):
            assert lib.r1_scene_build_bvh(sc, -1, bad, C.byref(ms)) == -1 and b"unknown bvh builder" in lib.r1_last_error()
        for builder in (r1.BVH_BUILD_HOST, r1.BVH_BUILD_DEVICE):
            assert lib.r1_scene_build_bvh(sc, -1, builder, None) in (-2, -3)       # not committed (R1_ERR_STATE) / no device (R1_ERR_CUDA)
            assert lib.r1_scene_build_bvh(sc, 0, builder, C.byref(ms)) in (-2, -3)
        assert lib.r1_bvh_export_device(sc, -1, None, 0, None, 0, C.byref(nn), None, None) == -2
        assert lib.r1_bvh_export_device(sc, 0, None, 0, None, 0, C.byref(nn), None, None) == -2
    finally:
        lib.r1_scene_destroy(sc)
