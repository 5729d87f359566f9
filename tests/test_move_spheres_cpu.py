"""CPU checks of moving spheres on the device (r1_scene_move_spheres, DESIGN.md section 4.10) through the refit's restatement,
tests/refit_restatement.py.

At unchanged positions the restated refit returns both builders' trees byte for byte: the host tree (r1_bvh_export) and the device
builder's (lbvh_restatement.build).  Refitted to moved spheres, a tree keeps the structure DESIGN.md section 4.8 requires of any BVH
the traversal runs (test_bvh_cpu.check_structure, against the moved scene), and the kernel's box test passes the winning sphere's
leaf and every ancestor for the oracle's Hitable::hit on the moved scene (test_bvh_cpu.check_conservative): small jitter, motion
that tangles the tree, every sphere collapsed onto one point, and a scene moved 1e6 away from the origin.  The device's refit is
compared with the restatement byte for byte on the GPU by tests/test_move_spheres_gpu.py.  Also: header, Python and library agree
on the new names, and the argument refusals need no device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import lbvh_restatement as lbvh
import refit_restatement as refit
from conftest import ROOT
from test_bvh_cpu import BUILTIN, EDGE, check_conservative, check_structure, cloud, host_scenes  # noqa: F401
from test_bvh_device_cpu import CAM, SPECIAL, special_spheres
from test_scan_edges_gpu import FLT_MAX, RawScene, aimed_rays


def tree_bytes(tree):
    nodes, leaves, depth = tree
    return nodes.tobytes(), leaves.tobytes(), depth


@pytest.fixture(scope="module")
def special_scenes(r1):
    out = {name: RawScene(CAM, special_spheres(r1, name), commit=False) for name in SPECIAL}
    yield out
    for s in out.values():
        s.close()


# ---- identity: a refit at unchanged positions returns both builders' trees ----------------------------------------------------

def check_identity(s):
    soa = s.soa()
    ex = refit.exact_of(soa)
    for tree in (s.bvh(), lbvh.build(soa)):
        assert tree_bytes(refit.refit(tree, ex)) == tree_bytes(tree)


@pytest.mark.parametrize("name", BUILTIN + EDGE)
def test_refit_at_unchanged_positions_is_the_identity(host_scenes, name):  # noqa: F811
    check_identity(host_scenes[name])


@pytest.mark.parametrize("name", SPECIAL)
def test_refit_at_unchanged_positions_is_the_identity_on_special_scenes(special_scenes, name):
    check_identity(special_scenes[name])


def test_refit_at_unchanged_positions_is_the_identity_on_a_cloud(cloud):  # noqa: F811
    check_identity(cloud)


# ---- moved scenes --------------------------------------------------------------------------------------------------------------

def moved_soa(soa, motion, seed=3):
    """a copy of soa with the centres of every sphere moved (radii, materials and inv_radius kept)"""
    rng = np.random.default_rng(seed)
    out = {k: v.copy() for k, v in soa.items()}
    c = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1).astype(np.float64)
    real = soa["inv_radius"] != 0
    span = np.abs(c[real]).max() + 1.0
    if motion == "jitter":
        c = c + rng.normal(scale=1e-3 * span, size=c.shape)
    elif motion == "tangle":                                             # every sphere jumps to another's place, plus noise
        c = c[rng.permutation(len(c))] + rng.normal(scale=0.05 * span, size=c.shape)
    elif motion == "collapse":
        c[:] = (1.5, 2.5, -3.5)
    elif motion == "far":
        c = c + 1e6
    out["cx"], out["cy"], out["cz"] = (c[:, k].astype(np.float32) for k in range(3))
    return out


class Moved:
    """a scene's moved SoA with a refitted tree, for check_structure and check_conservative"""

    def __init__(self, soa, tree):
        self._soa, self.tree = soa, tree

    def soa(self):
        return self._soa

    def bvh(self):
        return self.tree


def moved_rays(soa, seed=17, n=1500):
    rng = np.random.default_rng(seed)
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    c = np.stack([soa["cx"][real], soa["cy"][real], soa["cz"][real]], 1).astype(np.float64)
    mid, span = c.mean(0), np.abs(c - c.mean(0)).max() + 1.0
    o1 = mid + rng.uniform(-1.5 * span, 1.5 * span, (n, 3))
    d1 = rng.normal(size=(n, 3))
    d1 /= np.linalg.norm(d1, axis=1, keepdims=True)
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([0.5, 5.0, 50.0, 500.0], n))
    return np.concatenate([o1, o2]).astype(np.float32), np.concatenate([d1, d2]).astype(np.float32)


MOTIONS = ("jitter", "tangle", "collapse", "far")


@pytest.mark.parametrize("motion", MOTIONS)
@pytest.mark.parametrize("name", ("medium", "large", "flood488", "ties"))
def test_refit_trees_of_moved_scenes_keep_the_traversal_exact(oracle, host_scenes, name, motion):  # noqa: F811
    s = host_scenes[name]
    soa = moved_soa(s.soa(), motion)
    org, d = moved_rays(soa)
    for builder, tree in (("host", s.bvh()), ("device", lbvh.build(s.soa()))):
        m = Moved(soa, refit.refit(tree, refit.exact_of(soa)))
        check_structure(m, *m.tree)
        n = check_conservative(m, oracle, org, d, ((0.001, FLT_MAX), (0.5, 40.0)), "%s %s %s" % (name, motion, builder))
        assert n > 300


@pytest.mark.parametrize("motion", ("tangle", "far"))
def test_refit_trees_of_a_moved_cloud_keep_the_traversal_exact(oracle, cloud, motion):  # noqa: F811
    soa = moved_soa(cloud.soa(), motion)
    org, d = moved_rays(soa, n=1000)
    m = Moved(soa, refit.refit(lbvh.build(cloud.soa()), refit.exact_of(soa)))
    check_structure(m, *m.tree)
    assert check_conservative(m, oracle, org, d, ((0.001, FLT_MAX),), "cloud %s" % motion) > 300


def test_refit_boxes_contain_exactly_the_spheres_below(host_scenes):  # noqa: F811
    """each used slot's box is the union of its spheres' padded boxes: moving one sphere far changes exactly its root path"""
    s = host_scenes["large"]
    soa = s.soa()
    tree = s.bvh()
    k = int(tree[1]["index"][len(tree[1]) // 2])
    moved = {key: v.copy() for key, v in soa.items()}
    moved["cx"][k] += np.float32(5000)
    a = refit.refit(tree, refit.exact_of(soa))[0]
    b = refit.refit(tree, refit.exact_of(moved))[0]
    from test_bvh_cpu import path_slots
    path = set(map(tuple, path_slots(*tree[:2])[k]))
    changed = {(int(n), j) for n in range(len(a)) for j in (0, 1) if a[n]["hi%d" % j][0] != b[n]["hi%d" % j][0]}
    assert changed == {(int(n), int(j)) for n, j in path}


# ---- interface -----------------------------------------------------------------------------------------------------------------

def test_header_python_and_library_agree_on_the_names(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    for fn in ("r1_scene_move_spheres", "r1_scene_export_device"):
        assert re.search(r"\bint %s\(" % fn, header) and fn in r1.EXPORTED
    assert "#define R1_ABI_VERSION 2" in header and r1.lib.r1_abi_version() == 2
    assert callable(r1.Scene.move_spheres) and callable(r1.Scene.device_records)


def test_move_refuses_bad_arguments_without_a_device(r1):
    lib = r1.lib
    ms = C.c_double(0)
    buf = (C.c_float * 12)()
    assert lib.r1_scene_move_spheres(None, -1, 0, 1, buf, None, None, C.byref(ms)) == -1
    nb = C.c_uint64(0)
    assert lib.r1_scene_export_device(None, -1, None, 0, C.byref(nb)) == -1
    sc = lib.r1_scene_create(4)
    try:
        for j in range(3):
            assert lib.r1_scene_add_sphere(sc, j, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0) == j
        cases = ((0, 4, buf), (3, 1, buf), (2, 2, buf), (1, 0xFFFFFFFF, buf), (0xFFFFFFFF, 2, buf), (0, 1, None), (2, 1, None))
        for first, n, ptr in cases:
            assert lib.r1_scene_move_spheres(sc, -1, first, n, ptr, None, None, C.byref(ms)) == -1, (first, n)
            assert lib.r1_scene_move_spheres(sc, 0, first, n, ptr, buf, None, None) == -1, (first, n)
        assert b"null centres" in lib.r1_last_error()
        # valid arguments: refused by the state check (not committed) or the device lookup, never a crash
        for first, n in ((0, 3), (1, 2), (3, 0), (0, 0)):
            assert lib.r1_scene_move_spheres(sc, -1, first, n, buf, None, None, C.byref(ms)) in (-2, -3)
            assert lib.r1_scene_move_spheres(sc, 0, first, n, buf, buf, None, None) in (-2, -3)
        assert lib.r1_scene_export_device(sc, -1, None, 0, C.byref(nb)) == -2
        assert lib.r1_scene_export_device(sc, 0, None, 0, C.byref(nb)) == -2
    finally:
        lib.r1_scene_destroy(sc)


def test_python_checks_tensors_before_the_library(r1):
    torch = pytest.importorskip("torch")
    s = RawScene(CAM, [(0.0, 0.0, 0.0, 1.0, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0.0)], commit=False)
    try:
        with pytest.raises(ValueError, match="CUDA tensor"):
            s.move_spheres(torch.zeros(1, 3))
        with pytest.raises(ValueError, match="CUDA tensor"):
            s.move_spheres(np.zeros((1, 3), np.float32))
    finally:
        s.close()
