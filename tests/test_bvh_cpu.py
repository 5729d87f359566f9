"""CPU checks of the BVH variant (R1_VARIANT_MEGAKERNEL_BVH): the interface agrees on its value, the tree r1_bvh_export returns
has the structure DESIGN.md section 4.8 states, and the kernel's box test -- restated here in float32 in the kernel's operation
order (r1_device.cuh, bvh_child) -- passes the winning sphere's leaf and every ancestor at t_best = t_winner for the oracle's
Hitable::hit on every edge scene and on a 100 000-sphere cloud.  With the order-free acceptance rule that is what makes the
traversal return the brute-force scan's hit.  The kernels themselves are tested on the GPU by tests/test_bvh_gpu.py."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_scan_edges_gpu import (FLOODS, SWEEP, T_BOUND, RawScene, _f, aimed_rays, boundary_queries, boundary_rays, make_scene,
                                 scene_rays, tangent_rays)

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene as scene_tool  # noqa: E402

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)
GAMMA = F32(1.0 / 512.0)
UP = F32(1.0 + 2.0 ** -20)
RADIUS_PAD = 1.0 + 2.0 ** -16
BUILTIN = ("small", "medium", "large", "synth4096")
EDGE = tuple("n%d" % n for n in SWEEP) + tuple("flood%d" % n for n in FLOODS) + ("ties",)


# ---- interface ----------------------------------------------------------------------------------------------------------------

def test_header_python_and_executable_agree_on_the_value(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    values = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(R1_VARIANT_\w+)\s*=\s*(\d+)", header)}
    assert values["R1_VARIANT_MEGAKERNEL_BVH"] == 11
    assert 8 not in values.values() and 10 not in values.values()
    assert r1.VARIANT_MEGAKERNEL_BVH == 11 and r1.VARIANTS["bvh"] == 11
    assert sorted(values.values()) == sorted(set(r1.VARIANTS.values()))
    assert "int r1_bvh_export(" in header and "r1_bvh_export" in r1.EXPORTED
    main = open(os.path.join(ROOT, "rays1bench_b200", "csrc", "rays1_main.cpp")).read()
    usage = [l for l in main.splitlines() if "--variant" in l and l.startswith("//")]
    assert len(usage) == 1 and "|bvh|" in usage[0] and "|tensor-stream|" in usage[0]
    assert re.search(r'!strcmp\(v, "bvh"\)\) cfg\.variant = R1_VARIANT_MEGAKERNEL_BVH;', main)


def test_unknown_variants_are_refused_and_11_reaches_the_device_check(r1):
    lib = r1.lib
    sc = lib.r1_scene_create(8)
    assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0) == 0
    p = r1.RenderParams(16, 9, 1, 4, 0, 0, 0, 1, 1, 0, 0, -1)
    res = r1.Result()
    rgb = np.zeros(16 * 9 * 3, np.uint8)
    one = np.zeros(3, np.float32)
    for v in (8, 10, 12, -1):
        p.variant = v
        assert lib.r1_render(sc, C.byref(p), rgb, C.byref(res)) == -1 and b"unknown variant" in lib.r1_last_error()
        assert lib.r1_render_device(sc, C.byref(p), None, None, None, C.byref(res)) == -1
    p.variant = r1.VARIANT_MEGAKERNEL_BVH
    assert lib.r1_render(sc, C.byref(p), rgb, C.byref(res)) in (-2, -3)      # not committed (R1_ERR_STATE) / no device (R1_ERR_CUDA)
    assert lib.r1_render_device(sc, C.byref(p), None, None, None, C.byref(res)) in (-2, -3)
    idx, t = np.zeros(1, np.int32), np.zeros(1, np.float32)
    assert lib.r1_trace_rays(sc, 1, one, one, 0.001, 1.0, r1.VARIANT_MEGAKERNEL_BVH, idx, t, one, one) in (-2, -3)
    lib.r1_scene_destroy(sc)


# ---- structure ------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def host_scenes(r1, tmp_path_factory):
    d = tmp_path_factory.mktemp("bvh_cpu")
    out = {}
    for name in BUILTIN:
        out[name] = r1.create_scene(name, commit=False)
    for name in EDGE:
        out[name] = make_scene(r1, name, d, commit=False)
    yield out
    for s in out.values():
        s.close()


@pytest.fixture(scope="module")
def cloud(r1, tmp_path_factory):
    cam, sph = scene_tool.cloud_scene(100000, seed=5)
    path = str(tmp_path_factory.mktemp("cloud") / "cloud.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path, commit=False)
    yield s
    s.close()


def slot_boxes(nodes):
    """(lo, hi) of every (node, slot) as float32 [n_nodes, 2, 3]"""
    lo = np.stack([nodes["lo0"], nodes["lo1"]], 1)
    hi = np.stack([nodes["hi0"], nodes["hi1"]], 1)
    return lo, hi


def leaf_slots(nodes):
    """(node, slot, first, count) of every leaf reference"""
    node, slot = np.nonzero(nodes["child"] < -1)
    v = ~nodes["child"][node, slot]
    return node, slot, v >> 3, v & 7


def check_structure(s, nodes, leaves, depth):
    soa = s.soa()
    n = len(soa["cx"])
    real = np.nonzero(soa["inv_radius"] != 0)[0]
    assert depth <= 64 and len(nodes) >= 1
    # every real sphere exactly once, nothing else; records bit-equal to the SoA
    idx = leaves["index"]
    assert np.array_equal(np.sort(idx), real)
    ex = np.stack([soa["cx"], soa["cy"], soa["cz"], soa["radius_sq"]], 1)
    assert np.array_equal(leaves["exact"].view(np.uint32), ex[idx].view(np.uint32))
    assert not leaves["pad"].any()
    # leaves: 1 .. 4 records, ascending index, covering the record array exactly once in order
    node, slot, first, count = leaf_slots(nodes)
    assert count.min(initial=1) >= 1 and count.max(initial=1) <= 4
    order = np.argsort(first)
    assert np.array_equal(first[order], np.concatenate([[0], np.cumsum(count[order])[:-1]]) if len(first) else first)
    assert count.sum() == len(leaves)
    for f, c in zip(first, count):
        assert np.all(np.diff(idx[f:f + c]) > 0)
    # inner references: every node but the root is referenced once, by a parent with a lower index
    ch = nodes["child"]
    inner = ch[ch >= 0]
    assert np.array_equal(np.sort(inner), np.arange(1, len(nodes)))
    parent = np.full(len(nodes), -1)
    pn, ps = np.nonzero(ch >= 0)
    parent[ch[pn, ps]] = pn
    assert np.all(parent[1:] < np.arange(1, len(nodes)))
    # depth: inner nodes on the way to each node
    dep = np.ones(len(nodes), np.int64)
    for k in range(1, len(nodes)):
        dep[k] = dep[parent[k]] + 1
    assert dep.max() == depth
    # boxes: a parent's slot box contains both boxes of the child node; diag bounds the slot box's diagonal
    lo, hi = slot_boxes(nodes)
    if len(pn):
        c = ch[pn, ps]
        for j in (0, 1):
            live = ch[c, j] != -1
            assert np.all(lo[pn, ps][live] <= lo[c, j][live]) and np.all(hi[c, j][live] <= hi[pn, ps][live])
    used = ch != -1
    diag = np.sqrt(((hi.astype(np.float64) - lo) ** 2).sum(-1))
    assert np.all(nodes["diag"][used] >= diag[used])
    # every sphere's leaf box contains [c - r (1 + 2^-16), c + r (1 + 2^-16)] (evaluated in double)
    rec = np.concatenate([np.arange(f, f + c) for f, c in zip(first, count)]) if len(count) else np.zeros(0, int)
    rec_slot = np.repeat(np.arange(len(node)), count)
    cc = ex[idx[rec], :3].astype(np.float64)
    rp = np.sqrt(ex[idx[rec], 3].astype(np.float64)) * RADIUS_PAD
    assert np.all(lo[node[rec_slot], slot[rec_slot]] <= cc - rp[:, None])
    assert np.all(cc + rp[:, None] <= hi[node[rec_slot], slot[rec_slot]])
    assert n >= len(real)


@pytest.mark.parametrize("name", BUILTIN + EDGE)
def test_structure(host_scenes, name):
    s = host_scenes[name]
    nodes, leaves, depth = s.bvh()
    check_structure(s, nodes, leaves, depth)


def test_structure_of_a_cloud(cloud):
    nodes, leaves, depth = cloud.bvh()
    check_structure(cloud, nodes, leaves, depth)
    assert len(leaves) == cloud.count() - 7 and depth <= 40       # the 7 placeholders of the padding to 8 are left out


def test_padding_and_nonpositive_radii_are_left_out(r1):
    sph = [_f(0, 0, 0, 1) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), _f(3, 0, 0, 0) + (r1.MAT_NONE,) + _f(0, 0, 0, 0),
           _f(6, 0, 0, -2) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), _f(9, 0, 0, 0.5) + (r1.MAT_METAL,) + _f(0.5, 0.5, 0.5, 0.1)]
    s = RawScene(_f(0, 0, 20, 0, 0, 0, 40, 0, 20), sph, commit=False)
    try:
        nodes, leaves, depth = s.bvh()
        assert sorted(leaves["index"]) == [0, 3] and len(nodes) == 1 and depth == 1
        assert nodes["child"][0, 1] == -1                               # one leaf under the root, no second child
        r1._check(r1.lib.r1_scene_pad(s.handle, 8), "r1_scene_pad")
        nodes2, leaves2, _ = s.bvh()
        assert sorted(leaves2["index"]) == [0, 3]
        r1._check(r1.lib.r1_scene_add_sphere(s.handle, 12, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0), "add")   # drops the cached tree
        assert sorted(s.bvh()[1]["index"]) == [0, 3, 8]
    finally:
        s.close()


def test_coincident_centres_still_give_small_leaves(r1):
    """1 000 spheres at one point (and 1 000 exact duplicates): split by index order, leaves of <= 4, depth of a halving tree"""
    for radii in (np.linspace(0.1, 2.0, 1000), np.full(1000, 0.5)):
        sph = [_f(1, 2, 3, r) + (r1.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0) for r in radii]
        s = RawScene(_f(0, 0, 20, 0, 0, 0, 40, 0, 20), sph, commit=False)
        try:
            nodes, leaves, depth = s.bvh()
            check_structure(s, nodes, leaves, depth)
            count = ~nodes["child"][nodes["child"] < -1] & 7
            assert count.max() <= 4 and depth <= 9                      # ceil(log2(1000 / 4)) + 1
        finally:
            s.close()


def test_two_builds_are_byte_equal(r1, tmp_path):
    for name in ("large", "synth4096"):
        a, b = r1.create_scene(name, commit=False), r1.create_scene(name, commit=False)
        na, la, da = a.bvh()
        nb, lb, db = b.bvh()
        assert na.tobytes() == nb.tobytes() and la.tobytes() == lb.tobytes() and da == db
        a.close(); b.close()
    for name in ("flood488", "ties"):
        a, b = make_scene(r1, name, tmp_path, commit=False), make_scene(r1, name, tmp_path, commit=False)
        assert a.bvh()[0].tobytes() == b.bvh()[0].tobytes() and a.bvh()[1].tobytes() == b.bvh()[1].tobytes()
        a.close(); b.close()


def test_export_checks_buffer_sizes(r1):
    s = r1.create_scene("medium", commit=False)
    nn, nl, dep = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    assert r1.lib.r1_bvh_export(s.handle, None, 0, None, 0, C.byref(nn), C.byref(nl), C.byref(dep)) == 0 and nn.value > 0
    small = np.zeros(64 * nn.value - 1, np.uint8)
    assert r1.lib.r1_bvh_export(s.handle, small.ctypes.data, small.nbytes, None, 0, None, None, None) == -1
    assert b"node buffer too small" in r1.lib.r1_last_error()
    s.close()


# ---- conservativeness of the box test against the oracle ---------------------------------------------------------------------

def box_test(lo, hi, diag, o, d, t_min, t_lim):
    """bvh_child in float32, the kernel's operation order; lo / hi / o / d [k, 3], diag / t_lim [k].  Returns pass [k]."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = F32(1) / d
        dl = lo - o
        dh = hi - o
        g = np.fmax(np.fmax(dl, -dh), F32(0))
        w = GAMMA * (((g[:, 0] + g[:, 1]) + g[:, 2]) + diag)
        tl = (dl - w[:, None]) * inv
        th = (dh + w[:, None]) * inv
        neg = np.signbit(d)
        nr = np.where(neg, th, tl)
        fr = np.where(neg, tl, th)
        near = np.fmax(np.fmax(nr[:, 0], nr[:, 1]), np.fmax(nr[:, 2], F32(t_min)))
        far = np.fmin(np.fmin(fr[:, 0], fr[:, 1]), np.fmin(fr[:, 2], t_lim))
        return near <= far * UP


def path_slots(nodes, leaves):
    """per sphere index: the (node, slot) pairs from the root down to its leaf"""
    ch = nodes["child"]
    parent = np.full((len(nodes), 2), -1)
    pn, ps = np.nonzero(ch >= 0)
    parent[ch[pn, ps]] = np.stack([pn, ps], 1)
    node, slot, first, count = leaf_slots(nodes)
    out = {}
    for nd, sl, f, c in zip(node, slot, first, count):
        path = [(nd, sl)]
        k = nd
        while k != 0:
            k, s = parent[k]
            path.append((k, s))
        for i in leaves["index"][f:f + c]:
            out[int(i)] = path
    return out


def check_conservative(s, oracle, org, d, windows, what):
    nodes, leaves, _ = s.bvh()
    paths = path_slots(nodes, leaves)
    lo, hi = slot_boxes(nodes)
    so = oracle.scene_create_from_soa(s.soa())
    checked = 0
    try:
        for t_min, t_max in windows:
            idx, t, _, _ = oracle.hit(so, org, d, t_min, t_max)
            ray, pn, ps = [], [], []
            for k in np.nonzero(idx >= 0)[0]:
                for nd, sl in paths[int(idx[k])]:
                    ray.append(k); pn.append(nd); ps.append(sl)
            ray, pn, ps = np.array(ray, int), np.array(pn, int), np.array(ps, int)
            ok = box_test(lo[pn, ps], hi[pn, ps], nodes["diag"][pn, ps], org[ray], d[ray], F32(t_min), t[ray])
            assert ok.all(), "%s [%g, %g]: ray %d, sphere %d: the box test skips the winner's (node %d, slot %d)" % (
                what, t_min, t_max, ray[~ok][0], idx[ray[~ok][0]], pn[~ok][0], ps[~ok][0])
            checked += int((idx >= 0).sum())
    finally:
        oracle.scene_destroy(so)
    return checked


def zero_component_rays(soa, rng, n=300):
    """axis-aligned and in-plane directions with +0 and -0 components, from around aimed spheres"""
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    o, _ = aimed_rays(soa, rng.choice(real, n), rng, rng.uniform(0.5, 30.0, n))
    c = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1)[rng.choice(real, n)]
    d = c - o
    for k in range(n):
        zero = rng.choice(3, rng.integers(1, 3), replace=False)
        d[k, zero] = 0.0
        if not d[k].any():
            d[k, 1] = -1.0
    d = d / np.linalg.norm(d, axis=1, keepdims=True)
    sign = np.where(rng.uniform(size=d.shape) < 0.5, -1.0, 1.0)
    d = np.where(d == 0, sign * 0.0, d)                                       # +0 and -0
    return o.astype(F32), d.astype(F32)


def surface_rays(soa, rng, n=300):
    """rays starting on sphere surfaces (up to rounding) in random directions"""
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    i = rng.choice(real, n)
    c = np.stack([soa["cx"][i], soa["cy"][i], soa["cz"][i]], 1).astype(np.float64)
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    o = c + u / soa["inv_radius"][i, None]
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o.astype(F32), d.astype(F32)


def all_rays(name, soa, seed=12):
    rng = np.random.default_rng(seed)
    o1, d1 = scene_rays(name, soa)                                            # random, grazing and far (5 .. 20 000), floods, ties
    o2, d2 = zero_component_rays(soa, rng)
    o3, d3 = surface_rays(soa, rng)
    parts = [(o1, d1), (o2, d2), (o3, d3)]
    if name == "ties":
        parts.append(tangent_rays())
    return (np.concatenate([p[0] for p in parts]).astype(F32), np.concatenate([p[1] for p in parts]).astype(F32))


@pytest.mark.parametrize("name", EDGE + BUILTIN)
def test_box_test_passes_the_winners_path(oracle, host_scenes, name):
    s = host_scenes[name]
    soa = s.soa()
    org, d = all_rays(name if name in EDGE else "n%d" % 200, soa)
    n = check_conservative(s, oracle, org, d, ((0.001, FLT_MAX), (0.5, 40.0), (T_BOUND, FLT_MAX)), name)
    assert n > 500


@pytest.mark.parametrize("name", ("ties", "n120", "flood96"))
def test_box_test_at_root_boundaries(oracle, host_scenes, name):
    """per hit ray, t_max = t / t + ulp and t_min = t / t - ulp (the tie and root-boundary queries of test_scan_edges_gpu)"""
    s = host_scenes[name]
    soa = s.soa()
    nodes, leaves, _ = s.bvh()
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min in (0.001, T_BOUND):
            org, d, t = boundary_rays(name, soa, so, oracle, t_min)
            assert len(org) >= 40
            for k in range(len(org)):
                for lo, hi in boundary_queries(t_min, t[k]):
                    check_conservative(s, oracle, org[k:k + 1], d[k:k + 1], ((lo, hi),), "%s ray %d" % (name, k))
    finally:
        oracle.scene_destroy(so)


def test_box_test_on_a_cloud(oracle, cloud):
    """100 000 overlapping spheres: random rays, rays grazing spheres from 5 .. 20 000 units, +-0 components, surface starts"""
    soa = cloud.soa()
    rng = np.random.default_rng(77)
    n = 3000
    span = float(np.abs(soa["cx"][:-8]).max())
    o1 = (rng.uniform(-1.2 * span, 1.2 * span, (n, 3)) + [0, span, 0]).astype(F32)
    d1 = rng.normal(size=(n, 3))
    d1 = (d1 / np.linalg.norm(d1, axis=1, keepdims=True)).astype(F32)
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    o2, d2 = aimed_rays(soa, rng.choice(real, n), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n))
    o3, d3 = zero_component_rays(soa, rng)
    o4, d4 = surface_rays(soa, rng)
    org = np.concatenate([o1, o2, o3, o4]).astype(F32)
    d = np.concatenate([d1, d2, d3, d4]).astype(F32)
    assert check_conservative(cloud, oracle, org, d, ((0.001, FLT_MAX), (0.5, 40.0)), "cloud") > 4000
