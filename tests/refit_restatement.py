"""CPU restatement of the BVH refit of r1_scene_move_spheres (r1_bvh_device.cu refit_nodes, DESIGN.md section 4.10), from its
specification and in numpy.

The device refits bottom-up with one thread per node and atomic arrival counters; this goes level by level, deepest first.  The
result is specified as a function of the tree's topology and the spheres' exact records alone:
  - child references, record order and depth are unchanged; slots with child -1 keep their bytes;
  - every leaf record's {cx, cy, cz, radius_sq} becomes the sphere's exact record;
  - every other slot gets the float union of the padded sphere boxes [c - rp, c + rp] rounded outward,
    rp = sqrt((double) r2) (1 + 2^-16), of the spheres under it, and diag = round_up(sqrt(d2) (1 + 1e-12)) of that box.
`refit(tree, exact)` takes (nodes, leaves, depth) as Scene.bvh() returns them and exact [n, 4] float32 (cx, cy, cz, radius_sq per
sphere index), and returns the refitted (nodes, leaves, depth)."""
import numpy as np

import lbvh_restatement as lbvh


def exact_of(soa):
    """[n, 4] float32: the exact records {cx, cy, cz, radius_sq} of a SoA"""
    return np.stack([soa["cx"], soa["cy"], soa["cz"], soa["radius_sq"]], 1).astype(np.float32)


def record_boxes(ex):
    """padded boxes (lo, hi) [k, 3] float32 of exact records [k, 4] (step 1 of the builders)"""
    rp = np.sqrt(ex[:, 3].astype(np.float64)) * lbvh.RADIUS_PAD
    c = ex[:, :3].astype(np.float64)
    return lbvh.box_bounds(c, rp)


def diag_bound(lo, hi):
    """[k] float32: round_up(sqrt(w0^2 + w1^2 + w2^2) (1 + 1e-12)) in double, the builders' order"""
    w = hi.astype(np.float64) - lo.astype(np.float64)
    d2 = (w[:, 0] * w[:, 0] + w[:, 1] * w[:, 1]) + w[:, 2] * w[:, 2]
    return lbvh.round_up(np.sqrt(d2) * lbvh.DIAG_PAD).astype(np.float32)


def node_depths(nodes):
    """depth of every node (root = 1) from the child references, and its (parent, slot) (-1 for the root)"""
    ch = nodes["child"]
    parent = np.full((len(nodes), 2), -1, np.int64)
    pn, ps = np.nonzero(ch >= 0)
    parent[ch[pn, ps]] = np.stack([pn, ps], 1)
    depth = np.zeros(len(nodes), np.int64)
    depth[0] = 1
    frontier = np.array([0])
    d = 1
    while len(frontier):
        kids = ch[frontier]
        kids = kids[kids >= 0]
        d += 1
        depth[kids] = d
        frontier = kids
    return depth, parent


def refit(tree, exact):
    nodes, leaves, depth = tree
    nodes, leaves = nodes.copy(), leaves.copy()
    leaves["exact"] = exact[leaves["index"]]
    ch = nodes["child"]
    inf = np.float32(np.inf)
    # slot boxes, inf / -inf where a slot is empty or not yet known
    lo = np.full((len(nodes), 2, 3), inf, np.float32)
    hi = np.full((len(nodes), 2, 3), -inf, np.float32)
    # leaf slots: unions of their records' boxes (the records cover the array once, in order of `first`)
    node, slot = np.nonzero(ch < -1)
    v = ~ch[node, slot]
    first, count = v >> 3, v & 7
    if len(node):
        rlo, rhi = record_boxes(leaves["exact"])
        order = np.argsort(first)
        lo[node[order], slot[order]] = np.minimum.reduceat(rlo, first[order], axis=0)
        hi[node[order], slot[order]] = np.maximum.reduceat(rhi, first[order], axis=0)
    # inner slots, deepest children first: the union of the child node's used slots
    dep, parent = node_depths(nodes)
    for d in range(int(dep.max()), 1, -1):
        kids = np.nonzero(dep == d)[0]
        p, s = parent[kids, 0], parent[kids, 1]
        lo[p, s] = np.minimum(lo[kids, 0], lo[kids, 1])
        hi[p, s] = np.maximum(hi[kids, 0], hi[kids, 1])
    used = ch != -1
    n_idx, s_idx = np.nonzero(used)
    for k in (0, 1):
        sel = s_idx == k
        nn = n_idx[sel]
        nodes["lo%d" % k][nn] = lo[nn, k]
        nodes["hi%d" % k][nn] = hi[nn, k]
        nodes["diag"][nn, k] = diag_bound(lo[nn, k], hi[nn, k])
    return nodes, leaves, depth
