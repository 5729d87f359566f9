"""CPU restatement of the device BVH builder (r1_bvh_device.cuh, DESIGN.md section 4.9), from its specification and in numpy.

The device builds bottom-up (Karras' radix tree over the sorted keys, an atomic-counter refit, preorder numbers from kept-subtree
sizes); this builds top-down: every sorted range of more than 4 keys splits at its highest differing key bit and nodes are
emitted in preorder, child 0 (the lower keys) first.  Both give one tree, so the two must agree byte for byte.
`build(soa)` returns (nodes, leaves, depth) as the structured arrays of Scene.bvh()."""
import numpy as np

from rays1bench_b200 import BVH_LEAF, BVH_NODE

LEAF_MAX = 4
RADIUS_PAD = 1.0 + 2.0 ** -16
DIAG_PAD = 1.0 + 1e-12


def round_down(v):
    """float64 -> float32 toward -inf (r1_bvh.h round_down, __double2float_rd)"""
    f = v.astype(np.float32)
    return np.where(f.astype(np.float64) > v, np.nextafter(f, np.float32(-np.inf)), f)


def round_up(v):
    f = np.asarray(v).astype(np.float32)
    return np.where(f.astype(np.float64) < v, np.nextafter(f, np.float32(np.inf)), f)


def box_bounds(c, rp):
    """float64 centres [k, 3] (float32 values) and radii [k] -> the floats below c - rp and above c + rp, exactly (r1_bvh.h box_lo /
    box_hi, __dsub_rd / __dadd_ru then directed to float): TwoSum gives the error of the double sum and so the side it rounded to"""
    out = []
    for sgn, rnd, step in ((-1.0, round_down, -np.inf), (1.0, round_up, np.inf)):
        b = sgn * rp[:, None]
        with np.errstate(invalid="ignore"):                 # infinite centres: err is NaN and the box stays infinite
            v = c + b
            bv = v - c
            err = (c - (v - bv)) + (b - bv)
        f = rnd(v)
        off = (f.astype(np.float64) == v) & (err * sgn > 0)
        out.append(np.where(off, np.nextafter(f, np.float32(step)), f))
    return out[0], out[1]


def spread3(v):
    """bit b of a 10-bit value -> bit 3b"""
    out = np.zeros_like(v, dtype=np.uint64)
    for b in range(10):
        out |= ((v >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b)
    return out


def sphere_boxes(soa, real):
    """step 1: [n_real, 3] lo and hi of the padded sphere boxes, rounded outward to float32"""
    c = np.stack([soa["cx"][real], soa["cy"][real], soa["cz"][real]], 1).astype(np.float64)
    rp = np.sqrt(soa["radius_sq"][real].astype(np.float64)) * RADIUS_PAD
    return box_bounds(c, rp)


def sorted_keys(soa, real):
    """steps 2-3: the keys morton << 32 | index of the real spheres, ascending"""
    c = np.stack([soa["cx"][real], soa["cy"][real], soa["cz"][real]], 1)
    lo, hi = c.min(0), c.max(0)                                         # float32 min / max: exact
    q = np.zeros(c.shape, np.uint64)
    for k in range(3):
        ext = np.float64(hi[k]) - np.float64(lo[k])
        if ext > 0:
            f = np.floor((c[:, k].astype(np.float64) - np.float64(lo[k])) / ext * 1024.0)
            q[:, k] = np.minimum(1023.0, f).astype(np.uint64)
    morton = (spread3(q[:, 0]) << np.uint64(2)) | (spread3(q[:, 1]) << np.uint64(1)) | spread3(q[:, 2])
    return np.sort((morton << np.uint64(32)) | real.astype(np.uint64))


def build(soa):
    real = np.nonzero(soa["inv_radius"] != 0)[0]
    assert len(real) < 1 << 28
    keys = sorted_keys(soa, real) if len(real) else np.zeros(0, np.uint64)
    ids = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
    blo, bhi = sphere_boxes(soa, real) if len(real) else (np.zeros((0, 3), np.float32),) * 2
    pos = np.zeros(len(soa["cx"]), np.int64)
    pos[real] = np.arange(len(real))
    slo, shi = blo[pos[ids]], bhi[pos[ids]]                              # boxes in sorted order
    m = len(keys)
    exact = np.stack([soa["cx"], soa["cy"], soa["cz"], soa["radius_sq"]], 1).astype(np.float32)

    leaves = np.zeros(m, BVH_LEAF)
    nodes = np.zeros(max(m, 1), BVH_NODE)                                # preorder; fewer than m are used
    used = [0]
    depth = [1]

    def new_node():
        used[0] += 1
        return used[0] - 1

    def put_slot(node, slot, lo, hi, ref):
        nodes["lo%d" % slot][node], nodes["hi%d" % slot][node] = lo, hi
        nodes["child"][node, slot] = ref
        d2 = 0.0
        for k in range(3):
            w = np.float64(hi[k]) - np.float64(lo[k])
            d2 = d2 + w * w
        nodes["diag"][node, slot] = round_up(np.sqrt(d2) * DIAG_PAD)

    def leaf(a, b):
        """records of sorted positions [a, b), ascending sphere index; returns the child reference and the box"""
        order = np.sort(ids[a:b])
        leaves["exact"][a:b] = exact[order]
        leaves["index"][a:b] = order
        return np.int32(~np.int32((a << 3) | (b - a))), slo[a:b].min(0), shi[a:b].max(0)

    def child(a, b, d):
        """the subtree of sorted positions [a, b) below an inner node at depth d - 1"""
        if b - a <= LEAF_MAX:
            return leaf(a, b)
        return inner(a, b, d)

    def inner(a, b, d):
        me = new_node()
        depth[0] = max(depth[0], d)
        bit = int(keys[a] ^ keys[b - 1]).bit_length() - 1               # highest differing bit
        split = a + int(np.searchsorted((keys[a:b] >> np.uint64(bit)) & np.uint64(1), 1))
        r0, lo0, hi0 = child(a, split, d + 1)
        r1, lo1, hi1 = child(split, b, d + 1)
        put_slot(me, 0, lo0, hi0, r0)
        put_slot(me, 1, lo1, hi1, r1)
        return me, np.minimum(lo0, lo1), np.maximum(hi0, hi1)

    if m > LEAF_MAX:
        inner(0, m, 1)
    else:
        root = new_node()
        nodes["child"][root] = -1
        if m:
            ref, lo, hi = leaf(0, m)
            put_slot(root, 0, lo, hi, ref)
    return nodes[:used[0]].copy(), leaves, depth[0]
