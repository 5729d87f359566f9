// r1_bvh.h -- host builder of the bounding volume hierarchy of R1_VARIANT_MEGAKERNEL_BVH (DESIGN.md section 4.8).
//
// A binned-SAH BVH2 over the spheres that can be hit (inv_radius != 0), built single-threaded in double precision.  The build is
// a function of the scene alone: two builds of one scene give the same bytes.
//
//   node (64 B):  lo0[3] hi0[3] lo1[3] hi1[3]   the boxes of child 0 and child 1
//                 child[2]                      >= 0: index of an inner node; < 0: leaf, ~child = first record << 3 | count
//                                               (count 1 .. kLeafMax; ~child == 0, i.e. child == kEmpty: no child)
//                 diag[2]                       upper bound on the length of each box's diagonal
//   leaf record (32 B):  {cx, cy, cz, radius_sq} bit-equal to the scene's exact record, original sphere index, 3 x 0
//
// Node 0 is the root.  Its own box is not stored (every ray tests its two children).  A leaf's records are in ascending index
// order.  Each sphere's box is [c - rp, c + rp] with rp = sqrt(radius_sq) (1 + 2^-16), the exact bounds rounded outward to float
// (box_lo / box_hi); an inner box is the union of its spheres' boxes.  The traversal widens every box per ray (r1_device.cuh,
// bvh_child): the two together contain every point the exact test can accept, DESIGN.md section 4.8 derives the bound.
//
// Depth: the root is at depth 1; no inner node is deeper than kMaxDepth, which is also the traversal stack size.  Where the SAH
// split would leave a child that a halving build could no longer fit under kMaxDepth, the node splits at the object median
// instead, and spheres whose centres coincide split by index order.  Both halve the count, so the bound holds for any scene of
// fewer than 2^62 spheres.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

namespace r1 {
namespace bvh {

constexpr int kMaxDepth = 64;      // inner-node depth bound = traversal stack entries
constexpr int kLeafMax = 4;        // spheres per leaf
constexpr int kBins = 16;          // SAH bins per axis
constexpr int32_t kEmpty = -1;     // child reference of a missing child (a root with fewer than two children)
constexpr double kRadiusPad = 1.0 + 1.0 / 65536.0;

struct Node {
    float lo0[3], hi0[3], lo1[3], hi1[3];
    int32_t child[2];
    float diag[2];
};
static_assert(sizeof(Node) == 64, "one node = 64 bytes = 4 float4");

struct LeafRec {
    float cx, cy, cz, radius_sq;
    int32_t index, pad[3];
};
static_assert(sizeof(LeafRec) == 32, "one leaf record = 32 bytes = 2 float4");

struct Bvh {
    std::vector<Node> nodes;
    std::vector<LeafRec> leaves;
    uint32_t depth = 0;            // deepest inner node (root = 1)
};

inline int32_t leaf_ref(uint32_t first, uint32_t count) { return (int32_t)~((first << 3) | count); }

namespace detail {

struct Box {
    double lo[3], hi[3];
    Box() { for (int k = 0; k < 3; ++k) { lo[k] = std::numeric_limits<double>::infinity(); hi[k] = -std::numeric_limits<double>::infinity(); } }
    void grow(const Box &b) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], b.lo[k]); hi[k] = std::max(hi[k], b.hi[k]); } }
    double area() const
    {
        const double x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
        return x * y + y * z + z * x;
    }
};

inline float round_down(double v)
{
    float f = (float)v;
    if ((double)f > v) f = std::nextafter(f, -std::numeric_limits<float>::infinity());
    return f;
}
inline float round_up(double v)
{
    float f = (float)v;
    if ((double)f < v) f = std::nextafter(f, std::numeric_limits<float>::infinity());
    return f;
}
// The float below / above the exact c - rp / c + rp (rp >= 0).  The double sum rounds; its exact error (Knuth's TwoSum) says on
// which side of it the exact value lies.  Without it, rp below half a double ulp of c (|c| above 2^53 rp) gave the box [c, c].
inline float box_lo(float c, double rp)
{
    const double v = (double)c - rp, bv = v - (double)c, err = ((double)c - (v - bv)) + (-rp - bv);
    float f = round_down(v);
    if ((double)f == v && err < 0) f = std::nextafter(f, -std::numeric_limits<float>::infinity());
    return f;
}
inline float box_hi(float c, double rp)
{
    const double v = (double)c + rp, bv = v - (double)c, err = ((double)c - (v - bv)) + (rp - bv);
    float f = round_up(v);
    if ((double)f == v && err > 0) f = std::nextafter(f, std::numeric_limits<float>::infinity());
    return f;
}

// levels of inner nodes a halving build needs for n spheres
inline int halving_levels(size_t n)
{
    int h = 0;
    while (n > (size_t)kLeafMax) { n = (n + 1) / 2; ++h; }
    return h;
}

struct Builder {
    const float *cx, *cy, *cz, *r2;
    std::vector<Box> box;              // per sphere: float box, held in double
    std::vector<uint32_t> ids;
    Bvh *out;

    double centre(uint32_t i, int k) const { return k == 0 ? cx[i] : k == 1 ? cy[i] : cz[i]; }

    Box range_box(size_t b, size_t e) const
    {
        Box r;
        for (size_t j = b; j < e; ++j) r.grow(box[ids[j]]);
        return r;
    }

    // builds ids[b, e) below an inner node at depth `depth - 1`; returns the child reference and its box
    int32_t build(size_t b, size_t e, int depth, Box &bb)
    {
        bb = range_box(b, e);
        const size_t n = e - b;
        if (n <= (size_t)kLeafMax) {
            std::sort(ids.begin() + (long)b, ids.begin() + (long)e);
            const uint32_t first = (uint32_t)out->leaves.size();
            for (size_t j = b; j < e; ++j) {
                const uint32_t i = ids[j];
                LeafRec rec;
                memset(&rec, 0, sizeof(rec));
                rec.cx = cx[i]; rec.cy = cy[i]; rec.cz = cz[i]; rec.radius_sq = r2[i]; rec.index = (int32_t)i;
                out->leaves.push_back(rec);
            }
            return leaf_ref(first, (uint32_t)n);
        }
        const uint32_t me = (uint32_t)out->nodes.size();
        out->nodes.push_back(Node());
        out->depth = std::max(out->depth, (uint32_t)depth);
        const size_t mid = split(b, e, depth);
        Box lb, rb;
        const int32_t l = build(b, mid, depth + 1, lb);
        const int32_t r = build(mid, e, depth + 1, rb);
        set_child(me, 0, l, lb);
        set_child(me, 1, r, rb);
        return (int32_t)me;
    }

    void set_child(uint32_t node, int slot, int32_t ref, const Box &b)
    {
        Node &nd = out->nodes[node];
        float *lo = slot ? nd.lo1 : nd.lo0, *hi = slot ? nd.hi1 : nd.hi0;
        double d2 = 0;
        for (int k = 0; k < 3; ++k) {
            lo[k] = (float)b.lo[k];                                       // sphere boxes are floats: their unions are exact
            hi[k] = (float)b.hi[k];
            d2 += (b.hi[k] - b.lo[k]) * (b.hi[k] - b.lo[k]);
        }
        nd.child[slot] = ref;
        nd.diag[slot] = round_up(std::sqrt(d2) * (1.0 + 1e-12));
    }

    // partitions ids[b, e) (e - b > kLeafMax) and returns the split point; the inner node being split is at `depth`
    size_t split(size_t b, size_t e, int depth)
    {
        const size_t n = e - b;
        double cmin[3], cmax[3];
        for (int k = 0; k < 3; ++k) { cmin[k] = std::numeric_limits<double>::infinity(); cmax[k] = -cmin[k]; }
        for (size_t j = b; j < e; ++j)
            for (int k = 0; k < 3; ++k) { const double c = centre(ids[j], k); cmin[k] = std::min(cmin[k], c); cmax[k] = std::max(cmax[k], c); }
        int widest = 0;
        for (int k = 1; k < 3; ++k) if (cmax[k] - cmin[k] > cmax[widest] - cmin[widest]) widest = k;
        if (!(cmax[widest] - cmin[widest] > 0)) {                         // all centres coincide: split by index order
            std::sort(ids.begin() + (long)b, ids.begin() + (long)e);
            return b + (n + 1) / 2;
        }
        // binned SAH: cost(split) = area(left) * n_left + area(right) * n_right; ties keep the lowest axis and plane
        const int room = kMaxDepth - depth;                               // child inner nodes may sit at depth + 1 .. kMaxDepth
        double best = std::numeric_limits<double>::infinity();
        int best_axis = -1, best_plane = -1;
        for (int k = 0; k < 3; ++k) {
            const double ext = cmax[k] - cmin[k];
            if (!(ext > 0)) continue;
            Box bins[kBins];
            size_t cnt[kBins] = {};
            for (size_t j = b; j < e; ++j) {
                const int bi = bin_of(centre(ids[j], k), cmin[k], ext);
                bins[bi].grow(box[ids[j]]);
                ++cnt[bi];
            }
            double right_area[kBins];
            size_t right_cnt[kBins];
            Box acc;
            size_t c = 0;
            for (int i = kBins - 1; i > 0; --i) { acc.grow(bins[i]); c += cnt[i]; right_area[i] = c ? acc.area() : 0.0; right_cnt[i] = c; }
            Box left;
            size_t lc = 0;
            for (int i = 0; i < kBins - 1; ++i) {
                left.grow(bins[i]);
                lc += cnt[i];
                const size_t rc = right_cnt[i + 1];
                if (lc == 0 || rc == 0) continue;
                if (halving_levels(lc) > room || halving_levels(rc) > room) continue;
                const double cost = left.area() * (double)lc + right_area[i + 1] * (double)rc;
                if (cost < best) { best = cost; best_axis = k; best_plane = i; }
            }
        }
        if (best_axis >= 0) {
            const int k = best_axis, plane = best_plane;
            const double lo = cmin[k], ext = cmax[k] - cmin[k];
            auto it = std::stable_partition(ids.begin() + (long)b, ids.begin() + (long)e,
                                            [&](uint32_t i) { return bin_of(centre(i, k), lo, ext) <= plane; });
            return (size_t)(it - ids.begin());
        }
        // object median on the widest axis, ties by index: halves the count, so the subtree fits in halving_levels(n)
        const size_t mid = b + (n + 1) / 2;
        const int k = widest;
        std::nth_element(ids.begin() + (long)b, ids.begin() + (long)mid, ids.begin() + (long)e, [&](uint32_t x, uint32_t y) {
            const double a = centre(x, k), c = centre(y, k);
            return a < c || (a == c && x < y);
        });
        return mid;
    }

    static int bin_of(double c, double lo, double ext)
    {
        const double f = (c - lo) / ext * kBins;
        return f >= kBins - 1 ? kBins - 1 : (f <= 0 ? 0 : (int)f);
    }
};

}  // namespace detail

// Builds the BVH of the n spheres (the scene's SoA).  Spheres with inv_radius == 0 are left out: they can never be hit
// (rayweek1.cpp:288-292; the placeholders r1_scene_pad adds and radius <= 0).  Returns false if the scene is too large for the
// 28-bit leaf-record field of a child reference.
inline bool build(const float *cx, const float *cy, const float *cz, const float *radius_sq, const float *inv_radius, uint32_t n, Bvh &out)
{
    out = Bvh();
    detail::Builder bld;
    bld.cx = cx; bld.cy = cy; bld.cz = cz; bld.r2 = radius_sq; bld.out = &out;
    bld.box.resize(n);
    for (uint32_t i = 0; i < n; ++i) {
        if (inv_radius[i] == 0) continue;
        bld.ids.push_back(i);
        const double rp = std::sqrt((double)radius_sq[i]) * kRadiusPad;
        const double c[3] = { cx[i], cy[i], cz[i] };
        for (int k = 0; k < 3; ++k) { bld.box[i].lo[k] = detail::box_lo((float)c[k], rp); bld.box[i].hi[k] = detail::box_hi((float)c[k], rp); }
    }
    if (bld.ids.size() >= (1u << 28)) return false;
    out.nodes.reserve(bld.ids.size() / 2 + 1);
    out.leaves.reserve(bld.ids.size());
    out.nodes.push_back(Node());                                      // the root is always an inner node
    memset(&out.nodes[0], 0, sizeof(Node));
    out.depth = 1;
    const size_t n_real = bld.ids.size();
    if (n_real <= (size_t)kLeafMax) {                                 // one leaf (or none) under the root
        out.nodes[0].child[0] = out.nodes[0].child[1] = kEmpty;
        if (n_real) {
            detail::Box bb;
            const int32_t ref = bld.build(0, n_real, 2, bb);
            bld.set_child(0, 0, ref, bb);
        }
        return true;
    }
    const size_t mid = bld.split(0, n_real, 1);
    detail::Box lb, rb;
    const int32_t l = bld.build(0, mid, 2, lb);
    const int32_t r = bld.build(mid, n_real, 2, rb);
    bld.set_child(0, 0, l, lb);
    bld.set_child(0, 1, r, rb);
    return true;
}

}  // namespace bvh
}  // namespace r1
