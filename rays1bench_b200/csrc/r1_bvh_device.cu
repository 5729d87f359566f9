// r1_bvh_device.cu -- device builder of the BVH of R1_VARIANT_MEGAKERNEL_BVH: a linear BVH (DESIGN.md section 4.9).
//
// Morton codes of the sphere centres, one radix sort, Karras' binary radix tree (HPG 2012) over the sorted keys, collapsed to
// leaves of <= 4 spheres, refit bottom-up and numbered in depth-first preorder.  The output has r1_bvh.h's layout and the same
// box and diagonal arithmetic, so the traversal (bvh_trace) and its correctness argument are unchanged.  The tree is a function
// of the scene alone, specified step by step below, and tests/lbvh_restatement.py restates it on the CPU bit for bit:
//
//   1. box of a real sphere (inv_radius != 0): rp = sqrt((double)r2) (1 + 2^-16), [c - rp, c + rp] exactly, rounded outward to float
//   2. q_k = ext_k > 0 ? min(1023, floor((c_k - lo_k) / ext_k * 1024)) : 0 over the centroid bounds [lo, hi] of the real spheres,
//      ext_k = hi_k - lo_k, in double; morton = interleave(x -> bit 3b + 2, y -> 3b + 1, z -> 3b)
//   3. key = morton << 32 | sphere index: unique, sorted ascending over bits [0, 62)
//   4. radix tree: every inner node splits its sorted range at the highest differing key bit
//   5. a node of <= 4 spheres is a leaf (records in sorted order, re-sorted by sphere index within the leaf); the root stays inner
//   6. boxes are unions of sphere boxes; diag = round_up(sqrt(sum_k (hi_k - lo_k)^2) (1 + 1e-12)), k = 0, 1, 2 in that order
//   7. inner nodes in preorder, child 0 (the lower keys) first; leaf `first` = the leaf's first position in sorted order
//
// Every double operation is an explicit _rn intrinsic: nvcc would otherwise contract a product and a sum into an FMA, which
// the host builder and the restatement do not.
#include "r1_bvh_device.h"

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/rays1_b200.h"
#include "r1_bvh.h"
#include "r1_internal.h"

namespace r1 {
namespace lbvh {

constexpr int kThreads = 256;
constexpr int kMortonBits = 30;
constexpr int kKeyBits = kMortonBits + 32;        // sort over [0, 62)

// Read back by the host between phases.
struct Header {
    unsigned int error;                 // a real sphere with a non-finite centre or radius_sq
    unsigned int n_real;                // real spheres = leaf records
    unsigned int cursor;                // key slots handed out
    unsigned int depth;                 // deepest kept inner node (root = 1)
    unsigned int bounds[6];             // centroid lo[3] (ordered-uint min), hi[3] (ordered-uint max)
};

// float -> uint with the same order (-0 sorts below +0; min / max of the floats are exact either way)
__device__ __forceinline__ unsigned int ordered(float f)
{
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unordered(unsigned int u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

__device__ __forceinline__ bool finite4(float4 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w); }

// step 1: the padded box of a sphere, [box_lo(c_k, rp), box_hi(c_k, rp)] per axis with rp = padded_radius(radius_sq)
__device__ __forceinline__ double padded_radius(float r2) { return __dmul_rn(__dsqrt_rn((double)r2), bvh::kRadiusPad); }
// (directed in both steps: the float below / above the exact c -+ rp, even where rp is below half a double ulp of c)
__device__ __forceinline__ float box_lo(float c, double rp) { return __double2float_rd(__dsub_rd((double)c, rp)); }
__device__ __forceinline__ float box_hi(float c, double rp) { return __double2float_ru(__dadd_ru((double)c, rp)); }

// step 1 for every sphere; centroid bounds and the real-sphere count
__global__ void __launch_bounds__(kThreads) lbvh_boxes(const float4 *__restrict__ exact, const float4 *__restrict__ shade, uint32_t n,
                                                       float4 *__restrict__ box, Header *hdr)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (shade[2 * (size_t)i + 1].x == 0.0f) return;               // inv_radius == 0: never hit, not in the tree
    const float4 e = exact[i];
    if (!finite4(e)) { atomicOr(&hdr->error, 1u); return; }
    const double rp = padded_radius(e.w);
    const float c[3] = { e.x, e.y, e.z };
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) {
        lo[k] = box_lo(c[k], rp);
        hi[k] = box_hi(c[k], rp);
        atomicMin(&hdr->bounds[k], ordered(c[k]));
        atomicMax(&hdr->bounds[3 + k], ordered(c[k]));
    }
    box[2 * (size_t)i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
    box[2 * (size_t)i + 1] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    atomicAdd(&hdr->n_real, 1u);
}

__device__ __forceinline__ uint32_t quantise(float c, float lo, float hi)
{
    const double ext = __dsub_rn((double)hi, (double)lo);
    if (!(ext > 0.0)) return 0;
    const double f = floor(__dmul_rn(__ddiv_rn(__dsub_rn((double)c, (double)lo), ext), 1024.0));
    return f >= 1023.0 ? 1023u : (uint32_t)f;                      // f >= 0: c >= lo
}

__device__ __forceinline__ uint32_t spread3(uint32_t v)           // bit b -> bit 3b
{
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

// steps 2-3: one key per real sphere, in any slot order (the sort orders them; keys are unique)
__global__ void __launch_bounds__(kThreads) lbvh_keys(const float4 *__restrict__ exact, const float4 *__restrict__ shade, uint32_t n,
                                                      Header *hdr, unsigned long long *__restrict__ keys)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (shade[2 * (size_t)i + 1].x == 0.0f) return;
    const float4 e = exact[i];
    if (!finite4(e)) return;                                       // refused after lbvh_boxes
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) { lo[k] = unordered(hdr->bounds[k]); hi[k] = unordered(hdr->bounds[3 + k]); }
    const uint32_t m = (spread3(quantise(e.x, lo[0], hi[0])) << 2) | (spread3(quantise(e.y, lo[1], hi[1])) << 1) | spread3(quantise(e.z, lo[2], hi[2]));
    const uint32_t slot = atomicAdd(&hdr->cursor, 1u);
    keys[slot] = ((unsigned long long)m << 32) | i;
}

// Radix tree over m >= 2 sorted keys: inner nodes 0 .. m - 2 (0 = root), key leaves m - 1 + j.  Per inner node: its two children,
// its range [first, last]; per node: its parent.
struct Tree {
    int2 *child;                        // m - 1
    int2 *range;                        // m - 1: first, last
    int *parent;                        // 2m - 1 (root: -1)
    float4 *box;                        // 2m - 1 x 2: lo, hi
    int *kept;                          // 2m - 1: kept inner nodes in the subtree (a node of > kLeafMax keys is kept)
    unsigned int *arrivals;             // m - 1, zeroed
};

__device__ __forceinline__ int delta(const unsigned long long *keys, int m, int i, int j)
{
    return (j < 0 || j >= m) ? -1 : __clzll(keys[i] ^ keys[j]);
}

// step 4: Karras (HPG 2012, Fig. 4), one thread per inner node
__global__ void __launch_bounds__(kThreads) lbvh_hierarchy(const unsigned long long *__restrict__ keys, int m, Tree t)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m - 1) return;
    const int d = delta(keys, m, i, i + 1) > delta(keys, m, i, i - 1) ? 1 : -1;
    const int dmin = delta(keys, m, i, i - d);
    int lmax = 2;
    while (delta(keys, m, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int s = lmax / 2; s >= 1; s /= 2)
        if (delta(keys, m, i, i + (l + s) * d) > dmin) l += s;
    const int j = i + l * d;
    const int dnode = delta(keys, m, i, j);
    int s = 0, step = l;
    do {
        step = (step + 1) >> 1;
        if (delta(keys, m, i, i + (s + step) * d) > dnode) s += step;
    } while (step > 1);
    const int split = i + s * d + min(d, 0);
    const int first = min(i, j), last = max(i, j);
    const int left = first == split ? m - 1 + split : split;
    const int right = last == split + 1 ? m - 1 + split + 1 : split + 1;
    t.child[i] = make_int2(left, right);
    t.range[i] = make_int2(first, last);
    t.parent[left] = i;
    t.parent[right] = i;
    if (i == 0) t.parent[0] = -1;
}

// step 6 (boxes) and the kept-subtree sizes step 7 numbers by: Karras' refit, one thread per key leaf; at every inner node the
// second arriving child continues and the first exits.  Float min / max are exact, so no result depends on arrival order.
__global__ void __launch_bounds__(kThreads) lbvh_refit(const unsigned long long *__restrict__ keys, int m, const float4 *__restrict__ sphere_box, Tree t)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t idx = (uint32_t)keys[j];
    int v = m - 1 + j;
    __stcg(&t.box[2 * v], sphere_box[2 * (size_t)idx]);
    __stcg(&t.box[2 * v + 1], sphere_box[2 * (size_t)idx + 1]);
    __stcg(&t.kept[v], 0);
    for (;;) {
        const int p = __ldcg(&t.parent[v]);
        if (p < 0) return;
        __threadfence();
        if (atomicAdd(&t.arrivals[p], 1u) == 0) return;         // the sibling is not done yet: it continues from p
        __threadfence();
        const int2 c = __ldcg(&t.child[p]);
        const float4 l0 = __ldcg(&t.box[2 * c.x]), h0 = __ldcg(&t.box[2 * c.x + 1]);
        const float4 l1 = __ldcg(&t.box[2 * c.y]), h1 = __ldcg(&t.box[2 * c.y + 1]);
        __stcg(&t.box[2 * p], make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.0f));
        __stcg(&t.box[2 * p + 1], make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.0f));
        const int2 r = __ldcg(&t.range[p]);
        __stcg(&t.kept[p], (r.y - r.x + 1 > bvh::kLeafMax ? 1 : 0) + __ldcg(&t.kept[c.x]) + __ldcg(&t.kept[c.y]));
        v = p;
    }
}

// r1_bvh.h's set_child: the bound on the diagonal of a slot's box
__device__ __forceinline__ float diag_bound(float4 lo, float4 hi)
{
    const double wx = __dsub_rn((double)hi.x, (double)lo.x), wy = __dsub_rn((double)hi.y, (double)lo.y), wz = __dsub_rn((double)hi.z, (double)lo.z);
    double d2 = __dmul_rn(wx, wx);
    d2 = __dadd_rn(d2, __dmul_rn(wy, wy));
    d2 = __dadd_rn(d2, __dmul_rn(wz, wz));
    return __double2float_ru(__dmul_rn(__dsqrt_rn(d2), 1.0 + 1e-12));
}

// one 64-byte node {lo0, hi0, lo1, hi1, child[2], diag[2]}; an empty slot (ref kEmpty) is all zero but its reference
__device__ __forceinline__ void put_node(float4 *node, float4 lo0, float4 hi0, int32_t ref0, float4 lo1, float4 hi1, int32_t ref1)
{
    const float d0 = ref0 == bvh::kEmpty ? 0.0f : diag_bound(lo0, hi0), d1 = ref1 == bvh::kEmpty ? 0.0f : diag_bound(lo1, hi1);
    node[0] = make_float4(lo0.x, lo0.y, lo0.z, hi0.x);
    node[1] = make_float4(hi0.y, hi0.z, lo1.x, lo1.y);
    node[2] = make_float4(lo1.z, hi1.x, hi1.y, hi1.z);
    node[3] = make_float4(__int_as_float(ref0), __int_as_float(ref1), d0, d1);
}

__device__ __forceinline__ void order2(uint32_t &a, uint32_t &b) { const uint32_t x = min(a, b); b = max(a, b); a = x; }

// the records of a leaf over sorted positions [first, first + count): the scene's exact records, ascending sphere index
__device__ __forceinline__ int32_t put_leaf(const unsigned long long *keys, const float4 *exact, int first, int count, float4 *leaves)
{
    uint32_t id[bvh::kLeafMax];
#pragma unroll
    for (int a = 0; a < bvh::kLeafMax; ++a) id[a] = a < count ? (uint32_t)keys[first + a] : 0xffffffffu;
    order2(id[0], id[1]); order2(id[2], id[3]); order2(id[0], id[2]); order2(id[1], id[3]); order2(id[1], id[2]);   // sorting network
#pragma unroll
    for (int a = 0; a < bvh::kLeafMax; ++a) {
        if (a < count) {
            leaves[2 * (size_t)(first + a)] = exact[id[a]];
            leaves[2 * (size_t)(first + a) + 1] = make_float4(__int_as_float((int)id[a]), 0.0f, 0.0f, 0.0f);
        }
    }
    return (int32_t)~(((uint32_t)first << 3) | (uint32_t)count);   // bvh::leaf_ref
}

// step 7: one thread per kept inner node finds its preorder number and depth from the path to the root, then writes its node
// and the records of its leaf children
__global__ void __launch_bounds__(kThreads) lbvh_emit(const unsigned long long *__restrict__ keys, int m, const float4 *__restrict__ exact,
                                                      Tree t, float4 *__restrict__ nodes, float4 *__restrict__ leaves, Header *hdr)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m - 1) return;
    const int2 r = t.range[i];
    if (r.y - r.x + 1 <= bvh::kLeafMax) return;                   // collapsed into a leaf of its parent
    int number = 0, depth = 1;
    for (int v = i; v != 0; ++depth) {
        const int p = t.parent[v];
        const int2 c = t.child[p];
        number += c.x == v ? 1 : 1 + t.kept[c.x];
        v = p;
    }
    atomicMax(&hdr->depth, (unsigned int)depth);
    const int2 c = t.child[i];
    int32_t ref[2];
#pragma unroll
    for (int slot = 0; slot < 2; ++slot) {
        const int v = slot ? c.y : c.x;
        const int2 rv = v < m - 1 ? t.range[v] : make_int2(v - (m - 1), v - (m - 1));
        if (rv.y - rv.x + 1 > bvh::kLeafMax) ref[slot] = slot ? number + 1 + t.kept[c.x] : number + 1;
        else ref[slot] = put_leaf(keys, exact, rv.x, rv.y - rv.x + 1, leaves);
    }
    put_node(nodes + 4 * (size_t)number, t.box[2 * c.x], t.box[2 * c.x + 1], ref[0], t.box[2 * c.y], t.box[2 * c.y + 1], ref[1]);
}

// step 5's root of 0 .. kLeafMax real spheres: one leaf in slot 0 (none for 0 spheres), slot 1 empty and zero
__global__ void lbvh_small_root(const unsigned long long *__restrict__ keys, int m, const float4 *__restrict__ exact, const float4 *__restrict__ sphere_box,
                                float4 *__restrict__ nodes, float4 *__restrict__ leaves, Header *hdr)
{
    const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    hdr->depth = 1;
    if (m == 0) { put_node(nodes, zero, zero, bvh::kEmpty, zero, zero, bvh::kEmpty); return; }
    const float inf = __int_as_float(0x7f800000);
    float4 lo = make_float4(inf, inf, inf, 0.0f), hi = make_float4(-inf, -inf, -inf, 0.0f);
    for (int j = 0; j < m; ++j) {
        const uint32_t idx = (uint32_t)keys[j];
        const float4 a = sphere_box[2 * (size_t)idx], b = sphere_box[2 * (size_t)idx + 1];
        lo = make_float4(fminf(lo.x, a.x), fminf(lo.y, a.y), fminf(lo.z, a.z), 0.0f);
        hi = make_float4(fmaxf(hi.x, b.x), fmaxf(hi.y, b.y), fmaxf(hi.z, b.z), 0.0f);
    }
    put_node(nodes, lo, hi, put_leaf(keys, exact, 0, m, leaves), zero, zero, bvh::kEmpty);
}

// ---- refit (DESIGN.md section 4.10): new boxes and leaf records for moved spheres, same topology ---------------------------------
//
// Works on any tree in r1_bvh.h's layout, whichever builder made it and however its nodes are numbered (node 0 is the root).  Every
// slot whose child is not kEmpty gets the float union of the padded boxes (step 1) of the spheres under it and its diagonal bound;
// every leaf record gets the scene's new exact record.  Empty slots and child references keep their bytes.

// parent[v] = p << 1 | slot for every node v referenced by slot `slot` of node p; the root keeps the -1 it was filled with
__global__ void __launch_bounds__(kThreads) refit_parents(const float4 *__restrict__ nodes, uint32_t n_nodes, int *__restrict__ parent)
{
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    const float4 c = nodes[4 * (size_t)v + 3];
    const int32_t ref[2] = { __float_as_int(c.x), __float_as_int(c.y) };
    for (int slot = 0; slot < 2; ++slot)
        if (ref[slot] >= 0) parent[ref[slot]] = (int)(v << 1) | slot;
}

// writes a slot's box and diagonal bound; 4-byte stores, because the two slots of a node share float4s and may be written by two threads
__device__ __forceinline__ void put_slot(float4 *node, int slot, float4 lo, float4 hi)
{
    float *f = reinterpret_cast<float *>(node);
    __stcg(f + 6 * slot + 0, lo.x); __stcg(f + 6 * slot + 1, lo.y); __stcg(f + 6 * slot + 2, lo.z);
    __stcg(f + 6 * slot + 3, hi.x); __stcg(f + 6 * slot + 4, hi.y); __stcg(f + 6 * slot + 5, hi.z);
    __stcg(f + 14 + slot, diag_bound(lo, hi));
}

__device__ __forceinline__ void get_slot(const float4 *node, int slot, float4 &lo, float4 &hi)
{
    const float *f = reinterpret_cast<const float *>(node);
    lo = make_float4(__ldcg(f + 6 * slot + 0), __ldcg(f + 6 * slot + 1), __ldcg(f + 6 * slot + 2), 0.0f);
    hi = make_float4(__ldcg(f + 6 * slot + 3), __ldcg(f + 6 * slot + 4), __ldcg(f + 6 * slot + 5), 0.0f);
}

__device__ __forceinline__ int inner_children(int32_t r0, int32_t r1) { return (r0 >= 0 ? 1 : 0) + (r1 >= 0 ? 1 : 0); }

// One thread per node: the boxes of its leaf slots (and their records), then an arrival at the node.  A node is complete after 1 +
// (its inner children) arrivals; the last arriving thread writes the node's box into its parent's slot and arrives there.  No thread
// waits for another, and float min / max are exact, so the arrival order cannot show.
__global__ void __launch_bounds__(kThreads) refit_nodes(float4 *__restrict__ nodes, float4 *__restrict__ leaves, uint32_t n_nodes,
                                                       const float4 *__restrict__ exact, const int *__restrict__ parent, unsigned int *arrivals)
{
    const uint32_t v0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (v0 >= n_nodes) return;
    const float inf = __int_as_float(0x7f800000);
    {
        float4 *node = nodes + 4 * (size_t)v0;
        const float4 c = node[3];
        const int32_t ref[2] = { __float_as_int(c.x), __float_as_int(c.y) };
        for (int slot = 0; slot < 2; ++slot) {
            if (ref[slot] >= 0 || ref[slot] == bvh::kEmpty) continue;
            const uint32_t v = ~(uint32_t)ref[slot], first = v >> 3, count = v & 7u;
            float4 lo = make_float4(inf, inf, inf, 0.0f), hi = make_float4(-inf, -inf, -inf, 0.0f);
            for (uint32_t a = 0; a < count; ++a) {
                const size_t rec = first + a;
                const float4 e = exact[__float_as_int(leaves[2 * rec + 1].x)];
                leaves[2 * rec] = e;
                const double rp = padded_radius(e.w);
                lo = make_float4(fminf(lo.x, box_lo(e.x, rp)), fminf(lo.y, box_lo(e.y, rp)), fminf(lo.z, box_lo(e.z, rp)), 0.0f);
                hi = make_float4(fmaxf(hi.x, box_hi(e.x, rp)), fmaxf(hi.y, box_hi(e.y, rp)), fmaxf(hi.z, box_hi(e.z, rp)), 0.0f);
            }
            put_slot(node, slot, lo, hi);
        }
    }
    for (uint32_t v = v0;;) {
        const float4 *node = nodes + 4 * (size_t)v;
        const int32_t r0 = __float_as_int(__ldcg(reinterpret_cast<const float *>(node) + 12)), r1 = __float_as_int(__ldcg(reinterpret_cast<const float *>(node) + 13));
        __threadfence();
        if (atomicAdd(&arrivals[v], 1u) != (unsigned int)inner_children(r0, r1)) return;   // not the last arrival
        __threadfence();
        const int p = __ldcg(&parent[v]);
        if (p < 0) return;                                         // the root: its own box is not stored
        // the union of the node's used slots; an empty slot (kEmpty) holds zeros, not a box, and is left out whichever slot it is
        float4 lo = make_float4(inf, inf, inf, 0.0f), hi = make_float4(-inf, -inf, -inf, 0.0f);
        for (int slot = 0; slot < 2; ++slot) {
            if ((slot ? r1 : r0) == bvh::kEmpty) continue;
            float4 l, h;
            get_slot(node, slot, l, h);
            lo = make_float4(fminf(lo.x, l.x), fminf(lo.y, l.y), fminf(lo.z, l.z), 0.0f);
            hi = make_float4(fmaxf(hi.x, h.x), fmaxf(hi.y, h.y), fmaxf(hi.z, h.z), 0.0f);
        }
        put_slot(nodes + 4 * (size_t)(p >> 1), p & 1, lo, hi);
        v = (uint32_t)(p >> 1);
    }
}

#define R1_LBVH_CUDA(expr)                                                                                   \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess) return r1_set_error(R1_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

namespace {
struct Scratch {                        // one cudaMalloc, freed on every path out of build()
    void *p = nullptr;
    ~Scratch() { if (p) cudaFree(p); }
    template <typename T> T *as() { return static_cast<T *>(p); }
};
}  // namespace

// Three phases with a read-back after each of the first two: the real-sphere count sizes the sort, the kept-node count sizes the
// tree's block.  Scratch is allocated per build: this is set-up, not a render.
int build(const float4 *exact, const float4 *shade, uint32_t n, Built *out, double *ms)
{
    PhaseTimer tm;
    Scratch d_hdr, d_sbox;
    R1_LBVH_CUDA(cudaMalloc(&d_hdr.p, sizeof(Header)));
    R1_LBVH_CUDA(cudaMalloc(&d_sbox.p, (size_t)n * 32 + 16));
    Header h;
    memset(&h, 0, sizeof(h));
    for (int k = 0; k < 3; ++k) h.bounds[k] = 0xffffffffu;
    R1_LBVH_CUDA(cudaMemcpy(d_hdr.p, &h, sizeof(h), cudaMemcpyHostToDevice));
    Header *hdr = d_hdr.as<Header>();
    const float4 *sbox = d_sbox.as<float4>();
    const unsigned blocks_n = (n + kThreads - 1) / kThreads;

    // phase 1: sphere boxes, centroid bounds, real-sphere count
    R1_LBVH_CUDA(tm.start());
    if (n) lbvh_boxes<<<blocks_n, kThreads>>>(exact, shade, n, d_sbox.as<float4>(), hdr);
    R1_LBVH_CUDA(cudaGetLastError());
    R1_LBVH_CUDA(tm.stop());
    R1_LBVH_CUDA(cudaMemcpy(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost));
    if (h.error) return r1_set_error(R1_ERR_ARG, "a sphere that can be hit has a non-finite centre or radius_sq");
    if (h.n_real >= (1u << 28)) return r1_set_error(R1_ERR_LIMIT, "the bvh takes fewer than 2^28 spheres that can be hit");
    const int m = (int)h.n_real;
    const bool tree = m > bvh::kLeafMax;                          // else the root holds one leaf (or none)

    Scratch d_keys, d_sorted, d_temp, d_child, d_range, d_parent, d_box, d_kept, d_arrivals;
    R1_LBVH_CUDA(cudaMalloc(&d_keys.p, (size_t)m * 8 + 16));
    R1_LBVH_CUDA(cudaMalloc(&d_sorted.p, (size_t)m * 8 + 16));
    size_t temp_bytes = 0;
    R1_LBVH_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, d_keys.as<unsigned long long>(), d_sorted.as<unsigned long long>(), m, 0, kKeyBits));
    R1_LBVH_CUDA(cudaMalloc(&d_temp.p, temp_bytes + 16));
    Tree t;
    memset(&t, 0, sizeof(t));
    if (tree) {
        R1_LBVH_CUDA(cudaMalloc(&d_child.p, (size_t)(m - 1) * 8));
        R1_LBVH_CUDA(cudaMalloc(&d_range.p, (size_t)(m - 1) * 8));
        R1_LBVH_CUDA(cudaMalloc(&d_parent.p, (size_t)(2 * m - 1) * 4));
        R1_LBVH_CUDA(cudaMalloc(&d_box.p, (size_t)(2 * m - 1) * 32));
        R1_LBVH_CUDA(cudaMalloc(&d_kept.p, (size_t)(2 * m - 1) * 4));
        R1_LBVH_CUDA(cudaMalloc(&d_arrivals.p, (size_t)(m - 1) * 4));
        R1_LBVH_CUDA(cudaMemset(d_arrivals.p, 0, (size_t)(m - 1) * 4));
        t.child = d_child.as<int2>(); t.range = d_range.as<int2>(); t.parent = d_parent.as<int>(); t.box = d_box.as<float4>();
        t.kept = d_kept.as<int>(); t.arrivals = d_arrivals.as<unsigned int>();
    }
    const unsigned long long *keys = d_sorted.as<unsigned long long>();
    const unsigned blocks_m = (m + kThreads - 1) / kThreads;

    // phase 2: keys, sort, radix tree, refit
    R1_LBVH_CUDA(tm.start());
    if (m > 0) {
        lbvh_keys<<<blocks_n, kThreads>>>(exact, shade, n, hdr, d_keys.as<unsigned long long>());
        R1_LBVH_CUDA(cudaGetLastError());
        R1_LBVH_CUDA(cub::DeviceRadixSort::SortKeys(d_temp.p, temp_bytes, d_keys.as<unsigned long long>(), d_sorted.as<unsigned long long>(), m, 0, kKeyBits));
    }
    if (tree) {
        lbvh_hierarchy<<<blocks_m, kThreads>>>(keys, m, t);
        R1_LBVH_CUDA(cudaGetLastError());
        lbvh_refit<<<blocks_m, kThreads>>>(keys, m, sbox, t);
        R1_LBVH_CUDA(cudaGetLastError());
    }
    R1_LBVH_CUDA(tm.stop());
    uint32_t n_nodes = 1;
    if (tree) R1_LBVH_CUDA(cudaMemcpy(&n_nodes, t.kept, 4, cudaMemcpyDeviceToHost));   // kept nodes under the root, inner node 0

    // phase 3: nodes in preorder and leaf records, into the tree's own block
    Scratch blk;
    const size_t nb = (size_t)n_nodes * sizeof(bvh::Node), lb = (size_t)m * sizeof(bvh::LeafRec);
    R1_LBVH_CUDA(cudaMalloc(&blk.p, nb + lb + 16));
    float4 *nodes = blk.as<float4>(), *leaves = reinterpret_cast<float4 *>(static_cast<unsigned char *>(blk.p) + nb);
    R1_LBVH_CUDA(tm.start());
    if (tree) lbvh_emit<<<blocks_m, kThreads>>>(keys, m, exact, t, nodes, leaves, hdr);
    else lbvh_small_root<<<1, 1>>>(keys, m, exact, sbox, nodes, leaves, hdr);
    R1_LBVH_CUDA(cudaGetLastError());
    R1_LBVH_CUDA(tm.stop());
    R1_LBVH_CUDA(cudaMemcpy(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost));
    // 62 at most (DESIGN.md section 4.9); checked because the traversal stack holds kMaxDepth entries
    if (h.depth > (uint32_t)bvh::kMaxDepth) return r1_set_error(R1_ERR_LIMIT, "bvh depth %u exceeds %d", h.depth, bvh::kMaxDepth);
    *out = Built{ blk.p, n_nodes, (uint32_t)m, h.depth };
    blk.p = nullptr;
    if (ms) *ms = tm.ms;
    return R1_OK;
}

int refit(float4 *nodes, float4 *leaves, uint32_t n_nodes, const float4 *exact, int *parent, unsigned int *arrivals, bool parents_ready, cudaStream_t stream)
{
    const unsigned blocks = (n_nodes + kThreads - 1) / kThreads;
    if (!parents_ready) {
        R1_LBVH_CUDA(cudaMemsetAsync(parent, 0xff, (size_t)n_nodes * sizeof(int), stream));
        refit_parents<<<blocks, kThreads, 0, stream>>>(nodes, n_nodes, parent);
        R1_LBVH_CUDA(cudaGetLastError());
    }
    R1_LBVH_CUDA(cudaMemsetAsync(arrivals, 0, (size_t)n_nodes * sizeof(unsigned int), stream));
    refit_nodes<<<blocks, kThreads, 0, stream>>>(nodes, leaves, n_nodes, exact, parent, arrivals);
    R1_LBVH_CUDA(cudaGetLastError());
    return R1_OK;
}

}  // namespace lbvh
}  // namespace r1
