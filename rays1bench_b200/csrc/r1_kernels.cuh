// r1_kernels.cuh -- sm_100a kernels of the Rays1 trace loop: persistent-thread megakernel, framebuffer resolve,
// parity kernels and the FP32 FMA peak microbenchmark.  (The wavefront variant lives in r1_wavefront.cuh.)
// file:line citations are relative to /root/reference/.
#pragma once
#include "r1_device.cuh"
#include "r1_tensor.cuh"

namespace r1 {

constexpr unsigned kFull = 0xffffffffu;

// Work decomposition.  The persistent megakernels: work items are single samples g = lp * spp + s, handed to WARPS 32..2048
// at a time from one 64-bit counter (the warp sample pool, WarpPool below).  The wavefront variant: unit
// u = lp * n_chunks + c = `samples_per_unit` consecutive samples of one pixel (1 sample for spp <= 256), handed to LANES from a
// 32-bit counter.  Either way every finished sample is added to its pixel's accumulator in 64-bit FIXED POINT (2^-24) with a
// fire-and-forget atomic (RED.ADD.64).  Integer addition is associative: the sums, and therefore the RGB8 image, are
// bit-identical for every GPU count, CTA shape, scheduling and kernel variant, whatever order the samples arrive in.
// (The reference sums floats sequentially per pixel, rayweek1.cpp:757-765; radiance per sample is in [0, 1], so 24
// fractional bits lose < 3e-8 per sample -- float32 itself resolves no better near 1 -- and 2^20 samples fit with room.)
struct RenderArgs {
    DevScene scene;
    unsigned long long *accum;       // npix_local x 4 (r, g, b, -): sum of per-sample radiance * 2^24
    unsigned long long *num_rays;    // += one per traced ray (rayweek1.cpp:517)
    unsigned int *unit_counter;      // next unit to hand out
    uint8_t *rgb;                    // npix_local * 3, local rows packed, row 0 = bottom
    int32_t width, height, spp, max_bounces;
    int32_t rank, world, row_tile;
    uint32_t npix_local, n_units;
    int32_t samples_per_unit, n_chunks;
    float inv_w, inv_h, inv_spp;
    uint64_t seed;                   // Rng::seed_hash(global seed)
    uint64_t magic_chunks, magic_width, magic_row_tile;  // floor(2^64 / d) + 1: exact n / d for 32-bit n via one 64-bit mul-high (0 when d == 1)
    uint32_t sched_kmax, sched_div;      // guided self-scheduling: min(kmax, max(1, left / (lanes * div))) x 32 samples per warp
                                         // per atomic (the sample pool)
    // sample-pool scheduling (megakernel_pool): work items are single samples g = lp * spp + s, handed out 32 at a time
    unsigned long long *sample_counter;  // next sample to hand out (64-bit: 3840 x 2160 x 1024 = 8.5e9 samples)
    uint64_t n_samples, magic_spp;       // npix_local * spp; floor(2^64 / spp) + 1 (exact g / spp for g < 2^64 / spp; 0 when spp == 1)
};

// The BVH megakernel_pool<kScanBvh> traverses (r1_bvh.h): written on the launching stream before every launch of that kernel
// (r1_core.cu).  It is not a RenderArgs field because the wavefront kernels take a second parameter behind RenderArgs, whose
// offset -- and so their code -- would change with its size.
struct BvhArgs { const float4 *nodes, *leaves; };
__constant__ BvhArgs c_bvh;

// A batch of views (r1_render_views): the kernels' kViews instances render K images of one scene as one work space of
// K x npix local pixels, batch pixel plp = v * npix + lp.  View v's camera and hashed seed come from table[v]; everything past the
// primary ray -- pool entries, accumulators, resolve -- carries plp and never needs v.  Written on the launching stream before
// every batch launch, for the reason c_bvh is.
struct ViewRec { Camera cam; uint64_t seed; };   // the 22 constants; Rng::seed_hash(seed of the view)
static_assert(sizeof(ViewRec) == 96, "view records are loaded as six float4");
struct ViewArgs {
    const ViewRec *table;
    uint32_t npix;                    // local pixels of one view
    uint64_t magic_npix;              // div_magic(npix)
};
__constant__ ViewArgs c_views;

constexpr int kSmemSpheres = 16 + R1_RSQRT12_ENTRIES * 2;   // megakernel: byte offset of the staged spheres (mbarrier, rsqrtss table first)
constexpr float kFixedScale = 16777216.0f;                 // 2^24: one sample saturates at 2^32 - 1 (radiance 256; scenes stay <= 1)
constexpr float kFixedInvScale = 5.9604644775390625e-8f;   // 2^-24

// n / d for n, d < 2^32 with the precomputed magic (d == 1 -> magic 0)
__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint64_t magic) { return magic ? (uint32_t)__umul64hi((uint64_t)n, magic) : n; }
__host__ inline uint64_t div_magic(uint32_t d) { return d <= 1 ? 0ull : (~0ull / d) + 1ull; }

// ------------------------------------------------------------------------------------------------ TMA staging
// One 1-D bulk copy (cp.async.bulk -> UBLKCP) brings [scan | exact] = n_pad * 32 bytes into shared memory; an
// mbarrier with a transaction count signals arrival.  Every CTA reads the same <= 128 KB, which stays L2-resident.
__device__ __forceinline__ void stage_spheres(const DevScene &sc, float4 *s_spheres, uint64_t *bar)
{
    const uint32_t bytes = (uint32_t)sc.n_pad * 32u;
    const uint32_t bar_s = (uint32_t)__cvta_generic_to_shared(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(s_spheres)),
                     "l"(sc.scan), "r"(bytes), "r"(bar_s)
                     : "memory");
    }
    __syncthreads();  // barrier initialised before anyone polls it
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done)
                     : "r"(bar_s)
                     : "memory");
    }
}

// y of local row lr under the interleaved row-tile partition (tile k -> rank k % world)
__device__ __host__ __forceinline__ int global_row(int lr, int row_tile, int rank, int world)
{
    return ((lr / row_tile) * world + rank) * row_tile + (lr % row_tile);
}

// ------------------------------------------------------------------------------------------------ shared path steps
// The three steps of the per-path state machine, shared by the megakernel and the wavefront kernels so that both
// execute the same instructions on the same values (bit-identical images).

// unit -> (local pixel, global pixel, first sample, end sample)
__device__ __forceinline__ void unit_begin(const RenderArgs &a, uint32_t unit, uint32_t &lp, uint32_t &pixel, float &fx, float &fy, int &s, int &s_end)
{
    lp = fast_div(unit, a.magic_chunks);
    const uint32_t c = unit - lp * (uint32_t)a.n_chunks;
    const uint32_t lr = fast_div(lp, a.magic_width);
    const int x = (int)(lp - lr * (uint32_t)a.width);
    const uint32_t tile = fast_div(lr, a.magic_row_tile);                        // global_row() without the integer divisions
    const int y = (int)((tile * (uint32_t)a.world + (uint32_t)a.rank) * (uint32_t)a.row_tile + (lr - tile * (uint32_t)a.row_tile));
    pixel = (uint32_t)y * (uint32_t)a.width + (uint32_t)x;
    fx = (float)x; fy = (float)y;
    s = (int)c * a.samples_per_unit;
    s_end = min(s + a.samples_per_unit, a.spp);
}

// one finished sample -> the pixel's fixed-point accumulator (order-free, see RenderArgs)
__device__ __forceinline__ uint32_t quantise_radiance(float c)
{
    // cvt.rni.u32.f32 saturates: NaN (a degenerate path: zero-length scatter direction) and negatives become 0, anything above
    // 2^32 / 2^24 = 256 becomes 2^32 - 1 -- no clamp instructions needed, and 2^20 samples of at most 2^32 fit the 64-bit sums
    return __float2uint_rn(c * kFixedScale);
}
__device__ __forceinline__ void accumulate_quantised(const RenderArgs &a, uint32_t lp, uint32_t r, uint32_t g, uint32_t b)
{
    unsigned long long *dst = a.accum + (size_t)lp * 4;
    atomicAdd(dst + 0, (unsigned long long)r);
    atomicAdd(dst + 1, (unsigned long long)g);
    atomicAdd(dst + 2, (unsigned long long)b);
}
__device__ __forceinline__ void accumulate_sample(const RenderArgs &a, uint32_t lp, f3 c)
{
    accumulate_quantised(a, lp, quantise_radiance(c.x), quantise_radiance(c.y), quantise_radiance(c.z));
}

// total-rays counter (rayweek1.cpp:809-813): warp reduce, one 64-bit atomic per warp
__device__ __forceinline__ void count_rays(const RenderArgs &a, uint32_t nrays, unsigned lane)
{
    unsigned long long total = nrays;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) total += __shfl_xor_sync(kFull, total, off);
    if (lane == 0 && total) atomicAdd(a.num_rays, total);
}

// start sample s of a pixel: jitter (rayweek1.cpp:759), lens disk + camera ray (:760, :381-386); seed = Rng::seed_hash(global seed)
__device__ __forceinline__ void primary_ray(const RenderArgs &a, const Camera &cam, uint64_t seed, uint32_t pixel, float fx, float fy, int s,
                                            const uint16_t *__restrict__ tab, Rng &rng, f3 &o, f3 &d)
{
    rng.seed(pixel, (uint32_t)s, seed);
    const float u = fmul(fadd(rng.rand01(0), fx), a.inv_w), v = fmul(fadd(rng.rand01(1), fy), a.inv_h);
    float px, py;
    random_in_unit_disk(rng, 2, px, py);
    camera_ray(cam, u, v, px, py, tab, o, d);
}
// the render's own camera and seed
__device__ __forceinline__ void primary_ray(const RenderArgs &a, uint32_t pixel, float fx, float fy, int s, const uint16_t *__restrict__ tab, Rng &rng, f3 &o,
                                            f3 &d)
{
    primary_ray(a, a.scene.cam, a.seed, pixel, fx, fy, s, tab, rng, o, d);
}

// color() body after hit() (rayweek1.cpp:515-536).  Returns true when the path ends (contrib = its radiance);
// otherwise o / d / thr / depth hold the scattered ray.  `e` is the hit sphere's exact record.
__device__ __forceinline__ bool shade_step(const RenderArgs &a, int hit, float t, float4 e, const uint16_t *__restrict__ tab, f3 &o, f3 &d, f3 &thr, int &depth,
                                           const Rng &rng, f3 &contrib)
{
    contrib = mk3(0, 0, 0);
    if (hit < 0) {
        const f3 sk = sky(d);
        contrib = mk3(fmul(thr.x, sk.x), fmul(thr.y, sk.y), fmul(thr.z, sk.z));
        return true;
    }
    if (depth >= a.max_bounces) return true;   // :523 -- no scatter (and no RNG draw) past the cap
    f3 p, n, atten, nd, rs = mk3(0, 0, 0);
    float ru = 0.0f;
    const ShadeRec sh = load_shade(a.scene, hit);
    hit_finalise(e, sh.inv_radius, o, d, t, p, n);
    const int kind = sh.kind;
    const float4 mat = sh.mat;
    // One code path for every material: draw 0 of this bounce is Dielectric's coin AND the radius variable of the unit-ball
    // sample Lambertian / Metal use (a dielectric hit throws its ball sample away).  Branching on the material first made the
    // warp run the ~50 instructions of the ball sample once per material present in it.
    const uint32_t draw0 = kDrawsPrimary + kDrawsPerBounce * (uint32_t)depth;
    ru = rng.rand01(draw0);
    rs = random_in_unit_sphere(rng, draw0, ru);
    if (!scatter(kind, mat, sh.inv_ior, sh.r0s, d, p, n, rs, ru, tab, atten, nd)) return true;
    thr = mk3(fmul(thr.x, atten.x), fmul(thr.y, atten.y), fmul(thr.z, atten.z));
    o = p; d = nd; ++depth;
    return false;
}

// ------------------------------------------------------------------------------------------------ megakernel, warp sample pool
// Persistent CTAs; every lane runs  loop { take a sample | SCAN | shade }  so that all 32 lanes enter every scan with a live
// ray and divergence is confined to the short take / shade steps.
// Replaces render_tile + color + TileRenderScheduler (rayweek1.cpp:722-842, 515-536).
// kScan: which Hitable::hit implementation the lanes run
enum ScanKind { kScanCoop = 0, kScanLanePacked = 1, kScanLaneScalar = 2, kScanLaneDeferred = 3, kScanBvh = 4 };   // kScanBvh: megakernel_pool only
__host__ __device__ constexpr int scan_filter(int kScan) { return kScan == kScanLaneScalar ? 0 : 1; }

// The START of a path is taken out of the divergent part.  A lane that fetched its own next sample and generated its primary
// ray at once would do so together with whichever other lanes happen to finish in the same iteration: 12 of 32 lanes on the
// large scene, so the ~300 instructions of fetch + decode + RNG seeding + jitter + lens sample + Camera::getRay would be paid
// at 37 % occupancy in every iteration (round 1's lane-fetch scheduling, DESIGN.md section 4.1).
// Here each WARP keeps a pool of up to 32 ready-made primary rays in shared memory.  When the lanes in need outnumber the pool,
// the whole warp produces the next 32 consecutive samples at once -- one atomicAdd per 32 samples, every lane busy -- and a
// finishing lane just pops a ray (ballot + popc ranks, three 16-byte loads).  Work items are single samples (no unit ranges:
// the path state has no unit / sample bookkeeping, registers the scan loop can use), numbered g = lp * spp + s in 64 bits.
// Which lane traces which sample is irrelevant to the result: RNG streams are keyed by (pixel, sample) and the accumulators are
// integer sums -- the image is bit-identical to the other variants'.
// Every persistent kernel takes its work this way, and all of them produce through pool_produce.
// megakernel_tc3 and megakernel_tcs pop through pool_take; megakernel_pool writes the same pop out (faster there), and
// megakernel_pool2, which ranks two slots per lane, pops on its own.
struct __align__(16) WarpPool {
    float4 a[32];                     // origin.xyz, local pixel index (uint bits; kPoolInvalid = past the end of the work)
    float4 b[32];                     // direction.xyz, rng key word 0 (uint bits)
    uint32_t k1[32];                  // rng key word 1
};
constexpr uint32_t kPoolInvalid = 0xffffffffu;

// The producer side of a warp's pool; warp-uniform.
struct PoolState {
    bool dry;                         // the sample counter has run past the end
    uint32_t ready;                   // rays in the pool, entries [0, ready)
    // The warp's private range of samples [w_next, w_end).  Scan-heavy scenes take 32 samples per atomic; small scenes, where a
    // scan is a few hundred instructions and one atomic per 32 samples would saturate the counter's L2 line, take up to
    // sched_kmax x 32, shrinking as left / (sched_div x lanes) so that the last warps finish together.
    unsigned long long w_next, w_end;
};

// The whole warp produces the next 32 consecutive samples into its pool (every lane has popped what it takes from it): takes a
// new range when its own is used up, decodes sample g = lp * spp + s under the interleaved row-tile partition and generates the
// primary ray.  lanes_x = lanes of the grid x sched_div.  kViews: plp is a batch pixel (c_views), decoded per lane -- the 32
// samples of a warp can straddle a view boundary.
template <bool kViews>
__device__ __forceinline__ void pool_produce(const RenderArgs &a, WarpPool &pool, PoolState &ps, const uint16_t *tab, unsigned lane, uint32_t lanes_x)
{
    __syncwarp();
    if (ps.w_next >= ps.w_end) {
        unsigned long long base = 0;
        uint32_t k = 1;
        if (lane == 0) {
            const unsigned long long left = a.n_samples > ps.w_end ? a.n_samples - ps.w_end : 0ull;
            const unsigned long long want_k = left / lanes_x;
            k = want_k >= a.sched_kmax ? a.sched_kmax : (want_k < 1 ? 1u : (uint32_t)want_k);
            base = atomicAdd(a.sample_counter, 32ull * k);
        }
        base = __shfl_sync(kFull, base, 0);
        k = __shfl_sync(kFull, k, 0);
        ps.w_next = base;
        ps.w_end = base + 32ull * k < a.n_samples ? base + 32ull * k : a.n_samples;
    }
    if (ps.w_next >= a.n_samples) {
        ps.dry = true;
        ps.ready = 0;
    } else {
        const unsigned long long g = ps.w_next + lane;
        ps.w_next += 32;
        float4 pa = make_float4(0, 0, 0, __uint_as_float(kPoolInvalid)), pb = make_float4(0, 0, 0, 0);
        uint32_t pk1 = 0;
        if (g < a.n_samples) {
            const uint32_t plp = a.magic_spp ? (uint32_t)__umul64hi(g, a.magic_spp) : (uint32_t)g;
            const uint32_t smp = (uint32_t)(g - (unsigned long long)plp * (uint32_t)a.spp);
            uint32_t lp = plp, v = 0;
            if constexpr (kViews) {
                v = fast_div(plp, c_views.magic_npix);
                lp = plp - v * c_views.npix;
            }
            const uint32_t lr = fast_div(lp, a.magic_width);
            const int x = (int)(lp - lr * (uint32_t)a.width);
            const uint32_t tile = fast_div(lr, a.magic_row_tile);
            const int y = (int)((tile * (uint32_t)a.world + (uint32_t)a.rank) * (uint32_t)a.row_tile + (lr - tile * (uint32_t)a.row_tile));
            Rng r;
            f3 po, pd;
            if constexpr (kViews) {
                union { float4 q[6]; ViewRec rec; } vr;
                const float4 *src = reinterpret_cast<const float4 *>(c_views.table + v);
#pragma unroll
                for (int k = 0; k < 6; ++k) vr.q[k] = __ldg(src + k);
                primary_ray(a, vr.rec.cam, vr.rec.seed, (uint32_t)y * (uint32_t)a.width + (uint32_t)x, (float)x, (float)y, (int)smp, tab, r, po, pd);
            } else {
                primary_ray(a, (uint32_t)y * (uint32_t)a.width + (uint32_t)x, (float)x, (float)y, (int)smp, tab, r, po, pd);
            }
            pa = make_float4(po.x, po.y, po.z, __uint_as_float(plp));
            pb = make_float4(pd.x, pd.y, pd.z, __uint_as_float(r.k0));
            pk1 = r.k1;
        }
        pool.a[lane] = pa; pool.b[lane] = pb; pool.k1[lane] = pk1;
        ps.ready = 32;
    }
    __syncwarp();
}

// Lanes without a path (`want`, ballot `need`) take a ray from the warp's pool; the warp produces more when the pool runs short.
// A lane that finds the work exhausted keeps its o / d.
template <bool kViews>
__device__ __forceinline__ void pool_take(const RenderArgs &a, WarpPool &pool, PoolState &ps, const uint16_t *tab, unsigned lane, unsigned lt_mask,
                                          uint32_t lanes_x, unsigned need, bool want, bool &active, bool &exhausted, f3 &o, f3 &d, uint32_t &lp, Rng &rng,
                                          f3 &thr, int &depth)
{
    const uint32_t n_need = (uint32_t)__popc(need), rank = (uint32_t)__popc(need & lt_mask);
    int entry = -1;
    if (want && rank < ps.ready) entry = (int)(ps.ready - 1u - rank);
    const uint32_t n_first = min(n_need, ps.ready);
    float4 ea = make_float4(0, 0, 0, __uint_as_float(kPoolInvalid)), eb = make_float4(0, 0, 0, 0);
    uint32_t ek1 = 0;
    if (entry >= 0) { ea = pool.a[entry]; eb = pool.b[entry]; ek1 = pool.k1[entry]; }   // pop before the pool is overwritten
    if (n_need > ps.ready && !ps.dry) {                          // warp-uniform: not enough rays
        pool_produce<kViews>(a, pool, ps, tab, lane, lanes_x);
        const uint32_t rank2 = rank - n_first;                   // rank among the lanes the old pool could not serve
        if (want && entry < 0 && rank2 < ps.ready) {
            entry = (int)(ps.ready - 1u - rank2);
            ea = pool.a[entry]; eb = pool.b[entry]; ek1 = pool.k1[entry];
        }
        ps.ready -= min(n_need - n_first, ps.ready);
    } else {                                                     // the pool serves everybody (or there is nothing left to produce)
        ps.ready -= n_first;
    }
    if (want) {
        if (entry >= 0 && __float_as_uint(ea.w) != kPoolInvalid) {
            o = mk3(ea.x, ea.y, ea.z); d = mk3(eb.x, eb.y, eb.z); lp = __float_as_uint(ea.w);
            rng.k0 = __float_as_uint(eb.w); rng.k1 = ek1;
            thr = mk3(1, 1, 1); depth = 0; active = true;
        } else {
            exhausted = true;                                    // past the end of the work
        }
    }
}

template <int kScan, bool kStaged, int kThreads, int kBlocksPerSM, bool kViews>
__global__ void __launch_bounds__(kThreads, kBlocksPerSM) megakernel_pool(const __grid_constant__ RenderArgs a)
{
    // shared memory: [mbarrier 16 B | rsqrtss table 4 KB | staged spheres n_pad * 32 B | per-warp scan scratch (coop / deferred) | per-warp pools]
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint16_t *s_tab = reinterpret_cast<uint16_t *>(smem_raw + 16);
    for (int i = threadIdx.x; i < R1_RSQRT12_ENTRIES / 2; i += kThreads)
        reinterpret_cast<uint32_t *>(s_tab)[i] = reinterpret_cast<const uint32_t *>(g_rsqrt12)[i];
    const float4 *s_scan, *s_exact;
    if (kStaged) {
        float4 *s_spheres = reinterpret_cast<float4 *>(smem_raw + kSmemSpheres);
        stage_spheres(a.scene, s_spheres, reinterpret_cast<uint64_t *>(smem_raw));   // its __syncthreads also publishes the table
        s_scan = s_spheres;
        s_exact = s_spheres + a.scene.n_pad;
    } else {  // scenes beyond the staging limit scan straight from global memory (L1/L2 resident)
        s_scan = a.scene.scan;
        s_exact = a.scene.exact;
        __syncthreads();
    }
    const uint16_t *tab = s_tab;
    const int n_pad = a.scene.n_pad;
    const unsigned lane = threadIdx.x & 31u, lt_mask = (1u << lane) - 1u;
    constexpr bool kScratch = kScan == kScanCoop || kScan == kScanLaneDeferred;
    unsigned char *after_spheres = smem_raw + kSmemSpheres + (kStaged ? (size_t)n_pad * 32 : 0);
    WarpScratch *ws = reinterpret_cast<WarpScratch *>(after_spheres) + (threadIdx.x >> 5);
    WarpPool &pool = reinterpret_cast<WarpPool *>(after_spheres + (kScratch ? sizeof(WarpScratch) * (kThreads / 32) : 0))[threadIdx.x >> 5];

    bool active = false, exhausted = false;
    PoolState ps;
    ps.dry = false; ps.ready = 0; ps.w_next = 0; ps.w_end = 0;
    const uint32_t lanes_x = gridDim.x * blockDim.x * a.sched_div;
    uint32_t lp = 0, nrays = 0;
    int depth = 0;
    f3 thr = mk3(1, 1, 1);
    f3 o = mk3(0.0f, 1.0e18f, 0.0f), d = mk3(0.0f, 0.0f, 0.0f);  // idle lanes scan a ray that passes no filter
    Rng rng;
    rng.k0 = 0; rng.k1 = 0;

    for (;;) {
        // -- lanes without a path take a ray from the warp's pool; the warp produces more when the pool runs short.  pool_take's
        //    logic, written out: through pool_take this kernel measured 0.8-3.4 % slower on B200 (DESIGN.md section 4.12)
        const bool want = !active && !exhausted;
        const unsigned need = __ballot_sync(kFull, want);
        if (need) {
            const uint32_t n_need = (uint32_t)__popc(need), rank = (uint32_t)__popc(need & lt_mask);
            int entry = -1;                                      // pool entry this lane pops
            if (want && rank < ps.ready) entry = (int)(ps.ready - 1u - rank);
            const uint32_t n_first = min(n_need, ps.ready);
            if (n_need > ps.ready && !ps.dry) {                  // warp-uniform: not enough rays
                float4 ea = make_float4(0, 0, 0, 0), eb = make_float4(0, 0, 0, 0);
                uint32_t ek1 = 0;
                if (entry >= 0) { ea = pool.a[entry]; eb = pool.b[entry]; ek1 = pool.k1[entry]; }   // pop before the pool is overwritten
                pool_produce<kViews>(a, pool, ps, tab, lane, lanes_x);
                const uint32_t rank2 = rank - n_first;           // rank among the lanes the old pool could not serve
                if (want && entry < 0 && rank2 < ps.ready) {
                    entry = (int)(ps.ready - 1u - rank2);
                    ea = pool.a[entry]; eb = pool.b[entry]; ek1 = pool.k1[entry];
                }
                ps.ready -= min(n_need - n_first, ps.ready);
                if (want) {
                    if (entry >= 0 && __float_as_uint(ea.w) != kPoolInvalid) {
                        o = mk3(ea.x, ea.y, ea.z); d = mk3(eb.x, eb.y, eb.z); lp = __float_as_uint(ea.w);
                        rng.k0 = __float_as_uint(eb.w); rng.k1 = ek1;
                        thr = mk3(1, 1, 1); depth = 0; active = true;
                    } else {
                        exhausted = true;                        // past the end of the work
                        o = mk3(0.0f, 1.0e18f, 0.0f); d = mk3(0.0f, 0.0f, 0.0f);
                    }
                }
            } else {                                             // the pool serves everybody (or there is nothing left to produce)
                ps.ready -= n_first;
                if (want) {
                    bool got = false;
                    if (entry >= 0) {
                        const float4 ea = pool.a[entry], eb = pool.b[entry];
                        if (__float_as_uint(ea.w) != kPoolInvalid) {
                            o = mk3(ea.x, ea.y, ea.z); d = mk3(eb.x, eb.y, eb.z); lp = __float_as_uint(ea.w);
                            rng.k0 = __float_as_uint(eb.w); rng.k1 = pool.k1[entry];
                            thr = mk3(1, 1, 1); depth = 0; active = true; got = true;
                        }
                    }
                    if (!got) {
                        exhausted = true;
                        o = mk3(0.0f, 1.0e18f, 0.0f); d = mk3(0.0f, 0.0f, 0.0f);
                    }
                }
            }
        }
        if (__all_sync(kFull, exhausted)) break;

        // -- Hitable::hit (rayweek1.cpp:152-339): uniform trip count, all lanes
        float t = kTMax;
        int hit = -1;
        if (kScan == kScanCoop) scan_coop<(kThreads <= 512 ? 2 : 1)>(*ws, s_scan, s_exact, n_pad, o, d, kTMin, kTMax, t, hit);
        else if (kScan == kScanLaneDeferred) scan_deferred(*reinterpret_cast<DeferScratch *>(ws), s_scan, s_exact, a.scene.n8, o, d, kTMin, kTMax, t, hit);
        else if (kScan == kScanBvh) { if (active) bvh_trace(c_bvh.nodes, c_bvh.leaves, o, d, kTMin, t, hit); }   // idle lanes do not traverse
        else scan<scan_filter(kScan)>(s_scan, s_exact, a.scene.n8, o, d, kTMin, t, hit);

        // -- color() body (rayweek1.cpp:515-536)
        if (active) {
            ++nrays;
            f3 contrib;
            const float4 e = hit >= 0 ? s_exact[hit] : make_float4(0, 0, 0, 0);
            if (shade_step(a, hit, t, e, tab, o, d, thr, depth, rng, contrib)) {
                accumulate_sample(a, lp, contrib);
                active = false;
                o = mk3(0.0f, 1.0e18f, 0.0f); d = mk3(0.0f, 0.0f, 0.0f);    // (overwritten by the pop at the top of the loop)
            }
        }
    }
    count_rays(a, nrays, lane);
}

// ------------------------------------------------------------------------------------------------ megakernel, two paths per lane
// megakernel_pool with TWO paths per lane (R1_VARIANT_MEGAKERNEL_DUAL): both rays of a lane are tested against every sphere load,
// so the chunk loop issues 32 LDS.128 per 64 ray-sphere tests instead of per 32 (181 instead of 202 instructions per 32 tests),
// and a warp carries two independent FFMA2 streams.  The path state is 13 registers per path since the sample pool took the unit
// bookkeeping out, so two paths fit a 768-thread CTA (80 registers) where round 1's two-path kernel needed 128 registers and 512
// threads.  Everything else -- pool, production, shading, accumulators -- is megakernel_pool's; same bytes out.
// Measured on B200: large 6095 (768 threads) / 6054 (512) against 6178 Mrays/s for one path per lane at 1024 threads, 4096-sphere
// scene 820 against 825, medium 32.7 G against 34.1 G: the chunk loop is bound by the FMA pipe (FFMA2 / FADD2 issue), not by the
// LDS count, so the saved loads buy nothing and the lower occupancy costs a little.  Kept as an A/B variant only.
template <bool kStaged, int kThreads, int kBlocksPerSM>
__global__ void __launch_bounds__(kThreads, kBlocksPerSM) megakernel_pool2(const __grid_constant__ RenderArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint16_t *s_tab = reinterpret_cast<uint16_t *>(smem_raw + 16);
    for (int i = threadIdx.x; i < R1_RSQRT12_ENTRIES / 2; i += kThreads)
        reinterpret_cast<uint32_t *>(s_tab)[i] = reinterpret_cast<const uint32_t *>(g_rsqrt12)[i];
    const float4 *s_scan, *s_exact;
    if (kStaged) {
        float4 *s_spheres = reinterpret_cast<float4 *>(smem_raw + kSmemSpheres);
        stage_spheres(a.scene, s_spheres, reinterpret_cast<uint64_t *>(smem_raw));
        s_scan = s_spheres;
        s_exact = s_spheres + a.scene.n_pad;
    } else {
        s_scan = a.scene.scan;
        s_exact = a.scene.exact;
        __syncthreads();
    }
    const uint16_t *tab = s_tab;
    const unsigned lane = threadIdx.x & 31u, lt_mask = (1u << lane) - 1u;
    WarpPool &pool = reinterpret_cast<WarpPool *>(smem_raw + kSmemSpheres + (kStaged ? (size_t)a.scene.n_pad * 32 : 0))[threadIdx.x >> 5];

    bool active[2] = { false, false };
    PoolState ps;
    ps.dry = false; ps.ready = 0; ps.w_next = 0; ps.w_end = 0;
    const uint32_t lanes_x = gridDim.x * blockDim.x * a.sched_div;
    uint32_t lp[2] = { 0, 0 }, nrays = 0;
    int depth[2] = { 0, 0 };
    f3 thr[2] = { mk3(1, 1, 1), mk3(1, 1, 1) };
    f3 o[2] = { mk3(0.0f, 1.0e18f, 0.0f), mk3(0.0f, 1.0e18f, 0.0f) }, d[2] = { mk3(0, 0, 0), mk3(0, 0, 0) };
    Rng rng[2];
    rng[0].k0 = rng[0].k1 = rng[1].k0 = rng[1].k1 = 0;

    for (;;) {
        // -- refill: slot 0 of every lane first, then slot 1 (ranks over the 64 slots of the warp)
        const unsigned need0 = __ballot_sync(kFull, !active[0]), need1 = __ballot_sync(kFull, !active[1]);
        if (need0 | need1) {
            const uint32_t n0 = (uint32_t)__popc(need0), n_need = n0 + (uint32_t)__popc(need1);
            const uint32_t rank[2] = { (uint32_t)__popc(need0 & lt_mask), n0 + (uint32_t)__popc(need1 & lt_mask) };
            uint32_t served = 0;                                 // warp-uniform: slots with rank < served have been handled
            for (;;) {
                const uint32_t avail = ps.ready;
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (!active[r] && rank[r] >= served && rank[r] < served + avail) {
                        const int entry = (int)(avail - 1u - (rank[r] - served));
                        const float4 ea = pool.a[entry], eb = pool.b[entry];
                        if (__float_as_uint(ea.w) != kPoolInvalid) {
                            o[r] = mk3(ea.x, ea.y, ea.z); d[r] = mk3(eb.x, eb.y, eb.z); lp[r] = __float_as_uint(ea.w);
                            rng[r].k0 = __float_as_uint(eb.w); rng[r].k1 = pool.k1[entry];
                            thr[r] = mk3(1, 1, 1); depth[r] = 0; active[r] = true;
                        }
                    }
                }
                const uint32_t take = min(avail, n_need - served);
                ps.ready -= take;
                served += avail;
                if (served >= n_need || ps.dry) break;
                pool_produce<false>(a, pool, ps, tab, lane, lanes_x);   // everything in the pool has been popped: ready == 0
                if (ps.dry) break;
            }
#pragma unroll
            for (int r = 0; r < 2; ++r)
                if (!active[r]) { o[r] = mk3(0.0f, 1.0e18f, 0.0f); d[r] = mk3(0.0f, 0.0f, 0.0f); }   // nothing left for this slot
        }
        // the warp is done when the work has run dry, the pool is empty and no slot holds a path
        if (ps.dry && ps.ready == 0 && __all_sync(kFull, !active[0] && !active[1])) break;

        // -- Hitable::hit for both rays against the same sphere loads
        float t[2] = { kTMax, kTMax };
        int hit[2] = { -1, -1 };
        scan_dual(s_scan, s_exact, a.scene.n8, o, d, kTMin, t, hit);

        // -- color() body for each live path
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            if (active[r]) {
                ++nrays;
                f3 contrib;
                const float4 e = hit[r] >= 0 ? s_exact[hit[r]] : make_float4(0, 0, 0, 0);
                if (shade_step(a, hit[r], t[r], e, tab, o[r], d[r], thr[r], depth[r], rng[r], contrib)) {
                    accumulate_sample(a, lp[r], contrib);
                    active[r] = false;
                }
            }
        }
    }
    count_rays(a, nrays, lane);
}

// ------------------------------------------------------------------------------------------------ megakernel, tensor-core filter
// R1_VARIANT_MEGAKERNEL_TENSOR (DESIGN.md section 4.0): the path state machine of megakernel_pool with the filter on the tensor
// cores (r1_tensor.cuh).  CTA = kGroups ray groups of 128 threads (4 warps, warp w of a group owns TMEM lanes 32 w .. 32 w + 31,
// one ray per lane).  Per scan every thread writes its ray's lifted TF32 row into the group's A tile, and the scene's B tile
// (resident in shared memory) is walked in chunks of 128 spheres: four tcgen05.mma (M = 128, N = 128, K = 8) per chunk into a
// 128-column accumulator buffer, tcgen05.commit onto the group's `full` mbarrier.  No warp issues on behalf of the others: the
// LAST ray warp of a group to arrive -- with its row written (first chunk of a scan) or with its 32 lanes of the buffer read
// (next chunk) -- issues the tcgen05.mma itself, with arrivals counted in shared memory (atomicAdd).  The ray warps read their
// filter values with tcgen05.ld and resolve the flagged spheres with the same exact test as every other variant -- same hits,
// same bytes out.
//
// The four 128-column TMEM buffers are POOLED: a group holds one only while it scans (first MMA issued ... last chunk read) and
// hands it back for the exact tests of the last chunk, shading, the pop and the row build, so a CTA carries more ray groups
// (4 .. 7) than TMEM has buffers.  free_mask: bit b = buffer b is free; the last warp to write its row takes a buffer
// (atomicAnd), the last reader of the last chunk returns it (atomicOr).
struct TcControl {
    uint64_t full[8];                 // per group: accumulator chunk complete (tcgen05.commit; the exit arrival), count 1
    uint32_t arrived_a[8];            // per group: ray warps with their row written (low byte) / out of work (next byte)
    uint32_t arrived_e[8];            // per group: ray warps that have read the current chunk
    uint32_t exit_flag[8];
    uint32_t buf_of[8];               // per group: the buffer its current scan holds
    uint32_t free_mask;
    uint32_t tmem_base;
    uint32_t pad_[2];
};
static_assert(sizeof(TcControl) % 16 == 0, "TcControl is followed by 16-byte aligned tiles");

constexpr size_t tc3_smem_bytes(int groups, int n32)
{
    return (size_t)kSmemSpheres + 256 + (size_t)n32 * tc::kRowBytes + (size_t)n32 * 16 + (size_t)groups * 128 * tc::kRowBytes +
           (size_t)groups * 4 * sizeof(WarpPool) + 256;          // + alignment slack
}

template <int kGroups, bool kViews>
__global__ void __launch_bounds__(kGroups * 128, 1) megakernel_tc3(const __grid_constant__ RenderArgs a)
{
    constexpr int kChunk = 128, kPool = 4;
    static_assert(kGroups >= 4 && kGroups <= 7, "bad configuration");
    constexpr int kPieces = kChunk / 32;
    // shared memory: [16 B | rsqrtss table 4 KB | control | B tile n32 x 128 B | exact n32 x 16 B | A tiles kGroups x 16 KB | pools]
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint16_t *s_tab = reinterpret_cast<uint16_t *>(smem_raw + 16);
    unsigned char *p = smem_raw + ((kSmemSpheres + 127) & ~127);
    TcControl &ctl = *reinterpret_cast<TcControl *>(p);
    p += (sizeof(TcControl) + 127) & ~127;
    unsigned char *s_b = p;
    const int n32 = a.scene.n32;
    p += (size_t)n32 * tc::kRowBytes;
    float4 *s_exact = reinterpret_cast<float4 *>(p);
    p += (size_t)n32 * 16;
    unsigned char *s_a = p;
    p += (size_t)kGroups * 128 * tc::kRowBytes;
    WarpPool *pools = reinterpret_cast<WarpPool *>(p);

    for (int i = threadIdx.x; i < R1_RSQRT12_ENTRIES / 2; i += blockDim.x)
        reinterpret_cast<uint32_t *>(s_tab)[i] = reinterpret_cast<const uint32_t *>(g_rsqrt12)[i];
    for (int i = threadIdx.x; i < n32 * (tc::kRowBytes / 16); i += blockDim.x)
        reinterpret_cast<uint4 *>(s_b)[i] = reinterpret_cast<const uint4 *>(a.scene.tcb)[i];
    for (int i = threadIdx.x; i < n32; i += blockDim.x)
        s_exact[i] = i < a.scene.n_pad ? a.scene.exact[i] : make_float4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int g = 0; g < 8; ++g) {
            tc::mbar_init(&ctl.full[g], 1);
            ctl.arrived_a[g] = 0; ctl.arrived_e[g] = 0; ctl.exit_flag[g] = 0; ctl.buf_of[g] = 0;
        }
        ctl.free_mask = (1u << kPool) - 1u;
        tc::fence_mbar_init();
    }
    tc::fence_proxy_async();                                     // the B tile is read by the tensor core (async proxy)
    if (threadIdx.x < 32) tc::tmem_alloc(&ctl.tmem_base, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(&ctl.tmem_base);
    const int nchunks = (n32 + kChunk - 1) / kChunk;
    const unsigned lane = threadIdx.x & 31u;
    const int g = threadIdx.x >> 7, w = (threadIdx.x >> 5) & 3, r = threadIdx.x & 127;
    const uint16_t *tab = s_tab;
    const unsigned lt_mask = (1u << lane) - 1u;
    WarpPool &pool = pools[threadIdx.x >> 5];
    unsigned char *a_tile = s_a + (size_t)g * 128 * tc::kRowBytes;
    const uint32_t a_smem = tc::smem_u32(a_tile), b_smem = tc::smem_u32(s_b);
    const uint32_t t_lane = tmem_base + ((uint32_t)(w * 32) << 16);
    bool active = false, exhausted = false;
    PoolState ps;
    ps.dry = false; ps.ready = 0; ps.w_next = 0; ps.w_end = 0;
    const uint32_t lanes_x = gridDim.x * blockDim.x * a.sched_div;
    uint32_t lp = 0, it = 0, nrays = 0;
    int depth = 0;
    f3 thr = mk3(1, 1, 1), o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    Rng rng;
    rng.k0 = 0; rng.k1 = 0;

    for (;;) {
        const bool want = !active && !exhausted;
        const unsigned need = __ballot_sync(kFull, want);
        if (need) pool_take<kViews>(a, pool, ps, tab, lane, lt_mask, lanes_x, need, want, active, exhausted, o, d, lp, rng, thr, depth);
        const bool warp_done = __all_sync(kFull, exhausted);

        tc::write_ray_row(a_tile, r, o, d, active);
        tc::fence_proxy_async();
        tc::tc_fence_before();                                   // this warp's reads of the previous scan's last chunk are complete
        __syncwarp();
        if (lane == 0) {
            const uint32_t mine = 1u + (warp_done ? 0x100u : 0u);
            __threadfence_block();
            const uint32_t tot = atomicAdd(&ctl.arrived_a[g], mine) + mine;
            if ((tot & 0xffu) == 4u) {                           // last of the group: start the scan (or end the group)
                *reinterpret_cast<volatile uint32_t *>(&ctl.arrived_a[g]) = 0u;
                __threadfence_block();
                if ((tot >> 8) == 4u) {
                    *reinterpret_cast<volatile uint32_t *>(&ctl.exit_flag[g]) = 1u;
                    __threadfence_block();
                    tc::mbar_arrive(&ctl.full[g]);
                } else {
                    uint32_t b = 0, spins = 0;
                    for (;;) {                                   // take a free accumulator buffer
                        const uint32_t m = *reinterpret_cast<volatile uint32_t *>(&ctl.free_mask);
                        if (m) {
                            b = (uint32_t)__ffs((int)m) - 1u;
                            if (atomicAnd(&ctl.free_mask, ~(1u << b)) & (1u << b)) break;
                        } else {
                            __nanosleep(64);
                            if (++spins > (1u << 24)) __trap();
                        }
                    }
                    __threadfence_block();
                    *reinterpret_cast<volatile uint32_t *>(&ctl.buf_of[g]) = b;
                    tc::tc_fence_after();
                    tc::mma_chunk(tmem_base + b * kChunk, a_smem, b_smem, min(kChunk, n32), tc::kLBO, tc::kSBO);
                    tc::mma_commit(&ctl.full[g]);
                }
            }
        }
        __syncwarp();

        float t = kTMax;
        int hit = -1;
        bool leave = false;
        uint32_t b = 0;
        for (int c = 0; c < nchunks; ++c, ++it) {
            tc::mbar_wait(&ctl.full[g], it & 1u, true);
            if (c == 0) {
                if (*reinterpret_cast<volatile uint32_t *>(&ctl.exit_flag[g])) { leave = true; break; }
                b = *reinterpret_cast<volatile uint32_t *>(&ctl.buf_of[g]);
            }
            const uint32_t t_buf = t_lane + b * kChunk;
            tc::tc_fence_after();
            const int pieces = min(kPieces, (n32 - c * kChunk) >> 5);   // warp-uniform: the last chunk may be short
            uint32_t cand[kPieces + 1];
#pragma unroll
            for (int h = 0; h < kPieces; h += 2) {               // two loads in flight, eight independent sign-gather chains
                cand[h] = 0; cand[h + 1] = 0;
                if (kGroups <= 5 && h + 1 < pieces) {           // (6 and 7 groups have 72 .. 80 registers: one load at a time)
                    uint32_t v0[32], v1[32];
                    tc::tmem_ld32_issue(t_buf + 32 * h, v0);
                    tc::tmem_ld32_issue(t_buf + 32 * h + 32, v1);
                    tc::tmem_wait(v0, v1);
                    cand[h] = tc::flagged(v0);
                    cand[h + 1] = tc::flagged(v1);
                } else {
                    if (h < pieces) {
                        uint32_t v[32];
                        tc::tmem_ld32(t_buf + 32 * h, v);
                        cand[h] = tc::flagged(v);
                    }
                    if (h + 1 < pieces) {
                        uint32_t v[32];
                        tc::tmem_ld32(t_buf + 32 * h + 32, v);
                        cand[h + 1] = tc::flagged(v);
                    }
                }
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                if (atomicAdd(&ctl.arrived_e[g], 1u) == 3u) {        // last reader
                    *reinterpret_cast<volatile uint32_t *>(&ctl.arrived_e[g]) = 0u;
                    __threadfence_block();
                    if (c + 1 < nchunks) {                           // the buffer is free for the next chunk of this scan
                        tc::tc_fence_after();
                        tc::mma_chunk(tmem_base + b * kChunk, a_smem, b_smem + (uint32_t)(c + 1) * (kChunk / 8) * tc::kSBO, min(kChunk, n32 - (c + 1) * kChunk),
                                      tc::kLBO, tc::kSBO);
                        tc::mma_commit(&ctl.full[g]);
                    } else {
                        atomicOr(&ctl.free_mask, 1u << b);           // scan over: hand the buffer back
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int h = 0; h < kPieces; ++h)
                if (cand[h]) exact_candidates(cand[h], s_exact, c * kChunk + 32 * h, o, d, kTMin, t, hit);
        }
        if (leave) break;

        if (active) {
            ++nrays;
            f3 contrib;
            const float4 e = hit >= 0 ? s_exact[hit] : make_float4(0, 0, 0, 0);
            if (shade_step(a, hit, t, e, tab, o, d, thr, depth, rng, contrib)) {
                accumulate_sample(a, lp, contrib);
                active = false;
            }
        }
    }
    count_rays(a, nrays, lane);
    tc::tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tc::tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ megakernel, streamed tensor-core filter
// R1_VARIANT_MEGAKERNEL_TENSOR_STREAM (DESIGN.md section 4.7): megakernel_tc3's scan with the sphere operand STREAMED through a
// ring of kStages shared-memory stages instead of resident, so that shared memory no longer depends on the scene.  A stage holds
// one 128-sphere chunk: its 16 KB of operand rows (one contiguous range of the K-major layout) and its 2 KB of exact records,
// brought in by two cp.async.bulk on the stage's `landed` mbarrier.
//
// Fills are numbered f = 0, 1, 2, ...: fill f is chunk f mod nchunks in stage f mod kStages.  Every live ray group consumes every
// fill in order; a scan is the nchunks fills from a multiple of nchunks, so the exact tests still run in ascending sphere order.
// Each warp releases a fill once its group's MMA on it is complete (the warp has waited for it) and its own exact tests are done:
// byte g of the stage's ring word counts the warps of group g.  The thread whose release completes the fill -- every group still
// consuming has all four warps in -- refills the stage with fill f + kStages (tc3's last-arriver idiom, no producer warp), so the
// groups drift apart by at most the ring depth.  A group out of work sets its bit in `exited`: from then on it counts as done for
// every fill, and it completes the fills only it was holding up.  The ring word {fill number | release bytes} changes atomically,
// and a refill is claimed with a compare-and-swap on it, so a releaser and a leaving group that both see a fill complete refill
// it once.  Fill numbers are kept modulo 2 kStages nchunks, which preserves the stage, the chunk and the mbarrier parity.
constexpr int kTcsChunk = 128;
constexpr int kTcsMaxStages = 8;
constexpr uint32_t kTcsOpBytes = kTcsChunk * tc::kRowBytes;   // 16 KB of operand rows
constexpr uint32_t kTcsStageBytes = kTcsOpBytes + kTcsChunk * 16;   // + 2 KB of exact records

struct TcsControl {
    uint64_t mma[4];                      // per group: accumulator chunk complete (tcgen05.commit; the exit arrival), count 1
    uint64_t landed[kTcsMaxStages];       // per stage: fill landed (complete_tx)
    uint64_t ring[kTcsMaxStages];         // per stage: fill number << 32 | byte g = warps of group g done with it
    uint32_t arrived_a[4];                // per group: ray warps with their row written (low byte) / out of work (next byte)
    uint32_t arrived_e[4];                // per group: ray warps that have read the current chunk
    uint32_t exit_flag[4];
    uint32_t exited;                      // bit g: group g is out of work and consumes no more fills
    uint32_t tmem_base;
    uint32_t pad_[2];
};
static_assert(sizeof(TcsControl) % 16 == 0, "TcsControl is followed by 16-byte aligned stages");

// The sphere operand at every scene size: the end of the scene block, after the shading records (r1_scene_commit)
__device__ __forceinline__ const unsigned char *tcs_operand(const DevScene &sc) { return reinterpret_cast<const unsigned char *>(sc.shade + 2 * (size_t)sc.n_pad); }

// Fill a stage with chunk c (one thread): the rows that exist (the last chunk may be short) and the n_pad exact records that
// exist -- n32 is padded to 32, n_pad only to 16, and the columns without a record are padding rows no ray flags.
__device__ __forceinline__ void tcs_fill(const DevScene &sc, unsigned char *stage, uint64_t *landed, int c)
{
    const uint32_t op_bytes = (uint32_t)min(kTcsChunk, sc.n32 - c * kTcsChunk) * tc::kRowBytes;
    const uint32_t ex_bytes = (uint32_t)min(kTcsChunk, sc.n_pad - c * kTcsChunk) * 16u;
    const uint32_t bar = tc::smem_u32(landed);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(op_bytes + ex_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(stage)),
                 "l"(tcs_operand(sc) + (size_t)c * kTcsOpBytes), "r"(op_bytes), "r"(bar)
                 : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(stage + kTcsOpBytes)),
                 "l"(sc.exact + (size_t)c * kTcsChunk), "r"(ex_bytes), "r"(bar)
                 : "memory");
}

// A fill is complete when every group still consuming has all four warps in.  With every group gone nothing is refilled.
template <int kGroups>
__device__ __forceinline__ bool tcs_fill_complete(uint32_t released, uint32_t exited)
{
    bool done = exited != (1u << kGroups) - 1u;
#pragma unroll
    for (int g = 0; g < kGroups; ++g)
        if (!((exited >> g) & 1u) && ((released >> (8 * g)) & 0xffu) != 4u) done = false;
    return done;
}
// Refill a completed stage with fill f + kStages -- once: the compare-and-swap on the whole ring word fails for everyone else
template <int kStages>
__device__ __forceinline__ void tcs_refill(const DevScene &sc, TcsControl &ctl, unsigned char *stages, int s, uint64_t word, uint32_t wrap, int nchunks)
{
    uint32_t next = (uint32_t)(word >> 32) + kStages;
    if (next >= wrap) next -= wrap;
    if (atomicCAS(reinterpret_cast<unsigned long long *>(&ctl.ring[s]), word, (unsigned long long)next << 32) != word) return;
    tcs_fill(sc, stages + (size_t)s * kTcsStageBytes, &ctl.landed[s], (int)(next % (uint32_t)nchunks));
}
// One warp (lane 0) of group g is done with the fill in stage s
template <int kGroups, int kStages>
__device__ __forceinline__ void tcs_release(const DevScene &sc, TcsControl &ctl, unsigned char *stages, int s, int g, uint32_t wrap, int nchunks)
{
    __threadfence_block();
    const unsigned long long inc = 1ull << (8 * g);
    const uint64_t word = atomicAdd(reinterpret_cast<unsigned long long *>(&ctl.ring[s]), inc) + inc;
    __threadfence_block();                                       // the release before the read of `exited` (see tcs_leave)
    if (tcs_fill_complete<kGroups>((uint32_t)word, *reinterpret_cast<volatile uint32_t *>(&ctl.exited))) tcs_refill<kStages>(sc, ctl, stages, s, word, wrap, nchunks);
}
// Group g is out of work (its warps hold no fill): it stops counting as a consumer and completes the fills that waited only for it.
// Its bit is published before it reads the ring words, and a releaser adds its byte before it reads `exited`: of a racing pair at
// least one sees the other, and the compare-and-swap lets only one of them refill.
template <int kGroups, int kStages>
__device__ __forceinline__ void tcs_leave(const DevScene &sc, TcsControl &ctl, unsigned char *stages, int g, uint32_t wrap, int nchunks)
{
    const uint32_t exited = atomicOr(&ctl.exited, 1u << g) | (1u << g);
    __threadfence_block();
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
        const uint64_t word = *reinterpret_cast<volatile uint64_t *>(&ctl.ring[s]);
        if (tcs_fill_complete<kGroups>((uint32_t)word, exited)) tcs_refill<kStages>(sc, ctl, stages, s, word, wrap, nchunks);
    }
}

constexpr size_t tcs_smem_bytes(int groups, int stages)
{
    return (size_t)((kSmemSpheres + 127) & ~127) + ((sizeof(TcsControl) + 127) & ~(size_t)127) + (size_t)stages * kTcsStageBytes +
           (size_t)groups * 128 * tc::kRowBytes + (size_t)groups * 4 * sizeof(WarpPool);
}

template <int kGroups, int kStages, bool kViews>
__global__ void __launch_bounds__(kGroups * 128, 1) megakernel_tcs(const __grid_constant__ RenderArgs a)
{
    constexpr int kChunk = kTcsChunk, kPieces = kChunk / 32;
    static_assert(kGroups >= 1 && kGroups <= 4 && kStages >= 2 && kStages <= kTcsMaxStages, "bad configuration");
    constexpr uint32_t kTmemCols = kGroups == 1 ? 128 : (kGroups == 2 ? 256 : 512);   // one 128-column accumulator per group
    // shared memory: [16 B | rsqrtss table 4 KB | control | stages kStages x 18 KB | A tiles kGroups x 16 KB | pools]
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint16_t *s_tab = reinterpret_cast<uint16_t *>(smem_raw + 16);
    unsigned char *p = smem_raw + ((kSmemSpheres + 127) & ~127);
    TcsControl &ctl = *reinterpret_cast<TcsControl *>(p);
    p += (sizeof(TcsControl) + 127) & ~127;
    unsigned char *s_stages = p;
    p += (size_t)kStages * kTcsStageBytes;
    unsigned char *s_a = p;
    p += (size_t)kGroups * 128 * tc::kRowBytes;
    WarpPool *pools = reinterpret_cast<WarpPool *>(p);

    const int n32 = a.scene.n32;
    const int nchunks = (n32 + kChunk - 1) / kChunk;
    const uint32_t wrap = 2u * kStages * (uint32_t)nchunks;
    for (int i = threadIdx.x; i < R1_RSQRT12_ENTRIES / 2; i += blockDim.x)
        reinterpret_cast<uint32_t *>(s_tab)[i] = reinterpret_cast<const uint32_t *>(g_rsqrt12)[i];
    if (threadIdx.x == 0) {
        for (int g = 0; g < 4; ++g) {
            tc::mbar_init(&ctl.mma[g], 1);
            ctl.arrived_a[g] = 0; ctl.arrived_e[g] = 0; ctl.exit_flag[g] = 0;
        }
        for (int s = 0; s < kStages; ++s) {
            tc::mbar_init(&ctl.landed[s], 1);
            ctl.ring[s] = (uint64_t)s << 32;
        }
        ctl.exited = 0;
        tc::fence_mbar_init();
        tc::fence_proxy_async();
        for (int s = 0; s < kStages; ++s) tcs_fill(a.scene, s_stages + (size_t)s * kTcsStageBytes, &ctl.landed[s], s % nchunks);
    }
    if (threadIdx.x < 32) tc::tmem_alloc(&ctl.tmem_base, kTmemCols);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(&ctl.tmem_base);
    const unsigned lane = threadIdx.x & 31u;
    const int g = threadIdx.x >> 7, w = (threadIdx.x >> 5) & 3, r = threadIdx.x & 127;
    const uint16_t *tab = s_tab;
    const unsigned lt_mask = (1u << lane) - 1u;
    WarpPool &pool = pools[threadIdx.x >> 5];
    unsigned char *a_tile = s_a + (size_t)g * 128 * tc::kRowBytes;
    const uint32_t a_smem = tc::smem_u32(a_tile), stages_smem = tc::smem_u32(s_stages);
    const uint32_t t_acc = tmem_base + (uint32_t)(g * kChunk);
    const uint32_t t_lane = t_acc + ((uint32_t)(w * 32) << 16);
    bool active = false, exhausted = false;
    PoolState ps;
    ps.dry = false; ps.ready = 0; ps.w_next = 0; ps.w_end = 0;
    const uint32_t lanes_x = gridDim.x * blockDim.x * a.sched_div;
    uint32_t lp = 0, it = 0, nrays = 0, fpos = 0;               // fpos: the fill that starts this group's next scan
    int depth = 0;
    f3 thr = mk3(1, 1, 1), o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    Rng rng;
    rng.k0 = 0; rng.k1 = 0;

    for (;;) {
        const bool want = !active && !exhausted;
        const unsigned need = __ballot_sync(kFull, want);
        if (need) pool_take<kViews>(a, pool, ps, tab, lane, lt_mask, lanes_x, need, want, active, exhausted, o, d, lp, rng, thr, depth);
        const bool warp_done = __all_sync(kFull, exhausted);

        tc::write_ray_row(a_tile, r, o, d, active);
        tc::fence_proxy_async();
        tc::tc_fence_before();                                   // this warp's reads of the previous scan's last chunk are complete
        __syncwarp();
        if (lane == 0) {
            const uint32_t mine = 1u + (warp_done ? 0x100u : 0u);
            __threadfence_block();
            const uint32_t tot = atomicAdd(&ctl.arrived_a[g], mine) + mine;
            if ((tot & 0xffu) == 4u) {                           // last of the group: start the scan (or end the group)
                *reinterpret_cast<volatile uint32_t *>(&ctl.arrived_a[g]) = 0u;
                __threadfence_block();
                if ((tot >> 8) == 4u) {
                    *reinterpret_cast<volatile uint32_t *>(&ctl.exit_flag[g]) = 1u;
                    __threadfence_block();
                    tcs_leave<kGroups, kStages>(a.scene, ctl, s_stages, g, wrap, nchunks);
                    tc::mbar_arrive(&ctl.mma[g]);
                } else {
                    const int s = (int)(fpos % kStages);
                    tc::mbar_wait(&ctl.landed[s], (fpos / kStages) & 1u, true);
                    tc::tc_fence_after();
                    tc::mma_chunk(t_acc, a_smem, stages_smem + (uint32_t)s * kTcsStageBytes, min(kChunk, n32), tc::kLBO, tc::kSBO);
                    tc::mma_commit(&ctl.mma[g]);
                }
            }
        }
        __syncwarp();

        float t = kTMax;
        int hit = -1;
        bool leave = false;
        for (int c = 0; c < nchunks; ++c, ++it) {
            tc::mbar_wait(&ctl.mma[g], it & 1u, true);
            if (c == 0 && *reinterpret_cast<volatile uint32_t *>(&ctl.exit_flag[g])) { leave = true; break; }
            const uint32_t f = fpos + (uint32_t)c;
            const int s = (int)(f % kStages);
            tc::tc_fence_after();
            const int pieces = min(kPieces, (n32 - c * kChunk) >> 5);   // warp-uniform: the last chunk may be short
            uint32_t cand[kPieces];
#pragma unroll
            for (int h = 0; h < kPieces; h += 2) {               // two loads in flight, eight independent sign-gather chains
                cand[h] = 0; cand[h + 1] = 0;
                if (h + 1 < pieces) {
                    uint32_t v0[32], v1[32];
                    tc::tmem_ld32_issue(t_lane + 32 * h, v0);
                    tc::tmem_ld32_issue(t_lane + 32 * h + 32, v1);
                    tc::tmem_wait(v0, v1);
                    cand[h] = tc::flagged(v0);
                    cand[h + 1] = tc::flagged(v1);
                } else if (h < pieces) {
                    uint32_t v[32];
                    tc::tmem_ld32(t_lane + 32 * h, v);
                    cand[h] = tc::flagged(v);
                }
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                if (atomicAdd(&ctl.arrived_e[g], 1u) == 3u) {        // last reader: the accumulator is free for the next chunk
                    *reinterpret_cast<volatile uint32_t *>(&ctl.arrived_e[g]) = 0u;
                    __threadfence_block();
                    if (c + 1 < nchunks) {
                        const uint32_t f1 = f + 1u;
                        const int s1 = (int)(f1 % kStages);
                        tc::mbar_wait(&ctl.landed[s1], (f1 / kStages) & 1u, true);
                        tc::tc_fence_after();
                        tc::mma_chunk(t_acc, a_smem, stages_smem + (uint32_t)s1 * kTcsStageBytes, min(kChunk, n32 - (c + 1) * kChunk), tc::kLBO, tc::kSBO);
                        tc::mma_commit(&ctl.mma[g]);
                    }
                }
            }
            __syncwarp();
            tc::mbar_wait(&ctl.landed[s], (f / kStages) & 1u);   // complete (the MMA read it): makes the exact records visible here
            const float4 *s_exact = reinterpret_cast<const float4 *>(s_stages + (size_t)s * kTcsStageBytes + kTcsOpBytes) - c * kChunk;
#pragma unroll
            for (int h = 0; h < kPieces; ++h)
                if (cand[h]) exact_candidates(cand[h], s_exact, c * kChunk + 32 * h, o, d, kTMin, t, hit);
            __syncwarp();
            if (lane == 0) tcs_release<kGroups, kStages>(a.scene, ctl, s_stages, s, g, wrap, nchunks);
        }
        if (leave) break;
        fpos += (uint32_t)nchunks;
        if (fpos >= wrap) fpos -= wrap;

        if (active) {
            ++nrays;
            f3 contrib;
            const float4 e = hit >= 0 ? a.scene.exact[hit] : make_float4(0, 0, 0, 0);   // the stage may hold another chunk by now
            if (shade_step(a, hit, t, e, tab, o, d, thr, depth, rng, contrib)) {
                accumulate_sample(a, lp, contrib);
                active = false;
            }
        }
    }
    count_rays(a, nrays, lane);
    tc::tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) {                                      // no bulk copy may still be writing when the CTA ends
        for (int s = 0; s < kStages; ++s) {
            const uint32_t f = (uint32_t)(*reinterpret_cast<volatile uint64_t *>(&ctl.ring[s]) >> 32);
            tc::mbar_wait(&ctl.landed[s], (f / kStages) & 1u);
        }
    }
    if (threadIdx.x < 32) tc::tmem_dealloc(tmem_base, kTmemCols);
}

// TMEM read throughput: every warp reads 32 lanes x 32 columns (4 KB) per tcgen05.ld, `iters` times over its lane quarter's 512
// columns.  Bounds the tensor-core filter: one 4-byte filter value per (ray, sphere) has to come out of TMEM.
__global__ void __launch_bounds__(1024, 1) tmem_read_kernel(int iters, uint32_t *sink)
{
    __shared__ uint32_t slot;
    if (threadIdx.x < 32) tc::tmem_alloc(&slot, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t base = *reinterpret_cast<volatile uint32_t *>(&slot) + ((uint32_t)(((threadIdx.x >> 5) & 3) * 32) << 16);
    uint32_t acc = 0;
    for (int i = 0; i < iters; ++i) {
        uint32_t v[32];
        tc::tmem_ld32(base + (uint32_t)((i + (threadIdx.x >> 7)) & 15) * 32u, v);
#pragma unroll
        for (int j = 0; j < 32; j += 8) acc ^= v[j];
    }
    if (acc == 0x12345678u) sink[0] = acc;                       // keeps the loads alive
    tc::tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tc::tmem_dealloc(*reinterpret_cast<volatile uint32_t *>(&slot), 512);
}

// ------------------------------------------------------------------------------------------------ resolve
// rayweek1.cpp:765-775: average, gamma 2 (sqrtf), quantise (int)(c * 255.99f) -> RGB8.
__device__ __forceinline__ uint8_t quantise(unsigned long long sum, float inv_spp)
{
    const float mean = fmul(fmul(__ull2float_rn(sum), kFixedInvScale), inv_spp);   // col *= 1 / spp  (:765)
    const float c = __fsqrt_rn(mean);                                              // :767
    return (uint8_t)(int)fmul(c, 255.99f);                                         // :769-775
}
__global__ void __launch_bounds__(256) resolve(const __grid_constant__ RenderArgs a)
{
    for (uint32_t lp = blockIdx.x * blockDim.x + threadIdx.x; lp < a.npix_local; lp += gridDim.x * blockDim.x) {
        const ulonglong2 rg = *reinterpret_cast<const ulonglong2 *>(a.accum + (size_t)lp * 4);
        const unsigned long long b = a.accum[(size_t)lp * 4 + 2];
        uint8_t *out = a.rgb + (size_t)lp * 3;
        out[0] = quantise(rg.x, a.inv_spp); out[1] = quantise(rg.y, a.inv_spp); out[2] = quantise(b, a.inv_spp);
    }
}

// Multi-GPU epilogue: slice r of `gathered` = rank r's local rows; scatter them to their global rows.
__global__ void __launch_bounds__(256) deinterleave_rows(const uint8_t *gathered, size_t stride, uint8_t *out, int width, int height, int row_tile, int world)
{
    const size_t row_bytes = (size_t)width * 3, total = row_bytes * (size_t)height;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(i / row_bytes);
        const size_t xb = i - (size_t)y * row_bytes;
        const int tile = y / row_tile, rank = tile % world;
        const int lr = (tile / world) * row_tile + (y - tile * row_tile);
        out[i] = gathered[(size_t)rank * stride + (size_t)lr * row_bytes + xb];
    }
}

// ------------------------------------------------------------------------------------------------ parity kernels
template <int kScan>
__global__ void __launch_bounds__(128) trace_rays_kernel(const __grid_constant__ DevScene sc, int n, const float *org, const float *dir,
                                                         float t_min, float t_max, int32_t *index, float *t_out, float *p_out, float *n_out)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4 *s_spheres = reinterpret_cast<float4 *>(smem_raw + 16);
    stage_spheres(sc, s_spheres, reinterpret_cast<uint64_t *>(smem_raw));
    WarpScratch *ws = reinterpret_cast<WarpScratch *>(smem_raw + 16 + (size_t)sc.n_pad * 32) + (threadIdx.x >> 5);
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = k < n;                               // the whole warp takes part in the cooperative scan
    f3 o = mk3(0.0f, 1.0e18f, 0.0f), d = mk3(0.0f, 0.0f, 0.0f);
    if (live) { o = mk3(org[3 * k], org[3 * k + 1], org[3 * k + 2]); d = mk3(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]); }
    float t = t_max;
    int hit = -1;
    if (kScan == kScanCoop) scan_coop<2>(*ws, s_spheres, s_spheres + sc.n_pad, sc.n_pad, o, d, t_min, t_max, t, hit);
    else if (kScan == kScanLaneDeferred) scan_deferred(*reinterpret_cast<DeferScratch *>(ws), s_spheres, s_spheres + sc.n_pad, sc.n8, o, d, t_min, t_max, t, hit);
    else scan<scan_filter(kScan)>(s_spheres, s_spheres + sc.n_pad, sc.n8, o, d, t_min, t, hit);
    if (!live) return;
    f3 p = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
    if (hit >= 0) hit_finalise(s_spheres[sc.n_pad + hit], load_shade(sc, hit).inv_radius, o, d, t, p, nrm);
    index[k] = hit;
    t_out[k] = hit >= 0 ? t : 0.0f;
    p_out[3 * k] = p.x; p_out[3 * k + 1] = p.y; p_out[3 * k + 2] = p.z;
    n_out[3 * k] = nrm.x; n_out[3 * k + 1] = nrm.y; n_out[3 * k + 2] = nrm.z;
}

// Hitable::hit through the BVH (R1_VARIANT_MEGAKERNEL_BVH): bvh_trace, then hit_finalise from the scene's exact and shading
// records by original index.  Any sphere count; nothing staged.
__global__ void __launch_bounds__(128) trace_rays_bvh_kernel(const __grid_constant__ DevScene sc, int n, const float *org, const float *dir,
                                                             float t_min, float t_max, int32_t *index, float *t_out, float *p_out, float *n_out,
                                                             const float4 *nodes, const float4 *leaves)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const f3 o = mk3(org[3 * k], org[3 * k + 1], org[3 * k + 2]), d = mk3(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]);
    float t = t_max;
    int hit = -1;
    bvh_trace(nodes, leaves, o, d, t_min, t, hit);
    f3 p = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
    if (hit >= 0) hit_finalise(__ldg(sc.exact + hit), load_shade(sc, hit).inv_radius, o, d, t, p, nrm);
    index[k] = hit;
    t_out[k] = hit >= 0 ? t : 0.0f;
    p_out[3 * k] = p.x; p_out[3 * k + 1] = p.y; p_out[3 * k + 2] = p.z;
    n_out[3 * k] = nrm.x; n_out[3 * k + 1] = nrm.y; n_out[3 * k + 2] = nrm.z;
}

// Hitable::hit through the filter of megakernel_tc3: the same device functions (write_ray_row, mma_chunk in chunks of 128
// spheres with the per-chunk N, the last chunk read in (n32 - 128 c) / 32 pieces of 32 columns, two TMEM loads in flight,
// exact_candidates, hit_finalise) with the caller's t_min / t_max.  One CTA = 128 rays, one 128-column accumulator buffer, the
// MMA issued by thread 0; no buffer pool, so only the arithmetic and the chunking of tc3 are under test here.
constexpr int kTraceTcChunk = 128;                               // = megakernel_tc3's kChunk
constexpr size_t trace_rays_tc_smem_bytes(int n32)
{
    return 128 + (size_t)n32 * tc::kRowBytes + 128 * tc::kRowBytes + (size_t)n32 * 16;
}
__global__ void __launch_bounds__(128, 1) trace_rays_tc_kernel(const __grid_constant__ DevScene sc, int n, const float *org, const float *dir,
                                                               float t_min, float t_max, int32_t *index, float *t_out, float *p_out, float *n_out)
{
    constexpr int kChunk = kTraceTcChunk, kPieces = kChunk / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw);      // [mbarrier | TMEM address | pad to 128 | B | A | exact]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem_raw + 8);
    const int n32 = sc.n32;
    unsigned char *s_b = smem_raw + 128;
    unsigned char *a_tile = s_b + (size_t)n32 * tc::kRowBytes;
    float4 *s_exact = reinterpret_cast<float4 *>(a_tile + 128 * tc::kRowBytes);
    for (int i = threadIdx.x; i < n32 * (tc::kRowBytes / 16); i += blockDim.x)
        reinterpret_cast<uint4 *>(s_b)[i] = reinterpret_cast<const uint4 *>(sc.tcb)[i];
    for (int i = threadIdx.x; i < n32; i += blockDim.x)
        s_exact[i] = i < sc.n_pad ? sc.exact[i] : make_float4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        tc::mbar_init(full, 1);
        tc::fence_mbar_init();
    }
    const int k = blockIdx.x * 128 + threadIdx.x;
    const bool live = k < n;                                     // rays past n write a row that flags nothing
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    if (live) { o = mk3(org[3 * k], org[3 * k + 1], org[3 * k + 2]); d = mk3(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]); }
    tc::write_ray_row(a_tile, threadIdx.x, o, d, live);
    tc::fence_proxy_async();                                     // the tiles are read by the tensor core (async proxy)
    if (threadIdx.x < 32) tc::tmem_alloc(tmem_slot, kChunk);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(tmem_slot);
    const uint32_t t_lane = tmem_base + ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
    const uint32_t a_smem = tc::smem_u32(a_tile), b_smem = tc::smem_u32(s_b);
    const int nchunks = (n32 + kChunk - 1) / kChunk;
    float t = t_max;
    int hit = -1;
    for (int c = 0; c < nchunks; ++c) {
        if (threadIdx.x == 0) {
            tc::tc_fence_after();
            tc::mma_chunk(tmem_base, a_smem, b_smem + (uint32_t)c * (kChunk / 8) * tc::kSBO, min(kChunk, n32 - c * kChunk), tc::kLBO, tc::kSBO);
            tc::mma_commit(full);
        }
        tc::mbar_wait(full, (uint32_t)c & 1u);
        tc::tc_fence_after();
        const int pieces = min(kPieces, (n32 - c * kChunk) >> 5);   // the last chunk may be short
        uint32_t cand[kPieces];
#pragma unroll
        for (int h = 0; h < kPieces; h += 2) {
            cand[h] = 0; cand[h + 1] = 0;
            if (h + 1 < pieces) {
                uint32_t v0[32], v1[32];
                tc::tmem_ld32_issue(t_lane + 32 * h, v0);
                tc::tmem_ld32_issue(t_lane + 32 * h + 32, v1);
                tc::tmem_wait(v0, v1);
                cand[h] = tc::flagged(v0);
                cand[h + 1] = tc::flagged(v1);
            } else if (h < pieces) {
                uint32_t v[32];
                tc::tmem_ld32(t_lane + 32 * h, v);
                cand[h] = tc::flagged(v);
            }
        }
        tc::tc_fence_before();
        __syncthreads();                                         // every warp has read the buffer: the next chunk may overwrite it
#pragma unroll
        for (int h = 0; h < kPieces; ++h)
            if (cand[h]) exact_candidates(cand[h], s_exact, c * kChunk + 32 * h, o, d, t_min, t, hit);
    }
    if (threadIdx.x < 32) tc::tmem_dealloc(tmem_base, kChunk);
    if (!live) return;
    f3 p = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
    if (hit >= 0) hit_finalise(s_exact[hit], load_shade(sc, hit).inv_radius, o, d, t, p, nrm);
    index[k] = hit;
    t_out[k] = hit >= 0 ? t : 0.0f;
    p_out[3 * k] = p.x; p_out[3 * k + 1] = p.y; p_out[3 * k + 2] = p.z;
    n_out[3 * k] = nrm.x; n_out[3 * k + 1] = nrm.y; n_out[3 * k + 2] = nrm.z;
}

// Filter values of n rays against every sphere (parity / error measurement of the tensor filter): e[ray * n32 + sphere].
// The MMA chunks of trace_rays_tc_kernel -- 128 spheres with the per-chunk N into one 128-column accumulator, issued by
// thread 0 -- with the raw values written out instead of tested.
constexpr size_t filter_probe_smem_bytes(int n32) { return 128 + (size_t)n32 * tc::kRowBytes + 128 * tc::kRowBytes; }
__global__ void __launch_bounds__(128, 1) tc_filter_probe_kernel(const __grid_constant__ DevScene sc, int n, const float *__restrict__ org,
                                                               const float *__restrict__ dir, float *__restrict__ e_out)
{
    constexpr int kChunk = kTraceTcChunk;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw);      // [mbarrier | TMEM address | pad to 128 | B | A]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem_raw + 8);
    const int n32 = sc.n32;
    unsigned char *s_b = smem_raw + 128;
    unsigned char *a_tile = s_b + (size_t)n32 * tc::kRowBytes;
    for (int i = threadIdx.x; i < n32 * (tc::kRowBytes / 16); i += blockDim.x)
        reinterpret_cast<uint4 *>(s_b)[i] = reinterpret_cast<const uint4 *>(sc.tcb)[i];
    if (threadIdx.x == 0) {
        tc::mbar_init(full, 1);
        tc::fence_mbar_init();
    }
    const int ray = blockIdx.x * 128 + threadIdx.x;
    const bool live = ray < n;                                   // rays past n write a row that flags nothing
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    if (live) { o = mk3(org[3 * ray], org[3 * ray + 1], org[3 * ray + 2]); d = mk3(dir[3 * ray], dir[3 * ray + 1], dir[3 * ray + 2]); }
    tc::write_ray_row(a_tile, threadIdx.x, o, d, live);
    tc::fence_proxy_async();                                     // the tiles are read by the tensor core (async proxy)
    if (threadIdx.x < 32) tc::tmem_alloc(tmem_slot, kChunk);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(tmem_slot);
    const uint32_t t_lane = tmem_base + ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
    const uint32_t a_smem = tc::smem_u32(a_tile), b_smem = tc::smem_u32(s_b);
    const int nchunks = (n32 + kChunk - 1) / kChunk;
    for (int c = 0; c < nchunks; ++c) {
        if (threadIdx.x == 0) {
            tc::tc_fence_after();
            tc::mma_chunk(tmem_base, a_smem, b_smem + (uint32_t)c * (kChunk / 8) * tc::kSBO, min(kChunk, n32 - c * kChunk), tc::kLBO, tc::kSBO);
            tc::mma_commit(full);
        }
        tc::mbar_wait(full, (uint32_t)c & 1u);
        tc::tc_fence_after();
        const int pieces = min(kChunk / 32, (n32 - c * kChunk) >> 5);   // the last chunk may be short
        for (int h = 0; h < pieces; ++h) {
            uint32_t v[32];
            tc::tmem_ld32(t_lane + 32 * h, v);
            if (live)
#pragma unroll
                for (int j = 0; j < 32; ++j) e_out[(size_t)ray * n32 + c * kChunk + 32 * h + j] = __uint_as_float(v[j]);
        }
        tc::tc_fence_before();
        __syncthreads();                                         // every warp has read the buffer: the next chunk may overwrite it
    }
    if (threadIdx.x < 32) tc::tmem_dealloc(tmem_base, kChunk);
}

// Hitable::hit through the filter of megakernel_tcs at any scene size: the chunks stream through a ring of two stages filled by
// tcs_fill (its addressing, the short last chunk, the exact records that exist), the rest as in trace_rays_tc_kernel.  One CTA =
// one ray group, so chunk c is simply fill c; the multi-group release protocol is exercised by the renders.
constexpr int kTraceTcsStages = 2;
constexpr size_t trace_rays_tcs_smem_bytes() { return 128 + (size_t)kTraceTcsStages * kTcsStageBytes + 128 * tc::kRowBytes; }
__global__ void __launch_bounds__(128, 1) trace_rays_tcs_kernel(const __grid_constant__ DevScene sc, int n, const float *org, const float *dir,
                                                                float t_min, float t_max, int32_t *index, float *t_out, float *p_out, float *n_out)
{
    constexpr int kChunk = kTcsChunk, kPieces = kChunk / 32, kStages = kTraceTcsStages;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw);      // [MMA mbarrier | stage mbarriers | TMEM address | pad to 128 | stages | A]
    uint64_t *landed = full + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(landed + kStages);
    unsigned char *s_stages = smem_raw + 128;
    unsigned char *a_tile = s_stages + (size_t)kStages * kTcsStageBytes;
    const int n32 = sc.n32;
    const int nchunks = (n32 + kChunk - 1) / kChunk;
    if (threadIdx.x == 0) {
        tc::mbar_init(full, 1);
        for (int s = 0; s < kStages; ++s) tc::mbar_init(&landed[s], 1);
        tc::fence_mbar_init();
        tc::fence_proxy_async();
        for (int s = 0; s < kStages && s < nchunks; ++s) tcs_fill(sc, s_stages + (size_t)s * kTcsStageBytes, &landed[s], s);
    }
    const int k = blockIdx.x * 128 + threadIdx.x;
    const bool live = k < n;                                     // rays past n write a row that flags nothing
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    if (live) { o = mk3(org[3 * k], org[3 * k + 1], org[3 * k + 2]); d = mk3(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]); }
    tc::write_ray_row(a_tile, threadIdx.x, o, d, live);
    tc::fence_proxy_async();                                     // the A tile is read by the tensor core (async proxy)
    if (threadIdx.x < 32) tc::tmem_alloc(tmem_slot, kChunk);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(tmem_slot);
    const uint32_t t_lane = tmem_base + ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
    const uint32_t a_smem = tc::smem_u32(a_tile), stages_smem = tc::smem_u32(s_stages);
    float t = t_max;
    int hit = -1;
    for (int c = 0; c < nchunks; ++c) {
        const int s = c % kStages;
        const uint32_t parity = (uint32_t)(c / kStages) & 1u;
        if (threadIdx.x == 0) {
            tc::mbar_wait(&landed[s], parity);
            tc::tc_fence_after();
            tc::mma_chunk(tmem_base, a_smem, stages_smem + (uint32_t)s * kTcsStageBytes, min(kChunk, n32 - c * kChunk), tc::kLBO, tc::kSBO);
            tc::mma_commit(full);
        }
        tc::mbar_wait(full, (uint32_t)c & 1u);
        tc::tc_fence_after();
        const int pieces = min(kPieces, (n32 - c * kChunk) >> 5);   // the last chunk may be short
        uint32_t cand[kPieces];
#pragma unroll
        for (int h = 0; h < kPieces; h += 2) {
            cand[h] = 0; cand[h + 1] = 0;
            if (h + 1 < pieces) {
                uint32_t v0[32], v1[32];
                tc::tmem_ld32_issue(t_lane + 32 * h, v0);
                tc::tmem_ld32_issue(t_lane + 32 * h + 32, v1);
                tc::tmem_wait(v0, v1);
                cand[h] = tc::flagged(v0);
                cand[h + 1] = tc::flagged(v1);
            } else if (h < pieces) {
                uint32_t v[32];
                tc::tmem_ld32(t_lane + 32 * h, v);
                cand[h] = tc::flagged(v);
            }
        }
        tc::tc_fence_before();
        tc::mbar_wait(&landed[s], parity);                       // complete: makes the bulk copy's exact records visible here
        const float4 *s_exact = reinterpret_cast<const float4 *>(s_stages + (size_t)s * kTcsStageBytes + kTcsOpBytes) - c * kChunk;
#pragma unroll
        for (int h = 0; h < kPieces; ++h)
            if (cand[h]) exact_candidates(cand[h], s_exact, c * kChunk + 32 * h, o, d, t_min, t, hit);
        __syncthreads();                                         // every warp is done with the accumulator and with the stage
        if (threadIdx.x == 0 && c + kStages < nchunks) tcs_fill(sc, s_stages + (size_t)s * kTcsStageBytes, &landed[s], c + kStages);
    }
    if (threadIdx.x < 32) tc::tmem_dealloc(tmem_base, kChunk);
    if (!live) return;
    f3 p = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
    if (hit >= 0) hit_finalise(sc.exact[hit], load_shade(sc, hit).inv_radius, o, d, t, p, nrm);
    index[k] = hit;
    t_out[k] = hit >= 0 ? t : 0.0f;
    p_out[3 * k] = p.x; p_out[3 * k + 1] = p.y; p_out[3 * k + 2] = p.z;
    n_out[3 * k] = nrm.x; n_out[3 * k + 1] = nrm.y; n_out[3 * k + 2] = nrm.z;
}

__global__ void scatter_kernel(const __grid_constant__ DevScene sc, int n, const float *dir_in, const float *p, const float *nrm,
                               const int32_t *index, const float *rs, const float *ru, int32_t *ok, float *atten, float *dir_out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int i = index[k];
    f3 a = mk3(0, 0, 0), dd = mk3(0, 0, 0);
    bool r = false;
    const ShadeRec sh = load_shade(sc, i >= 0 && i < sc.n_pad ? i : 0);
    if (i >= 0 && i < sc.n_pad && sh.kind >= 0)
        r = scatter(sh.kind, sh.mat, sh.inv_ior, sh.r0s, mk3(dir_in[3 * k], dir_in[3 * k + 1], dir_in[3 * k + 2]), mk3(p[3 * k], p[3 * k + 1], p[3 * k + 2]),
                    mk3(nrm[3 * k], nrm[3 * k + 1], nrm[3 * k + 2]), mk3(rs[3 * k], rs[3 * k + 1], rs[3 * k + 2]), ru[k], g_rsqrt12, a, dd);
    ok[k] = r ? 1 : 0;
    atten[3 * k] = a.x; atten[3 * k + 1] = a.y; atten[3 * k + 2] = a.z;
    dir_out[3 * k] = dd.x; dir_out[3 * k + 1] = dd.y; dir_out[3 * k + 2] = dd.z;
}

__global__ void get_ray_kernel(const __grid_constant__ DevScene sc, int n, const float *su, const float *tv, const float *disk, float *org, float *dir)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    f3 o, d;
    camera_ray(sc.cam, su[k], tv[k], disk[2 * k], disk[2 * k + 1], g_rsqrt12, o, d);
    org[3 * k] = o.x; org[3 * k + 1] = o.y; org[3 * k + 2] = o.z;
    dir[3 * k] = d.x; dir[3 * k + 1] = d.y; dir[3 * k + 2] = d.z;
}

__global__ void rng_kernel(uint32_t pixel, uint32_t sample, uint32_t seed, int n, uint32_t *out)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        Rng rng;
        rng.seed(pixel, sample, Rng::seed_hash(seed));
        for (int i = 0; i < n; ++i) out[i] = rng.draw((uint32_t)i);
    }
}

// The random points of the integrator for given (pixel, sample) keys: primary_ray's lens-disk sample and shade_step's (ru, unit-ball
// sample) of every depth, from the same device functions and draw indices -- the values a CPU cannot reproduce (SFU approximations).
__global__ void sample_points_kernel(int n, const uint32_t *pixel, const uint32_t *sample, uint64_t seed_mix, int bounces, float *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Rng rng;
    rng.seed(pixel[k], sample[k], seed_mix);
    float *o = out + (size_t)k * (2 + 4 * (size_t)bounces);
    float px, py;
    random_in_unit_disk(rng, 2, px, py);
    o[0] = px; o[1] = py;
    for (int depth = 0; depth < bounces; ++depth) {
        const uint32_t draw0 = kDrawsPrimary + kDrawsPerBounce * (uint32_t)depth;
        const float ru = rng.rand01(draw0);
        const f3 rs = random_in_unit_sphere(rng, draw0, ru);
        float *q = o + 2 + 4 * depth;
        q[0] = ru; q[1] = rs.x; q[2] = rs.y; q[3] = rs.z;
    }
}

// ------------------------------------------------------------------------------------------------ replay (parity)
// SURVEY.md 8f rank 4: the pixel loop of render_tile (rayweek1.cpp:752-765) for one pixel per thread, driven by the
// REFERENCE's generators from recorded states instead of the counter-based RNG: xorshift32 13/17/15 (mymath.h:17-25), the
// x4 stream for jitter and the unit-ball rejection loop (mymath.h:41-73, 224-235), the scalar stream for the lens-disk
// rejection loop and the dielectric coin (rayweek1.cpp:353-362, 503).  Everything else -- camera_ray, scan, exact test,
// hit_finalise, scatter, sky -- is the production device code, so this compares the GPU integrator with the reference's
// color() sample by sample.  Attenuations are multiplied innermost-first like the recursion (rayweek1.cpp:525).
struct RefRng {
    uint32_t state, s4[4];
    __device__ __forceinline__ static uint32_t step(uint32_t &x) { x ^= x << 13; x ^= x >> 17; x ^= x << 15; return x; }
    __device__ __forceinline__ float rand01() { return fmul((float)(step(state) & 0xFFFFFFu), 5.9604644775390625e-8f); }
    __device__ __forceinline__ float rand02() { return __fdiv_rn((float)(step(state) & 0xFFFFFFu), 8388608.0f); }
    __device__ __forceinline__ void rand_x4(float scale, float (&out)[4])
    {
#pragma unroll
        for (int k = 0; k < 4; ++k) out[k] = fmul((float)(int)(step(s4[k]) & 0xFFFFFFu), scale);
    }
};

__global__ void __launch_bounds__(128) replay_pixels_kernel(const __grid_constant__ DevScene sc, int n, const int32_t *xy, int image_w, int image_h,
                                                            int spp, int max_bounces, const uint32_t *state_in, const uint32_t *state4_in,
                                                            float *color_sum, uint32_t *rays_out)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4 *s_spheres = reinterpret_cast<float4 *>(smem_raw + 16);
    stage_spheres(sc, s_spheres, reinterpret_cast<uint64_t *>(smem_raw));
    const float4 *s_scan = s_spheres, *s_exact = s_spheres + sc.n_pad;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    RefRng rng;
    rng.state = state_in[k];
#pragma unroll
    for (int j = 0; j < 4; ++j) rng.s4[j] = state4_in[4 * k + j];
    const float inv_w = 1.0f / image_w, inv_h = 1.0f / image_h;
    const float fx = (float)xy[2 * k], fy = (float)xy[2 * k + 1];
    f3 col = mk3(0, 0, 0);
    uint32_t rays = 0;
    for (int smp = 0; smp < spp; ++smp) {
        float xi[4];
        rng.rand_x4((float)(1.0 / 16777216.0), xi);                                   // myrand01_x4, lanes 0 and 1 (:759)
        const float u = fmul(fadd(xi[0], fx), inv_w), v = fmul(fadd(xi[1], fy), inv_h);
        float px, py;
        do {                                                                           // random_in_unit_disk: first draw lands in y (gcc)
            py = fsub(rng.rand02(), 1.0f);
            px = fsub(rng.rand02(), 1.0f);
        } while (fadd(fmul(px, px), fmul(py, py)) >= 1.0f);
        f3 o, d;
        camera_ray(sc.cam, u, v, px, py, g_rsqrt12, o, d);
        f3 stack[51];
        int depth = 0;
        f3 leaf = mk3(0, 0, 0);
        for (;;) {
            ++rays;
            float t = kTMax;
            int hit = -1;
            scan<1>(s_scan, s_exact, sc.n8, o, d, kTMin, t, hit);
            if (hit < 0) { leaf = sky(d); break; }
            if (depth >= max_bounces) break;
            f3 p, nrm, atten, nd, rs = mk3(0, 0, 0);
            float ru = 0.0f;
            const ShadeRec sh = load_shade(sc, hit);
            hit_finalise(s_exact[hit], sh.inv_radius, o, d, t, p, nrm);
            const int kind = sh.kind;
            if (kind == 2) {
                ru = rng.rand01();                                                     // Dielectric: one scalar draw (:503)
            } else {
                float r4[4];
                do {                                                                   // random_in_unit_sphere on the x4 stream
                    rng.rand_x4((float)(1.0 / 8388608.0), r4);
                    rs = mk3(fsub(r4[0], 1.0f), fsub(r4[1], 1.0f), fsub(r4[2], 1.0f));
                } while (fadd(fadd(fmul(rs.x, rs.x), fmul(rs.y, rs.y)), fmul(rs.z, rs.z)) >= 1.0f);
            }
            if (!scatter(kind, sh.mat, sh.inv_ior, sh.r0s, d, p, nrm, rs, ru, g_rsqrt12, atten, nd)) break;
            stack[depth++] = atten;
            o = p; d = nd;
        }
        while (depth > 0) { --depth; leaf = mk3(fmul(stack[depth].x, leaf.x), fmul(stack[depth].y, leaf.y), fmul(stack[depth].z, leaf.z)); }
        col = add3(col, leaf);
    }
    color_sum[3 * k] = col.x; color_sum[3 * k + 1] = col.y; color_sum[3 * k + 2] = col.z;
    rays_out[k] = rays;
}

// ------------------------------------------------------------------------------------------------ FP32 peak
// 16 independent accumulator chains per thread; packed = FFMA2 on float2 accumulators.  FLOPs = 2 per FMA.
template <bool kPacked>
__global__ void __launch_bounds__(256) fma_peak_kernel(int iters, float seed, float *sink, long long *cycles)
{
    long long c0, c1;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c0), "+f"(seed));  // seed is an in/out operand: the chains start after this read
    float r = 0.0f;
    if (kPacked) {
        float2 acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = make_float2(seed + k, seed - k);
        const float2 m = make_float2(1.0000001f, 0.9999999f), b = make_float2(seed, -seed);
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = __ffma2_rn(acc[k], m, b);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) r += acc[k].x + acc[k].y;
    } else {
        float acc[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = seed + k;
        const float m = 1.0000001f, b = seed;
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = ffma(acc[k], m, b);
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) r += acc[k];
    }
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c1), "+f"(r));     // r is an in/out operand: read after the chains finish
    if (r == 123.456f) sink[0] = r;  // keep the chains alive
    if (blockIdx.x == 0 && threadIdx.x == 0) cycles[0] = c1 - c0;
}

}  // namespace r1
