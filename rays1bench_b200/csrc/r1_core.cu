// r1_core.cu -- implementation of the device-facing C ABI (include/rays1_b200.h part 1): scene storage, upload,
// render orchestration on one device, parity entry points.  No CPU fallback anywhere: every compute entry point
// returns R1_ERR_CUDA if the CUDA runtime reports an error (including "no device").
// file:line citations are relative to /root/reference/.
#include "../../include/rays1_b200.h"
#include "r1_bvh.h"
#include "r1_bvh_device.h"
#include "r1_internal.h"
#include "r1_kernels.cuh"
#include "r1_move.h"
#include "r1_wavefront.cuh"

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

namespace {

thread_local std::string g_error;

#define fail r1_set_error

#define R1_CUDA(expr)                                                                                        \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess) return fail(R1_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Per-device state of a committed scene: one allocation [scan | exact | mat | inv_radius | kind], one H2D copy.
struct DeviceCtx {
    int device = -1;
    void *block = nullptr;
    size_t block_bytes = 0;
    r1::DevScene dev;
    uint64_t generation = 0;            // r1_scene::generation at the commit
    void *bvh_block = nullptr;          // R1_VARIANT_MEGAKERNEL_BVH: [nodes | leaf records], uploaded on first use or r1_scene_build_bvh
    const float4 *bvh_nodes = nullptr, *bvh_leaves = nullptr;
    uint32_t bvh_n_nodes = 0, bvh_n_leaves = 0, bvh_depth = 0;
    // r1_scene_move_spheres: set once spheres were moved here (the records no longer match the host SoA, the host tree no longer fits)
    bool moved = false;
    void *refit_block = nullptr;        // the tree's [parent | arrivals] for refits, n_nodes words each; freed with the tree
    bool refit_parents = false;         // parent holds the tree's parent references
    unsigned int *move_flag = nullptr;  // result word of the move's value check
};

// Per-device scratch shared by every scene of the process (pixel accumulators, counters, staging, events).
// It outlives scenes so that a render does not pay cudaMalloc/cudaFree; renders on one device are serialised by the
// caller, as the reference's benchmark() calls are (rayweek1.cpp:969-984).
struct Scratch {
    bool ready = false;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    unsigned long long *accum = nullptr; size_t accum_cap = 0;   // npix_local x 4 fixed-point sums
    unsigned int *unit_counter = nullptr;
    unsigned long long *sample_counter = nullptr;
    uint8_t *rgb = nullptr; size_t rgb_cap = 0;
    unsigned long long *num_rays = nullptr;
    unsigned long long *host_rays = nullptr;  // pinned
    r1::ViewRec *views = nullptr; size_t views_cap = 0;          // the view table of the last batch (r1_render_views_device)
    r1::WavefrontBuffers wf;
    // scene blocks of destroyed scenes, kept for the next commit on this device: the reference-facing call builds a new scene
    // per benchmark() (rayweek1.cpp:969-984), and a cudaMalloc + cudaFree per scene and device is most of what the 8-GPU
    // in-process path pays on top of the render (8 serial commits inside a 13 ms step)
    struct Block { void *ptr; size_t bytes; };
    std::vector<Block> scene_blocks;
    cudaEvent_t ev[4] = { nullptr, nullptr, nullptr, nullptr };
    uint32_t last_launches = 0, last_units = 0;
    uint64_t last_samples = 0;
    bool last_wavefront = false;
};

std::mutex g_scratch_mutex;
std::map<int, Scratch> g_scratch;

}  // namespace

int r1_set_error(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

struct r1_scene {
    // SphereSOA (soa_sphere.h:38-53) with the Material hierarchy flattened to (kind, albedo, param)
    std::vector<float> cx, cy, cz, radius_sq, inv_radius, albedo, param;
    std::vector<int32_t> kind;
    r1::Camera cam;
    bool have_camera = false;
    std::map<int, DeviceCtx> ctx;
    int current = -1;  // device of the last commit
    std::unique_ptr<r1::bvh::Bvh> bvh;  // R1_VARIANT_MEGAKERNEL_BVH: built on first need, dropped when the spheres change
    uint64_t generation = 0;            // counts changes to the spheres
};

namespace {

constexpr size_t kSceneBlockCache = 4;   // blocks kept per device (<= 4 x 260 KB)

void free_ctx(DeviceCtx &c)
{
    if (c.device < 0) return;
    if (c.bvh_block || c.refit_block || c.move_flag) {
        cudaSetDevice(c.device);
        if (c.bvh_block) cudaFree(c.bvh_block);
        if (c.refit_block) cudaFree(c.refit_block);
        if (c.move_flag) cudaFree(c.move_flag);
    }
    bool kept = false;
    {
        std::lock_guard<std::mutex> lock(g_scratch_mutex);
        auto it = g_scratch.find(c.device);
        if (it != g_scratch.end() && it->second.ready && it->second.scene_blocks.size() < kSceneBlockCache) {
            it->second.scene_blocks.push_back({ c.block, c.block_bytes });
            kept = true;
        }
    }
    if (!kept) {
        cudaSetDevice(c.device);
        cudaFree(c.block);
    }
    c = DeviceCtx();
}

// a device block of at least `bytes` for a scene: from the device's cache of released blocks, else cudaMalloc
int take_scene_block(Scratch &scr, size_t bytes, void **out, size_t *out_bytes)
{
    {
        std::lock_guard<std::mutex> lock(g_scratch_mutex);
        for (size_t i = 0; i < scr.scene_blocks.size(); ++i) {
            if (scr.scene_blocks[i].bytes >= bytes && scr.scene_blocks[i].bytes <= 2 * bytes + 4096) {
                *out = scr.scene_blocks[i].ptr; *out_bytes = scr.scene_blocks[i].bytes;
                scr.scene_blocks.erase(scr.scene_blocks.begin() + (long)i);
                return R1_OK;
            }
        }
    }
    R1_CUDA(cudaMalloc(out, bytes));
    *out_bytes = bytes;
    return R1_OK;
}

int get_scratch(int device, Scratch **out)
{
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    Scratch &sc = g_scratch[device];
    if (!sc.ready) {
        R1_CUDA(cudaSetDevice(device));
        R1_CUDA(cudaDeviceGetAttribute(&sc.sm_count, cudaDevAttrMultiProcessorCount, device));
        R1_CUDA(cudaDeviceGetAttribute(&sc.cc_major, cudaDevAttrComputeCapabilityMajor, device));
        R1_CUDA(cudaDeviceGetAttribute(&sc.cc_minor, cudaDevAttrComputeCapabilityMinor, device));
        R1_CUDA(cudaMalloc(&sc.unit_counter, sizeof(unsigned int)));
        R1_CUDA(cudaMalloc(&sc.sample_counter, sizeof(unsigned long long)));
        R1_CUDA(cudaMalloc(&sc.num_rays, sizeof(unsigned long long)));
        R1_CUDA(cudaMallocHost(&sc.host_rays, sizeof(unsigned long long)));
        for (auto &e : sc.ev) R1_CUDA(cudaEventCreate(&e));
        sc.ready = true;
    }
    *out = &sc;
    return R1_OK;
}

void v3_unit(float *v)
{
    const float inv = 1.0f / std::sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
    v[0] *= inv; v[1] *= inv; v[2] *= inv;
}

template <typename T>
int grow(T *&ptr, size_t &cap, size_t need)
{
    if (need <= cap) return R1_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr; cap = 0;
    R1_CUDA(cudaMalloc(&ptr, need * sizeof(T)));
    cap = need;
    return R1_OK;
}

int get_ctx(r1_scene *scene, DeviceCtx **out, int device = -1)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (device < 0) device = scene->current;
    auto it = scene->ctx.find(device);
    if (device < 0 || it == scene->ctx.end()) return fail(R1_ERR_STATE, "scene not committed to device %d (call r1_scene_commit)", device);
    R1_CUDA(cudaSetDevice(device));
    *out = &it->second;
    return R1_OK;
}

// Interleave granularity of the multi-GPU partition.  Measured on the large scene at 8 ranks: 8-row tiles leave the ranks'
// ray counts 4.5 % apart (max / mean), single rows 0.08 %.
constexpr int kDefaultRowTile = 1;

// One sample per unit up to 256 spp (more only to keep the unit count below 2^32 on huge renders): the accumulators are
// order-free, so the unit size affects scheduling granularity only, never the image.
int samples_per_unit(int spp) { return std::max(1, (spp + 255) / 256); }

// Pixels per r1::resolve launch: its 32-bit grid-stride index (at most sm_count x 8 x 256 apart) cannot wrap below 2^31 pixels.
constexpr uint32_t kResolvePixels = 1u << 31;

struct Partition { int local_rows; uint32_t npix_local; };

Partition partition(int width, int height, int row_tile, int rank, int world)
{
    Partition p;
    p.local_rows = (int)r1_local_rows(height, row_tile, rank, world);
    p.npix_local = (uint32_t)p.local_rows * (uint32_t)width;
    return p;
}

// One persistent CTA per SM; kThreads = 512 / 768 / 1024 (4 / 6 / 8 warps per scheduler; ptxas fits 96 / 76 / 64 registers
// without spills).  Shared memory = 16 + n_pad * 32 bytes.
constexpr int kDefaultThreads = 1024;     // per-lane scans: 64 registers
constexpr int kDefaultThreadsCoop = 512;  // cooperative scan: 4 rays per lane in flight, 127 registers

// streamed tensor-core filter (r1::megakernel_tcs, R1_VARIANT_MEGAKERNEL_TENSOR_STREAM): `threads` / 128 = ray groups per CTA (one
// 128-column TMEM accumulator each), kDefaultTcsStages = depth of the operand ring.  Shared memory does not depend on the scene.
// Measured on synth4096 at 1280x720x250 (B200, 1000 W; DESIGN.md section 4.7, profiles/r03_bench_tensor_stream.json): 4 groups with
// 2 / 3 / 4 / 6 stages 1279 / 1324 / 1350 / 1358 Mrays/s; 3 / 2 / 1 groups with 6 stages 1120 / 806 / 415 (PACKED: 827).
constexpr int kDefaultTcsGroups = 4, kDefaultTcsStages = 6;

// BVH traversal (megakernel_pool<kScanBvh>, R1_VARIANT_MEGAKERNEL_BVH): nothing is staged.
// Measured at 640x360x32 (B200, DESIGN.md section 4.8), Mrays/s for 512 / 768 / 1024 threads: large
// 7143 / 8264 / 8531, 10^5-sphere cloud 527 / 705 / 789, 10^5-sphere grid 2603 / 3331 / 3565.  Samples per atomic (sched_kmax x 32,
// shrinking by sched_div) at 512 threads, kmax,div = 64,16 / 8,16 / 1,1: large 7143 / 7114 / 6716, cloud 527 / 529 / 525.
constexpr int kDefaultThreadsBvh = 1024;
constexpr uint32_t kBvhSchedKmax = 64, kBvhSchedDiv = 16;

// The tuning knobs of the environment.  Read on every render, so that a caller can change them between renders.
struct Knobs {
    bool force_unstaged = false;        // R1_FORCE_UNSTAGED: scan from global memory even where the scene could be staged
    uint32_t sched_kmax = 0, sched_div = 0;   // R1_SCHED "kmax,div" (1 .. 4096, 1 .. 1024) overrides the scheduling; 0: not set
};

Knobs read_knobs()
{
    Knobs k;
    k.force_unstaged = getenv("R1_FORCE_UNSTAGED") != nullptr;
    if (const char *e = getenv("R1_SCHED")) {
        unsigned kmax = 0, div = 0;
        if (sscanf(e, "%u,%u", &kmax, &div) == 2 && kmax >= 1 && kmax <= 4096 && div >= 1 && div <= 1024) { k.sched_kmax = kmax; k.sched_div = div; }
    }
    return k;
}

// Samples per atomic (guided self-scheduling).  The sample pool: a WARP takes kmax x 32 consecutive samples per atomicAdd, shrinking
// as left / (div x lanes) towards the end.  Measured on B200 (large scene, Mrays/s, full image | rank 0 of 8 = the per-GPU share of
// the 8-GPU partition):  1,1: 6066 | 6057   2,16: 6102 | 6088   4,16: 6121 | 6088   8,16: 6132 | 6103.  Small scenes need long
// ranges: with 32 samples per atomic the one counter line in L2 saturates (small scene 39 G rays/s instead of 58).  BVH traversals
// are short at every scene size (DESIGN.md section 4.8).
void pick_schedule(const r1::DevScene &dev, int variant, const Knobs &k, r1::RenderArgs &a)
{
    if (variant == R1_VARIANT_MEGAKERNEL_BVH) { a.sched_kmax = kBvhSchedKmax; a.sched_div = kBvhSchedDiv; }
    else if (dev.n8 >= 256) { a.sched_kmax = 8; a.sched_div = 16; }
    else { a.sched_kmax = 64; a.sched_div = 16; }
    if (k.sched_kmax) { a.sched_kmax = k.sched_kmax; a.sched_div = k.sched_div; }
}

using RenderKernel = void (*)(r1::RenderArgs);

// Launches a persistent render kernel: blocks_per_sm CTAs per SM (at least one), but never more CTAs than ceil(work / work_per_cta),
// the CTAs that have work to take.  `what` names the kernel in the shared-memory refusal.
int launch_persistent(RenderKernel kern, int threads, size_t smem, unsigned long long work, unsigned long long work_per_cta, int blocks_per_sm,
                      int sm_count, const char *what, const r1::RenderArgs &args, cudaStream_t stream)
{
    if (smem > 227 * 1024) return fail(R1_ERR_LIMIT, "%s: %d threads need %zu bytes of shared memory for this scene (227 KB available)", what, threads, smem);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned long long max_ctas = std::max<unsigned long long>(1, (work + work_per_cta - 1) / work_per_cta);
    const int grid = (int)std::min<unsigned long long>((unsigned long long)sm_count * (unsigned long long)std::max(blocks_per_sm, 1), max_ctas);
    kern<<<grid, threads, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

// [mbarrier 16 B | rsqrtss table 4 KB | staged spheres n_pad * 32 B | per-warp scan scratch (coop / deferred) | per-warp sample pools]
size_t megakernel_smem(int scan, bool staged, int n_pad, int threads)
{
    return r1::kSmemSpheres + (staged ? (size_t)n_pad * 32 : 0) +
           (scan == r1::kScanCoop || scan == r1::kScanLaneDeferred ? sizeof(r1::WarpScratch) * (threads / 32) : 0) + sizeof(r1::WarpPool) * (threads / 32);
}

// r1::megakernel_pool with the packed, scalar, cooperative or deferred scan.  kViews (a batch of views, packed scan only): the
// default thread count is the only instance.
template <int kScan, bool kStaged, bool kViews>
int launch_megakernel(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    int threads = prm.threads > 0 ? prm.threads : (kScan == r1::kScanCoop ? kDefaultThreadsCoop : kDefaultThreads);
    // The deferred scan's 2 KB of queue per warp: with the sample pool, 1024 threads and more than 3 936 staged spheres exceed
    // 227 KB of shared memory.  The default then runs 768 threads (the image does not depend on the thread count).
    if (prm.threads <= 0 && megakernel_smem(kScan, kStaged, args.scene.n_pad, threads) > 227 * 1024) threads = 768;
    RenderKernel kern = nullptr;
    if constexpr (!kViews) {
        if (threads == 512) kern = r1::megakernel_pool<kScan, kStaged, 512, 1, false>;
        if (threads == 768) kern = r1::megakernel_pool<kScan, kStaged, 768, 1, false>;
    }
    if (threads == 1024) kern = r1::megakernel_pool<kScan, kStaged, 1024, 1, kViews>;
    if (!kern) return fail(R1_ERR_ARG, "threads must be 512, 768 or 1024 (got %d)", threads);
    return launch_persistent(kern, threads, megakernel_smem(kScan, kStaged, args.scene.n_pad, threads), args.n_samples, threads, prm.blocks_per_sm, sm_count,
                             "megakernel_pool", args, stream);
}

template <bool kViews>
int launch_megakernel_bvh(int sm_count, const r1::RenderArgs &args, const float4 *nodes, const float4 *leaves, const r1_render_params &prm,
                          cudaStream_t stream)
{
    const int threads = prm.threads > 0 ? prm.threads : kDefaultThreadsBvh;
    const r1::BvhArgs b = { nodes, leaves };
    R1_CUDA(cudaMemcpyToSymbolAsync(r1::c_bvh, &b, sizeof(b), 0, cudaMemcpyHostToDevice, stream));
    RenderKernel kern = nullptr;
    if constexpr (!kViews) {
        if (threads == 512) kern = r1::megakernel_pool<r1::kScanBvh, false, 512, 1, false>;
        if (threads == 768) kern = r1::megakernel_pool<r1::kScanBvh, false, 768, 1, false>;
    }
    if (threads == 1024) kern = r1::megakernel_pool<r1::kScanBvh, false, 1024, 1, kViews>;
    if (!kern) return fail(R1_ERR_ARG, "the bvh variant runs 512, 768 or 1024 threads (got %d)", threads);
    return launch_persistent(kern, threads, megakernel_smem(r1::kScanBvh, false, args.scene.n_pad, threads), args.n_samples, threads, prm.blocks_per_sm,
                             sm_count, "bvh variant", args, stream);
}

// two paths per lane (r1::megakernel_pool2, R1_VARIANT_MEGAKERNEL_DUAL)
template <bool kStaged>
int launch_megakernel_dual(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    const int threads = prm.threads > 0 ? prm.threads : 768;
    RenderKernel kern = nullptr;
    if (threads == 512) kern = r1::megakernel_pool2<kStaged, 512, 1>;
    if (threads == 768) kern = r1::megakernel_pool2<kStaged, 768, 1>;
    if (!kern) return fail(R1_ERR_ARG, "the dual variant runs 512 or 768 threads (got %d)", threads);
    return launch_persistent(kern, threads, megakernel_smem(r1::kScanLanePacked, kStaged, args.scene.n_pad, threads), args.n_samples, 2ull * threads,
                             prm.blocks_per_sm, sm_count, "dual variant", args, stream);
}

// tensor-core filter (r1::megakernel_tc3, R1_VARIANT_MEGAKERNEL_TENSOR): `threads` / 128 = ray groups per CTA, one CTA per SM
template <bool kViews>
int launch_megakernel_tc(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    if (!args.scene.tcb) return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (its operand lives in shared memory)", r1::tc::kMaxSpheres);
    // ray groups per CTA; measured on the large scene: 4 groups 9.70, 5: 10.34, 6: 9.92, 7: 9.69 G rays/s
    const int groups = prm.threads > 0 ? prm.threads / 128 : 5;
    RenderKernel kern = nullptr;
    if (groups == 5) kern = r1::megakernel_tc3<5, kViews>;
    if constexpr (!kViews) {
        if (groups == 4) kern = r1::megakernel_tc3<4, false>;
        if (groups == 6) kern = r1::megakernel_tc3<6, false>;
        if (groups == 7) kern = r1::megakernel_tc3<7, false>;
    }
    if (!kern) return fail(R1_ERR_ARG, "the tensor variant runs 4 .. 7 groups of 128 ray threads per CTA (threads = 512 .. 896)");
    return launch_persistent(kern, groups * 128, r1::tc3_smem_bytes(groups, args.scene.n32), args.n_samples, groups * 128, 1, sm_count, "tensor variant", args,
                             stream);
}

// streamed tensor-core filter (r1::megakernel_tcs): one CTA per SM
template <bool kViews>
int launch_megakernel_tcs(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    const int groups = prm.threads > 0 ? prm.threads / 128 : kDefaultTcsGroups;
    RenderKernel kern = nullptr;
    if (groups == 4) kern = r1::megakernel_tcs<4, kDefaultTcsStages, kViews>;
    if constexpr (!kViews) {
        if (groups == 3) kern = r1::megakernel_tcs<3, kDefaultTcsStages, false>;
        if (groups == 2) kern = r1::megakernel_tcs<2, kDefaultTcsStages, false>;
        if (groups == 1) kern = r1::megakernel_tcs<1, kDefaultTcsStages, false>;
    }
    if (!kern) return fail(R1_ERR_ARG, "the tensor-stream variant runs 1 .. 4 groups of 128 ray threads per CTA (threads = 128 .. 512, got %d groups)", groups);
    return launch_persistent(kern, groups * 128, r1::tcs_smem_bytes(groups, kDefaultTcsStages), args.n_samples, groups * 128, 1, sm_count, "tensor-stream variant",
                             args, stream);
}

// The host BVH of the scene, built on first need (r1_bvh.h).
int scene_bvh(r1_scene *scene, const r1::bvh::Bvh **out)
{
    if (!scene->bvh) {
        std::unique_ptr<r1::bvh::Bvh> b(new r1::bvh::Bvh());
        if (!r1::bvh::build(scene->cx.data(), scene->cy.data(), scene->cz.data(), scene->radius_sq.data(), scene->inv_radius.data(),
                            (uint32_t)scene->cx.size(), *b))
            return fail(R1_ERR_LIMIT, "the bvh takes fewer than 2^28 spheres that can be hit");
        if (b->depth > (uint32_t)r1::bvh::kMaxDepth) return fail(R1_ERR_LIMIT, "bvh depth %u exceeds %d", b->depth, r1::bvh::kMaxDepth);
        scene->bvh = std::move(b);
    }
    *out = scene->bvh.get();
    return R1_OK;
}

// Makes blk = [n_nodes nodes | n_leaves leaf records] the tree BVH renders and traces on c's device use, freeing the one it replaces.
void set_ctx_bvh(DeviceCtx &c, void *blk, uint32_t n_nodes, uint32_t n_leaves, uint32_t depth)
{
    if (c.bvh_block) cudaFree(c.bvh_block);
    if (c.refit_block) cudaFree(c.refit_block);
    c.refit_block = nullptr;
    c.refit_parents = false;
    c.bvh_block = blk;
    c.bvh_nodes = static_cast<const float4 *>(blk);
    c.bvh_leaves = reinterpret_cast<const float4 *>(static_cast<unsigned char *>(blk) + (size_t)n_nodes * sizeof(r1::bvh::Node));
    c.bvh_n_nodes = n_nodes; c.bvh_n_leaves = n_leaves; c.bvh_depth = depth;
}

// The host tree on c's device: a synchronous copy into an allocation of its own, freed with the context.  ms (optional): CUDA
// events around the copies.
int upload_bvh(DeviceCtx &c, const r1::bvh::Bvh &b, double *ms)
{
    const size_t nb = b.nodes.size() * sizeof(r1::bvh::Node), lb = b.leaves.size() * sizeof(r1::bvh::LeafRec);
    R1_CUDA(cudaSetDevice(c.device));
    void *blk = nullptr;
    R1_CUDA(cudaMalloc(&blk, nb + lb + 16));
    r1::PhaseTimer tm;
    cudaError_t e = ms ? tm.start() : cudaSuccess;
    if (e == cudaSuccess) e = cudaMemcpy(blk, b.nodes.data(), nb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && lb) e = cudaMemcpy(static_cast<unsigned char *>(blk) + nb, b.leaves.data(), lb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && ms) e = tm.stop();
    if (e != cudaSuccess) { cudaFree(blk); return fail(R1_ERR_CUDA, "bvh upload: %s", cudaGetErrorString(e)); }
    if (ms) *ms = tm.ms;
    set_ctx_bvh(c, blk, (uint32_t)b.nodes.size(), (uint32_t)b.leaves.size(), b.depth);
    return R1_OK;
}

// The scene's BVH on the context's device: unless r1_scene_build_bvh put one there, the host tree is built and uploaded on the
// first BVH render or trace.  Refused when the spheres changed after the commit: the device's shading and exact records would no
// longer match the tree.
int ctx_bvh(r1_scene *scene, DeviceCtx &c)
{
    if (c.bvh_block) return R1_OK;
    if (c.moved)
        return fail(R1_ERR_STATE, "spheres were moved on device %d and it holds no bvh of them: build one with r1_scene_build_bvh(..., R1_BVH_BUILD_DEVICE, ...)", c.device);
    if (c.generation != scene->generation) return fail(R1_ERR_STATE, "the scene's spheres changed after it was committed to device %d (commit it again)", c.device);
    const r1::bvh::Bvh *b = nullptr;
    int rc = scene_bvh(scene, &b);
    if (rc) return rc;
    return upload_bvh(c, *b, nullptr);
}

// R1_VARIANT_MEGAKERNEL = the fastest megakernel for the scene.  Measured on B200: the tensor-core filter wins on the large scene
// (485 spheres: 10.3 against 6.2 G rays/s) and loses where a scan is short (medium, 58 spheres: 25 against 34 G).  Explicit
// tuning knobs (blocks_per_sm, threads, R1_FORCE_UNSTAGED) address the packed kernel.
int resolve_variant(const r1::DevScene &dev, const r1_render_params &prm, const Knobs &k)
{
    if (prm.variant != R1_VARIANT_MEGAKERNEL) return prm.variant;
    const bool tuned = prm.blocks_per_sm > 0 || prm.threads > 0 || k.force_unstaged;
    if (dev.tcb && dev.n8 >= 256 && !tuned) return R1_VARIANT_MEGAKERNEL_TENSOR;
    return R1_VARIANT_MEGAKERNEL_PACKED;
}

// 8 and 10 stay unassigned (include/rays1_b200.h)
bool known_variant(int v) { return v >= 0 && v <= R1_VARIANT_MEGAKERNEL_BVH && v != 8 && v != 10; }

int validate(const r1_render_params *p)
{
    if (!p) return fail(R1_ERR_ARG, "null params");
    if (p->width <= 0 || p->height <= 0 || p->spp <= 0 || p->max_bounces < 0) return fail(R1_ERR_ARG, "width/height/spp must be > 0, max_bounces >= 0");
    if (p->world <= 0 || p->rank < 0 || p->rank >= p->world) return fail(R1_ERR_ARG, "bad rank/world %d/%d", p->rank, p->world);
    if ((uint64_t)p->width * (uint64_t)p->height > (1ull << 31)) return fail(R1_ERR_ARG, "image too large");
    // the pixel accumulators hold sums of radiance * 2^24 in 64 bits, one sample saturating at 2^32 - 1 (r1_kernels.cuh): 2^20
    // samples per pixel cannot wrap them
    if (p->spp > (1 << 20)) return fail(R1_ERR_LIMIT, "spp %d exceeds the accumulator limit of 2^20 samples per pixel", p->spp);
    if (!known_variant(p->variant)) return fail(R1_ERR_ARG, "unknown variant %d", p->variant);
    return R1_OK;
}

}  // namespace

extern "C" {

int r1_abi_version(void) { return R1_ABI_VERSION; }
const char *r1_last_error(void) { return g_error.c_str(); }

int r1_device_count(void)
{
    int n = 0;
    R1_CUDA(cudaGetDeviceCount(&n));
    return n;
}

r1_scene *r1_scene_create(uint32_t capacity_hint)
{
    r1_scene *s = new r1_scene();
    memset(&s->cam, 0, sizeof(s->cam));
    s->cx.reserve(capacity_hint); s->cy.reserve(capacity_hint); s->cz.reserve(capacity_hint);
    s->radius_sq.reserve(capacity_hint); s->inv_radius.reserve(capacity_hint);
    s->albedo.reserve(3 * (size_t)capacity_hint); s->param.reserve(capacity_hint); s->kind.reserve(capacity_hint);
    return s;
}

void r1_scene_destroy(r1_scene *scene)
{
    if (!scene) return;
    for (auto &kv : scene->ctx) free_ctx(kv.second);
    delete scene;
}

}  // extern "C"

namespace {
// The 22 camera constants in r1_scene_get_camera's order, to and from r1::Camera.
void camera_to_constants(const r1::Camera &c, float *out)
{
    const float *src[7] = { c.origin, c.llc, c.horizontal, c.vertical, c.u, c.v, c.w };
    for (int k = 0; k < 7; ++k) memcpy(out + 3 * k, src[k], 12);
    out[21] = c.lens_radius;
}

void camera_from_constants(const float *cam, r1::Camera &c)
{
    float *dst[7] = { c.origin, c.llc, c.horizontal, c.vertical, c.u, c.v, c.w };
    for (int k = 0; k < 7; ++k) memcpy(dst[k], cam + 3 * k, 12);
    c.lens_radius = cam[21];
}
}  // namespace

extern "C" {

// Camera::init (rayweek1.cpp:366-379)
int r1_camera_constants(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov_deg, float aspect, float aperture,
                        float focus_dist, float out[22])
{
    if (!lookfrom || !lookat || !vup || !out) return fail(R1_ERR_ARG, "null argument");
    r1::Camera c;
    // The reference's builders call Camera::init with constants, so gcc folds it at compile time -- after the fast-math
    // reassociation of `vfov * (float)M_PI / 180 / 2` into vfov * C, C = (float)M_PI * (1.0f / 360.0f) -- with tanf and the 1 / sqrtf
    // of unit_vector correctly rounded and everything else in source order.  Evaluated the same way here, the 22 constants have the
    // reference's exact bits for its three scenes (checked against the constants recorded from its binary, tests/test_abi_cpu.py).
    c.lens_radius = aperture / 2;
    const float half_angle_per_degree = (float)M_PI * (1.0f / 360.0f);
    const float half_height = (float)tan((double)(vfov_deg * half_angle_per_degree));
    const float half_width = aspect * half_height;
    for (int k = 0; k < 3; ++k) { c.origin[k] = lookfrom[k]; c.w[k] = lookfrom[k] - lookat[k]; }
    v3_unit(c.w);
    c.u[0] = vup[1] * c.w[2] - vup[2] * c.w[1];
    c.u[1] = vup[2] * c.w[0] - vup[0] * c.w[2];
    c.u[2] = vup[0] * c.w[1] - vup[1] * c.w[0];
    v3_unit(c.u);
    c.v[0] = c.w[1] * c.u[2] - c.w[2] * c.u[1];
    c.v[1] = c.w[2] * c.u[0] - c.w[0] * c.u[2];
    c.v[2] = c.w[0] * c.u[1] - c.w[1] * c.u[0];
    for (int k = 0; k < 3; ++k) {
        c.llc[k] = ((c.origin[k] - (half_width * focus_dist) * c.u[k]) - (half_height * focus_dist) * c.v[k]) - focus_dist * c.w[k];
        c.horizontal[k] = (2 * half_width * focus_dist) * c.u[k];
        c.vertical[k] = (2 * half_height * focus_dist) * c.v[k];
    }
    camera_to_constants(c, out);
    return R1_OK;
}

int r1_scene_set_camera(r1_scene *scene, const float lookfrom[3], const float lookat[3], const float vup[3], float vfov_deg, float aspect,
                        float aperture, float focus_dist)
{
    if (!scene || !lookfrom || !lookat || !vup) return fail(R1_ERR_ARG, "null argument");
    float cam[22];
    const int rc = r1_camera_constants(lookfrom, lookat, vup, vfov_deg, aspect, aperture, focus_dist, cam);
    if (rc) return rc;
    return r1_scene_set_camera_raw(scene, cam);
}

int r1_scene_set_camera_raw(r1_scene *scene, const float cam[22])
{
    if (!scene || !cam) return fail(R1_ERR_ARG, "null argument");
    camera_from_constants(cam, scene->cam);
    scene->have_camera = true;
    return R1_OK;
}

// SphereSOA::add (soa_sphere.cpp:70-85)
int r1_scene_add_sphere(r1_scene *scene, float cx, float cy, float cz, float radius, int mat_kind, float r, float g, float b, float param)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (mat_kind < R1_MAT_NONE || mat_kind > R1_MAT_DIELECTRIC) return fail(R1_ERR_ARG, "unknown material kind %d", mat_kind);
    if (mat_kind == R1_MAT_NONE && radius > 0) return fail(R1_ERR_ARG, "a sphere with radius > 0 needs a material");
    if (mat_kind == R1_MAT_METAL) param = param < 1 ? param : 1;  // Metal ctor, rayweek1.cpp:424
    scene->bvh.reset();
    ++scene->generation;
    scene->cx.push_back(cx); scene->cy.push_back(cy); scene->cz.push_back(cz);
    float radius_sq, inv_radius;
    r1::enc::radius_terms(radius, radius_sq, inv_radius);   // r1_encode.h: r1_scene_move_spheres derives new radii's terms the same way
    scene->radius_sq.push_back(radius_sq);
    scene->inv_radius.push_back(inv_radius);
    scene->kind.push_back(mat_kind);
    scene->albedo.push_back(r); scene->albedo.push_back(g); scene->albedo.push_back(b);
    scene->param.push_back(param);
    return (int)scene->cx.size() - 1;
}

int r1_scene_pad(r1_scene *scene, uint32_t multiple)
{
    if (!scene || multiple == 0) return fail(R1_ERR_ARG, "bad argument");
    while (scene->cx.size() % multiple != 0) {
        int rc = r1_scene_add_sphere(scene, 999999999.0f, 999999999.0f, 999999999.0f, 0.0f, R1_MAT_NONE, 0, 0, 0, 0);
        if (rc < 0) return rc;
    }
    return R1_OK;
}

uint32_t r1_scene_count(const r1_scene *scene) { return scene ? (uint32_t)scene->cx.size() : 0; }

int r1_scene_get_soa(const r1_scene *scene, float *cx, float *cy, float *cz, float *radius_sq, float *inv_radius, int32_t *kind, float *albedo,
                     float *param)
{
    if (!scene || !cx || !cy || !cz || !radius_sq || !inv_radius || !kind || !albedo || !param) return fail(R1_ERR_ARG, "null argument");
    const size_t n = scene->cx.size();
    memcpy(cx, scene->cx.data(), n * 4); memcpy(cy, scene->cy.data(), n * 4); memcpy(cz, scene->cz.data(), n * 4);
    memcpy(radius_sq, scene->radius_sq.data(), n * 4); memcpy(inv_radius, scene->inv_radius.data(), n * 4);
    memcpy(kind, scene->kind.data(), n * 4); memcpy(albedo, scene->albedo.data(), 3 * n * 4); memcpy(param, scene->param.data(), n * 4);
    return R1_OK;
}

int r1_scene_get_camera(const r1_scene *scene, float *out)
{
    if (!scene || !out) return fail(R1_ERR_ARG, "null argument");
    camera_to_constants(scene->cam, out);
    return R1_OK;
}

// The sphere operand of the tensor-core filter (r1_tensor.cuh): n32 rows of 128 bytes, spheres that can never be hit and the
// padding up to a multiple of 32 as rows no ray can flag.  Host arithmetic only.
static void build_tensor_operand(const r1_scene *scene, unsigned char *dst, int n32)
{
    const int n = (int)scene->cx.size();
    memset(dst, 0, (size_t)n32 * r1::tc::kRowBytes);
    for (int i = 0; i < n32; ++i) {
        const bool real = i < n && scene->inv_radius[i] != 0;      // rayweek1.cpp:288-292: inv_radius == 0 spheres never hit
        r1::tc::sphere_row_host(dst, i, real, real ? scene->cx[i] : 0.0, real ? scene->cy[i] : 0.0, real ? scene->cz[i] : 0.0,
                                real ? scene->radius_sq[i] : 0.0);
    }
}

int r1_tensor_operand(const r1_scene *scene, void *out, uint64_t out_bytes, uint32_t *n32_out)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    const int n32 = ((int)scene->cx.size() + 31) / 32 * 32;
    if (n32_out) *n32_out = (uint32_t)n32;
    if (n32 == 0 || n32 > r1::tc::kMaxSpheres) return fail(R1_ERR_LIMIT, "the tensor-core filter takes 1 .. %d spheres (this scene pads to %d)", r1::tc::kMaxSpheres, n32);
    if (!out) return R1_OK;                                        // size query
    if (out_bytes < (uint64_t)n32 * r1::tc::kRowBytes) return fail(R1_ERR_ARG, "operand buffer too small: %llu < %llu bytes", (unsigned long long)out_bytes,
                                                                   (unsigned long long)n32 * r1::tc::kRowBytes);
    build_tensor_operand(scene, static_cast<unsigned char *>(out), n32);
    return R1_OK;
}

int r1_bvh_export(const r1_scene *scene, void *nodes, uint64_t nodes_bytes, void *leaves, uint64_t leaves_bytes, uint32_t *n_nodes,
                  uint32_t *n_leaf_records, uint32_t *depth)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    const r1::bvh::Bvh *b = nullptr;
    { const int rc = scene_bvh(const_cast<r1_scene *>(scene), &b); if (rc) return rc; }   // the cached tree is derived state, not a change to the scene
    if (n_nodes) *n_nodes = (uint32_t)b->nodes.size();
    if (n_leaf_records) *n_leaf_records = (uint32_t)b->leaves.size();
    if (depth) *depth = b->depth;
    const uint64_t nb = b->nodes.size() * sizeof(r1::bvh::Node), lb = b->leaves.size() * sizeof(r1::bvh::LeafRec);
    if (nodes) {
        if (nodes_bytes < nb) return fail(R1_ERR_ARG, "node buffer too small: %llu < %llu bytes", (unsigned long long)nodes_bytes, (unsigned long long)nb);
        memcpy(nodes, b->nodes.data(), nb);
    }
    if (leaves) {
        if (leaves_bytes < lb) return fail(R1_ERR_ARG, "leaf buffer too small: %llu < %llu bytes", (unsigned long long)leaves_bytes, (unsigned long long)lb);
        memcpy(leaves, b->leaves.data(), lb);
    }
    return R1_OK;
}

int r1_scene_commit(r1_scene *scene, int device)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (!scene->have_camera) return fail(R1_ERR_STATE, "camera not set");
    if (scene->cx.empty()) return fail(R1_ERR_STATE, "scene has no spheres");
    int ndev = 0;
    R1_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(R1_ERR_ARG, "device %d out of range (%d visible)", device, ndev);
    R1_CUDA(cudaSetDevice(device));
    Scratch *scr = nullptr;
    int rc = get_scratch(device, &scr);
    if (rc) return rc;
    if (scr->cc_major != 10) return fail(R1_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, scr->cc_major, scr->cc_minor);

    {   // drop a previous commit to this device first; the new context is published only once the upload succeeded
        auto prev = scene->ctx.find(device);
        if (prev != scene->ctx.end()) { free_ctx(prev->second); scene->ctx.erase(prev); }
        if (scene->current == device) scene->current = -1;
    }
    DeviceCtx c;
    c.device = device;

    const int n = (int)scene->cx.size();
    const int n_pad = (n + 15) / 16 * 16;  // one scan supergroup = 16 spheres (the reference pads to SIMD_WIDTH = 8, rayweek1.cpp:575)
    // host image of the device block: [scan n_pad f4 | exact n_pad f4 | shade n_pad x 2 f4 | tensor-filter operand n32 x 128 B].
    // The operand is built for every scene: the streamed filter (r1::tcs_operand) finds it after `shade` at any size, while `tcb`,
    // the resident filter's pointer, stays null above tc::kMaxSpheres.
    const int n32 = (n + 31) / 32 * 32;
    const bool tensor_ok = n32 > 0 && n32 <= r1::tc::kMaxSpheres;
    const size_t tcb_off = (size_t)n_pad * (16 + 16 + 32);
    const size_t bytes = tcb_off + (size_t)n32 * r1::tc::kRowBytes;
    std::vector<unsigned char> host(bytes, 0);
    float *scan = reinterpret_cast<float *>(host.data());
    float4 *exact = reinterpret_cast<float4 *>(host.data()) + n_pad;
    float4 *shade = exact + n_pad;
    for (int i = 0; i < n_pad; ++i) {
        const bool real = i < n && scene->inv_radius[i] != 0;  // rayweek1.cpp:288-292: inv_radius == 0 spheres never hit
        // supergroup lanes and kk (r1_encode.h; r1_scene_move_spheres encodes moved spheres with the same function on the device)
        if (real) r1::enc::scan_lanes(scan, i, true, scene->cx[i], scene->cy[i], scene->cz[i], scene->radius_sq[i]);
        else r1::enc::scan_lanes(scan, i, false, 0.0f, 0.0f, 0.0f, 0.0f);
        if (i < n) {
            exact[i] = make_float4(scene->cx[i], scene->cy[i], scene->cz[i], scene->radius_sq[i]);
            // material and inv_radius (r1_encode.h; r1_scene_set_materials encodes new materials with the same function on the device)
            r1::enc::shade_records(scene->kind[i], scene->albedo[3 * i], scene->albedo[3 * i + 1], scene->albedo[3 * i + 2], scene->param[i],
                                   scene->inv_radius[i], shade[2 * i], shade[2 * i + 1]);
        } else {
            r1::enc::shade_records(R1_MAT_NONE, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, shade[2 * i], shade[2 * i + 1]);
        }
    }
    build_tensor_operand(scene, host.data() + tcb_off, n32);
    rc = take_scene_block(*scr, bytes, &c.block, &c.block_bytes);
    if (rc) return rc;
    {
        const cudaError_t e = cudaMemcpy(c.block, host.data(), bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFree(c.block); return fail(R1_ERR_CUDA, "scene upload: %s", cudaGetErrorString(e)); }
    }
    float4 *d4 = reinterpret_cast<float4 *>(c.block);
    c.dev.scan = d4;
    c.dev.exact = d4 + n_pad;
    c.dev.shade = d4 + 2 * (size_t)n_pad;
    c.dev.n_pad = n_pad;
    c.dev.n8 = (n + 7) / 8 * 8;
    c.dev.n_real = n;
    c.dev.cam = scene->cam;
    c.dev.tcb = tensor_ok ? reinterpret_cast<const unsigned char *>(c.block) + tcb_off : nullptr;
    c.dev.n32 = n32;
    c.generation = scene->generation;
    scene->ctx[device] = c;
    scene->current = device;
    return R1_OK;
}

int64_t r1_local_rows(int height, int row_tile, int rank, int world)
{
    if (row_tile <= 0) row_tile = kDefaultRowTile;
    int64_t rows = 0;
    for (int k = rank, y = rank * row_tile; y < height; k += world, y += world * row_tile) rows += std::min(row_tile, height - y);
    return rows;
}

int64_t r1_local_pixels(int width, int height, int row_tile, int rank, int world) { return r1_local_rows(height, row_tile, rank, world) * width; }

int r1_global_row(int local_row, int row_tile, int rank, int world)
{
    if (row_tile <= 0) row_tile = kDefaultRowTile;
    return r1::global_row(local_row, row_tile, rank, world);
}

int r1_deinterleave_rows(int device, const void *d_gathered, uint64_t stride, void *d_out, int width, int height, int row_tile, int world,
                         void *cuda_stream)
{
    if (!d_gathered || !d_out || width <= 0 || height <= 0 || world <= 0) return fail(R1_ERR_ARG, "bad argument");
    if (row_tile <= 0) row_tile = kDefaultRowTile;
    R1_CUDA(cudaSetDevice(device));
    const size_t total = (size_t)width * height * 3;
    const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
    r1::deinterleave_rows<<<grid, 256, 0, (cudaStream_t)cuda_stream>>>((const uint8_t *)d_gathered, (size_t)stride, (uint8_t *)d_out, width, height,
                                                                        row_tile, world);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

}  // extern "C"

namespace {

// A batch of views (r1_render_views_device): n host camera records of 22 floats and n seeds (null: the render's seed for every view).
struct Views { uint32_t n; const float *cams; const uint32_t *seeds; };

// The refusals of a batch that need no device, in the header's order.  `outputs`: the output pointers are not null.
int check_views(const r1_render_params *params, uint32_t n_views, const float *cams, bool outputs)
{
    int rc = validate(params);
    if (rc) return rc;
    if (n_views == 0) return fail(R1_ERR_ARG, "a batch needs at least one view");
    if (!cams || !outputs) return fail(R1_ERR_ARG, "null argument");
    const int v = params->variant;
    if (v != R1_VARIANT_MEGAKERNEL && v != R1_VARIANT_MEGAKERNEL_PACKED && v != R1_VARIANT_MEGAKERNEL_TENSOR && v != R1_VARIANT_MEGAKERNEL_TENSOR_STREAM &&
        v != R1_VARIANT_MEGAKERNEL_BVH)
        return fail(R1_ERR_ARG, "a batch of views renders with the megakernel, packed, tensor, tensor-stream or bvh variant, not %d", v);
    if (params->threads > 0 || params->blocks_per_sm > 0) return fail(R1_ERR_ARG, "a batch of views runs with default tuning only (threads and blocks_per_sm <= 0)");
    const Partition part = partition(params->width, params->height, params->row_tile, params->rank, params->world);
    const uint64_t batch_pix = (uint64_t)n_views * part.npix_local;
    // a batch pixel is a 32-bit pool entry, and 0xffffffff marks an empty one (kPoolInvalid)
    if (batch_pix >= 0xffffffffull) return fail(R1_ERR_LIMIT, "too many pixels in the batch (%u views x %u local pixels)", n_views, part.npix_local);
    if ((long double)batch_pix * params->spp * params->spp >= 18.0e18L)
        return fail(R1_ERR_LIMIT, "too many samples (%llu x %d spp)", (unsigned long long)batch_pix, params->spp);
    return R1_OK;
}

// r1_render_device, and with `views` r1_render_views_device: enqueues the memsets, the trace kernel and the resolve on the stream.
int enqueue_render(r1_scene *scene, const r1_render_params *params, const Views *views, void *d_rgb, void *d_num_rays, void *cuda_stream, r1_result *result)
{
    int rc = validate(params);
    if (rc) return rc;
    DeviceCtx *cp = nullptr;
    rc = get_ctx(scene, &cp, params->device);
    if (rc) return rc;
    DeviceCtx &c = *cp;
    Scratch *xp = nullptr;
    rc = get_scratch(c.device, &xp);
    if (rc) return rc;
    Scratch &x = *xp;
    if (!d_rgb || !d_num_rays) return fail(R1_ERR_ARG, "null device buffer");
    r1_render_params prm = *params;
    if (prm.row_tile <= 0) prm.row_tile = kDefaultRowTile;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (prm.variant == R1_VARIANT_MEGAKERNEL_BVH) {   // first use on this device: build / upload before the first event
        rc = ctx_bvh(scene, c);
        if (rc) return rc;
    }

    const Partition part = partition(prm.width, prm.height, prm.row_tile, prm.rank, prm.world);
    r1::RenderArgs a;
    memset(&a, 0, sizeof(a));
    a.scene = c.dev;
    a.width = prm.width; a.height = prm.height; a.spp = prm.spp; a.max_bounces = prm.max_bounces;
    a.rank = prm.rank; a.world = prm.world; a.row_tile = prm.row_tile;
    a.npix_local = views ? views->n * part.npix_local : part.npix_local;   // a batch: the views' pixels one after the other
    a.samples_per_unit = samples_per_unit(prm.spp);
    a.n_chunks = (prm.spp + a.samples_per_unit - 1) / a.samples_per_unit;
    if (!views) {   // work units are the wavefront variant's; the kernels a batch runs take samples
        const uint64_t n_units = (uint64_t)a.npix_local * (uint64_t)a.n_chunks;
        if (n_units >= (1ull << 32) - (1ull << 24)) return fail(R1_ERR_LIMIT, "too many work units (%llu)", (unsigned long long)n_units);
        a.n_units = (uint32_t)n_units;
    }
    a.seed = r1::Rng::seed_hash(prm.seed);
    a.inv_w = 1.0f / prm.width; a.inv_h = 1.0f / prm.height;  // rayweek1.cpp:746
    a.inv_spp = (float)(1.0f / prm.spp);                       // rayweek1.cpp:765
    a.magic_chunks = r1::div_magic((uint32_t)a.n_chunks);
    a.magic_width = r1::div_magic((uint32_t)prm.width);
    a.magic_row_tile = r1::div_magic((uint32_t)prm.row_tile);
    const Knobs knobs = read_knobs();
    const int variant = resolve_variant(c.dev, prm, knobs);
    pick_schedule(c.dev, variant, knobs, a);
    a.rgb = (uint8_t *)d_rgb;
    a.num_rays = (unsigned long long *)d_num_rays;
    a.unit_counter = x.unit_counter;
    a.sample_counter = x.sample_counter;
    a.n_samples = (uint64_t)a.npix_local * (uint64_t)prm.spp;
    a.magic_spp = r1::div_magic((uint32_t)prm.spp);
    // __umul64hi(g, magic_spp) is the exact g / spp for g < 2^64 / spp
    if ((long double)a.n_samples * (long double)prm.spp >= 18.0e18L) return fail(R1_ERR_LIMIT, "too many samples (%llu x %d spp)", (unsigned long long)a.npix_local, prm.spp);

    x.last_launches = 0;
    x.last_wavefront = prm.variant == R1_VARIANT_WAVEFRONT;
    x.last_units = a.n_units;
    x.last_samples = (uint64_t)a.npix_local * (uint64_t)prm.spp;
    R1_CUDA(cudaMemsetAsync(d_num_rays, 0, sizeof(unsigned long long), stream));
    R1_CUDA(cudaEventRecord(x.ev[0], stream));
    if (a.npix_local > 0) {
        rc = grow(x.accum, x.accum_cap, (size_t)a.npix_local * 4);
        if (rc) return rc;
        a.accum = x.accum;
        R1_CUDA(cudaMemsetAsync(x.accum, 0, (size_t)a.npix_local * 4 * sizeof(unsigned long long), stream));
        R1_CUDA(cudaMemsetAsync(x.unit_counter, 0, sizeof(unsigned int), stream));
        R1_CUDA(cudaMemsetAsync(x.sample_counter, 0, sizeof(unsigned long long), stream));
        if (views) {   // the view table, on the stream: a batch enqueued before keeps its own
            std::vector<r1::ViewRec> recs(views->n);
            for (uint32_t v = 0; v < views->n; ++v) {
                camera_from_constants(views->cams + 22 * (size_t)v, recs[v].cam);
                recs[v].seed = r1::Rng::seed_hash(views->seeds ? views->seeds[v] : prm.seed);
            }
            rc = grow(x.views, x.views_cap, views->n);
            if (rc) return rc;
            R1_CUDA(cudaMemcpyAsync(x.views, recs.data(), recs.size() * sizeof(r1::ViewRec), cudaMemcpyHostToDevice, stream));
            const r1::ViewArgs va = { x.views, part.npix_local, r1::div_magic(part.npix_local) };
            R1_CUDA(cudaMemcpyToSymbolAsync(r1::c_views, &va, sizeof(va), 0, cudaMemcpyHostToDevice, stream));
        }
        // scenes of up to 4096 spheres are staged in shared memory; R1_FORCE_UNSTAGED=1 exercises the global-memory path on small scenes
        const bool staged = c.dev.n_pad <= r1::kMaxStagedSpheres && !knobs.force_unstaged;
        R1_CUDA(cudaEventRecord(x.ev[1], stream));
        if (variant == R1_VARIANT_WAVEFRONT) {
            if (c.dev.n_pad > r1::kMaxStagedSpheres) return fail(R1_ERR_LIMIT, "the wavefront variant stages at most %d spheres", r1::kMaxStagedSpheres);
            uint32_t launches = 0;
            rc = r1::wavefront_render(x.wf, a, x.sm_count, stream, &launches);
            if (rc) return fail(R1_ERR_CUDA, "wavefront: %s", cudaGetErrorString((cudaError_t)rc));
            x.last_launches += launches;
        } else if (views) {   // one instance per production kernel, default tuning (check_views)
            if (variant == R1_VARIANT_MEGAKERNEL_PACKED) rc = staged ? launch_megakernel<r1::kScanLanePacked, true, true>(x.sm_count, a, prm, stream)
                                                                  : launch_megakernel<r1::kScanLanePacked, false, true>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR) rc = launch_megakernel_tc<true>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR_STREAM) rc = launch_megakernel_tcs<true>(x.sm_count, a, prm, stream);
            else rc = launch_megakernel_bvh<true>(x.sm_count, a, c.bvh_nodes, c.bvh_leaves, prm, stream);
            if (rc) return rc;
            x.last_launches += 1;
        } else {
            if (variant == R1_VARIANT_MEGAKERNEL_PACKED) rc = staged ? launch_megakernel<r1::kScanLanePacked, true, false>(x.sm_count, a, prm, stream)
                                                                  : launch_megakernel<r1::kScanLanePacked, false, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_COOP) rc = staged ? launch_megakernel<r1::kScanCoop, true, false>(x.sm_count, a, prm, stream)
                                                                            : launch_megakernel<r1::kScanCoop, false, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_DEFERRED) rc = staged ? launch_megakernel<r1::kScanLaneDeferred, true, false>(x.sm_count, a, prm, stream)
                                                                                : launch_megakernel<r1::kScanLaneDeferred, false, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR) rc = launch_megakernel_tc<false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR_STREAM) rc = launch_megakernel_tcs<false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_BVH) rc = launch_megakernel_bvh<false>(x.sm_count, a, c.bvh_nodes, c.bvh_leaves, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_DUAL) rc = staged ? launch_megakernel_dual<true>(x.sm_count, a, prm, stream)
                                                                            : launch_megakernel_dual<false>(x.sm_count, a, prm, stream);
            else rc = staged ? launch_megakernel<r1::kScanLaneScalar, true, false>(x.sm_count, a, prm, stream)
                             : launch_megakernel<r1::kScanLaneScalar, false, false>(x.sm_count, a, prm, stream);
            if (rc) return rc;
            x.last_launches += 1;
        }
        R1_CUDA(cudaEventRecord(x.ev[2], stream));
        // resolve's grid-stride index is 32-bit: it ends only while npix_local + stride stays below 2^32.  A single render has at most
        // 2^31 pixels (validate); a batch up to 2^32 - 2, so it is resolved in pieces of at most 2^31 pixels.
        for (uint32_t first = 0; first < a.npix_local; first += std::min<uint32_t>(a.npix_local - first, kResolvePixels)) {
            r1::RenderArgs ra = a;
            ra.accum = a.accum + (size_t)first * 4;
            ra.rgb = a.rgb + (size_t)first * 3;
            ra.npix_local = std::min<uint32_t>(a.npix_local - first, kResolvePixels);
            const int rgrid = (int)std::min<uint64_t>(((uint64_t)ra.npix_local + 255) / 256, (uint64_t)x.sm_count * 8);
            r1::resolve<<<rgrid, 256, 0, stream>>>(ra);
            R1_CUDA(cudaGetLastError());
            x.last_launches += 1;
        }
    } else {
        R1_CUDA(cudaEventRecord(x.ev[1], stream));
        R1_CUDA(cudaEventRecord(x.ev[2], stream));
    }
    R1_CUDA(cudaEventRecord(x.ev[3], stream));
    if (result) {
        memset(result, 0, sizeof(*result));
        result->num_samples = x.last_samples;
        result->launches = x.last_launches;
        result->n_units = x.last_units;
    }
    return R1_OK;
}

}  // namespace

extern "C" {

int r1_render_device(r1_scene *scene, const r1_render_params *params, void *d_rgb, void *d_num_rays, void *cuda_stream, r1_result *result)
{
    return enqueue_render(scene, params, nullptr, d_rgb, d_num_rays, cuda_stream, result);
}

int r1_render_views_device(r1_scene *scene, const r1_render_params *params, uint32_t n_views, const float *cams, const uint32_t *seeds, void *d_rgb,
                           void *d_num_rays, void *cuda_stream, r1_result *result)
{
    int rc = check_views(params, n_views, cams, d_rgb && d_num_rays);
    if (rc) return rc;
    int ndev = 0;
    R1_CUDA(cudaGetDeviceCount(&ndev));   // no device: R1_ERR_CUDA, whether or not the scene was committed
    const Views views = { n_views, cams, seeds };
    return enqueue_render(scene, params, &views, d_rgb, d_num_rays, cuda_stream, result);
}

int r1_render_wait(r1_scene *scene, int device, r1_result *result)
{
    DeviceCtx *cp = nullptr;
    int rc = get_ctx(scene, &cp, device);
    if (rc) return rc;
    Scratch *xp = nullptr;
    rc = get_scratch(cp->device, &xp);
    if (rc) return rc;
    Scratch &x = *xp;
    R1_CUDA(cudaEventSynchronize(x.ev[3]));
    if (result) {
        float ms_all = 0, ms_trace = 0;
        R1_CUDA(cudaEventElapsedTime(&ms_all, x.ev[0], x.ev[3]));
        R1_CUDA(cudaEventElapsedTime(&ms_trace, x.ev[1], x.ev[2]));
        result->kernel_ms = ms_all;
        result->trace_ms = ms_trace;
        result->num_samples = x.last_samples;
        result->launches = x.last_launches;
        result->n_units = x.last_units;
        if (x.last_wavefront && x.wf.d_iterations) {  // wavefront: 3 kernels per loop iteration, counted on the device
            uint32_t iters = 0;
            R1_CUDA(cudaMemcpy(&iters, x.wf.d_iterations, sizeof(iters), cudaMemcpyDeviceToHost));
            result->launches += 3 * iters;
        }
    }
    return R1_OK;
}

int r1_wavefront_graph_builds(int device)
{
    Scratch *xp = nullptr;
    int rc = get_scratch(device, &xp);
    if (rc) return rc;
    return (int)xp->wf.graph_builds;
}

int r1_render(r1_scene *scene, const r1_render_params *params, uint8_t *rgb_host, r1_result *result)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = validate(params);
    if (rc) return rc;
    if (!rgb_host) return fail(R1_ERR_ARG, "null rgb_host");
    DeviceCtx *cp = nullptr;
    rc = get_ctx(scene, &cp, params->device);
    if (rc) return rc;
    Scratch *xp = nullptr;
    rc = get_scratch(cp->device, &xp);
    if (rc) return rc;
    Scratch &x = *xp;
    const Partition part = partition(params->width, params->height, params->row_tile, params->rank, params->world);
    const size_t bytes = (size_t)part.npix_local * 3;
    rc = grow(x.rgb, x.rgb_cap, std::max<size_t>(bytes, 16));
    if (rc) return rc;
    r1_result res;
    rc = r1_render_device(scene, params, x.rgb, x.num_rays, nullptr, &res);
    if (rc) return rc;
    if (bytes) R1_CUDA(cudaMemcpyAsync(rgb_host, x.rgb, bytes, cudaMemcpyDeviceToHost, nullptr));
    R1_CUDA(cudaMemcpyAsync(x.host_rays, x.num_rays, sizeof(unsigned long long), cudaMemcpyDeviceToHost, nullptr));
    R1_CUDA(cudaStreamSynchronize(nullptr));
    rc = r1_render_wait(scene, params->device, &res);
    if (rc) return rc;
    res.num_rays = *x.host_rays;
    res.elapsed_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (result) *result = res;
    return R1_OK;
}

int r1_render_views(r1_scene *scene, const r1_render_params *params, uint32_t n_views, const float *cams, const uint32_t *seeds, uint8_t *rgb_host,
                    uint64_t *sums_host, r1_result *result)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = check_views(params, n_views, cams, rgb_host != nullptr);
    if (rc) return rc;
    int ndev = 0;
    R1_CUDA(cudaGetDeviceCount(&ndev));
    DeviceCtx *cp = nullptr;
    rc = get_ctx(scene, &cp, params->device);
    if (rc) return rc;
    Scratch *xp = nullptr;
    rc = get_scratch(cp->device, &xp);
    if (rc) return rc;
    Scratch &x = *xp;
    const size_t npix = (size_t)n_views * partition(params->width, params->height, params->row_tile, params->rank, params->world).npix_local;
    rc = grow(x.rgb, x.rgb_cap, std::max<size_t>(npix * 3, 16));
    if (rc) return rc;
    r1_result res;
    rc = r1_render_views_device(scene, params, n_views, cams, seeds, x.rgb, x.num_rays, nullptr, &res);
    if (rc) return rc;
    if (npix) R1_CUDA(cudaMemcpyAsync(rgb_host, x.rgb, npix * 3, cudaMemcpyDeviceToHost, nullptr));
    R1_CUDA(cudaMemcpyAsync(x.host_rays, x.num_rays, sizeof(unsigned long long), cudaMemcpyDeviceToHost, nullptr));
    R1_CUDA(cudaStreamSynchronize(nullptr));
    rc = r1_render_wait(scene, params->device, &res);
    if (rc) return rc;
    res.num_rays = *x.host_rays;
    if (sums_host && npix) {
        std::vector<unsigned long long> accum(npix * 4);   // (r, g, b, unused) per batch pixel
        R1_CUDA(cudaMemcpy(accum.data(), x.accum, accum.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (size_t p = 0; p < npix; ++p)
            for (int c = 0; c < 3; ++c) sums_host[3 * p + c] = accum[4 * p + c];
    }
    res.elapsed_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (result) *result = res;
    return R1_OK;
}

}  // extern "C"

// ---- parity entry points -------------------------------------------------------------------------------------

namespace {
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) { R1_CUDA(cudaMalloc(&p, std::max<size_t>(bytes, 16))); return R1_OK; }
    int upload(const void *src, size_t bytes) { int rc = alloc(bytes); if (rc) return rc; R1_CUDA(cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice)); return R1_OK; }
    int download(void *dst, size_t bytes) { R1_CUDA(cudaMemcpy(dst, p, bytes, cudaMemcpyDeviceToHost)); return R1_OK; }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};
#define R1_TRY(expr) do { int rc_ = (expr); if (rc_) return rc_; } while (0)

// CUDA events around work enqueued on one stream (device_ms of r1_scene_move_spheres and r1_scene_set_materials)
struct StreamTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    ~StreamTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    int start(cudaStream_t stream)
    {
        R1_CUDA(cudaEventCreate(&a));
        R1_CUDA(cudaEventCreate(&b));
        R1_CUDA(cudaEventRecord(a, stream));
        return R1_OK;
    }
    int stop(cudaStream_t stream, double *ms_out)
    {
        R1_CUDA(cudaEventRecord(b, stream));
        R1_CUDA(cudaEventSynchronize(b));
        float ms = 0;
        R1_CUDA(cudaEventElapsedTime(&ms, a, b));
        *ms_out = ms;
        return R1_OK;
    }
};

// the records of c's block, in r1_scene_commit's layout
r1::move::Records ctx_records(DeviceCtx &c)
{
    float4 *block = static_cast<float4 *>(c.block);
    return { block, block + c.dev.n_pad, block + 2 * (size_t)c.dev.n_pad, static_cast<unsigned char *>(c.block) + (size_t)c.dev.n_pad * (16 + 16 + 32) };
}

// r1_trace_rays through the BVH: any sphere count
int trace_rays_bvh(r1_scene *scene, DeviceCtx &c, int n, const float *org, const float *dir, float t_min, float t_max, int32_t *index, float *t,
                   float *p, float *normal)
{
    R1_TRY(ctx_bvh(scene, c));
    DevBuf d_org, d_dir, d_idx, d_t, d_p, d_n;
    R1_TRY(d_org.upload(org, (size_t)n * 12)); R1_TRY(d_dir.upload(dir, (size_t)n * 12));
    R1_TRY(d_idx.alloc((size_t)n * 4)); R1_TRY(d_t.alloc((size_t)n * 4)); R1_TRY(d_p.alloc((size_t)n * 12)); R1_TRY(d_n.alloc((size_t)n * 12));
    r1::trace_rays_bvh_kernel<<<(n + 127) / 128, 128>>>(c.dev, n, d_org.as<float>(), d_dir.as<float>(), t_min, t_max, d_idx.as<int32_t>(), d_t.as<float>(),
                                                        d_p.as<float>(), d_n.as<float>(), c.bvh_nodes, c.bvh_leaves);
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d_idx.download(index, (size_t)n * 4)); R1_TRY(d_t.download(t, (size_t)n * 4));
    R1_TRY(d_p.download(p, (size_t)n * 12)); R1_TRY(d_n.download(normal, (size_t)n * 12));
    return R1_OK;
}

// The LBVH of the committed scene, built on c's device (r1_bvh_device.cu) and installed as its tree.
int build_device_bvh(DeviceCtx &c, double *ms)
{
    R1_CUDA(cudaSetDevice(c.device));
    r1::lbvh::Built out;
    R1_TRY(r1::lbvh::build(c.dev.exact, c.dev.shade, (uint32_t)c.dev.n_real, &out, ms));
    set_ctx_bvh(c, out.block, out.n_nodes, out.n_leaves, out.depth);
    return R1_OK;
}

}  // namespace

extern "C" {

int r1_scene_build_bvh(r1_scene *scene, int device, int builder, double *device_ms)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (builder != R1_BVH_BUILD_HOST && builder != R1_BVH_BUILD_DEVICE) return fail(R1_ERR_ARG, "unknown bvh builder %d", builder);
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp, device));
    if (cp->generation != scene->generation) return fail(R1_ERR_STATE, "the scene's spheres changed after it was committed to device %d (commit it again)", cp->device);
    double ms = 0;
    if (builder == R1_BVH_BUILD_HOST) {
        if (cp->moved)
            return fail(R1_ERR_STATE, "spheres were moved on device %d: the host tree describes the committed positions (build with R1_BVH_BUILD_DEVICE, or commit again)", cp->device);
        const r1::bvh::Bvh *b = nullptr;
        R1_TRY(scene_bvh(scene, &b));
        R1_TRY(upload_bvh(*cp, *b, &ms));
    } else {
        R1_TRY(build_device_bvh(*cp, &ms));
    }
    if (device_ms) *device_ms = ms;
    return R1_OK;
}

int r1_bvh_export_device(r1_scene *scene, int device, void *nodes, uint64_t nodes_bytes, void *leaves, uint64_t leaves_bytes, uint32_t *n_nodes,
                         uint32_t *n_leaf_records, uint32_t *depth)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (device < 0) device = scene->current;
    auto it = scene->ctx.find(device);
    if (device < 0 || it == scene->ctx.end()) return fail(R1_ERR_STATE, "scene not committed to device %d (call r1_scene_commit)", device);
    const DeviceCtx &c = it->second;
    if (!c.bvh_block) return fail(R1_ERR_STATE, "device %d holds no bvh of this scene", device);
    if (n_nodes) *n_nodes = c.bvh_n_nodes;
    if (n_leaf_records) *n_leaf_records = c.bvh_n_leaves;
    if (depth) *depth = c.bvh_depth;
    const uint64_t nb = (uint64_t)c.bvh_n_nodes * sizeof(r1::bvh::Node), lb = (uint64_t)c.bvh_n_leaves * sizeof(r1::bvh::LeafRec);
    if (nodes && nodes_bytes < nb) return fail(R1_ERR_ARG, "node buffer too small: %llu < %llu bytes", (unsigned long long)nodes_bytes, (unsigned long long)nb);
    if (leaves && leaves_bytes < lb) return fail(R1_ERR_ARG, "leaf buffer too small: %llu < %llu bytes", (unsigned long long)leaves_bytes, (unsigned long long)lb);
    R1_CUDA(cudaSetDevice(c.device));
    if (nodes) R1_CUDA(cudaMemcpy(nodes, c.bvh_nodes, nb, cudaMemcpyDeviceToHost));
    if (leaves && lb) R1_CUDA(cudaMemcpy(leaves, c.bvh_leaves, lb, cudaMemcpyDeviceToHost));
    return R1_OK;
}

int r1_scene_move_spheres(r1_scene *scene, int device, uint32_t first, uint32_t n, const float *d_centre, const float *d_radius, void *cuda_stream,
                          double *device_ms)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    const uint64_t count = scene->cx.size();
    if ((uint64_t)first + n > count)
        return fail(R1_ERR_ARG, "spheres %u .. %u + %u - 1 are out of range (the scene has %llu)", first, first, n, (unsigned long long)count);
    if (n > 0 && !d_centre) return fail(R1_ERR_ARG, "null centres");
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp, device));
    DeviceCtx &c = *cp;
    if (c.generation != scene->generation) return fail(R1_ERR_STATE, "the scene's spheres changed after it was committed to device %d (commit it again)", c.device);
    if (device_ms) *device_ms = 0;
    if (n == 0) return R1_OK;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (!c.move_flag) R1_CUDA(cudaMalloc(&c.move_flag, 16));
    if (c.bvh_block && !c.refit_block) R1_CUDA(cudaMalloc(&c.refit_block, (size_t)c.bvh_n_nodes * 8 + 16));
    StreamTimer ev;
    if (device_ms) R1_TRY(ev.start(stream));
    const r1::move::Records rec = ctx_records(c);
    R1_TRY(r1::move::check(rec, first, n, d_centre, d_radius, c.move_flag, stream));   // nothing is written unless every value passes
    R1_TRY(r1::move::encode(rec, first, n, d_centre, d_radius, stream));
    c.moved = true;                                                // the records no longer match the host scene
    if (c.bvh_block) {
        int *parent = static_cast<int *>(c.refit_block);
        unsigned int *arrivals = reinterpret_cast<unsigned int *>(parent + c.bvh_n_nodes);
        float4 *nodes = static_cast<float4 *>(c.bvh_block);
        R1_TRY(r1::lbvh::refit(nodes, const_cast<float4 *>(c.bvh_leaves), c.bvh_n_nodes, rec.exact, parent, arrivals, c.refit_parents, stream));
        c.refit_parents = true;
    }
    if (device_ms) R1_TRY(ev.stop(stream, device_ms));
    R1_CUDA(cudaStreamSynchronize(stream));
    return R1_OK;
}

int r1_scene_move_camera(r1_scene *scene, int device, const float cam[22])
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (!cam) return fail(R1_ERR_ARG, "null camera constants");
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp, device));
    if (cp->generation != scene->generation) return fail(R1_ERR_STATE, "the scene's spheres changed after it was committed to device %d (commit it again)", cp->device);
    camera_from_constants(cam, cp->dev.cam);   // read by value when a render or parity kernel is launched
    return R1_OK;
}

int r1_scene_set_materials(r1_scene *scene, int device, uint32_t first, uint32_t n, const int32_t *d_kind, const float *d_albedo, const float *d_param,
                           void *cuda_stream, double *device_ms)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    const uint64_t count = scene->cx.size();
    if ((uint64_t)first + n > count)
        return fail(R1_ERR_ARG, "spheres %u .. %u + %u - 1 are out of range (the scene has %llu)", first, first, n, (unsigned long long)count);
    if (n > 0 && !d_kind && !d_albedo && !d_param) return fail(R1_ERR_ARG, "no material field given (kind, albedo and param are all null)");
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp, device));
    DeviceCtx &c = *cp;
    if (c.generation != scene->generation) return fail(R1_ERR_STATE, "the scene's spheres changed after it was committed to device %d (commit it again)", c.device);
    if (device_ms) *device_ms = 0;
    if (n == 0) return R1_OK;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (d_kind && !c.move_flag) R1_CUDA(cudaMalloc(&c.move_flag, 16));
    StreamTimer ev;
    if (device_ms) R1_TRY(ev.start(stream));
    const r1::move::Records rec = ctx_records(c);
    if (d_kind) R1_TRY(r1::move::check_materials(rec, first, n, d_kind, c.move_flag, stream));   // only new kinds can be refused
    R1_TRY(r1::move::encode_materials(rec, first, n, d_kind, d_albedo, d_param, stream));
    // neither the geometry nor the tree changes: c.moved stays as it is, and a device without a tree may still upload the host's
    if (device_ms) R1_TRY(ev.stop(stream, device_ms));
    R1_CUDA(cudaStreamSynchronize(stream));
    return R1_OK;
}

int r1_scene_export_device(r1_scene *scene, int device, void *out, uint64_t out_bytes, uint64_t *bytes)
{
    if (!scene) return fail(R1_ERR_ARG, "null scene");
    if (device < 0) device = scene->current;
    auto it = scene->ctx.find(device);
    if (device < 0 || it == scene->ctx.end()) return fail(R1_ERR_STATE, "scene not committed to device %d (call r1_scene_commit)", device);
    const DeviceCtx &c = it->second;
    const uint64_t nb = (uint64_t)c.dev.n_pad * (16 + 16 + 32) + (uint64_t)c.dev.n32 * r1::tc::kRowBytes;   // r1_scene_commit's layout
    if (bytes) *bytes = nb;
    if (!out) return R1_OK;
    if (out_bytes < nb) return fail(R1_ERR_ARG, "record buffer too small: %llu < %llu bytes", (unsigned long long)out_bytes, (unsigned long long)nb);
    R1_CUDA(cudaSetDevice(c.device));
    R1_CUDA(cudaMemcpy(out, c.block, nb, cudaMemcpyDeviceToHost));
    return R1_OK;
}

int r1_trace_rays(r1_scene *scene, int n, const float *org, const float *dir, float t_min, float t_max, int variant, int32_t *index, float *t,
                  float *p, float *normal)
{
    // The exact test lifts discr to 2^-100 before its square root, and the cooperative and deferred scans merge roots as unsigned
    // keys: both agree with Hitable::hit only for t_min >= 2^-24 (r1_device.cuh, exact_test).  Renders use 0.001.  !(>=) rejects NaN.
    if (!(t_min >= 0x1p-24f)) return fail(R1_ERR_ARG, "t_min must be >= 2^-24 (5.96e-8), got %g", (double)t_min);
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || (n > 0 && (!org || !dir || !index || !t || !p || !normal))) return fail(R1_ERR_ARG, "bad argument");
    // R1_VARIANT_MEGAKERNEL resolves as in r1_render; the variants without a per-ray kernel of their own are refused
    r1_render_params prm;
    memset(&prm, 0, sizeof(prm));
    prm.variant = variant;
    if (!known_variant(variant)) return fail(R1_ERR_ARG, "unknown variant %d", variant);
    const int v = resolve_variant(cp->dev, prm, read_knobs());
    if (v == R1_VARIANT_WAVEFRONT || v == R1_VARIANT_MEGAKERNEL_DUAL) return fail(R1_ERR_ARG, "r1_trace_rays has no kernel for variant %d (wavefront, dual)", v);
    if (v == R1_VARIANT_MEGAKERNEL_TENSOR && !cp->dev.tcb)
        return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (this scene pads to %d)", r1::tc::kMaxSpheres, cp->dev.n32);
    if (n == 0) return R1_OK;
    if (v == R1_VARIANT_MEGAKERNEL_BVH) return trace_rays_bvh(scene, *cp, n, org, dir, t_min, t_max, index, t, p, normal);
    // the streamed filter takes any size; the other kernels stage the whole scene in shared memory
    if (v != R1_VARIANT_MEGAKERNEL_TENSOR_STREAM && cp->dev.n_pad > r1::kMaxStagedSpheres) return fail(R1_ERR_LIMIT, "r1_trace_rays stages at most %d spheres", r1::kMaxStagedSpheres);
    DevBuf d_org, d_dir, d_idx, d_t, d_p, d_n;
    R1_TRY(d_org.upload(org, (size_t)n * 12)); R1_TRY(d_dir.upload(dir, (size_t)n * 12));
    R1_TRY(d_idx.alloc((size_t)n * 4)); R1_TRY(d_t.alloc((size_t)n * 4)); R1_TRY(d_p.alloc((size_t)n * 12)); R1_TRY(d_n.alloc((size_t)n * 12));
    const size_t smem = v == R1_VARIANT_MEGAKERNEL_TENSOR          ? r1::trace_rays_tc_smem_bytes(cp->dev.n32)
                        : v == R1_VARIANT_MEGAKERNEL_TENSOR_STREAM ? r1::trace_rays_tcs_smem_bytes()
                                                                   : 16 + (size_t)cp->dev.n_pad * 32 + sizeof(r1::WarpScratch) * 4;
    const int grid = (n + 127) / 128;
    auto launch = [&](auto kern) -> int {
        R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 128, smem>>>(cp->dev, n, d_org.as<float>(), d_dir.as<float>(), t_min, t_max, d_idx.as<int32_t>(), d_t.as<float>(), d_p.as<float>(),
                                  d_n.as<float>());
        return R1_OK;
    };
    if (v == R1_VARIANT_MEGAKERNEL_SCALAR) R1_TRY(launch(r1::trace_rays_kernel<r1::kScanLaneScalar>));
    else if (v == R1_VARIANT_MEGAKERNEL_COOP) R1_TRY(launch(r1::trace_rays_kernel<r1::kScanCoop>));
    else if (v == R1_VARIANT_MEGAKERNEL_DEFERRED) R1_TRY(launch(r1::trace_rays_kernel<r1::kScanLaneDeferred>));
    else if (v == R1_VARIANT_MEGAKERNEL_TENSOR) R1_TRY(launch(r1::trace_rays_tc_kernel));
    else if (v == R1_VARIANT_MEGAKERNEL_TENSOR_STREAM) R1_TRY(launch(r1::trace_rays_tcs_kernel));
    else R1_TRY(launch(r1::trace_rays_kernel<r1::kScanLanePacked>));
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d_idx.download(index, (size_t)n * 4)); R1_TRY(d_t.download(t, (size_t)n * 4));
    R1_TRY(d_p.download(p, (size_t)n * 12)); R1_TRY(d_n.download(normal, (size_t)n * 12));
    return R1_OK;
}

const char *r1_kernel_name(r1_scene *scene, int variant)
{
    DeviceCtx *cp = nullptr;
    if (get_ctx(scene, &cp)) return "";
    r1_render_params prm;
    memset(&prm, 0, sizeof(prm));
    prm.variant = variant;
    switch (resolve_variant(cp->dev, prm, read_knobs())) {
    case R1_VARIANT_WAVEFRONT: return "wf_intersect + wf_shade (graph loop)";
    case R1_VARIANT_MEGAKERNEL_TENSOR: return "megakernel_tc3";
    case R1_VARIANT_MEGAKERNEL_DUAL: return "megakernel_pool2";
    case R1_VARIANT_MEGAKERNEL_TENSOR_STREAM: return "megakernel_tcs";
    case R1_VARIANT_MEGAKERNEL_BVH: return "megakernel_bvh";
    default: return "megakernel_pool";
    }
}

int r1_filter_probe(r1_scene *scene, int n, const float *org, const float *dir, int layout, float *e)
{
    if (layout != 0) return fail(R1_ERR_ARG, "r1_filter_probe: layout must be 0, got %d", layout);
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || (n > 0 && (!org || !dir || !e))) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    if (!cp->dev.tcb) return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (its operand lives in shared memory)", r1::tc::kMaxSpheres);
    const int n32 = cp->dev.n32;
    DevBuf d_org, d_dir, d_e;
    R1_TRY(d_org.upload(org, (size_t)n * 12)); R1_TRY(d_dir.upload(dir, (size_t)n * 12));
    R1_TRY(d_e.alloc((size_t)n * n32 * 4));
    const size_t smem = r1::filter_probe_smem_bytes(n32);
    R1_CUDA(cudaFuncSetAttribute(r1::tc_filter_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    r1::tc_filter_probe_kernel<<<(n + 127) / 128, 128, smem>>>(cp->dev, n, d_org.as<float>(), d_dir.as<float>(), d_e.as<float>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d_e.download(e, (size_t)n * n32 * 4));
    return R1_OK;
}

int r1_scatter(r1_scene *scene, int n, const float *dir_in, const float *p, const float *normal, const int32_t *index, const float *rand_sphere,
               const float *rand_u, int32_t *ok, float *atten, float *dir_out)
{
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || (n > 0 && (!dir_in || !p || !normal || !index || !rand_sphere || !rand_u || !ok || !atten || !dir_out))) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    DevBuf a, b, c, d, e, f, g, h, i;
    R1_TRY(a.upload(dir_in, (size_t)n * 12)); R1_TRY(b.upload(p, (size_t)n * 12)); R1_TRY(c.upload(normal, (size_t)n * 12));
    R1_TRY(d.upload(index, (size_t)n * 4)); R1_TRY(e.upload(rand_sphere, (size_t)n * 12)); R1_TRY(f.upload(rand_u, (size_t)n * 4));
    R1_TRY(g.alloc((size_t)n * 4)); R1_TRY(h.alloc((size_t)n * 12)); R1_TRY(i.alloc((size_t)n * 12));
    r1::scatter_kernel<<<(n + 127) / 128, 128>>>(cp->dev, n, a.as<float>(), b.as<float>(), c.as<float>(), d.as<int32_t>(), e.as<float>(), f.as<float>(),
                                                 g.as<int32_t>(), h.as<float>(), i.as<float>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(g.download(ok, (size_t)n * 4)); R1_TRY(h.download(atten, (size_t)n * 12)); R1_TRY(i.download(dir_out, (size_t)n * 12));
    return R1_OK;
}

int r1_get_ray(r1_scene *scene, int n, const float *su, const float *tv, const float *disk, float *org, float *dir)
{
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || (n > 0 && (!su || !tv || !disk || !org || !dir))) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    DevBuf a, b, c, d, e;
    R1_TRY(a.upload(su, (size_t)n * 4)); R1_TRY(b.upload(tv, (size_t)n * 4)); R1_TRY(c.upload(disk, (size_t)n * 8));
    R1_TRY(d.alloc((size_t)n * 12)); R1_TRY(e.alloc((size_t)n * 12));
    r1::get_ray_kernel<<<(n + 127) / 128, 128>>>(cp->dev, n, a.as<float>(), b.as<float>(), c.as<float>(), d.as<float>(), e.as<float>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d.download(org, (size_t)n * 12)); R1_TRY(e.download(dir, (size_t)n * 12));
    return R1_OK;
}

int r1_replay_pixels(r1_scene *scene, int n, const int32_t *xy, int width, int height, int spp, int max_bounces, const uint32_t *state,
                     const uint32_t *state4, float *color_sum, uint32_t *num_rays)
{
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || width <= 0 || height <= 0 || spp <= 0 || max_bounces < 0 || max_bounces > 50 || (n > 0 && (!xy || !state || !state4 || !color_sum || !num_rays)))
        return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    if (cp->dev.n_pad > r1::kMaxStagedSpheres) return fail(R1_ERR_LIMIT, "r1_replay_pixels stages at most %d spheres", r1::kMaxStagedSpheres);
    DevBuf a, b, c, d, e;
    R1_TRY(a.upload(xy, (size_t)n * 8)); R1_TRY(b.upload(state, (size_t)n * 4)); R1_TRY(c.upload(state4, (size_t)n * 16));
    R1_TRY(d.alloc((size_t)n * 12)); R1_TRY(e.alloc((size_t)n * 4));
    const size_t smem = 16 + (size_t)cp->dev.n_pad * 32;
    R1_CUDA(cudaFuncSetAttribute(r1::replay_pixels_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    r1::replay_pixels_kernel<<<(n + 127) / 128, 128, smem>>>(cp->dev, n, a.as<int32_t>(), width, height, spp, max_bounces, b.as<uint32_t>(), c.as<uint32_t>(),
                                                            d.as<float>(), e.as<uint32_t>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d.download(color_sum, (size_t)n * 12)); R1_TRY(e.download(num_rays, (size_t)n * 4));
    return R1_OK;
}

int r1_rng_draws(uint32_t pixel, uint32_t sample, uint32_t seed, int n, uint32_t *out)
{
    if (n < 0 || (n > 0 && !out)) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    DevBuf d;
    R1_TRY(d.alloc((size_t)n * 4));
    r1::rng_kernel<<<1, 32>>>(pixel, sample, seed, n, d.as<uint32_t>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d.download(out, (size_t)n * 4));
    return R1_OK;
}

int r1_sample_points(int n, const uint32_t *pixel, const uint32_t *sample, uint32_t seed, int bounces, float *out)
{
    if (n < 0 || bounces < 0 || bounces > 1024 || (n > 0 && (!pixel || !sample || !out))) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    const size_t per_key = 2 + 4 * (size_t)bounces;
    DevBuf d_pixel, d_sample, d_out;
    R1_TRY(d_pixel.upload(pixel, (size_t)n * 4)); R1_TRY(d_sample.upload(sample, (size_t)n * 4));
    R1_TRY(d_out.alloc((size_t)n * per_key * 4));
    r1::sample_points_kernel<<<(n + 127) / 128, 128>>>(n, d_pixel.as<uint32_t>(), d_sample.as<uint32_t>(), r1::Rng::seed_hash(seed), bounces, d_out.as<float>());
    R1_CUDA(cudaGetLastError());
    R1_CUDA(cudaDeviceSynchronize());
    R1_TRY(d_out.download(out, (size_t)n * per_key * 4));
    return R1_OK;
}

int r1_render_sums(r1_scene *scene, const r1_render_params *params, uint64_t *sums, uint8_t *rgb_host, r1_result *result)
{
    R1_TRY(validate(params));
    if (!scene || !sums || !rgb_host) return fail(R1_ERR_ARG, "null argument");
    int ndev = 0;
    R1_CUDA(cudaGetDeviceCount(&ndev));
    R1_TRY(r1_render(scene, params, rgb_host, result));   // returns after the render and its copies have completed
    const Partition part = partition(params->width, params->height, params->row_tile, params->rank, params->world);
    if (part.npix_local == 0) return R1_OK;
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp, params->device));
    Scratch *xp = nullptr;
    R1_TRY(get_scratch(cp->device, &xp));
    std::vector<unsigned long long> accum((size_t)part.npix_local * 4);   // (r, g, b, unused) per local pixel
    R1_CUDA(cudaMemcpy(accum.data(), xp->accum, accum.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    for (size_t lp = 0; lp < part.npix_local; ++lp)
        for (int c = 0; c < 3; ++c) sums[3 * lp + c] = accum[4 * lp + c];
    return R1_OK;
}

int r1_tmem_read_peak(int device, int warps, double *bytes_per_second_per_sm)
{
    if (!bytes_per_second_per_sm || warps < 1 || warps > 32) return fail(R1_ERR_ARG, "bad argument");
    R1_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    R1_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf sink;
    R1_TRY(sink.alloc(16));
    cudaEvent_t e0, e1;
    R1_CUDA(cudaEventCreate(&e0)); R1_CUDA(cudaEventCreate(&e1));
    const int iters = 20000;
    r1::tmem_read_kernel<<<prop.multiProcessorCount, warps * 32>>>(100, sink.as<uint32_t>());   // warm-up
    R1_CUDA(cudaEventRecord(e0));
    r1::tmem_read_kernel<<<prop.multiProcessorCount, warps * 32>>>(iters, sink.as<uint32_t>());
    R1_CUDA(cudaEventRecord(e1));
    R1_CUDA(cudaEventSynchronize(e1));
    R1_CUDA(cudaGetLastError());
    float ms = 0;
    R1_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *bytes_per_second_per_sm = (double)warps * iters * 4096.0 / (ms * 1e-3);
    return R1_OK;
}

int r1_fma_peak(int device, int packed, double *tflops, double *sm_mhz_est)
{
    if (!tflops) return fail(R1_ERR_ARG, "null argument");
    R1_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    R1_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf sink, cyc;
    R1_TRY(sink.alloc(16)); R1_TRY(cyc.alloc(16));
    const int iters = 1 << 16, threads = 256, grid = prop.multiProcessorCount * 8;
    struct Events {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Events() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
    } ev;
    R1_CUDA(cudaEventCreate(&ev.e0)); R1_CUDA(cudaEventCreate(&ev.e1));
    cudaEvent_t e0 = ev.e0, e1 = ev.e1;
    double best_ms = 1e30, mhz = 0;
    for (int rep = 0; rep < 4; ++rep) {  // first repetition is the warm-up
        R1_CUDA(cudaEventRecord(e0));
        if (packed) r1::fma_peak_kernel<true><<<grid, threads>>>(iters, 0.5f, sink.as<float>(), cyc.as<long long>());
        else r1::fma_peak_kernel<false><<<grid, threads>>>(iters, 0.5f, sink.as<float>(), cyc.as<long long>());
        R1_CUDA(cudaEventRecord(e1));
        R1_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        R1_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        long long cycles = 0;
        R1_TRY(cyc.download(&cycles, sizeof(cycles)));
        // all 8 x 256-thread CTAs per SM are resident (one wave), so one CTA's cycle count spans the kernel
        if (rep > 0 && ms < best_ms) { best_ms = ms; mhz = (double)cycles / (ms * 1e-3) / 1e6; }
    }
    const double fmas = (double)grid * threads * (double)iters * 16.0;  // 16 scalar FMAs or 8 packed (= 16) per iteration
    *tflops = 2.0 * fmas / (best_ms * 1e-3) / 1e12;
    if (sm_mhz_est) *sm_mhz_est = mhz;
    return R1_OK;
}

}  // extern "C"
