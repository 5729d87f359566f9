// r1_core.cu -- implementation of the device-facing C ABI (include/rays1_b200.h part 1): scene storage, upload,
// render orchestration on one device, parity entry points.  No CPU fallback anywhere: every compute entry point
// returns R1_ERR_CUDA if the CUDA runtime reports an error (including "no device").
// file:line citations are relative to /root/reference/.
#include "../../include/rays1_b200.h"
#include "r1_internal.h"
#include "r1_kernels.cuh"
#include "r1_wavefront.cuh"

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
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
};

namespace {

constexpr size_t kSceneBlockCache = 4;   // blocks kept per device (<= 4 x 260 KB)

void free_ctx(DeviceCtx &c)
{
    if (c.device < 0) return;
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

template <int kScan, bool kStaged, int kThreads>
int launch_megakernel_lanefetch(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    constexpr int kBlocks = 1;
    auto kern = r1::megakernel<kScan, kStaged, kThreads, kBlocks>;
    const size_t smem = r1::kSmemSpheres + (kStaged ? (size_t)args.scene.n_pad * 32 : 0) + (kScan == r1::kScanCoop || kScan == r1::kScanLaneDeferred ? sizeof(r1::WarpScratch) * (kThreads / 32) : 0);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count * kBlocks;
    if (prm.blocks_per_sm > 0) grid = sm_count * prm.blocks_per_sm;
    // never launch more lanes than there are units
    const long long max_ctas = ((long long)args.n_units + kThreads - 1) / kThreads;
    if (grid > max_ctas) grid = (int)std::max<long long>(1, max_ctas);
    kern<<<grid, kThreads, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

// warp sample-pool scheduling (r1::megakernel_pool): the default; R1_POOL=0 selects the per-lane unit fetch of r1::megakernel
size_t megakernel_pool_smem(int scan, bool staged, int n_pad, int threads)
{
    return r1::kSmemSpheres + (staged ? (size_t)n_pad * 32 : 0) +
           (scan == r1::kScanCoop || scan == r1::kScanLaneDeferred ? sizeof(r1::WarpScratch) * (threads / 32) : 0) + sizeof(r1::WarpPool) * (threads / 32);
}

template <int kScan, bool kStaged, int kThreads>
int launch_megakernel_pool(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    constexpr int kBlocks = 1;
    auto kern = r1::megakernel_pool<kScan, kStaged, kThreads, kBlocks>;
    const size_t smem = megakernel_pool_smem(kScan, kStaged, args.scene.n_pad, kThreads);
    if (smem > 227 * 1024) return fail(R1_ERR_LIMIT, "%d threads need %zu bytes of shared memory for this scene (227 KB available)", kThreads, smem);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count * kBlocks;
    if (prm.blocks_per_sm > 0) grid = sm_count * prm.blocks_per_sm;
    const unsigned long long max_ctas = (args.n_samples + kThreads - 1) / kThreads;   // never launch more lanes than there are samples
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kThreads, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

// two paths per lane (r1::megakernel_pool2, R1_VARIANT_MEGAKERNEL_DUAL)
template <bool kStaged, int kThreads>
int launch_megakernel_dual_t(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    auto kern = r1::megakernel_pool2<kStaged, kThreads, 1>;
    const size_t smem = r1::kSmemSpheres + (kStaged ? (size_t)args.scene.n_pad * 32 : 0) + sizeof(r1::WarpPool) * (kThreads / 32);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count * (prm.blocks_per_sm > 0 ? prm.blocks_per_sm : 1);
    const unsigned long long max_ctas = (args.n_samples + 2 * kThreads - 1) / (2 * kThreads);
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kThreads, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

template <bool kStaged>
int launch_megakernel_dual(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    const int threads = prm.threads > 0 ? prm.threads : 768;
    if (threads == 512) return launch_megakernel_dual_t<kStaged, 512>(sm_count, args, prm, stream);
    if (threads == 768) return launch_megakernel_dual_t<kStaged, 768>(sm_count, args, prm, stream);
    return fail(R1_ERR_ARG, "the dual variant runs 512 or 768 threads (got %d)", threads);
}

// tensor-core filter (r1::megakernel_tc, R1_VARIANT_MEGAKERNEL_TENSOR): `threads` selects the number of 128-ray groups per CTA,
// R1_TC_CFG="chunk,buffers" the TMEM pipeline (columns per accumulator buffer, buffers per group; groups x buffers x chunk <= 512)
template <int kGroups, int kChunk, int kBufs, bool kATmem>
int launch_megakernel_tc_t(int sm_count, const r1::RenderArgs &args, cudaStream_t stream)
{
    auto kern = r1::megakernel_tc<kGroups, kChunk, kBufs, kATmem>;
    const size_t smem = r1::tc_smem_bytes(kGroups, args.scene.n32);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count;                                         // one CTA per SM: it owns all 512 TMEM columns
    const unsigned long long max_ctas = (args.n_samples + kGroups * 128 - 1) / (kGroups * 128);
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kGroups * 160, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

template <int kGroups, int kChunk, int kBufs>
int launch_megakernel_tc2_t(int sm_count, const r1::RenderArgs &args, cudaStream_t stream)
{
    auto kern = r1::megakernel_tc2<kGroups, kChunk, kBufs>;
    const size_t smem = r1::tc2_smem_bytes(kGroups, args.scene.n32);
    if (smem > 227 * 1024) return fail(R1_ERR_LIMIT, "tensor variant: %d ray groups need %zu bytes of shared memory for this scene", kGroups, smem);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count;
    const unsigned long long max_ctas = (args.n_samples + kGroups * 128 - 1) / (kGroups * 128);
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kGroups * 128, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

template <int kGroups>
int launch_megakernel_tc3_t(int sm_count, const r1::RenderArgs &args, cudaStream_t stream)
{
    auto kern = r1::megakernel_tc3<kGroups>;
    const size_t smem = r1::tc2_smem_bytes(kGroups, args.scene.n32);
    if (smem > 227 * 1024) return fail(R1_ERR_LIMIT, "tensor variant: %d ray groups need %zu bytes of shared memory for this scene", kGroups, smem);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count;
    const unsigned long long max_ctas = (args.n_samples + kGroups * 128 - 1) / (kGroups * 128);
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kGroups * 128, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

// streamed tensor-core filter (r1::megakernel_tcs, R1_VARIANT_MEGAKERNEL_TENSOR_STREAM): `threads` / 128 = ray groups per CTA (one
// 128-column TMEM accumulator each), R1_TCS_STAGES = depth of the operand ring.  Shared memory does not depend on the scene.
// Measured on synth4096 at 1280x720x250 (B200, 1000 W; DESIGN.md section 4.7, profiles/r03_bench_tensor_stream.json): 4 groups with
// 2 / 3 / 4 / 6 stages 1279 / 1324 / 1350 / 1358 Mrays/s; 3 / 2 / 1 groups with 6 stages 1120 / 806 / 415 (PACKED: 827).
constexpr int kDefaultTcsGroups = 4, kDefaultTcsStages = 6;

template <int kGroups, int kStages>
int launch_megakernel_tcs_t(int sm_count, const r1::RenderArgs &args, cudaStream_t stream)
{
    auto kern = r1::megakernel_tcs<kGroups, kStages>;
    const size_t smem = r1::tcs_smem_bytes(kGroups, kStages);
    if (smem > 227 * 1024) return fail(R1_ERR_LIMIT, "tensor-stream variant: %d ray groups and %d stages need %zu bytes of shared memory", kGroups, kStages, smem);
    R1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count;                                         // one CTA per SM
    const unsigned long long max_ctas = (args.n_samples + kGroups * 128 - 1) / (kGroups * 128);
    if ((unsigned long long)grid > max_ctas) grid = (int)std::max<unsigned long long>(1, max_ctas);
    kern<<<grid, kGroups * 128, smem, stream>>>(args);
    R1_CUDA(cudaGetLastError());
    return R1_OK;
}

int launch_megakernel_tcs(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    const int groups = prm.threads > 0 ? prm.threads / 128 : kDefaultTcsGroups;
    const int stages = getenv("R1_TCS_STAGES") ? atoi(getenv("R1_TCS_STAGES")) : kDefaultTcsStages;
    if (groups == 4 && stages == 2) return launch_megakernel_tcs_t<4, 2>(sm_count, args, stream);
    if (groups == 4 && stages == 3) return launch_megakernel_tcs_t<4, 3>(sm_count, args, stream);
    if (groups == 4 && stages == 4) return launch_megakernel_tcs_t<4, 4>(sm_count, args, stream);
    if (groups == 4 && stages == 6) return launch_megakernel_tcs_t<4, 6>(sm_count, args, stream);
    if (groups == 3 && stages == 6) return launch_megakernel_tcs_t<3, 6>(sm_count, args, stream);
    if (groups == 2 && stages == 6) return launch_megakernel_tcs_t<2, 6>(sm_count, args, stream);
    if (groups == 1 && stages == 6) return launch_megakernel_tcs_t<1, 6>(sm_count, args, stream);
    return fail(R1_ERR_ARG, "the tensor-stream variant runs 1 .. 4 groups of 128 ray threads per CTA (threads = 128 .. 512) with a 6-stage ring, "
                            "or 4 groups with 2, 3, 4 or 6 stages (got %d groups, %d stages)", groups, stages);
}

int launch_megakernel_tc(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    if (!args.scene.tcb) return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (its operand lives in shared memory)", r1::tc::kMaxSpheres);
    if (!getenv("R1_TC1") && !getenv("R1_TC2")) {
        // r1::megakernel_tc3 (default): the last ray warp to arrive issues the MMA, accumulator buffers pooled among the groups;
        // R1_TC3 (or threads / 128) = ray groups per CTA.  Measured on the large scene: 4 groups 9.70, 5: 10.34, 6: 9.92, 7: 9.69 G rays/s
        const int groups = getenv("R1_TC3") ? atoi(getenv("R1_TC3")) : (prm.threads > 0 ? prm.threads / 128 : 5);
        if (groups == 4) return launch_megakernel_tc3_t<4>(sm_count, args, stream);
        if (groups == 5) return launch_megakernel_tc3_t<5>(sm_count, args, stream);
        if (groups == 6) return launch_megakernel_tc3_t<6>(sm_count, args, stream);
        if (groups == 7) return launch_megakernel_tc3_t<7>(sm_count, args, stream);
        return fail(R1_ERR_ARG, "the tensor variant runs 4 .. 7 groups of 128 ray threads per CTA (threads = 512 .. 896)");
    }
    if (!getenv("R1_TC1")) {   // R1_TC2 = groups (A/B): r1::megakernel_tc2, one accumulator buffer (or two: R1_TC2_BUFS=2) owned by each group
        const int groups = atoi(getenv("R1_TC2"));
        const int bufs = getenv("R1_TC2_BUFS") ? atoi(getenv("R1_TC2_BUFS")) : 1;
        if (groups == 4 && bufs == 2) return launch_megakernel_tc2_t<4, 64, 2>(sm_count, args, stream);
        if (groups == 3 && bufs == 2) return launch_megakernel_tc2_t<3, 64, 2>(sm_count, args, stream);
        if (groups == 4) return launch_megakernel_tc2_t<4, 128, 1>(sm_count, args, stream);
        if (groups == 5) return launch_megakernel_tc2_t<5, 96, 1>(sm_count, args, stream);
        if (groups == 6) return launch_megakernel_tc2_t<6, 64, 1>(sm_count, args, stream);
        if (groups == 7) return launch_megakernel_tc2_t<7, 64, 1>(sm_count, args, stream);
        return fail(R1_ERR_ARG, "R1_TC2 must be 3 .. 7");
    }
    // R1_TC1=1: r1::megakernel_tc, one MMA-issuing warp per group (A/B)
    const int threads = prm.threads > 0 ? prm.threads : (getenv("R1_TC_THREADS") ? atoi(getenv("R1_TC_THREADS")) : 512);
    int chunk = 128, bufs = 1, atmem = 0;
    if (const char *e = getenv("R1_TC_CFG")) sscanf(e, "%d,%d,%d", &chunk, &bufs, &atmem);
#define R1_TC_CASE(G, C, B, A) if (threads == G * 128 && chunk == C && bufs == B && atmem == A) return launch_megakernel_tc_t<G, C, B, A != 0>(sm_count, args, stream)
    R1_TC_CASE(4, 128, 1, 0); R1_TC_CASE(4, 64, 2, 0); R1_TC_CASE(4, 96, 1, 1); R1_TC_CASE(4, 32, 3, 1);
    R1_TC_CASE(3, 128, 1, 0); R1_TC_CASE(3, 64, 2, 0); R1_TC_CASE(3, 128, 1, 1); R1_TC_CASE(3, 64, 2, 1);
    R1_TC_CASE(2, 128, 2, 0); R1_TC_CASE(2, 256, 1, 0); R1_TC_CASE(2, 96, 2, 1); R1_TC_CASE(2, 224, 1, 1);
#undef R1_TC_CASE
    return fail(R1_ERR_ARG, "tensor variant: no kernel for %d ray threads, chunk %d, %d buffers, A in %s", threads, chunk, bufs, atmem ? "TMEM" : "shared memory");
}

template <int kScan, bool kStaged, int kThreads>
int launch_megakernel_t(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    const bool pool = !(getenv("R1_POOL") && atoi(getenv("R1_POOL")) == 0);   // read per render, like the other tuning knobs
    if (pool) return launch_megakernel_pool<kScan, kStaged, kThreads>(sm_count, args, prm, stream);
    return launch_megakernel_lanefetch<kScan, kStaged, kThreads>(sm_count, args, prm, stream);
}

template <int kScan, bool kStaged>
int launch_megakernel(int sm_count, const r1::RenderArgs &args, const r1_render_params &prm, cudaStream_t stream)
{
    int threads = prm.threads > 0 ? prm.threads : (kScan == r1::kScanCoop ? kDefaultThreadsCoop : kDefaultThreads);
    // The deferred scan's 2 KB of queue per warp: with the sample pool, 1024 threads and more than 3 936 staged spheres exceed
    // 227 KB of shared memory.  The default then runs 768 threads (the image does not depend on the thread count).
    const bool pool = !(getenv("R1_POOL") && atoi(getenv("R1_POOL")) == 0);
    if (prm.threads <= 0 && pool && megakernel_pool_smem(kScan, kStaged, args.scene.n_pad, threads) > 227 * 1024) threads = 768;
    if (threads == 512) return launch_megakernel_t<kScan, kStaged, 512>(sm_count, args, prm, stream);
    if (threads == 768) return launch_megakernel_t<kScan, kStaged, 768>(sm_count, args, prm, stream);
    if (threads == 1024) return launch_megakernel_t<kScan, kStaged, 1024>(sm_count, args, prm, stream);
    return fail(R1_ERR_ARG, "threads must be 512, 768 or 1024 (got %d)", threads);
}

// R1_VARIANT_MEGAKERNEL = the fastest megakernel for the scene.  Measured on B200: the tensor-core filter wins on the large scene
// (485 spheres: 10.3 against 6.2 G rays/s) and loses where a scan is short (medium, 58 spheres: 25 against 34 G).  Explicit
// tuning knobs (blocks_per_sm, threads, R1_POOL=0) address the packed kernel; R1_AUTO_TENSOR=0 keeps it everywhere.
int resolve_variant(const r1::DevScene &dev, const r1_render_params &prm)
{
    if (prm.variant != R1_VARIANT_MEGAKERNEL) return prm.variant;
    const bool tuned = prm.blocks_per_sm > 0 || prm.threads > 0 || (getenv("R1_POOL") && atoi(getenv("R1_POOL")) == 0) || getenv("R1_FORCE_UNSTAGED");
    const bool off = getenv("R1_AUTO_TENSOR") && atoi(getenv("R1_AUTO_TENSOR")) == 0;
    if (dev.tcb && dev.n8 >= 256 && !tuned && !off) return R1_VARIANT_MEGAKERNEL_TENSOR;
    return R1_VARIANT_MEGAKERNEL_PACKED;
}

int validate(const r1_render_params *p)
{
    if (!p) return fail(R1_ERR_ARG, "null params");
    if (p->width <= 0 || p->height <= 0 || p->spp <= 0 || p->max_bounces < 0) return fail(R1_ERR_ARG, "width/height/spp must be > 0, max_bounces >= 0");
    if (p->world <= 0 || p->rank < 0 || p->rank >= p->world) return fail(R1_ERR_ARG, "bad rank/world %d/%d", p->rank, p->world);
    if ((uint64_t)p->width * (uint64_t)p->height > (1ull << 31)) return fail(R1_ERR_ARG, "image too large");
    // the pixel accumulators hold sums of radiance * 2^24 in 64 bits, one sample saturating at 2^32 - 1 (r1_kernels.cuh): 2^20
    // samples per pixel cannot wrap them
    if (p->spp > (1 << 20)) return fail(R1_ERR_LIMIT, "spp %d exceeds the accumulator limit of 2^20 samples per pixel", p->spp);
    if (p->variant < 0 || p->variant > R1_VARIANT_MEGAKERNEL_TENSOR_STREAM || p->variant == 8) return fail(R1_ERR_ARG, "unknown variant %d", p->variant);
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

// Camera::init (rayweek1.cpp:366-379)
int r1_scene_set_camera(r1_scene *scene, const float lookfrom[3], const float lookat[3], const float vup[3], float vfov_deg, float aspect,
                        float aperture, float focus_dist)
{
    if (!scene || !lookfrom || !lookat || !vup) return fail(R1_ERR_ARG, "null argument");
    r1::Camera &c = scene->cam;
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
    scene->have_camera = true;
    return R1_OK;
}

int r1_scene_set_camera_raw(r1_scene *scene, const float cam[22])
{
    if (!scene || !cam) return fail(R1_ERR_ARG, "null argument");
    r1::Camera &c = scene->cam;
    float *dst[7] = { c.origin, c.llc, c.horizontal, c.vertical, c.u, c.v, c.w };
    for (int k = 0; k < 7; ++k) memcpy(dst[k], cam + 3 * k, 12);
    c.lens_radius = cam[21];
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
    scene->cx.push_back(cx); scene->cy.push_back(cy); scene->cz.push_back(cz);
    scene->radius_sq.push_back(radius * radius);
    scene->inv_radius.push_back(radius > 0 ? (1.0f / radius) : 0);
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
    const r1::Camera &c = scene->cam;
    const float *src[7] = { c.origin, c.llc, c.horizontal, c.vertical, c.u, c.v, c.w };
    for (int k = 0; k < 7; ++k) memcpy(out + 3 * k, src[k], 12);
    out[21] = c.lens_radius;
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
    const float inf = std::numeric_limits<float>::infinity();
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
        // supergroup layout (r1_device.cuh): group g = i / 4 at float4 index (g >> 2) * 16 + (g & 3); cy / cz / r2f at +4 / +8 / +12
        const int g = i / 4, k = i % 4, f4 = (g >> 2) * 16 + (g & 3);
        scan[4 * (f4 + 0) + k] = real ? -scene->cx[i] : 0.0f;
        scan[4 * (f4 + 4) + k] = real ? -scene->cy[i] : 0.0f;
        scan[4 * (f4 + 8) + k] = real ? -scene->cz[i] : 0.0f;
        // kk = |c|^2 - r^2 - 2^-17 |c|^2, evaluated in double and rounded DOWN (r1_device.cuh "Filter arithmetic")
        if (real) {
            const double c2 = (double)scene->cx[i] * scene->cx[i] + (double)scene->cy[i] * scene->cy[i] + (double)scene->cz[i] * scene->cz[i];
            const double kk = c2 - (double)scene->radius_sq[i] - c2 / 131072.0;
            float kf = (float)kk;
            if ((double)kf > kk) kf = std::nextafter(kf, -inf);
            scan[4 * (f4 + 12) + k] = std::nextafter(kf, -inf);
        } else {
            scan[4 * (f4 + 12) + k] = inf;
        }
        int32_t kind = R1_MAT_NONE;
        float inv_r = 0.0f;
        if (i < n) {
            exact[i] = make_float4(scene->cx[i], scene->cy[i], scene->cz[i], scene->radius_sq[i]);
            shade[2 * i] = make_float4(scene->albedo[3 * i], scene->albedo[3 * i + 1], scene->albedo[3 * i + 2], scene->param[i]);
            inv_r = scene->inv_radius[i];
            kind = scene->kind[i];
        }
        float kind_bits, inv_ior = 0.0f, r0s = 0.0f;
        memcpy(&kind_bits, &kind, 4);
        if (kind == R1_MAT_DIELECTRIC) {   // Dielectric::scatter's two divisions (rayweek1.cpp:482, :456), once per sphere, IEEE float
            const volatile float ior = scene->param[i];
            inv_ior = 1.0f / ior;
            r0s = (1.0f - ior) / (ior + 1.0f);
        }
        shade[2 * i + 1] = make_float4(inv_r, kind_bits, inv_ior, r0s);
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

int r1_render_device(r1_scene *scene, const r1_render_params *params, void *d_rgb, void *d_num_rays, void *cuda_stream, r1_result *result)
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

    const Partition part = partition(prm.width, prm.height, prm.row_tile, prm.rank, prm.world);
    r1::RenderArgs a;
    memset(&a, 0, sizeof(a));
    a.scene = c.dev;
    a.width = prm.width; a.height = prm.height; a.spp = prm.spp; a.max_bounces = prm.max_bounces;
    a.rank = prm.rank; a.world = prm.world; a.row_tile = prm.row_tile;
    a.npix_local = part.npix_local;
    a.samples_per_unit = samples_per_unit(prm.spp);
    a.n_chunks = (prm.spp + a.samples_per_unit - 1) / a.samples_per_unit;
    const uint64_t n_units = (uint64_t)a.npix_local * (uint64_t)a.n_chunks;
    if (n_units >= (1ull << 32) - (1ull << 24)) return fail(R1_ERR_LIMIT, "too many work units (%llu)", (unsigned long long)n_units);
    a.n_units = (uint32_t)n_units;
    a.seed = r1::Rng::seed_hash(prm.seed);
    a.inv_w = 1.0f / prm.width; a.inv_h = 1.0f / prm.height;  // rayweek1.cpp:746
    a.inv_spp = (float)(1.0f / prm.spp);                       // rayweek1.cpp:765
    a.magic_chunks = r1::div_magic((uint32_t)a.n_chunks);
    a.magic_width = r1::div_magic((uint32_t)prm.width);
    a.magic_row_tile = r1::div_magic((uint32_t)prm.row_tile);
    // Samples per atomic (guided self-scheduling).  r1::megakernel_pool: a WARP takes kmax x 32 consecutive samples per atomicAdd,
    // shrinking as left / (div x lanes) towards the end.  Measured on B200 (large scene, Mrays/s, full image | rank 0 of 8 = the
    // per-GPU share of the 8-GPU partition):  1,1: 6066 | 6057   2,16: 6102 | 6088   4,16: 6121 | 6088   8,16: 6132 | 6103.
    // Small scenes need long ranges: with 32 samples per atomic the one counter line in L2 saturates (small scene 39 G rays/s
    // instead of 58).  r1::megakernel (R1_POOL=0) hands units to LANES; its round-1 tuning is kept: 1 unit per fetch on
    // scan-heavy scenes (ranges held by lanes at the end of a render are a serial tail), up to 64 on small ones.
    const bool pool_sched = !(getenv("R1_POOL") && atoi(getenv("R1_POOL")) == 0);
    if (c.dev.n8 >= 256) { a.sched_kmax = pool_sched ? 8 : 1; a.sched_div = pool_sched ? 16 : 1; }
    else { a.sched_kmax = 64; a.sched_div = 16; }
    a.tc_flags = getenv("R1_TC_FLAGS") ? (uint32_t)atoi(getenv("R1_TC_FLAGS")) : 1u;
    if (const char *e = getenv("R1_SCHED")) {  // tuning knob: "kmax,div"
        unsigned k = 0, d = 0;
        if (sscanf(e, "%u,%u", &k, &d) == 2 && k >= 1 && k <= 4096 && d >= 1 && d <= 1024) { a.sched_kmax = k; a.sched_div = d; }
    }
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
        // scenes of up to 4096 spheres are staged in shared memory; R1_FORCE_UNSTAGED=1 exercises the global-memory path on small scenes
        const bool staged = c.dev.n_pad <= r1::kMaxStagedSpheres && !getenv("R1_FORCE_UNSTAGED");
        R1_CUDA(cudaEventRecord(x.ev[1], stream));
        const int variant = resolve_variant(c.dev, prm);
        if (variant == R1_VARIANT_WAVEFRONT) {
            if (c.dev.n_pad > r1::kMaxStagedSpheres) return fail(R1_ERR_LIMIT, "the wavefront variant stages at most %d spheres", r1::kMaxStagedSpheres);
            uint32_t launches = 0;
            rc = r1::wavefront_render(x.wf, a, x.sm_count, stream, &launches);
            if (rc) return fail(R1_ERR_CUDA, "wavefront: %s", cudaGetErrorString((cudaError_t)rc));
            x.last_launches += launches;
        } else {
            if (variant == R1_VARIANT_MEGAKERNEL_PACKED) rc = staged ? launch_megakernel<r1::kScanLanePacked, true>(x.sm_count, a, prm, stream)
                                                                  : launch_megakernel<r1::kScanLanePacked, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_COOP) rc = staged ? launch_megakernel<r1::kScanCoop, true>(x.sm_count, a, prm, stream)
                                                                            : launch_megakernel<r1::kScanCoop, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_DEFERRED) rc = staged ? launch_megakernel<r1::kScanLaneDeferred, true>(x.sm_count, a, prm, stream)
                                                                                : launch_megakernel<r1::kScanLaneDeferred, false>(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR) rc = launch_megakernel_tc(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_TENSOR_STREAM) rc = launch_megakernel_tcs(x.sm_count, a, prm, stream);
            else if (variant == R1_VARIANT_MEGAKERNEL_DUAL) rc = staged ? launch_megakernel_dual<true>(x.sm_count, a, prm, stream)
                                                                            : launch_megakernel_dual<false>(x.sm_count, a, prm, stream);
            else rc = staged ? launch_megakernel<r1::kScanLaneScalar, true>(x.sm_count, a, prm, stream)
                             : launch_megakernel<r1::kScanLaneScalar, false>(x.sm_count, a, prm, stream);
            if (rc) return rc;
            x.last_launches += 1;
        }
        R1_CUDA(cudaEventRecord(x.ev[2], stream));
        const int rgrid = (int)std::min<uint64_t>(((uint64_t)a.npix_local + 255) / 256, (uint64_t)x.sm_count * 8);
        r1::resolve<<<rgrid, 256, 0, stream>>>(a);
        R1_CUDA(cudaGetLastError());
        x.last_launches += 1;
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
}  // namespace

extern "C" {

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
    if (variant < 0 || variant > R1_VARIANT_MEGAKERNEL_TENSOR_STREAM || variant == 8) return fail(R1_ERR_ARG, "unknown variant %d", variant);
    const int v = resolve_variant(cp->dev, prm);
    if (v == R1_VARIANT_WAVEFRONT || v == R1_VARIANT_MEGAKERNEL_DUAL) return fail(R1_ERR_ARG, "r1_trace_rays has no kernel for variant %d (wavefront, dual)", v);
    if (v == R1_VARIANT_MEGAKERNEL_TENSOR && !cp->dev.tcb)
        return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (this scene pads to %d)", r1::tc::kMaxSpheres, cp->dev.n32);
    if (n == 0) return R1_OK;
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
    switch (resolve_variant(cp->dev, prm)) {
    case R1_VARIANT_WAVEFRONT: return "wf_intersect + wf_shade (graph loop)";
    case R1_VARIANT_MEGAKERNEL_TENSOR: return getenv("R1_TC1") ? "megakernel_tc" : (getenv("R1_TC2") ? "megakernel_tc2" : "megakernel_tc3");
    case R1_VARIANT_MEGAKERNEL_DUAL: return "megakernel_pool2";
    case R1_VARIANT_MEGAKERNEL_TENSOR_STREAM: return "megakernel_tcs";
    default: return (getenv("R1_POOL") && atoi(getenv("R1_POOL")) == 0) ? "megakernel" : "megakernel_pool";
    }
}

int r1_filter_probe(r1_scene *scene, int n, const float *org, const float *dir, int layout, float *e)
{
    DeviceCtx *cp = nullptr;
    R1_TRY(get_ctx(scene, &cp));
    if (n < 0 || (n > 0 && (!org || !dir || !e))) return fail(R1_ERR_ARG, "bad argument");
    if (n == 0) return R1_OK;
    if (!cp->dev.tcb) return fail(R1_ERR_LIMIT, "the tensor-core filter takes scenes of 1 .. %d spheres (its operand lives in shared memory)", r1::tc::kMaxSpheres);
    const int n32 = cp->dev.n32;
    DevBuf d_org, d_dir, d_e;
    R1_TRY(d_org.upload(org, (size_t)n * 12)); R1_TRY(d_dir.upload(dir, (size_t)n * 12));
    R1_TRY(d_e.alloc((size_t)n * n32 * 4));
    const size_t smem = ((sizeof(r1::TcControl) + 127) & ~(size_t)127) + (size_t)n32 * r1::tc::kRowBytes + 128 * r1::tc::kRowBytes;
    R1_CUDA(cudaFuncSetAttribute(r1::tc_filter_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // layout 1 swaps the two stride fields of the shared-memory descriptors (bring-up aid; 0 is the layout the renderer uses)
    const uint32_t lbo = layout == 1 ? r1::tc::kSBO : r1::tc::kLBO, sbo = layout == 1 ? r1::tc::kLBO : r1::tc::kSBO;
    r1::tc_filter_probe_kernel<<<(n + 127) / 128, 160, smem>>>(cp->dev, n, d_org.as<float>(), d_dir.as<float>(), d_e.as<float>(), lbo, sbo);
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
