// r1_wavefront.cuh -- wavefront variant of the trace loop: the same per-path state machine as the megakernel
// (unit_begin / primary_ray / shade_step), but with the path state in HBM and the stages split into kernels:
//
//   wf_init       every slot takes a unit and generates its first primary ray
//   loop (a CUDA-graph WHILE node: the host never waits inside the loop)
//     wf_intersect  the compacted list of live slots: Hitable::hit with R rays per lane sharing each sphere load; classifies each slot
//                   (miss / lambertian / metal / dielectric) and appends it to that class's queue, compacted with
//                   warp ballot + one atomic per warp per class
//     wf_shade      walks the queues class by class, so a warp shades 32 rays of ONE material (or 32 misses, which also
//                   start the next sample / take the next unit): full lanes where the megakernel runs 5-12 of 32
//     wf_decide     one thread: loop again while any slot is alive; resets the queue counters
//
// Finished samples go to the same fixed-point pixel accumulators as the megakernel's, so both variants produce
// bit-identical images.  State: one 64-byte record per slot, ~2.4 M slots.
#pragma once
#include <cstring>
#include "r1_kernels.cuh"

namespace r1 {

constexpr int kWfRays = 2;          // rays per lane in wf_intersect (measured: 4 x 512 threads 3815, 2 x 768 3988, 2 x 1024 4070,
constexpr int kWfThreads = 1024;    //  1 x 1024 3914 Mrays/s on the large scene -- the candidate loop, not the sphere loads, bounds it)
constexpr uint32_t kDead = 0xffffffffu;

// One 64-byte record per slot (two 32-byte sectors): intersect touches the first sector only, shade reads and writes both.
//   [0] origin.xyz, hit t      [1] dir.xyz, hit sphere index (int bits)
//   [2] throughput.rgb, depth (int bits)      [3] unit (kDead = slot retired), sample index, rng key words k0, k1  (uint bits)
// (The first layout kept six separate SoA arrays: wf_shade, which visits slots in class-queue order, then moved six
// scattered sectors per ray in each direction and took 90 ms per frame.)
struct WfState {
    float4 *slots;      // 4 float4 per slot
    uint32_t *queue;    // 4 classes x n_slots slot indices
    uint32_t *alive[2]; // compacted lists of live slots: intersect reads alive[parity], shade fills alive[parity ^ 1]
    uint32_t *counters; // [0..3] class queue lengths, [4] live slots after shade, [5] loop iterations so far,
                        // [6] parity, [7] length of alive[parity], [8] next tile of wf_intersect
    uint32_t n_slots;
};

// what an instantiated loop graph was captured with: it can be launched again as long as none of this changed
struct WfGraphKey {
    RenderArgs a;
    WfState w;
    int igrid, sgrid;
    size_t smem;
};
struct WavefrontBuffers {
    void *pool = nullptr;
    size_t pool_bytes = 0;
    cudaGraphExec_t exec = nullptr;    // instantiated WHILE-loop graph, cached across renders
    WfGraphKey key;                    // valid while exec != nullptr
    uint32_t graph_builds = 0;         // how many times the graph had to be (re)built (diagnostics / tests)
    uint32_t *d_iterations = nullptr;  // device counter of loop iterations of the last render
};

inline void wavefront_free(WavefrontBuffers &b)
{
    if (b.exec) cudaGraphExecDestroy(b.exec);
    if (b.pool) cudaFree(b.pool);
    b = WavefrontBuffers();
}

__device__ __forceinline__ void wf_store_path(const WfState &w, uint32_t slot, f3 o, f3 d, f3 thr, int depth, uint32_t unit, int s, const Rng &rng)
{
    float4 *rec = w.slots + (size_t)slot * 4;
    rec[0] = make_float4(o.x, o.y, o.z, 0.0f);
    rec[1] = make_float4(d.x, d.y, d.z, __int_as_float(-1));
    rec[2] = make_float4(thr.x, thr.y, thr.z, __int_as_float(depth));
    rec[3] = make_float4(__uint_as_float(unit), __uint_as_float((uint32_t)s), __uint_as_float(rng.k0), __uint_as_float(rng.k1));
}
__device__ __forceinline__ void wf_retire(const WfState &w, uint32_t slot)
{
    w.slots[(size_t)slot * 4 + 3] = make_float4(__uint_as_float(kDead), 0.0f, 0.0f, 0.0f);
}

// slot i starts unit i (the unit counter is preset to min(n_slots, n_units))
__global__ void __launch_bounds__(256) wf_init(const __grid_constant__ RenderArgs a, const __grid_constant__ WfState w)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const uint32_t first = a.n_units < w.n_slots ? a.n_units : w.n_slots;
        *a.unit_counter = first;
        w.counters[7] = first;                              // slots 0 .. first-1 are alive, in order
    }
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < w.n_slots; slot += gridDim.x * blockDim.x) {
        if (slot < a.n_units) {
            uint32_t lp, pixel; float fx, fy; int s, s_end;
            unit_begin(a, slot, lp, pixel, fx, fy, s, s_end);
            Rng rng; f3 o, d;
            primary_ray(a, pixel, fx, fy, s, g_rsqrt12, rng, o, d);
            wf_store_path(w, slot, o, d, mk3(1, 1, 1), 0, slot, s, rng);
            w.alive[0][slot] = slot;
        } else {
            wf_retire(w, slot);
        }
    }
}

// Hitable::hit for every live slot; R rays per lane; classification + queue compaction.
template <int R, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) wf_intersect(const __grid_constant__ RenderArgs a, const __grid_constant__ WfState w)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4 *s_spheres = reinterpret_cast<float4 *>(smem_raw + 16);
    stage_spheres(a.scene, s_spheres, reinterpret_cast<uint64_t *>(smem_raw));
    const float4 *s_scan = s_spheres, *s_exact = s_spheres + a.scene.n_pad;
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n_alive = w.counters[7];
    const uint32_t *alive = w.alive[w.counters[6] & 1u];
    const uint32_t n_tiles = (n_alive + 32 * R - 1) / (32 * R);
    uint32_t nrays = 0;
    for (;;) {
        // tiles are handed out dynamically (one atomic per warp per 32 * R rays): the exact-candidate work per tile varies, and a
        // static split left the SMs idle for 30 % of the kernel
        uint32_t tile = 0;
        if (lane == 0) tile = atomicAdd(&w.counters[8], 1u);
        tile = __shfl_sync(kFull, tile, 0);
        if (tile >= n_tiles) break;
        f3 o[R], d[R];
        float t[R];
        int hit[R];
        uint32_t slots[R];
        bool live[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t i = tile * (32 * R) + r * 32 + lane;
            live[r] = i < n_alive;
            slots[r] = live[r] ? alive[i] : 0u;
            o[r] = mk3(0.0f, 1.0e18f, 0.0f); d[r] = mk3(0.0f, 0.0f, 0.0f);   // lanes past the end scan a ray that passes no filter
            if (live[r]) {
                const float4 ro = w.slots[(size_t)slots[r] * 4], rd = w.slots[(size_t)slots[r] * 4 + 1];
                o[r] = mk3(ro.x, ro.y, ro.z); d[r] = mk3(rd.x, rd.y, rd.z);
            }
            t[r] = kTMax; hit[r] = -1;
        }
        scan_multi<R, (R >= 4 ? 4 : 8)>(s_scan, s_exact, a.scene.n8, o, d, kTMin, t, hit);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t slot = slots[r];
            int cls = -1;
            if (live[r]) {
                ++nrays;
                w.slots[(size_t)slot * 4].w = t[r];                       // same 32-byte sector as the ray
                w.slots[(size_t)slot * 4 + 1].w = __int_as_float(hit[r]);
                cls = hit[r] < 0 ? 0 : 1 + __float_as_int(__ldg(a.scene.shade + 2 * hit[r] + 1).y);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {          // ballot + popc compaction: one atomic per warp per class
                const unsigned m = __ballot_sync(kFull, cls == c);
                if (m) {
                    const int leader = __ffs(m) - 1;
                    unsigned base = 0;
                    if ((int)lane == leader) base = atomicAdd(&w.counters[c], (unsigned)__popc(m));
                    base = __shfl_sync(kFull, base, leader);
                    if (cls == c) w.queue[(size_t)c * w.n_slots + base + __popc(m & ((1u << lane) - 1u))] = slot;
                }
            }
        }
    }
    count_rays(a, nrays, lane);
}

// color() + (on path end) accumulate, next sample / next unit, next primary ray -- class by class.
__global__ void __launch_bounds__(256) wf_shade(const __grid_constant__ RenderArgs a, const __grid_constant__ WfState w)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n0 = w.counters[0], n1 = w.counters[1], n2 = w.counters[2], n3 = w.counters[3];
    // each class is padded to a multiple of 32 entries so that a warp never mixes classes
    const uint32_t p0 = (n0 + 31) & ~31u, p1 = (n1 + 31) & ~31u, p2 = (n2 + 31) & ~31u, p3 = (n3 + 31) & ~31u;
    const uint32_t total = p0 + p1 + p2 + p3;
    uint32_t *next_alive = w.alive[(w.counters[6] & 1u) ^ 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        uint32_t c, j;
        if (i < p0) { c = 0; j = i; }
        else if (i < p0 + p1) { c = 1; j = i - p0; }
        else if (i < p0 + p1 + p2) { c = 2; j = i - p0 - p1; }
        else { c = 3; j = i - p0 - p1 - p2; }
        const uint32_t n_c = c == 0 ? n0 : c == 1 ? n1 : c == 2 ? n2 : n3;
        const bool valid = j < n_c;
        bool ended = false, alive = false;
        uint32_t slot = 0, unit = 0;
        int s = 0, depth = 0;
        f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0), thr = mk3(1, 1, 1), contrib = mk3(0, 0, 0);
        Rng rng; rng.k0 = 0; rng.k1 = 0;
        if (valid) {
            slot = w.queue[(size_t)c * w.n_slots + j];
            const float4 *rec = w.slots + (size_t)slot * 4;
            const float4 ro = rec[0], rd = rec[1], th = rec[2], m = rec[3];
            o = mk3(ro.x, ro.y, ro.z); d = mk3(rd.x, rd.y, rd.z); thr = mk3(th.x, th.y, th.z); depth = __float_as_int(th.w);
            unit = __float_as_uint(m.x); s = (int)__float_as_uint(m.y); rng.k0 = __float_as_uint(m.z); rng.k1 = __float_as_uint(m.w);
            const int hit = __float_as_int(rd.w);
            const float4 e = hit >= 0 ? __ldg(a.scene.exact + hit) : make_float4(0, 0, 0, 0);
            ended = shade_step(a, hit, ro.w, e, g_rsqrt12, o, d, thr, depth, rng, contrib);
            alive = true;
        }
        // path ended: add the sample to its pixel, then the next sample of the unit or the next unit (warp-aggregated atomic)
        uint32_t lp, pixel; float fx, fy; int s0, s_end;
        bool want_unit = false;
        if (ended) {
            unit_begin(a, unit, lp, pixel, fx, fy, s0, s_end);
            accumulate_sample(a, lp, contrib);
            want_unit = ++s == s_end;
        }
        const unsigned need = __ballot_sync(kFull, want_unit);
        if (need) {
            const int leader = __ffs(need) - 1;
            unsigned base = 0;
            if ((int)lane == leader) base = atomicAdd(a.unit_counter, (unsigned)__popc(need));
            base = __shfl_sync(kFull, base, leader);
            if (want_unit) {
                unit = base + __popc(need & ((1u << lane) - 1u));
                if (unit < a.n_units) unit_begin(a, unit, lp, pixel, fx, fy, s, s_end);
                else { alive = false; unit = kDead; }
            }
        }
        if (valid) {
            if (ended && alive) {
                primary_ray(a, pixel, fx, fy, s, g_rsqrt12, rng, o, d);
                thr = mk3(1, 1, 1);
                depth = 0;
            }
            if (alive) wf_store_path(w, slot, o, d, thr, depth, unit, s, rng);
            else wf_retire(w, slot);
        }
        // live slots go to the next iteration's compacted list (ballot + popc, one atomic per warp)
        const unsigned am = __ballot_sync(kFull, valid && alive);
        if (am) {
            const int leader = __ffs(am) - 1;
            unsigned base = 0;
            if ((int)lane == leader) base = atomicAdd(&w.counters[4], (unsigned)__popc(am));
            base = __shfl_sync(kFull, base, leader);
            if (valid && alive) next_alive[base + __popc(am & ((1u << lane) - 1u))] = slot;
        }
    }
}

// loop control: one thread.  Sets the WHILE node's condition through `handle`; host_flag, when not null, receives the live-slot
// count (the graph passes null).
__global__ void wf_decide(const __grid_constant__ WfState w, cudaGraphConditionalHandle handle, uint32_t *host_flag)
{
    const uint32_t alive = w.counters[4];
    for (int k = 0; k < 5; ++k) w.counters[k] = 0;
    w.counters[8] = 0;                                      // wf_intersect's tile counter
    w.counters[5] += 1;
    w.counters[6] ^= 1u;
    w.counters[7] = alive;
    if (handle) cudaGraphSetConditional(handle, alive ? 1u : 0u);
    if (host_flag) *host_flag = alive;
}

#define R1_WF_CUDA(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return (int)e_; } while (0)

inline uint32_t wavefront_slots(uint32_t n_units, int sm_count)
{
    // a multiple of one full wave of wf_intersect (SMs x warps x 32 lanes x R rays) so that every warp gets the same number of tiles
    const uint64_t wave = (uint64_t)sm_count * kWfThreads * kWfRays;
    uint64_t slots = wave * 8;
    const uint64_t need = ((uint64_t)n_units + 32 * kWfRays - 1) / (32 * kWfRays) * (32 * kWfRays);
    if (slots > need) slots = need;
    return (uint32_t)slots;
}

// returns a cudaError_t (0 = ok).  Asynchronous on `stream`; the unit counter must already be zeroed.
inline int wavefront_render(WavefrontBuffers &b, const RenderArgs &a, int sm_count, cudaStream_t stream, uint32_t *launches)
{
    *launches = 0;
    WfState w;
    memset(&w, 0, sizeof(w));   // padding too: the graph cache compares the struct bytewise
    w.n_slots = wavefront_slots(a.n_units, sm_count);
    const size_t n = w.n_slots;
    const size_t bytes = n * (64 + 16 + 8) + 64 + 256;
    if (bytes > b.pool_bytes) {
        if (b.pool) cudaFree(b.pool);
        b.pool = nullptr; b.pool_bytes = 0;
        R1_WF_CUDA(cudaMalloc(&b.pool, bytes));
        b.pool_bytes = bytes;
    }
    unsigned char *p = static_cast<unsigned char *>(b.pool);
    w.slots = reinterpret_cast<float4 *>(p); p += n * 64;
    w.queue = reinterpret_cast<uint32_t *>(p); p += n * 16;
    w.alive[0] = reinterpret_cast<uint32_t *>(p); p += n * 4;
    w.alive[1] = reinterpret_cast<uint32_t *>(p); p += n * 4;
    w.counters = reinterpret_cast<uint32_t *>(p);

    b.d_iterations = w.counters + 5;
    R1_WF_CUDA(cudaMemsetAsync(w.counters, 0, 64, stream));
    const int init_grid = (int)std::min<size_t>((n + 255) / 256, (size_t)sm_count * 8);
    wf_init<<<init_grid, 256, 0, stream>>>(a, w);
    R1_WF_CUDA(cudaGetLastError());
    *launches += 1;

    const size_t smem = 16 + (size_t)a.scene.n_pad * 32;
    const auto ikern = wf_intersect<kWfRays, kWfThreads>;
    R1_WF_CUDA(cudaFuncSetAttribute(ikern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t n_tiles = (w.n_slots + 32 * kWfRays - 1) / (32 * kWfRays);
    const int igrid = (int)std::min<uint32_t>((uint32_t)sm_count, (n_tiles * 32 + kWfThreads - 1) / kWfThreads);
    const int sgrid = sm_count * 8;

    // the loop as a CUDA-graph WHILE node: intersect -> shade -> decide, repeated on the device until no slot is alive.
    // Kernel arguments are baked into the instantiated graph, so it is cached and re-launched while they stay the same
    // (every render of a benchmark loop); any change -- another scene block, image size, buffers, grid -- rebuilds it.
    WfGraphKey key;
    memset(&key, 0, sizeof(key));
    key.a = a; key.w = w; key.igrid = igrid; key.sgrid = sgrid; key.smem = smem;
    if (b.exec && memcmp(&key, &b.key, sizeof(key)) != 0) {
        R1_WF_CUDA(cudaStreamSynchronize(stream));   // the previous render's graph may still be running on this stream
        cudaGraphExecDestroy(b.exec);
        b.exec = nullptr;
    }
    if (!b.exec) {
        cudaGraph_t graph = nullptr;
        R1_WF_CUDA(cudaGraphCreate(&graph, 0));
        cudaGraphConditionalHandle handle;
        R1_WF_CUDA(cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault));
        cudaGraphNodeParams cond = { cudaGraphNodeTypeConditional };
        cond.conditional.handle = handle;
        cond.conditional.type = cudaGraphCondTypeWhile;
        cond.conditional.size = 1;
        cudaGraphNode_t node;
        R1_WF_CUDA(cudaGraphAddNode(&node, graph, nullptr, 0, &cond));
        cudaGraph_t body = cond.conditional.phGraph_out[0];
        cudaStream_t cap;
        R1_WF_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
        R1_WF_CUDA(cudaStreamBeginCaptureToGraph(cap, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
        ikern<<<igrid, kWfThreads, smem, cap>>>(a, w);
        wf_shade<<<sgrid, 256, 0, cap>>>(a, w);
        wf_decide<<<1, 1, 0, cap>>>(w, handle, nullptr);
        R1_WF_CUDA(cudaStreamEndCapture(cap, nullptr));
        R1_WF_CUDA(cudaStreamDestroy(cap));
        R1_WF_CUDA(cudaGraphInstantiate(&b.exec, graph, 0));
        R1_WF_CUDA(cudaGraphDestroy(graph));
        b.key = key;
        ++b.graph_builds;
    }
    R1_WF_CUDA(cudaGraphLaunch(b.exec, stream));
    // 3 kernels per loop iteration; the iteration count lives on the device (d_iterations) and is read by r1_render_wait
    *launches += 0;
    return 0;
}

}  // namespace r1
