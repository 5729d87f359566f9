// r1_bvh_device.h -- the device BVH builder of r1_bvh_device.cu, as r1_core.cu calls it.  A translation unit of its own: the
// radix sort's headers would otherwise move the global symbols every render kernel addresses, and so change their code.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace r1 {

// CUDA events around phases of set-up work on the current device's legacy stream; ms sums the phases, not the host time between.
struct PhaseTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    double ms = 0;
    ~PhaseTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    cudaError_t start()
    {
        cudaError_t e = cudaSuccess;
        if (!a && (e = cudaEventCreate(&a)) != cudaSuccess) return e;
        if (!b && (e = cudaEventCreate(&b)) != cudaSuccess) return e;
        return cudaEventRecord(a, nullptr);
    }
    cudaError_t stop()
    {
        float t = 0;
        cudaError_t e = cudaEventRecord(b, nullptr);
        if (e == cudaSuccess) e = cudaEventSynchronize(b);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&t, a, b);
        ms += t;
        return e;
    }
};

namespace lbvh {

struct Built {
    void *block;                        // cudaMalloc'ed [n_nodes x 64 B nodes | n_leaves x 32 B leaf records]; the caller frees it
    uint32_t n_nodes, n_leaves, depth;
};

// The linear BVH of spheres 0 .. n - 1 of a committed scene on the current device, from its exact records and shading records
// (inv_radius = shade[2 i + 1].x).  Returns R1_OK, or an R1_ERR_* code with r1_set_error's message: R1_ERR_ARG for a sphere that
// can be hit with a non-finite centre or radius_sq, R1_ERR_LIMIT from 2^28 such spheres, R1_ERR_CUDA.  ms: device time of the
// kernels and the sort.
int build(const float4 *exact, const float4 *shade, uint32_t n, Built *out, double *ms);

// Refits a tree in r1_bvh.h's layout in place to the scene's exact records (DESIGN.md section 4.10): same topology, child references
// and record order; every used slot gets the union of the padded boxes of its spheres and their diagonal bound, every leaf record the
// sphere's exact record.  parent / arrivals: n_nodes words of scratch each; parent is derived from the child references unless
// parents_ready says it already holds that (it depends on the topology alone).  Asynchronous on `stream`.
int refit(float4 *nodes, float4 *leaves, uint32_t n_nodes, const float4 *exact, int *parent, unsigned int *arrivals, bool parents_ready,
          cudaStream_t stream);

}  // namespace lbvh
}  // namespace r1
