// r1_move.cu -- moving committed spheres (r1_scene_move_spheres, DESIGN.md section 4.10) and changing their materials
// (r1_scene_set_materials, section 4.11) on the device: a check of the new values, then the records r1_scene_commit would write for
// them, from the same functions (r1_encode.h).
#include "r1_move.h"

#include "../../include/rays1_b200.h"
#include "r1_encode.h"
#include "r1_internal.h"

namespace r1 {
namespace move {

constexpr int kThreads = 256;

__device__ __forceinline__ bool finite4(float a, float b, float c, float d) { return isfinite(a) && isfinite(b) && isfinite(c) && isfinite(d); }

// bit 0: a new radius changes whether its sphere can be hit; bit 1: a sphere that can be hit gets a non-finite centre or radius_sq
__global__ void __launch_bounds__(kThreads) move_check(const float4 *__restrict__ exact, const float4 *__restrict__ shade, uint32_t first, uint32_t n,
                                                       const float *__restrict__ centre, const float *__restrict__ radius, unsigned int *flag)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const size_t i = (size_t)first + j;
    const float inv_old = shade[2 * i + 1].x;
    float r2 = exact[i].w, inv = inv_old;
    if (radius) enc::radius_terms(radius[j], r2, inv);
    const bool real = inv_old != 0.0f;
    if ((inv != 0.0f) != real) atomicOr(flag, 1u);
    if (real && !finite4(centre[3 * (size_t)j], centre[3 * (size_t)j + 1], centre[3 * (size_t)j + 2], r2)) atomicOr(flag, 2u);
}

// one thread per sphere: its scan lanes, exact record, inv_radius and operand row (8 x 16 bytes)
__global__ void __launch_bounds__(kThreads) move_encode(Records r, uint32_t first, uint32_t n, const float *__restrict__ centre,
                                                        const float *__restrict__ radius)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = first + j;
    const float cx = centre[3 * (size_t)j], cy = centre[3 * (size_t)j + 1], cz = centre[3 * (size_t)j + 2];
    float r2 = r.exact[i].w, inv = r.shade[2 * (size_t)i + 1].x;
    if (radius) enc::radius_terms(radius[j], r2, inv);
    const bool real = inv != 0.0f;                                 // unchanged by the move (move_check)
    enc::scan_lanes(reinterpret_cast<float *>(r.scan), (int)i, real, real ? cx : 0.0f, real ? cy : 0.0f, real ? cz : 0.0f, real ? r2 : 0.0f);
    r.exact[i] = make_float4(cx, cy, cz, r2);
    reinterpret_cast<float *>(r.shade)[4 * (2 * (size_t)i + 1)] = inv;
    uint32_t w[tc::kK];
    tc::sphere_row_words(real, real ? cx : 0.0, real ? cy : 0.0, real ? cz : 0.0, real ? r2 : 0.0, w);
    unsigned char *row = r.operand + tc::row_offset((int)i, 0);
#pragma unroll
    for (int kc = 0; kc < tc::kK / 4; ++kc)
        *reinterpret_cast<uint4 *>(row + kc * tc::kLBO) = make_uint4(w[4 * kc], w[4 * kc + 1], w[4 * kc + 2], w[4 * kc + 3]);
}

#define R1_MOVE_CUDA(expr)                                                                                   \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess) return r1_set_error(R1_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int check(const Records &r, uint32_t first, uint32_t n, const float *centre, const float *radius, unsigned int *d_flag, cudaStream_t stream)
{
    R1_MOVE_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(unsigned int), stream));
    move_check<<<(n + kThreads - 1) / kThreads, kThreads, 0, stream>>>(r.exact, r.shade, first, n, centre, radius, d_flag);
    R1_MOVE_CUDA(cudaGetLastError());
    unsigned int flag = 0;
    R1_MOVE_CUDA(cudaMemcpyAsync(&flag, d_flag, sizeof(flag), cudaMemcpyDeviceToHost, stream));
    R1_MOVE_CUDA(cudaStreamSynchronize(stream));
    if (flag & 1u) return r1_set_error(R1_ERR_ARG, "a new radius changes whether its sphere can be hit (radius > 0 and finite against inv_radius != 0): commit the scene again");
    if (flag & 2u) return r1_set_error(R1_ERR_ARG, "a sphere that can be hit would get a non-finite centre or radius_sq");
    return R1_OK;
}

int encode(const Records &r, uint32_t first, uint32_t n, const float *centre, const float *radius, cudaStream_t stream)
{
    move_encode<<<(n + kThreads - 1) / kThreads, kThreads, 0, stream>>>(r, first, n, centre, radius);
    R1_MOVE_CUDA(cudaGetLastError());
    return R1_OK;
}

// ---- materials (r1_scene_set_materials, DESIGN.md section 4.11) ----------------------------------------------------------------

// bit 0: a kind outside R1_MAT_NONE .. R1_MAT_DIELECTRIC; bit 1: R1_MAT_NONE for a sphere that can be hit (inv_radius != 0)
__global__ void __launch_bounds__(kThreads) material_check(const float4 *__restrict__ shade, uint32_t first, uint32_t n,
                                                           const int32_t *__restrict__ kind, unsigned int *flag)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int32_t k = kind[j];
    if (k < R1_MAT_NONE || k > R1_MAT_DIELECTRIC) atomicOr(flag, 1u);
    if (k == R1_MAT_NONE && shade[2 * ((size_t)first + j) + 1].x != 0.0f) atomicOr(flag, 2u);
}

// one thread per sphere: both shade records from the new fields and the kept ones (inv_radius is always kept)
__global__ void __launch_bounds__(kThreads) material_encode(float4 *__restrict__ shade, uint32_t first, uint32_t n, const int32_t *__restrict__ kind,
                                                            const float *__restrict__ albedo, const float *__restrict__ param)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const size_t i = (size_t)first + j;
    const float4 mat = shade[2 * i], geo = shade[2 * i + 1];
    const int32_t k = kind ? kind[j] : (int32_t)enc::bits(geo.y);
    const float r = albedo ? albedo[3 * (size_t)j] : mat.x, g = albedo ? albedo[3 * (size_t)j + 1] : mat.y, b = albedo ? albedo[3 * (size_t)j + 2] : mat.z;
    float4 m, e;
    enc::shade_records(k, r, g, b, param ? param[j] : mat.w, geo.x, m, e);
    shade[2 * i] = m;
    shade[2 * i + 1] = e;
}

int check_materials(const Records &r, uint32_t first, uint32_t n, const int32_t *kind, unsigned int *d_flag, cudaStream_t stream)
{
    R1_MOVE_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(unsigned int), stream));
    material_check<<<(n + kThreads - 1) / kThreads, kThreads, 0, stream>>>(r.shade, first, n, kind, d_flag);
    R1_MOVE_CUDA(cudaGetLastError());
    unsigned int flag = 0;
    R1_MOVE_CUDA(cudaMemcpyAsync(&flag, d_flag, sizeof(flag), cudaMemcpyDeviceToHost, stream));
    R1_MOVE_CUDA(cudaStreamSynchronize(stream));
    if (flag & 1u) return r1_set_error(R1_ERR_ARG, "unknown material kind (R1_MAT_NONE .. R1_MAT_DIELECTRIC = -1 .. 2)");
    if (flag & 2u) return r1_set_error(R1_ERR_ARG, "a sphere that can be hit (inv_radius != 0) needs a material: R1_MAT_NONE refused");
    return R1_OK;
}

int encode_materials(const Records &r, uint32_t first, uint32_t n, const int32_t *kind, const float *albedo, const float *param, cudaStream_t stream)
{
    material_encode<<<(n + kThreads - 1) / kThreads, kThreads, 0, stream>>>(r.shade, first, n, kind, albedo, param);
    R1_MOVE_CUDA(cudaGetLastError());
    return R1_OK;
}

}  // namespace move
}  // namespace r1
