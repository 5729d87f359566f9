// r1_move.h -- the device side of r1_scene_move_spheres and r1_scene_set_materials (r1_move.cu), as r1_core.cu calls it.  A translation unit of its own, like
// the BVH builder: the render kernels of r1_core.cu keep their code byte for byte.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace r1 {
namespace move {

// The records of a committed scene on one device (r1_scene_commit's block): scan and exact n_pad float4 each, shade 2 n_pad float4,
// then the tensor-filter operand, n32 rows of 128 bytes.
struct Records {
    float4 *scan, *exact, *shade;
    unsigned char *operand;
};

// Checks the new values of spheres first .. first + n - 1 (centre: n x 3 floats, radius: n floats or null = keep) before anything is
// written: R1_ERR_ARG if one changes whether its sphere can be hit (inv_radius != 0) or gives a sphere that can be hit a non-finite
// centre or radius_sq.  d_flag: one device word of scratch.  Waits for `stream`.
int check(const Records &r, uint32_t first, uint32_t n, const float *centre, const float *radius, unsigned int *d_flag, cudaStream_t stream);

// Rewrites those spheres' scan lanes, exact records, inv_radius and operand rows with r1_encode.h, as r1_scene_commit writes them for
// a scene with the new values.  Asynchronous on `stream`.
int encode(const Records &r, uint32_t first, uint32_t n, const float *centre, const float *radius, cudaStream_t stream);

// Checks the new kinds of spheres first .. first + n - 1 (kind: n int32) before anything is written: R1_ERR_ARG for a kind outside
// R1_MAT_NONE .. R1_MAT_DIELECTRIC, or R1_MAT_NONE for a sphere that can be hit (inv_radius != 0).  d_flag: one device word of
// scratch.  Waits for `stream`.
int check_materials(const Records &r, uint32_t first, uint32_t n, const int32_t *kind, unsigned int *d_flag, cudaStream_t stream);

// Rewrites those spheres' shade records with r1_encode.h's shade_records from the new fields (kind: n int32, albedo: n x 3 floats,
// param: n floats; null = keep that field) and the kept inv_radius.  Asynchronous on `stream`.
int encode_materials(const Records &r, uint32_t first, uint32_t n, const int32_t *kind, const float *albedo, const float *param, cudaStream_t stream);

}  // namespace move
}  // namespace r1
