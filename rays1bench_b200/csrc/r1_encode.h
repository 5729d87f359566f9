// r1_encode.h -- the device records of one sphere, in one definition for the host and the device: r1_scene_commit encodes a scene
// with these functions on the host, and r1_scene_move_spheres / r1_scene_set_materials (r1_move.cu) re-encode spheres with them on
// the device.  The two must write the same bytes (DESIGN.md sections 4.10, 4.11), so every double operation goes through dmul /
// dadd / dsub / ddiv, which are the _rn intrinsics on the device (nvcc would otherwise contract a product and a sum into an FMA) and
// the plain operators on the host.  Conversions between float and double are exact (float -> double) or round to nearest (double ->
// float) on both.
//
// Records of sphere i in the committed block [scan | exact | shade | tensor operand]:
//   scan    supergroup lanes -cx, -cy, -cz, kk (r1_device.cuh "Filter arithmetic"): scan_lanes
//   exact   {cx, cy, cz, radius_sq}
//   shade   [2i] material, [2i + 1] {inv_radius, kind, 1 / ior, r0}: shade_records; only inv_radius depends on the geometry
//   operand the sphere's row of the tensor-core filter's B operand (r1_tensor.cuh): sphere_row_words
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rays1_b200.h"

#include <cmath>
#include <cstring>

#define R1_HD __host__ __device__ __forceinline__

namespace r1 {
namespace enc {

R1_HD double dmul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
R1_HD double dadd(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
R1_HD double dsub(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
R1_HD double ddiv(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
R1_HD uint32_t bits(float x)
{
    uint32_t b;
    memcpy(&b, &x, 4);
    return b;
}
R1_HD float from_bits(uint32_t b)
{
    float x;
    memcpy(&x, &b, 4);
    return x;
}
R1_HD float neg(float x) { return from_bits(bits(x) ^ 0x80000000u); }   // the sign flip of the host's unary minus, NaN included

// r1_scene_add_sphere's derived values (SphereSOA::add, soa_sphere.cpp:70-85): radius * radius and radius > 0 ? 1 / radius : 0, IEEE
R1_HD void radius_terms(float radius, float &radius_sq, float &inv_radius)
{
#ifdef __CUDA_ARCH__
    radius_sq = __fmul_rn(radius, radius);
    inv_radius = radius > 0 ? __fdiv_rn(1.0f, radius) : 0.0f;
#else
    radius_sq = radius * radius;
    inv_radius = radius > 0 ? (1.0f / radius) : 0;
#endif
}

// The range of the expanded filters (r1_device.cuh "Filter arithmetic", r1_tensor.cuh; DESIGN.md section 4.1).  Their error bounds
// are relative and hold while no term overflows, which |c|^2 < 2^120 and |o|^2 < 2^120 guarantee with a wide margin.  A sphere that
// can be hit with |c|^2 >= 2^120 (double; so from |c| = 2^60 on, and for infinite centres) is a FAR sphere: its filter records make
// it a candidate of every ray.  A ray with |o|^2 >= 2^120 (float, or NaN) gets filter constants that flag every sphere that can be
// hit.  The exact test decides both, and placeholders stay out.  From |c| = 2^60 on the margins exceed r^2 of any sphere the
// ray's line passes within |c| of, so far spheres were candidates of nearly every ray already; the encoding only keeps that true
// where |c|^2 overflows float (|c| > 2^64).
constexpr double kFarC2 = 0x1p120;
constexpr float kFarKK = -0x1p122f;                     // the kk of a far sphere, whose every other lane or feature is 0

// The four scan lanes of sphere i in the supergroup layout (r1_device.cuh): group g = i / 4 at float4 index (g >> 2) * 16 + (g & 3);
// cy / cz / kk at +4 / +8 / +12.  kk = |c|^2 - r^2 - 2^-17 |c|^2, evaluated in double, rounded down, then one more ulp down.  A sphere
// that can never be hit (`real` false) gets 0, 0, 0, +inf: no ray flags it.  A far sphere gets 0, 0, 0, kFarKK: every ray flags it.
R1_HD void scan_lanes(float *scan, int i, bool real, float cx, float cy, float cz, float radius_sq)
{
    const int g = i / 4, k = i % 4, f4 = (g >> 2) * 16 + (g & 3);
    const float inf = from_bits(0x7f800000u);
    const double c2 = real ? dadd(dadd(dmul((double)cx, (double)cx), dmul((double)cy, (double)cy)), dmul((double)cz, (double)cz)) : 0.0;
    const bool far = c2 >= kFarC2;                      // false for NaN: those keep the records r1_scene_commit has always written
    scan[4 * (f4 + 0) + k] = real && !far ? neg(cx) : 0.0f;
    scan[4 * (f4 + 4) + k] = real && !far ? neg(cy) : 0.0f;
    scan[4 * (f4 + 8) + k] = real && !far ? neg(cz) : 0.0f;
    if (far) {
        scan[4 * (f4 + 12) + k] = kFarKK;
    } else if (real) {
        const double kk = dsub(dsub(c2, (double)radius_sq), ddiv(c2, 131072.0));
        float kf = (float)kk;
        if ((double)kf > kk) kf = nextafterf(kf, -inf);
        scan[4 * (f4 + 12) + k] = nextafterf(kf, -inf);
    } else {
        scan[4 * (f4 + 12) + k] = inf;
    }
}

// The two shade records of a sphere with material (kind, r, g, b, param): mat = {r, g, b, param}, Metal's param clamped as its ctor
// does (rayweek1.cpp:424: param < 1 ? param : 1, so a NaN fuzz becomes 1); geo = {inv_radius, kind's bits, 1 / ior, (1 - ior) /
// (ior + 1)}, Dielectric::scatter's two divisions (rayweek1.cpp:482, :456) done once per sphere in IEEE float, 0 and 0 for other
// kinds.  r1_scene_commit's host scene holds Metal params clamped already; clamping again changes no bit.
R1_HD void shade_records(int32_t kind, float r, float g, float b, float param, float inv_radius, float4 &mat, float4 &geo)
{
    if (kind == R1_MAT_METAL) param = param < 1 ? param : 1;
    float inv_ior = 0.0f, r0 = 0.0f;
    if (kind == R1_MAT_DIELECTRIC) {
#ifdef __CUDA_ARCH__
        inv_ior = __fdiv_rn(1.0f, param);
        r0 = __fdiv_rn(__fsub_rn(1.0f, param), __fadd_rn(param, 1.0f));
#else
        const volatile float ior = param;
        inv_ior = 1.0f / ior;
        r0 = (1.0f - ior) / (ior + 1.0f);
#endif
    }
    mat = make_float4(r, g, b, param);
    geo = make_float4(inv_radius, from_bits((uint32_t)kind), inv_ior, r0);
}

}  // namespace enc

namespace tc {

constexpr int kFeatures = 11;
constexpr int kK = 32;                                  // 4 x (K = 8 tf32)
constexpr int kRowBytes = kK * 4;                       // one ray / sphere row
// canonical K-major, no-swizzle operand layout (core matrix = 8 rows x 16 bytes, stored contiguously):
//   byte offset of (row r, k) = (r / 8) * kSBO + (k / 4) * kLBO + (r % 8) * 16 + (k % 4) * 4
constexpr uint32_t kLBO = 128;                          // between the core matrices of adjacent K
constexpr uint32_t kSBO = (kK / 4) * 128;               // between 8-row groups: 1024 bytes
constexpr int kMaxSpheres = 768;                        // B tile of the whole scene resident in shared memory: 96 KB
constexpr double kMargin = 1.0 / 65536.0;               // 2^-16 of |c|^2 (sphere side) and of |o|^2 (ray side)
constexpr float kPadKK = 1.0e30f;                       // padded sphere rows: e = -1e30

__host__ __device__ __forceinline__ uint32_t row_offset(int r, int k) { return (uint32_t)(r >> 3) * kSBO + (uint32_t)(k >> 2) * kLBO + (uint32_t)(r & 7) * 16u + (uint32_t)(k & 3) * 4u; }

// ---- the sphere operand ------------------------------------------------------------------------------------------------------
R1_HD uint32_t tf32_rna_bits(float x)                   // cvt.rna.tf32.f32: round to nearest, ties away, low 13 bits zero
{
    const uint32_t b = enc::bits(x);
    if ((b & 0x7f800000u) == 0x7f800000u) return b & 0xffffe000u;
    return (b + 0x1000u) & 0xffffe000u;
}
R1_HD void split_tf32(double v, uint32_t &hi, uint32_t &lo)
{
    hi = tf32_rna_bits((float)v);
    lo = tf32_rna_bits((float)enc::dsub(v, (double)enc::from_bits(hi)));
}
// The 11 lifted features of one sphere (the B operand's row before the TF32 split); `real` = false for padding and for spheres
// that can never be hit.  A far sphere (enc::kFarC2) gets 0 x 9, kFarKK, 1: every live ray row flags it (its feature 10 lies in
// [-2^120, 2^121], r1_tensor.cuh ray_row), and the idle row (-2^126) does not.
struct Features {
    double f[kFeatures];
};
R1_HD Features sphere_features(bool real, double cx, double cy, double cz, double radius_sq)
{
    Features r = { { 0, 0, 0, 0, 0, 0, 0, 0, 0, (double)kPadKK, 0 } };
    double *f = r.f;
    const bool far = real && enc::dadd(enc::dadd(enc::dmul(cx, cx), enc::dmul(cy, cy)), enc::dmul(cz, cz)) >= enc::kFarC2;
    if (far) {
        f[9] = (double)enc::kFarKK;
        f[10] = 1.0;
    } else if (real) {
#ifdef __CUDA_ARCH__
        using namespace enc;
        const double nx = -cx, ny = -cy, nz = -cz, c2 = dadd(dadd(dmul(cx, cx), dmul(cy, cy)), dmul(cz, cz));
        f[0] = dmul(nx, nx); f[1] = dmul(ny, ny); f[2] = dmul(nz, nz); f[3] = dmul(nx, ny); f[4] = dmul(nx, nz); f[5] = dmul(ny, nz);
        f[6] = nx; f[7] = ny; f[8] = nz;
        f[9] = dsub(dsub(c2, radius_sq), dmul(c2, kMargin));
#else
        // The same operations in the same order, spelled with operators: with NaN inputs the host compiler is free to pick which
        // operand's NaN a product returns, and this spelling keeps the bytes r1_scene_commit has always written for them.  The device
        // never encodes a NaN (r1_scene_move_spheres refuses them), and for every other input the two spellings round alike.
        const double nx = -cx, ny = -cy, nz = -cz, c2 = cx * cx + cy * cy + cz * cz;
        f[0] = nx * nx; f[1] = ny * ny; f[2] = nz * nz; f[3] = nx * ny; f[4] = nx * nz; f[5] = ny * nz;
        f[6] = nx; f[7] = ny; f[8] = nz;
        f[9] = c2 - radius_sq - c2 * kMargin;
#endif
        f[10] = 1.0;
    }
    return r;
}
// The 32 words of one sphere row in K order: {hi x 11 | hi x 11 | lo x 10} of the features (the ray side pairs them hi, lo, hi)
R1_HD void sphere_row_words(bool real, double cx, double cy, double cz, double radius_sq, uint32_t (&w)[kK])
{
    const Features ft = sphere_features(real, cx, cy, cz, radius_sq);
    for (int j = 0; j < kFeatures; ++j) {
        uint32_t hi, lo;
        split_tf32(ft.f[j], hi, lo);
        w[j] = hi;
        w[kFeatures + j] = hi;
        if (j < kFeatures - 1) w[2 * kFeatures + j] = lo;
    }
}
// one sphere row of the B tile in shared-memory layout: sphere_row_words, written at row i
inline void sphere_row_host(unsigned char *tile, int i, bool real, double cx, double cy, double cz, double radius_sq)
{
    const Features ft = sphere_features(real, cx, cy, cz, radius_sq);
    for (int j = 0; j < kFeatures; ++j) {
        uint32_t hi, lo;
        split_tf32(ft.f[j], hi, lo);
        memcpy(tile + row_offset(i, j), &hi, 4);                                // x ray hi
        memcpy(tile + row_offset(i, kFeatures + j), &hi, 4);                    // x ray lo
        if (j < kFeatures - 1) memcpy(tile + row_offset(i, 2 * kFeatures + j), &lo, 4);   // x ray hi
    }
}

}  // namespace tc
}  // namespace r1
