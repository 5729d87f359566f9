// rays1-b200: the nearest-hit FILTER on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM).
//
// The filter of r1_device.cuh evaluates, per (ray, sphere),   e = (o.d - c.d)^2 - (|c|^2 - r^2 - margins - 2 o.c + |o|^2)
// and flags the sphere when e >= 0; the exact test (bit-identical to the reference's Hitable::hit, rayweek1.cpp:152-339)
// decides.  e is a polynomial of degree 2 in the sphere centre, so it is ONE dot product of a lifted ray vector with a lifted
// sphere vector, n = -c:
//     sphere:  nx^2  ny^2  nz^2  nx ny  nx nz  ny nz   nx  ny  nz   kk   1          kk = |c|^2 - r^2 - margin_s
//     ray:     dx^2  dy^2  dz^2  2dxdy  2dxdz  2dydz   2 (o.d d - o)    -1   (o.d)^2 - |o|^2 (1 - margin_r)
// i.e. a GEMM  E[rays x spheres] = R[rays x 11] S^T  -- 128 rays x 128 spheres per tcgen05.mma.  TF32 operands carry 11
// significant bits, so every feature is split  x = hi + lo  (both TF32) and the three products hi hi + lo hi + hi lo go into
// the K dimension:  K = 11 + 11 + 10 = 32 (the constant sphere feature has no low part) = four K = 8 instructions.
// Per test the CUDA cores are left with ONE instruction (the sign bit of e into the candidate mask) instead of eight packed FMA.
// The split products carry 2^-21 relative error and the accumulation order inside the tensor core is not documented, so the
// margins are wider than the FP32 filter's (kMargin in r1_encode.h, against 2^-17); the measured error is in DESIGN.md section 4.0 and
// tests/test_gpu_parity.py::test_tensor_filter_is_conservative checks the filter against the exact test on the GPU.
#pragma once
#include <cstdint>
#include <cstring>

#include "r1_encode.h"   // the operand layout and the sphere rows (kFeatures .. sphere_row_host)

namespace r1 {
namespace tc {

#ifdef __CUDACC__
// ---- PTX wrappers ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ bool mbar_try(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done != 0;
}
__device__ __forceinline__ bool mbar_try_hint(uint64_t *bar, uint32_t parity, uint32_t ns)   // suspends up to `ns` before it reports failure
{
    uint32_t done;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
                 : "memory");
    return done != 0;
}
// A barrier that never completes would hang the GPU; a protocol error traps instead (the launch then fails loudly).
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity, bool hint = false)
{
    uint32_t spins = 0;
    if (hint) {
        while (!mbar_try_hint(bar, parity, 100000u))
            if (++spins > (1u << 22)) __trap();
    } else {
        while (!mbar_try(bar, parity))
            if (++spins > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t *slot, uint32_t ncols)      // whole warp
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) { asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory"); }

// shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor): start >> 4 [0,14), LBO >> 4 [16,30),
// SBO >> 4 [32,46), version 1 [46,48), layout type 0 = no swizzle [61,64)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// instruction descriptor (InstrDescriptor): D = f32 [4,6), A = B = tf32 [7,10) [10,13), both K-major, N >> 3 [17,23), M >> 4 [24,29)
__device__ __forceinline__ uint32_t instr_desc(int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24); }

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc),
                 "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory"); }

// 32 consecutive columns of this thread's TMEM lane (warp w reads lanes 32 (w % 4) .. +31), complete on return
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, "
                 "%23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]),
                   "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]),
                   "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr)
                 : "memory");
    // the registers are defined only after wait::ld: tie them to it so that no use can be scheduled above
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]),
                   "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]),
                   "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
// the same in two steps: issue (the registers are undefined until tmem_wait), and one wait for two loads in flight
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_wait(uint32_t (&a)[32], uint32_t (&b)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]), "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]), "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31]),
                   "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]), "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15]), "+r"(b[16]), "+r"(b[17]), "+r"(b[18]), "+r"(b[19]), "+r"(b[20]), "+r"(b[21]), "+r"(b[22]), "+r"(b[23]), "+r"(b[24]), "+r"(b[25]), "+r"(b[26]), "+r"(b[27]), "+r"(b[28]), "+r"(b[29]), "+r"(b[30]), "+r"(b[31])
                 :
                 : "memory");
}
// sign bits of 32 filter values into a candidate mask: first sphere -> bit 31, set = flagged (e >= 0)
__device__ __forceinline__ uint32_t flagged(const uint32_t (&v)[32])
{
    // four independent funnel-shift chains of 8 (one chain of 32 is a 32-deep dependency)
    uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        m0 = __funnelshift_l(v[j], m0, 1);
        m1 = __funnelshift_l(v[8 + j], m1, 1);
        m2 = __funnelshift_l(v[16 + j], m2, 1);
        m3 = __funnelshift_l(v[24 + j], m3, 1);
    }
    return ~((m0 << 24) | (m1 << 16) | (m2 << 8) | m3);
}

// ---- device: the ray operand -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tf32_rna(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// The lifted TF32 row of one ray.  Rays without a path (`live` false) get a row that flags nothing: 0 x 9, -1, -2^126, so
// e = -(kk + 2^126) < 0 for every sphere with r^2 < 2^126, far spheres (r1_encode.h kFarC2) included, and -1e30 for padding.
// A live ray with |o|^2 >= 2^120 (or NaN) is out of the filter's range (r1_device.cuh "Filter arithmetic"): its row 0 x 9, -1, 2^121
// flags every sphere that can be hit (e = 2^121 - kk > 0 with kk < 2^120, or kk = -2^122) and no padding row (e = -1e30).  Every
// row is finite, so no product the tensor core forms is infinite or NaN.
__device__ __forceinline__ void ray_row(f3 o, f3 d, bool live, uint32_t (&row)[kK])
{
    float f[kFeatures];
    const float od = dot3(o, d), oo = dot3(o, o);
    f[0] = fmul(d.x, d.x); f[1] = fmul(d.y, d.y); f[2] = fmul(d.z, d.z);
    f[3] = fmul(fadd(d.x, d.x), d.y); f[4] = fmul(fadd(d.x, d.x), d.z); f[5] = fmul(fadd(d.y, d.y), d.z);
    f[6] = fmul(2.0f, fsub(fmul(od, d.x), o.x)); f[7] = fmul(2.0f, fsub(fmul(od, d.y), o.y)); f[8] = fmul(2.0f, fsub(fmul(od, d.z), o.z));
    f[9] = -1.0f;
    f[10] = fsub(fmul(od, od), fmul(oo, (float)(1.0 - kMargin)));
    const bool in_range = oo < 0x1p120f;
    if (!live || !in_range) {
#pragma unroll
        for (int j = 0; j < 9; ++j) f[j] = 0.0f;
        f[10] = live ? 0x1p121f : -0x1p126f;
    }
#pragma unroll
    for (int j = 0; j < kFeatures; ++j) {
        const uint32_t hi = tf32_rna(f[j]);
        row[j] = hi;
        row[kFeatures + j] = tf32_rna(fsub(f[j], __uint_as_float(hi)));
        if (j < kFeatures - 1) row[2 * kFeatures + j] = hi;
    }
}
// Row r of a 128-ray A tile in shared memory
__device__ __forceinline__ void write_ray_row(unsigned char *a_tile, int r, f3 o, f3 d, bool live)
{
    uint32_t row[kK];
    ray_row(o, d, live, row);
    unsigned char *base = a_tile + (uint32_t)(r >> 3) * kSBO + (uint32_t)(r & 7) * 16u;
#pragma unroll
    for (int kc = 0; kc < kK / 4; ++kc)
        *reinterpret_cast<uint4 *>(base + kc * kLBO) = make_uint4(row[4 * kc], row[4 * kc + 1], row[4 * kc + 2], row[4 * kc + 3]);
}

// The four K = 8 steps of one accumulator chunk:  D[128 x n] = A[128 x 32] B[n x 32]^T   (one thread)
__device__ __forceinline__ void mma_chunk(uint32_t d_tmem, uint32_t a_smem, uint32_t b_smem, int n, uint32_t lbo, uint32_t sbo)
{
    const uint32_t idesc = instr_desc(n);
#pragma unroll
    for (int k = 0; k < kK / 8; ++k)
        mma_tf32(d_tmem, smem_desc(a_smem + 2 * k * kLBO, lbo, sbo), smem_desc(b_smem + 2 * k * kLBO, lbo, sbo), idesc, k > 0);
}
#endif  // __CUDACC__

}  // namespace tc
}  // namespace r1
