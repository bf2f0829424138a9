// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma /
// commit / ld / fences).  Everything here is header-only and device-only.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace gb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* d) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(d)) : "memory");
}
// 2D tiled load: coordinates are (inner, outer) element indices; signed, OOB zero-filled.
// 1-D bulk copy global -> shared (16-byte aligned address/size), completion counted on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gptr, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gptr), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* d, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(d)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// TMEM -> registers: each thread of the warp reads 32 (or 16) consecutive 32-bit columns of its lane.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Explicit shared-state-space accesses.  Pointers carved out of the dynamic shared-memory arena reach the compiler as generic
// addresses and turn into LD.E / ST.E (generic path, long scoreboard); these stay LDS / STS.
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ long long ld_shared_b64(uint32_t addr) {
    long long v;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(addr) : "memory");
    return v;
}

// Shared-memory matrix descriptor for a K-major bf16 tile stored as rows of 128 bytes (64 bf16) with the
// 128-byte swizzle TMA produces (CU_TENSOR_MAP_SWIZZLE_128B).  Atom = 8 rows x 128 B, so the stride between
// 8-row groups (SBO) is 1024 B; LBO is unused for a single swizzle atom along K.
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
    uint64_t desc = 0;
    desc |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);  // start address, bits [0,14)
    desc |= static_cast<uint64_t>(0) << 16;                     // LBO (ignored)
    desc |= static_cast<uint64_t>(1024 >> 4) << 32;             // SBO = 1024 B
    desc |= static_cast<uint64_t>(1) << 46;                     // descriptor version (sm_100)
    desc |= static_cast<uint64_t>(2) << 61;                     // layout type: SWIZZLE_128B
    return desc;
}

// kind::f16 instruction descriptor: bf16 A/B (K-major), fp32 accumulate, M x N tile.
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
    return (1u << 4)      // c_format = F32
           | (1u << 7)    // a_format = BF16
           | (1u << 10)   // b_format = BF16
           | (0u << 15)   // a_major  = K
           | (0u << 16)   // b_major  = K
           | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// ---------------------------------------------------------------- small math helpers
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
// erf-GELU (nn.GELU default).  erf by Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7, branch-free: 2 MUFU + 9 FMA-class ops instead of
// erff's ~25-instruction piecewise polynomial); the result is stored as bf16 (ulp 2^-8 relative), five orders of magnitude coarser.
__device__ __forceinline__ float gelu_erf(float x) {
    const float z = fabsf(x) * 0.70710678118654752440f;
    const float t = __frcp_rn(fmaf(0.3275911f, z, 1.0f));
    float pl = fmaf(t, 1.061405429f, -1.453152027f);
    pl = fmaf(t, pl, 1.421413741f);
    pl = fmaf(t, pl, -0.284496736f);
    pl = fmaf(t, pl, 0.254829592f);
    const float e = 1.0f - t * pl * __expf(-z * z);          // erf(|x| / sqrt 2)
    return 0.5f * x * (1.0f + copysignf(e, x));
}
__device__ __forceinline__ float silu(float x) { return x / (1.0f + __expf(-x)); }

}  // namespace gb

// ---------------------------------------------------------------- 2-CTA (cta_group::2) helpers
namespace gb {
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// split cluster barrier: arrive early (no memory ordering needed, it only proves "this CTA is running"), wait late
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.aligned;" ::: "memory"); }
// TMA load issued by either CTA of a pair; the transaction bytes are credited to the LEADER CTA's mbarrier (the barrier's
// shared::cluster address with the peer bit cleared names CTA 0's copy of the same offset).
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* d, uint64_t* bar, int32_t c0, int32_t c1) {
    const uint32_t bar_addr = smem_u32(bar) & 0xFEFFFFFFu;
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(d)), "r"(bar_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 remAddr32;\n\t"
        "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t}\n" ::"r"(smem_u32(bar)), "r"(cta)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_holder) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)), "n"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
}  // namespace gb
