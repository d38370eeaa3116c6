// Inline-PTX wrappers for the sm_100a features the engine uses: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld / fences) and the shared-memory + instruction descriptors.
// Bit layouts follow the PTX ISA "tcgen05" chapter (matrix descriptor, instruction descriptor).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "mw_common.cuh"

namespace mw {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------ packed fp32 pairs (FFMA2 / FADD2 / FMUL2 on sm_100)
// Two independent IEEE fp32 operations per instruction: the same bits as two scalar ones at half the issue slots.
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// ------------------------------------------------------------------ L2 eviction priority
// A cache policy (createpolicy) carried by a load as `.L2::cache_hint` sets the L2 eviction priority of the lines it touches.
// The PTX ISA's priority list includes evict_unchanged ("do not change eviction priority order as part of this access"),
// which implies that an access with any other priority re-marks a line that is already resident.  Hints may be ignored by
// the hardware; they never change what a load returns.  The policy is a pure value (no `volatile`): ptxas folds it into
// the load's uniform memory descriptor.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 16 read-only bytes, not allocated in L1, with an L2 cache policy.  Not `volatile`: the data must not change during the
// kernel (ld.global.nc), so the compiler may schedule the load freely.
__device__ __forceinline__ uint4 ldg_nc_hint(const void* p, uint64_t pol) {
    uint4 r;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
        : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return r;
}
// the 128-byte line holding p into L2, marked evict_last
__device__ __forceinline__ void prefetch_l2_evict_last(const void* p) {
    asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(p));
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (the launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("mw: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
            __trap();
        }
    }
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ------------------------------------------------------------------ tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T, 16-bit inputs (mw_h), fp32 accumulate.  One thread issues.
__device__ __forceinline__ void umma_h16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets row (lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
// store 32 lanes x 32 consecutive fp32 columns (thread i of the warp writes row lane base + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, SWIZZLE_128B.
//   bits [0,14)  start address >> 4          bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4     bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
// K-major operand (rows of 64 bf16 = one 128-byte swizzle row): 8-row groups are 1024 B apart (SBO),
// LBO unused.  MN-major operand (64 contiguous MN elements per 128-byte row, 8 K-rows per atom):
// SBO = stride between 8-row K groups (1024 B), LBO = stride between 64-element MN blocks.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor for kind::f16: 16-bit x 16-bit -> fp32 (MW_UMMA_FMT: 0 = fp16, 1 = bf16, mw_common.cuh).
//   [4,6) D format (1 = f32)  [7,10) A format  [10,13) B format
//   [15] A major (0 = K)  [16] B major (0 = K, 1 = MN)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_h16(int M, int N, int b_mn_major = 0) {
    return (1u << 4) | (MW_UMMA_FMT << 7) | (MW_UMMA_FMT << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------ thread-block clusters / distributed shared memory
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// address of the same shared-memory offset inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

}  // namespace ptx
}  // namespace mw
