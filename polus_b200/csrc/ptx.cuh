// Inline-PTX wrappers for the Blackwell (sm_100a) async machinery: mbarrier, TMA, tcgen05/TMEM.
#pragma once
#include <stdint.h>
#include <cuda.h>

namespace ptx {

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
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("polus_b200: mbarrier wait timeout (block %d thread %d bar %u parity %u)\n",
                   (int)blockIdx.x, (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// 2-CTA variant: executed by BOTH CTAs of the pair; the completion bytes land on the LEADER CTA's barrier
// (peer bit 24 of the shared::cluster address cleared).
__device__ __forceinline__ void tma_load_4d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                                int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu),
        "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// 1-D bulk copy global -> shared (bytes and both addresses multiples of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// TMA store: swizzled smem block -> global (rows/columns outside the tensor map are clipped)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// TMA prefetch of one box into L2 (no shared-memory destination, no barrier): warms the L2 for a load that a LATER CTA will issue
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// TMA reduction: global[tile] += smem block (element type from the tensor map; fp32 add done at L2)
__device__ __forceinline__ void tma_reduce_add_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// make generic-proxy writes to shared memory visible to the async proxy (TMA engine)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(cta)
        : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_slot) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_slot)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
                 : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                              uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (count 1) on the barrier at this smem offset in every CTA of `cta_mask` (default: both CTAs of a 2-CTA cluster)
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask = 3) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(cta_mask)
        : "memory");
}

template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_slot)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = TMEM lane).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
          "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor (sm_100 "version 1"), 128-byte swizzle.
//   [0,14)  start address >> 4     [16,30) leading byte offset >> 4
//   [32,46) stride byte offset >> 4 [46,48) version = 1   [61,64) layout type (2 = SWIZZLE_128B)
// K-major tile  : rows of 64 bf16 (128 B), 8-row swizzle atoms 1024 B apart  -> SBO = 1024, LBO unused (1)
// MN-major tile : [MN/64][BLOCK_K][64] bf16; 8-k atoms 1024 B apart (SBO), 64-wide MN groups
//                 BLOCK_K*128 B apart (LBO)
__device__ __forceinline__ uint64_t umma_desc_base(uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ uint64_t umma_desc(uint64_t base, uint32_t smem_addr) {
    return base | (uint64_t)((smem_addr >> 4) & 0x3FFF);
}
// Instruction descriptor, kind::f16, bf16 x bf16 -> fp32.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4)                         // D format: F32
           | (1u << 7)                       // A format: BF16
           | (1u << 10)                      // B format: BF16
           | ((uint32_t)a_mn_major << 15)    // A major
           | ((uint32_t)b_mn_major << 16)    // B major
           | ((uint32_t)(N >> 3) << 17)      // N
           | ((uint32_t)(M >> 4) << 24);     // M
}

}  // namespace ptx
