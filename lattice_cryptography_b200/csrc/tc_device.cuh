// tc_device.cuh — the sm_100a asynchronous primitives of the tensor-core kernels: mbarriers, bulk global->shared copies,
// and tcgen05 (tensor-memory allocation, MMA, commit, loads).  Operands are K-major and unswizzled: a matrix of R rows
// is a sequence of 16-byte K columns, each holding its R rows of 16 bytes back to back (core matrices of 8 rows x 16
// bytes, 128 bytes apart along M / N, R * 16 bytes apart along K).
#pragma once
#include <cstdint>

namespace lcb {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* b, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_addr(b)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_tx(uint64_t* b, unsigned bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_addr(b)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra WAIT;\n\t"
        "}" ::"r"(smem_addr(b)),
        "r"(parity)
        : "memory");
}

// bytes (multiple of 16, both addresses 16-byte aligned) from global to shared, completion counted on bar as tx bytes
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

// generic-proxy shared-memory writes -> visible to the tensor cores (async proxy)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp: allocates `cols` tensor-memory columns, base address written to *slot
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, unsigned cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t base, unsigned cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// shared-memory matrix descriptor, no swizzle: lbo = byte distance of adjacent core matrices along K, sbo = along M / N
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
           (1ull << 46);
}

// instruction descriptor of kind::i8: u8 x u8 -> s32, both operands K-major
__host__ __device__ constexpr uint32_t umma_idesc_u8(int m, int n) {
    return (2u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// single thread: D[tmem] (+)= A * B^T
__device__ __forceinline__ void umma_u8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}

// single thread: bar receives one arrival when every MMA this thread issued so far has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(bar))
                 : "memory");
}

// whole warp: 16 consecutive 32-bit columns of the warp's 32 lanes (lane i of the warp reads tensor-memory lane
// 32 (warp % 4) + i; taddr carries that lane offset in its upper half)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
        "[%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace lcb
