// tma_util.cuh — mbarrier / TMA bulk-copy wrappers (inline PTX) shared by the TMA-staged step kernels.
#pragma once
#include <cstdint>

namespace snn {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// consumer-side wait: spin (a sleep or a suspend-time hint changes neither the power draw nor the time, DESIGN.md §2)
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// producer-side wait: back off 256 ns between probes so that the spinning lane does not eat issue slots of the consumers
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (true) {
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}\n" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(256);
    }
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// order prior generic-proxy observations (an acquire of a peer's arrival flag) before subsequent async-proxy (TMA) reads
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

}  // namespace snn
