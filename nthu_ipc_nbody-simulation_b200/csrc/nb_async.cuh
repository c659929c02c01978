// Device helpers shared by the large-N steppers (nb_large.cu, nb_sym.cu): 1-D TMA bulk copies into shared memory
// completed on an mbarrier, and the system-scope counters through which ranks signal that their rows have arrived.
#pragma once
#include <cstdint>

namespace nb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_sys(unsigned long long* p) {
    asm volatile("red.release.sys.global.add.u64 [%0], %1;" ::"l"(p), "l"(1ULL) : "memory");
}

// Spins until *counter >= target.  A lost peer must not hang the GPU: 2e10 clk (~10 s) after t0 the wait gives up and
// writes `code` to *status, which the host reports.
__device__ __forceinline__ void wait_counter(const unsigned long long* counter, unsigned long long target, int* status,
                                             int code, long long t0) {
    while (ld_acquire_sys(counter) < target) {
        if (clock64() - t0 > 20000000000LL) {
            *status = code;
            break;
        }
    }
}
__device__ __forceinline__ void wait_counter(const unsigned long long* counter, unsigned long long target, int* status,
                                             int code) {
    wait_counter(counter, target, status, code, clock64());
}

}  // namespace nb
