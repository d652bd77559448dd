// rz_ptx.cuh -- PTX wrappers for mbarriers and bulk global -> shared copies, used by the staged K1 kernels
// (rz_k1_bitboard.cu) and the tcgen05 tower (rz_net_tc.cu).
#pragma once
#include <stdint.h>

namespace rz {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait (~4 s of SM clocks): a protocol bug traps and is reported to the host instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    long long t0 = 0;
    for (uint32_t spin = 0; !ok; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!ok && (spin & 1023) == 1023) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 8000000000LL) __trap();
        }
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace ptx
}  // namespace rz
