// stage.cuh -- the per-lane shared-memory staging of the hash kernels (keccak_kernels.cu, verify_fused.cu): slot geometry,
// the per-warp mbarrier and the bulk-copy engine (cp.async.bulk -> SASS UBLKCP).
#pragma once
#include <stdint.h>

#include "keccak_f1600.cuh"

namespace phant {

// window = what one bulk copy brings in: BLOCKS rate blocks + 15 bytes of skew, rounded to 16 x odd so that the 16-byte
// windows of a quarter warp fall in distinct banks.  The lane's slot is 32 bytes longer than the window (still 16 x odd):
// the final block is padded IN the slot (absorb_final_smem), which needs 140 bytes behind the block's start; with only
// the window, a last block that follows BLOCKS-1 full ones at a skew of 13..15 did not fit and took the masked path --
// 3 of 16 such messages at arbitrary alignment, and because lanes of one warp then split between the two paths the warp
// paid for both (C3: 3.93 -> 3.30 G perm/s).  + 16 bytes behind the last slot: the reader may touch 4 bytes past a message.
constexpr int stage_window(int blocks)
{
    int s = (blocks * KECCAK_RATE + 15 + 15) / 16;
    if (s % 2 == 0) ++s;
    return 16 * s;
}
constexpr int stage_slot(int blocks) { return stage_window(blocks) + 32; }
constexpr int stage_smem(int blocks, int warps) { return 128 + warps * 32 * stage_slot(blocks) + 16; }
static_assert(stage_smem(4, 12) <= 232448, "default shape must fit the 227 KB a CTA may opt into");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

} // namespace phant
