// peer_sync.cuh -- system-scope flag accesses of the peer-memory epilogue (comm.cu "peer transport"), shared by the kernels
// that end a proof batch (walk_kernel.cu, verify_fused.cu).
#pragma once
#include <stdint.h>

namespace phant {
namespace {

// system-scope flag accesses for the peer epilogue
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v)
{
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// spin until flags[r] >= value for every r < world (bounded: a peer that died must not hang this GPU)
__device__ __forceinline__ void wait_flags(const unsigned long long* flags, uint32_t world, unsigned long long value, uint32_t* err)
{
    const unsigned long long t0 = global_timer_ns();
    for (uint32_t r = 0; r < world; ++r)
        while (ld_acquire_sys(flags + r) < value)
            if (global_timer_ns() - t0 > 4000000000ull) { *err = 1; return; }
}

} // namespace
} // namespace phant
