// keccak_f1600.cuh -- Keccak-f[1600] and the Keccak-256 sponge for one thread (sm_100a).
//
// One sponge per THREAD: the 25 64-bit lanes live in 50 registers, every index below is a compile-time
// constant after unrolling, so there is no local memory and no cross-lane traffic.  Integer work only:
// theta/chi fold into LOP3 (3-input logic), rho is two funnel shifts (SHF) per lane.  This is the
// B200 statement of the function phant reaches through src/crypto/hasher.zig:4-8 (Zig std Keccak256);
// the native twin in the reference tree is ethash/lib/keccak/keccak.c:58-269 (permutation) and
// :301-354 (sponge).  Round constants are the standard ones (keccak.c:38-46).
#pragma once
#include <stdint.h>

namespace phant {

__constant__ uint64_t KECCAK_RC[24] = {
    0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull,
    0x000000000000808bull, 0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull,
    0x000000000000008aull, 0x0000000000000088ull, 0x0000000080008009ull, 0x000000008000000aull,
    0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull, 0x8000000000008003ull,
    0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
    0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};

constexpr int KECCAK_RATE = 136;       // bytes absorbed per permutation (Keccak-256)
constexpr int KECCAK_RATE_WORDS = 17;  // 64-bit lanes per block

// 64-bit rotate left by a compile-time amount, as two 32-bit funnel shifts.
template <int N>
__device__ __forceinline__ uint64_t rol64(uint64_t x)
{
    if constexpr (N == 0) return x;
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    uint32_t rlo, rhi;
    if constexpr (N == 32) {
        rlo = hi; rhi = lo;
    } else if constexpr (N < 32) {
        rlo = __funnelshift_l(hi, lo, N);
        rhi = __funnelshift_l(lo, hi, N);
    } else {
        rlo = __funnelshift_l(lo, hi, N - 32);
        rhi = __funnelshift_l(hi, lo, N - 32);
    }
    return ((uint64_t)rhi << 32) | rlo;
}

// theta + rho + pi for one input lane: B[pi(I)] = rol(A[I] ^ D[I % 5], RHO[I]) with
// D[x] = C[x-1] ^ rol(C[x+1], 1) folded into the lane's own 3-input XOR (one LOP3 per half instead of
// forming D first: 122 LOP3 + 58 SHF per round, measured 4.27 vs 3.99 G perm/s register-resident).
#define PHANT_RHOPI(I, J, R) b[J] = rol64<R>(a[I] ^ c[((I) % 5 + 4) % 5] ^ r1[((I) % 5 + 1) % 5]);

__device__ __forceinline__ void keccak_round(uint64_t (&a)[25], uint64_t rc)
{
    uint64_t c[5], r1[5], b[25];
#pragma unroll
    for (int x = 0; x < 5; ++x) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
    for (int x = 0; x < 5; ++x) r1[x] = rol64<1>(c[x]);
    // lane I=x+5y moves to J=y+5((2x+3y)%5) rotated by RHO[I]
    PHANT_RHOPI(0, 0, 0)    PHANT_RHOPI(1, 10, 1)   PHANT_RHOPI(2, 20, 62)  PHANT_RHOPI(3, 5, 28)   PHANT_RHOPI(4, 15, 27)
    PHANT_RHOPI(5, 16, 36)  PHANT_RHOPI(6, 1, 44)   PHANT_RHOPI(7, 11, 6)   PHANT_RHOPI(8, 21, 55)  PHANT_RHOPI(9, 6, 20)
    PHANT_RHOPI(10, 7, 3)   PHANT_RHOPI(11, 17, 10) PHANT_RHOPI(12, 2, 43)  PHANT_RHOPI(13, 12, 25) PHANT_RHOPI(14, 22, 39)
    PHANT_RHOPI(15, 23, 41) PHANT_RHOPI(16, 8, 45)  PHANT_RHOPI(17, 18, 15) PHANT_RHOPI(18, 3, 21)  PHANT_RHOPI(19, 13, 8)
    PHANT_RHOPI(20, 14, 18) PHANT_RHOPI(21, 24, 2)  PHANT_RHOPI(22, 9, 61)  PHANT_RHOPI(23, 19, 56) PHANT_RHOPI(24, 4, 14)
#pragma unroll
    for (int y = 0; y < 25; y += 5) {
#pragma unroll
        for (int x = 0; x < 5; ++x) a[y + x] = b[y + x] ^ (~b[y + (x + 1) % 5] & b[y + (x + 2) % 5]);
    }
    a[0] ^= rc;
}

// The 24th round when only the 256-bit digest (lanes 0..3) is read afterwards: theta needs every column parity, but rho/pi
// and chi only have to produce row 0 -- B[0..4] come from lanes 0, 6, 12, 18, 24.  40 LOP3 + 18 SHF instead of 122 + 58.
// Lanes 4..24 of `a` are left stale.
__device__ __forceinline__ void keccak_last_round_digest(uint64_t (&a)[25], uint64_t rc)
{
    uint64_t c[5], r1[5], b[5];
#pragma unroll
    for (int x = 0; x < 5; ++x) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
    for (int x = 0; x < 5; ++x) r1[x] = rol64<1>(c[x]);
    PHANT_RHOPI(0, 0, 0) PHANT_RHOPI(6, 1, 44) PHANT_RHOPI(12, 2, 43) PHANT_RHOPI(18, 3, 21) PHANT_RHOPI(24, 4, 14)
#pragma unroll
    for (int x = 0; x < 4; ++x) a[x] = b[x] ^ (~b[(x + 1) % 5] & b[(x + 2) % 5]);
    a[0] ^= rc;
}
#undef PHANT_RHOPI

// UNROLL rounds per loop trip (24 % UNROLL == 0).  2 keeps the body inside the instruction cache.
// DIGEST_ONLY: the last permutation of a message -- the final trip is peeled and its last round pruned to row 0.
template <int UNROLL = 2, bool DIGEST_ONLY = false>
__device__ __forceinline__ void keccak_f1600(uint64_t (&a)[25])
{
    constexpr int LOOPED = DIGEST_ONLY ? 24 - UNROLL : 24;
#pragma unroll 1
    for (int r = 0; r < LOOPED; r += UNROLL) {
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) keccak_round(a, KECCAK_RC[r + k]);
    }
    if constexpr (DIGEST_ONLY) {
#pragma unroll
        for (int k = 0; k < UNROLL - 1; ++k) keccak_round(a, KECCAK_RC[LOOPED + k]);
        keccak_last_round_digest(a, KECCAK_RC[23]);
    }
}

// ---- byte-granular message access ------------------------------------------------------------
// A message starts at any byte address.  `w` points at the 8-byte aligned word holding its first
// byte and `sh` = 8 * (address & 7): message word k is the funnel of aligned words k and k+1.
struct MsgView {
    const uint64_t* w;
    uint32_t sh; // 0, 8, .. 56
};
__device__ __forceinline__ MsgView msg_view(const void* p)
{
    const uintptr_t a = (uintptr_t)p;
    return MsgView{(const uint64_t*)(a & ~(uintptr_t)7), (uint32_t)(a & 7) * 8};
}
__device__ __forceinline__ uint64_t funnel64(uint64_t lo, uint64_t hi, uint32_t sh)
{
    return sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
}

// Absorb one full 136-byte block starting at message word `base`.
template <int UNROLL>
__device__ __forceinline__ void absorb_full(uint64_t (&st)[25], const MsgView& v, uint32_t base)
{
    uint64_t w[KECCAK_RATE_WORDS + 1];
#pragma unroll
    for (int k = 0; k < KECCAK_RATE_WORDS; ++k) w[k] = v.w[base + k];
    // with a misaligned start the byte after the block is still a message byte of this block's
    // last word, so word base+17 always holds valid bytes when sh != 0
    w[KECCAK_RATE_WORDS] = v.sh ? v.w[base + KECCAK_RATE_WORDS] : 0;
#pragma unroll
    for (int k = 0; k < KECCAK_RATE_WORDS; ++k) st[k] ^= funnel64(w[k], w[k + 1], v.sh);
    keccak_f1600<UNROLL>(st);
}

// Absorb the last (partial, possibly empty) block: `rem` < 136 bytes at message word `base`, then
// pad 0x01 .. 0x80 (keccak.c:341-347) and permute.  Never touches a word holding no message byte.
template <int UNROLL>
__device__ __forceinline__ void absorb_final(uint64_t (&st)[25], const MsgView& v, uint32_t base, uint32_t rem)
{
    const uint32_t mis = v.sh >> 3;
#pragma unroll
    for (int k = 0; k < KECCAK_RATE_WORDS; ++k) {
        const int valid = (int)rem - 8 * k; // message bytes in this word (may be <= 0 or >= 8)
        uint64_t word = 0;
        if (valid > 0) {
            const uint64_t lo = v.w[base + k];
            const uint64_t hi = (mis + (valid > 8 ? 8 : valid) > 8) ? v.w[base + k + 1] : 0;
            word = funnel64(lo, hi, v.sh);
            if (valid < 8) word &= (1ull << (8 * valid)) - 1;
        }
        if (valid >= 0 && valid < 8) word ^= 1ull << (8 * valid); // 0x01 right after the message
        st[k] ^= word;
    }
    st[KECCAK_RATE_WORDS - 1] ^= 0x8000000000000000ull;
    keccak_f1600<UNROLL, true>(st); // callers read the digest only
}

// ---- shared-memory absorb (staged kernel) -------------------------------------------------------
// The message sits in the lane's shared-memory slot at byte address `sa` (any alignment).  Read it as aligned
// 32-bit words (LDS.32 on the LSU pipe) and fix the byte skew with ONE funnel shift per word: 34 SHF + 34 LOP3 on
// the ALU pipe per 136-byte block, against ~180 for the generic 64-bit path above.
#ifndef PHANT_HOST_SMEM
__device__ __forceinline__ uint32_t lds32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
#else // test harness (tests/hostcheck): "shared memory" is a host array, addresses are offsets into it
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) { uint32_t v; memcpy(&v, PHANT_HOST_SMEM + saddr, 4); return v; }
#endif
// `aligned`: the caller knows sa % 4 == 0 for every lane of the warp (a warp-uniform test), so the words are the block's bytes
// as they are and the 34 funnel shifts are skipped.  Only the absorb is duplicated; the permutation stays one copy.
template <int UNROLL, bool DIGEST_ONLY = false>
__device__ __forceinline__ void absorb_full_smem(uint64_t (&st)[25], uint32_t sa, bool aligned = false)
{
    if (aligned) {
#pragma unroll
        for (int k = 0; k < KECCAK_RATE_WORDS; ++k) st[k] ^= ((uint64_t)lds32(sa + 8 * k + 4) << 32) | lds32(sa + 8 * k);
    } else {
        const uint32_t a4 = sa & ~3u, sh = (sa & 3u) * 8;
        uint32_t w[2 * KECCAK_RATE_WORDS + 1];
#pragma unroll
        for (int j = 0; j < 2 * KECCAK_RATE_WORDS; ++j) w[j] = lds32(a4 + 4 * j);
        w[2 * KECCAK_RATE_WORDS] = sh ? lds32(a4 + 4 * 2 * KECCAK_RATE_WORDS) : 0; // holds block bytes only when skewed
#pragma unroll
        for (int k = 0; k < KECCAK_RATE_WORDS; ++k) {
            const uint32_t lo = __funnelshift_r(w[2 * k], w[2 * k + 1], sh);
            const uint32_t hi = __funnelshift_r(w[2 * k + 1], w[2 * k + 2], sh);
            st[k] ^= ((uint64_t)hi << 32) | lo;
        }
    }
    keccak_f1600<UNROLL, DIGEST_ONLY>(st);
}
// last block: rem < 136 message bytes at `sa`.  The 0x01 .. 00 .. 0x80 padding is WRITTEN INTO THE SLOT (stores go to the
// idle LSU pipe) and the block is then absorbed like a full one: no per-word masks or predicates on the ALU pipe, which
// is the pipe this kernel is bound by.  The slot is private to the lane, the block ends inside it (skew + 4*136 <= 559).
#ifndef PHANT_HOST_SMEM
__device__ __forceinline__ void sts32_(uint32_t saddr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }
#else
__device__ __forceinline__ void sts32_(uint32_t saddr, uint32_t v) { memcpy(PHANT_HOST_SMEM + saddr, &v, 4); }
#endif
// The same block with the padding applied in registers (masks): used when the 136-byte block would not fit behind `sa`
// inside the lane's slot (a message whose last few bytes follow four full blocks of the window).
template <int UNROLL>
__device__ __forceinline__ void absorb_final_smem_masked(uint64_t (&st)[25], uint32_t sa, uint32_t rem)
{
    const uint32_t a4 = sa & ~3u, sh = (sa & 3u) * 8;
    const uint32_t nfw = rem >> 2, tail = rem & 3u;
    const uint32_t bmask = (1u << (8 * tail)) - 1u, pad = 1u << (8 * tail);
    uint32_t prev = rem ? lds32(a4) : 0;
#pragma unroll
    for (int j = 0; j < 2 * KECCAK_RATE_WORDS; ++j) {
        uint32_t word = 0;
        if ((uint32_t)j < nfw || ((uint32_t)j == nfw && tail)) {
            const uint32_t next = lds32(a4 + 4 * (j + 1));
            word = __funnelshift_r(prev, next, sh);
            prev = next;
        }
        if ((uint32_t)j == nfw) word = (word & bmask) ^ pad;
        if (j == 2 * KECCAK_RATE_WORDS - 1) word ^= 0x80000000u;
        st[j >> 1] ^= (j & 1) ? ((uint64_t)word << 32) : (uint64_t)word;
    }
    keccak_f1600<UNROLL, true>(st);
}
// `room` = bytes from `sa` to the end of the lane's slot
template <int UNROLL>
__device__ __forceinline__ void absorb_final_smem(uint64_t (&st)[25], uint32_t sa, uint32_t rem, uint32_t room, bool aligned = false)
{
    if (room < KECCAK_RATE + 4) { absorb_final_smem_masked<UNROLL>(st, sa, rem); return; }
    const uint32_t a4 = sa & ~3u, s = sa & 3u;
    const uint32_t p0 = rem + s, p1 = KECCAK_RATE - 1 + s;      // byte positions (from a4) of the 0x01 and the 0x80
    const uint32_t q0 = p0 >> 2, b0 = p0 & 3u, q1 = p1 >> 2, b1 = p1 & 3u;
    uint32_t w0 = lds32(a4 + 4 * q0);
    w0 = (w0 & ((1u << (8 * b0)) - 1u)) | (1u << (8 * b0));     // keep the message bytes below, 0x01, zeros above
    if (q0 == q1) w0 |= 0x80u << (8 * b1);                      // rem == 135 (or the same word): 0x01 and 0x80 meet
    sts32_(a4 + 4 * q0, w0);
    for (uint32_t q = q0 + 1; q < q1; ++q) sts32_(a4 + 4 * q, 0u);
    if (q1 > q0) sts32_(a4 + 4 * q1, 0x80u << (8 * b1));        // bytes above b1 lie past the block and are never used
    absorb_full_smem<UNROLL, true>(st, sa, aligned);            // last permutation: only the digest lanes are finished
}

// Whole-message Keccak-256 from global or shared memory (generic pointer), any alignment.
template <int UNROLL = 2>
__device__ __forceinline__ void keccak256_thread(const uint8_t* p, uint64_t len, uint64_t (&digest)[4])
{
    uint64_t st[25];
#pragma unroll
    for (int i = 0; i < 25; ++i) st[i] = 0;
    const MsgView v = msg_view(p);
    uint32_t base = 0;
    while (len >= KECCAK_RATE) {
        absorb_full<UNROLL>(st, v, base);
        base += KECCAK_RATE_WORDS;
        len -= KECCAK_RATE;
    }
    absorb_final<UNROLL>(st, v, base, (uint32_t)len);
#pragma unroll
    for (int i = 0; i < 4; ++i) digest[i] = st[i];
}

} // namespace phant
