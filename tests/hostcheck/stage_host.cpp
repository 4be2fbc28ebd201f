// Test-only: the staged Keccak kernel's per-lane absorb path (phant_b200/csrc/keccak_f1600.cuh: absorb_full_smem,
// absorb_final_smem with its in-slot padding and masked fallback) compiled as HOST code, with "shared memory" a host array.
// The control flow around the absorb calls restates keccak256_staged_kernel's loop for ONE lane (window copy of <= WINDOW
// bytes from the 16-byte aligned address below the cursor, byte skew, full blocks, final block with `room`).
// stdin: "<pad_front> <hex message>" per line ("-" = empty); stdout: digest.  Argument "aligned": absorb with `aligned` set,
// as the kernel does when every lane's cursor is a multiple of 4 (a line whose pad_front is not is refused, exit code 2).
// Nothing in the product links this.
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#define __device__
#define __forceinline__ inline
#define __constant__ static const
static inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, uint32_t n) { n &= 31; return n ? (hi << n) | (lo >> (32 - n)) : hi; }
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t n) { n &= 31; return n ? (lo >> n) | (hi << (32 - n)) : lo; }
static uint8_t g_smem[4096];
#define PHANT_HOST_SMEM g_smem
#include "../../phant_b200/csrc/keccak_f1600.cuh"

using namespace phant;

// geometry of the default kernel shape (keccak_kernels.cu: stage_window(4) / stage_slot(4))
constexpr int BLOCKS = 4;
constexpr int WINDOW = 16 * (((BLOCKS * KECCAK_RATE + 15 + 15) / 16) | 1); // rounded to 16 x odd
constexpr int SLOT = WINDOW + 32;
static_assert(WINDOW == 560 && SLOT == 592, "keep in step with keccak_kernels.cu");

static void lane(const uint8_t* buf /*16-byte aligned, message at buf+front*/, uint64_t front, uint64_t len, bool aligned, uint8_t out[32],
                 int* used_masked)
{
    const uint32_t slot_s = 64; // the lane's slot inside g_smem (16-byte aligned, like the device slots)
    uint64_t cur = front, end = front + len;
    uint64_t st[25] = {0};
    bool done = false;
    while (!done) {
        const uint64_t need = end - cur, a0 = cur & ~(uint64_t)15;
        uint32_t cs = 0;
        if (need) {
            const uint64_t span = ((end - a0) + 15) & ~(uint64_t)15;
            cs = span < (uint64_t)WINDOW ? (uint32_t)span : WINDOW;
            memset(g_smem + slot_s, 0xEE, SLOT);    // stale bytes of the previous tile: must never matter
            memcpy(g_smem + slot_s, buf + a0, cs);  // the bulk copy
        }
        const uint32_t skew = (uint32_t)(cur - a0);
        const uint64_t in_slot = cs - skew;
        const uint64_t avail = need < in_slot ? need : in_slot;
        const uint32_t nfull = (uint32_t)(avail / KECCAK_RATE);
        uint32_t sa = slot_s + skew;
        for (uint32_t b = 0; b < nfull; ++b) { absorb_full_smem<2>(st, sa, aligned); sa += KECCAK_RATE; }
        if (avail == need) {
            const uint32_t room = slot_s + SLOT - sa;
            if (room < KECCAK_RATE + 4) ++*used_masked;
            absorb_final_smem<2>(st, sa, (uint32_t)(avail - (uint64_t)nfull * KECCAK_RATE), room, aligned);
            done = true;
        } else {
            cur += (uint64_t)nfull * KECCAK_RATE;
        }
    }
    memcpy(out, st, 32);
}

int main(int argc, char** argv)
{
    const bool aligned = argc > 1 && strcmp(argv[1], "aligned") == 0;
    static char line[1 << 17];
    int masked = 0;
    while (fgets(line, sizeof line, stdin)) {
        unsigned front = 0;
        int consumed = 0;
        if (sscanf(line, "%u %n", &front, &consumed) < 1) continue;
        char* hex = line + consumed;
        size_t hl = strlen(hex);
        while (hl && (hex[hl - 1] == '\n' || hex[hl - 1] == '\r')) hex[--hl] = 0;
        std::vector<uint8_t> buf(front + hl / 2 + 64 + 16, 0xA5); // 0xA5 neighbours: reading them into the state would show
        uint8_t* base = (uint8_t*)(((uintptr_t)buf.data() + 15) & ~(uintptr_t)15);
        size_t n = 0;
        if (strcmp(hex, "-") != 0)
            for (; 2 * n + 1 < hl; ++n) { unsigned v; sscanf(hex + 2 * n, "%2x", &v); base[front + n] = (uint8_t)v; }
        if (aligned && (front & 3)) { fprintf(stderr, "pad_front %u is not a multiple of 4\n", front); return 2; }
        uint8_t dg[32];
        lane(base, front, n, aligned, dg, &masked);
        for (int i = 0; i < 32; ++i) printf("%02x", dg[i]);
        printf("\n");
    }
    fprintf(stderr, "masked_fallbacks %d\n", masked);
    return 0;
}
