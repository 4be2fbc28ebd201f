// Test-only: ONE lane of verify_fused_kernel (phant_b200/csrc/verify_fused.cu) compiled as HOST code, with "shared memory" a
// host array.  The loop below restates the kernel's `while` body for a single lane: window copy of <= WINDOW bytes from the
// 16-byte aligned address below the cursor, full blocks, the final block padded IN the slot, the digest compared with the
// parent's reference, then walk_node reading the node from the slot (SlotBytes) on the first trip or from the node buffer
// (GlobalBytes) for a node longer than one window.  The absorb, the summary, the walk step and the slot geometry are the
// product headers themselves.  Built as a shared object by tests/test_fused_lane_host.py; nothing in the product links this.
//
// Unlike the ABI's contiguous CSR, every node has its own start address in `buf`, so a test can put any node at any byte
// skew.  Every proof runs twice: with the kernel's aligned absorb wherever the cursor is a multiple of 4, and with the
// unaligned absorb only; both must agree.  Each run checks what a wrong bound could never show in a verdict:
//   F_SLOT_BOUNDS  a read by walk_node through SlotBytes (at / load32 / load32_tail) left the lane's slot
//   F_ALIGN_DIFF   the aligned and the unaligned run disagree (status, val_off or val_len)
//   F_SUMMARY      summarize_node on the padded slot != summarize_node on the node alone
//   F_GUARD        bytes around the slot changed (the in-slot padding wrote outside it)
//   F_WINDOW       a window copy reached past the end of `buf` (the device would read past the node buffer)
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#define __device__
#define __forceinline__ inline
#define __constant__ static const
#define __restrict__
struct uint4 { uint32_t x, y, z, w; };
static inline uint4 __ldg(const uint4* p) { uint4 v; memcpy(&v, p, sizeof v); return v; }
static inline int __popc(uint32_t v) { return __builtin_popcount(v); }
static inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, uint32_t n) { n &= 31; return n ? (hi << n) | (lo >> (32 - n)) : hi; }
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t n) { n &= 31; return n ? (lo >> n) | (hi << (32 - n)) : lo; }
static inline size_t __cvta_generic_to_shared(const void* p) { return (size_t)p; } // stage.cuh's smem_u32: never called here
alignas(128) static uint8_t g_smem[4096];
#define PHANT_HOST_SMEM g_smem
#include "../../phant_b200/csrc/keccak_f1600.cuh"
#include "../../phant_b200/csrc/node_summary.cuh"
#include "../../phant_b200/csrc/stage.cuh"
#include "../../phant_b200/csrc/walk_one.cuh"

using namespace phant;

// geometry of the kernel's shape (verify_fused.cu launch_fused: BLOCKS = 4)
constexpr int BLOCKS = 4;
constexpr int WINDOW = stage_window(BLOCKS), SLOT = stage_slot(BLOCKS);
static_assert(WINDOW == 560 && SLOT == 592, "the tests' window and fallback bands assume the default shape");

enum { F_SLOT_BOUNDS = 1, F_ALIGN_DIFF = 2, F_SUMMARY = 4, F_GUARD = 8, F_WINDOW = 16 };
enum { C_TAIL_OK_TRUE, C_TAIL_OK_FALSE, C_MASKED, C_MULTI_WINDOW, C_ALIGNED_ABSORB, C_SLOT_WALKS, C_GLOBAL_WALKS, C_NODES, C_COUNT };

constexpr uint32_t SLOT_S = 1024;            // the lane's slot inside g_smem (16-byte aligned, like the device slots)
constexpr uint32_t GUARD = 256;              // bytes watched on either side of the slot
constexpr uint8_t STALE = 0xEE, GUARD_BYTE = 0x5A;

static uint64_t* g_count; // counters of the current run (nullptr: the second, unaligned-only run is not counted)
static inline void count(int c) { if (g_count) ++g_count[c]; }

// SlotBytes behind a bounds check: every byte any accessor touches must lie inside the lane's slot
struct CheckedSlot {
    SlotBytes s;
    mutable bool* oob;
    void touch(const uint8_t* lo, const uint8_t* hi) const // [lo, hi)
    {
        if (lo < g_smem + SLOT_S || hi > g_smem + SLOT_S + SLOT) *oob = true;
    }
    // SlotBytes::load32_at reads nine 32-bit words from the 4-byte aligned address at or below q
    void touch32(const uint8_t* q) const
    {
        const uint8_t* w = (const uint8_t*)((uintptr_t)q & ~(uintptr_t)3);
        touch(w, w + 36);
    }
    uint32_t at(uint32_t o) const { touch(s.p + o, s.p + o + 1); return s.at(o); }
    void load32(uint32_t o, uint32_t (&e)[8]) const { touch32(s.p + o); s.load32(o, e); }
    bool tail_ok(uint32_t e) const { const bool ok = s.tail_ok(e); count(ok ? C_TAIL_OK_TRUE : C_TAIL_OK_FALSE); return ok; }
    void load32_tail(uint32_t e, uint32_t (&t)[8]) const { touch32(s.p + e - 32); s.load32_tail(e, t); }
    uint64_t abs(uint32_t o) const { return s.abs(o); }
};

struct Batch {
    const uint8_t* buf; // 16-byte aligned node buffer
    uint64_t buf_len;
    const uint64_t* node_start;
    const uint64_t* node_len;
    const uint64_t* proof_first;
    const uint8_t* keys32;
    const uint8_t* roots32;
    uint64_t n_roots;
};

static bool guards_intact()
{
    for (uint32_t i = SLOT_S - GUARD; i < SLOT_S; ++i) if (g_smem[i] != GUARD_BYTE) return false;
    for (uint32_t i = SLOT_S + SLOT; i < SLOT_S + SLOT + GUARD; ++i) if (g_smem[i] != GUARD_BYTE) return false;
    return true;
}

// one lane of verify_fused_kernel for proof p; `use_aligned`: take the aligned absorb when the cursor is a multiple of 4
static int lane(const Batch& B, uint64_t p, bool use_aligned, uint64_t& voff, uint32_t& vlen, uint32_t& fail)
{
    uint64_t j = B.proof_first[p], jl = B.proof_first[p + 1], nbeg = 0, cur = 0, end = 0;
    uint32_t pos = 0, expect[8], kw[8];
    voff = 0; vlen = 0;
    load32_aligned(B.roots32 + (B.n_roots == 1 ? 0 : 32 * p), expect);
    load32_aligned(B.keys32 + 32 * p, kw);
    if (j == jl) return eq32_const(EMPTY_ROOT, expect) ? ST_ABSENT : ST_REJECT; // no node: only the empty trie proves anything
    nbeg = cur = B.node_start[j];
    end = nbeg + B.node_len[j];
    if (end - nbeg > 0xffffffffull) return ST_REJECT;
    uint64_t st[25] = {0};
    bool first_trip = true;
    for (;;) {
        const uint64_t need = end - cur, a0 = cur & ~(uint64_t)15;
        uint32_t cs = 0;
        if (need) {
            const uint64_t span = ((end - a0) + 15) & ~(uint64_t)15;
            cs = span < (uint64_t)WINDOW ? (uint32_t)span : WINDOW;
            if (a0 + cs > B.buf_len) { fail |= F_WINDOW; return ST_REJECT; }
            memset(g_smem + SLOT_S, STALE, SLOT);      // stale bytes of an earlier tile: must never matter
            memcpy(g_smem + SLOT_S, B.buf + a0, cs);   // the bulk copy
        } // need == 0 (an empty node): no copy, the slot keeps the previous node's bytes, as on the device
        const bool aligned = use_aligned && (cur & 3) == 0;
        const uint32_t skew = (uint32_t)(cur - a0);
        const uint64_t in_slot = cs - skew;
        const uint64_t avail = need < in_slot ? need : in_slot;
        const uint32_t nfull = (uint32_t)(avail / KECCAK_RATE);
        uint32_t sa = SLOT_S + skew;
        for (uint32_t b = 0; b < nfull; ++b) {
            absorb_full_smem<2>(st, sa, aligned);
            if (aligned) count(C_ALIGNED_ABSORB);
            sa += KECCAK_RATE;
        }
        if (avail != need) { // the node goes on past this window
            cur += (uint64_t)nfull * KECCAK_RATE;
            first_trip = false;
            continue;
        }
        const uint32_t room = SLOT_S + SLOT - sa;
        if (room < KECCAK_RATE + 4) count(C_MASKED);
        absorb_final_smem<2>(st, sa, (uint32_t)(avail - (uint64_t)nfull * KECCAK_RATE), room, aligned);
        if (aligned) count(C_ALIGNED_ABSORB);
        if (!guards_intact()) fail |= F_GUARD;
        count(C_NODES);
        if (!first_trip) count(C_MULTI_WINDOW);
        uint32_t diff = 0; // R1: the node's digest is the reference its parent named
        for (int w = 0; w < 4; ++w) diff |= ((uint32_t)st[w] ^ expect[2 * w]) | ((uint32_t)(st[w] >> 32) ^ expect[2 * w + 1]);
        const uint32_t len = (uint32_t)(end - nbeg);
        int r = ST_REJECT;
        ++j;
        if (first_trip) { // the summary the walk would read, against the same node with nothing around it
            std::vector<uint8_t> alone(len + 64, 0xA5);
            memcpy(alone.data(), B.buf + nbeg, len);
            if (summarize_node(g_smem + SLOT_S + skew, len) != summarize_node(alone.data(), len)) fail |= F_SUMMARY;
        }
        if (diff == 0) {
            if (first_trip) { // the whole node is in the slot
                const uint8_t* np = g_smem + SLOT_S + skew;
                bool oob = false;
                count(C_SLOT_WALKS);
                r = walk_node(CheckedSlot{SlotBytes{np, skew, nbeg}, &oob}, len, summarize_node(np, len), j == jl, kw, pos, expect, voff, vlen);
                if (oob) fail |= F_SLOT_BOUNDS;
            } else {
                count(C_GLOBAL_WALKS);
                r = walk_node(GlobalBytes{B.buf, nbeg}, len, 0u, j == jl, kw, pos, expect, voff, vlen);
            }
            if (r == ST_NEXT && j == jl) r = ST_REJECT; // R3: a hash reference needs a node
        }
        if (r != ST_NEXT) return r;
        // next node of the chain (its own start: the harness is not bound to a contiguous CSR)
        nbeg = cur = B.node_start[j];
        end = nbeg + B.node_len[j];
        if (end - nbeg > 0xffffffffull) return ST_REJECT;
        for (int i = 0; i < 25; ++i) st[i] = 0;
        first_trip = true;
    }
}

// status / val_off (offset in buf) / val_len per proof, as verify_fused_kernel stores them; fail = F_* bits per proof;
// counters[C_COUNT] are added to.  Returns the number of proofs with a non-zero fail.
extern "C" uint64_t fusedlane_run(const uint8_t* buf, uint64_t buf_len, const uint64_t* node_start, const uint64_t* node_len,
                                  const uint64_t* proof_first, uint64_t n_proofs, const uint8_t* keys32, const uint8_t* roots32,
                                  uint64_t n_roots, uint8_t* status, uint64_t* val_off, uint32_t* val_len, uint8_t* fail,
                                  uint64_t* counters)
{
    // the device node buffer is 16-byte aligned: copy into one that is, so that every window starts where the kernel's would
    std::vector<uint8_t> store(buf_len + 16);
    uint8_t* abuf = (uint8_t*)(((uintptr_t)store.data() + 15) & ~(uintptr_t)15);
    memcpy(abuf, buf, buf_len);
    const Batch B{abuf, buf_len, node_start, node_len, proof_first, keys32, roots32, n_roots};
    memset(g_smem, GUARD_BYTE, sizeof g_smem);
    memset(g_smem + SLOT_S, STALE, SLOT);
    uint64_t bad = 0;
    for (uint64_t p = 0; p < n_proofs; ++p) {
        uint32_t f = 0, vl2 = 0;
        uint64_t vo2 = 0;
        g_count = counters;
        int r = lane(B, p, true, val_off[p], val_len[p], f);
        g_count = nullptr;
        const int r2 = lane(B, p, false, vo2, vl2, f);
        if (r != ST_PRESENT) { val_off[p] = 0; val_len[p] = 0; }
        if (r2 != ST_PRESENT) { vo2 = 0; vl2 = 0; }
        if (r != r2 || val_off[p] != vo2 || val_len[p] != vl2) f |= F_ALIGN_DIFF;
        status[p] = (uint8_t)r;
        fail[p] = (uint8_t)f;
        bad += f != 0;
    }
    fprintf(stderr, "fused lane: tail_ok true %llu false %llu, masked fallbacks %llu, multi-window nodes %llu, aligned absorbs %llu, "
                    "slot walks %llu, global walks %llu, nodes %llu\n",
            (unsigned long long)counters[C_TAIL_OK_TRUE], (unsigned long long)counters[C_TAIL_OK_FALSE], (unsigned long long)counters[C_MASKED],
            (unsigned long long)counters[C_MULTI_WINDOW], (unsigned long long)counters[C_ALIGNED_ABSORB], (unsigned long long)counters[C_SLOT_WALKS],
            (unsigned long long)counters[C_GLOBAL_WALKS], (unsigned long long)counters[C_NODES]);
    return bad;
}
