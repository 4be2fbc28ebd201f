// walk_one.cuh -- the proof walk of ONE key, as the per-thread device function the kernels in walk_kernel.cu call.
//
// Kept in a header of its own so that the same source can also be compiled as HOST code by the test harness
// (tests/hostcheck/walk_host.cpp defines the CUDA qualifiers and the three intrinsics away) and fuzzed against the oracle
// on a machine without a GPU.  Rules R1-R4: DESIGN.md "Proof walk"; CPU statement: oracle/verify.c.
#pragma once
#include <stdint.h>

namespace phant {
namespace {

enum { ST_REJECT = 0, ST_PRESENT = 1, ST_ABSENT = 2, ST_MISSING = 3 };

// Bag mode: the witness is an unordered set of nodes; a hash reference is resolved through an open-addressing table
// keyed by the first 8 digest bytes (full 32-byte compare on hit).  table[slot] = node index or EMPTY.
constexpr uint32_t BAG_EMPTY = 0xffffffffu;
struct Bag {
    const uint32_t* table;
    uint32_t mask; // capacity - 1 (power of two)
};

struct Item {
    uint32_t is_list;
    uint32_t pay_off; // from the item's first byte
    uint32_t pay_len;
};

// 32 bytes at a 16-byte aligned address (digests, roots) as two 128-bit loads
__device__ __forceinline__ void load32_aligned(const uint8_t* a, uint32_t (&e)[8])
{
    const uint4 lo = __ldg(reinterpret_cast<const uint4*>(a)), hi = __ldg(reinterpret_cast<const uint4*>(a) + 1);
    e[0] = lo.x; e[1] = lo.y; e[2] = lo.z; e[3] = lo.w;
    e[4] = hi.x; e[5] = hi.y; e[6] = hi.z; e[7] = hi.w;
}
__device__ __forceinline__ bool eq32_aligned(const uint8_t* a, const uint32_t (&e)[8])
{
    uint32_t d[8];
    load32_aligned(a, d);
    uint32_t diff = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) diff |= d[i] ^ e[i];
    return diff == 0;
}
// 32 bytes at any address (a hash inside a node): the 48-byte aligned window around them as THREE 128-bit loads, then a word
// select and one funnel shift per word.  One proof per lane means every load instruction touches 32 different lines, so the
// walk is bound by the NUMBER of load instructions, not by bytes: three wide loads instead of nine narrow ones.  The window
// may reach 15 bytes before `a` and 16 bytes past `a + 32`; both stay inside the node buffer (16-byte aligned base, 16 bytes
// of slack behind the last node: include/phant_gpu.h).
__device__ __forceinline__ void load32(const uint8_t* a, uint32_t (&e)[8])
{
    const uintptr_t p = (uintptr_t)a;
    const uint4* q = reinterpret_cast<const uint4*>(p & ~(uintptr_t)15);
    const uint4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2);
    const uint32_t v[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
    const uint32_t w0 = (uint32_t)(p & 15) >> 2, sh = (uint32_t)(p & 3) * 8;
    uint32_t u[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) { // u[i] = v[w0 + i], w0 in 0..3, without dynamic register indexing
        const uint32_t a01 = (w0 & 1) ? v[i + 1] : v[i];
        const uint32_t a23 = (w0 & 1) ? v[i + 3 < 12 ? i + 3 : 11] : v[i + 2 < 12 ? i + 2 : 11];
        u[i] = (w0 & 2) ? a23 : a01;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) e[i] = __funnelshift_r(u[i], u[i + 1], sh);
}
__device__ __forceinline__ bool eq32_const(const uint8_t* a, const uint32_t (&e)[8])
{
    uint32_t diff = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t w = (uint32_t)a[4 * i] | ((uint32_t)a[4 * i + 1] << 8) | ((uint32_t)a[4 * i + 2] << 16) | ((uint32_t)a[4 * i + 3] << 24);
        diff |= w ^ e[i];
    }
    return diff == 0;
}

__constant__ uint8_t EMPTY_ROOT[32] = {0x56, 0xe8, 0x1f, 0x17, 0x1b, 0xcc, 0x55, 0xa6, 0xff, 0x83, 0x45,
                                       0xe6, 0x92, 0xc0, 0xf8, 0x6e, 0x5b, 0x48, 0xe0, 0x1b, 0x99, 0x6c,
                                       0xad, 0xc0, 0x01, 0x62, 0x2f, 0xb5, 0xe3, 0x63, 0xb4, 0x21};

__device__ __forceinline__ uint32_t bag_slot(const uint32_t (&e)[8], uint32_t mask)
{
    uint64_t h = ((uint64_t)e[1] << 32) | e[0];
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32; // the digest is uniform already; this only decorrelates from `mask`
    return (uint32_t)h & mask;
}
__device__ uint32_t bag_find(const Bag& bag, const uint8_t* __restrict__ digests, const uint32_t (&expect)[8])
{
    uint32_t s = bag_slot(expect, bag.mask);
    for (;;) {
        const uint32_t idx = bag.table[s];
        if (idx == BAG_EMPTY) return BAG_EMPTY;
        if (eq32_aligned(digests + 32ull * idx, expect)) return idx;
        s = (s + 1) & bag.mask;
    }
}

// ---- the node bytes a walk step reads: a node of the caller's buffer, or the same node staged in a lane's shared-memory slot.
// Offsets are local to the node; `at(0)` is its first byte.  `load32(o)` reads the 32 bytes at local offset o (inside the
// node); `tail_ok(e)` says whether `load32_tail(e)`, the 32 bytes ENDING at local offset e, may be read (they may start before
// the node: the leaf-path compare masks them off).  `abs(o)` is the offset in the caller's node buffer (the value slice returned).
struct GlobalBytes {
    const uint8_t* __restrict__ nodes;
    uint64_t base; // node_off of this node
    __device__ __forceinline__ uint32_t at(uint32_t o) const { return nodes[base + o]; }
    __device__ __forceinline__ void load32(uint32_t o, uint32_t (&e)[8]) const { ::phant::load32(nodes + base + o, e); }
    __device__ __forceinline__ bool tail_ok(uint32_t e) const { return base + e >= 48; } // the 48-byte window stays in the buffer
    __device__ __forceinline__ void load32_tail(uint32_t e, uint32_t (&t)[8]) const { ::phant::load32(nodes + (base + e - 32), t); }
    __device__ __forceinline__ uint64_t abs(uint32_t o) const { return base + o; }
};
// `p` = the node's first byte in the slot (a generic pointer into shared memory), `skew` = bytes of the slot in front of it
// (the slot is 16-byte aligned, the node starts at its 16-byte aligned window + skew).  32 bytes = 9 aligned 32-bit words and
// one funnel shift per word, all inside the slot: a 32-byte read ending at the node's end reaches at most 4 bytes past it.
struct SlotBytes {
    const uint8_t* p;
    uint32_t skew;
    uint64_t base;
    __device__ __forceinline__ uint32_t at(uint32_t o) const { return p[o]; }
    __device__ __forceinline__ void load32(uint32_t o, uint32_t (&e)[8]) const { load32_at(p + o, e); }
    __device__ __forceinline__ void load32_tail(uint32_t e, uint32_t (&t)[8]) const { load32_at(p + e - 32, t); }
    __device__ __forceinline__ static void load32_at(const uint8_t* q, uint32_t (&e)[8])
    {
        const uintptr_t a = (uintptr_t)q;
        const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)(a & 3) * 8;
        uint32_t u[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) u[i] = w[i];
#pragma unroll
        for (int i = 0; i < 8; ++i) e[i] = __funnelshift_r(u[i], u[i + 1], sh);
    }
    __device__ __forceinline__ bool tail_ok(uint32_t e) const { return skew + e >= 32; } // starts inside the slot
    __device__ __forceinline__ uint64_t abs(uint32_t o) const { return base + o; }
};

// Strict decode of one RLP item at local offset `at` of a node (avail bytes).  Returns its total size, 0 if malformed.
template <class Bytes>
__device__ __forceinline__ uint32_t rlp_item_at(const Bytes& nb, uint32_t at, uint32_t avail, Item& it)
{
    if (avail == 0) return 0;
    const uint32_t b = nb.at(at);
    if (b < 0x80) { it.is_list = 0; it.pay_off = 0; it.pay_len = 1; return 1; }
    const uint32_t is_list = b >= 0xc0;
    const uint32_t base_short = is_list ? 0xc0 : 0x80, base_long = is_list ? 0xf7 : 0xb7;
    it.is_list = is_list;
    if (b <= base_long) {
        const uint32_t len = b - base_short;
        if (1 + len > avail) return 0;
        if (!is_list && len == 1 && nb.at(at + 1) < 0x80) return 0; // single byte must encode as itself
        it.pay_off = 1; it.pay_len = len;
        return 1 + len;
    }
    const uint32_t n = b - base_long;
    if (n > 4 || 1 + n > avail) return 0;
    if (nb.at(at + 1) == 0) return 0;
    uint64_t len = 0;
    for (uint32_t i = 0; i < n; ++i) len = (len << 8) | nb.at(at + 1 + i);
    if (len <= 55) return 0;
    if (1 + n + len > avail) return 0;
    it.pay_off = 1 + n; it.pay_len = (uint32_t)len;
    return (uint32_t)(1 + n + len);
}

// nibble q of the key, q < 64
__device__ __forceinline__ uint32_t key_nibble(const uint32_t (&kw)[8], uint32_t q)
{
    const uint32_t wi = q >> 3;
    const uint32_t a01 = (wi & 1) ? kw[1] : kw[0], a23 = (wi & 1) ? kw[3] : kw[2], a45 = (wi & 1) ? kw[5] : kw[4], a67 = (wi & 1) ? kw[7] : kw[6];
    const uint32_t lo4 = (wi & 2) ? a23 : a01, hi4 = (wi & 2) ? a67 : a45;
    const uint32_t w = (wi & 4) ? hi4 : lo4;
    const uint32_t byte = (w >> (8 * ((q >> 1) & 3))) & 0xffu;
    return (q & 1) ? (byte & 15u) : (byte >> 4);
}

// One step of the walk: the node whose digest matched `expect` (rule R1, checked by the caller) is interpreted for the key.
// `len` = node size, `sm` = its summary (node_summary.cuh; 0 = parse it), `last_node` = it is the chain's last node, `pos` =
// key nibbles consumed so far.  Returns ST_NEXT with `expect` = the hash reference the next node must match, or a terminal
// status (with voff / vlen set for ST_PRESENT).  Embedded children (< 32 bytes) are walked in place, inside this step.
enum { ST_NEXT = 4 };
template <class Bytes>
__device__ __forceinline__ int walk_node(const Bytes& nb, uint32_t len, uint32_t sm, bool last_node, const uint32_t (&kw)[8], uint32_t& pos,
                                         uint32_t (&expect)[8], uint64_t& voff, uint32_t& vlen)
{
    // fast path: the node is a simple branch (canonical 17-item list, children empty or 32-byte hashes, empty value) and the
    // summary holds the child mask: no parse, one 32-byte fetch
    if ((sm & 3u) == 1u && pos < 64) {
        const uint32_t nibble = key_nibble(kw, pos);
        ++pos;
        const uint32_t mask = sm >> 8;
        if (!((mask >> nibble) & 1u)) return last_node ? ST_ABSENT : ST_REJECT; // empty slot (R3)
        const uint32_t before = __popc(mask & ((1u << nibble) - 1u));
        nb.load32(((sm >> 2) & 7u) + 33u * before + (nibble - before) + 1u, expect);
        return ST_NEXT;
    }
    uint32_t cur = 0, cur_len = len; // the item being interpreted: the node, then embedded children
    for (;;) {
        Item top;
        const uint32_t tot = rlp_item_at(nb, cur, cur_len, top);
        if (tot == 0 || !top.is_list || tot != cur_len) return ST_REJECT; // R2
        const uint32_t pay = cur + top.pay_off;
        const uint32_t pl = top.pay_len;

        // one pass over the items: remember item 0, item 1, the item at the key's nibble and item 16
        const uint32_t want = pos < 64 ? key_nibble(kw, pos) : 16u;
        Item it0{}, it1{}, itw{}, it16{};
        uint32_t off0 = 0, off1 = 0, offw = 0, off16 = 0;
        uint32_t cnt = 0, o = 0;
        while (o < pl) {
            if (cnt == 17) return ST_REJECT;
            Item it;
            const uint32_t t = rlp_item_at(nb, pay + o, pl - o, it);
            if (t == 0) return ST_REJECT;
            if (cnt == 0) { it0 = it; off0 = o; }
            if (cnt == 1) { it1 = it; off1 = o; }
            if (cnt == want) { itw = it; offw = o; }
            if (cnt == 16) { it16 = it; off16 = o; }
            o += t;
            ++cnt;
        }
        if (cnt != 17 && cnt != 2) return ST_REJECT;

        Item child;
        uint32_t child_off;
        if (cnt == 17) {
            if (pos == 64) { // key exhausted: the branch value decides
                if (it16.is_list || !last_node) return ST_REJECT;
                if (it16.pay_len == 0) return ST_ABSENT;
                voff = nb.abs(pay + off16 + it16.pay_off);
                vlen = it16.pay_len;
                return ST_PRESENT;
            }
            child = itw; child_off = offw;
            ++pos;
        } else {
            if (it0.is_list || it0.pay_len == 0) return ST_REJECT;
            const uint32_t hp = pay + off0 + it0.pay_off;
            const uint32_t h0 = nb.at(hp);
            const uint32_t flag = h0 >> 4;
            if (flag > 3) return ST_REJECT;
            if (!(flag & 1) && (h0 & 15)) return ST_REJECT;
            const uint32_t plen = 2 * (it0.pay_len - 1) + (flag & 1);
            if (plen > 64) return ST_REJECT;
            bool match = 64 - pos >= plen;
            if ((flag & 2) && pos + plen != 64) match = false; // a leaf only proves presence when its path ends the key: nothing to compare otherwise
            else if (match && (flag & 2) && plen >= 2 && nb.tail_ok(hp + it0.pay_len)) {
                // leaf whose path ends exactly at the key's end: its last plen/2 bytes must equal the key's last plen/2 bytes (and,
                // for an odd path, the low nibble of hp[0] the nibble before them) -- one wide load instead of a byte loop
                uint32_t tail[8];
                nb.load32_tail(hp + it0.pay_len, tail);
                const uint32_t nbytes = plen >> 1; // whole bytes compared: key bytes [32 - nbytes, 32)
                uint32_t diff = 0;
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    const int first = 32 - (int)nbytes - 4 * w; // first compared byte inside word w (<= 0: whole word, >= 4: none)
                    const uint32_t m = first <= 0 ? 0xffffffffu : (first >= 4 ? 0u : 0xffffffffu << (8 * first));
                    diff |= (tail[w] ^ kw[w]) & m;
                }
                if ((flag & 1) && (h0 & 15u) != key_nibble(kw, pos)) diff = 1;
                match = diff == 0;
            } else if (match) {
                // path nibble j: odd flag -> nibble 0 is hp[0]&15, then bytes; even -> bytes from hp[1]
                for (uint32_t j = 0; j < plen; ++j) {
                    const uint32_t q = j + 2 - (flag & 1); // nibble index inside hp (2 nibbles per byte)
                    const uint32_t hb = nb.at(hp + (q >> 1));
                    const uint32_t pn = (q & 1) ? (hb & 15u) : (hb >> 4);
                    if (pn != key_nibble(kw, pos + j)) { match = false; break; }
                }
            }
            if (flag & 2) { // leaf
                if (it1.is_list || !last_node) return ST_REJECT;
                if (match && pos + plen == 64) {
                    voff = nb.abs(pay + off1 + it1.pay_off);
                    vlen = it1.pay_len;
                    return ST_PRESENT;
                }
                return ST_ABSENT;
            }
            if (plen == 0) return ST_REJECT;
            if (!match) return last_node ? ST_ABSENT : ST_REJECT;
            pos += plen;
            child = it1; child_off = off1;
        }
        if (child.is_list) { // embedded child (< 32 bytes), walked in place
            const uint32_t tot_child = child.pay_off + child.pay_len;
            if (tot_child >= 32) return ST_REJECT;
            cur = pay + child_off;
            cur_len = tot_child;
            continue;
        }
        if (child.pay_len == 0) {
            if (cnt == 2) return ST_REJECT;
            return last_node ? ST_ABSENT : ST_REJECT;
        }
        if (child.pay_len != 32) return ST_REJECT;
        nb.load32(pay + child_off + child.pay_off, expect);
        return ST_NEXT;
    }
}

// The walk of one key over a chain (or, BAG, over the node set), from the digests the hash kernel left: walk_node per node.
template <bool BAG>
__device__ int walk_one(const uint8_t* __restrict__ nodes, const uint64_t* __restrict__ node_off,
                        const uint64_t* __restrict__ node_index, const Bag bag, uint64_t first,
                        uint64_t last, const uint8_t* __restrict__ key, const uint8_t* __restrict__ root,
                        const uint8_t* __restrict__ digests, const uint32_t* __restrict__ summary, uint64_t& voff, uint32_t& vlen)
{
    voff = 0; vlen = 0;
    uint32_t expect[8];
    load32_aligned(root, expect);
    // the key lives in registers (two 128-bit loads) instead of one byte load per trie level
    uint32_t kw[8];
    load32_aligned(key, kw);
    if (BAG) { // no chain: first/last only feed the "is this the last node" tests, which always pass
        first = 0;
        last = 1;
        if (eq32_const(EMPTY_ROOT, expect)) return ST_ABSENT;
    } else if (first == last) return eq32_const(EMPTY_ROOT, expect) ? ST_ABSENT : ST_REJECT;

    uint32_t pos = 0; // nibbles of the key consumed
    uint64_t i = first;
    for (;;) {
        uint64_t ni;
        if (BAG) {
            const uint32_t f = bag_find(bag, digests, expect);
            if (f == BAG_EMPTY) return ST_MISSING; // the witness does not contain the node this reference names
            ni = f;
            i = last - 1; // so that ++i below leaves i == last: every terminal test sees "last node"
        } else {
            if (i == last) return ST_REJECT; // R3: a hash reference needs a node
            ni = node_index ? node_index[i] : i; // deduplicated witness: the chain holds node indices
        }
        const uint64_t o = node_off[ni];
        const uint64_t l = node_off[ni + 1] - o;
        if (l > 0xffffffffull) return ST_REJECT;
        if (!BAG && !eq32_aligned(digests + 32 * ni, expect)) return ST_REJECT; // R1 (bag: the lookup compared it)
        const uint32_t sm = summary ? summary[ni] : 0;
        ++i;
        const int st = walk_node(GlobalBytes{nodes, o}, (uint32_t)l, sm, i == last, kw, pos, expect, voff, vlen);
        if (st != ST_NEXT) return st;
    }
}

} // namespace
} // namespace phant
