// walk_kernel.cu -- Merkle-Patricia proof walk (entry point V of include/phant_gpu.h).
//
// Fills the hook phant leaves open at src/engine_api/execution_payload.zig:177-178.  Every node of the
// batch has already been hashed by the batched Keccak kernel; this kernel walks each proof's chain:
// strict RLP decode of the branch / extension / leaf encodings that src/mpt/mpt.zig:170-281 produces,
// the child reference for the key's next nibble compared with the next node's digest (or followed in
// place when the child is embedded, mpt.zig:104,112), until a terminal decides present / absent.
// Rules R1-R4 are written out in DESIGN.md ("Proof walk"); oracle/verify.c is the CPU statement the
// tests hold this against.  One proof per thread: chains are short (<= ~12 nodes), independent, and
// the node bytes were just streamed through L2 by the hash kernel.
#include "common.cuh"

#include <stdlib.h>

#include "peer_sync.cuh"
#include "walk_one.cuh"  // Item / rlp_item_at / Bag / walk_one<BAG>

namespace phant {
namespace {

// MINB = CTAs of 128 threads the register allocator must fit per SM (8 -> <= 64 registers, 12 -> <= 40, 16 -> <= 32): the
// walk is latency-bound (dependent loads per node), so residency is traded against spills; measured, see launch_walk
template <bool BAG, int MINB, bool PEER = false>
__global__ void __launch_bounds__(128, MINB)
walk_kernel(const Bag bag, uint64_t n_proofs, const uint8_t* __restrict__ nodes, const uint64_t* __restrict__ node_off,
            const uint64_t* __restrict__ node_index, const uint64_t* __restrict__ proof_first, const uint8_t* __restrict__ keys32,
            const uint8_t* __restrict__ roots32, uint64_t n_roots, const uint8_t* __restrict__ digests,
            const uint32_t* __restrict__ summary, uint64_t* __restrict__ bitmap, uint8_t* __restrict__ status, uint64_t* __restrict__ val_off,
            uint32_t* __restrict__ val_len, const PeerOut peer)
{
    if (PEER) { // nobody may write into a remote buffer before its owner has copied the previous contents out
        if (threadIdx.x == 0 && peer.wait_done) wait_flags(peer.done, peer.world, peer.wait_done, peer.err);
        __syncthreads();
    }
    const uint64_t n_padded = (n_proofs + 31) & ~(uint64_t)31; // whole warps, so the ballot is complete
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_padded; p += (uint64_t)gridDim.x * blockDim.x) {
        int st = ST_REJECT;
        if (p < n_proofs) {
            uint64_t vo;
            uint32_t vl;
            st = walk_one<BAG>(nodes, node_off, node_index, bag, BAG ? 0 : proof_first[p], BAG ? 0 : proof_first[p + 1], keys32 + 32 * p,
                          roots32 + (n_roots == 1 ? 0 : 32 * p), digests, summary, vo, vl);
            if (status) status[p] = (uint8_t)st;
            if (val_off) val_off[p] = vo;
            if (val_len) val_len[p] = vl;
        }
        const uint32_t word = __ballot_sync(0xffffffffu, st == ST_PRESENT || st == ST_ABSENT); // missing node (3) is not an accept
        if (PEER) { // lane r stores the warp's word into rank r's gathered bitmap (this rank's slice): one store instruction
            const uint32_t lane = threadIdx.x & 31;
            if (lane < peer.world) peer.dst[lane][p >> 5] = word;
        } else if (bitmap && (threadIdx.x & 31) == 0) reinterpret_cast<uint32_t*>(bitmap)[p >> 5] = word;
    }
    if (PEER) { // the last CTA to finish publishes the step in every rank's flag array
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t t = atomicAdd(peer.ticket, 1u);
            if (t == gridDim.x - 1) {
                __threadfence_system();
                for (uint32_t r = 0; r < peer.world; ++r) st_release_sys(peer.ready[r], peer.step);
                *peer.ticket = 0;
            }
        }
    }
}

} // namespace

// tuning knob (development): PHANT_WALK_MINB = 6 | 8 | 10 | 12 | 16; the default is the measured best
static int walk_minb()
{
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("PHANT_WALK_MINB");
        v = e ? atoi(e) : 8;
        if (v != 6 && v != 10 && v != 12 && v != 16) v = 8;
    }
    return v;
}

cudaError_t launch_walk(cudaStream_t s, int device, uint64_t n_proofs, const uint8_t* nodes, const uint64_t* node_off,
                        const uint64_t* node_index, const uint64_t* proof_first, const uint8_t* keys32, const uint8_t* roots32, uint64_t n_roots,
                        const uint8_t* digests, const uint32_t* summary, uint64_t* bitmap, uint8_t* status, uint64_t* val_off,
                        uint32_t* val_len, const PeerOut* peer)
{
    if (n_proofs == 0) return cudaSuccess;
    uint64_t blocks = (n_proofs + 127) / 128;
    const uint64_t cap = (uint64_t)keccak_num_sms(device) * 16;
    if (blocks > cap) blocks = cap;
    if (peer) {
        walk_kernel<false, 8, true><<<(unsigned)blocks, 128, 0, s>>>(Bag{nullptr, 0}, n_proofs, nodes, node_off, node_index, proof_first, keys32, roots32, n_roots,
                                                                    digests, summary, bitmap, status, val_off, val_len, *peer);
        return cudaGetLastError();
    }
#define PHANT_WALK_ARGS Bag{nullptr, 0}, n_proofs, nodes, node_off, node_index, proof_first, keys32, roots32, n_roots, digests, summary, bitmap, status, val_off, val_len, PeerOut{}
    switch (walk_minb()) {
    case 6: walk_kernel<false, 6><<<(unsigned)blocks, 128, 0, s>>>(PHANT_WALK_ARGS); break;
    case 10: walk_kernel<false, 10><<<(unsigned)blocks, 128, 0, s>>>(PHANT_WALK_ARGS); break;
    case 12: walk_kernel<false, 12><<<(unsigned)blocks, 128, 0, s>>>(PHANT_WALK_ARGS); break;
    case 16: walk_kernel<false, 16><<<(unsigned)blocks, 128, 0, s>>>(PHANT_WALK_ARGS); break;
    default: walk_kernel<false, 8><<<(unsigned)blocks, 128, 0, s>>>(PHANT_WALK_ARGS); break;
    }
#undef PHANT_WALK_ARGS
    return cudaGetLastError();
}

// ---- bag mode: table build + walk ----
namespace {
__global__ void bag_insert_kernel(const uint8_t* __restrict__ digests, uint64_t n_nodes, uint32_t* __restrict__ table, uint32_t mask)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t e[8];
        load32_aligned(digests + 32 * i, e);
        uint32_t s = bag_slot(e, mask);
        for (;;) {
            const uint32_t prev = atomicCAS(&table[s], BAG_EMPTY, (uint32_t)i);
            if (prev == BAG_EMPTY) break;
            if (eq32_aligned(digests + 32ull * prev, e)) break; // the same node twice in the bag: one entry is enough
            s = (s + 1) & mask;
        }
    }
}
} // namespace

cudaError_t launch_bag_build(cudaStream_t s, int device, const uint8_t* digests, uint64_t n_nodes, uint32_t* table, uint32_t capacity)
{
    cudaError_t e = cudaMemsetAsync(table, 0xff, 4ull * capacity, s);
    if (e != cudaSuccess || n_nodes == 0) return e;
    uint64_t blocks = (n_nodes + 255) / 256;
    const uint64_t cap = (uint64_t)keccak_num_sms(device) * 8;
    if (blocks > cap) blocks = cap;
    bag_insert_kernel<<<(unsigned)blocks, 256, 0, s>>>(digests, n_nodes, table, capacity - 1);
    return cudaGetLastError();
}

cudaError_t launch_walk_bag(cudaStream_t s, int device, uint64_t n_keys, const uint8_t* nodes, const uint64_t* node_off, const uint8_t* keys32,
                            const uint8_t* roots32, uint64_t n_roots, const uint8_t* digests, const uint32_t* summary, const uint32_t* table,
                            uint32_t capacity, uint64_t* bitmap, uint8_t* status, uint64_t* val_off, uint32_t* val_len)
{
    if (n_keys == 0) return cudaSuccess;
    uint64_t blocks = (n_keys + 127) / 128;
    const uint64_t cap = (uint64_t)keccak_num_sms(device) * 16;
    if (blocks > cap) blocks = cap;
    walk_kernel<true, 8><<<(unsigned)blocks, 128, 0, s>>>(Bag{table, capacity - 1}, n_keys, nodes, node_off, nullptr, nullptr, keys32, roots32, n_roots,
                                                      digests, summary, bitmap, status, val_off, val_len, PeerOut{});
    return cudaGetLastError();
}

// ---- peer transport, receiving side: wait until every rank's words of this step have landed in MY buffer, copy the gathered
// bitmap to the caller's buffer, tell every rank that this buffer of mine may be overwritten again ----
namespace {
__global__ void __launch_bounds__(256)
peer_collect_kernel(const unsigned long long* __restrict__ ready /*my ready[buffer][0..world)*/, uint32_t world, unsigned long long step,
                    const unsigned long long* __restrict__ src, unsigned long long* __restrict__ dst, uint64_t n_words,
                    const PeerOut sig /* ready[] = the done flags in every rank */)
{
    if (threadIdx.x == 0) wait_flags(ready, world, step, sig.err);
    __syncthreads();
    // the words were written by other GPUs: read them around the L1 (ld.cv)
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = __ldcv(src + i);
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t t = atomicAdd(sig.ticket, 1u);
        if (t == gridDim.x - 1) {
            __threadfence_system();
            for (uint32_t r = 0; r < world; ++r) st_release_sys(sig.ready[r], step);
            *sig.ticket = 0;
        }
    }
}
} // namespace

cudaError_t launch_peer_collect(cudaStream_t s, const unsigned long long* ready, uint32_t world, unsigned long long step, const void* src, void* dst,
                                uint64_t bytes, const PeerOut& sig)
{
    const uint64_t n_words = bytes / 8;
    uint64_t blocks = (n_words + 255) / 256;
    if (blocks > 64) blocks = 64;
    if (blocks == 0) blocks = 1;
    peer_collect_kernel<<<(unsigned)blocks, 256, 0, s>>>(ready, world, step, (const unsigned long long*)src, (unsigned long long*)dst, n_words, sig);
    return cudaGetLastError();
}

} // namespace phant
