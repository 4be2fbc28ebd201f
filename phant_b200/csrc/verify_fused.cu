// verify_fused.cu -- proof verification of a CSR chain in ONE pass: each lane owns one proof and hashes and walks its nodes
// in turn (entry point V of include/phant_gpu.h when the witness is a plain chain, DESIGN.md section 4).
//
// The hash side is keccak256_staged_kernel (keccak_kernels.cu) unchanged: one persistent CTA of 12 warps per SM, a 624-byte
// shared-memory slot per lane filled by the bulk-copy engine behind one mbarrier per warp, the last block padded in the slot,
// the digest-only last round.  What changes is the unit of work: a lane takes proof order[idx], and when a node's last block
// is absorbed, the node is still in the slot -- its digest is compared with the reference its parent named (the root for the
// first node), and the walk step (walk_one.cuh, walk_node) reads the node's bytes from the slot to find the next reference.
// So the digests, the node summaries and the walk's re-read of every node never reach DRAM.
//
// A node longer than one window streams through the slot for hashing as in the hash kernel and is then walked from global
// memory (GlobalBytes): rare, and the same code.  A lane with a verdict stops requesting copies but keeps arriving on the
// warp's mbarrier until the whole warp is done.
#include "common.cuh"
#include "keccak_f1600.cuh"
#include "node_summary.cuh"
#include "peer_sync.cuh"
#include "stage.cuh"
#include "walk_one.cuh"

namespace phant {
namespace {

template <int UNROLL, int BLOCKS, int WARPS, bool PEER>
__global__ void __launch_bounds__(WARPS * 32, 1)
verify_fused_kernel(uint64_t n_proofs, const uint8_t* __restrict__ nodes, const uint64_t* __restrict__ node_off,
                    const uint64_t* __restrict__ proof_first, const uint32_t* __restrict__ order, const uint8_t* __restrict__ keys32,
                    const uint8_t* __restrict__ roots32, uint64_t n_roots, uint64_t* __restrict__ bitmap, uint8_t* __restrict__ status,
                    uint64_t* __restrict__ val_off, uint32_t* __restrict__ val_len, unsigned long long* __restrict__ perms, const PeerOut peer)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar = smem_u32(smem) + 8 * warp;
    constexpr int SLOT = stage_slot(BLOCKS), WINDOW = stage_window(BLOCKS);
    uint8_t* slot = smem + 128 + (warp * 32 + lane) * SLOT;
    const uint32_t slot_s = smem_u32(slot);
    if (lane == 0) mbar_init(bar, 32);
    fence_proxy_async();
    if (PEER) { // nobody may write into a remote buffer before its owner has copied the previous contents out
        if (threadIdx.x == 0 && peer.wait_done) wait_flags(peer.done, peer.world, peer.wait_done, peer.err);
    }
    __syncthreads();
    uint32_t parity = 0;
    uint64_t my_perms = 0;

    const uint64_t n_tiles = (n_proofs + 31) / 32;
    for (uint64_t tile = (uint64_t)blockIdx.x * WARPS + warp; tile < n_tiles; tile += (uint64_t)gridDim.x * WARPS) {
        const uint64_t idx = tile * 32 + lane;
        const bool active = idx < n_proofs;
        uint64_t p = 0, j = 0, jl = 0, nbeg = 0, cur = 0, end = 0, nxt = 0, voff = 0; // nxt: end of node j+1, loaded ahead
        uint32_t vlen = 0, pos = 0;
        uint32_t expect[8], kw[8];
        int verdict = ST_REJECT;
        bool done = !active;
        if (active) {
            p = order ? order[idx] : idx;
            j = proof_first[p];
            jl = proof_first[p + 1];
            load32_aligned(roots32 + (n_roots == 1 ? 0 : 32 * p), expect);
            load32_aligned(keys32 + 32 * p, kw);
            if (j == jl) { // no node: only the empty trie proves anything
                verdict = eq32_const(EMPTY_ROOT, expect) ? ST_ABSENT : ST_REJECT;
                done = true;
            } else {
                nbeg = cur = node_off[j];
                end = node_off[j + 1];
                if (j + 1 < jl) nxt = node_off[j + 2];
                if (end - nbeg > 0xffffffffull) done = true; // REJECT, as walk_one
            }
        }
        uint64_t st[25];
#pragma unroll
        for (int i = 0; i < 25; ++i) st[i] = 0;
        bool first_trip = true;

        while (!__all_sync(0xffffffffu, done)) {
            // -- ask the copy engine for this lane's next <= BLOCKS blocks (16-byte aligned window) --
            const uint64_t need = done ? 0 : end - cur;
            const uint64_t a0 = cur & ~(uint64_t)15;
            uint32_t cs = 0;
            if (need) {
                const uint64_t span = ((end - a0) + 15) & ~(uint64_t)15;
                cs = span < WINDOW ? (uint32_t)span : WINDOW;
                fence_proxy_async(); // my earlier reads and writes of the slot are ordered before the engine's writes
                mbar_arrive_expect_tx(bar, cs);
                bulk_g2s(slot_s, nodes + a0, cs, bar);
            } else {
                mbar_arrive(bar);
            }
            mbar_wait(bar, parity);
            parity ^= 1;
            // every lane's node starts at a multiple of 4 bytes (C2: always): absorb without the byte-skew funnel shifts
            const bool aligned = __all_sync(0xffffffffu, done || (cur & 3) == 0);
            if (done) continue;
            const uint32_t skew = (uint32_t)(cur - a0);
            const uint64_t in_slot = cs - skew; // node bytes present in the slot (cs == 0 -> need == 0: an empty node)
            const uint64_t avail = need < in_slot ? need : in_slot;
            const uint32_t nfull = (uint32_t)(avail / KECCAK_RATE);
            uint32_t sa = slot_s + skew;
            for (uint32_t b = 0; b < nfull; ++b) {
                absorb_full_smem<UNROLL>(st, sa, aligned);
                sa += KECCAK_RATE;
            }
            my_perms += nfull;
            if (avail != need) { // the node goes on past this window
                cur += (uint64_t)nfull * KECCAK_RATE;
                first_trip = false;
                continue;
            }
            // the node ends inside this window: pad (behind the node's bytes, which stay intact) and finish
            absorb_final_smem<UNROLL>(st, sa, (uint32_t)(avail - (uint64_t)nfull * KECCAK_RATE), slot_s + SLOT - sa, aligned);
            ++my_perms;
            uint32_t diff = 0; // R1: the node's digest is the reference its parent named
#pragma unroll
            for (int w = 0; w < 4; ++w) diff |= ((uint32_t)st[w] ^ expect[2 * w]) | ((uint32_t)(st[w] >> 32) ^ expect[2 * w + 1]);
            const uint32_t len = (uint32_t)(end - nbeg);
            int r = ST_REJECT;
            ++j;
            if (diff == 0) {
                if (first_trip) { // the whole node is in the slot
                    const uint8_t* np = slot + skew;
                    r = walk_node(SlotBytes{np, skew, nbeg}, len, summarize_node(np, len), j == jl, kw, pos, expect, voff, vlen);
                } else {
                    r = walk_node(GlobalBytes{nodes, nbeg}, len, 0u, j == jl, kw, pos, expect, voff, vlen);
                }
                if (r == ST_NEXT && j == jl) r = ST_REJECT; // R3: a hash reference needs a node
            }
            if (r != ST_NEXT) {
                verdict = r;
                done = true;
                continue;
            }
            // next node of the chain
            nbeg = cur = end;
            end = nxt;
            if (j + 1 < jl) nxt = node_off[j + 2]; // consumed when this node is done: the load is off the critical path
            if (end - nbeg > 0xffffffffull) { done = true; continue; } // REJECT, as walk_one
#pragma unroll
            for (int i = 0; i < 25; ++i) st[i] = 0;
            first_trip = true;
        }

        if (active) {
            if (status) status[p] = (uint8_t)verdict;
            if (val_off) val_off[p] = verdict == ST_PRESENT ? voff : 0;
            if (val_len) val_len[p] = verdict == ST_PRESENT ? vlen : 0;
        }
        const bool acc = active && (verdict == ST_PRESENT || verdict == ST_ABSENT); // missing node (3) is not an accept
        const uint32_t word = __ballot_sync(0xffffffffu, acc);
        if (PEER) { // lane r stores the warp's word into rank r's gathered bitmap (this rank's slice): one store instruction
            if (lane < peer.world) peer.dst[lane][tile] = word;
        } else if (bitmap) {
            // a warp that holds the 32 proofs of bitmap word `tile` stores the word; a regrouped warp sets its bits one by one
            if (__all_sync(0xffffffffu, !active || p == idx)) {
                if (lane == 0) reinterpret_cast<uint32_t*>(bitmap)[tile] = word;
            } else if (acc) {
                atomicOr(reinterpret_cast<uint32_t*>(bitmap) + (p >> 5), 1u << (p & 31));
            }
        }
    }
    for (int o = 16; o; o >>= 1) my_perms += __shfl_down_sync(0xffffffffu, my_perms, o);
    if (lane == 0 && my_perms) atomicAdd(perms, (unsigned long long)my_perms); // one atomic per warp
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

template <bool PEER>
cudaError_t launch_fused(cudaStream_t s, int device, uint64_t n_proofs, const uint8_t* nodes, const uint64_t* node_off,
                         const uint64_t* proof_first, const uint32_t* order, const uint8_t* keys32, const uint8_t* roots32, uint64_t n_roots,
                         uint64_t* bitmap, uint8_t* status, uint64_t* val_off, uint32_t* val_len, unsigned long long* perms, const PeerOut& peer)
{
    constexpr int BLOCKS = 4, WARPS = 12; // the hash kernel's measured best shape: 1 CTA of 12 warps per SM
    constexpr int SMEM = stage_smem(BLOCKS, WARPS);
    auto kernel = verify_fused_kernel<2, BLOCKS, WARPS, PEER>;
    static int ctas_cache[64] = {0}; // function attributes are per device
    int& ctas_per_sm = ctas_cache[(device >= 0 && device < 64) ? device : 0];
    if (!ctas_per_sm) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kernel, WARPS * 32, SMEM);
        if (e != cudaSuccess || ctas_per_sm < 1) { ctas_per_sm = 0; return e != cudaSuccess ? e : cudaErrorLaunchOutOfResources; }
    }
    const uint64_t tiles = (n_proofs + 31) / 32;
    uint64_t blocks = (tiles + WARPS - 1) / WARPS;
    const uint64_t cap = (uint64_t)keccak_num_sms(device) * ctas_per_sm; // persistent: every CTA resident, striding over the tiles
    if (blocks > cap) blocks = cap;
    kernel<<<(unsigned)blocks, WARPS * 32, SMEM, s>>>(n_proofs, nodes, node_off, proof_first, order, keys32, roots32, n_roots, bitmap, status,
                                                      val_off, val_len, perms, peer);
    return cudaGetLastError();
}

} // namespace

bool verify_fused_supported(const uint8_t* nodes) { return ((uintptr_t)nodes & 15) == 0; } // bulk copies need 16-byte alignment

cudaError_t launch_verify_fused(cudaStream_t s, int device, uint64_t n_proofs, const uint8_t* nodes, const uint64_t* node_off,
                                const uint64_t* proof_first, const uint32_t* order, const uint8_t* keys32, const uint8_t* roots32,
                                uint64_t n_roots, uint64_t* bitmap, uint8_t* status, uint64_t* val_off, uint32_t* val_len,
                                unsigned long long* perms, const PeerOut* peer)
{
    if (n_proofs == 0) return cudaSuccess;
    if (peer) {
        if (order) return cudaErrorInvalidValue; // the peer epilogue stores whole words: proofs in index order
        return launch_fused<true>(s, device, n_proofs, nodes, node_off, proof_first, nullptr, keys32, roots32, n_roots, bitmap, status, val_off,
                                  val_len, perms, *peer);
    }
    return launch_fused<false>(s, device, n_proofs, nodes, node_off, proof_first, order, keys32, roots32, n_roots, bitmap, status, val_off,
                               val_len, perms, PeerOut{});
}

} // namespace phant
