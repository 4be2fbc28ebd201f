// keccak_kernels.cu -- batched Keccak-256 over CSR messages (entry point K of include/phant_gpu.h).
//
// Replaces N calls of hasher.keccak256 (reference src/crypto/hasher.zig:4-8; per-node use in
// src/mpt/mpt.zig:203-209,241-247,273-280) by one launch.  Three kernels, same results:
//
//   staged  (default)  one sponge per thread, state in registers; each lane's message bytes are brought
//                      from HBM into its private shared-memory slot by the bulk-copy engine
//                      (cp.async.bulk -> SASS UBLKCP, completion on a per-warp mbarrier), 4 rate blocks
//                      per trip, and read back as aligned 32-bit words (one funnel shift fixes the byte
//                      skew).  No thread ever issues a global load for message bytes, so the strided
//                      (one-message-per-lane) access pattern never reaches the LSU as 32 uncoalesced
//                      sectors.  One CTA of 12 warps per SM (227 KB of slots).
//   direct             same sponge, message words loaded straight from global memory (fallback when
//                      the buffer is not 16-byte aligned / padded; also the simplest correct kernel).
//   warp               the layout BASELINE.json's north star describes: one WARP per sponge, lane i
//                      holds state lane i (25 of 32 lanes busy), coalesced 136-byte block loads, theta /
//                      pi / chi as warp shuffles.  Kept for comparison: it issues ~7x more
//                      instructions per permutation than one-sponge-per-thread (DESIGN.md).
//
// Messages may be regrouped by number of rate blocks (`order`), so that the 32 lanes of a warp run the
// same number of permutations.
#include "common.cuh"
#include "keccak_f1600.cuh"
#include "node_summary.cuh"
#include "stage.cuh"

#include <stdlib.h>
#include <string.h>

namespace phant {

// ------------------------------------------------------------------------------------------------
// direct
// ------------------------------------------------------------------------------------------------
template <int UNROLL>
__global__ void __launch_bounds__(128)
keccak256_direct_kernel(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ off,
                        const uint32_t* __restrict__ order, uint64_t n, uint8_t* __restrict__ out,
                        uint32_t* __restrict__ summary, const uint64_t* __restrict__ len)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t m = order ? order[i] : i;
        const uint64_t beg = off[m], end = len ? beg + len[m] : off[m + 1];
        uint64_t dg[4];
        keccak256_thread<UNROLL>(msgs + beg, end - beg, dg);
        if (summary) summary[m] = (end - beg) <= 4096 ? summarize_node(msgs + beg, (uint32_t)(end - beg)) : 0;
        uint64_t* o = reinterpret_cast<uint64_t*>(out + 32 * m);
        o[0] = dg[0]; o[1] = dg[1]; o[2] = dg[2]; o[3] = dg[3];
    }
}

// ------------------------------------------------------------------------------------------------
// staged: bulk-copy engine -> per-lane shared-memory slot -> registers
// ------------------------------------------------------------------------------------------------
template <int UNROLL, int BLOCKS, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
keccak256_staged_kernel(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ off,
                        const uint32_t* __restrict__ order, uint64_t n, uint8_t* __restrict__ out,
                        uint32_t* __restrict__ summary, const uint64_t* __restrict__ len)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar = smem_u32(smem) + 8 * warp;
    constexpr int SLOT = stage_slot(BLOCKS), WINDOW = stage_window(BLOCKS);
    uint8_t* slot = smem + 128 + (warp * 32 + lane) * SLOT;
    const uint32_t slot_s = smem_u32(slot);
    if (lane == 0) mbar_init(bar, 32);
    fence_proxy_async();
    __syncthreads();
    uint32_t parity = 0;

    const uint64_t n_tiles = (n + 31) / 32;
    for (uint64_t tile = (uint64_t)blockIdx.x * WARPS + warp; tile < n_tiles; tile += (uint64_t)gridDim.x * WARPS) {
        const uint64_t idx = tile * 32 + lane;
        const bool active = idx < n;
        uint64_t m = 0, cur = 0, end = 0;
        if (active) {
            m = order ? order[idx] : idx;
            cur = off[m];
            end = len ? cur + len[m] : off[m + 1]; // `len`: messages sit in fixed-stride slots (trie builders), not back to back
        }
        uint64_t st[25];
#pragma unroll
        for (int i = 0; i < 25; ++i) st[i] = 0;
        bool done = !active;
        bool first_trip = true;

        while (!__all_sync(0xffffffffu, done)) {
            // -- ask the copy engine for this lane's next <= 4 blocks (16-byte aligned window) --
            const uint64_t need = done ? 0 : end - cur;
            const uint64_t a0 = cur & ~(uint64_t)15;
            uint32_t cs = 0;
            if (need) {
                const uint64_t span = ((end - a0) + 15) & ~(uint64_t)15;
                cs = span < WINDOW ? (uint32_t)span : WINDOW;
                fence_proxy_async(); // my earlier reads of the slot are ordered before the engine's writes
                mbar_arrive_expect_tx(bar, cs);
                bulk_g2s(slot_s, msgs + a0, cs, bar);
            } else {
                mbar_arrive(bar);
            }
            mbar_wait(bar, parity);
            parity ^= 1;
            // every lane's node starts at a multiple of 4 bytes (C2: always): absorb without the byte-skew funnel shifts
            const bool aligned = __all_sync(0xffffffffu, done || (cur & 3) == 0);
            if (!done) {
                const uint32_t skew = (uint32_t)(cur - a0);
                const uint64_t in_slot = cs - skew; // message bytes present in the slot (cs == 0 -> need == 0)
                const uint64_t avail = need < in_slot ? need : in_slot;
                if (summary && first_trip) // the whole node is in the slot iff the message ends in this window
                    summary[m] = avail == need ? summarize_node(slot + skew, (uint32_t)need) : 0;
                const uint32_t nfull = (uint32_t)(avail / KECCAK_RATE);
                uint32_t sa = slot_s + skew;
                for (uint32_t b = 0; b < nfull; ++b) {
                    absorb_full_smem<UNROLL>(st, sa, aligned);
                    sa += KECCAK_RATE;
                }
                if (avail == need) { // the message ends inside this window: pad and finish
                    absorb_final_smem<UNROLL>(st, sa, (uint32_t)(avail - (uint64_t)nfull * KECCAK_RATE), slot_s + SLOT - sa, aligned);
                    done = true;
                } else {
                    cur += (uint64_t)nfull * KECCAK_RATE;
                }
            }
            first_trip = false;
        }
        if (active) {
            uint4* o = reinterpret_cast<uint4*>(out + 32 * m);
            o[0] = make_uint4((uint32_t)st[0], (uint32_t)(st[0] >> 32), (uint32_t)st[1], (uint32_t)(st[1] >> 32));
            o[1] = make_uint4((uint32_t)st[2], (uint32_t)(st[2] >> 32), (uint32_t)st[3], (uint32_t)(st[3] >> 32));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// warp: one sponge per warp (north-star layout)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t rolv64(uint64_t x, uint32_t n) { return n ? (x << n) | (x >> (64 - n)) : x; }

__global__ void __launch_bounds__(256)
keccak256_warp_kernel(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ off, uint64_t n,
                      uint8_t* __restrict__ out, const uint64_t* __restrict__ lens)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp_id = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    // per-lane constants: lane i = x + 5y holds A[x,y]
    const uint32_t x = lane % 5, y = (lane % 25) / 5;
    constexpr uint32_t RHO[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
    uint32_t rho = 0;
#pragma unroll
    for (int i = 0; i < 25; ++i) if (lane == (uint32_t)i) rho = RHO[i];
    // pi: destination (X,Y) takes source (x', y') with X = y', Y = 2x'+3y'  =>  x' = (X + 3Y) % 5, y' = X
    const uint32_t pi_src = ((x + 3 * y) % 5) + 5 * x;
    const uint32_t col1 = (x + 1) % 5, col4 = (x + 4) % 5;
    const uint32_t row1 = 5 * y + (x + 1) % 5, row2 = 5 * y + (x + 2) % 5;
    const uint32_t FULL = 0xffffffffu;

    for (uint64_t m = warp_id; m < n; m += n_warps) {
        const uint64_t beg = off[m], end = lens ? beg + lens[m] : off[m + 1];
        uint64_t len = end - beg;
        const MsgView v = msg_view(msgs + beg);
        uint64_t s = 0; // my state lane (lanes >= 25 carry junk that nobody reads)
        uint32_t base = 0;
        bool last = false;
        while (!last) {
            // ---- absorb one block: lanes 0..16 take word k = lane ----
            uint64_t word = 0;
            if (len >= KECCAK_RATE) {
                uint64_t lo = 0;
                if (lane <= KECCAK_RATE_WORDS && (lane < KECCAK_RATE_WORDS || v.sh)) lo = v.w[base + lane];
                const uint64_t hi = __shfl_down_sync(FULL, lo, 1);
                word = lane < KECCAK_RATE_WORDS ? funnel64(lo, hi, v.sh) : 0;
                len -= KECCAK_RATE;
                base += KECCAK_RATE_WORDS;
            } else {
                const uint32_t rem = (uint32_t)len, mis = v.sh >> 3;
                // aligned words that hold message bytes of this block: [0, ceil((mis+rem)/8))
                const uint32_t n_al = (mis + rem + 7) / 8;
                uint64_t lo = (rem && lane < n_al) ? v.w[base + lane] : 0;
                const uint64_t hi = __shfl_down_sync(FULL, lo, 1);
                if (lane < KECCAK_RATE_WORDS) {
                    const int valid = (int)rem - 8 * (int)lane;
                    if (valid > 0) {
                        word = funnel64(lo, hi, v.sh);
                        if (valid < 8) word &= (1ull << (8 * valid)) - 1;
                    }
                    if (valid >= 0 && valid < 8) word ^= 1ull << (8 * valid);
                    if (lane == KECCAK_RATE_WORDS - 1) word ^= 0x8000000000000000ull;
                }
                last = true;
            }
            s ^= word;
            // ---- Keccak-f[1600] across the warp ----
#pragma unroll 1
            for (int r = 0; r < 24; ++r) {
                uint64_t c = s;                                        // theta: column parity
                c ^= __shfl_sync(FULL, s, (lane + 5) % 25);
                c ^= __shfl_sync(FULL, s, (lane + 10) % 25);
                c ^= __shfl_sync(FULL, s, (lane + 15) % 25);
                c ^= __shfl_sync(FULL, s, (lane + 20) % 25);
                const uint64_t cm = __shfl_sync(FULL, c, col4), cp = __shfl_sync(FULL, c, col1);
                s ^= cm ^ rolv64(cp, 1);
                s = rolv64(s, rho);                                    // rho
                s = __shfl_sync(FULL, s, pi_src);                      // pi
                const uint64_t b1 = __shfl_sync(FULL, s, row1), b2 = __shfl_sync(FULL, s, row2);
                s ^= ~b1 & b2;                                         // chi
                if (lane == 0) s ^= KECCAK_RC[r];                      // iota
            }
        }
        if (lane < 4) reinterpret_cast<uint64_t*>(out + 32 * m)[lane] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// regrouping by permutation count: a stable 16-bucket counting sort in two launches of our own
// ------------------------------------------------------------------------------------------------
// Lanes of a warp run in lockstep, so a warp costs max(permutations) over its 32 items: `order` lists the item indices class
// by class (heaviest first), each class in ascending index order.  An item is either one message (`first` == nullptr: class =
// 15 - min(15, permutations - 1)) or one proof of a CSR chain, items i = nodes first[i] .. first[i+1] (the fused verify kernel:
// one lane hashes and walks a whole chain; class = 15 - min(15, (permutations - 1) / 4), one class per full branch node, so
// that chains of depth 4 .. 12 fall in distinct classes).
//   launch 1  keccak_class_kernel: block b histograms its contiguous chunk of messages (hist[b][16]) and adds the
//             chunk's permutation count to the statistics; the LAST block to finish turns the matrix into global start
//             positions in place (class-major exclusive scan: start[b][c] = sum of classes < c + sum over blocks < b);
//   launch 2  keccak_regroup_kernel: block b walks the same chunk tile by tile and writes each index at
//             start[b][c] + (messages of class c seen so far in the chunk): ranks by warp match + a per-tile warp table.
// No library sort, no temporary storage beyond 64 bytes per block, deterministic output.
constexpr int CLS_THREADS = 256, CLS_WARPS = CLS_THREADS / 32;

// permutations of item i (see above)
__device__ __forceinline__ uint64_t keccak_item_perms(const uint64_t* __restrict__ off, const uint64_t* __restrict__ first, uint64_t i)
{
    if (!first) return (off[i + 1] - off[i]) / KECCAK_RATE + 1;
    uint64_t nb = 0;
    for (uint64_t j = first[i], e = first[i + 1]; j < e; ++j) nb += (off[j + 1] - off[j]) / KECCAK_RATE + 1;
    return nb;
}
__device__ __forceinline__ uint32_t keccak_class_of(uint64_t nb, bool proofs)
{
    const uint64_t c = proofs ? (nb ? (nb - 1) / 4 : 0) : nb - 1;
    return (uint32_t)(15 - (c > 15 ? 15 : c));
}

__global__ void __launch_bounds__(CLS_THREADS)
keccak_class_kernel(const uint64_t* __restrict__ off, const uint64_t* __restrict__ first, uint64_t n, uint64_t chunk,
                    uint32_t* __restrict__ hist /* gridDim.x * 16 */, uint32_t* __restrict__ ticket, unsigned long long* __restrict__ perms)
{
    __shared__ uint32_t h[16];
    __shared__ uint32_t cls_total[16];
    __shared__ bool last;
    if (threadIdx.x < 16) h[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t lo = (uint64_t)blockIdx.x * chunk, hi = lo + chunk < n ? lo + chunk : n;
    unsigned long long local = 0;
    for (uint64_t i0 = lo; i0 < hi; i0 += CLS_THREADS) { // whole warps stay converged: the tail is handled by `valid`
        const uint64_t i = i0 + threadIdx.x;
        const bool valid = i < hi;
        uint32_t c = 16;
        if (valid) {
            const uint64_t nb = keccak_item_perms(off, first, i);
            c = keccak_class_of(nb, first != nullptr);
            local += nb;
        }
        const uint32_t peers = __match_any_sync(0xffffffffu, c);
        if (valid && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&h[c], __popc(peers));
    }
    for (int o = 16; o; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local && perms) atomicAdd(perms, local); // one atomic per warp
    __syncthreads();
    if (threadIdx.x < 16) hist[16 * blockIdx.x + threadIdx.x] = h[threadIdx.x];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // ---- the last block: hist[b][c] -> start[b][c], class-major ----
    const uint32_t nb = gridDim.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (uint32_t c = warp; c < 16; c += CLS_WARPS) { // totals per class
        uint32_t t = 0;
        for (uint32_t b = lane; b < nb; b += 32) t += __ldcg(&hist[16 * b + c]);
        for (int o = 16; o; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
        if (lane == 0) cls_total[c] = t;
    }
    __syncthreads();
    for (uint32_t c = warp; c < 16; c += CLS_WARPS) {
        uint32_t carry = 0;
        for (uint32_t k = 0; k < c; ++k) carry += cls_total[k];
        for (uint32_t b0 = 0; b0 < nb; b0 += 32) {
            const uint32_t b = b0 + lane;
            const uint32_t v = b < nb ? __ldcg(&hist[16 * b + c]) : 0;
            uint32_t incl = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += up;
            }
            if (b < nb) hist[16 * b + c] = carry + incl - v;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    if (threadIdx.x == 0) *ticket = 0; // ready for the next call on this stream
}

__global__ void __launch_bounds__(CLS_THREADS)
keccak_regroup_kernel(const uint64_t* __restrict__ off, const uint64_t* __restrict__ first, uint64_t n, uint64_t chunk,
                      const uint32_t* __restrict__ start /* gridDim.x * 16 */, uint32_t* __restrict__ order)
{
    __shared__ uint32_t base[16];
    __shared__ uint32_t wcnt[CLS_WARPS][16];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 16) base[threadIdx.x] = start[16 * blockIdx.x + threadIdx.x];
    const uint64_t lo = (uint64_t)blockIdx.x * chunk, hi = lo + chunk < n ? lo + chunk : n;
    for (uint64_t i0 = lo; i0 < hi; i0 += CLS_THREADS) {
        if (threadIdx.x < CLS_WARPS * 16) (&wcnt[0][0])[threadIdx.x] = 0;
        __syncthreads(); // also orders the previous tile's reads of base[] / wcnt[] before they change
        const uint64_t i = i0 + threadIdx.x;
        const bool valid = i < hi;
        const uint32_t c = valid ? keccak_class_of(keccak_item_perms(off, first, i), first != nullptr) : 16;
        const uint32_t peers = __match_any_sync(0xffffffffu, c);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
        if (valid && rank == 0) wcnt[warp][c] = __popc(peers);
        __syncthreads();
        if (valid) {
            uint32_t pos = base[c] + rank;
            for (uint32_t w = 0; w < warp; ++w) pos += wcnt[w][c];
            order[pos] = (uint32_t)i;
        }
        __syncthreads();
        if (threadIdx.x < 16) {
            uint32_t t = 0;
#pragma unroll
            for (int w = 0; w < CLS_WARPS; ++w) t += wcnt[w][threadIdx.x];
            base[threadIdx.x] += t;
        }
        __syncthreads(); // wcnt is cleared at the top of the next tile: not before the sums above have been taken
    }
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
int keccak_num_sms(int device)
{
    static int cached[64] = {0};
    if (device < 0 || device >= 64) device = 0;
    if (!cached[device]) cudaDeviceGetAttribute(&cached[device], cudaDevAttrMultiProcessorCount, device);
    return cached[device] ? cached[device] : 148;
}

template <int BLOCKS, int WARPS>
static cudaError_t launch_staged(cudaStream_t s, int device, int sms, const uint8_t* msgs, const uint64_t* off, const uint32_t* order, uint64_t n,
                                 uint8_t* out, uint32_t* summary, const uint64_t* len)
{
    constexpr int SMEM = stage_smem(BLOCKS, WARPS);
    static int ctas_cache[64] = {0}; // function attributes are per device
    int& ctas_per_sm = ctas_cache[(device >= 0 && device < 64) ? device : 0];
    if (!ctas_per_sm) {
        cudaError_t e = cudaFuncSetAttribute(keccak256_staged_kernel<2, BLOCKS, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) return e;
        cudaFuncSetAttribute(keccak256_staged_kernel<2, BLOCKS, WARPS>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, keccak256_staged_kernel<2, BLOCKS, WARPS>, WARPS * 32, SMEM);
        if (e != cudaSuccess || ctas_per_sm < 1) { ctas_per_sm = 0; return e != cudaSuccess ? e : cudaErrorLaunchOutOfResources; }
    }
    const uint64_t tiles = (n + 31) / 32;
    uint64_t blocks = (tiles + WARPS - 1) / WARPS;
    const uint64_t cap = (uint64_t)sms * ctas_per_sm; // persistent: every CTA resident, striding over the tiles
    if (blocks > cap) blocks = cap;
    keccak256_staged_kernel<2, BLOCKS, WARPS><<<(unsigned)blocks, WARPS * 32, SMEM, s>>>(msgs, off, order, n, out, summary, len);
    return cudaGetLastError();
}

cudaError_t launch_keccak(cudaStream_t s, int device, KeccakVariant variant, const uint8_t* msgs, const uint64_t* off,
                          const uint32_t* order, uint64_t n, uint8_t* out, uint32_t* summary, const uint64_t* len)
{
    if (n == 0) return cudaSuccess;
    const int sms = keccak_num_sms(device);
    switch (variant) {
    case KECCAK_STAGED: {
        // tuning knob (development): PHANT_STAGE_CFG=b<blocks>w<warps>; the default is the measured best
        static int cfg = -1;
        if (cfg < 0) {
            const char* e = getenv("PHANT_STAGE_CFG");
            cfg = 0;
            if (e) {
                const char* names[] = {"default", "b3w4", "b2w4", "b1w4", "b4w8", "b2w8", "b4w12", "b4w6", "b3w8", "b4w10", "b4w4"};
                for (int i = 0; i < 11; ++i) if (!strcmp(e, names[i])) cfg = i;
            }
        }
        switch (cfg) {
        case 1: return launch_staged<3, 4>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 2: return launch_staged<2, 4>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 3: return launch_staged<1, 4>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 4: return launch_staged<4, 8>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 5: return launch_staged<2, 8>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 6: return launch_staged<4, 12>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 7: return launch_staged<4, 6>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 8: return launch_staged<3, 8>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 9: return launch_staged<4, 10>(s, device, sms, msgs, off, order, n, out, summary, len);
        case 10: return launch_staged<4, 4>(s, device, sms, msgs, off, order, n, out, summary, len);
        default: return launch_staged<4, 12>(s, device, sms, msgs, off, order, n, out, summary, len); // measured best: 1 CTA of 12 warps per SM
        }
    }
    case KECCAK_DIRECT: {
        uint64_t blocks = (n + 127) / 128;
        const uint64_t cap = (uint64_t)sms * 8;
        if (blocks > cap) blocks = cap;
        keccak256_direct_kernel<2><<<(unsigned)blocks, 128, 0, s>>>(msgs, off, order, n, out, summary, len);
        break;
    }
    case KECCAK_WARP: {
        uint64_t blocks = (n + 7) / 8;
        const uint64_t cap = (uint64_t)sms * 8;
        if (blocks > cap) blocks = cap;
        keccak256_warp_kernel<<<(unsigned)blocks, 256, 0, s>>>(msgs, off, n, out, len);
        if (summary) cudaMemsetAsync(summary, 0, 4 * n, s); // this layout does not classify: the walk parses every node
        break;
    }
    }
    return cudaGetLastError();
}

// blocks * chunk >= n, chunk a multiple of the tile, blocks <= 8 per SM (the scan of the last block is O(16 * blocks))
static void class_geometry(int device, uint64_t n, uint64_t& blocks, uint64_t& chunk)
{
    const uint64_t cap = (uint64_t)keccak_num_sms(device) * 8;
    chunk = ((n + cap - 1) / cap + CLS_THREADS - 1) / CLS_THREADS * CLS_THREADS;
    blocks = (n + chunk - 1) / chunk;
}
uint64_t keccak_regroup_scratch_bytes(int device, uint64_t n)
{
    uint64_t blocks, chunk;
    class_geometry(device, n ? n : 1, blocks, chunk);
    return 64 * blocks;
}
cudaError_t launch_keccak_classify(cudaStream_t s, int device, const uint64_t* off, const uint64_t* first, uint64_t n, uint32_t* hist,
                                   uint32_t* ticket, unsigned long long* perms)
{
    if (n == 0) return cudaSuccess;
    uint64_t blocks, chunk;
    class_geometry(device, n, blocks, chunk);
    keccak_class_kernel<<<(unsigned)blocks, CLS_THREADS, 0, s>>>(off, first, n, chunk, hist, ticket, perms);
    return cudaGetLastError();
}
cudaError_t launch_keccak_regroup(cudaStream_t s, int device, const uint64_t* off, const uint64_t* first, uint64_t n, const uint32_t* start,
                                  uint32_t* order)
{
    if (n == 0) return cudaSuccess;
    uint64_t blocks, chunk;
    class_geometry(device, n, blocks, chunk);
    keccak_regroup_kernel<<<(unsigned)blocks, CLS_THREADS, 0, s>>>(off, first, n, chunk, start, order);
    return cudaGetLastError();
}

} // namespace phant
