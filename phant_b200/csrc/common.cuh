// common.cuh -- declarations shared by the translation units of libphantgpu.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace phant {

enum KeccakVariant { KECCAK_STAGED = 0, KECCAK_DIRECT = 1, KECCAK_WARP = 2 };

// keccak_kernels.cu
int keccak_num_sms(int device);
cudaError_t launch_keccak(cudaStream_t s, int device, KeccakVariant variant, const uint8_t* msgs, const uint64_t* off,
                          const uint32_t* order, uint64_t n, uint8_t* out, uint32_t* summary /*nullable*/,
                          const uint64_t* len = nullptr /*nullable: message m = msgs[off[m] .. off[m] + len[m])*/);
// regrouping by permutation count (stable 16-bucket counting sort, two launches): classify fills hist[blocks][16], counts the
// permutations (perms: nullable) and leaves global start positions in hist; regroup writes `order`.  Items are messages
// (first == nullptr) or proofs of a CSR chain (item i = nodes first[i] .. first[i+1] of `off`).
uint64_t keccak_regroup_scratch_bytes(int device, uint64_t n);
cudaError_t launch_keccak_classify(cudaStream_t s, int device, const uint64_t* off, const uint64_t* first /*nullable*/, uint64_t n,
                                   uint32_t* hist, uint32_t* ticket, unsigned long long* perms /*nullable*/);
cudaError_t launch_keccak_regroup(cudaStream_t s, int device, const uint64_t* off, const uint64_t* first /*nullable*/, uint64_t n,
                                  const uint32_t* start, uint32_t* order);

// Peer-memory epilogue of the proof walk (comm.cu "peer transport"): every warp stores its ballot word straight into the
// gathered bitmap of EVERY rank of the node through NVLink peer mappings (lane r < world stores to rank r: one predicated
// store instruction), and the last CTA to finish publishes "step s of rank `me` has landed" in every rank's flag array.
constexpr int PEER_MAX_WORLD = 16;
struct PeerOut {
    uint32_t* dst[PEER_MAX_WORLD];         // rank r's bitmap of this step's buffer, at THIS rank's slice (32-bit words)
    unsigned long long* ready[PEER_MAX_WORLD]; // in rank r's region: ready[buffer][me]
    const unsigned long long* done;        // in MY region: done[buffer][0..world): rank r has copied step (value) out of this buffer
    unsigned long long wait_done;          // wait until done[r] >= this for every r before touching remote memory (0 = no wait)
    unsigned long long step;               // value to publish
    uint32_t* ticket;                      // CTA counter (device memory of this rank)
    uint32_t* err;                         // set to 1 when a wait times out
    uint32_t world;
};

// walk_kernel.cu
cudaError_t launch_walk(cudaStream_t s, int device, uint64_t n_proofs, const uint8_t* nodes, const uint64_t* node_off,
                        const uint64_t* node_index /*nullable*/, const uint64_t* proof_first, const uint8_t* keys32, const uint8_t* roots32, uint64_t n_roots,
                        const uint8_t* digests, const uint32_t* summary /*nullable*/, uint64_t* bitmap, uint8_t* status,
                        uint64_t* val_off, uint32_t* val_len, const PeerOut* peer = nullptr /*nullable: fused gather over peer memory*/);

// verify_fused.cu: hash and walk every proof of a CSR chain in one kernel (one lane per proof, `order`: nullable proof
// order from the regrouping above); counts its permutations into *perms (one atomic per warp).  The bitmap must be zeroed
// by the caller (a regrouped warp sets the bits of proofs it does not hold a whole word of with atomicOr); with `peer` the
// words go to every rank's gathered bitmap and `order` must be nullptr.
bool verify_fused_supported(const uint8_t* nodes);
cudaError_t launch_verify_fused(cudaStream_t s, int device, uint64_t n_proofs, const uint8_t* nodes, const uint64_t* node_off,
                                const uint64_t* proof_first, const uint32_t* order, const uint8_t* keys32, const uint8_t* roots32,
                                uint64_t n_roots, uint64_t* bitmap, uint8_t* status, uint64_t* val_off, uint32_t* val_len,
                                unsigned long long* perms, const PeerOut* peer = nullptr);

cudaError_t launch_peer_collect(cudaStream_t s, const unsigned long long* ready, uint32_t world, unsigned long long step, const void* src, void* dst,
                                uint64_t bytes, const PeerOut& sig);

cudaError_t launch_bag_build(cudaStream_t s, int device, const uint8_t* digests, uint64_t n_nodes, uint32_t* table, uint32_t capacity);
cudaError_t launch_walk_bag(cudaStream_t s, int device, uint64_t n_keys, const uint8_t* nodes, const uint64_t* node_off, const uint8_t* keys32,
                            const uint8_t* roots32, uint64_t n_roots, const uint8_t* digests, const uint32_t* summary, const uint32_t* table,
                            uint32_t capacity, uint64_t* bitmap, uint8_t* status, uint64_t* val_off, uint32_t* val_len);

// synth.cu
cudaError_t launch_synth_c2(cudaStream_t s, int device, uint64_t seed, uint64_t first_index, uint64_t n, uint32_t depth,
                            int corrupt, uint8_t* nodes, uint64_t* node_off, uint64_t* proof_first, uint8_t* keys32,
                            uint8_t* roots32);
cudaError_t launch_synth_c3_sizes(cudaStream_t s, int device, uint64_t seed, uint64_t first_index, uint64_t n,
                                  uint64_t* n_nodes_per, uint64_t* n_bytes_per);
cudaError_t launch_synth_c3(cudaStream_t s, int device, uint64_t seed, uint64_t first_index, uint64_t n, int corrupt,
                            const uint64_t* node_first /* exclusive scan of nodes per proof, n+1 */,
                            const uint64_t* byte_first /* exclusive scan of bytes per proof, n+1 */, uint8_t* nodes,
                            uint64_t* node_off, uint8_t* keys32, uint8_t* roots32);

} // namespace phant
