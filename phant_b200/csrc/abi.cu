// abi.cu -- the extern "C" surface of libphantgpu.so (include/phant_gpu.h): context, scratch memory,
// host<->device staging, and the launch sequences behind each entry point.
#include "../../include/phant_gpu.h"
#include "common.cuh"
#include "ctx.cuh"

#include <cub/device/device_scan.cuh>

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>

using namespace phant;

#define CU(expr)                                                              \
    do {                                                                      \
        cudaError_t e_ = (expr);                                              \
        if (e_ != cudaSuccess) return ctx->fail(e_, #expr, __FILE__, __LINE__); \
    } while (0)

// ------------------------------------------------------------------------------------------------
// context plumbing
// ------------------------------------------------------------------------------------------------
int phant_gpu_ctx::fail(cudaError_t e, const char* what, const char* file, int line)
{
    snprintf(last_error, sizeof last_error, "%s: %s (%s:%d)", cudaGetErrorName(e), what, file, line);
    cudaGetLastError(); // clear the sticky-less error
    return e == cudaErrorMemoryAllocation ? PHANT_GPU_E_OOM : PHANT_GPU_E_CUDA;
}

int DevBuf::reserve(phant_gpu_ctx* ctx, size_t bytes)
{
    if (bytes <= cap) return 0;
    if (ptr) { cudaFree(ptr); ptr = nullptr; cap = 0; }
    size_t want = bytes + bytes / 8 + 256; // a little headroom so repeated calls of similar size do not realloc
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e != cudaSuccess) { want = bytes + 256; e = cudaMalloc(&ptr, want); }
    if (e != cudaSuccess) { ptr = nullptr; return ctx->fail(e, "cudaMalloc", __FILE__, __LINE__); }
    // zero once per (re)allocation: kernels read whole aligned words / 16-byte windows, i.e. up to 15 bytes past the
    // last message byte; those bytes are masked off, but they should not be uninitialised memory.  On the context's
    // stream, so that it is ordered before everything that fills the buffer (the stream is non-blocking: a memset on
    // the legacy stream would race with it).
    cudaMemsetAsync(ptr, 0, want, ctx->stream);
    cap = want;
    return 0;
}
void DevBuf::release()
{
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
}

void phant_gpu_ctx::time_begin(int which)
{
    if ((size_t)n_pairs >= pairs.size()) pairs.emplace_back();
    EventPair& p = pairs[n_pairs];
    if (!p.a) { cudaEventCreate(&p.a); cudaEventCreate(&p.b); }
    p.which = which;
    cudaEventRecord(p.a, stream);
}
void phant_gpu_ctx::time_end()
{
    cudaEventRecord(pairs[n_pairs].b, stream);
    ++n_pairs;
}
void phant_gpu_ctx::resolve_times()
{
    if (!n_pairs) return;
    cudaStreamSynchronize(stream);
    for (int i = 0; i < n_pairs; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pairs[i].a, pairs[i].b) == cudaSuccess) {
            if (pairs[i].which == 0) stats.keccak_ms += ms; else stats.walk_ms += ms;
        }
    }
    n_pairs = 0;
}

extern "C" int phant_gpu_abi_version(void) { return PHANT_GPU_ABI_VERSION; }

extern "C" const char* phant_gpu_strerror(int code)
{
    switch (code) {
    case PHANT_GPU_OK: return "ok";
    case PHANT_GPU_E_INVALID: return "invalid argument";
    case PHANT_GPU_E_NO_DEVICE: return "no usable CUDA device";
    case PHANT_GPU_E_OOM: return "out of device memory";
    case PHANT_GPU_E_CUDA: return "CUDA runtime error";
    case PHANT_GPU_E_COMM: return "collective communication error";
    case PHANT_GPU_E_MALFORMED: return "malformed RLP in builder input";
    default: return "unknown error";
    }
}

extern "C" int phant_gpu_create(phant_gpu_ctx** out, const phant_gpu_config* cfg)
{
    if (!out) return PHANT_GPU_E_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); return PHANT_GPU_E_NO_DEVICE; }
    // environment overrides (deployment knobs a Zig host need not plumb through): PHANT_GPU_DEVICE replaces cfg->device,
    // PHANT_GPU_FLAGS (decimal or 0x..) is OR-ed into cfg->flags; PHANT_GPU_NCCL_LIB names the NCCL library (comm.cu)
    int dev = cfg ? cfg->device : 0;
    uint32_t env_flags = 0;
    if (const char* e = getenv("PHANT_GPU_DEVICE")) { char* end = nullptr; const long v = strtol(e, &end, 10); if (end != e && *end == 0) dev = (int)v; }
    if (const char* e = getenv("PHANT_GPU_FLAGS")) { char* end = nullptr; const unsigned long v = strtoul(e, &end, 0); if (end != e && *end == 0) env_flags = (uint32_t)v; }
    if (dev < 0 || dev >= count) return PHANT_GPU_E_INVALID;
    if (cudaSetDevice(dev) != cudaSuccess) { cudaGetLastError(); return PHANT_GPU_E_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { cudaGetLastError(); return PHANT_GPU_E_NO_DEVICE; }
    if (prop.major < 10) return PHANT_GPU_E_NO_DEVICE; // sm_100a code only
    phant_gpu_ctx* ctx = new (std::nothrow) phant_gpu_ctx();
    if (!ctx) return PHANT_GPU_E_OOM;
    ctx->device = dev;
    ctx->flags = (cfg ? cfg->flags : 0) | env_flags;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        delete ctx;
        return PHANT_GPU_E_CUDA;
    }
    ctx->stream = ctx->own_stream;
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        cudaStreamDestroy(ctx->own_stream);
        delete ctx;
        return PHANT_GPU_E_CUDA;
    }
    *out = ctx;
    return PHANT_GPU_OK;
}

extern "C" void phant_gpu_destroy(phant_gpu_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    phant_gpu_comm_destroy(ctx);
    for (DevBuf* b : ctx->all_bufs()) b->release();
    for (EventPair& p : ctx->pairs)
        if (p.a) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (cudaEvent_t e : ctx->chunk_events) cudaEventDestroy(e);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

extern "C" int phant_gpu_set_flags(phant_gpu_ctx* ctx, uint32_t flags)
{
    if (!ctx) return PHANT_GPU_E_INVALID;
    ctx->flags = flags;
    return PHANT_GPU_OK;
}
extern "C" int phant_gpu_set_stream(phant_gpu_ctx* ctx, void* cuda_stream)
{
    if (!ctx) return PHANT_GPU_E_INVALID;
    ctx->resolve_times();
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return PHANT_GPU_OK;
}
extern "C" const char* phant_gpu_last_error(const phant_gpu_ctx* ctx) { return ctx ? ctx->last_error : "null context"; }

extern "C" int phant_gpu_synchronize(phant_gpu_ctx* ctx)
{
    if (!ctx) return PHANT_GPU_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->comm_stream) CU(cudaStreamSynchronize(ctx->comm_stream));
    return PHANT_GPU_OK;
}
extern "C" int phant_gpu_get_stats(phant_gpu_ctx* ctx, phant_gpu_stats* out)
{
    if (!ctx || !out) return PHANT_GPU_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    ctx->resolve_times();
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->perms_pending) {
        unsigned long long p = 0;
        CU(cudaMemcpy(&p, ctx->d_perms.ptr, sizeof p, cudaMemcpyDeviceToHost));
        ctx->stats.keccak_perms += p;
        CU(cudaMemset(ctx->d_perms.ptr, 0, sizeof p));
        ctx->perms_pending = false;
    }
    *out = ctx->stats;
    return PHANT_GPU_OK;
}
extern "C" int phant_gpu_reset_stats(phant_gpu_ctx* ctx)
{
    if (!ctx) return PHANT_GPU_E_INVALID;
    phant_gpu_stats tmp;
    int rc = phant_gpu_get_stats(ctx, &tmp);
    memset(&ctx->stats, 0, sizeof ctx->stats);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// K: hash a CSR message set that is already on the device
// ------------------------------------------------------------------------------------------------
int phant_gpu_ctx::hash_csr(const uint8_t* d_msgs, const uint64_t* d_off, uint64_t n, uint64_t total_bytes, uint8_t* d_out,
                            uint32_t* d_summary)
{
    phant_gpu_ctx* ctx = this;
    if (n == 0) return PHANT_GPU_OK;
    if (n > 0xffffffffull) return PHANT_GPU_E_INVALID; // message indices are 32-bit on the device
    NvtxRange nvtx("phant:keccak");
    KeccakVariant variant = KECCAK_STAGED;
    if (flags & PHANT_GPU_FLAG_KECCAK_DIRECT) variant = KECCAK_DIRECT;
    if (flags & PHANT_GPU_FLAG_KECCAK_WARP) variant = KECCAK_WARP;
    if (variant == KECCAK_STAGED && ((uintptr_t)d_msgs & 15)) variant = KECCAK_DIRECT; // bulk copies need 16-byte alignment

    // classify (always: it also counts the permutations for the stats) and, optionally, regroup -- two launches of our
    // own (keccak_kernels.cu "regrouping"), no library sort on the hot path
    if (int rc = d_perms.reserve(ctx, 64)) return rc;
    if (!perms_init) { CU(cudaMemsetAsync(d_perms.ptr, 0, 64, stream)); perms_init = true; } // [0] permutations, [1] block ticket
    if (int rc = d_idx.reserve(ctx, keccak_regroup_scratch_bytes(device, n))) return rc;
    CU(launch_keccak_classify(stream, device, d_off, nullptr, n, (uint32_t*)d_idx.ptr, (uint32_t*)((unsigned long long*)d_perms.ptr + 1),
                              (unsigned long long*)d_perms.ptr));
    stats.launches++;
    perms_pending = true;
    const uint32_t* order = nullptr;
    const bool regroup = !(flags & PHANT_GPU_FLAG_NO_BINNING) && variant != KECCAK_WARP && n >= 4096;
    if (regroup) {
        if (int rc = d_order.reserve(ctx, 4 * n)) return rc;
        CU(launch_keccak_regroup(stream, device, d_off, nullptr, n, (const uint32_t*)d_idx.ptr, (uint32_t*)d_order.ptr));
        stats.launches++;
        order = (const uint32_t*)d_order.ptr;
    }
    time_begin(0);
    CU(launch_keccak(stream, device, variant, d_msgs, d_off, order, n, d_out, d_summary));
    time_end();
    stats.launches++;
    stats.keccak_msgs += n;
    stats.keccak_bytes += total_bytes;
    return PHANT_GPU_OK;
}

int phant_gpu_ctx::hash_slots(const uint8_t* d_msgs, const uint64_t* d_off, const uint64_t* d_len, uint64_t n, uint8_t* d_out)
{
    phant_gpu_ctx* ctx = this;
    if (n == 0) return PHANT_GPU_OK;
    KeccakVariant variant = KECCAK_STAGED;
    if (flags & PHANT_GPU_FLAG_KECCAK_DIRECT) variant = KECCAK_DIRECT;
    if (flags & PHANT_GPU_FLAG_KECCAK_WARP) variant = KECCAK_WARP;
    if (variant == KECCAK_STAGED && ((uintptr_t)d_msgs & 15)) variant = KECCAK_DIRECT;
    time_begin(0);
    CU(launch_keccak(stream, device, variant, d_msgs, d_off, nullptr, n, d_out, nullptr, d_len));
    time_end();
    stats.launches++;
    stats.keccak_msgs += n;
    return PHANT_GPU_OK;
}

// offsets must start the CSR at off[0] (any value) and be monotone; returns total bytes via *total
static int check_offsets_host(const uint64_t* off, uint64_t n, uint64_t* total)
{
    for (uint64_t i = 0; i < n; ++i)
        if (off[i + 1] < off[i]) return PHANT_GPU_E_INVALID;
    *total = off[n];
    return PHANT_GPU_OK;
}

extern "C" int phant_gpu_keccak256_batch(phant_gpu_ctx* ctx, const uint8_t* msgs, const uint64_t* off, uint64_t n, uint8_t* out)
{
    if (!ctx || (n && (!off || !out))) return PHANT_GPU_E_INVALID;
    if (n == 0) return PHANT_GPU_OK;
    CU(cudaSetDevice(ctx->device));
    if (ctx->flags & PHANT_GPU_FLAG_DEVICE_PTRS) {
        uint64_t last = 0;
        CU(cudaMemcpyAsync(&last, off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (last && !msgs) return PHANT_GPU_E_INVALID;
        return ctx->hash_csr(msgs, off, n, last, out);
    }
    uint64_t total = 0;
    if (int rc = check_offsets_host(off, n, &total)) return rc;
    if (total && !msgs) return PHANT_GPU_E_INVALID;
    if (int rc = ctx->d_msgs.reserve(ctx, total + 64)) return rc;
    if (int rc = ctx->d_off.reserve(ctx, 8 * (n + 1))) return rc;
    if (int rc = ctx->d_out.reserve(ctx, 32 * n)) return rc;
    if (total) CU(cudaMemcpyAsync(ctx->d_msgs.ptr, msgs, total, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_off.ptr, off, 8 * (n + 1), cudaMemcpyHostToDevice, ctx->stream));
    ctx->stats.h2d_bytes += total + 8 * (n + 1);
    if (int rc = ctx->hash_csr((const uint8_t*)ctx->d_msgs.ptr, (const uint64_t*)ctx->d_off.ptr, n, total, (uint8_t*)ctx->d_out.ptr)) return rc;
    CU(cudaMemcpyAsync(out, ctx->d_out.ptr, 32 * n, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.d2h_bytes += 32 * n;
    CU(cudaStreamSynchronize(ctx->stream));
    return PHANT_GPU_OK;
}

// device pointers with the total supplied by the caller: fully asynchronous on the context's stream (the plain entry point
// has to read off[n] back, one host synchronisation per call)
extern "C" int phant_gpu_keccak256_batch_async(phant_gpu_ctx* ctx, const uint8_t* msgs, const uint64_t* off, uint64_t n, uint64_t total_bytes,
                                               uint8_t* out)
{
    if (!ctx || (n && (!off || !out)) || (total_bytes && !msgs)) return PHANT_GPU_E_INVALID;
    if (!(ctx->flags & PHANT_GPU_FLAG_DEVICE_PTRS)) return PHANT_GPU_E_INVALID;
    if (n == 0) return PHANT_GPU_OK;
    CU(cudaSetDevice(ctx->device));
    return ctx->hash_csr(msgs, off, n, total_bytes, out);
}

// ------------------------------------------------------------------------------------------------
// V: proof verification
// ------------------------------------------------------------------------------------------------
// A CSR chain (no node_index) is verified in one pass: verify_fused.cu hashes and walks each proof in the same lane, so the
// digests and node summaries of the two-pass path (hash_csr + walk_kernel) are never written.  Proofs are regrouped by their
// permutation count first (keccak_kernels.cu "regrouping", per proof instead of per node), so that the 32 lanes of a warp
// hash chains of similar length.  The two-pass path stays for deduplicated witnesses (a shared node is hashed once), for
// the KECCAK_DIRECT / KECCAK_WARP variants and for a node buffer that is not 16-byte aligned.
static bool fused_path(const phant_gpu_ctx* ctx, const uint8_t* nodes)
{
    return !(ctx->flags & (PHANT_GPU_FLAG_KECCAK_DIRECT | PHANT_GPU_FLAG_KECCAK_WARP)) && verify_fused_supported(nodes);
}
// `fence_and_clear`: device-pointer call -- wait for the collective still using `bitmap` (sharded calls), then zero it
static int verify_fused(phant_gpu_ctx* ctx, const uint8_t* nodes, const uint64_t* node_off, const uint64_t* proof_first, uint64_t np,
                        uint64_t n_nodes, uint64_t total, const uint8_t* keys32, const uint8_t* roots32, uint64_t n_roots, uint64_t* bitmap,
                        uint8_t* status, uint64_t* val_off, uint32_t* val_len, const PeerOut* peer, bool fence_and_clear)
{
    if (np > 0xffffffffull) return PHANT_GPU_E_INVALID; // proof indices are 32-bit on the device
    NvtxRange nvtx("phant:verify");
    cudaStream_t s = ctx->stream;
    if (int rc = ctx->d_perms.reserve(ctx, 64)) return rc;
    if (!ctx->perms_init) { CU(cudaMemsetAsync(ctx->d_perms.ptr, 0, 64, s)); ctx->perms_init = true; } // [0] permutations, [1] block ticket
    const uint32_t* order = nullptr;
    if (!peer && !(ctx->flags & PHANT_GPU_FLAG_NO_BINNING) && np >= 4096) {
        if (int rc = ctx->d_idx.reserve(ctx, keccak_regroup_scratch_bytes(ctx->device, np))) return rc;
        if (int rc = ctx->d_order.reserve(ctx, 4 * np)) return rc;
        CU(launch_keccak_classify(s, ctx->device, node_off, proof_first, np, (uint32_t*)ctx->d_idx.ptr,
                                  (uint32_t*)((unsigned long long*)ctx->d_perms.ptr + 1), nullptr));
        CU(launch_keccak_regroup(s, ctx->device, node_off, proof_first, np, (const uint32_t*)ctx->d_idx.ptr, (uint32_t*)ctx->d_order.ptr));
        ctx->stats.launches += 2;
        order = (const uint32_t*)ctx->d_order.ptr;
    }
    if (fence_and_clear) {
        if (int rc = ctx->wait_walk_fence()) return rc; // sharded call: the previous gather of this bitmap buffer (comm.cu)
        if (bitmap) CU(cudaMemsetAsync(bitmap, 0, ((np + 63) / 64) * 8, s));
    }
    ctx->time_begin(0);
    CU(launch_verify_fused(s, ctx->device, np, nodes, node_off, proof_first, order, keys32, roots32, n_roots, bitmap, status, val_off, val_len,
                           (unsigned long long*)ctx->d_perms.ptr, peer));
    ctx->time_end();
    ctx->stats.launches++;
    ctx->stats.keccak_msgs += n_nodes;
    ctx->stats.keccak_bytes += total;
    ctx->perms_pending = true;
    return PHANT_GPU_OK;
}

// host pointers + deduplicated witness: distinct nodes are hashed once, chains are index lists (one shot, no chunking:
// a chunk of proofs does not map to a contiguous range of nodes)
static int verify_dedup_host(phant_gpu_ctx* ctx, const phant_gpu_proof_batch* in, uint64_t* accept_bitmap, uint8_t* status,
                             uint64_t* val_off, uint32_t* val_len)
{
    const uint64_t np = in->n_proofs, n_nodes = in->n_nodes;
    if (n_nodes == 0) return PHANT_GPU_E_INVALID;
    uint64_t total = 0;
    if (int rc = check_offsets_host(in->node_off, n_nodes, &total)) return rc;
    if (total && !in->nodes) return PHANT_GPU_E_INVALID;
    for (uint64_t p = 0; p < np; ++p)
        if (in->proof_first[p + 1] < in->proof_first[p]) return PHANT_GPU_E_INVALID;
    const uint64_t n_refs = in->proof_first[np];
    for (uint64_t r = 0; r < n_refs; ++r)
        if (in->node_index[r] >= n_nodes) return PHANT_GPU_E_INVALID;
    const size_t bm_bytes = ((np + 63) / 64) * 8;
    if (int rc = ctx->d_msgs.reserve(ctx, total + 64)) return rc;
    if (int rc = ctx->d_off.reserve(ctx, 8 * (n_nodes + 1))) return rc;
    if (int rc = ctx->d_first.reserve(ctx, 8 * (np + 1))) return rc;
    if (int rc = ctx->d_index.reserve(ctx, 8 * (n_refs + 1))) return rc;
    if (int rc = ctx->d_keys.reserve(ctx, 32 * np)) return rc;
    if (int rc = ctx->d_roots.reserve(ctx, 32 * in->n_roots)) return rc;
    if (int rc = ctx->d_digests.reserve(ctx, 32 * n_nodes + 32)) return rc;
    if (int rc = ctx->d_summary.reserve(ctx, 4 * n_nodes + 32)) return rc;
    if (int rc = ctx->d_bitmap.reserve(ctx, bm_bytes)) return rc;
    if (int rc = ctx->d_status.reserve(ctx, np)) return rc;
    if (val_off) if (int rc = ctx->d_voff.reserve(ctx, 8 * np)) return rc;
    if (val_len) if (int rc = ctx->d_vlen.reserve(ctx, 4 * np)) return rc;
    cudaStream_t s = ctx->stream;
    if (total) CU(cudaMemcpyAsync(ctx->d_msgs.ptr, in->nodes, total, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ctx->d_off.ptr, in->node_off, 8 * (n_nodes + 1), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ctx->d_first.ptr, in->proof_first, 8 * (np + 1), cudaMemcpyHostToDevice, s));
    if (n_refs) CU(cudaMemcpyAsync(ctx->d_index.ptr, in->node_index, 8 * n_refs, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ctx->d_keys.ptr, in->keys32, 32 * np, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ctx->d_roots.ptr, in->roots32, 32 * in->n_roots, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += total + 8 * (n_nodes + 1) + 8 * (np + 1) + 8 * n_refs + 32 * np + 32 * in->n_roots;
    if (int rc = ctx->hash_csr((const uint8_t*)ctx->d_msgs.ptr, (const uint64_t*)ctx->d_off.ptr, n_nodes, total, (uint8_t*)ctx->d_digests.ptr,
                               (uint32_t*)ctx->d_summary.ptr)) return rc;
    CU(cudaMemsetAsync(ctx->d_bitmap.ptr, 0, bm_bytes, s));
    ctx->time_begin(1);
    CU(launch_walk(s, ctx->device, np, (const uint8_t*)ctx->d_msgs.ptr, (const uint64_t*)ctx->d_off.ptr, (const uint64_t*)ctx->d_index.ptr,
                   (const uint64_t*)ctx->d_first.ptr, (const uint8_t*)ctx->d_keys.ptr, (const uint8_t*)ctx->d_roots.ptr, in->n_roots,
                   (const uint8_t*)ctx->d_digests.ptr, (const uint32_t*)ctx->d_summary.ptr, (uint64_t*)ctx->d_bitmap.ptr,
                   (uint8_t*)ctx->d_status.ptr, val_off ? (uint64_t*)ctx->d_voff.ptr : nullptr, val_len ? (uint32_t*)ctx->d_vlen.ptr : nullptr));
    ctx->time_end();
    ctx->stats.launches++;
    if (accept_bitmap) { CU(cudaMemcpyAsync(accept_bitmap, ctx->d_bitmap.ptr, bm_bytes, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += bm_bytes; }
    if (status) { CU(cudaMemcpyAsync(status, ctx->d_status.ptr, np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += np; }
    if (val_off) { CU(cudaMemcpyAsync(val_off, ctx->d_voff.ptr, 8 * np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 8 * np; }
    if (val_len) { CU(cudaMemcpyAsync(val_len, ctx->d_vlen.ptr, 4 * np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 4 * np; }
    CU(cudaStreamSynchronize(s));
    return PHANT_GPU_OK;
}

extern "C" int phant_gpu_verify_proofs(phant_gpu_ctx* ctx, const phant_gpu_proof_batch* in, uint64_t* accept_bitmap,
                                       uint8_t* status, uint64_t* val_off, uint32_t* val_len)
{
    if (!ctx || !in) return PHANT_GPU_E_INVALID;
    const uint64_t np = in->n_proofs;
    if (np == 0) return PHANT_GPU_OK;
    if (!in->node_off || !in->proof_first || !in->keys32 || !in->roots32) return PHANT_GPU_E_INVALID;
    if (in->n_roots != 1 && in->n_roots != np) return PHANT_GPU_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    const size_t bm_bytes = ((np + 63) / 64) * 8;

    if (ctx->flags & PHANT_GPU_FLAG_DEVICE_PTRS) {
        uint64_t n_nodes = in->n_nodes, total = in->nodes_bytes;
        if (in->node_index && n_nodes == 0) return PHANT_GPU_E_INVALID; // the number of distinct nodes cannot be derived
        if (n_nodes == 0) { // not supplied: read the tails of the CSR arrays back (one sync each)
            CU(cudaMemcpyAsync(&n_nodes, in->proof_first + np, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            if (n_nodes) {
                CU(cudaMemcpyAsync(&total, in->node_off + n_nodes, 8, cudaMemcpyDeviceToHost, ctx->stream));
                CU(cudaStreamSynchronize(ctx->stream));
            }
        }
        if (!in->node_index && fused_path(ctx, in->nodes))
            return verify_fused(ctx, in->nodes, in->node_off, in->proof_first, np, n_nodes, total, in->keys32, in->roots32, in->n_roots,
                                accept_bitmap, status, val_off, val_len, (const PeerOut*)ctx->walk_peer, true); // asynchronous, as below
        if (int rc = ctx->d_digests.reserve(ctx, 32 * n_nodes + 32)) return rc;
        if (int rc = ctx->d_summary.reserve(ctx, 4 * n_nodes + 32)) return rc;
        if (int rc = ctx->hash_csr(in->nodes, in->node_off, n_nodes, total, (uint8_t*)ctx->d_digests.ptr, (uint32_t*)ctx->d_summary.ptr)) return rc;
        NvtxRange nvtx("phant:walk");
        if (int rc = ctx->wait_walk_fence()) return rc; // sharded call: the previous gather of this bitmap buffer (comm.cu)
        if (accept_bitmap) CU(cudaMemsetAsync(accept_bitmap, 0, bm_bytes, ctx->stream));
        ctx->time_begin(1);
        CU(launch_walk(ctx->stream, ctx->device, np, in->nodes, in->node_off, in->node_index, in->proof_first, in->keys32, in->roots32, in->n_roots,
                       (const uint8_t*)ctx->d_digests.ptr, (const uint32_t*)ctx->d_summary.ptr, accept_bitmap, status, val_off, val_len,
                       (const PeerOut*)ctx->walk_peer /* sharded call over the peer transport: fused gather (comm.cu) */));
        ctx->time_end();
        ctx->stats.launches++;
        return PHANT_GPU_OK; // asynchronous on the context's stream: phant_gpu_synchronize() to wait
    }

    // host pointers: validate the CSR arrays, stage everything, run, copy the verdicts back
    if (in->node_index) return verify_dedup_host(ctx, in, accept_bitmap, status, val_off, val_len);
    // (the CSR arrays are validated chunk by chunk below, while the previous chunk's DMA is in flight)
    const uint64_t n_nodes = in->proof_first[np];
    const uint64_t total = in->node_off[n_nodes];
    if (total && !in->nodes) return PHANT_GPU_E_INVALID;
    if (int rc = ctx->d_msgs.reserve(ctx, total + 64)) return rc;
    if (int rc = ctx->d_off.reserve(ctx, 8 * (n_nodes + 1))) return rc;
    if (int rc = ctx->d_first.reserve(ctx, 8 * (np + 1))) return rc;
    if (int rc = ctx->d_keys.reserve(ctx, 32 * np)) return rc;
    if (int rc = ctx->d_roots.reserve(ctx, 32 * in->n_roots)) return rc;
    const bool fused = fused_path(ctx, (const uint8_t*)ctx->d_msgs.ptr);
    if (!fused) { // the two-pass path keeps every digest and summary of the batch
        if (int rc = ctx->d_digests.reserve(ctx, 32 * n_nodes + 32)) return rc;
        if (int rc = ctx->d_summary.reserve(ctx, 4 * n_nodes + 32)) return rc;
    }
    if (int rc = ctx->d_bitmap.reserve(ctx, bm_bytes)) return rc;
    if (int rc = ctx->d_status.reserve(ctx, np)) return rc;
    if (val_off) if (int rc = ctx->d_voff.reserve(ctx, 8 * np)) return rc;
    if (val_len) if (int rc = ctx->d_vlen.reserve(ctx, 4 * np)) return rc;
    cudaStream_t s = ctx->stream, cs = ctx->copy_stream;
    // Pipeline: the witness crosses PCIe in chunks of whole proofs on the copy stream while the previous
    // chunk is hashed and walked on the compute stream.  Device arrays keep their full size and absolute
    // offsets, so a chunk is just a sub-range [p0, p1) of proofs = [n0, n1) of nodes = [b0, b1) of bytes.
    uint8_t* d_nodes = (uint8_t*)ctx->d_msgs.ptr;
    uint64_t* d_noff = (uint64_t*)ctx->d_off.ptr;
    uint64_t* d_pfirst = (uint64_t*)ctx->d_first.ptr;
    CU(cudaMemsetAsync(ctx->d_bitmap.ptr, 0, bm_bytes, s));
    CU(cudaMemcpyAsync(ctx->d_roots.ptr, in->roots32, 32 * in->n_roots, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += total + 8 * (n_nodes + 1) + 8 * (np + 1) + 32 * np + 32 * in->n_roots;
    // per chunk: large enough for PCIe efficiency, small enough to start early (PHANT_GPU_CHUNK_MB: development knob)
    static uint64_t chunk_mb = 0;
    if (!chunk_mb) { const char* e = getenv("PHANT_GPU_CHUNK_MB"); const long v = e ? atol(e) : 0; chunk_mb = v >= 1 && v <= 4096 ? (uint64_t)v : 128; }
    const uint64_t target_bytes = chunk_mb << 20;
    uint64_t p0 = 0;
    size_t chunk = 0;
    // the copy stream must not overwrite buffers a previous call's kernels may still read
    if (ctx->chunk_events.empty()) { cudaEvent_t e; CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->chunk_events.push_back(e); }
    CU(cudaEventRecord(ctx->chunk_events[0], s));
    CU(cudaStreamWaitEvent(cs, ctx->chunk_events[0], 0));
    while (p0 < np) {
        // grow the chunk proof by proof (64 at a time, so bitmap words never straddle chunks) up to the byte target
        uint64_t p1 = p0;
        const uint64_t n0 = in->proof_first[p0], b0 = n0 <= n_nodes ? in->node_off[n0] : 0;
        bool in_range = n0 <= n_nodes;
        do {
            p1 = p1 + 4096 < np ? p1 + 4096 : np;
            in_range = in_range && in->proof_first[p1] <= n_nodes;
        } while (in_range && p1 < np && in->node_off[in->proof_first[p1]] - b0 < target_bytes);
        if (!in_range) { // never leave DMA running on the caller's buffers behind an error return
            cudaStreamSynchronize(cs);
            cudaStreamSynchronize(s);
            return PHANT_GPU_E_INVALID;
        }
        const uint64_t n1 = in->proof_first[p1], b1 = in->node_off[n1];
        {   // monotone offsets inside the declared totals, or nothing of this chunk is touched
            bool ok = n0 <= n1 && n1 <= n_nodes && b0 <= b1 && b1 <= total;
            for (uint64_t p = p0; ok && p < p1; ++p) ok = in->proof_first[p] <= in->proof_first[p + 1];
            for (uint64_t j = n0; ok && j < n1; ++j) ok = in->node_off[j] <= in->node_off[j + 1];
            if (!ok) {
                cudaStreamSynchronize(cs);
                cudaStreamSynchronize(s);
                return PHANT_GPU_E_INVALID;
            }
        }
        nvtxRangePushA("phant:h2d chunk");
        if (b1 > b0) CU(cudaMemcpyAsync(d_nodes + b0, in->nodes + b0, b1 - b0, cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(d_noff + n0, in->node_off + n0, 8 * (n1 - n0 + 1), cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(d_pfirst + p0, in->proof_first + p0, 8 * (p1 - p0 + 1), cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync((uint8_t*)ctx->d_keys.ptr + 32 * p0, in->keys32 + 32 * p0, 32 * (p1 - p0), cudaMemcpyHostToDevice, cs));
        ++chunk;
        if (ctx->chunk_events.size() <= chunk) { cudaEvent_t e; CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->chunk_events.push_back(e); }
        CU(cudaEventRecord(ctx->chunk_events[chunk], cs));
        CU(cudaStreamWaitEvent(s, ctx->chunk_events[chunk], 0));
        nvtxRangePop();
        if (fused) {
            if (int rc = verify_fused(ctx, d_nodes, d_noff, d_pfirst + p0, p1 - p0, n1 - n0, b1 - b0, (const uint8_t*)ctx->d_keys.ptr + 32 * p0,
                                      (const uint8_t*)ctx->d_roots.ptr + (in->n_roots == 1 ? 0 : 32 * p0), in->n_roots,
                                      (uint64_t*)ctx->d_bitmap.ptr + p0 / 64, (uint8_t*)ctx->d_status.ptr + p0,
                                      val_off ? (uint64_t*)ctx->d_voff.ptr + p0 : nullptr, val_len ? (uint32_t*)ctx->d_vlen.ptr + p0 : nullptr,
                                      nullptr, false)) {
                cudaStreamSynchronize(cs); // as below: no DMA on the caller's buffers after we return
                cudaStreamSynchronize(s);
                return rc;
            }
            p0 = p1;
            continue;
        }
        if (int rc = ctx->hash_csr(d_nodes, d_noff + n0, n1 - n0, b1 - b0, (uint8_t*)ctx->d_digests.ptr + 32 * n0,
                                   (uint32_t*)ctx->d_summary.ptr + n0)) {
            cudaStreamSynchronize(cs); // as above: no DMA on the caller's buffers after we return
            cudaStreamSynchronize(s);
            return rc;
        }
        ctx->time_begin(1);
        CU(launch_walk(s, ctx->device, p1 - p0, d_nodes, d_noff, nullptr, d_pfirst + p0, (const uint8_t*)ctx->d_keys.ptr + 32 * p0,
                       (const uint8_t*)ctx->d_roots.ptr + (in->n_roots == 1 ? 0 : 32 * p0), in->n_roots, (const uint8_t*)ctx->d_digests.ptr,
                       (const uint32_t*)ctx->d_summary.ptr, (uint64_t*)ctx->d_bitmap.ptr + p0 / 64, (uint8_t*)ctx->d_status.ptr + p0, val_off ? (uint64_t*)ctx->d_voff.ptr + p0 : nullptr,
                       val_len ? (uint32_t*)ctx->d_vlen.ptr + p0 : nullptr));
        ctx->time_end();
        ctx->stats.launches++;
        p0 = p1;
    }
    if (accept_bitmap) { CU(cudaMemcpyAsync(accept_bitmap, ctx->d_bitmap.ptr, bm_bytes, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += bm_bytes; }
    if (status) { CU(cudaMemcpyAsync(status, ctx->d_status.ptr, np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += np; }
    if (val_off) { CU(cudaMemcpyAsync(val_off, ctx->d_voff.ptr, 8 * np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 8 * np; }
    if (val_len) { CU(cudaMemcpyAsync(val_len, ctx->d_vlen.ptr, 4 * np, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 4 * np; }
    CU(cudaStreamSynchronize(s));
    return PHANT_GPU_OK;
}

// ------------------------------------------------------------------------------------------------
// W: witness as a set of nodes
// ------------------------------------------------------------------------------------------------
extern "C" int phant_gpu_verify_witness(phant_gpu_ctx* ctx, const phant_gpu_witness* in, uint64_t* accept_bitmap, uint8_t* status,
                                        uint64_t* val_off, uint32_t* val_len)
{
    if (!ctx || !in) return PHANT_GPU_E_INVALID;
    const uint64_t nk = in->n_keys, nn = in->n_nodes;
    if (nk == 0) return PHANT_GPU_OK;
    if (!in->keys32 || !in->roots32 || (nn && !in->node_off) || (in->n_roots != 1 && in->n_roots != nk)) return PHANT_GPU_E_INVALID;
    if (nn > (1ull << 30)) return PHANT_GPU_E_INVALID; // table capacity (2 x nn rounded up to a power of two) must fit 32 bits
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const bool dev = ctx->flags & PHANT_GPU_FLAG_DEVICE_PTRS;
    const size_t bm_bytes = ((nk + 63) / 64) * 8;
    uint64_t total = in->nodes_bytes;
    const uint8_t* d_nodes = in->nodes; const uint64_t* d_noff = in->node_off; const uint8_t* d_keys = in->keys32; const uint8_t* d_roots = in->roots32;
    uint64_t* d_bitmap = accept_bitmap; uint8_t* d_status = status; uint64_t* d_voff = val_off; uint32_t* d_vlen = val_len;
    if (!dev) {
        total = 0;
        if (nn) { if (int rc = check_offsets_host(in->node_off, nn, &total)) return rc; }
        if (total && !in->nodes) return PHANT_GPU_E_INVALID;
        if (int rc = ctx->d_msgs.reserve(ctx, total + 64)) return rc;
        if (int rc = ctx->d_off.reserve(ctx, 8 * (nn + 1))) return rc;
        if (int rc = ctx->d_keys.reserve(ctx, 32 * nk)) return rc;
        if (int rc = ctx->d_roots.reserve(ctx, 32 * in->n_roots)) return rc;
        if (int rc = ctx->d_bitmap.reserve(ctx, bm_bytes)) return rc;
        if (int rc = ctx->d_status.reserve(ctx, nk)) return rc;
        if (val_off) if (int rc = ctx->d_voff.reserve(ctx, 8 * nk)) return rc;
        if (val_len) if (int rc = ctx->d_vlen.reserve(ctx, 4 * nk)) return rc;
        if (total) CU(cudaMemcpyAsync(ctx->d_msgs.ptr, in->nodes, total, cudaMemcpyHostToDevice, s));
        static const uint64_t zero2[2] = {0, 0};
        CU(cudaMemcpyAsync(ctx->d_off.ptr, nn ? in->node_off : zero2, 8 * (nn + 1), cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(ctx->d_keys.ptr, in->keys32, 32 * nk, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(ctx->d_roots.ptr, in->roots32, 32 * in->n_roots, cudaMemcpyHostToDevice, s));
        ctx->stats.h2d_bytes += total + 8 * (nn + 1) + 32 * nk + 32 * in->n_roots;
        d_nodes = (const uint8_t*)ctx->d_msgs.ptr; d_noff = (const uint64_t*)ctx->d_off.ptr; d_keys = (const uint8_t*)ctx->d_keys.ptr;
        d_roots = (const uint8_t*)ctx->d_roots.ptr; d_bitmap = (uint64_t*)ctx->d_bitmap.ptr; d_status = (uint8_t*)ctx->d_status.ptr;
        d_voff = val_off ? (uint64_t*)ctx->d_voff.ptr : nullptr; d_vlen = val_len ? (uint32_t*)ctx->d_vlen.ptr : nullptr;
    }
    uint32_t capacity = 64;
    while ((uint64_t)capacity < 2 * nn) capacity <<= 1; // load factor <= 0.5; nn <= 2^30 bounds this at 2^31
    if (int rc = ctx->d_digests.reserve(ctx, 32 * nn + 32)) return rc;
    if (int rc = ctx->d_summary.reserve(ctx, 4 * nn + 32)) return rc;
    if (int rc = ctx->d_index.reserve(ctx, 4ull * capacity)) return rc;
    if (int rc = ctx->hash_csr(d_nodes, d_noff, nn, total, (uint8_t*)ctx->d_digests.ptr, (uint32_t*)ctx->d_summary.ptr)) return rc;
    CU(launch_bag_build(s, ctx->device, (const uint8_t*)ctx->d_digests.ptr, nn, (uint32_t*)ctx->d_index.ptr, capacity));
    if (d_bitmap) CU(cudaMemsetAsync(d_bitmap, 0, bm_bytes, s));
    ctx->time_begin(1);
    CU(launch_walk_bag(s, ctx->device, nk, d_nodes, d_noff, d_keys, d_roots, in->n_roots, (const uint8_t*)ctx->d_digests.ptr,
                       (const uint32_t*)ctx->d_summary.ptr, (const uint32_t*)ctx->d_index.ptr, capacity, d_bitmap, d_status, d_voff, d_vlen));
    ctx->time_end();
    ctx->stats.launches += 2;
    if (!dev) {
        if (accept_bitmap) { CU(cudaMemcpyAsync(accept_bitmap, d_bitmap, bm_bytes, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += bm_bytes; }
        if (status) { CU(cudaMemcpyAsync(status, d_status, nk, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += nk; }
        if (val_off) { CU(cudaMemcpyAsync(val_off, d_voff, 8 * nk, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 8 * nk; }
        if (val_len) { CU(cudaMemcpyAsync(val_len, d_vlen, 4 * nk, cudaMemcpyDeviceToHost, s)); ctx->stats.d2h_bytes += 4 * nk; }
        CU(cudaStreamSynchronize(s));
    }
    return PHANT_GPU_OK;
}

// ------------------------------------------------------------------------------------------------
// B: logs blooms (src/types/receipt.zig:37-63)
// ------------------------------------------------------------------------------------------------
__global__ void bloom_set_kernel(const uint8_t* __restrict__ digests, const uint32_t* __restrict__ bloom_of_item, uint64_t n_items,
                                 uint64_t n_blooms, uint32_t* __restrict__ blooms /* n_blooms * 64 words */)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t b = bloom_of_item[i];
        if (b >= n_blooms) continue; // validated on the host for host pointers; never write out of bounds
        const uint8_t* h = digests + 32 * i;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const uint32_t bit_to_set = (((uint32_t)h[2 * j] << 8) | h[2 * j + 1]) & 0x07ffu; // big-endian 16-bit word, low 11 bits
            const uint32_t bit_index = 0x07ffu - bit_to_set;
            const uint32_t byte_index = bit_index >> 3;
            const uint32_t in_byte = 1u << (7 - (bit_index & 7));
            atomicOr(&blooms[64 * b + (byte_index >> 2)], in_byte << (8 * (byte_index & 3)));
        }
    }
}

extern "C" int phant_gpu_logs_bloom(phant_gpu_ctx* ctx, const uint8_t* items, const uint64_t* item_off, const uint32_t* bloom_of_item,
                                    uint64_t n_items, uint64_t n_blooms, uint8_t* blooms)
{
    if (!ctx || (n_blooms && !blooms) || (n_items && (!item_off || !bloom_of_item))) return PHANT_GPU_E_INVALID;
    if (n_blooms == 0) return n_items ? PHANT_GPU_E_INVALID : PHANT_GPU_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const bool dev = ctx->flags & PHANT_GPU_FLAG_DEVICE_PTRS;
    const uint8_t* d_items = items; const uint64_t* d_ioff = item_off; const uint32_t* d_map = bloom_of_item;
    uint32_t* d_blooms = (uint32_t*)blooms;
    uint64_t total = 0;
    if (!dev) {
        if (n_items) {
            if (int rc = check_offsets_host(item_off, n_items, &total)) return rc;
            if (total && !items) return PHANT_GPU_E_INVALID;
            for (uint64_t i = 0; i < n_items; ++i) if (bloom_of_item[i] >= n_blooms) return PHANT_GPU_E_INVALID;
        }
        if (int rc = ctx->d_msgs.reserve(ctx, total + 64)) return rc;
        if (int rc = ctx->d_off.reserve(ctx, 8 * (n_items + 1))) return rc;
        if (int rc = ctx->d_index.reserve(ctx, 4 * (n_items + 1))) return rc;
        if (int rc = ctx->d_out.reserve(ctx, 256 * n_blooms)) return rc;
        if (total) CU(cudaMemcpyAsync(ctx->d_msgs.ptr, items, total, cudaMemcpyHostToDevice, s));
        if (n_items) {
            CU(cudaMemcpyAsync(ctx->d_off.ptr, item_off, 8 * (n_items + 1), cudaMemcpyHostToDevice, s));
            CU(cudaMemcpyAsync(ctx->d_index.ptr, bloom_of_item, 4 * n_items, cudaMemcpyHostToDevice, s));
        }
        ctx->stats.h2d_bytes += total + 12 * n_items + 8;
        d_items = (const uint8_t*)ctx->d_msgs.ptr; d_ioff = (const uint64_t*)ctx->d_off.ptr; d_map = (const uint32_t*)ctx->d_index.ptr;
        d_blooms = (uint32_t*)ctx->d_out.ptr;
    } else if (n_items) {
        CU(cudaMemcpyAsync(&total, item_off + n_items, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    CU(cudaMemsetAsync(d_blooms, 0, 256 * n_blooms, s));
    if (n_items) {
        if (int rc = ctx->d_digests.reserve(ctx, 32 * n_items + 32)) return rc;
        if (int rc = ctx->hash_csr(d_items, d_ioff, n_items, total, (uint8_t*)ctx->d_digests.ptr)) return rc;
        uint64_t blocks = (n_items + 255) / 256;
        const uint64_t cap = (uint64_t)keccak_num_sms(ctx->device) * 8;
        if (blocks > cap) blocks = cap;
        bloom_set_kernel<<<(unsigned)blocks, 256, 0, s>>>((const uint8_t*)ctx->d_digests.ptr, d_map, n_items, n_blooms, d_blooms);
        CU(cudaGetLastError());
        ctx->stats.launches++;
    }
    if (!dev) {
        CU(cudaMemcpyAsync(blooms, d_blooms, 256 * n_blooms, cudaMemcpyDeviceToHost, s));
        ctx->stats.d2h_bytes += 256 * n_blooms;
        CU(cudaStreamSynchronize(s));
    }
    return PHANT_GPU_OK;
}

// ------------------------------------------------------------------------------------------------
// synthetic witnesses (device pointers)
// ------------------------------------------------------------------------------------------------
namespace phant { uint64_t synth_c2_bytes_per_proof(uint32_t depth); }

static int c3_scans(phant_gpu_ctx* ctx, uint64_t seed, uint64_t first_index, uint64_t n)
{
    // per-proof node / byte counts, then exclusive scans with a trailing total (n+1 entries)
    if (int rc = ctx->d_tmp_a.reserve(ctx, 8 * (n + 1))) return rc;
    if (int rc = ctx->d_tmp_b.reserve(ctx, 8 * (n + 1))) return rc;
    if (int rc = ctx->d_scan_a.reserve(ctx, 8 * (n + 1))) return rc;
    if (int rc = ctx->d_scan_b.reserve(ctx, 8 * (n + 1))) return rc;
    CU(cudaMemsetAsync((uint64_t*)ctx->d_tmp_a.ptr + n, 0, 8, ctx->stream));
    CU(cudaMemsetAsync((uint64_t*)ctx->d_tmp_b.ptr + n, 0, 8, ctx->stream));
    CU(launch_synth_c3_sizes(ctx->stream, ctx->device, seed, first_index, n, (uint64_t*)ctx->d_tmp_a.ptr, (uint64_t*)ctx->d_tmp_b.ptr));
    ctx->stats.launches++;
    size_t temp = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, temp, (const uint64_t*)ctx->d_tmp_a.ptr, (uint64_t*)ctx->d_scan_a.ptr, (int64_t)(n + 1), ctx->stream));
    if (int rc = ctx->d_cub.reserve(ctx, temp)) return rc;
    CU(cub::DeviceScan::ExclusiveSum(ctx->d_cub.ptr, temp, (const uint64_t*)ctx->d_tmp_a.ptr, (uint64_t*)ctx->d_scan_a.ptr, (int64_t)(n + 1), ctx->stream));
    CU(cub::DeviceScan::ExclusiveSum(ctx->d_cub.ptr, temp, (const uint64_t*)ctx->d_tmp_b.ptr, (uint64_t*)ctx->d_scan_b.ptr, (int64_t)(n + 1), ctx->stream));
    return PHANT_GPU_OK;
}

extern "C" int phant_gpu_synth_sizes(phant_gpu_ctx* ctx, int which, uint64_t seed, uint64_t first_index, uint64_t n, uint32_t depth,
                                     uint64_t* total_nodes, uint64_t* total_bytes)
{
    if (!ctx || !total_nodes || !total_bytes) return PHANT_GPU_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    if (which == 2) {
        if (depth < 2 || depth > 64) return PHANT_GPU_E_INVALID;
        *total_nodes = n * depth;
        *total_bytes = n * synth_c2_bytes_per_proof(depth);
        return PHANT_GPU_OK;
    }
    if (which != 3) return PHANT_GPU_E_INVALID;
    *total_nodes = *total_bytes = 0;
    if (n == 0) return PHANT_GPU_OK;
    if (int rc = c3_scans(ctx, seed, first_index, n)) return rc;
    CU(cudaMemcpyAsync(total_nodes, (uint64_t*)ctx->d_scan_a.ptr + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(total_bytes, (uint64_t*)ctx->d_scan_b.ptr + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return PHANT_GPU_OK;
}

extern "C" int phant_gpu_synth(phant_gpu_ctx* ctx, int which, uint64_t seed, uint64_t first_index, uint64_t n, uint32_t depth,
                               int corrupt, uint8_t* nodes, uint64_t* node_off, uint64_t* proof_first, uint8_t* keys32, uint8_t* roots32)
{
    if (!ctx || !nodes || !node_off || !proof_first || !keys32 || !roots32) return PHANT_GPU_E_INVALID;
    if (n == 0) return PHANT_GPU_OK;
    CU(cudaSetDevice(ctx->device));
    if (which == 2) {
        if (depth < 2 || depth > 64) return PHANT_GPU_E_INVALID;
        CU(launch_synth_c2(ctx->stream, ctx->device, seed, first_index, n, depth, corrupt, nodes, node_off, proof_first, keys32, roots32));
        ctx->stats.launches++;
    } else if (which == 3) {
        if (int rc = c3_scans(ctx, seed, first_index, n)) return rc;
        CU(cudaMemcpyAsync(proof_first, ctx->d_scan_a.ptr, 8 * (n + 1), cudaMemcpyDeviceToDevice, ctx->stream));
        CU(launch_synth_c3(ctx->stream, ctx->device, seed, first_index, n, corrupt, (const uint64_t*)ctx->d_scan_a.ptr,
                           (const uint64_t*)ctx->d_scan_b.ptr, nodes, node_off, keys32, roots32));
        ctx->stats.launches++;
    } else {
        return PHANT_GPU_E_INVALID;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return PHANT_GPU_OK;
}
