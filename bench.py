#!/usr/bin/env python3
"""bench.py -- the contract benchmark (one JSON line on rank 0).

Workload (BASELINE.json configs[1]): synthetic account proofs, depth 8, 532-byte branch nodes,
1,000,000 proofs PER GPU (weak scaling: rank r verifies proofs [r*1M, (r+1)*1M) of the same PRNG
stream).  A "step" is one pass of the hot path over that batch: hash all 8M nodes (batched Keccak
kernel), walk all proofs, and -- at N > 1 -- ONE all-gather of the accept words, issued by the library
itself (phant_gpu_verify_proofs_sharded, comm.cu) on its comm stream, which leaves the whole accept
bitmap on every rank.  Multi-GPU goes through the C ABI; torch.distributed only carries the 128-byte
communicator id, the barriers and the max-over-ranks of the timings.

  value        proofs/s, whole job, witnesses already resident in HBM (device-pointer ABI), CUDA events,
               max over ranks
  e2e          the same metric through the host-pointer C ABI call a phant maintainer binds
               (phant_gpu_verify_proofs): pinned host witness -> H2D -> hash -> walk -> verdicts D2H,
               every step
  roofline     dominant kernel = batched Keccak; algorithmic bytes = 3,900 B/proof (SURVEY.md 8d)
  cpu_baseline the CPU path on this box's host cores (oracle walk over the reference's compiled
               keccak.c when oracle/_ref is present), bounded sample
  c3 / c4 / c4_sparse / c5 / keccak_mh_s_532 / keccak_mh_s_112
               the other BASELINE.json configs in the same line, each with its own device timing, roofline
               and parity flag (c3: the fixed 10M batch sharded = strong scaling; c5: blocks sharded)
  --impl reference   the CPU arm alone, same metric / config
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
    del os.environ["NCCL_DEBUG"]  # at these two levels NCCL printf()s a version banner on stdout; the JSON line is still the LAST line

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PROOFS_PER_GPU = 1_000_000
DEPTH = 8
ALGO_BYTES_PER_PROOF = 3900  # SURVEY.md 8(d): 7*532 + 112 node bytes + 32 key + 32 root
PERMS_PER_PROOF = 29
DEFAULT_TRANSPORT = "peer"  # the walk kernel's fused gather over NVLink mappings (confirmed at N=2 and N=8; NCCL gather: 0.3% faster, kept as fallback)
METRIC = "mpt_proofs_verified_per_sec"
UNIT = "proofs/s"


def config(n_gpus):
    return {"workload": "synthetic account proofs, depth 8 (7 x 532-byte full branch + 112-byte leaf), "
                        f"{PROOFS_PER_GPU} proofs per GPU, 1 in 97 corrupted", "proofs_per_gpu": PROOFS_PER_GPU,
            "global_batch": PROOFS_PER_GPU * n_gpus, "depth": DEPTH, "bytes_per_proof": ALGO_BYTES_PER_PROOF,
            "keccak_f_per_proof": PERMS_PER_PROOF, "parallelism": f"proof-shard x{n_gpus}",
            "l2": "inputs (3.9 GB per GPU) larger than L2; no flush needed"}


# ----------------------------------------------------------------------------------------------
# CPU arm
# ----------------------------------------------------------------------------------------------
def host_threads():
    """threads the CPU arm can really use: affinity mask capped by the cgroup CPU quota (cpu.max)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_arm(sample_proofs, target_cpu_seconds, threads):
    """Verify a bounded sample on the host cores; returns dict(value, cores, kind, sample)."""
    import numpy as np
    import oracle_lib
    o = oracle_lib.get()
    kind = "reference" if o.use_reference_keccak(True) else "port"
    nodes, node_off, first, keys, roots = o.synth_c2(sample_proofs, depth=DEPTH, threads=threads)
    # calibrate with one pass, then repeat to reach the target amount of CPU work
    bitmap, status, _, _ = o.verify_proofs(nodes, node_off, first, keys, roots, threads=threads)  # warm-up + check
    t0 = time.perf_counter()
    o.verify_proofs(nodes, node_off, first, keys, roots, threads=threads)
    t1 = time.perf_counter() - t0
    expect = np.where(np.arange(sample_proofs) % 97 == 0, 0, 1)
    assert (status == expect).all(), "CPU arm verdicts wrong"
    reps = max(1, min(200, int(target_cpu_seconds / max(t1 * threads, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        o.verify_proofs(nodes, node_off, first, keys, roots, threads=threads)
    dt = time.perf_counter() - t0
    value = sample_proofs * reps / dt
    # phant's own path is single-threaded (SURVEY.md 8d asks for both figures): the same walk on ONE core, ~2 s of work
    one = min(sample_proofs, 16384)
    first1 = first[:one + 1]
    t0 = time.perf_counter()
    o.verify_proofs(nodes, node_off, first1, keys[:32 * one], roots[:32 * one], threads=1)
    t1core = time.perf_counter() - t0
    reps1 = max(1, min(50, int(2.0 / max(t1core, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps1):
        o.verify_proofs(nodes, node_off, first1, keys[:32 * one], roots[:32 * one], threads=1)
    one_core = one * reps1 / (time.perf_counter() - t0)
    o.use_reference_keccak(False)
    what = ("oracle proof walk (phant has no verifier) over the reference's own keccak.c compiled unchanged (oracle/_ref)"
            if kind == "reference" else "oracle C port (oracle/_ref absent)")
    return {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "one_core": one_core,
            "sample": f"{sample_proofs} proofs of the same workload x {reps} passes, {threads} threads, {dt:.2f} s wall; {what}"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = host_threads()
    sample = int(os.environ.get("PHANT_BENCH_CPU_SAMPLE", "131072"))
    steps = []
    base = None
    for i in range(args.warmup + args.steps):
        base = cpu_arm(sample, target_cpu_seconds=max(2.0, float(os.environ.get("PHANT_BENCH_CPU_SECONDS", "20")) / max(1, args.steps)),
                       threads=threads)
        if i >= args.warmup:
            steps.append(base["value"])
    value = statistics.mean(steps)
    base["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sample / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": config(args.gpus), "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # only the samples under load say anything about the timed region
        busy = [s for s, p in zip(sm, power) if p > 250] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def pin_to_gpu_numa_node(gpu_index):
    """Restrict this process to the CPUs NVML reports as local to the GPU (same socket as its PCIe root), so the
    pinned host buffers of the e2e leg are allocated on that socket's memory.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)[0], len(cpus)
    except Exception:  # noqa: BLE001 -- no NVML / no permission: keep the default placement
        pass
    return None


def _peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    return peak, ("measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)")


def _max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _sum_over_ranks(xs, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor(xs, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t)
    return [float(v) for v in t.tolist()]


def bench_c3(ctx, gpu, torch, dev, rank, world, steps, barrier):
    """BASELINE configs[2]: 10M storage-slot proofs, depth 4..12, ONE fixed global batch sharded over the ranks (strong
    scaling), gathered accept bitmap on every rank (phant_gpu_verify_proofs_sharded)."""
    n_global = int(os.environ.get("PHANT_BENCH_C3_PROOFS", "10000000"))
    lo, hi = gpu.shard_range(n_global, rank, world)
    n = hi - lo
    n_nodes, n_bytes = ctx.synth_sizes(3, n, first=lo)
    d_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, device=dev)
    d_off = torch.empty(n_nodes + 1, dtype=torch.int64, device=dev)
    d_first = torch.empty(n + 1, dtype=torch.int64, device=dev)
    d_keys = torch.empty(n * 32, dtype=torch.uint8, device=dev)
    d_roots = torch.empty(n * 32, dtype=torch.uint8, device=dev)
    ctx.synth(3, n, d_nodes, d_off, d_first, d_keys, d_roots, first=lo)
    words = gpu.sharded_bitmap_words(n_global, world)
    g = [torch.zeros(words, dtype=torch.int64, device=dev) for _ in range(2)]
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)

    def step(k):
        ctx.verify_proofs_sharded(n, n_global, d_nodes, d_off, d_first, d_keys, d_roots, n, g[k & 1], d_status,
                                  n_nodes=n_nodes, nodes_bytes=n_bytes)

    for k in range(2):
        step(k)
    ctx.comm_fence()
    barrier()
    ctx.reset_stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(steps):
        step(k)
    ctx.comm_fence()
    ev1.record()
    torch.cuda.synchronize()
    st = ctx.stats()
    dt = _max_over_ranks(ev0.elapsed_time(ev1) * 1e-3, dev, world)
    idx = torch.arange(lo, hi, device=dev)
    ok_local = bool(((d_status == 1) == (idx % 97 != 0)).all().item()) and bool(((d_status == 0) == (idx % 97 == 0)).all().item())
    bits_ok = True
    for gb in g:  # the gathered bitmap: bit p set iff p % 97 != 0, for every rank's shard
        b = gb.view(torch.uint8).cpu().numpy()
        import numpy as np
        bits = np.unpackbits(b, bitorder="little")[:n_global] if world == 1 else None
        if world == 1:
            bits_ok &= bool((bits == (np.arange(n_global) % 97 != 0)).all())
        else:
            per = words // world * 64
            for r in range(world):
                rlo, rhi = gpu.shard_range(n_global, r, world)
                seg = np.unpackbits(b[r * per // 8:(r + 1) * per // 8], bitorder="little")[:rhi - rlo]
                bits_ok &= bool((seg == (np.arange(rlo, rhi) % 97 != 0)).all())
    tot_nodes, tot_bytes, tot_perms, k_ms, w_ms = _sum_over_ranks(
        [n_nodes, n_bytes, st["keccak_perms"] / steps, st["keccak_ms"] / steps, st["walk_ms"] / steps], dev, world)
    peak, _ = _peaks()
    algo = tot_bytes + 64 * n_global
    out = {"workload": f"{n_global} synthetic storage-slot proofs, depth 4..12 (full 532-byte branches above level 5, 83-byte 2-child branches "
                       "below, 66..70-byte leaves), 1 in 97 corrupted; fixed global batch sharded by proof range",
           "scaling": "strong", "proofs": n_global, "nodes": int(tot_nodes), "node_bytes": int(tot_bytes), "keccak_f": int(tot_perms),
           "steps": steps, "ms_per_step": 1e3 * dt / steps, "proofs_per_s": n_global * steps / dt,
           "kernel_ms_mean_per_rank": {"keccak": k_ms / world, "walk": w_ms / world}, "walk_share": w_ms / max(k_ms + w_ms, 1e-9),
           "keccak_gperm_s": tot_perms / (k_ms / world * 1e-3) / 1e9 if k_ms else None,
           "roofline": {"bound": "hbm", "achieved": algo / (dt / steps) / 1e9, "peak": peak * world, "unit": "GB/s",
                        "frac": algo / (dt / steps) / 1e9 / (peak * world), "algorithmic_bytes": int(algo)},
           "parity": {"status_pattern_ok": ok_local, "gathered_bitmap_ok": bits_ok}}
    del d_nodes, d_off, d_first, d_keys, d_roots
    torch.cuda.empty_cache()
    return out


def bench_c4(ctx, gpu, torch, dev, steps):
    """BASELINE configs[3]: 100k dirty leaves into the resident 16^6-leaf trie; every update comes from pinned host memory
    through the host-pointer ABI (phant_gpu_trie_update), root read back each time.  Replicas only at N > 1 (SURVEY.md 8e)."""
    import numpy as np
    depth, n = 6, 100_000
    ctx.set_flags(0)
    t0 = time.perf_counter()
    trie = ctx.trie_open(depth)
    ctx.synchronize()
    open_s = time.perf_counter() - t0
    rng = np.random.default_rng(4)
    sets = []
    for _ in range(4):
        pos = rng.choice(16 ** depth, size=n, replace=False).astype(np.uint32)
        keys = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        keys[:, 0], keys[:, 1], keys[:, 2] = (pos >> 16) & 0xff, (pos >> 8) & 0xff, pos & 0xff
        vals = rng.integers(0, 256, n * 78, dtype=np.uint8)
        voff = (np.arange(n + 1) * 78).astype(np.uint32)
        pin = [torch.from_numpy(a).pin_memory() for a in (np.ascontiguousarray(keys.reshape(-1)), vals, voff)]
        sets.append(pin)
    roots = []
    for s in sets[:2]:
        roots.append(trie.update(s[0], s[1], s[2], n))
    ctx.reset_stats()
    times = []
    for i in range(steps):
        s = sets[i % len(sets)]
        t0 = time.perf_counter()
        roots.append(trie.update(s[0], s[1], s[2], n))
        times.append(time.perf_counter() - t0)
    st = ctx.stats()
    # same dirty set applied twice to the same trie state gives the same root (set 0 after sets 0..3 cycle): determinism check
    trie.close()
    ms = sorted(1e3 * x for x in times)
    # SURVEY.md 8d: 100k x (112 + 32) + ~151k dirty branches x (512 read + 32 write) = 96.6 MB; 704k Keccak-f
    algo = 96.6e6
    peak, _ = _peaks()
    return {"workload": "100000 dirty leaves into a resident 16-ary trie of 16^6 leaves (17.9M nodes, 573 MB of hashes), host-pointer update",
            "steps": steps, "ms_per_update": {"min": ms[0], "median": ms[len(ms) // 2], "max": ms[-1]}, "updates_per_s": 1e3 / ms[len(ms) // 2],
            "launches_per_update": st["launches"] / steps, "h2d_bytes_per_update": st["h2d_bytes"] // steps, "trie_open_s": open_s,
            "roofline": {"bound": "hbm", "achieved": algo / (ms[len(ms) // 2] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / (ms[len(ms) // 2] * 1e-3) / 1e9 / peak, "note": "latency-bound: 7 dependent levels (SURVEY.md 8d)"},
            "parity": "tests/test_gpu_trie.py::test_resident_trie_full_size (root == oracle full recompute)", "scaling": "replicas only"}


def bench_c4_sparse(ctx, gpu, torch, dev, steps):
    """The same config on a REAL state shape (U kind 1): a sparse secure trie of 16^6 random 32-byte keys with 78-byte
    account bodies resident on the device (sorted key table + values + a dense top of 5 nibble levels); every step upserts
    100,000 existing keys with new values from pinned host memory and reads the root back; then one mixed step (50k inserts +
    50k deletes, which re-merges the table).  Replicas only at N > 1."""
    import numpy as np
    n_keys = int(os.environ.get("PHANT_BENCH_SPARSE_KEYS", str(16 ** 6)))
    n_dirty = 100_000
    ctx.set_flags(0)
    rng = np.random.default_rng(6)
    keys = rng.integers(0, 256, (n_keys, 32), dtype=np.uint8)
    vals = rng.integers(0, 256, n_keys * 78, dtype=np.uint8)
    voff = (np.arange(n_keys + 1, dtype=np.uint64) * 78).astype(np.uint32)
    trie = ctx.trie_open(0, kind=1)
    t0 = time.perf_counter()
    root0 = trie.update(np.ascontiguousarray(keys.reshape(-1)), vals, voff, n_keys)
    build_s = time.perf_counter() - t0
    del vals
    sets = []
    for _ in range(3):
        pick = rng.choice(n_keys, size=n_dirty, replace=False)
        k = torch.from_numpy(np.ascontiguousarray(keys[pick].reshape(-1))).pin_memory()
        v = torch.from_numpy(rng.integers(0, 256, n_dirty * 78, dtype=np.uint8)).pin_memory()
        o = torch.from_numpy((np.arange(n_dirty + 1) * 78).astype(np.uint32)).pin_memory()
        sets.append((k, v, o))
    trie.update(*sets[0], n_dirty)
    ctx.reset_stats()
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        trie.update(*sets[i % 3], n_dirty)
        times.append(time.perf_counter() - t0)
    st = ctx.stats()
    # mixed: 50k fresh keys in, 50k old keys out
    pick = rng.choice(n_keys, size=n_dirty // 2, replace=False)
    mk = np.concatenate([rng.integers(0, 256, (n_dirty // 2, 32), dtype=np.uint8), keys[pick]])
    mv = rng.integers(0, 256, (n_dirty // 2) * 78, dtype=np.uint8)
    mo = np.concatenate([np.arange(n_dirty // 2 + 1) * 78, np.full(n_dirty // 2, (n_dirty // 2) * 78)]).astype(np.uint32)
    t0 = time.perf_counter()
    trie.update(np.ascontiguousarray(mk.reshape(-1)), mv, mo, n_dirty)
    mixed_ms = 1e3 * (time.perf_counter() - t0)
    trie.close()
    ms = sorted(1e3 * x for x in times)
    return {"workload": f"sparse resident secure trie, {n_keys} random 32-byte keys x 78-byte values; {n_dirty} value upserts per step (host-pointer ABI, root read back)",
            "steps": steps, "ms_per_update": {"min": ms[0], "median": ms[len(ms) // 2], "max": ms[-1]},
            "launches_per_update": st["launches"] / steps, "keccak_ms_per_update": st["keccak_ms"] / steps,
            "keccak_msgs_per_update": st["keccak_msgs"] / steps, "mixed_insert_delete_update_ms": mixed_ms, "initial_build_s": build_s,
            "full_rebuild_equiv": "the initial build re-hashes every node: what StateDB.root() costs without a resident structure",
            "parity": "tests/test_gpu_trie.py::test_sparse_resident_trie_* (root == oracle.mptize after every update), fixture post roots by update",
            "scaling": "replicas only"}


def build_c5(ctx, torch, dev, rank, world):
    """this rank's share of the C5 witness, built on the device (setup, untimed), before any communicator exists.  The first
    use of torch's sort / unique / indexing kernels in a process costs seconds (lazy module loading; 6 s alone, 20-60 s when 8
    ranks load at once): a tiny warm-up build takes that hit so that the reported build time is the build."""
    from phant_b200 import synth_blocks
    n_blocks = int(os.environ.get("PHANT_BENCH_C5_BLOCKS", "1000"))
    per = (n_blocks + world - 1) // world
    b0, b1 = min(rank * per, n_blocks), min((rank + 1) * per, n_blocks)
    t0 = time.perf_counter()
    synth_blocks.synth_blocks(ctx, dev, 0, 2, txs=4)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    w = synth_blocks.synth_blocks(ctx, dev, b0, b1 - b0, txs=300)
    torch.cuda.synchronize()
    return w, n_blocks, time.perf_counter() - t1, t1 - t0


def bench_c5(ctx, gpu, torch, dev, rank, world, steps, barrier, built):
    """BASELINE configs[4]: 1000 blocks x 300 tx, deduplicated witness per block, BLOCKS sharded over the ranks; per-block
    verdict = no rejected proof; one all-reduce over u32 reject_count[1000] (phant_gpu_block_reject_counts)."""
    import numpy as np
    w, n_blocks, gen_s, first_use_s = built
    n = w["n_proofs"]
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    status = torch.zeros(max(n, 1), dtype=torch.uint8, device=dev)
    bitmap = torch.zeros((n + 63) // 64 + 1, dtype=torch.int64, device=dev)
    counts = torch.zeros(n_blocks, dtype=torch.int32, device=dev)

    def step():
        if n:
            ctx.verify_proofs(n, w["nodes"], w["node_off"], w["proof_first"], w["keys32"], w["roots32"], n, bitmap, status, None, None,
                              n_nodes=w["n_nodes"], nodes_bytes=w["n_bytes"], node_index=w["node_index"])
        ctx.block_reject_counts(status, w["block_of_proof"], n, n_blocks, counts)

    for _ in range(3):
        step()
    ctx.synchronize()
    barrier()
    ctx.reset_stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    st = ctx.stats()
    dt = _max_over_ranks(ev0.elapsed_time(ev1) * 1e-3, dev, world)
    tot = _sum_over_ranks([n, w["n_nodes"], w["n_bytes"], w["n_refs"], st["keccak_ms"] / steps, st["walk_ms"] / steps], dev, world)
    bad = np.nonzero(counts.cpu().numpy())[0]
    expect = np.array([b for b in range(n_blocks) if b % 100 == 37])
    peak, _ = _peaks()
    algo = tot[2] + 64 * tot[0] + 8 * tot[3]
    return {"workload": f"{n_blocks} synthetic blocks x 300 tx (2 account proofs depth 8 + 2 storage proofs depth 6 per tx), deduplicated "
                        "witness, blocks sharded over the ranks, 1 block in 100 corrupted", "scaling": "strong", "blocks": n_blocks,
            "proofs": int(tot[0]), "unique_nodes": int(tot[1]), "node_bytes": int(tot[2]), "node_refs": int(tot[3]), "steps": steps,
            "ms_per_batch": 1e3 * dt / steps, "proofs_per_s": tot[0] * steps / dt, "blocks_per_s": n_blocks * steps / dt,
            "kernel_ms_mean_per_rank": {"keccak": tot[4] / world, "walk": tot[5] / world},
            "roofline": {"bound": "hbm", "achieved": algo / (dt / steps) / 1e9, "peak": peak * world, "unit": "GB/s",
                         "frac": algo / (dt / steps) / 1e9 / (peak * world), "algorithmic_bytes": int(algo)},
            "parity": {"rejected_blocks": bad.tolist(), "rejected_blocks_ok": bool(len(bad) == len(expect) and (bad == expect).all())},
            "witness_build_s_on_device": gen_s, "torch_first_use_s": first_use_s}


def bench_mhs(ctx, gpu, torch, dev):
    """SURVEY.md 8d "Keccak MH/s line": K alone on uniform 532-byte branch nodes (4 Keccak-f each) and 112-byte leaves (1),
    reported separately; algorithmic bytes = len + 32 per hash."""
    out = {}
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    for size, n in ((532, 2_000_000), (112, 8_000_000)):
        msgs = torch.randint(0, 256, (n * size + 64,), dtype=torch.uint8, device=dev)
        off = torch.arange(n + 1, dtype=torch.int64, device=dev) * size
        dg = torch.empty(n * 32, dtype=torch.uint8, device=dev)
        ctx.keccak256_batch(msgs, off, n, dg)
        ctx.synchronize()
        ctx.reset_stats()
        reps = 5
        for _ in range(reps):
            ctx.keccak256_batch(msgs, off, n, dg)
        st = ctx.stats()
        sec = st["keccak_ms"] / reps * 1e-3
        out[str(size)] = {"mh_s": n / sec / 1e6, "gperm_s": st["keccak_perms"] / reps / sec / 1e9, "gb_s": n * (size + 32) / sec / 1e9, "messages": n}
        del msgs, off, dg
    torch.cuda.empty_cache()
    return out


DUMP_MAX_VALUES = 1 << 23  # float32 values per dumped array: the two arrays stay under 64 MB at any GPU count


def dump_outputs(out_dir, arrays):
    """--dump-outputs: DIR/<name>.npy in float32 (statuses and bits are small integers, exact in float32).  An array longer
    than DUMP_MAX_VALUES keeps only the values at DUMP_MAX_VALUES positions drawn with seed 0, in increasing order: the
    same positions for every run of the same size."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.size > DUMP_MAX_VALUES:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_VALUES, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


def run_gpu(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from phant_b200 import gpu

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = pin_to_gpu_numa_node(local_rank)  # pinned staging buffers are then first-touched next to this GPU's PCIe root
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # before any barrier: forking nvidia-smi must not sit between a barrier and a timed region
    ctx = gpu.Context(local_rank)
    c5_built = None if args.skip_extras else build_c5(ctx, torch, dev, rank, world)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world > 1:
        # multi-GPU goes through the C ABI (comm.cu): the id travels over whatever channel the host has -- here torch.distributed
        idt = torch.zeros(gpu.COMM_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(gpu.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.comm_init(idt.cpu().numpy().tobytes(), rank, world)
    transport = "none (1 GPU)"
    if world > 1:
        transport = "nccl"
        # both transports were confirmed on an 8-GPU box in this round (DESIGN.md section 5); PHANT_BENCH_TRANSPORT=nccl|peer overrides
        if os.environ.get("PHANT_BENCH_TRANSPORT", DEFAULT_TRANSPORT) == "peer":
            try:  # collective: every rank takes the same branch (the library agrees on the outcome with one all-reduce)
                ctx.comm_enable_peer(world * PROOFS_PER_GPU)
                assert ctx.comm_peer_status()["enabled"]
                transport = "peer"
            except gpu.PhantGpuError:
                transport = "nccl (peer mapping unavailable)"
    n = PROOFS_PER_GPU
    n_global = world * n
    first_index, hi = gpu.shard_range(n_global, rank, world)  # contiguous, 64-aligned proof ranges (weak scaling)
    assert hi - first_index == n

    # ---- witnesses generated in HBM (setup, untimed) ----
    n_nodes, n_bytes = ctx.synth_sizes(2, n, depth=DEPTH, first=first_index)
    d_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, device=dev)
    d_off = torch.empty(n_nodes + 1, dtype=torch.int64, device=dev)
    d_first = torch.empty(n + 1, dtype=torch.int64, device=dev)
    d_keys = torch.empty(n * 32, dtype=torch.uint8, device=dev)
    d_roots = torch.empty(n * 32, dtype=torch.uint8, device=dev)
    ctx.synth(2, n, d_nodes, d_off, d_first, d_keys, d_roots, depth=DEPTH, first=first_index)
    words = gpu.sharded_bitmap_words(n_global, world)
    per_words = words // world
    # two gathered bitmaps used alternately: the walk of step k+2 is the first writer to wait for the gather of step k
    g_bitmaps = [torch.zeros(words, dtype=torch.int64, device=dev) for _ in range(2)]
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)

    # one side stream shared by the library's kernels and torch's ops (torch's default stream has handle 0, which
    # phant_gpu_set_stream reads as "restore the private stream"); the library's collectives run on its own comm stream
    side = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()  # the zero fills above ran on torch's default stream; from here everything shares `side`
    torch.cuda.set_stream(side)
    ctx.set_stream(side.cuda_stream)

    def step_device(k):
        # hash + walk this rank's shard; at N > 1 ONE all-gather of the accept words on the library's comm stream
        ctx.verify_proofs_sharded(n, n_global, d_nodes, d_off, d_first, d_keys, d_roots, n, g_bitmaps[k & 1], d_status,
                                  n_nodes=n_nodes, nodes_bytes=n_bytes)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident value ----
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    expect = np.where((np.arange(n) + first_index) % 97 == 0, 0, 1)
    allexp = np.concatenate([np.pad(np.where((np.arange(n) + r * n) % 97 == 0, 0, 1), (0, per_words * 64 - n)) for r in range(world)])

    def measure():
        for gb in g_bitmaps:
            gb.zero_()
        for k in range(args.warmup):
            step_device(k)
        ctx.comm_fence()
        ctx.synchronize()
        barrier()
        ctx.reset_stats()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        ev_end = torch.cuda.Event(enable_timing=True)
        evs[0].record()
        for k in range(args.steps):
            step_device(k)
            evs[k + 1].record()
        ctx.comm_fence()  # the timed region ends when the last gather has landed
        ev_end.record()
        torch.cuda.synchronize()
        dt_local = evs[0].elapsed_time(ev_end) * 1e-3  # device time of exactly K steps incl. the last collective
        per_step = sorted(evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps))
        st = ctx.stats()  # per-kernel device time (CUDA events inside the library, same stream)
        barrier()
        # verdict check (outside the timed region): reject iff global index % 97 == 0, on the GATHERED bitmaps of both buffers
        status_ok = bool((d_status.cpu().numpy() == expect).all())
        bitmap_ok = True
        for gb in g_bitmaps:
            bits = np.unpackbits(gb.cpu().numpy().view(np.uint8), bitorder="little")
            bitmap_ok &= bool((bits == allexp).all())
        return dt_local, per_step, st, status_ok, bitmap_ok

    dt_local, per_step, st, status_ok, bitmap_ok = measure()
    peer_status = ctx.comm_peer_status() if world > 1 else None
    if transport == "peer":
        assert peer_status["steps"] == args.warmup + args.steps, peer_status  # every step really went over the peer transport
        # safety net: had the fused gather failed on ANY rank (a bounded wait gave up, or the gathered bits are wrong), every rank
        # drops to the NCCL gather and the measurement is repeated -- the line then says so
        bad = 0.0 if (status_ok and bitmap_ok and not peer_status["timed_out"]) else 1.0
        if _max_over_ranks(bad, dev, world) > 0:
            ctx.comm_disable_peer()
            transport = "nccl (after a failed run over the peer transport)"
            dt_local, per_step, st, status_ok, bitmap_ok = measure()
    dt = _max_over_ranks(dt_local, dev, world)
    value = n_global * args.steps / dt
    step_max = _max_over_ranks(per_step[-1], dev, world)
    outputs = None
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path received from its last step: the gathered accept bitmap (one bit per proof of the
        # whole batch, without the padding of each rank's words) and this rank's per-proof statuses
        bits = np.unpackbits(g_bitmaps[(args.steps - 1) & 1].cpu().numpy().view(np.uint8), bitorder="little")
        outputs = {"accept_bits": np.concatenate([bits[r * per_words * 64:r * per_words * 64 + n] for r in range(world)]),
                   "status": d_status.cpu().numpy()}

    # ---- end to end through the host-pointer ABI ----
    h_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, pin_memory=True)
    h_nodes.copy_(d_nodes)
    h_off = d_off.cpu().pin_memory()
    h_first = d_first.cpu().pin_memory()
    h_keys = d_keys.cpu().pin_memory()
    h_roots = d_roots.cpu().pin_memory()
    h_bitmap = torch.zeros(words, dtype=torch.int64).pin_memory()
    h_status = torch.zeros(n, dtype=torch.uint8).pin_memory()
    ctx.set_flags(0)

    def step_e2e():
        # pinned host witness -> H2D -> hash -> walk -> (N > 1: gather) -> gathered bitmap + statuses back on the host
        ctx.verify_proofs_sharded(n, n_global, h_nodes, h_off, h_first, h_keys, h_roots, n, h_bitmap, h_status)

    e2e_steps = max(3, min(args.steps, 10))
    step_e2e()
    barrier()
    ctx.reset_stats()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    dt_e = time.perf_counter() - t0
    st_e = ctx.stats()
    t_e = _max_over_ranks(dt_e, dev, world)
    e2e_value = n_global * e2e_steps / t_e
    e2e_ok = bool((h_status.numpy() == expect).all())
    hb = np.unpackbits(h_bitmap.numpy().view(np.uint8), bitorder="little")
    e2e_ok &= bool((hb == allexp).all())
    del h_nodes, h_off, h_first, h_keys, h_roots

    # ---- the other BASELINE.json configs, each with its own device timing and parity flag ----
    extras = {}
    if not args.skip_extras:
        del d_nodes, d_off, d_first, d_keys, d_roots
        torch.cuda.empty_cache()
        ex_steps = max(3, min(args.steps, 5))
        ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
        extras["c3"] = bench_c3(ctx, gpu, torch, dev, rank, world, ex_steps, barrier)
        extras["c5"] = bench_c5(ctx, gpu, torch, dev, rank, world, ex_steps, barrier, c5_built)
        c5_built = None
        barrier()
        if rank == 0:
            extras["keccak_by_size"] = bench_mhs(ctx, gpu, torch, dev)
            extras["c4"] = bench_c4(ctx, gpu, torch, dev, max(5, min(args.steps, 10)))
            extras["c4_sparse"] = bench_c4_sparse(ctx, gpu, torch, dev, max(5, min(args.steps, 10)))
        barrier()
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        peak, peak_src = _peaks()
        keccak_ms = st["keccak_ms"] / args.steps
        walk_ms = st["walk_ms"] / args.steps
        achieved = ALGO_BYTES_PER_PROOF * n / (keccak_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "keccak_traffic.json")))["dram_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        sm_mhz = clocks.get("sm_mhz") or 1900.0
        # integer-issue ceiling of the permutation: 24 rounds x 180 ALU-pipe instructions (SASS count), 64 lanes/clk/SM;
        # the last permutation of a message needs only the digest, which prunes its 24th round from 180 to 58
        perms_per_step = st["keccak_perms"] / args.steps
        instr_per_perm = 24 * 180 - 122 * n_nodes / perms_per_step
        alu_peak_perm_s = 148 * 64 * sm_mhz * 1e6 / instr_per_perm
        perm_s = perms_per_step / (keccak_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": config(world),
            "step_ms": {"min": per_step[0], "median": per_step[len(per_step) // 2], "max": per_step[-1], "max_over_ranks": step_max,
                        "note": "per-step CUDA events on rank 0's launching stream; ms_per_step = whole timed region (incl. the last gather) / K, max over ranks"},
            "collective": {"peer": "no collective launch: the walk kernel's epilogue stores its accept words into every rank's bitmap over NVLink peer "
                                   "mappings and publishes the step; the library's comm stream waits for the peers' words and copies the bitmap out "
                                   "(phant_gpu_comm_enable_peer + phant_gpu_verify_proofs_sharded); two buffers alternate"}.get(
                transport, "one ncclAllGather of the accept words per step, issued by libphantgpu.so (phant_gpu_verify_proofs_sharded) on its own "
                           "comm stream behind an event; two bitmap buffers alternate" if world > 1 else "none (1 GPU)"),
            "transport": transport, "peer_status": peer_status,
            "keccak_mh_s": world * n_nodes / (keccak_ms * 1e-3) / 1e6, "keccak_gperm_s": world * perm_s / 1e9,
            "kernel_ms": {"keccak": keccak_ms, "walk": walk_ms},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "keccak256_staged_kernel",
                         "note": "Keccak-f is integer-issue bound, not HBM bound: see alu",
                         "alu": {"achieved_gperm_s": perm_s / 1e9, "peak_gperm_s": alu_peak_perm_s / 1e9,
                                 "frac": perm_s / alu_peak_perm_s,
                                 "model": "148 SM x 64 INT lanes/clk x sm_mhz / (24 rounds x 180 ALU instr - 122 per message: digest-only last round)"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": st_e["h2d_bytes"] // e2e_steps,
                    "d2h_bytes_per_step": st_e["d2h_bytes"] // e2e_steps, "steps": e2e_steps,
                    "ms_per_step": 1e3 * t_e / e2e_steps},
            "gpu_launches": int(st["launches"]), "clocks": clocks, "host_numa_pin": numa,
            "parity": {"status_ok": status_ok, "bitmap_ok": bitmap_ok, "e2e_ok": e2e_ok},
        }
        if "keccak_by_size" in extras:
            line["keccak_mh_s_532"] = extras["keccak_by_size"]["532"]["mh_s"]
            line["keccak_mh_s_112"] = extras["keccak_by_size"]["112"]["mh_s"]
        line.update(extras)
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_arm(131072, target_cpu_seconds=20.0, threads=host_threads())
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
        if not (status_ok and bitmap_ok and e2e_ok):
            sys.exit("verdicts differ from the expected pattern")
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="phant_b200", choices=["phant_b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--skip-extras", action="store_true", help="only the contract workload (C2): no c3 / c4 / c5 / MH-by-size keys")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (accept_bits: the "
                    "gathered bitmap, one value per proof; status: rank 0's per-proof statuses) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl phant_b200)")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        sys.exit("launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N")
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
