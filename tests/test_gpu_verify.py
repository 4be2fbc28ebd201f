"""V: proof walk on the GPU vs the oracle (status, accept bitmap, value slice: bit-exact)."""
import numpy as np
import pytest

import oracle_lib
from helpers import secure_account_items
from test_oracle_proofs import batch_of, mutations

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from phant_b200 import gpu
    c = gpu.Context(0)
    yield c
    c.close()


def gpu_verify(ctx, nodes, node_off, first, keys, roots, flags=0):
    n = len(first) - 1
    bitmap = np.zeros((n + 63) // 64, np.uint64)
    status = np.full(n, 77, np.uint8)
    voff = np.zeros(n, np.uint64)
    vlen = np.zeros(n, np.uint32)
    ctx.set_flags(flags)
    ctx.verify_proofs(n, np.ascontiguousarray(nodes), node_off, first, np.ascontiguousarray(keys), np.ascontiguousarray(roots),
                      roots.size // 32, bitmap, status, voff, vlen)
    return bitmap, status, voff, vlen


def assert_same(ctx, oracle, proofs, flags=0):
    nodes, node_off, first, keys, roots = batch_of(proofs)
    want = oracle.verify_proofs(nodes, node_off, first, keys, roots)
    got = gpu_verify(ctx, nodes, node_off, first, keys, roots, flags)
    assert (got[1] == want[1]).all(), np.nonzero(got[1] != want[1])[0][:10]
    assert (got[0] == want[0]).all()
    present = want[1] == 1
    assert (got[2][present] == want[2][present]).all() and (got[3][present] == want[3][present]).all()
    return want[1]


@pytest.mark.parametrize("flags", [0, 1 << 4, 1 << 5])
def test_fixture_proofs_and_mutations(ctx, oracle, golden, flags):
    g = golden("fixture_states.json.gz")
    rng = np.random.default_rng(3)
    proofs = []
    for tkey, accounts in sorted(g["tables"].items())[:30]:
        if not accounts:
            continue
        items = secure_account_items(oracle.keccak256, oracle.mptize, accounts)
        trie = oracle.trie(items)
        root = trie.root()
        mine = [(trie.prove(k), k, root) for k, _ in items[:50]]
        for _ in range(4):
            k = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
            mine.append((trie.prove(k), k, root))
        proofs += mine
        for i in rng.choice(len(mine), size=min(4, len(mine)), replace=False):
            proofs += mutations(*mine[int(i)], rng)
    st = assert_same(ctx, oracle, proofs, flags)
    assert {0, 1, 2} <= set(st.tolist())


def test_embedded_and_empty(ctx, oracle):
    base = bytes(range(31))
    kv = sorted((base + bytes([b]), bytes([v])) for b, v in [(0x10, 1), (0x11, 2), (0x1f, 3), (0x20, 4), (0x77, 5)])
    trie = oracle.trie(kv)
    root = trie.root()
    proofs = [(trie.prove(k), k, root) for k, _ in kv]
    proofs += [(trie.prove(k), k, root) for k in [base + bytes([0x12]), base + bytes([0x30]), bytes([0xff]) + base]]
    rng = np.random.default_rng(5)
    for p in list(proofs[:5]):
        proofs += mutations(*p, rng)
    empty = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")
    proofs += [([], bytes(32), empty), ([], bytes(32), bytes(32))]
    assert_same(ctx, oracle, proofs)


def test_single_root_broadcast(ctx, oracle):
    rng = np.random.default_rng(8)
    keys = sorted(rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(300))
    trie = oracle.trie([(k, b"v" * 50) for k in keys])
    root = trie.root()
    proofs = [(trie.prove(k), k, root) for k in keys]
    nodes, node_off, first, keysa, _ = batch_of(proofs)
    roots = np.frombuffer(root, np.uint8)
    want = oracle.verify_proofs(nodes, node_off, first, keysa, roots)
    got = gpu_verify(ctx, nodes, node_off, first, keysa, roots)
    assert (got[1] == want[1]).all() and (want[1] == 1).all()


@pytest.mark.parametrize("which", [2, 3])
def test_device_synth_equals_oracle_synth(ctx, oracle, which):
    """phant_b200/csrc/synth.cu vs oracle/synth.c: byte-identical witnesses, then identical verdicts."""
    import torch
    n = 2000
    n_nodes, n_bytes = ctx.synth_sizes(which, n, depth=8, first=1000)
    d_nodes = torch.zeros(n_bytes + 64, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(n_nodes + 1, dtype=torch.int64, device="cuda")
    d_first = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    d_keys = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
    d_roots = torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()  # torch's fills run on torch's stream, the library on its own (non-blocking) one
    ctx.synth(which, n, d_nodes, d_off, d_first, d_keys, d_roots, depth=8, first=1000)
    o = oracle.synth_c2(n, depth=8, first=1000) if which == 2 else oracle.synth_c3(n, first=1000)
    assert n_bytes == int(o[1][-1]) and n_nodes == len(o[1]) - 1
    assert (d_nodes.cpu().numpy()[:n_bytes] == o[0][:n_bytes]).all()
    assert (d_off.cpu().numpy().astype(np.uint64) == o[1]).all()
    assert (d_first.cpu().numpy().astype(np.uint64) == o[2]).all()
    assert (d_keys.cpu().numpy() == o[3]).all() and (d_roots.cpu().numpy() == o[4]).all()
    want = oracle.verify_proofs(*o, threads=8)
    got = gpu_verify(ctx, *o)
    assert (got[1] == want[1]).all() and (got[0] == want[0]).all()
    expect = np.where((np.arange(n) + 1000) % 97 == 0, 0, 1)
    assert (got[1] == expect).all()


def test_full_size_c2_property(ctx):
    """BASELINE config: 1M account proofs, depth 8, generated and verified in HBM; reject iff index % 97 == 0."""
    import torch
    from phant_b200 import gpu
    n = 1_000_000
    n_nodes, n_bytes = ctx.synth_sizes(2, n, depth=8)
    assert n_bytes == n * 3836
    d_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n_nodes + 1, dtype=torch.int64, device="cuda")
    d_first = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_keys = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    d_roots = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    ctx.synth(2, n, d_nodes, d_off, d_first, d_keys, d_roots, depth=8)
    d_status = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_bitmap = torch.zeros((n + 63) // 64, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    ctx.verify_proofs(n, d_nodes, d_off, d_first, d_keys, d_roots, n, d_bitmap, d_status, None, None)
    ctx.synchronize()
    ctx.set_flags(0)
    st = d_status.cpu().numpy()
    expect = np.where(np.arange(n) % 97 == 0, 0, 1)
    assert (st == expect).all()
    bm = d_bitmap.cpu().numpy().view(np.uint64)
    bits = np.unpackbits(bm.view(np.uint8), bitorder="little")[:n]
    assert (bits == expect).all()


def test_host_pipeline_many_chunks_and_bad_csr(ctx, oracle):
    """host-pointer path crosses PCIe in chunks: 40k proofs (153 MB, so two chunks at the default 128 MB) must give the same
    verdicts as the oracle; corrupt CSR arrays must be refused with E_INVALID, not read out of bounds.  Many small chunks:
    test_gpu_fused_layout.py::test_chunked_host_path."""
    from phant_b200 import gpu
    n = 40_000
    o = oracle.synth_c2(n, depth=8, first=7)
    want = oracle.verify_proofs(*o, threads=8)
    got = gpu_verify(ctx, *o)
    assert (got[1] == want[1]).all() and (got[0] == want[0]).all()
    nodes, node_off, first, keys, roots = o
    bad_off = node_off.copy()
    bad_off[12345] = bad_off[12346] + 9          # not monotone
    with pytest.raises(gpu.PhantGpuError) as e:
        gpu_verify(ctx, nodes, bad_off, first, keys, roots)
    assert e.value.code == -1
    bad_first = first.copy()
    bad_first[20000] = first[-1] + 5              # beyond n_nodes
    with pytest.raises(gpu.PhantGpuError) as e:
        gpu_verify(ctx, nodes, node_off, bad_first, keys, roots)
    assert e.value.code == -1
    # and the context is still usable afterwards
    got = gpu_verify(ctx, *o)
    assert (got[1] == want[1]).all()


def test_deduplicated_block_witness(ctx, oracle):
    """config C5 shape: per-block virtual tries, distinct nodes stored once, chains are node-index lists; verdicts,
    bitmap and value slices must equal the oracle's, host-pointer and device-pointer paths alike."""
    import torch
    from phant_b200 import gpu
    w = oracle.synth_blocks(60, txs=50, first=0, threads=8)      # blocks 37 is corrupted
    n = w["n_proofs"]
    want = oracle.verify_proofs(w["nodes"], w["node_off"], w["proof_first"], w["keys32"], w["roots32"], threads=8, node_index=w["node_index"])
    assert w["n_refs"] > w["n_nodes"]                              # something is shared
    bitmap = np.zeros((n + 63) // 64, np.uint64)
    status = np.full(n, 77, np.uint8)
    voff = np.zeros(n, np.uint64)
    vlen = np.zeros(n, np.uint32)
    ctx.set_flags(0)
    ctx.verify_proofs(n, w["nodes"], w["node_off"], w["proof_first"], w["keys32"], w["roots32"], n, bitmap, status, voff, vlen,
                      n_nodes=w["n_nodes"], nodes_bytes=w["n_bytes"], node_index=w["node_index"])
    assert (status == want[1]).all() and (bitmap == want[0]).all()
    ok = want[1] == 1
    assert (voff[ok] == want[2][ok]).all() and (vlen[ok] == want[3][ok]).all()
    rej_blocks = set(w["block_of_proof"][status == 0].tolist())
    assert rej_blocks == {37}
    # device pointers
    d = {k: torch.from_numpy(v.view(np.int64) if v.dtype == np.uint64 else v).cuda() for k, v in w.items() if isinstance(v, np.ndarray)}
    d_status = torch.zeros(n, dtype=torch.uint8, device="cuda")
    d_bitmap = torch.zeros((n + 63) // 64, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    ctx.verify_proofs(n, d["nodes"], d["node_off"], d["proof_first"], d["keys32"], d["roots32"], n, d_bitmap, d_status, None, None,
                      n_nodes=w["n_nodes"], nodes_bytes=w["n_bytes"], node_index=d["node_index"])
    ctx.synchronize()
    ctx.set_flags(0)
    assert (d_status.cpu().numpy() == want[1]).all()
    # a node index out of range is refused, not dereferenced
    bad = w["node_index"].copy()
    bad[5] = w["n_nodes"] + 3
    with pytest.raises(gpu.PhantGpuError) as e:
        ctx.verify_proofs(n, w["nodes"], w["node_off"], w["proof_first"], w["keys32"], w["roots32"], n, bitmap, status, None, None,
                          n_nodes=w["n_nodes"], nodes_bytes=w["n_bytes"], node_index=bad)
    assert e.value.code == -1


def test_full_size_c3_property(ctx):
    """BASELINE config: 10M storage proofs, mixed depth 4..12 (28 GB of nodes in HBM); reject iff index % 97 == 0."""
    import torch
    from phant_b200 import gpu
    n = 10_000_000
    n_nodes, n_bytes = ctx.synth_sizes(3, n)
    d_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n_nodes + 1, dtype=torch.int64, device="cuda")
    d_first = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_keys = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    d_roots = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    ctx.synth(3, n, d_nodes, d_off, d_first, d_keys, d_roots)
    d_status = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_bitmap = torch.zeros((n + 63) // 64, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    ctx.verify_proofs(n, d_nodes, d_off, d_first, d_keys, d_roots, n, d_bitmap, d_status, None, None, n_nodes=n_nodes, nodes_bytes=n_bytes)
    ctx.synchronize()
    ctx.set_flags(0)
    depth = (d_first[1:] - d_first[:-1]).cpu().numpy()
    assert depth.min() == 4 and depth.max() == 12
    expect = np.where(np.arange(n) % 97 == 0, 0, 1)
    assert (d_status.cpu().numpy() == expect).all()
    del d_nodes, d_off
    torch.cuda.empty_cache()


def test_witness_as_unordered_node_set(ctx, oracle, golden):
    """W: bag-of-nodes witnesses (execution-witness shape) -- GPU vs oracle, incl. missing nodes, junk nodes, fixture tries"""
    from test_oracle_proofs import shuffled_bag
    rng = np.random.default_rng(12)
    w = oracle.synth_blocks(8, txs=60, first=30, threads=8)       # block 37 is corrupted
    victim = int(w["node_index"][int(w["proof_first"][11]) + 3])
    for drop, extra in ((None, 0), (None, 40), (victim, 10)):
        nodes, node_off = shuffled_bag(w, rng, drop=drop, extra=extra)
        want = oracle.verify_bag(nodes, node_off, w["keys32"], w["roots32"], threads=8)
        n = w["n_proofs"]
        bitmap = np.zeros((n + 63) // 64, np.uint64)
        status = np.full(n, 77, np.uint8)
        voff = np.zeros(n, np.uint64)
        vlen = np.zeros(n, np.uint32)
        ctx.set_flags(0)
        ctx.verify_witness(len(node_off) - 1, nodes, node_off, n, w["keys32"], w["roots32"], n, bitmap, status, voff, vlen)
        assert (status == want[0]).all(), np.nonzero(status != want[0])[0][:10]
        ok = status == 1
        assert (voff[ok] == want[1][ok]).all() and (vlen[ok] == want[2][ok]).all()
        bits = np.unpackbits(bitmap.view(np.uint8), bitorder="little")[:n]
        assert (bits == ((status == 1) | (status == 2))).all()
        if drop is not None:
            assert (status == 3).any()
    # a real trie: fixture accounts, present + absent keys, one root for all
    g = golden("fixture_states.json.gz")
    accounts = max(g["tables"].values(), key=len)[:120]
    items = secure_account_items(oracle.keccak256, oracle.mptize, accounts)
    trie = oracle.trie(items)
    bag = {}
    keys = [k for k, _ in items] + [oracle.keccak256(bytes([i])) for i in range(20)]
    for k in keys:
        for nd in trie.prove(k):
            bag[nd] = 1
    nodes, node_off = oracle_lib.csr(list(bag), np.uint64)
    keys32 = np.frombuffer(b"".join(keys), np.uint8)
    root = np.frombuffer(trie.root(), np.uint8)
    want = oracle.verify_bag(nodes, node_off, keys32, root)
    status = np.zeros(len(keys), np.uint8)
    ctx.verify_witness(len(node_off) - 1, nodes, node_off, len(keys), keys32, root, 1, None, status, None, None)
    assert (status == want[0]).all() and (status[:len(items)] == 1).all() and (status[len(items):] == 2).all()


def test_proof_kat_without_the_oracle(golden):
    """CUDA walk against the committed vectors only (no oracle in the loop): statuses, accept bits and value slices"""
    from phant_b200 import gpu
    from test_oracle_proofs import batch_of, kat_batch
    g = golden("proof_kat.json.gz")
    proofs = kat_batch(g)
    nodes, node_off, first, keys, roots = batch_of(proofs)
    n = len(proofs)
    ctx = gpu.Context(0)
    for flags in (0, gpu.FLAG_KECCAK_DIRECT):
        ctx.set_flags(flags)
        bitmap = np.zeros((n + 63) // 64, np.uint64)
        status = np.full(n, 9, np.uint8)
        voff = np.zeros(n, np.uint64)
        vlen = np.zeros(n, np.uint32)
        ctx.verify_proofs(n, nodes, node_off, first, np.ascontiguousarray(keys), np.ascontiguousarray(roots), n, bitmap, status, voff, vlen)
        for i, c in enumerate(g["cases"]):
            assert int(status[i]) == c["status"], (flags, c["name"])
            assert bool((int(bitmap[i // 64]) >> (i % 64)) & 1) == (c["status"] != 0), c["name"]
            if c["status"] == 1:
                assert nodes[int(voff[i]):int(voff[i]) + int(vlen[i])].tobytes().hex() == c["value"], c["name"]
    ctx.close()


def _rlp_items(b):
    """payload items of one RLP list (used on the proven account body: nonce, balance, storage root, code hash)"""
    assert b[0] >= 0xc0
    if b[0] <= 0xf7:
        o, end = 1, 1 + b[0] - 0xc0
    else:
        ll = b[0] - 0xf7
        o, end = 1 + ll, 1 + ll + int.from_bytes(b[1:1 + ll], "big")
    assert end == len(b)
    out = []
    while o < end:
        c = b[o]
        if c < 0x80:
            out.append(b[o:o + 1]); o += 1
        elif c <= 0xb7:
            out.append(b[o + 1:o + 1 + c - 0x80]); o += 1 + c - 0x80
        else:
            ll = c - 0xb7
            n = int.from_bytes(b[o + 1:o + 1 + ll], "big")
            out.append(b[o + 1 + ll:o + 1 + ll + n]); o += 1 + ll + n
    return out


def test_every_fixture_account_and_storage_slot_under_the_fixture_roots(ctx, oracle, golden):
    """SURVEY.md 8c anchor, complete: ONE batch with an inclusion proof for every account of all 91 fixture pre/post
    tables plus absent keys, verified under the stateRoot THE FIXTURE states (genesisBlockHeader.stateRoot / last valid
    blockHeader.stateRoot) -- the expected status comes from the fixture, not from the oracle walk; then ONE batch with
    every storage slot of every account, verified under the storageRoot the GPU just proved inside that account's leaf
    (account proof -> storage_root -> slot proof), plus one absent slot per storage trie."""
    from helpers import rlp_int_be
    g = golden("fixture_states.json.gz")
    root_of = {}
    for t in g["tests"]:
        for tab, root in ((t["pre"], t["pre_root"]), (t["post"], t["post_root"])):
            assert root_of.setdefault(tab, root) == root
    assert set(root_of) == set(g["tables"])  # every table is pinned by a header field
    rng = np.random.default_rng(21)
    proofs, expect, want_val, slot_jobs = [], [], [], []
    for tab, accounts in sorted(g["tables"].items()):
        froot = bytes.fromhex(root_of[tab])
        if not accounts:
            absent = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
            proofs.append(([], absent, froot)); expect.append(2); want_val.append(None)   # empty trie: keccak(0x80)
            continue
        items = secure_account_items(oracle.keccak256, oracle.mptize, accounts)
        trie = oracle.trie(items)            # used to CUT the proofs; what they must hash up to is the fixture's root
        by_key = {oracle.keccak256(bytes.fromhex(a["address"])): a for a in accounts}
        for k, v in items:
            if any(int(x, 16) for x in by_key[k]["storage"].values()):
                slot_jobs.append((len(proofs), by_key[k]))
            proofs.append((trie.prove(k), k, froot)); expect.append(1); want_val.append(v)
        for _ in range(2):
            k = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
            if k not in by_key:
                proofs.append((trie.prove(k), k, froot)); expect.append(2); want_val.append(None)
    nodes, node_off, first, keys, roots = batch_of(proofs)
    bitmap, status, voff, vlen = gpu_verify(ctx, nodes, node_off, first, keys, roots)
    assert (status == np.array(expect, np.uint8)).all(), np.nonzero(status != np.array(expect))[0][:10]
    bits = np.unpackbits(bitmap.view(np.uint8), bitorder="little")[:len(proofs)]
    assert bits.all()
    n_acc = 0
    for i, v in enumerate(want_val):
        if v is not None:
            assert nodes[int(voff[i]):int(voff[i]) + int(vlen[i])].tobytes() == v
            n_acc += 1
    assert n_acc >= 1100, n_acc
    # ---- storage slots under the storage roots proven above ----
    sproofs, sexpect, sval = [], [], []
    for i, a in slot_jobs:
        body = nodes[int(voff[i]):int(voff[i]) + int(vlen[i])].tobytes()
        sroot = _rlp_items(body)[2]
        assert len(sroot) == 32
        st = sorted((oracle.keccak256(bytes.fromhex(k)), rlp_int_be(bytes.fromhex(v))) for k, v in a["storage"].items() if int(v, 16) != 0)
        trie = oracle.trie(st)
        for k, v in st:
            sproofs.append((trie.prove(k), k, sroot)); sexpect.append(1); sval.append(v)
        absent = oracle.keccak256(b"absent slot" + a["address"].encode())
        sproofs.append((trie.prove(absent), absent, sroot)); sexpect.append(2); sval.append(None)
    assert sum(e == 1 for e in sexpect) >= 70
    nodes, node_off, first, keys, roots = batch_of(sproofs)
    bitmap, status, voff, vlen = gpu_verify(ctx, nodes, node_off, first, keys, roots)
    assert (status == np.array(sexpect, np.uint8)).all()
    for i, v in enumerate(sval):
        if v is not None:
            assert nodes[int(voff[i]):int(voff[i]) + int(vlen[i])].tobytes() == v
    # and the same two batches give the same answers on the oracle (the fixture decided; the oracle must agree)
    want = oracle.verify_proofs(nodes, node_off, first, keys, roots, threads=4)
    assert (want[1] == status).all()


@pytest.mark.parametrize("which,n,chunk", [(2, 1_000_000, 250_000), (3, 1_200_000, 300_000)])
def test_full_size_status_and_values_vs_oracle(ctx, oracle, which, n, chunk):
    """BASELINE sizes against the ORACLE, not a pattern: 1M account proofs (C2) and 1.2M storage proofs (C3), every status,
    accept bit and value slice compared with oracle.verify_proofs chunk by chunk (the oracle generator regenerates each
    chunk from (seed, index); the host-pointer ABI verifies it)."""
    for lo in range(0, n, chunk):
        o = oracle.synth_c2(chunk, depth=8, first=lo, threads=8) if which == 2 else oracle.synth_c3(chunk, first=lo, threads=8)
        want = oracle.verify_proofs(*o, threads=8)
        got = gpu_verify(ctx, *o)
        assert (got[1] == want[1]).all() and (got[0] == want[0]).all()
        ok = want[1] == 1
        assert ok.sum() > 0.98 * chunk
        assert (got[2][ok] == want[2][ok]).all() and (got[3][ok] == want[3][ok]).all()
        assert (want[1] == np.where((np.arange(chunk) + lo) % 97 == 0, 0, 1)).all()


def test_device_built_block_witnesses_vs_oracle(ctx, oracle):
    """the C5 workload bench.py measures is BUILT on the device (phant_b200/synth_blocks.py: torch lays the bytes out, the
    library's Keccak hashes every level): what the GPU verifier says about it must be what the oracle says about the same
    bytes -- statuses, accept bits, value slices, per-block reject counts -- and only block 37 may be refused"""
    import torch
    from phant_b200 import gpu, synth_blocks
    first, nb, txs = 30, 12, 40
    w = synth_blocks.synth_blocks(ctx, "cuda", first, nb, txs=txs)
    n = w["n_proofs"]
    h = {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in w.items()}
    want = oracle.verify_proofs(h["nodes"], h["node_off"].astype(np.uint64), h["proof_first"].astype(np.uint64), h["keys32"], h["roots32"], threads=8,
                                node_index=h["node_index"].astype(np.uint64))
    d_status = torch.zeros(n, dtype=torch.uint8, device="cuda")
    d_bitmap = torch.zeros((n + 63) // 64, dtype=torch.int64, device="cuda")
    d_voff = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_vlen = torch.zeros(n, dtype=torch.int32, device="cuda")
    d_counts = torch.zeros(first + nb, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
    ctx.verify_proofs(n, w["nodes"], w["node_off"], w["proof_first"], w["keys32"], w["roots32"], n, d_bitmap, d_status, d_voff, d_vlen,
                      n_nodes=w["n_nodes"], nodes_bytes=w["n_bytes"], node_index=w["node_index"])
    ctx.block_reject_counts(d_status, w["block_of_proof"], n, first + nb, d_counts)
    ctx.synchronize()
    ctx.set_flags(0)
    status = d_status.cpu().numpy()
    assert (status == want[1]).all() and (d_bitmap.cpu().numpy().view(np.uint64) == want[0]).all()
    ok = status == 1
    assert (d_voff.cpu().numpy().view(np.uint64)[ok] == want[2][ok]).all() and (d_vlen.cpu().numpy().view(np.uint32)[ok] == want[3][ok]).all()
    counts = d_counts.cpu().numpy()
    assert counts[37] == 1 and counts.sum() == 1 and (status == 0).sum() == 1
