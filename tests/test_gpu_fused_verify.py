"""V on a plain CSR chain runs the fused kernel (verify_fused.cu: each lane hashes and walks one proof); the same witness with
node_index = arange(n_nodes) runs the two-pass path (hash_csr + walk_kernel).  Status, accept bitmap, val_off and val_len
must be byte-identical between the two, and equal to the oracle."""
import numpy as np
import pytest

from helpers import secure_account_items
from test_fuzz_walk import base_proofs, damage
from test_oracle_proofs import batch_of, mutations

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from phant_b200 import gpu
    c = gpu.Context(0)
    yield c
    c.close()


def run_host(ctx, nodes, node_off, first, keys, roots, node_index=None):
    n = len(first) - 1
    bitmap = np.zeros((n + 63) // 64, np.uint64)
    status = np.full(n, 77, np.uint8)
    voff = np.full(n, 7, np.uint64)
    vlen = np.full(n, 7, np.uint32)
    ctx.set_flags(0)
    ctx.verify_proofs(n, np.ascontiguousarray(nodes), node_off, first, np.ascontiguousarray(keys), np.ascontiguousarray(roots),
                      roots.size // 32, bitmap, status, voff, vlen, n_nodes=len(node_off) - 1, nodes_bytes=int(node_off[-1]),
                      node_index=node_index)
    return bitmap, status, voff, vlen


def assert_fused_equals_two_pass(ctx, oracle, nodes, node_off, first, keys, roots):
    ctx.reset_stats()
    fused = run_host(ctx, nodes, node_off, first, keys, roots)
    st = ctx.stats()
    assert st["walk_ms"] == 0 and st["keccak_perms"] > 0  # the fused path ran: no walk kernel
    two = run_host(ctx, nodes, node_off, first, keys, roots, node_index=np.arange(len(node_off) - 1, dtype=np.uint64))
    for a, b, what in zip(fused, two, ("bitmap", "status", "val_off", "val_len")):
        assert (a == b).all(), (what, np.nonzero(a != b)[0][:10])
    want = oracle.verify_proofs(nodes, node_off, first, keys, roots, threads=8)
    assert (fused[1] == want[1]).all() and (fused[0] == want[0]).all()
    return fused[1]


def fixture_proofs(oracle, golden, rng, tables=30):
    g = golden("fixture_states.json.gz")
    proofs = []
    for _, accounts in sorted(g["tables"].items())[:tables]:
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
    return proofs


def shaped_proofs(oracle, rng):
    """embedded children, extensions, branch values, nodes longer than one staging window, the empty trie"""
    base = bytes(range(31))
    kv = sorted((base + bytes([b]), bytes([v])) for b, v in [(0x10, 1), (0x11, 2), (0x1f, 3), (0x20, 4), (0x77, 5)])
    t = oracle.trie(kv)
    proofs = [(t.prove(k), k, t.root()) for k, _ in kv]
    proofs += [(t.prove(k), k, t.root()) for k in [base + bytes([0x12]), base + bytes([0x30]), bytes([0xff]) + base]]
    # values of 540 .. 2000 bytes: leaves that stream through the slot in several windows
    keys = sorted(rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(60))
    kv = [(k, rng.integers(0, 256, int(rng.choice([540, 600, 1100, 2000])), dtype=np.uint8).tobytes()) for k in keys]
    t = oracle.trie(kv)
    proofs += [(t.prove(k), k, t.root()) for k in keys]
    proofs += [(t.prove(k), k, t.root()) for k in (rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(10))]
    empty = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")
    proofs += [([], bytes(32), empty), ([], bytes(32), bytes(32))]
    for p in list(proofs[:12]):
        proofs += mutations(*p, rng)
    return proofs


def test_fixtures_mutations_and_shapes(ctx, oracle, golden):
    rng = np.random.default_rng(11)
    proofs = fixture_proofs(oracle, golden, rng) + shaped_proofs(oracle, rng)
    proofs = proofs[:len(proofs) - (len(proofs) % 32 == 0)]  # not a whole number of warps
    assert len(proofs) % 32
    st = assert_fused_equals_two_pass(ctx, oracle, *batch_of(proofs))
    assert {0, 1, 2} <= set(st.tolist())


def test_damaged_proofs_regrouped(ctx, oracle):
    """> 4096 proofs of mixed lengths, so the proofs are regrouped by permutation count before the fused kernel: warps then
    hold proofs from all over the batch, and reject early at different nodes"""
    rng = np.random.default_rng(12)
    base = base_proofs(oracle, rng) + shaped_proofs(oracle, rng)
    proofs = []
    while len(proofs) < 9000:
        p = base[int(rng.integers(0, len(base)))]
        proofs.append(damage(p, rng) if rng.random() < 0.4 else p)
    proofs = proofs[:9000 - 13]
    st = assert_fused_equals_two_pass(ctx, oracle, *batch_of(proofs))
    assert {0, 1, 2} <= set(st.tolist())


@pytest.mark.parametrize("which,n", [(2, 1_000_000), (3, 300_000)])
def test_device_pointers_c2_c3(ctx, which, n):
    """device-pointer path at benchmark size (C2) and over C3's depths 4 .. 12: fused == two-pass, byte for byte"""
    import torch
    from phant_b200 import gpu
    n_nodes, n_bytes = ctx.synth_sizes(which, n, depth=8, first=0)
    d_nodes = torch.empty(n_bytes + 64, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n_nodes + 1, dtype=torch.int64, device="cuda")
    d_first = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_keys = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    d_roots = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.synth(which, n, d_nodes, d_off, d_first, d_keys, d_roots, depth=8, first=0)
    d_index = torch.arange(n_nodes, dtype=torch.int64, device="cuda")
    out = []
    for node_index in (None, d_index):
        d_status = torch.full((n,), 77, dtype=torch.uint8, device="cuda")
        d_bitmap = torch.zeros((n + 63) // 64, dtype=torch.int64, device="cuda")
        d_voff = torch.full((n,), 7, dtype=torch.int64, device="cuda")
        d_vlen = torch.full((n,), 7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.set_flags(gpu.FLAG_DEVICE_PTRS)
        ctx.reset_stats()
        ctx.verify_proofs(n, d_nodes, d_off, d_first, d_keys, d_roots, n, d_bitmap, d_status, d_voff, d_vlen,
                          n_nodes=n_nodes, nodes_bytes=n_bytes, node_index=node_index)
        ctx.synchronize()
        st = ctx.stats()
        ctx.set_flags(0)
        if node_index is None:  # classify + regroup + the fused kernel
            assert st["launches"] == 3 and st["walk_ms"] == 0 and st["keccak_msgs"] == n_nodes and st["keccak_bytes"] == n_bytes
        out.append([t.cpu().numpy() for t in (d_bitmap, d_status, d_voff, d_vlen)])
    for a, b, what in zip(out[0], out[1], ("bitmap", "status", "val_off", "val_len")):
        assert (a == b).all(), (what, np.nonzero(a != b)[0][:10])
    expect = np.where(np.arange(n) % 97 == 0, 0, 1)
    assert (out[0][1] == expect).all()
