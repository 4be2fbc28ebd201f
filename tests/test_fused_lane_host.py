"""One lane of the fused verify kernel (verify_fused.cu) compiled as HOST code (tests/hostcheck/fused_host.cpp: the product's
absorb, summary, slot accessor and walk step, shared memory a host array) and compared with the oracle: status, val_off and
val_len.  Every node is placed at a chosen byte skew, so the slot reads, the padding written behind a node, the change from
slot to global walk for nodes longer than one window and the aligned absorb are all reached, at every skew 0..15.  Each proof
also runs with the unaligned absorb only, and the harness fails a proof whose slot reads leave the lane's slot, whose summary
depends on the bytes around the node, or whose padding writes outside the slot.  The product never runs this way; the
-m gpu tests (test_gpu_fused_layout.py) run the kernel itself."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_fuzz_walk import base_proofs, damage
from test_gpu_fused_verify import shaped_proofs
from test_oracle_proofs import batch_of

HERE = os.path.dirname(os.path.abspath(__file__))
COUNTERS = ("tail_ok_true", "tail_ok_false", "masked", "multi_window", "aligned_absorb", "slot_walks", "global_walks", "nodes")
EMPTY_ROOT = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")


@pytest.fixture(scope="module")
def fusedlane(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("fusedlane") / "libfusedhost.so")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so,
                    os.path.join(HERE, "hostcheck", "fused_host.cpp")], check=True)
    lib = C.CDLL(so)
    lib.fusedlane_run.restype = C.c_uint64
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def place(proofs, skews):
    """every node at its own start: a 16-byte aligned address + its skew, after the previous node; gaps and 16 bytes of slack
    behind the last node are 0xA5.  skews[i][j] = skew of node j of proof i."""
    starts, lens, pos = [], [], 0
    for (nl, _, _), sk in zip(proofs, skews):
        for nd, s in zip(nl, sk):
            start = ((pos + 15) & ~15) + int(s)
            starts.append(start)
            lens.append(len(nd))
            pos = start + len(nd)
    buf = np.full(((pos + 15) & ~15) + 16, 0xA5, np.uint8)
    k = 0
    for nl, _, _ in proofs:
        for nd in nl:
            buf[starts[k]:starts[k] + len(nd)] = np.frombuffer(nd, np.uint8)
            k += 1
    return buf, np.array(starts or [0], np.uint64), np.array(lens or [0], np.uint64)


def random_skews(proofs, rng, first=None, last=None):
    """per node a random skew 0..15; `first` / `last` (per proof, or one int) pin the first / the last node's"""
    out = []
    for i, (nl, _, _) in enumerate(proofs):
        sk = [int(x) for x in rng.integers(0, 16, len(nl))]
        if nl and first is not None:
            sk[0] = first if isinstance(first, int) else int(first[i])
        if nl and last is not None:
            sk[-1] = last if isinstance(last, int) else int(last[i])
        out.append(sk)
    return out


def check(lib, oracle, proofs, skews):
    """run the lanes, compare with the oracle; -> (status, counters)"""
    nodes, node_off, first, keys, roots = batch_of(proofs)
    _, want_st, want_off, want_len = oracle.verify_proofs(nodes, node_off, first, keys, roots, threads=4)
    buf, start, length = place(proofs, skews)
    n = len(proofs)
    status, voff, vlen = np.full(n, 9, np.uint8), np.zeros(n, np.uint64), np.zeros(n, np.uint32)
    fail, counters = np.zeros(n, np.uint8), np.zeros(len(COUNTERS), np.uint64)
    keys, roots = np.ascontiguousarray(keys), np.ascontiguousarray(roots)
    bad = lib.fusedlane_run(_p(buf), C.c_uint64(buf.size), _p(start), _p(length), _p(first), C.c_uint64(n), _p(keys), _p(roots),
                            C.c_uint64(n), _p(status), _p(voff), _p(vlen), _p(fail), _p(counters))
    where = np.nonzero(fail)[0]
    assert bad == 0 and where.size == 0, ("harness checks failed (F_* bits)", where[:10], fail[where[:10]],
                                          [skews[i] for i in where[:3]], [[len(x) for x in proofs[i][0]] for i in where[:3]])
    wrong = np.nonzero(status != want_st)[0]
    assert wrong.size == 0, ("status", wrong[:10], status[wrong[:10]], want_st[wrong[:10]], [skews[i] for i in wrong[:3]])
    # val_off is an offset into this layout's buffer: map it back through the node holding it to the oracle's contiguous CSR
    ok = status == 1
    g = np.searchsorted(start, voff[ok], side="right") - 1
    mapped = node_off[g] + (voff[ok] - start[g])
    wrong = np.nonzero((mapped != want_off[ok]) | (vlen[ok] != want_len[ok]))[0]
    assert wrong.size == 0, ("val_off / val_len", np.nonzero(ok)[0][wrong[:10]], mapped[wrong[:10]], want_off[ok][wrong[:10]])
    assert (voff[~ok] == 0).all() and (vlen[~ok] == 0).all()
    return status, dict(zip(COUNTERS, counters.tolist()))


def at_every_skew(proofs, rng, pin="first"):
    """the proofs 16 times over, the pinned node at skew 0, 1, .. 15, the other nodes at random skews"""
    rep = [p for _ in range(16) for p in proofs]
    pinned = [s for s in range(16) for _ in proofs]
    return rep, random_skews(rep, rng, **{pin: pinned})


def flip_byte(nd, rng):
    b = bytearray(nd)
    b[int(rng.integers(0, len(b)))] ^= 1 << int(rng.integers(0, 8))
    return bytes(b)


def last_nibble_changed(key):
    return key[:31] + bytes([key[31] ^ 0x01])


def present_absent_flipped(nl, key, root, rng):
    j = int(rng.integers(0, len(nl)))
    return [(nl, key, root), (nl, last_nibble_changed(key), root), (nl[:j] + [flip_byte(nl[j], rng)] + nl[j + 1:], key, root)]


def test_skew_sweep(fusedlane, oracle):
    """the fuzz base proofs and the shaped proofs of the GPU fused test, first node at every skew 0..15"""
    rng = np.random.default_rng(71)
    proofs = base_proofs(oracle, rng) + shaped_proofs(oracle, rng)
    rep, skews = at_every_skew(proofs, rng)
    st, cnt = check(fusedlane, oracle, rep, skews)
    assert {0, 1, 2} <= set(st.tolist())
    assert all(cnt[k] > 0 for k in COUNTERS if k != "masked"), cnt  # no node of these ends 544..559 bytes into a window


def leaf_of_every_length(oracle, rng, lo, hi, stride=1):
    """{leaf length: (proof nodes, key, root)} of single-leaf tries, one per reachable length in [lo, hi]"""
    out = {}
    for v in range(1, hi):
        key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
        t = oracle.trie([(key, rng.integers(0, 256, v, dtype=np.uint8).tobytes())])
        nl = t.prove(key)
        if lo <= len(nl[0]) <= hi and (len(nl[0]) - lo) % stride == 0:
            out.setdefault(len(nl[0]), (nl, key, t.root()))
    return out


def test_leaf_length_sweep(fusedlane, oracle):
    """single leaves of 36..1200 bytes at every skew (a 64-nibble leaf is at least 36 bytes): the window edge (skew + len 560
    fits, 561 does not), the masked final block (a tail after 544 bytes) and nodes of 2..9 windows; present, absent (last key
    nibble changed) and one flipped byte each"""
    rng = np.random.default_rng(72)
    leaves = leaf_of_every_length(oracle, rng, 36, 1200)
    assert set(range(555, 566)) <= set(leaves)
    proofs = [c for nl, key, root in leaves.values() for c in present_absent_flipped(nl, key, root, rng)]
    rep, skews = at_every_skew(proofs, rng)
    st, cnt = check(fusedlane, oracle, rep, skews)
    assert set(st.tolist()) == {0, 1, 2}
    for k in ("tail_ok_true", "masked", "multi_window", "aligned_absorb", "global_walks", "slot_walks"):
        assert cnt[k] > 0, cnt


def test_two_node_chains_cross_the_window(fusedlane, oracle):
    """branch + long leaf (slot walk, then a leaf of 36..1200 bytes at every skew, some walked from global memory), and a
    branch made longer than one window by its value, followed by a leaf (global walk, then slot walk)"""
    rng = np.random.default_rng(73)
    proofs = []
    for L in list(range(36, 1200, 7)) + list(range(540, 580)):
        v = max(1, L - 36)
        k1 = bytes([0x1F]) + rng.integers(0, 256, 31, dtype=np.uint8).tobytes()
        k2 = bytes([0x2F]) + rng.integers(0, 256, 31, dtype=np.uint8).tobytes()
        t = oracle.trie([(k1, rng.integers(0, 256, v, dtype=np.uint8).tobytes()), (k2, b"\x05" * 40)])
        proofs += present_absent_flipped(t.prove(k1), k1, t.root(), rng)
    st1, cnt1 = check(fusedlane, oracle, *at_every_skew(proofs, rng, pin="last"))
    assert set(st1.tolist()) == {0, 1, 2} and cnt1["global_walks"] > 0 and cnt1["masked"] > 0
    # prefix keys: the 31-byte key's value sits in the branch at nibble 62, the 32-byte keys hang below it as hashed leaves
    proofs = []
    for v in list(range(30, 700, 23)) + [400, 460, 500]:
        for kids in (2, 16):
            base = rng.integers(0, 256, 31, dtype=np.uint8).tobytes()
            kv = [(base, rng.integers(0, 256, v, dtype=np.uint8).tobytes())]
            kv += [(base + bytes([16 * x + 3]), rng.integers(0, 256, 40, dtype=np.uint8).tobytes()) for x in range(0, 16, 16 // kids)]
            t = oracle.trie(sorted(kv))
            k = base + bytes([0x03])
            nl = t.prove(k)
            assert len(nl) == 3
            proofs += present_absent_flipped(nl, k, t.root(), rng)
    rep, _ = at_every_skew(proofs, rng)
    skews = [[int(rng.integers(0, 16)), s, int(rng.integers(0, 16))] for s in range(16) for _ in proofs]
    st2, cnt2 = check(fusedlane, oracle, rep, skews)
    assert set(st2.tolist()) == {0, 1, 2} and cnt2["multi_window"] > 0 and cnt2["global_walks"] > 0


def test_leaf_paths_of_every_length(fusedlane, oracle):
    """leaves whose paths have 1..63 nibbles, hashed and embedded in their branch: the leaf-path compare reads the 32 bytes
    ending at the path's end, which start in front of the node when the path ends early -- tail_ok says no at small skews
    and yes at large ones"""
    rng = np.random.default_rng(74)
    proofs = []
    for shared in list(range(0, 29, 2)) + [29, 30, 31, 31]:
        prefix = rng.integers(0, 256, shared, dtype=np.uint8).tobytes()
        keys = sorted({prefix + rng.integers(0, 256, 32 - shared, dtype=np.uint8).tobytes() for _ in range(int(rng.integers(2, 12)))})
        kv = [(k, rng.integers(0, 256, int(rng.choice([1, 2, 5, 20, 40])), dtype=np.uint8).tobytes()) for k in keys]
        t = oracle.trie(kv)
        for k in keys:
            proofs += present_absent_flipped(t.prove(k), k, t.root(), rng)
        for _ in range(3):
            k = prefix + rng.integers(0, 256, 32 - shared, dtype=np.uint8).tobytes()
            proofs.append((t.prove(k), k, t.root()))
    st, cnt = check(fusedlane, oracle, *at_every_skew(proofs, rng, pin="last"))
    assert set(st.tolist()) == {0, 1, 2}
    assert cnt["tail_ok_true"] > 0 and cnt["tail_ok_false"] > 0, cnt


def rlp_branch(children):
    """a 17-item branch: children[n] = 32-byte reference or b'' (empty), empty value"""
    pay = b"".join(b"\xa0" + c if c else b"\x80" for c in children) + b"\x80"
    return (bytes([0xc0 + len(pay)]) if len(pay) <= 55 else bytes([0xf8, len(pay)]) if len(pay) < 256 else
            bytes([0xf9, len(pay) >> 8, len(pay) & 255])) + pay


def test_empty_nodes(fusedlane, oracle):
    """zero-length nodes: inside a chain, behind a leaf, as the first node under keccak(''), and named by a branch whose child
    reference is keccak('') (the digest matches, the walk rejects the empty node); the empty proof"""
    rng = np.random.default_rng(75)
    k_empty = oracle.keccak256(b"")
    base = [p for p in base_proofs(oracle, rng) if len(p[0]) >= 2][:20]
    proofs = []
    for nl, key, root in base:
        j = int(rng.integers(1, len(nl)))
        proofs += [(nl[:j] + [b""] + nl[j:], key, root), (nl + [b""], key, root), ([b""] + nl, key, root)]
    children = [b""] * 16
    children[3], children[9] = k_empty, oracle.keccak256(b"\x01" * 40)
    br = rlp_branch(children)
    rb = oracle.keccak256(br)
    k3, k7 = bytes([0x3A]) + bytes(31), bytes([0x7A]) + bytes(31)
    leaf = bytes(rng.integers(0, 256, 40, dtype=np.uint8))
    proofs += [([br, b""], k3, rb), ([br, b"", leaf], k3, rb), ([br], k7, rb), ([br, b""], k7, rb), ([b""], k3, k_empty),
               ([b"", b""], k3, k_empty), ([], k3, EMPTY_ROOT), ([], k3, rb)]
    st, _ = check(fusedlane, oracle, *at_every_skew(proofs, rng))
    assert {0, 2} <= set(st.tolist())


def test_damaged_proofs(fusedlane, oracle):
    rng = np.random.default_rng(515)
    base = base_proofs(oracle, rng)
    cases = [damage(base[int(rng.integers(0, len(base)))], rng) for _ in range(6000)]
    st, _ = check(fusedlane, oracle, cases, random_skews(cases, rng))
    assert set(st.tolist()) == {0, 1, 2}
