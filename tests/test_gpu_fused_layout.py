"""The fused verify kernel (verify_fused.cu) on layouts chosen to reach its aligned absorb and its chunked host path, compared
with the oracle only (status, accept bitmap, val_off, val_len).

Every C2 node is 532 or 112 bytes, a multiple of 4, so a C2 batch keeps every node start at a multiple of 4 and every warp
takes the aligned absorb.  Damage that keeps the lengths (bit flips, another last key nibble, another root, a dropped 532-byte
node) keeps it so; a leading filler node of 4, 8 or 12 bytes moves every node to another slot skew and keeps it so, one of 1,
2 or 3 bytes leaves no node start at a multiple of 4 and forces the unaligned absorb."""
import os
import subprocess
import sys

import numpy as np
import pytest

from test_gpu_fused_verify import run_host
from test_oracle_proofs import batch_of

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    from phant_b200 import gpu
    c = gpu.Context(0)
    yield c
    c.close()


def c2_proofs(oracle, n, first=0):
    nodes, node_off, pf, keys, roots = oracle.synth_c2(n, depth=8, first=first)
    return [([nodes[int(node_off[j]):int(node_off[j + 1])].tobytes() for j in range(int(pf[i]), int(pf[i + 1]))],
             keys[32 * i:32 * i + 32].tobytes(), roots[32 * i:32 * i + 32].tobytes()) for i in range(n)]


def damage_keeping_lengths(proof, kind, rng):
    """0 intact, 1 bit flips in one node, 2 last key nibble changed (ABSENT), 3 another root, 4 one 532-byte node dropped"""
    nl, key, root = proof
    if kind == 1:
        j = int(rng.integers(0, len(nl)))
        b = bytearray(nl[j])
        for bit in rng.integers(0, 8 * len(b), int(rng.integers(1, 4))):
            b[bit >> 3] ^= 1 << (bit & 7)
        nl = nl[:j] + [bytes(b)] + nl[j + 1:]
    elif kind == 2:
        key = key[:31] + bytes([key[31] ^ 0x01])
    elif kind == 3:
        root = bytes([root[0] ^ 0x80]) + root[1:]
    elif kind == 4:
        j = int(rng.integers(0, len(nl) - 1))
        nl = nl[:j] + nl[j + 1:]
    return nl, key, root


def damaged_c2(oracle, n, rng, first=0):
    return [damage_keeping_lengths(p, int(k), rng) for p, k in zip(c2_proofs(oracle, n, first), rng.integers(0, 5, n))]


def compare(got, want, what=""):
    for a, b, name in zip(got, want, ("bitmap", "status", "val_off", "val_len")):
        assert (a == b).all(), (what, name, np.nonzero(a != b)[0][:10], a[np.nonzero(a != b)[0][:5]], b[np.nonzero(a != b)[0][:5]])


@pytest.mark.parametrize("n", [3001, 9001])
def test_aligned_warps_at_every_shift(ctx, oracle, n):
    """damaged C2 behind a filler node of 0..12 bytes; n < 4096 runs in proof order, n > 4096 regrouped (not a multiple of 32)"""
    rng = np.random.default_rng(n)
    proofs = damaged_c2(oracle, n, rng)
    junk_key, junk_root = rng.integers(0, 256, 32, dtype=np.uint8).tobytes(), rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    for shift in (0, 4, 8, 12, 1, 2, 3):
        batch = ([([bytes(rng.integers(0, 256, shift, dtype=np.uint8))], junk_key, junk_root)] if shift else []) + proofs
        nodes, node_off, first, keys, roots = batch_of(batch)
        starts = node_off[1 if shift else 0:-1]
        if shift % 4 == 0:
            assert (starts % 4 == 0).all()  # every warp: the aligned absorb
        else:
            assert (starts % 4 == shift).all()  # no warp: the unaligned absorb
        assert len({int(s) % 16 for s in starts}) > 1  # and more than one slot skew
        want = oracle.verify_proofs(nodes, node_off, first, keys, roots, threads=8)
        ctx.reset_stats()
        got = run_host(ctx, nodes, node_off, first, keys, roots)
        st = ctx.stats()
        assert st["walk_ms"] == 0 and st["launches"] == (3 if len(batch) >= 4096 else 1), (shift, st)  # the fused kernel ran
        compare(got, want, shift)
        assert set(want[1][1 if shift else 0:].tolist()) == {0, 1, 2}


CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[3])
from phant_b200 import gpu
a = np.load(sys.argv[1])
n = len(a["first"]) - 1
ctx = gpu.Context(0)
bitmap, status = np.zeros((n + 63) // 64, np.uint64), np.full(n, 77, np.uint8)
voff, vlen = np.full(n, 7, np.uint64), np.full(n, 7, np.uint32)
ctx.verify_proofs(n, a["nodes"], a["node_off"], a["first"], a["keys"], a["roots"], a["roots"].size // 32, bitmap, status, voff, vlen)
st = ctx.stats()
ctx.close()
np.savez(sys.argv[2], bitmap=bitmap, status=status, voff=voff, vlen=vlen, launches=st["launches"], walk_ms=st["walk_ms"])
"""


@pytest.mark.parametrize("roots", ["per_proof", "one"])
def test_chunked_host_path(oracle, tmp_path, roots):
    """host pointers in 1 MB chunks (PHANT_GPU_CHUNK_MB, read once per process: a child process): every chunk is 4096 proofs
    and regrouped, the last partial one is not.  Per-proof roots (damaged C2), or one root for the whole batch (damaged copies
    of one C2 proof)"""
    rng = np.random.default_rng(21 if roots == "one" else 22)
    n = 4 * 4096 + 3629
    if roots == "one":
        one = c2_proofs(oracle, 2, first=1)[1]
        proofs = [damage_keeping_lengths(one, int(k), rng) for k in rng.integers(0, 5, n)]
        nodes, node_off, first, keys, _ = batch_of(proofs)
        roots32 = np.frombuffer(one[2], np.uint8).copy()
    else:
        nodes, node_off, first, keys, roots32 = batch_of(damaged_c2(oracle, n, rng, first=7))
    assert (node_off % 4 == 0).all()
    want = oracle.verify_proofs(nodes, node_off, first, keys, roots32, threads=8)
    assert set(want[1].tolist()) == {0, 1, 2}
    src, dst = tmp_path / "in.npz", tmp_path / "out.npz"
    np.savez(src, nodes=nodes, node_off=node_off, first=first, keys=np.ascontiguousarray(keys), roots=np.ascontiguousarray(roots32))
    subprocess.run([sys.executable, "-c", CHILD, str(src), str(dst), ROOT], check=True, cwd=ROOT,
                   env={**os.environ, "PHANT_GPU_CHUNK_MB": "1"})
    out = np.load(dst)
    assert int(out["walk_ms"]) == 0 and int(out["launches"]) == 4 * 3 + 1  # 4 regrouped chunks (3 launches each) + 1 in order
    compare([out["bitmap"], out["status"], out["voff"], out["vlen"]], want, roots)
