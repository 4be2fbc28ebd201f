"""Pin the CPU oracle against every known answer the reference holds for this path (SURVEY.md 8c).

CPU-only.  If these fail nothing else in the suite means anything: the GPU parity tests compare against
this oracle.
"""
import numpy as np
import pytest

from helpers import compiled_reference_keccak_messages, compiled_reference_secure_tries, index_trie_items, inputs_sha256


def test_keccak_reference_table(oracle, golden):
    """ethash/test/unittests/test_keccak.cpp:25-195 -- every prefix length of test_text."""
    g = golden("keccak_kat.json")
    text = g["text"].encode()
    assert len(g["cases"]) >= 160
    for c in g["cases"]:
        assert oracle.keccak256(text[:c["len"]]).hex() == c["keccak256"], c["len"]


def test_keccak_unaligned(oracle, golden):
    """ethash/test/unittests/test_keccak.cpp:221-240 -- same table at byte offsets 1..7."""
    g = golden("keccak_kat.json")
    text = g["text"].encode()
    for shift in range(1, 8):
        buf = np.zeros(len(text) + 16, np.uint8)
        buf[shift:shift + len(text)] = np.frombuffer(text, np.uint8)
        off = np.array([shift, shift + 0], np.uint64)
        for c in g["cases"][::7]:
            off[1] = shift + c["len"]
            assert oracle.keccak256_batch(buf, off)[0].tobytes().hex() == c["keccak256"]


def test_keccak_constants(oracle):
    """keccak('') = src/blockchain/vm.zig:22, keccak(0x80) = src/mpt/mpt.zig:10, keccak(0xc0) = src/types/block.zig:13."""
    assert oracle.keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert oracle.keccak256(b"\x80").hex() == "56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421"
    assert oracle.keccak256(b"\xc0").hex() == "1dcc4de8dec75d7aab85b567b6ccd41ad312451b948a7413f0a142fd40d49347"


def test_port_equals_compiled_reference_keccak(oracle, golden):
    """The port vs the reference's keccak.c compiled unchanged (oracle/_ref; digests stored by
    tests/golden/make_compiled_reference_kat.py), random lengths 0..1200."""
    g = golden("compiled_reference_kat.json")
    msgs = compiled_reference_keccak_messages()
    assert inputs_sha256(msgs) == g["keccak_inputs_sha256"], "the messages differ from those the digests were computed for"
    assert [len(m) for m in msgs] == [c["len"] for c in g["keccak"]]
    for m, c in zip(msgs, g["keccak"]):
        assert oracle.keccak256(m).hex() == c["keccak256"], len(m)


def test_mptize_reference_roots(oracle, golden):
    """src/mpt/mpt.zig:326-385 -- the seven `mptize` roots."""
    for c in golden("mptize_kat.json")["cases"]:
        kv = [(bytes.fromhex(k), bytes.fromhex(v)) for k, v in c["kv"]]
        assert oracle.mptize(kv).hex() == c["root"], c["name"]


def test_mptize_rejects_unsorted(oracle):
    with pytest.raises(ValueError):
        oracle.mptize([(b"\x02", b"a"), (b"\x01", b"b")])
    with pytest.raises(ValueError):
        oracle.mptize([(b"\x01", b"a"), (b"\x01", b"b")])


def test_evmone_topologies(oracle, golden):
    """evmone/test/unittests/state_mpt_test.cpp:157-333 -- root after each insertion, all >= 32-byte nodes."""
    g = golden("evmone_mpt_kat.json")
    for grp in g["topologies"]:
        for upto in range(1, len(grp) + 1):
            kv = sorted((bytes.fromhex(e["key"]), bytes.fromhex(e["value"])) for e in grp[:upto])
            assert oracle.mptize(kv).hex() == grp[upto - 1]["root_after_insert"]
    for e in g["examples"]:
        kv = sorted((bytes.fromhex(k), bytes.fromhex(v)) for k, v in e["kv"])
        assert oracle.mptize(kv).hex() == e["root"], e["name"]


def test_evmone_state_roots(oracle, golden):
    """evmone/test/unittests/state_mpt_hash_test.cpp:19-66 (go-ethereum derived)."""
    for s in golden("evmone_mpt_kat.json")["states"]:
        assert oracle.state_root(s["accounts"]).hex() == s["root"], s["name"]


def test_fixture_state_roots(oracle, golden):
    """84 + 84 state roots: root(pre) == genesis stateRoot, root(postState) == last valid block's stateRoot."""
    g = golden("fixture_states.json.gz")
    roots = {k: oracle.state_root(v).hex() for k, v in g["tables"].items()}
    assert len(g["tests"]) == 84
    for t in g["tests"]:
        assert roots[t["pre"]] == t["pre_root"], (t["file"], t["name"], "pre")
        assert roots[t["post"]] == t["post_root"], (t["file"], t["name"], "post")


def test_fixture_list_roots(oracle, golden):
    """87 + 87 index-trie roots (src/blockchain/blockchain.zig:209-235 key order) vs the block headers."""
    g = golden("fixture_states.json.gz")
    n = 0
    for t in g["tests"]:
        for b in t["blocks"]:
            txs = [bytes.fromhex(x) for x in b["tx_values"]]
            wds = [bytes.fromhex(x) for x in b["wd_values"]]
            assert oracle.mptize(index_trie_items(txs)).hex() == b["transactionsTrie"]
            assert oracle.mptize(index_trie_items(wds)).hex() == b["withdrawalsRoot"]
            n += 1
    assert n == 87


def test_secure_trie_equals_compiled_evmone(oracle, golden):
    """Random secure tries: mptize restatement vs the reference's vendored evmone MPT compiled unchanged (oracle/_ref;
    roots stored by tests/golden/make_compiled_reference_kat.py)."""
    g = golden("compiled_reference_kat.json")
    tries = compiled_reference_secure_tries()
    assert inputs_sha256([k + v for kv in tries for k, v in kv]) == g["secure_trie_inputs_sha256"], \
        "the tries differ from those the roots were computed for"
    assert [len(kv) for kv in tries] == [c["n"] for c in g["secure_trie"]]
    for kv, c in zip(tries, g["secure_trie"]):
        assert oracle.mptize(kv).hex() == c["root"], len(kv)


def test_logs_bloom_reference_vector(oracle, golden):
    """Receipt.addToBloom (src/types/receipt.zig:50-63): the three-log receipt of
    evmone/test/unittests/state_mpt_hash_test.cpp:118-190 and its on-chain logsBloom."""
    g = golden("logs_bloom_kat.json")
    items, own = [], []
    for addr, topics in g["logs"]:
        items.append(bytes.fromhex(addr)); own.append(0)
        for t in topics:
            items.append(bytes.fromhex(t)); own.append(0)
    assert oracle.logs_bloom(items, own, 1)[0].tobytes().hex() == g["bloom"]


def test_tx_hash_reference_vectors(oracle, golden):
    """src/types/transaction.zig:275-314: three mainnet transactions (legacy, EIP-2930, EIP-1559)."""
    for c in golden("tx_hash_kat.json")["cases"]:
        assert oracle.keccak256(bytes.fromhex(c["encoded"])).hex() == c["hash"]


def test_receipts_root_reference_vector(oracle, golden):
    """evmone/test/unittests/state_mpt_hash_test.cpp:192-245: blooms + receipt encodings + index trie, all on the CPU side"""
    from phant_b200.host import Log, Receipt
    g = golden("logs_bloom_kat.json")
    receipts = []
    for r in g["receipts"]:
        logs = [Log(bytes.fromhex(l["address"]), [bytes.fromhex(x) for x in l["topics"]], bytes.fromhex(l["data"])) for l in r["logs"]]
        rc = Receipt(r["succeeded"], r["gas_used"], logs, tx_type=r["type"])
        items = [x for l in logs for x in [l.address] + l.topics]
        rc.bloom = oracle.logs_bloom(items, [0] * len(items), 1)[0].tobytes() if items else bytes(256)
        receipts.append(rc)
    assert oracle.mptize(index_trie_items([r.encode() for r in receipts])).hex() == g["receipts_root"]


def test_oracle_mptize_vs_independent_python(oracle, golden):
    """the C oracle against a second, independently written statement of mpt.zig (tests/helpers.py::py_mptize): first on the
    reference's own 7 roots (so the Python statement is itself pinned), then on random tries with prefix keys, branch
    values, embedded children, extensions, empty and long values"""
    import numpy as np
    from helpers import py_mptize
    for c in golden("mptize_kat.json")["cases"]:
        kv = [(bytes.fromhex(k), bytes.fromhex(v)) for k, v in c["kv"]]
        assert py_mptize(oracle.keccak256, kv).hex() == c["root"], c["name"]
    assert py_mptize(oracle.keccak256, []) == oracle.mptize([])
    rng = np.random.default_rng(4242)
    for trial in range(300):
        n = int(rng.choice([1, 2, 3, 5, 8, 20, 60]))
        keys = set()
        while len(keys) < n:
            base = bytes(rng.integers(0, 3, int(rng.integers(0, 5)), dtype=np.uint8) * 17)  # nibble-repeating bytes: shared runs
            keys.add(base + bytes(rng.integers(0, 256, int(rng.integers(0, 3)), dtype=np.uint8)))
        kv = [(k, rng.integers(0, 256, int(rng.choice([0, 1, 1, 2, 10, 31, 32, 33, 60, 200])), dtype=np.uint8).tobytes()) for k in sorted(keys)]
        assert py_mptize(oracle.keccak256, kv) == oracle.mptize(kv), (trial, kv)


def test_oracle_state_root_vs_independent_python(oracle, golden):
    """oracle_state_root (C) against keys / leaves assembled in Python and the independent py_mptize, on fixture states and
    random ones (zero slots, empty code, big balances)"""
    import numpy as np
    from helpers import py_mptize, secure_account_items
    g = golden("fixture_states.json.gz")
    for name in list(g["tables"])[:6]:
        acc = g["tables"][name]
        items = secure_account_items(oracle.keccak256, lambda kv: py_mptize(oracle.keccak256, kv), acc)
        assert py_mptize(oracle.keccak256, items) == oracle.state_root(acc), name
    rng = np.random.default_rng(7)
    for trial in range(20):
        acc = []
        for _ in range(int(rng.choice([1, 2, 9, 40]))):
            st = {rng.integers(0, 256, 32, dtype=np.uint8).tobytes().hex(): (bytes(int(rng.integers(0, 33))) + rng.integers(0, 256, 32, dtype=np.uint8).tobytes())[:32].hex()
                  for _ in range(int(rng.choice([0, 1, 4])))}
            acc.append({"address": rng.integers(0, 256, 20, dtype=np.uint8).tobytes().hex(), "nonce": int(rng.choice([0, 1, 128, 2 ** 40])),
                        "balance": "%064x" % int(rng.choice([0, 127, 128, 2 ** 255 + 5])), "code": rng.integers(0, 256, int(rng.choice([0, 1, 200])), dtype=np.uint8).tobytes().hex(),
                        "storage": st})
        items = secure_account_items(oracle.keccak256, lambda kv: py_mptize(oracle.keccak256, kv), acc)
        assert py_mptize(oracle.keccak256, items) == oracle.state_root(acc), trial


def test_rlp_encoder_vectors(oracle, golden):
    """evmone/test/unittests/state_rlp_test.cpp: the wire format zig-rlp (absent from the tree) must produce; pins the RLP
    helpers that prepare builder inputs in the host mirror (phant_b200/host.py) and in the tests (tests/helpers.py), and --
    through a one-account state -- the account body the oracle's and the device's state-root builders emit"""
    from helpers import rlp_int_be, rlp_list, rlp_str, rlp_uint
    from phant_b200 import host
    g = golden("rlp_kat.json")
    for c in g["uint64"]:
        v, want = c["value"], c["rlp"]
        assert host._rlp_uint(v).hex() == want == rlp_uint(v).hex() == rlp_int_be(v.to_bytes(8, "big")).hex(), v
    for c in g["long_strings"]:
        for enc in (host._rlp_str, rlp_str):
            r = enc(bytes(c["len"]))
            assert len(r) == c["len"] + 1 + (r[0] - 0xb7) and r[:10].hex() == c["first10"], c
    empty_root = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")
    empty_hash = oracle.keccak256(b"")
    body = [rlp_uint(0), rlp_uint(1), rlp_str(empty_root), rlp_str(empty_hash)]
    assert rlp_list(body).hex() == g["account_nonce0_balance1_empty"] == host._rlp_list(body).hex()
    assert rlp_int_be(bytes.fromhex("%064x" % 0x01ff)).hex() == g["storage_value_0x01ff"]
    leaf = g["leaf_node"]
    assert rlp_list([rlp_str(bytes.fromhex(leaf["path"])), rlp_str(bytes.fromhex(leaf["value"]))]).hex() == leaf["rlp"]
    # the same account body inside the oracle's state root: one account (nonce 0, balance 1, no code, no storage)
    addr = bytes(19) + b"\x07"
    acct = {"address": addr.hex(), "nonce": 0, "balance": "%064x" % 1, "code": "", "storage": {}}
    key = oracle.keccak256(addr)
    leaf_rlp = rlp_list([rlp_str(b"\x20" + key), rlp_str(bytes.fromhex(g["account_nonce0_balance1_empty"]))])
    assert oracle.state_root([acct]) == oracle.keccak256(leaf_rlp)


def test_fixture_header_hashes(oracle, golden):
    """src/blockchain/blockchain.zig:135-137 compares parent_hash with the hash of the previous header: in every fixture,
    keccak256(rlp(header)) of each valid block equals its `hash` field and the next block's `parentHash` (87 headers)"""
    g = golden("fixture_states.json.gz")
    n = 0
    for t in g["tests"]:
        prev = t["genesis_hash"]
        for b in t["blocks"]:
            assert oracle.keccak256(bytes.fromhex(b["header_rlp"])).hex() == b["hash"]
            assert b["parentHash"] == prev
            prev = b["hash"]
            n += 1
    assert n == 87
